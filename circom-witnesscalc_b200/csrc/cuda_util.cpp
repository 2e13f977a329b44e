// Host-side device plumbing shared by the engine, the R1CS checker, the device input parser, the NTT and the C ABI.
#include "cuda_util.hpp"

#include <sched.h>
#include <stdio.h>
#include <stdlib.h>

#include <thread>
#include <vector>

namespace gw {

int cuda_device_count() {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
  return n;
}

void check_device(int device) {
  const int n = cuda_device_count();
  if (n == 0) throw Error(NO_DEVICE_ERROR);
  if (device < 0 || device >= n) throw Error("CUDA device index out of range");
}

// Pins the CALLING thread to the CPUs of the NUMA node the GPU hangs off (sysfs: numa_node of its PCI function,
// cpulist of that node), so that the thread's pinned allocations are node-local and its copies do not cross the
// socket interconnect.  Only ever called on threads this library created.  GW_NUMA=0 turns it off.
static void bind_thread_near_device(int device) {
  const char* numa = getenv("GW_NUMA");
  if (numa && *numa && atoi(numa) == 0) return;
  char bus[32] = {0};
  if (cudaDeviceGetPCIBusId(bus, (int)sizeof bus, device) != cudaSuccess) return;
  for (char* c = bus; *c; c++) if (*c >= 'A' && *c <= 'Z') *c = (char)(*c - 'A' + 'a');
  char path[160];
  snprintf(path, sizeof path, "/sys/bus/pci/devices/%s/numa_node", bus);
  FILE* f = fopen(path, "r");
  if (!f) return;
  int node = -1;
  if (fscanf(f, "%d", &node) != 1) node = -1;
  fclose(f);
  if (node < 0) return;
  snprintf(path, sizeof path, "/sys/devices/system/node/node%d/cpulist", node);
  f = fopen(path, "r");
  if (!f) return;
  char list[4096] = {0};
  const bool got = fgets(list, (int)sizeof list, f) != nullptr;
  fclose(f);
  if (!got) return;
  cpu_set_t allowed, want;
  CPU_ZERO(&allowed); CPU_ZERO(&want);
  if (sched_getaffinity(0, sizeof allowed, &allowed) != 0) return;
  int n_want = 0;
  for (const char* c = list; *c;) {
    while (*c == ',' || *c == ' ' || *c == '\n') c++;
    if (*c < '0' || *c > '9') break;
    long lo = strtol(c, const_cast<char**>(&c), 10), hi = lo;
    if (*c == '-') hi = strtol(c + 1, const_cast<char**>(&c), 10);
    for (long k = lo; k <= hi && k < CPU_SETSIZE; k++) if (CPU_ISSET((int)k, &allowed)) { CPU_SET((int)k, &want); n_want++; }
  }
  if (n_want > 0) sched_setaffinity(0, sizeof want, &want);
}

void run_shards(size_t B, int n_gpus, int first_device, const std::function<void(int, size_t, size_t)>& fn) {
  std::vector<std::thread> th;
  std::vector<std::string> errs(n_gpus);
  for (int g = 0; g < n_gpus; g++) {
    const size_t lo = B * g / n_gpus, hi = B * (g + 1) / n_gpus;
    if (hi == lo) continue;
    th.emplace_back([=, &errs, &fn]() {
      try {
        bind_thread_near_device(first_device + g);
        fn(first_device + g, lo, hi);
      } catch (const std::exception& e) { errs[g] = e.what(); }
    });
  }
  for (auto& t : th) t.join();
  for (auto& e : errs) if (!e.empty()) throw Error(e);
}

}  // namespace gw
