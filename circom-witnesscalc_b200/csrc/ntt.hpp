// Batched number-theoretic transforms over the BN254 scalar field (gw_fr_ntt_batch_device) and the Groth16 quotient
// transforms of ABC rows (R1cs::quotient_device).  Kernels and tables: ntt.cu; arithmetic: ntt.cuh.
#pragma once
#include <stddef.h>
#include <stdint.h>

namespace gw {

static const uint32_t NTT_INVERSE = 1u;      // GW_NTT_INVERSE
static const uint32_t NTT_COSET = 2u;        // GW_NTT_COSET
static const uint32_t NTT_MAX_LOG = 24;      // supported domains: 2^0 .. 2^24

// checks the arguments of ntt_batch_device without touching a device (throws gw::Error); returns the effective pitch
size_t ntt_check_args(const void* d_data, uint32_t log_n, size_t pitch, uint32_t flags);

// in place: vector v at d_data + v * pitch, 2^log_n canonical 32-byte entries out, any 256-bit values in; natural order
void ntt_batch_device(int device, void* d_data, size_t n_vectors, uint32_t log_n, size_t pitch, uint32_t flags, void* stream);

// B rows of d_work (row r at d_work + r * pitch, pitch >= 3 * n * 32, a multiple of 16): A | B | C of n = 2^log_n
// entries each, canonical.  Leaves h_i = A_odd[i] * B_odd[i] - C_odd[i] in the first n entries of each row, where
// X_odd is the forward transform on the coset g * <w_n> (g = w_2n) of the inverse transform of X.  The rest of each row
// is clobbered.
void ntt_quotient_device(int device, void* d_work, size_t B, uint32_t log_n, size_t pitch, void* stream);

}  // namespace gw
