//! Hand-written declarations of include/graph_witness.h (what bindgen generates in the reference, build.rs:9-26).
#![allow(non_camel_case_types)]
use std::ffi::{c_char, c_int, c_void};

pub const GW_ERROR_CODE_OK: c_int = 0;
pub const GW_ERROR_CODE_ERROR: c_int = 1;

#[repr(C)]
pub struct gw_status_t {
    pub code: c_int,
    pub error_msg: *mut c_char,
}

#[repr(C)]
pub struct gw_graph_t {
    _private: [u8; 0],
}

#[repr(C)]
#[derive(Default, Clone, Copy)]
pub struct gw_graph_info_t {
    pub n_nodes: u64,
    pub n_ops: u64,
    pub n_inputs: u32,
    pub n_witness: u32,
    pub n_input_signals: u32,
    pub n_instrs: u32,
    pub n_regs: u32,
    pub n_spill: u32,
    pub n_mul: u64,
    pub n_div: u64,
    pub n_spill_ld: u64,
    pub n_spill_st: u64,
    pub n_slots: u32,
    pub n_dot: u32,
    pub n_dot_mac: u32,
    pub n_mul_instr: u32,
    pub n_inversions: u32,
    pub threads: u32,
    pub sets_per_thread: u32,
    pub n_narrow_instr: u32,
    pub bit_eligible: u32,
    pub bit_luts: u32,
    pub bit_steps: u32,
    pub bit_wide: u32,
}

#[repr(C)]
pub struct gw_r1cs_t {
    _private: [u8; 0],
}

#[repr(C)]
#[derive(Default, Clone, Copy)]
pub struct gw_r1cs_info_t {
    pub n_wires: u32,
    pub n_pub_out: u32,
    pub n_pub_in: u32,
    pub n_prv_in: u32,
    pub n_constraints: u32,
    pub n_consts: u32,
    pub n_labels: u64,
    pub n_terms: u64,
    pub n_mac_terms: u64,
    pub n_chunks: u64,
}

pub const GW_R1CS_OK: u32 = 0xFFFF_FFFF;
pub const GW_R1CS_ABC_GROTH16: u32 = 1;
pub const GW_NTT_INVERSE: u32 = 1;
pub const GW_NTT_COSET: u32 = 2;

pub type gw_witness_chunk_fn = unsafe extern "C" fn(
    user: *mut c_void, device: c_int, first_set: usize, n_sets: usize, rows: *const u8, row_bytes: usize, flags: *const u32,
) -> c_int;

extern "C" {
    pub fn gw_calc_witness(inputs: *const c_char, graph_data: *const c_void, graph_data_len: usize,
                           wtns_data: *mut *mut c_void, wtns_len: *mut usize, status: *const gw_status_t) -> c_int;
    pub fn gw_graph_load(graph_data: *const c_void, graph_data_len: usize, graph: *mut *mut gw_graph_t,
                         status: *mut gw_status_t) -> c_int;
    pub fn gw_graph_free(graph: *mut gw_graph_t);
    pub fn gw_graph_info(graph: *const gw_graph_t, info: *mut gw_graph_info_t) -> c_int;
    pub fn gw_graph_input_signal(graph: *const gw_graph_t, i: u32, name: *mut *const c_char, offset: *mut u32,
                                 len: *mut u32) -> c_int;
    pub fn gw_calc_witness_batch(graph: *mut gw_graph_t, inputs: *const u8, n_sets: usize, witness: *mut u8,
                                 flags: *mut u32, n_gpus: c_int, status: *mut gw_status_t) -> c_int;
    pub fn gw_calc_witness_batch_stream(graph: *mut gw_graph_t, first_device: c_int, n_gpus: c_int, inputs: *const u8,
                                        n_sets: usize, chunk_sets: usize, f: gw_witness_chunk_fn, user: *mut c_void,
                                        status: *mut gw_status_t) -> c_int;
    pub fn gw_wtns_header(n_witness: u32, dst76: *mut u8);
    pub fn gw_r1cs_load(data: *const c_void, len: usize, r1cs: *mut *mut gw_r1cs_t, status: *mut gw_status_t) -> c_int;
    pub fn gw_r1cs_free(r1cs: *mut gw_r1cs_t);
    pub fn gw_r1cs_info(r1cs: *const gw_r1cs_t, info: *mut gw_r1cs_info_t) -> c_int;
    pub fn gw_r1cs_check_batch(r1cs: *mut gw_r1cs_t, witness: *const u8, n_sets: usize, row_pitch: usize,
                               first_failed: *mut u32, n_gpus: c_int, status: *mut gw_status_t) -> c_int;
    pub fn gw_r1cs_check_batch_device(r1cs: *mut gw_r1cs_t, device: c_int, d_witness: *const c_void, n_sets: usize,
                                      row_pitch: usize, d_first_failed: *mut u32, cuda_stream: *mut c_void,
                                      status: *mut gw_status_t) -> c_int;
    pub fn gw_calc_witness_batch_check(graph: *mut gw_graph_t, r1cs: *mut gw_r1cs_t, first_device: c_int, n_gpus: c_int,
                                       inputs: *const u8, n_sets: usize, witness: *mut u8, flags: *mut u32,
                                       first_failed: *mut u32, status: *mut gw_status_t) -> c_int;
    pub fn gw_r1cs_abc_len(r1cs: *const gw_r1cs_t, options: u32) -> u64;
    pub fn gw_r1cs_abc_batch(r1cs: *mut gw_r1cs_t, witness: *const u8, n_sets: usize, row_pitch: usize, abc: *mut u8,
                             abc_pitch: usize, options: u32, first_failed: *mut u32, n_gpus: c_int,
                             status: *mut gw_status_t) -> c_int;
    pub fn gw_r1cs_abc_batch_device(r1cs: *mut gw_r1cs_t, device: c_int, d_witness: *const c_void, n_sets: usize,
                                    row_pitch: usize, d_abc: *mut c_void, abc_pitch: usize, options: u32,
                                    d_first_failed: *mut u32, cuda_stream: *mut c_void,
                                    status: *mut gw_status_t) -> c_int;
    pub fn gw_fr_ntt_batch_device(device: c_int, d_data: *mut c_void, n_vectors: usize, log_n: u32, pitch: usize, flags: u32,
                                  cuda_stream: *mut c_void, status: *mut gw_status_t) -> c_int;
    pub fn gw_r1cs_quotient_batch(r1cs: *mut gw_r1cs_t, witness: *const u8, n_sets: usize, row_pitch: usize, h: *mut u8,
                                  h_pitch: usize, first_failed: *mut u32, n_gpus: c_int, status: *mut gw_status_t) -> c_int;
    pub fn gw_r1cs_quotient_batch_device(r1cs: *mut gw_r1cs_t, device: c_int, d_witness: *const c_void, n_sets: usize,
                                         row_pitch: usize, d_work: *mut c_void, work_pitch: usize, d_first_failed: *mut u32,
                                         cuda_stream: *mut c_void, status: *mut gw_status_t) -> c_int;
    pub fn gw_inputs_parse_batch_device(graph: *const gw_graph_t, device: c_int, text: *const c_char, text_len: usize,
                                        d_inputs: *mut c_void, max_sets: usize, n_sets: *mut usize, cuda_stream: *mut c_void,
                                        status: *mut gw_status_t) -> c_int;
    pub fn gw_calc_witness_latency_batch(graph: *mut gw_graph_t, first_device: c_int, n_gpus: c_int, inputs: *const u8,
                                         n_sets: usize, witness: *mut u8, flags: *mut u32, status: *mut gw_status_t) -> c_int;
    pub fn gw_calc_witness_latency_batch_device(graph: *mut gw_graph_t, device: c_int, d_inputs: *const c_void, n_sets: usize,
                                                d_witness: *mut c_void, d_flags: *mut u32, cuda_stream: *mut c_void,
                                                status: *mut gw_status_t) -> c_int;
}
