//! Raw bindings of include/lzkp_b200.h plus the two safe calls libzkp's `src/backend/snark.rs` needs.
//! Conventions (see the header): 0 = ok, negative = error, `lzkp_last_error()` has the message; all
//! byte formats are ark-serialize's; the caller owns every buffer.
#![allow(non_camel_case_types)]
use std::ffi::CStr;
use std::os::raw::{c_char, c_int, c_void};

#[repr(C)]
pub struct lzkp_pk {
    _private: [u8; 0],
}
#[repr(C)]
pub struct lzkp_vk {
    _private: [u8; 0],
}
#[repr(C)]
#[derive(Default, Clone, Copy)]
pub struct lzkp_pk_options {
    pub window_bits: c_int,
    pub table_budget_bytes: u64,
    pub max_chunk: u32,
    pub shard_index: u32,
    pub shard_count: u32,
}
pub const LZKP_CIRCUIT_EQUALITY: c_int = 0;
pub const LZKP_CIRCUIT_MEMBERSHIP: c_int = 1;

extern "C" {
    pub fn lzkp_init(devices: *const c_int, n_devices: c_int) -> c_int;
    pub fn lzkp_device_count() -> c_int;
    pub fn lzkp_last_error() -> *const c_char;
    pub fn lzkp_pk_load_ex(pk: *const u8, len: usize, validate: c_int, opt: *const lzkp_pk_options,
                           out: *mut *mut lzkp_pk) -> c_int;
    pub fn lzkp_pk_free(pk: *mut lzkp_pk);
    pub fn lzkp_circuit_builtin(pk: *mut lzkp_pk, kind: c_int, param: u32) -> c_int;
    pub fn lzkp_key_sizes(m: u32, n_inst: u32, n_wit: u32, pk_len: *mut usize, vk_len: *mut usize) -> c_int;
    pub fn lzkp_setup_builtin(kind: c_int, param: u32, toxic: *const u8, pk_out: *mut u8, pk_cap: usize,
                              vk_out: *mut u8, vk_cap: usize) -> c_int;
    pub fn lzkp_prove_batch(pk: *mut lzkp_pk, n: usize, z: *const u8, r: *const u8, s: *const u8,
                            proofs_out: *mut u8, status: *mut i32) -> c_int;
    pub fn lzkp_prove_equality_batch(pk: *mut lzkp_pk, n: usize, a: *const u64, b: *const u64,
                                     commitments: *const u8, r: *const u8, s: *const u8, proofs_out: *mut u8,
                                     commitments_out: *mut u8, status: *mut i32) -> c_int;
    pub fn lzkp_prove_membership_batch(pk: *mut lzkp_pk, n: usize, value: *const u64, sets: *const u64,
                                       set_len: *const u32, set_stride: u32, commitments: *const u8,
                                       r: *const u8, s: *const u8, proofs_out: *mut u8,
                                       commitments_out: *mut u8, status: *mut i32) -> c_int;
    pub fn lzkp_prove_equality_enveloped(pk: *mut lzkp_pk, n: usize, a: *const u64, b: *const u64, r: *const u8,
                                         s: *const u8, envelopes_out: *mut u8, envelope_len: *mut u32,
                                         status: *mut i32) -> c_int;
    pub fn lzkp_prove_membership_enveloped(pk: *mut lzkp_pk, n: usize, value: *const u64, sets: *const u64,
                                           set_len: *const u32, set_stride: u32, r: *const u8, s: *const u8,
                                           envelopes_out: *mut u8, envelope_stride: u32, envelope_len: *mut u32,
                                           status: *mut i32) -> c_int;
    pub fn lzkp_vk_load(vk: *const u8, len: usize, out: *mut *mut lzkp_vk) -> c_int;
    pub fn lzkp_vk_free(vk: *mut lzkp_vk);
    pub fn lzkp_vk_info(vk: *const lzkp_vk, info: *mut u64) -> c_int;
    pub fn lzkp_verify_batch(vk: *mut lzkp_vk, n: usize, proofs: *const u8, public_inputs: *const u8, n_pub: usize,
                             ok_out: *mut u8) -> c_int;
    pub fn lzkp_verify_batch_device(vk: *mut lzkp_vk, n: usize, d_proofs: *const c_void, d_public_inputs: *const c_void,
                                    n_pub: usize, d_ok: *mut c_void, stream: *mut c_void) -> c_int;
    pub fn lzkp_commit_value_snark(value: u64, out: *mut u8) -> c_int;
    pub fn lzkp_msm_g1(bases: *const u8, scalars: *const u8, n: usize, out: *mut u8) -> c_int;
    pub fn lzkp_msm_g2(bases: *const u8, scalars: *const u8, n: usize, out: *mut u8) -> c_int;
    pub fn lzkp_ntt(data: *mut u8, log_n: u32, inverse: c_int, coset: c_int) -> c_int;
    pub fn lzkp_prove_batch_device(pk: *mut lzkp_pk, n: usize, d_z: *const c_void, d_r: *const c_void,
                                   d_s: *const c_void, d_proofs: *mut c_void, d_status: *mut c_void,
                                   stream: *mut c_void) -> c_int;
}

pub fn last_error() -> String {
    unsafe { CStr::from_ptr(lzkp_last_error()).to_string_lossy().into_owned() }
}

/// A proving key resident in HBM, bound to one of libzkp's two circuits.  Send + Sync: the library
/// serializes calls on one key internally.
pub struct DevicePk(*mut lzkp_pk);
unsafe impl Send for DevicePk {}
unsafe impl Sync for DevicePk {}

impl DevicePk {
    /// `pk_bytes` = `ProvingKey::<Bn254>::serialize_uncompressed` (what snark.rs:97-101 persists).
    pub fn load(pk_bytes: &[u8], kind: c_int, param: u32, validate: bool) -> Result<Self, String> {
        let mut h: *mut lzkp_pk = std::ptr::null_mut();
        let opt = lzkp_pk_options::default();
        let rc = unsafe { lzkp_pk_load_ex(pk_bytes.as_ptr(), pk_bytes.len(), validate as c_int, &opt, &mut h) };
        if rc != 0 {
            return Err(last_error());
        }
        let pk = DevicePk(h);
        if unsafe { lzkp_circuit_builtin(pk.0, kind, param) } != 0 {
            return Err(last_error());
        }
        Ok(pk)
    }

    /// n equality proofs in one device call; `None` where the reference would return an empty Vec.
    pub fn prove_equality(&self, a: &[u64], b: &[u64], commitments: &[[u8; 32]], r: &[[u8; 32]],
                          s: &[[u8; 32]]) -> Result<Vec<Option<[u8; 256]>>, String> {
        let n = a.len();
        // the C side reads n entries from every slice: a shorter one would be an out-of-bounds read from safe code
        if b.len() != n || commitments.len() != n || r.len() != n || s.len() != n {
            return Err(format!("prove_equality: slice lengths differ (a {}, b {}, commitments {}, r {}, s {})",
                               n, b.len(), commitments.len(), r.len(), s.len()));
        }
        let mut proofs = vec![0u8; 256 * n];
        let mut status = vec![0i32; n];
        let rc = unsafe {
            lzkp_prove_equality_batch(self.0, n, a.as_ptr(), b.as_ptr(), commitments.as_ptr() as *const u8,
                                      r.as_ptr() as *const u8, s.as_ptr() as *const u8, proofs.as_mut_ptr(),
                                      std::ptr::null_mut(), status.as_mut_ptr())
        };
        if rc != 0 {
            return Err(last_error());
        }
        Ok((0..n).map(|i| if status[i] == 0 {
            let mut p = [0u8; 256];
            p.copy_from_slice(&proofs[256 * i..256 * (i + 1)]);
            Some(p)
        } else { None }).collect())
    }
}

impl Drop for DevicePk {
    fn drop(&mut self) {
        unsafe { lzkp_pk_free(self.0) }
    }
}
