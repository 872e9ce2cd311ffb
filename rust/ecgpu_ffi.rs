//! ecgpu_ffi.rs — reference-side binding of libecgpu.so (SOURCE ONLY: this repository's environment has no Rust
//! toolchain, so this file is not compiled here; the compiled equivalents are elliptic-curves_b200/host/ecgpu.hpp,
//! exercised method by method by tests/test_host_cpp.py, and the ctypes binding elliptic-curves_b200/ecgpu/__init__.py).
//! It would live in the reference as `k256/src/arithmetic/gpu.rs` behind a `gpu` feature.  INTEGRATION.md shows where
//! each wrapper plugs into the existing trait surface; the wrappers here work on the crates' PUBLIC byte encodings
//! (`Scalar::to_bytes`, `AffineCoordinates::{x, y}`, `FieldElement::to_bytes`), never on the internal limb layouts.
#![allow(non_camel_case_types, dead_code)]

use core::ffi::c_char;

#[repr(C)]
pub struct ecg_ctx {
    _private: [u8; 0],
}

pub const ECG_OK: i32 = 0;
pub const ECG_EINVAL: i32 = 1;
pub const ECG_ESCALAR_RANGE: i32 = 2;
pub const ECG_ENOT_ON_CURVE: i32 = 3;
pub const ECG_ECUDA: i32 = 4;
pub const ECG_ENCCL: i32 = 5;
pub const ECG_ENOMEM: i32 = 6;
pub const ECG_SECP256K1: i32 = 0;
pub const ECG_NISTP256: i32 = 1;
pub const ECG_FLAG_DEVICE_PTRS: u32 = 1;
pub const ECG_FLAG_ZEROIZE: u32 = 2;
pub const ECG_FLAG_CONSTTIME: u32 = 4;
pub const ECG_FOP_ADD: i32 = 0;
pub const ECG_FOP_SUB: i32 = 1;
pub const ECG_FOP_NEG: i32 = 2;
pub const ECG_FOP_MUL: i32 = 3;
pub const ECG_FOP_SQR: i32 = 4;
pub const ECG_FOP_INV: i32 = 5;

#[link(name = "ecgpu")]
unsafe extern "C" {
    pub fn ecg_ctx_create(device_ids: *const i32, n_devices: i32, flags: u32, out: *mut *mut ecg_ctx) -> i32;
    pub fn ecg_ctx_destroy(ctx: *mut ecg_ctx);
    pub fn ecg_last_error(ctx: *const ecg_ctx) -> *const c_char;
    pub fn ecg_last_error_index(ctx: *const ecg_ctx) -> usize;
    pub fn ecg_ctx_set_stream(ctx: *mut ecg_ctx, cuda_stream: *mut core::ffi::c_void) -> i32;
    /// `ProjectivePoint * Scalar` over a batch (k256/src/arithmetic/mul.rs:236-295)
    pub fn ecg_mul_batch(ctx: *mut ecg_ctx, curve: i32, n: usize, k: *const u8, p_xy: *const u8, p_inf: *const u8,
                         out_xy: *mut u8, out_inf: *mut u8) -> i32;
    /// x coordinate only: `(public * secret).to_affine().x` (k256/src/ecdh.rs:46-60)
    pub fn ecg_mul_batch_x(ctx: *mut ecg_ctx, curve: i32, n: usize, k: *const u8, p_xy: *const u8, p_inf: *const u8,
                           out_x: *mut u8, out_inf: *mut u8) -> i32;
    /// `ProjectivePoint::mul_by_generator` (mul.rs:180-232)
    pub fn ecg_mul_gen_batch(ctx: *mut ecg_ctx, curve: i32, n: usize, k: *const u8, out_xy: *mut u8, out_inf: *mut u8) -> i32;
    /// `LinearCombination::lincomb` (mul.rs:66-175)
    pub fn ecg_lincomb(ctx: *mut ecg_ctx, curve: i32, n: usize, k: *const u8, p_xy: *const u8, p_inf: *const u8,
                       out_xy: *mut u8, out_inf: *mut u8) -> i32;
    /// the same sum left as a Jacobian X||Y||Z (one per rank; combined by `ecg_point_sum`)
    pub fn ecg_lincomb_partial(ctx: *mut ecg_ctx, curve: i32, n: usize, k: *const u8, p_xy: *const u8, p_inf: *const u8,
                               out_xyz: *mut u8) -> i32;
    pub fn ecg_point_sum(ctx: *mut ecg_ctx, curve: i32, m: usize, xyz: *const u8, out_xy: *mut u8, out_inf: *mut u8) -> i32;
    /// `MulByGeneratorVartime::mul_by_generator_and_mul_add_vartime` (mul.rs:303-310)
    pub fn ecg_mul_gen_add_batch(ctx: *mut ecg_ctx, curve: i32, n: usize, a: *const u8, b: *const u8, p_xy: *const u8,
                                 p_inf: *const u8, out_xy: *mut u8, out_inf: *mut u8) -> i32;
    /// `BatchNormalize::batch_normalize` on Jacobian (X:Y:Z), x = X/Z^2
    pub fn ecg_batch_normalize(ctx: *mut ecg_ctx, curve: i32, n: usize, xyz: *const u8, out_xy: *mut u8, out_inf: *mut u8) -> i32;
    /// `BatchNormalize::batch_normalize` on the reference's own homogeneous (X:Y:Z), x = X/Z (projective.rs:367-391)
    pub fn ecg_batch_normalize_hom(ctx: *mut ecg_ctx, curve: i32, n: usize, xyz: *const u8, out_xy: *mut u8, out_inf: *mut u8) -> i32;
    /// `FieldElement::{add, sub, neg, mul, square, invert}` (field.rs:116-196)
    pub fn ecg_field_op_batch(ctx: *mut ecg_ctx, curve: i32, op: i32, n: usize, a: *const u8, b: *const u8, out: *mut u8) -> i32;
    /// `GroupDigest::hash_from_bytes` / `encode_from_bytes` over a batch (hash2curve/src/group_digest.rs:88-118):
    /// message i = msgs[offsets[i]..offsets[i+1]], n + 1 offsets; secp256k1 / P-256 XMD:SHA-256 SSWU suites
    pub fn ecg_hash_to_curve_batch(ctx: *mut ecg_ctx, curve: i32, n: usize, msgs: *const u8, offsets: *const u64, dst: *const u8,
                                   dst_len: usize, nonuniform: i32, out_xy: *mut u8, out_inf: *mut u8) -> i32;
    /// `hash2curve::hash_to_scalar` over a batch (group_digest.rs:131-143)
    pub fn ecg_hash_to_scalar_batch(ctx: *mut ecg_ctx, curve: i32, n: usize, msgs: *const u8, offsets: *const u64, dst: *const u8,
                                    dst_len: usize, out: *mut u8) -> i32;
    /// `FieldElement::sqrt` (field.rs:200-235)
    pub fn ecg_field_sqrt_batch(ctx: *mut ecg_ctx, curve: i32, n: usize, a: *const u8, out: *mut u8, is_square: *mut u8) -> i32;
    /// `schnorr::VerifyingKey::verify_raw` over a batch (schnorr/verifying.rs:76-99)
    pub fn ecg_schnorr_verify_batch(ctx: *mut ecg_ctx, n: usize, pk_x: *const u8, msg32: *const u8, sig64: *const u8,
                                    valid: *mut u8) -> i32;
    /// `ecdsa::VerifyingKey::verify_prehash` over a batch (ecdsa.rs:93-121)
    pub fn ecg_ecdsa_verify_batch(ctx: *mut ecg_ctx, curve: i32, n: usize, z32: *const u8, sig64: *const u8, q_xy: *const u8,
                                  low_s_only: i32, valid: *mut u8) -> i32;
    /// `ecdsa::VerifyingKey::recover_from_prehash` over a batch (k256/src/ecdsa.rs:45-88), `recid` = `RecoveryId::to_byte`
    pub fn ecg_ecdsa_recover_batch(ctx: *mut ecg_ctx, curve: i32, n: usize, z32: *const u8, sig64: *const u8, recid: *const u8,
                                   low_s_only: i32, out_xy: *mut u8, valid: *mut u8) -> i32;
    /// `sm2::dsa::VerifyingKey::verify_prehash` over a batch (sm2/src/dsa/verifying.rs:138-175)
    pub fn ecg_sm2dsa_verify_batch(ctx: *mut ecg_ctx, n: usize, e32: *const u8, sig64: *const u8, q_xy: *const u8, valid: *mut u8) -> i32;
    /// `sm2::pke::EncryptingKey::encrypt` over a batch with the caller's ephemeral scalars (sm2/src/pke/encrypting.rs:166-230)
    pub fn ecg_sm2pke_encrypt_batch(ctx: *mut ecg_ctx, n: usize, msgs: *const u8, offsets: *const u64, k32: *const u8, pb_xy: *const u8,
                                    mode: i32, compressed: i32, out: *mut u8, status: *mut u8) -> i32;
    /// `sm2::pke::DecryptingKey::decrypt` over a batch (sm2/src/pke/decrypting.rs:174-222)
    pub fn ecg_sm2pke_decrypt_batch(ctx: *mut ecg_ctx, n: usize, cts: *const u8, offsets: *const u64, d32: *const u8, mode: i32,
                                    out: *mut u8, pt_len: *mut u64, valid: *mut u8) -> i32;
    /// `AffinePoint::decompress` over a batch (primeorder/src/affine.rs:179-198)
    pub fn ecg_decompress_batch(ctx: *mut ecg_ctx, curve: i32, n: usize, sec1_33: *const u8, out_xy: *mut u8,
                                out_inf: *mut u8, valid: *mut u8) -> i32;
    pub fn ecg_kernel_launches(ctx: *const ecg_ctx) -> u64;
}

#[derive(Debug)]
pub enum GpuError {
    Cuda(String),
    /// `Scalar::from_repr` would have returned `None` for this element
    ScalarRange(usize),
    /// `AffinePoint::from_coordinates` would have returned `None` for this element
    NotOnCurve(usize),
    /// a zero secret scalar, an identity peer or an identity result where the reference's types rule them out
    Identity(usize),
    Invalid,
}

pub type Bytes32 = [u8; 32];
pub type PointXY = [u8; 64]; // x || y, canonical big-endian
pub type PointXYZ = [u8; 96]; // X || Y || Z
pub type Sec1 = [u8; 33];

/// One `ecg_ctx`; `!Sync` by construction (raw pointer): one engine per calling thread.
pub struct GpuEngine {
    ctx: *mut ecg_ctx,
    curve: i32,
}

impl GpuEngine {
    /// `zeroize`: clear the device-side copies of inputs and intermediates after every call (ECG_FLAG_ZEROIZE).
    /// `consttime`: `ECG_FLAG_CONSTTIME` — masked table selects, branch-free sign folding, `k*G` through the variable-base
    /// routine, per-term `lincomb`: the ctx to use where the scalars are secret (the default is the `*_vartime` analogue).
    pub fn new(curve: i32, devices: &[i32], zeroize: bool, consttime: bool) -> Result<Self, GpuError> {
        let mut ctx = core::ptr::null_mut();
        let flags = (if zeroize { ECG_FLAG_ZEROIZE } else { 0 }) | (if consttime { ECG_FLAG_CONSTTIME } else { 0 });
        // SAFETY: out-pointer is valid; the library copies `devices` before returning.
        match unsafe { ecg_ctx_create(devices.as_ptr(), devices.len() as i32, flags, &mut ctx) } {
            ECG_OK => Ok(Self { ctx, curve }),
            _ => Err(GpuError::Cuda("ecg_ctx_create failed: no CUDA device (there is no CPU fallback)".into())),
        }
    }

    /// `out[i] = k[i] * P[i]` — batch form of `Mul<Scalar> for ProjectivePoint` / `MulVartime`.
    pub fn mul_batch(&mut self, k: &[Bytes32], p_xy: &[PointXY], p_inf: &[u8]) -> Result<(Vec<PointXY>, Vec<u8>), GpuError> {
        let n = k.len();
        assert!(p_xy.len() == n && p_inf.len() == n);
        let (mut out_xy, mut out_inf) = (vec![[0u8; 64]; n], vec![0u8; n]);
        // SAFETY: all slices hold exactly n elements of the layout include/ecgpu.h specifies.
        let rc = unsafe {
            ecg_mul_batch(self.ctx, self.curve, n, k.as_ptr().cast(), p_xy.as_ptr().cast(), p_inf.as_ptr(),
                          out_xy.as_mut_ptr().cast(), out_inf.as_mut_ptr())
        };
        self.check(rc).map(|_| (out_xy, out_inf))
    }

    /// `out[i] = k[i] * G` — `ProjectivePoint::mul_by_generator[_vartime]` / `MulBackend::mul_by_generator`.
    pub fn mul_by_generator_batch(&mut self, k: &[Bytes32]) -> Result<(Vec<PointXY>, Vec<u8>), GpuError> {
        let n = k.len();
        let (mut out_xy, mut out_inf) = (vec![[0u8; 64]; n], vec![0u8; n]);
        // SAFETY: as above.
        let rc = unsafe { ecg_mul_gen_batch(self.ctx, self.curve, n, k.as_ptr().cast(), out_xy.as_mut_ptr().cast(), out_inf.as_mut_ptr()) };
        self.check(rc).map(|_| (out_xy, out_inf))
    }

    /// `sum_i k[i] * P[i]` — `LinearCombination<[(ProjectivePoint, Scalar)]>::lincomb` (the caller passes the affine
    /// images of its points: `batch_normalize` below, or the crate's own).  Returns `(x || y, is_identity)`.
    pub fn lincomb(&mut self, k: &[Bytes32], p_xy: &[PointXY], p_inf: &[u8]) -> Result<(PointXY, bool), GpuError> {
        let n = k.len();
        assert!(p_xy.len() == n && p_inf.len() == n);
        let (mut out_xy, mut out_inf) = ([0u8; 64], 0u8);
        // SAFETY: as above; the two outputs are 64 + 1 bytes.
        let rc = unsafe {
            ecg_lincomb(self.ctx, self.curve, n, k.as_ptr().cast(), p_xy.as_ptr().cast(), p_inf.as_ptr(), out_xy.as_mut_ptr(), &mut out_inf)
        };
        self.check(rc).map(|_| (out_xy, out_inf != 0))
    }

    /// This rank's share of a distributed `lincomb`: the un-normalised sum (Jacobian X || Y || Z).
    pub fn lincomb_partial(&mut self, k: &[Bytes32], p_xy: &[PointXY], p_inf: &[u8]) -> Result<PointXYZ, GpuError> {
        let n = k.len();
        assert!(p_xy.len() == n && p_inf.len() == n);
        let mut out = [0u8; 96];
        // SAFETY: as above.
        let rc = unsafe { ecg_lincomb_partial(self.ctx, self.curve, n, k.as_ptr().cast(), p_xy.as_ptr().cast(), p_inf.as_ptr(), out.as_mut_ptr()) };
        self.check(rc).map(|_| out)
    }

    /// Sum of the ranks' partial points, normalised.
    pub fn point_sum(&mut self, parts: &[PointXYZ]) -> Result<(PointXY, bool), GpuError> {
        let (mut out_xy, mut out_inf) = ([0u8; 64], 0u8);
        // SAFETY: as above.
        let rc = unsafe { ecg_point_sum(self.ctx, self.curve, parts.len(), parts.as_ptr().cast(), out_xy.as_mut_ptr(), &mut out_inf) };
        self.check(rc).map(|_| (out_xy, out_inf != 0))
    }

    /// `a[i] * G + b[i] * P[i]` — `MulByGeneratorVartime::mul_by_generator_and_mul_add_vartime`.
    pub fn mul_by_generator_and_mul_add_batch(&mut self, a: &[Bytes32], b: &[Bytes32], p_xy: &[PointXY], p_inf: &[u8])
        -> Result<(Vec<PointXY>, Vec<u8>), GpuError> {
        let n = a.len();
        assert!(b.len() == n && p_xy.len() == n && p_inf.len() == n);
        let (mut out_xy, mut out_inf) = (vec![[0u8; 64]; n], vec![0u8; n]);
        // SAFETY: as above.
        let rc = unsafe {
            ecg_mul_gen_add_batch(self.ctx, self.curve, n, a.as_ptr().cast(), b.as_ptr().cast(), p_xy.as_ptr().cast(), p_inf.as_ptr(),
                                  out_xy.as_mut_ptr().cast(), out_inf.as_mut_ptr())
        };
        self.check(rc).map(|_| (out_xy, out_inf))
    }

    /// `BatchNormalize::batch_normalize` for `ProjectivePoint`s given as the reference's homogeneous (X : Y : Z).
    pub fn batch_normalize(&mut self, xyz: &[PointXYZ]) -> Result<(Vec<PointXY>, Vec<u8>), GpuError> {
        let n = xyz.len();
        let (mut out_xy, mut out_inf) = (vec![[0u8; 64]; n], vec![0u8; n]);
        // SAFETY: as above.
        let rc = unsafe { ecg_batch_normalize_hom(self.ctx, self.curve, n, xyz.as_ptr().cast(), out_xy.as_mut_ptr().cast(), out_inf.as_mut_ptr()) };
        self.check(rc).map(|_| (out_xy, out_inf))
    }

    /// Same for Jacobian inputs (x = X / Z^2), the form `lincomb_partial` produces.
    pub fn batch_normalize_jacobian(&mut self, xyz: &[PointXYZ]) -> Result<(Vec<PointXY>, Vec<u8>), GpuError> {
        let n = xyz.len();
        let (mut out_xy, mut out_inf) = (vec![[0u8; 64]; n], vec![0u8; n]);
        // SAFETY: as above.
        let rc = unsafe { ecg_batch_normalize(self.ctx, self.curve, n, xyz.as_ptr().cast(), out_xy.as_mut_ptr().cast(), out_inf.as_mut_ptr()) };
        self.check(rc).map(|_| (out_xy, out_inf))
    }

    /// `FieldElement` arithmetic over a batch (`op` = ECG_FOP_*; `b` ignored by the unary operations).
    pub fn field_op_batch(&mut self, op: i32, a: &[Bytes32], b: Option<&[Bytes32]>) -> Result<Vec<Bytes32>, GpuError> {
        let n = a.len();
        let mut out = vec![[0u8; 32]; n];
        let bp = match b {
            Some(s) => {
                assert!(s.len() == n);
                s.as_ptr().cast()
            }
            None => core::ptr::null(),
        };
        // SAFETY: as above.
        let rc = unsafe { ecg_field_op_batch(self.ctx, self.curve, op, n, a.as_ptr().cast(), bp, out.as_mut_ptr().cast()) };
        self.check(rc).map(|_| out)
    }

    /// `FieldElement::sqrt` over a batch: `None` where the input is not a square.
    pub fn field_sqrt_batch(&mut self, a: &[Bytes32]) -> Result<Vec<Option<Bytes32>>, GpuError> {
        let n = a.len();
        let (mut out, mut ok) = (vec![[0u8; 32]; n], vec![0u8; n]);
        // SAFETY: as above.
        let rc = unsafe { ecg_field_sqrt_batch(self.ctx, self.curve, n, a.as_ptr().cast(), out.as_mut_ptr().cast(), ok.as_mut_ptr()) };
        self.check(rc).map(|_| out.into_iter().zip(ok).map(|(r, o)| if o != 0 { Some(r) } else { None }).collect())
    }

    /// `GroupDigest::hash_from_bytes` (`nonuniform = false`) / `encode_from_bytes` (`true`) for a batch of messages.
    pub fn hash_to_curve_batch(&mut self, msgs: &[&[u8]], dst: &[u8], nonuniform: bool) -> Result<(Vec<[u8; 64]>, Vec<u8>), GpuError> {
        let n = msgs.len();
        let mut offsets = Vec::with_capacity(n + 1);
        let mut data = Vec::new();
        offsets.push(0u64);
        for m in msgs {
            data.extend_from_slice(m);
            offsets.push(data.len() as u64);
        }
        let (mut out_xy, mut out_inf) = (vec![[0u8; 64]; n], vec![0u8; n]);
        // SAFETY: `data` holds offsets[n] bytes, `offsets` n + 1 values, the outputs n records; all outlive the call.
        let rc = unsafe {
            ecg_hash_to_curve_batch(self.ctx, self.curve, n, data.as_ptr(), offsets.as_ptr(), dst.as_ptr(), dst.len(), nonuniform as i32,
                                    out_xy.as_mut_ptr().cast(), out_inf.as_mut_ptr())
        };
        self.check(rc).map(|_| (out_xy, out_inf))
    }

    /// `hash2curve::hash_to_scalar` for a batch of messages: big-endian scalars below the group order.
    pub fn hash_to_scalar_batch(&mut self, msgs: &[&[u8]], dst: &[u8]) -> Result<Vec<Bytes32>, GpuError> {
        let n = msgs.len();
        let mut offsets = Vec::with_capacity(n + 1);
        let mut data = Vec::new();
        offsets.push(0u64);
        for m in msgs {
            data.extend_from_slice(m);
            offsets.push(data.len() as u64);
        }
        let mut out = vec![[0u8; 32]; n];
        // SAFETY: as above.
        let rc = unsafe {
            ecg_hash_to_scalar_batch(self.ctx, self.curve, n, data.as_ptr(), offsets.as_ptr(), dst.as_ptr(), dst.len(), out.as_mut_ptr().cast())
        };
        self.check(rc).map(|_| out)
    }

    /// BIP340 batch verification: one bool per (key, message, signature).  secp256k1 only.
    pub fn schnorr_verify_batch(&mut self, pk: &[Bytes32], msg: &[Bytes32], sig: &[[u8; 64]]) -> Result<Vec<bool>, GpuError> {
        let n = pk.len();
        assert!(msg.len() == n && sig.len() == n);
        let mut valid = vec![0u8; n];
        // SAFETY: as above.
        let rc = unsafe { ecg_schnorr_verify_batch(self.ctx, n, pk.as_ptr().cast(), msg.as_ptr().cast(), sig.as_ptr().cast(), valid.as_mut_ptr()) };
        self.check(rc).map(|_| valid.into_iter().map(|v| v != 0).collect())
    }

    /// ECDSA `verify_prehash` over a batch; `low_s_only` = `EcdsaCurve::NORMALIZE_S`.
    pub fn ecdsa_verify_batch(&mut self, z: &[Bytes32], sig: &[[u8; 64]], q_xy: &[PointXY], low_s_only: bool) -> Result<Vec<bool>, GpuError> {
        let n = z.len();
        assert!(sig.len() == n && q_xy.len() == n);
        let mut valid = vec![0u8; n];
        // SAFETY: as above.
        let rc = unsafe {
            ecg_ecdsa_verify_batch(self.ctx, self.curve, n, z.as_ptr().cast(), sig.as_ptr().cast(), q_xy.as_ptr().cast(), low_s_only as i32,
                                   valid.as_mut_ptr())
        };
        self.check(rc).map(|_| valid.into_iter().map(|v| v != 0).collect())
    }

    /// `VerifyingKey::recover_from_prehash` over a batch: `None` where the reference returns `Err`.
    pub fn ecdsa_recover_batch(&mut self, z: &[Bytes32], sig: &[[u8; 64]], recid: &[u8], low_s_only: bool) -> Result<Vec<Option<PointXY>>, GpuError> {
        let n = z.len();
        assert!(sig.len() == n && recid.len() == n);
        let mut out = vec![[0u8; 64]; n];
        let mut valid = vec![0u8; n];
        // SAFETY: as above.
        let rc = unsafe {
            ecg_ecdsa_recover_batch(self.ctx, self.curve, n, z.as_ptr().cast(), sig.as_ptr().cast(), recid.as_ptr(), low_s_only as i32,
                                    out.as_mut_ptr().cast(), valid.as_mut_ptr())
        };
        self.check(rc).map(|_| out.into_iter().zip(valid).map(|(q, v)| if v != 0 { Some(q) } else { None }).collect())
    }

    /// SM2DSA `verify_prehash` over a batch: `e` = SM3(Z_A || M) per signature (`VerifyingKey::hash_msg`).
    pub fn sm2dsa_verify_batch(&mut self, e: &[Bytes32], sig: &[[u8; 64]], q_xy: &[PointXY]) -> Result<Vec<bool>, GpuError> {
        let n = e.len();
        assert!(sig.len() == n && q_xy.len() == n);
        let mut valid = vec![0u8; n];
        // SAFETY: as above.
        let rc = unsafe { ecg_sm2dsa_verify_batch(self.ctx, n, e.as_ptr().cast(), sig.as_ptr().cast(), q_xy.as_ptr().cast(), valid.as_mut_ptr()) };
        self.check(rc).map(|_| valid.into_iter().map(|v| v != 0).collect())
    }

    /// `EncryptingKey::encrypt` (mode C1C3C2 = 0 / C1C2C3 = 1, digest SM3) over a slice of messages for one recipient key,
    /// with the caller's ephemeral scalars (the reference draws k from its RNG inside `encrypt`).  `Ok(None)` at i where
    /// the KDF output was all zero (draw another k and retry that message) or the message / k was refused.
    pub fn sm2pke_encrypt_batch(&mut self, pb: &PointXY, k: &[Bytes32], msgs: &[&[u8]], mode: i32, compressed: bool)
                                -> Result<Vec<Option<Vec<u8>>>, GpuError> {
        let n = msgs.len();
        assert!(k.len() == n);
        let ovh = 32 + if compressed { 33 } else { 65 };
        let mut offsets = Vec::with_capacity(n + 1);
        let mut data = Vec::new();
        offsets.push(0u64);
        for m in msgs {
            data.extend_from_slice(m);
            offsets.push(data.len() as u64);
        }
        let pbs: Vec<PointXY> = vec![*pb; n];
        let (mut out, mut status) = (vec![0u8; data.len() + n * ovh], vec![0u8; n]);
        // SAFETY: `data` holds offsets[n] bytes, `offsets` n + 1 values, `k` / `pbs` n records, `out` offsets[n] + n * ovh bytes.
        let rc = unsafe {
            ecg_sm2pke_encrypt_batch(self.ctx, n, data.as_ptr(), offsets.as_ptr(), k.as_ptr().cast(), pbs.as_ptr().cast(), mode,
                                     compressed as i32, out.as_mut_ptr(), status.as_mut_ptr())
        };
        self.check(rc).map(|_| (0..n).map(|i| {
            let (lo, hi) = (offsets[i] as usize + i * ovh, offsets[i + 1] as usize + (i + 1) * ovh);
            if status[i] == 1 { Some(out[lo..hi].to_vec()) } else { None }
        }).collect())
    }

    /// `DecryptingKey::decrypt` over a slice of ciphertexts under one secret key: `None` where the reference returns `Err`.
    pub fn sm2pke_decrypt_batch(&mut self, d: &Bytes32, cts: &[&[u8]], mode: i32) -> Result<Vec<Option<Vec<u8>>>, GpuError> {
        let n = cts.len();
        let mut offsets = Vec::with_capacity(n + 1);
        let mut data = Vec::new();
        offsets.push(0u64);
        for c in cts {
            data.extend_from_slice(c);
            offsets.push(data.len() as u64);
        }
        let ds: Vec<Bytes32> = vec![*d; n];
        let (mut out, mut len, mut valid) = (vec![0u8; data.len()], vec![0u64; n], vec![0u8; n]);
        // SAFETY: `data` / `out` hold offsets[n] bytes, `offsets` n + 1 values, `ds` / `len` / `valid` n records.
        let rc = unsafe {
            ecg_sm2pke_decrypt_batch(self.ctx, n, data.as_ptr(), offsets.as_ptr(), ds.as_ptr().cast(), mode, out.as_mut_ptr(), len.as_mut_ptr(),
                                     valid.as_mut_ptr())
        };
        self.check(rc).map(|_| (0..n).map(|i| {
            let lo = offsets[i] as usize;
            if valid[i] != 0 { Some(out[lo..lo + len[i] as usize].to_vec()) } else { None }
        }).collect())
    }

    /// `AffinePoint::decompress` over a batch of SEC1 compressed records: `None` where decoding fails.
    pub fn decompress_batch(&mut self, rec: &[Sec1]) -> Result<Vec<Option<(PointXY, bool)>>, GpuError> {
        let n = rec.len();
        let (mut out_xy, mut out_inf, mut valid) = (vec![[0u8; 64]; n], vec![0u8; n], vec![0u8; n]);
        // SAFETY: as above.
        let rc = unsafe {
            ecg_decompress_batch(self.ctx, self.curve, n, rec.as_ptr().cast(), out_xy.as_mut_ptr().cast(), out_inf.as_mut_ptr(), valid.as_mut_ptr())
        };
        self.check(rc).map(|_| (0..n).map(|i| if valid[i] != 0 { Some((out_xy[i], out_inf[i] != 0)) } else { None }).collect())
    }

    /// ECDH over a batch: the x coordinates of `secret[i] * public[i]`.  VARIABLE TIME in the secret (window tables are
    /// indexed by scalar digits) — the reference's `diffie_hellman` is constant time, hence the name; create the engine
    /// with `zeroize = true`.  Zero scalars and identity results are errors, as `NonZeroScalar` / `PublicKey` imply.
    pub fn diffie_hellman_vartime(&mut self, secret: &[Bytes32], public_xy: &[PointXY]) -> Result<Vec<Bytes32>, GpuError> {
        let n = secret.len();
        assert!(public_xy.len() == n);
        if let Some(i) = secret.iter().position(|s| s.iter().all(|&b| b == 0)) {
            return Err(GpuError::Identity(i));
        }
        let (mut out_x, mut out_inf) = (vec![[0u8; 32]; n], vec![0u8; n]);
        // SAFETY: as above; a null P_inf means "no identities among the inputs".
        let rc = unsafe {
            ecg_mul_batch_x(self.ctx, self.curve, n, secret.as_ptr().cast(), public_xy.as_ptr().cast(), core::ptr::null(),
                            out_x.as_mut_ptr().cast(), out_inf.as_mut_ptr())
        };
        self.check(rc)?;
        match out_inf.iter().position(|&f| f != 0) {
            Some(i) => Err(GpuError::Identity(i)),
            None => Ok(out_x),
        }
    }

    fn check(&self, rc: i32) -> Result<(), GpuError> {
        match rc {
            ECG_OK => Ok(()),
            // SAFETY: ctx is live for the lifetime of self.
            ECG_ESCALAR_RANGE => Err(GpuError::ScalarRange(unsafe { ecg_last_error_index(self.ctx) })),
            ECG_ENOT_ON_CURVE => Err(GpuError::NotOnCurve(unsafe { ecg_last_error_index(self.ctx) })),
            ECG_EINVAL => Err(GpuError::Invalid),
            _ => Err(GpuError::Cuda(unsafe { core::ffi::CStr::from_ptr(ecg_last_error(self.ctx)) }.to_string_lossy().into_owned())),
        }
    }
}

impl Drop for GpuEngine {
    fn drop(&mut self) {
        // SAFETY: created by ecg_ctx_create, destroyed exactly once.
        unsafe { ecg_ctx_destroy(self.ctx) }
    }
}

// ---- trait-shaped adapters (k256 types) -------------------------------------------------------------------------------
// These are the functions INTEGRATION.md section 3 plugs into the reference's seams; they only use public API:
//   Scalar::to_bytes (k256/src/arithmetic/scalar.rs:96-98), AffineCoordinates::{x, y} and AffinePoint::from_coordinates
//   (k256/src/arithmetic/affine.rs:131-155), ProjectivePoint::batch_normalize (k256/src/arithmetic/projective.rs:345-365).
#[cfg(feature = "k256-types")]
pub mod k256_glue {
    use super::*;
    use elliptic_curve::{group::Curve, point::AffineCoordinates, BatchNormalize, PrimeField};
    use k256::{AffinePoint, FieldBytes, ProjectivePoint, Scalar};

    fn pack_affine(points: &[AffinePoint]) -> (Vec<PointXY>, Vec<u8>) {
        let mut xy = vec![[0u8; 64]; points.len()];
        let mut inf = vec![0u8; points.len()];
        for (i, p) in points.iter().enumerate() {
            if bool::from(p.is_identity()) {
                inf[i] = 1;
            } else {
                xy[i][..32].copy_from_slice(&p.x());
                xy[i][32..].copy_from_slice(&p.y());
            }
        }
        (xy, inf)
    }

    fn unpack_affine(xy: &PointXY, is_identity: bool) -> AffinePoint {
        if is_identity {
            return AffinePoint::IDENTITY;
        }
        // outputs are canonical and on the curve by construction; from_coordinates re-validates (affine.rs:134-147)
        AffinePoint::from_coordinates(FieldBytes::from_slice(&xy[..32]), FieldBytes::from_slice(&xy[32..])).unwrap()
    }

    /// `LinearCombination<[(ProjectivePoint, Scalar)]>::lincomb` on the GPU (k256/src/arithmetic/mul.rs:85-109).
    pub fn lincomb(eng: &mut GpuEngine, pairs: &[(ProjectivePoint, Scalar)]) -> Result<ProjectivePoint, GpuError> {
        let proj: Vec<ProjectivePoint> = pairs.iter().map(|(p, _)| *p).collect();
        let affine: Vec<AffinePoint> = ProjectivePoint::batch_normalize(proj.as_slice());
        let (xy, inf) = pack_affine(&affine);
        let k: Vec<Bytes32> = pairs.iter().map(|(_, s)| s.to_bytes().into()).collect();
        let (out, is_identity) = eng.lincomb(&k, &xy, &inf)?;
        Ok(unpack_affine(&out, is_identity).into())
    }

    /// The batch of independent multiplications the reference has no API for: `out[i] = points[i] * scalars[i]`.
    pub fn batch_mul(eng: &mut GpuEngine, pairs: &[(AffinePoint, Scalar)]) -> Result<Vec<AffinePoint>, GpuError> {
        let pts: Vec<AffinePoint> = pairs.iter().map(|(p, _)| *p).collect();
        let (xy, inf) = pack_affine(&pts);
        let k: Vec<Bytes32> = pairs.iter().map(|(_, s)| s.to_bytes().into()).collect();
        let (oxy, oinf) = eng.mul_batch(&k, &xy, &inf)?;
        Ok(oxy.iter().zip(oinf).map(|(p, f)| unpack_affine(p, f != 0)).collect())
    }
}
