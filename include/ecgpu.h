/* ecgpu.h — C ABI of libecgpu.so: B200-native batched elliptic-curve scalar multiplication
 * (secp256k1 / NIST P-256).
 *
 * The reference (RustCrypto/elliptic-curves @ 739304e) has NO FFI boundary; its seams are Rust traits.
 * Each entry point below names the trait method(s) / function(s) it stands in for (paths relative to the
 * reference checkout).  INTEGRATION.md shows the `extern "C"` block and the trait-shaped Rust wrappers a
 * maintainer would add on the reference side.
 *
 * Conventions (mirroring the reference's: infallible arithmetic, fallible decoding):
 *  - scalars   : 32-byte big-endian, must be < n      (Scalar::from_repr, k256/src/arithmetic/scalar.rs:310-316,
 *                                                      p256/src/arithmetic/scalar.rs:306-312) else ECG_ESCALAR_RANGE
 *  - points    : 64 bytes x||y, each 32-byte big-endian < p and on the curve
 *                (AffinePoint::from_coordinates, k256/src/arithmetic/affine.rs:134-147) else ECG_ENOT_ON_CURVE;
 *                identity = flag byte 1 (coordinates ignored on input, written as 64 zero bytes on output:
 *                AffinePoint::IDENTITY, k256/src/arithmetic/affine.rs:53-57)
 *  - field elts: 32-byte big-endian canonical (< p)   (FieldElement::to_bytes, k256/src/arithmetic/field.rs:110-112)
 *  - caller owns every buffer; the library reads/writes them only during the call; no exceptions cross.
 *  - a ctx is not safe for concurrent calls; distinct ctxs are independent.
 *  - there is NO CPU fallback: without a CUDA device every compute entry fails with ECG_ECUDA.
 */
#ifndef ECGPU_H
#define ECGPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct ecg_ctx ecg_ctx;

typedef enum {
  ECG_OK = 0,
  ECG_EINVAL = 1,        /* bad argument (null pointer, unknown curve/op, unsupported flag combination) */
  ECG_ESCALAR_RANGE = 2, /* some scalar >= n */
  ECG_ENOT_ON_CURVE = 3, /* some point coordinate >= p or point not on the curve */
  ECG_ECUDA = 4,         /* CUDA runtime error (see ecg_last_error) */
  ECG_ENCCL = 5,         /* reserved: collective error (the library itself issues no collectives) */
  ECG_ENOMEM = 6
} ecg_status;

/* Curves.  The hot path (SURVEY 8(a)-(e)) is secp256k1 and P-256; the other ids are the widening row "more curves
 * through the same templates" (SURVEY 8(f) rank 4): every prime-order Weierstrass curve the reference implements
 * (p384/src/arithmetic.rs:43-75, sm2/src/arithmetic.rs:44-67, bp256/src/{r1,t1}/arithmetic.rs:34-53,
 * bp384/src/{r1,t1}/arithmetic.rs:34-53, bignp256/src/arithmetic.rs:38-57, p224/src/arithmetic.rs:40-56,
 * p192/src/arithmetic.rs:38-54, p521/src/arithmetic.rs:45-90), a = -3 and general-a alike (primeorder/src/point_arithmetic.rs:54-208, :212-319).
 * Record sizes follow the curve: a scalar / field element is FB = 32 bytes for the 256-bit curves, 48 for P-384 and
 * brainpoolP384, 28 for P-224, 24 for P-192, 66 for P-521 — read "32 / 64 / 96" in every size below as "FB / 2 FB / 3 FB".
 * Byte order is the one the reference uses for the curve: big-endian everywhere except bign-curve256v1, whose field
 * elements and scalars are little-endian (bignp256/src/arithmetic/field.rs:65, bignp256/src/lib.rs:102).
 * Every curve is served by the hot-path entries (mul_batch[_x], mul_gen_batch, lincomb[_partial], point_sum,
 * batch_normalize[_hom], field_op_batch) and by mul_gen_add_batch; ecdsa_verify_batch serves every curve the reference
 * defines ECDSA for (all but sm2 and bign-curve256v1, whose signature schemes differ); hash to curve the four curves with
 * an RFC 9380 suite in the reference; SEC1 decompression every curve (one exponentiation by (p + 1) / 4 where p = 3 mod 4,
 * Tonelli-Shanks for P-224); the field square root every curve but P-224 (where the reference's root is the one its
 * external bignum crate's Tonelli-Shanks happens to return); BIP340 is secp256k1's alone, SM2DSA and SM2 public-key
 * encryption sm2's.  What a curve does not serve answers ECG_EINVAL. */
typedef enum {
  ECG_SECP256K1 = 0,
  ECG_NISTP256 = 1,
  ECG_NISTP384 = 2,
  ECG_SM2 = 3,
  ECG_BP256R1 = 4,   /* brainpoolP256r1: general a */
  ECG_BP256T1 = 5,   /* brainpoolP256t1: a = -3 */
  ECG_BIGNP256 = 6,  /* bign-curve256v1 (STB 34.101.45): little-endian records */
  ECG_BP384R1 = 7,   /* brainpoolP384r1: general a */
  ECG_BP384T1 = 8,   /* brainpoolP384t1: a = -3 */
  ECG_NISTP224 = 9,
  ECG_NISTP192 = 10,
  ECG_NISTP521 = 11  /* 66-byte records (FieldBytesSize = U66, p521/src/lib.rs:63-64) */
} ecg_curve;

typedef enum {
  ECG_FOP_ADD = 0,
  ECG_FOP_SUB = 1,
  ECG_FOP_NEG = 2, /* b ignored */
  ECG_FOP_MUL = 3,
  ECG_FOP_SQR = 4, /* b ignored */
  ECG_FOP_INV = 5  /* b ignored; inv(0) = 0 */
} ecg_field_op;

/* ctx flags */
#define ECG_FLAG_DEVICE_PTRS 1u /* every data pointer is a device pointer on device_ids[0] (n_devices must be 1);
                                   32/64/96-byte record arrays must be 4-byte aligned (ECG_EINVAL otherwise) */

#define ECG_FLAG_ZEROIZE 2u     /* before a call returns, overwrite the library's device-side copies of its inputs and
                                   every intermediate derived from them (staged scalars and points, window tables,
                                   Jacobian results, batch-inversion scratch, bucket arenas) with zeros — for callers
                                   that pass secret scalars (the reference zeroizes secrets on drop); costs one
                                   memset per buffer and call */

#define ECG_FLAG_CONSTTIME 4u   /* scalar-independent execution for the entries that take secret scalars — ecg_mul_batch[_x],
                                   ecg_mul_gen_batch, ecg_lincomb[_partial], the scalar multiplications of
                                   ecg_sm2pke_{encrypt,decrypt}_batch — the analogue of the reference's constant-time
                                   `Mul` / `lincomb` (k256/src/arithmetic/mul.rs:112-163, LookupTable::select
                                   primeorder/src/tables/lookup.rs:43-65): window-table entries are fetched by a masked scan
                                   over all entries, the GLV sign folding is branch-free, k*G runs through the variable-base
                                   routine (no table indexed by 16 scalar bits, like mul_backend::VariableOnly), lincomb
                                   always takes the per-term path (the bucket method's access pattern is the scalars).
                                   Left data-dependent: the exceptional-case branches of the Jacobian formulas, reachable
                                   only for k = 0 (not a NonZeroScalar) and a negligible set of scalars; kernel timing also
                                   depends on inputs being rejected.  The default (flag clear) is the vartime analogue. */

/* Create a context on the given CUDA devices (NULL/0 = device 0).  With several devices a host-pointer
 * batch is split into contiguous index ranges, one per device (SURVEY.md §8(e)); there is no
 * inter-device traffic.  Replaces nothing in the reference (it has no runtime state except the lazily
 * built generator table, primeorder/src/tables/basepoint.rs:29-31; here too the fixed-base table is built on
 * first use, on the device, ~30 ms and 32 MiB per curve and device). */
ecg_status ecg_ctx_create(const int* device_ids, int n_devices, unsigned flags, ecg_ctx** out);
void ecg_ctx_destroy(ecg_ctx* ctx);
const char* ecg_last_error(const ecg_ctx* ctx);
/* index of the first offending element of the last failed call with ECG_ESCALAR_RANGE / ECG_ENOT_ON_CURVE */
size_t ecg_last_error_index(const ecg_ctx* ctx);

/* Run this ctx's work on a caller-provided cudaStream_t (e.g. PyTorch's current stream) instead of the
 * ctx-owned stream; device 0 of the ctx only.  NULL restores the owned stream (which is non-blocking: it does NOT
 * synchronise with the legacy default stream) — to run on the legacy default stream itself pass cudaStreamLegacy. */
ecg_status ecg_ctx_set_stream(ecg_ctx* ctx, void* cuda_stream);

/* out[i] = k[i] * P[i].
 * Replaces `ProjectivePoint * Scalar` / `mul_vartime` for a batch of independent pairs:
 *   k256/src/arithmetic/mul.rs:236-295 (Mul, MulVartime impls), primeorder/src/projective.rs:133-144, :847-858
 * followed by to_affine (k256/src/arithmetic/projective.rs:64-75).
 * k: n*32, P_xy: n*64, P_inf: n bytes or NULL (no identities), out_xy: n*64, out_inf: n bytes. */
ecg_status ecg_mul_batch(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* k, const uint8_t* P_xy,
                         const uint8_t* P_inf, uint8_t* out_xy, uint8_t* out_inf);

/* out[i] = k[i] * G.
 * Replaces ProjectivePoint::mul_by_generator[_vartime] (k256/src/arithmetic/mul.rs:180-232),
 * BasepointTable::mul (primeorder/src/tables/basepoint.rs:82-125), MulBackend::mul_by_generator
 * (primeorder/src/mul_backend.rs:11-29). */
ecg_status ecg_mul_gen_batch(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* k, uint8_t* out_xy,
                             uint8_t* out_inf);

/* out = sum_i k[i] * P[i]   (one point).
 * Replaces LinearCombination::lincomb / lincomb_vartime (k256/src/arithmetic/mul.rs:66-175,
 * primeorder/src/projective.rs:480-557). */
ecg_status ecg_lincomb(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* k, const uint8_t* P_xy,
                       const uint8_t* P_inf, uint8_t out_xy[64], uint8_t* out_inf);

/* Same sum, but the result is left un-normalised as X||Y||Z (3*32 bytes big-endian, Jacobian:
 * x = X/Z^2, y = Y/Z^3, Z = 0 for the identity) so that partial sums from several ranks can be combined
 * with ecg_point_sum after one small gather (SURVEY.md §8(e), config 5). */
ecg_status ecg_lincomb_partial(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* k, const uint8_t* P_xy,
                               const uint8_t* P_inf, uint8_t out_xyz[96]);

/* out = sum of m Jacobian points given as m*96 bytes (X||Y||Z), normalised to affine (m is the number of ranks).
 * Pointers follow the ctx flags like every other entry: with ECG_FLAG_DEVICE_PTRS the points are read straight from
 * device memory (e.g. the receive buffer of the all_gather that is config 5's one exchange step) and the 64 + 1 result
 * bytes are written to device memory: import -> sum -> normalise, no host staging. */
ecg_status ecg_point_sum(ecg_ctx* ctx, ecg_curve curve, size_t m, const uint8_t* xyz, uint8_t out_xy[64],
                         uint8_t* out_inf);

/* out[i] = a[i] * G + b[i] * P[i].
 * Replaces MulByGeneratorVartime::mul_by_generator_and_mul_add_vartime (k256/src/arithmetic/mul.rs:303-310,
 * primeorder/src/mul_backend.rs:31-40) — the ECDSA / BIP340 verification shape. */
ecg_status ecg_mul_gen_add_batch(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* a, const uint8_t* b,
                                 const uint8_t* P_xy, const uint8_t* P_inf, uint8_t* out_xy, uint8_t* out_inf);

/* ---- first widening step (SURVEY.md section 8(f), rank 1): batched signature verification ------------------
 * Invalid encodings (r, s, public key out of range / off curve) are NOT API errors: valid[i] = 0, like the
 * reference's per-signature Err(Error). */

/* BIP340 Schnorr verification, secp256k1: valid[i] = 1 iff sig[i] (r || s, 64 bytes) is a valid signature of the
 * 32-byte message msg32[i] under the x-only public key pk_x[i].
 * Replaces VerifyingKey::verify_raw over a batch (k256/src/schnorr/verifying.rs:76-99), including
 * VerifyingKey::from_bytes (lift_x, :36-52) and the tagged challenge hash (k256/src/schnorr.rs:85,221-227). */
ecg_status ecg_schnorr_verify_batch(ecg_ctx* ctx, size_t n, const uint8_t* pk_x, const uint8_t* msg32,
                                    const uint8_t* sig64, uint8_t* valid);

/* ECDSA verification: z32[i] = the prehash after bits2field, one FB-byte big-endian record (reduced mod n inside),
 * sig64[i] = r || s (2 FB bytes, Signature::try_from encoding), Q_xy[i] = public key x || y (2 FB).  low_s_only != 0
 * additionally rejects s > n/2 (EcdsaCurve::NORMALIZE_S: true for k256 only, k256/src/ecdsa.rs:104-106).  Replaces
 * ecdsa_core::VerifyingKey::verify_prehash over a batch for every curve the reference gives an EcdsaCurve impl:
 * k256/src/ecdsa.rs:93-121, p256/src/ecdsa.rs, p192 / p224 / p384 / p521 src/ecdsa.rs, bp256/src/{r1,t1}/ecdsa.rs,
 * bp384/src/{r1,t1}/ecdsa.rs (ECG_SM2, ECG_BIGNP256: ECG_EINVAL — SM2DSA and the bign scheme are not ECDSA). */
ecg_status ecg_ecdsa_verify_batch(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* z32, const uint8_t* sig64,
                                  const uint8_t* Q_xy, int low_s_only, uint8_t* valid);

/* Public-key recovery over a batch (secp256k1 — the Ethereum ecrecover shape — and P-256): z32 = the prehash, sig64 = r || s,
 * recid = one byte per signature (RecoveryId::to_byte: bit 0 = y of R is odd, bit 1 = x of R was reduced, i.e. x = r + n).
 * R = decompress(x, y parity); Q = u1*G + u2*R with u1 = -z r^-1, u2 = s r^-1 (mod n).  valid[i] = 1 and out_xy = Q.x || Q.y
 * when 0 < r, s < n, recid < 4, x < p has a point and Q != O (then the closing verify_prehash of the reference holds by
 * construction; low_s_only = EcdsaCurve::NORMALIZE_S refuses s > n/2 as that verification does on secp256k1); otherwise
 * valid[i] = 0 and 64 zero bytes.  Replaces ecdsa_core::VerifyingKey::recover_from_prehash / recover_from_digest as k256 and
 * p256 re-export it (k256/src/ecdsa.rs:45-88; vectors :182-262). */
ecg_status ecg_ecdsa_recover_batch(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* z32, const uint8_t* sig64,
                                   const uint8_t* recid, int low_s_only, uint8_t* out_xy, uint8_t* valid);

/* SM2DSA verify_prehash over a batch (curve sm2 only, so no curve argument): e32 = the 32-byte digest e = SM3(Z_A || M)
 * the caller computed (Z_A = the identity hash of sm2/src/distid.rs:21-47), sig64 = r || s, Q_xy = the public key.
 * valid[i] = 1 iff r, s in [1, n-1], t = r + s mod n != 0, Q on the curve and (e + x(s*G + t*Q)) mod n == r.
 * Replaces sm2::dsa::VerifyingKey::verify_prehash (sm2/src/dsa/verifying.rs:138-175).  The bign signature scheme
 * (bignp256/src/ecdsa/verifying.rs:92-150) hashes the x coordinate with belt-hash between the group step and the
 * verdict; its group step R = (s1 + H)*G + (s0 + 2^128)*Q is ecg_mul_gen_add_batch on ECG_BIGNP256. */
ecg_status ecg_sm2dsa_verify_batch(ecg_ctx* ctx, size_t n, const uint8_t* e32, const uint8_t* sig64, const uint8_t* Q_xy,
                                   uint8_t* valid);

/* SM2 public-key encryption (GB/T 32918.4; curve sm2 only, so no curve argument), digest SM3.  Records are variable-length
 * and packed as for hash to curve: record i = data[offsets[i] .. offsets[i+1]), n + 1 non-decreasing uint64 offsets.  With
 * ECG_FLAG_DEVICE_PTRS every data pointer is a device pointer (offsets and pt_len 8-byte aligned, k32 / d32 / Pb_xy
 * 4-byte aligned) and the offsets are not checked on the host.  Both entries run on the ctx's first device.  A bad
 * ciphertext, key or nonce is a per-record verdict, not an API error; ECG_EINVAL means a null pointer, decreasing
 * offsets, an unknown mode or a misaligned device pointer.  mode 0 = C1C3C2 (the reference's default), 1 = C1C2C3.
 *
 * C_i = SM2-Enc(Pb_i, M_i; k_i).  k32: n*32 ephemeral scalars (the caller's randomness; the reference draws k inside,
 * sm2/src/pke/encrypting.rs:186-188), Pb_xy: n*64 recipient keys.  compressed != 0: C1 = 02|03 || x (what
 * EncryptingKey::encrypt emits, encrypting.rs:90), else 04 || x || y (OpenSSL / GM/T 0003 interoperability).
 * Record i is written at out + (offsets[i] - offsets[0]) + i*ovh, ovh = 32 + (compressed ? 33 : 65), length len_i + ovh,
 * laid out as Cipher::to_slice (sm2/src/pke.rs:181-213).  status[i]: 1 = ok; 0 = refused (k not in [1, n-1], Pb not
 * on the curve, empty message), record zeroed; 2 = the KDF output was all zero, draw another k (the reference's retry
 * loop, encrypting.rs:184-209), record zeroed.  Replaces EncryptingKey::encrypt / encrypt_digest::<_, Sm3>
 * (encrypting.rs:166-230). */
ecg_status ecg_sm2pke_encrypt_batch(ecg_ctx* ctx, size_t n, const uint8_t* msgs, const uint64_t* offsets, const uint8_t* k32,
                                    const uint8_t* Pb_xy, int mode, int compressed, uint8_t* out, uint8_t* status);

/* M_i = SM2-Dec(d_i, C_i).  Ciphertext i = cts[offsets[i] .. offsets[i+1]), C1 in any SEC1 form the reference accepts
 * (02 / 03 compressed, 04 uncompressed, 05 compact; Cipher::from_slice, sm2/src/pke.rs:122-160).  d32: n*32 secret
 * scalars, valid only in [1, n-1].  out has the size of cts: plaintext i at out + (offsets[i] - offsets[0]), pt_len[i]
 * bytes; every other byte of record i's range is written as zero, as is the whole range when valid[i] = 0.  valid[i] = 1
 * iff the record parses, d is in range and SM3(x2 || M' || y2) equals C3 (compared without an early exit).  Replaces
 * DecryptingKey::decrypt / decrypt_digest::<Sm3> (sm2/src/pke/decrypting.rs:174-222). */
ecg_status ecg_sm2pke_decrypt_batch(ecg_ctx* ctx, size_t n, const uint8_t* cts, const uint64_t* offsets, const uint8_t* d32,
                                    int mode, uint8_t* out, uint64_t* pt_len, uint8_t* valid);

/* SEC1 compressed point decoding (rank 2 of SURVEY 8(f)): records of 1 + FB bytes (02|03 || x; all zero bytes = the
 * identity; 33 bytes for the 256-bit curves, 49 for the 384-bit ones, 29 for P-224, 25 for P-192, 67 for P-521).
 * valid[i] = 0 when the tag is unknown, x >= p, or x^3 + ax + b has no square root; out_xy / out_inf as in ecg_mul_batch.  Replaces AffinePoint::decompress / from_sec1_point over a batch
 * (primeorder/src/affine.rs:179-198, :212-232; k256/src/arithmetic/affine.rs DecompressPoint; sqrt:
 * k256/src/arithmetic/field.rs:200-235, p256/src/arithmetic/field.rs:121-147, p521/src/arithmetic/field.rs:386; the
 * primefield-generated fields of p384 / sm2 / brainpool / p192, primefield/src/monty.rs:467, through the same
 * (p + 1) / 4 exponent; P-224, p = 1 mod 4, through Tonelli-Shanks — decompress selects the root by the tag's parity, so
 * the result does not depend on which root the square root finds).  The x bytes are the curve's FieldBytes, i.e.
 * little-endian for bign-curve256v1, as from_repr reads them inside decompress. */
ecg_status ecg_decompress_batch(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* sec1_33, uint8_t* out_xy,
                                uint8_t* out_inf, uint8_t* valid);

/* Projective (Jacobian X||Y||Z, n*96 bytes) -> affine, one shared inversion per thread-group
 * (Montgomery's trick).  Replaces BatchNormalize::batch_normalize (k256/src/arithmetic/projective.rs:345-391,
 * primeorder/src/projective.rs:435-478).  Coordinates must be < p. */
ecg_status ecg_batch_normalize(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* xyz, uint8_t* out_xy,
                               uint8_t* out_inf);

/* Same for the reference's OWN projective form: homogeneous (X:Y:Z) with x = X/Z, y = Y/Z and identity (0:1:0)
 * (k256/src/arithmetic/projective.rs:49-53, to_affine :64-75, batch_normalize :367-391; primeorder/src/projective.rs
 * :435-478), so a reference-side caller passes ProjectivePoint coordinates unchanged. */
ecg_status ecg_batch_normalize_hom(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* xyz, uint8_t* out_xy,
                                   uint8_t* out_inf);

/* out_x[i] = x coordinate of k[i] * P[i] (n*32 bytes; 32 zero bytes + flag for the identity): the ECDH shape,
 * SharedSecret = (public * secret).to_affine().x (k256/src/ecdh.rs:46-60, elliptic-curve's diffie_hellman).  The y
 * coordinate is never formed (2 of the 7 normalisation multiplications, 32 of the 65 result bytes per point). */
ecg_status ecg_mul_batch_x(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* k, const uint8_t* P_xy,
                           const uint8_t* P_inf, uint8_t* out_x, uint8_t* out_inf);

/* out[i] = sqrt(a[i]) as the reference returns it, a^((p+1)/4), with is_square[i] = 1; FB zero bytes and
 * is_square[i] = 0 when a[i] is not a square (CtOption::none).  Replaces FieldElement::sqrt
 * (k256/src/arithmetic/field.rs:200-235, p256/src/arithmetic/field.rs:121-147; every curve with p = 3 (mod 4);
 * ECG_NISTP224: ECG_EINVAL). */
ecg_status ecg_field_sqrt_batch(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* a, uint8_t* out,
                                uint8_t* is_square);

/* ---- hash to curve (SURVEY.md section 8(f) rank 4: "hash-to-curve front end"), RFC 9380 with expand_message_xmd: the
 * four Weierstrass suites the reference implements — secp256k1_XMD:SHA-256_SSWU_{RO,NU}_ (k256/src/arithmetic/
 * hash2curve.rs:14-20), P256_XMD:SHA-256_SSWU_{RO,NU}_ (p256/.../hash2curve.rs:13-19), P384_XMD:SHA-384_SSWU_{RO,NU}_
 * (p384/.../hash2curve.rs:13-19), P521_XMD:SHA-512_SSWU_{RO,NU}_ (p521/.../hash2curve.rs:13-19); other curves: ECG_EINVAL.
 * Outputs are the curve's records (2 FB bytes per point, FB per scalar).
 * Message i is msgs[offsets[i] .. offsets[i+1]) (offsets: n + 1 non-decreasing uint64 values; with ECG_FLAG_DEVICE_PTRS
 * msgs, offsets and the outputs are device pointers, offsets 8-byte aligned).  dst / dst_len: the domain separation tag,
 * always a host pointer; empty -> ECG_EINVAL (ExpandMsgXmdError::EmptyDst, hash2curve/src/hash2field/expand_msg.rs:101-106),
 * longer than 255 bytes -> replaced by H("H2C-OVERSIZE-DST-" || dst), H the suite's hash, as in the reference (expand_msg.rs:107-121).
 * nonuniform = 0: out[i] = hash_to_curve(msg_i) (GroupDigest::hash_from_bytes, hash2curve/src/group_digest.rs:88-97:
 * two field elements, two maps, one addition); nonuniform != 0: encode_to_curve (encode_from_bytes, :110-118). */
ecg_status ecg_hash_to_curve_batch(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* msgs, const uint64_t* offsets,
                                   const uint8_t* dst, size_t dst_len, int nonuniform, uint8_t* out_xy, uint8_t* out_inf);

/* out[i] = hash_to_scalar(msg_i) as one FB-byte big-endian record: hash_to_field with the group order as modulus and the suite's L (48 / 72 / 98)
 * (hash2curve/src/group_digest.rs:131-143 with Reduce<Array<u8, U48>> for Scalar, k256/src/arithmetic/hash2curve.rs:151-166,
 * p256/src/arithmetic/hash2curve.rs:77-94) — the VOPRF DeriveKeyPair / HashToScalar primitive. */
ecg_status ecg_hash_to_scalar_batch(ecg_ctx* ctx, ecg_curve curve, size_t n, const uint8_t* msgs, const uint64_t* offsets,
                                    const uint8_t* dst, size_t dst_len, uint8_t* out);

/* out[i] = a[i] op b[i] in F_p.
 * Replaces FieldElement add/sub/neg/mul/square/invert: k256/src/arithmetic/field.rs:116-196 over
 * field_5x52.rs:203-414; p256/src/arithmetic/field.rs:67-118 over field64.rs:7-144. */
ecg_status ecg_field_op_batch(ecg_ctx* ctx, ecg_curve curve, int op, size_t n, const uint8_t* a,
                              const uint8_t* b, uint8_t* out);

/* ---- measurement helpers (not part of the reference-facing surface) ---- */

/* Integer-pipe microbenchmark on device 0 of the ctx: which = 0 IMAD.WIDE.U32.X carry chains (the
 * field-multiplier's instruction), 1 = IMAD (32-bit lo), 2 = IADD3 carry chains, 3 = fused field-mul
 * throughput (secp256k1), 4 = same for P-256.  Returns operations per second (thread-level instructions
 * of the named kind, or field multiplications for 3/4). */
ecg_status ecg_microbench(ecg_ctx* ctx, int which, int iters, double* ops_per_s, double* elapsed_ms);

/* When enabled, every call brackets its dominant kernel (variable-base / fixed-base scalar multiplication)
 * with CUDA events on the launching stream; ecg_timing_read returns the accumulated device milliseconds
 * (max over the ctx's devices per call) and the number of calls since ecg_timing_enable. */
ecg_status ecg_timing_enable(ecg_ctx* ctx, int on);
ecg_status ecg_timing_read(const ecg_ctx* ctx, double* dominant_kernel_ms_sum, uint64_t* calls);

/* number of CUDA kernels this ctx has launched since creation */
uint64_t ecg_kernel_launches(const ecg_ctx* ctx);

const char* ecg_version(void);

#ifdef __cplusplus
}
#endif
#endif /* ECGPU_H */
