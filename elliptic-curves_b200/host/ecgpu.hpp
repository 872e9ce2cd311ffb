// ecgpu.hpp — C++ host-side mirror of the reference's operator surface for the scalar-multiplication path,
// header-only, over the C ABI in include/ecgpu.h.  (The reference is Rust; this image has no Rust toolchain, so the
// host layer above the ABI is C++; INTEGRATION.md shows the equivalent Rust shim.)
//
// Names follow the reference's traits so that call sites read the same:
//   Engine::mul(points, scalars)                      <->  ProjectivePoint * Scalar            (k256/src/arithmetic/mul.rs:249-274)
//   Engine::mul_vartime(...)                          <->  MulVartime::mul_vartime             (mul.rs:276-295)   [same kernel]
//   Engine::mul_by_generator(scalars)                 <->  ProjectivePoint::mul_by_generator   (mul.rs:180-232)
//   Engine::lincomb(points, scalars)                  <->  LinearCombination::lincomb          (mul.rs:66-109)
//   Engine::mul_by_generator_and_mul_add_vartime(...) <->  MulByGeneratorVartime::...          (mul.rs:303-310)
//   Engine::batch_normalize(jacobian)                 <->  BatchNormalize::batch_normalize     (projective.rs:345-365)
//   Engine::hash_to_curve / encode_to_curve / hash_to_scalar <-> GroupDigest::hash_from_bytes / encode_from_bytes,
//                                                         hash2curve::hash_to_scalar (hash2curve/src/group_digest.rs:88-143)
//   Engine::sm2pke_encrypt / sm2pke_decrypt          <->  sm2::pke::EncryptingKey::encrypt / DecryptingKey::decrypt
// The typed surface below is for the 256-bit curves with big-endian records (secp256k1, P-256, sm2, brainpoolP256r1/t1);
// the other curves of include/ecgpu.h (48 / 28 / 24-byte records, bign's little-endian records) are reached through the
// C ABI directly or the Python mirror, which sizes its buffers per curve.
// Fallible decoding mirrors CtOption/Result: out-of-range scalars / off-curve points throw DecodeError carrying the
// index of the first offender; arithmetic itself is total.
#pragma once
#include <algorithm>
#include <array>
#include <cstdint>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/ecgpu.h"

namespace ecgpu {

using Scalar = std::array<uint8_t, 32>;  // big-endian, < n          (Scalar::to_bytes)
struct AffinePoint {                     // AffinePoint { x, y, infinity } (k256/src/arithmetic/affine.rs:37-49)
  std::array<uint8_t, 32> x{}, y{};
  uint8_t infinity = 0;
  static AffinePoint identity() {
    AffinePoint p;
    p.infinity = 1;
    return p;
  }
};
struct JacobianPoint {  // X, Y, Z big-endian; x = X/Z^2, y = Y/Z^3; Z = 0 is the identity
  std::array<uint8_t, 32> X{}, Y{}, Z{};
};
struct ProjectivePoint {  // the reference's own form: homogeneous, x = X/Z, y = Y/Z, identity (0:1:0)
  std::array<uint8_t, 32> X{}, Y{}, Z{};  // (k256/src/arithmetic/projective.rs:49-53)
};

struct Error : std::runtime_error {
  ecg_status code;
  Error(ecg_status c, const std::string& m) : std::runtime_error(m), code(c) {}
};
struct DecodeError : Error {  // Scalar::from_repr / AffinePoint::from_coordinates returned None in the reference
  size_t index;
  DecodeError(ecg_status c, const std::string& m, size_t i) : Error(c, m), index(i) {}
};

class Engine {
 public:
  // zeroize: clear the device-side copies of scalars, window tables and intermediates after every call
  // (ECG_FLAG_ZEROIZE; the reference zeroizes secrets on drop)
  // consttime: ECG_FLAG_CONSTTIME — scalar-independent table selects and sign folding, k*G through the variable-base
  // routine, per-term lincomb (the analogue of the reference's constant-time Mul; costs measured in bench.py configs.8)
  explicit Engine(ecg_curve curve, const std::vector<int>& devices = {0}, bool zeroize = false, bool consttime = false) : curve_(curve) {
    ecg_status st = ecg_ctx_create(devices.data(), (int)devices.size(), (zeroize ? ECG_FLAG_ZEROIZE : 0u) | (consttime ? ECG_FLAG_CONSTTIME : 0u), &ctx_);
    if (st != ECG_OK) throw Error(st, "ecg_ctx_create failed (no CUDA device? there is no CPU fallback)");
  }
  ~Engine() { ecg_ctx_destroy(ctx_); }
  Engine(const Engine&) = delete;
  Engine& operator=(const Engine&) = delete;

  std::vector<AffinePoint> mul(const std::vector<AffinePoint>& points, const std::vector<Scalar>& scalars) {
    size_t n = check_sizes(points.size(), scalars.size());
    pack(points);
    std::vector<uint8_t> out(64 * n), oinf(n);
    check(ecg_mul_batch(ctx_, curve_, n, flat(scalars), xy_.data(), inf_.data(), out.data(), oinf.data()));
    return unpack(out, oinf);
  }
  std::vector<AffinePoint> mul_vartime(const std::vector<AffinePoint>& p, const std::vector<Scalar>& k) { return mul(p, k); }

  std::vector<AffinePoint> mul_by_generator(const std::vector<Scalar>& scalars) {
    size_t n = scalars.size();
    std::vector<uint8_t> out(64 * n), oinf(n);
    check(ecg_mul_gen_batch(ctx_, curve_, n, flat(scalars), out.data(), oinf.data()));
    return unpack(out, oinf);
  }
  std::vector<AffinePoint> mul_by_generator_vartime(const std::vector<Scalar>& k) { return mul_by_generator(k); }

  AffinePoint lincomb(const std::vector<AffinePoint>& points, const std::vector<Scalar>& scalars) {
    size_t n = check_sizes(points.size(), scalars.size());
    pack(points);
    std::vector<uint8_t> out(64), oinf(1);
    check(ecg_lincomb(ctx_, curve_, n, flat(scalars), xy_.data(), inf_.data(), out.data(), oinf.data()));
    return unpack(out, oinf)[0];
  }
  AffinePoint lincomb_vartime(const std::vector<AffinePoint>& p, const std::vector<Scalar>& k) { return lincomb(p, k); }

  // a[i]*G + b[i]*P[i]
  std::vector<AffinePoint> mul_by_generator_and_mul_add_vartime(const std::vector<Scalar>& a, const std::vector<Scalar>& b,
                                                                const std::vector<AffinePoint>& points) {
    size_t n = check_sizes(points.size(), a.size());
    check_sizes(n, b.size());
    pack(points);
    std::vector<uint8_t> out(64 * n), oinf(n);
    check(ecg_mul_gen_add_batch(ctx_, curve_, n, flat(a), flat(b), xy_.data(), inf_.data(), out.data(), oinf.data()));
    return unpack(out, oinf);
  }

  std::vector<AffinePoint> batch_normalize(const std::vector<JacobianPoint>& pts) {
    size_t n = pts.size();
    std::vector<uint8_t> out(64 * n), oinf(n);
    check(ecg_batch_normalize(ctx_, curve_, n, reinterpret_cast<const uint8_t*>(pts.data()), out.data(), oinf.data()));
    return unpack(out, oinf);
  }

  // BatchNormalize::batch_normalize on the reference's homogeneous coordinates (projective.rs:367-391)
  std::vector<AffinePoint> batch_normalize(const std::vector<ProjectivePoint>& pts) {
    size_t n = pts.size();
    std::vector<uint8_t> out(64 * n), oinf(n);
    check(ecg_batch_normalize_hom(ctx_, curve_, n, reinterpret_cast<const uint8_t*>(pts.data()), out.data(), oinf.data()));
    return unpack(out, oinf);
  }
  // FieldElement::sqrt over a batch; ok[i] = false (and a zero root) where the input is not a square
  std::vector<std::array<uint8_t, 32>> field_sqrt(const std::vector<std::array<uint8_t, 32>>& a, std::vector<bool>* ok = nullptr) {
    size_t n = a.size();
    std::vector<std::array<uint8_t, 32>> r(n);
    std::vector<uint8_t> sq(n);
    check(ecg_field_sqrt_batch(ctx_, curve_, n, reinterpret_cast<const uint8_t*>(a.data()), reinterpret_cast<uint8_t*>(r.data()), sq.data()));
    if (ok) ok->assign(sq.begin(), sq.end());
    return r;
  }

  // ---- widening (SURVEY 8(f)): verification, wire format, key agreement ----
  using Bytes32 = std::array<uint8_t, 32>;
  using Sig64 = std::array<uint8_t, 64>;
  using Sec1Compressed = std::array<uint8_t, 33>;

  // schnorr::VerifyingKey::verify_raw over a batch (k256/src/schnorr/verifying.rs:76-99); secp256k1 only
  std::vector<bool> schnorr_verify(const std::vector<Bytes32>& pk_x, const std::vector<Bytes32>& msg, const std::vector<Sig64>& sig) {
    size_t n = check_sizes(pk_x.size(), msg.size());
    check_sizes(n, sig.size());
    std::vector<uint8_t> valid(n);
    check(ecg_schnorr_verify_batch(ctx_, n, reinterpret_cast<const uint8_t*>(pk_x.data()), reinterpret_cast<const uint8_t*>(msg.data()),
                                   reinterpret_cast<const uint8_t*>(sig.data()), valid.data()));
    return std::vector<bool>(valid.begin(), valid.end());
  }
  // ecdsa::VerifyingKey::verify_prehash over a batch (k256/src/ecdsa.rs:93-121); low_s_only = EcdsaCurve::NORMALIZE_S
  std::vector<bool> ecdsa_verify_prehash(const std::vector<Bytes32>& z, const std::vector<Sig64>& sig, const std::vector<AffinePoint>& q,
                                         bool low_s_only) {
    size_t n = check_sizes(z.size(), sig.size());
    check_sizes(n, q.size());
    pack(q);
    std::vector<uint8_t> valid(n);
    check(ecg_ecdsa_verify_batch(ctx_, curve_, n, reinterpret_cast<const uint8_t*>(z.data()), reinterpret_cast<const uint8_t*>(sig.data()),
                                 xy_.data(), low_s_only ? 1 : 0, valid.data()));
    return std::vector<bool>(valid.begin(), valid.end());
  }
  // ecdsa::VerifyingKey::recover_from_prehash over a batch (k256/src/ecdsa.rs:45-88): recid = RecoveryId::to_byte per signature;
  // ok[i] = false (and an all-zero point) where recovery fails
  std::vector<AffinePoint> ecdsa_recover_prehash(const std::vector<Bytes32>& z, const std::vector<Sig64>& sig, const std::vector<uint8_t>& recid,
                                                 bool low_s_only, std::vector<bool>* ok = nullptr) {
    size_t n = check_sizes(z.size(), sig.size());
    check_sizes(n, recid.size());
    std::vector<uint8_t> out(64 * n), valid(n), noinf(n, 0);
    check(ecg_ecdsa_recover_batch(ctx_, curve_, n, reinterpret_cast<const uint8_t*>(z.data()), reinterpret_cast<const uint8_t*>(sig.data()),
                                  recid.data(), low_s_only ? 1 : 0, out.data(), valid.data()));
    if (ok) ok->assign(valid.begin(), valid.end());
    return unpack(out, noinf);
  }
  // sm2::dsa::VerifyingKey::verify_prehash over a batch (sm2/src/dsa/verifying.rs:138-175): e = SM3(Z_A || M) per signature
  std::vector<bool> sm2dsa_verify_prehash(const std::vector<Bytes32>& e, const std::vector<Sig64>& sig, const std::vector<AffinePoint>& q) {
    size_t n = check_sizes(e.size(), sig.size());
    check_sizes(n, q.size());
    pack(q);
    std::vector<uint8_t> valid(n);
    check(ecg_sm2dsa_verify_batch(ctx_, n, reinterpret_cast<const uint8_t*>(e.data()), reinterpret_cast<const uint8_t*>(sig.data()), xy_.data(),
                                  valid.data()));
    return std::vector<bool>(valid.begin(), valid.end());
  }
  // AffinePoint::decompress over a batch (primeorder/src/affine.rs:179-198); ok[i] = false where x is not on the curve
  std::vector<AffinePoint> decompress(const std::vector<Sec1Compressed>& rec, std::vector<bool>* ok = nullptr) {
    size_t n = rec.size();
    std::vector<uint8_t> out(64 * n), oinf(n), valid(n);
    check(ecg_decompress_batch(ctx_, curve_, n, reinterpret_cast<const uint8_t*>(rec.data()), out.data(), oinf.data(), valid.data()));
    if (ok) ok->assign(valid.begin(), valid.end());
    return unpack(out, oinf);
  }
  // to_sec1_point(true) / GroupEncoding::to_bytes (primeorder/src/affine.rs:387-402): byte layout only, no device work
  static Sec1Compressed compress(const AffinePoint& p) {
    Sec1Compressed r{};
    if (p.infinity) return r;  // identity = 33 zero bytes
    r[0] = 2 + (p.y[31] & 1);
    std::copy(p.x.begin(), p.x.end(), r.begin() + 1);
    return r;
  }
  // diffie_hellman (k256/src/ecdh.rs:46-60): x-coordinate of secret[i] * public[i], through ecg_mul_batch_x (y is never
  // formed).  VARIABLE TIME in the secret — the kernels index window tables by scalar digits and branch on exceptional
  // cases, the reference's diffie_hellman is constant time — hence the name; construct the Engine with zeroize = true.
  // Like the reference's NonZeroScalar / PublicKey inputs, a zero scalar, an identity peer or an identity result is an
  // error, never an all-zero shared secret.
  std::vector<Bytes32> diffie_hellman_vartime(const std::vector<Scalar>& secret, const std::vector<AffinePoint>& pub) {
    size_t n = check_sizes(pub.size(), secret.size());
    for (size_t i = 0; i < n; i++) {
      if (pub[i].infinity) throw DecodeError(ECG_EINVAL, "diffie_hellman_vartime: identity public key", i);
      if (std::all_of(secret[i].begin(), secret[i].end(), [](uint8_t b) { return b == 0; }))
        throw DecodeError(ECG_EINVAL, "diffie_hellman_vartime: zero secret scalar", i);
    }
    pack(pub);
    std::vector<Bytes32> r(n);
    std::vector<uint8_t> oinf(n);
    check(ecg_mul_batch_x(ctx_, curve_, n, flat(secret), xy_.data(), nullptr, reinterpret_cast<uint8_t*>(r.data()), oinf.data()));
    for (size_t i = 0; i < n; i++)
      if (oinf[i]) throw DecodeError(ECG_EINVAL, "diffie_hellman_vartime: identity shared point", i);
    return r;
  }
  // PublicKey::from_secret_scalar over a batch, SEC1-compressed.  VARIABLE TIME in the secret (see above).
  std::vector<Sec1Compressed> derive_public_keys_vartime(const std::vector<Scalar>& secret) {
    for (size_t i = 0; i < secret.size(); i++)
      if (std::all_of(secret[i].begin(), secret[i].end(), [](uint8_t b) { return b == 0; }))
        throw DecodeError(ECG_EINVAL, "derive_public_keys_vartime: zero secret scalar", i);
    std::vector<AffinePoint> p = mul_by_generator(secret);
    std::vector<Sec1Compressed> r(p.size());
    for (size_t i = 0; i < p.size(); i++) r[i] = compress(p[i]);
    return r;
  }

  // GroupDigest::hash_from_bytes (nonuniform = false) / encode_from_bytes (true) over a batch of messages, RFC 9380 with
  // expand_message_xmd<SHA-256> (hash2curve/src/group_digest.rs:88-118; suites of k256 / p256 arithmetic/hash2curve.rs)
  std::vector<AffinePoint> hash_to_curve(const std::vector<std::string>& msgs, const std::string& dst, bool nonuniform = false) {
    size_t n = msgs.size();
    std::vector<uint64_t> offs(n + 1, 0);
    std::string all;
    for (size_t i = 0; i < n; i++) {
      all += msgs[i];
      offs[i + 1] = all.size();
    }
    std::vector<uint8_t> out(64 * n), oinf(n);
    check(ecg_hash_to_curve_batch(ctx_, curve_, n, reinterpret_cast<const uint8_t*>(all.data()), offs.data(),
                                  reinterpret_cast<const uint8_t*>(dst.data()), dst.size(), nonuniform ? 1 : 0, out.data(), oinf.data()));
    return unpack(out, oinf);
  }
  std::vector<AffinePoint> encode_to_curve(const std::vector<std::string>& msgs, const std::string& dst) { return hash_to_curve(msgs, dst, true); }
  // hash2curve::hash_to_scalar over a batch (group_digest.rs:131-143, L = 48)
  std::vector<Scalar> hash_to_scalar(const std::vector<std::string>& msgs, const std::string& dst) {
    size_t n = msgs.size();
    std::vector<uint64_t> offs(n + 1, 0);
    std::string all;
    for (size_t i = 0; i < n; i++) {
      all += msgs[i];
      offs[i + 1] = all.size();
    }
    std::vector<Scalar> r(n);
    check(ecg_hash_to_scalar_batch(ctx_, curve_, n, reinterpret_cast<const uint8_t*>(all.data()), offs.data(),
                                   reinterpret_cast<const uint8_t*>(dst.data()), dst.size(), reinterpret_cast<uint8_t*>(r.data())));
    return r;
  }

  // SM2 public-key encryption, digest SM3 (Engine(ECG_SM2, ...) only; mode 0 = C1C3C2, 1 = C1C2C3).
  // EncryptingKey::encrypt over a batch (sm2/src/pke/encrypting.rs:166-230) with the caller's ephemeral scalars k: one
  // recipient key, one ciphertext per message; an empty vector where status != 1 (0 refused, 2: draw another k).
  std::vector<std::vector<uint8_t>> sm2pke_encrypt(const AffinePoint& pb, const std::vector<Scalar>& k, const std::vector<std::string>& msgs,
                                                   int mode = 0, bool compressed = true, std::vector<uint8_t>* status = nullptr) {
    const size_t n = check_sizes(k.size(), msgs.size()), ovh = 32 + (compressed ? 33 : 65);
    std::vector<uint64_t> offs(n + 1, 0);
    std::string all;
    for (size_t i = 0; i < n; i++) {
      all += msgs[i];
      offs[i + 1] = all.size();
    }
    pack(std::vector<AffinePoint>(n, pb));
    std::vector<uint8_t> out(all.size() + n * ovh), st(n);
    check(ecg_sm2pke_encrypt_batch(ctx_, n, reinterpret_cast<const uint8_t*>(all.data()), offs.data(), flat(k), xy_.data(), mode,
                                   compressed ? 1 : 0, out.data(), st.data()));
    std::vector<std::vector<uint8_t>> r(n);
    for (size_t i = 0; i < n; i++)
      if (st[i] == 1) r[i].assign(out.begin() + offs[i] + i * ovh, out.begin() + offs[i + 1] + (i + 1) * ovh);
    if (status) *status = st;
    return r;
  }
  // DecryptingKey::decrypt over a batch (sm2/src/pke/decrypting.rs:174-222): one secret key; valid[i] = 0 where the
  // reference returns Err (its plaintext is then empty)
  std::vector<std::vector<uint8_t>> sm2pke_decrypt(const Scalar& d, const std::vector<std::vector<uint8_t>>& cts, int mode = 0,
                                                   std::vector<bool>* valid = nullptr) {
    const size_t n = cts.size();
    std::vector<uint64_t> offs(n + 1, 0), len(n);
    std::vector<uint8_t> all;
    for (size_t i = 0; i < n; i++) {
      all.insert(all.end(), cts[i].begin(), cts[i].end());
      offs[i + 1] = all.size();
    }
    std::vector<Scalar> ds(n, d);
    std::vector<uint8_t> out(all.size()), ok(n);
    check(ecg_sm2pke_decrypt_batch(ctx_, n, all.data(), offs.data(), flat(ds), mode, out.data(), len.data(), ok.data()));
    std::vector<std::vector<uint8_t>> r(n);
    for (size_t i = 0; i < n; i++)
      if (ok[i]) r[i].assign(out.begin() + offs[i], out.begin() + offs[i] + len[i]);
    if (valid) valid->assign(ok.begin(), ok.end());
    return r;
  }

  uint64_t kernel_launches() const { return ecg_kernel_launches(ctx_); }

 private:
  static size_t check_sizes(size_t a, size_t b) {
    if (a != b) throw Error(ECG_EINVAL, "points/scalars length mismatch");
    return a;
  }
  static const uint8_t* flat(const std::vector<Scalar>& s) { return reinterpret_cast<const uint8_t*>(s.data()); }
  void pack(const std::vector<AffinePoint>& pts) {
    xy_.resize(64 * pts.size());
    inf_.resize(pts.size());
    for (size_t i = 0; i < pts.size(); i++) {
      std::copy(pts[i].x.begin(), pts[i].x.end(), xy_.begin() + 64 * i);
      std::copy(pts[i].y.begin(), pts[i].y.end(), xy_.begin() + 64 * i + 32);
      inf_[i] = pts[i].infinity;
    }
  }
  static std::vector<AffinePoint> unpack(const std::vector<uint8_t>& xy, const std::vector<uint8_t>& inf) {
    std::vector<AffinePoint> r(inf.size());
    for (size_t i = 0; i < r.size(); i++) {
      std::copy(xy.begin() + 64 * i, xy.begin() + 64 * i + 32, r[i].x.begin());
      std::copy(xy.begin() + 64 * i + 32, xy.begin() + 64 * i + 64, r[i].y.begin());
      r[i].infinity = inf[i];
    }
    return r;
  }
  void check(ecg_status st) {
    if (st == ECG_OK) return;
    std::string m = ecg_last_error(ctx_);
    if (st == ECG_ESCALAR_RANGE || st == ECG_ENOT_ON_CURVE) throw DecodeError(st, m, ecg_last_error_index(ctx_));
    throw Error(st, m);
  }
  ecg_curve curve_;
  ecg_ctx* ctx_ = nullptr;
  std::vector<uint8_t> xy_, inf_;
};

}  // namespace ecgpu
