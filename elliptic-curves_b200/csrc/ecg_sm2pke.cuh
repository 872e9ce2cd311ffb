// ecg_sm2pke.cuh — SM2 public-key encryption around the variable-base kernel (sm2/src/pke.rs, pke/encrypting.rs:166-230,
// pke/decrypting.rs:174-222; GB/T 32918.4).  Group 1 (sm2) only.
//
//   decryption:  prep (parse C1, decode it, range-check d)  ->  [d]C1 = (x2, y2)  ->  sm2pke_kdf_kernel<false>
//   encryption:  prep (range-check k, Pb on the curve, M non-empty)  ->  [k]Pb = (x2, y2), [k]G = C1  ->  sm2pke_kdf_kernel<true>
//
// The KDF is SM3(x2 || y2 || BE32(j)), j = 1, 2, ... (pke.rs:349-381).  x2 || y2 is exactly one 64-byte block, so its
// midstate is computed once and every KDF block costs one compression (the counter block): 1 + ceil(L / 32) compressions
// for L message bytes, instead of 2 ceil(L / 32).  C3 = SM3(x2 || M || y2) streams alongside: ceil((L + 73) / 64).
// One thread per record; messages are read and written byte by byte at arbitrary offsets, as in h2c_kernel.
#pragma once
#include "ecg_kernels.cuh"
#include "ecg_sm3.cuh"

namespace ecg {

// bytes of C1 for a SEC1 tag over 32-byte field elements (sec1 Tag::message_len): 00 identity 1, 02 / 03 compressed and
// 05 compact 33, 04 uncompressed 65; 0 for any other tag (Tag::from_u8 refuses it)
ECG_D uint32_t sm2pke_c1_len(uint32_t tag) { return tag == 0 ? 1u : (tag == 2 || tag == 3 || tag == 5) ? 33u : tag == 4 ? 65u : 0u; }

// ciphertext record -> (C1 affine in internal form, ok).  Cipher::from_slice (pke.rs:122-160): the record holds at least
// C1 and the 32-byte C3 (C2 may be empty); C1 is decoded as FromSec1Point does (primeorder/src/affine.rs:204-229):
// uncompressed = from_coordinates, compressed = decompress by the tag's parity, compact = the even root, then
// y = min(y, p - y) (to_compact, :64-73).  The identity (tag 00) fails the reference's [h]C1 != O check: with a prime
// order any nonzero multiplier gives the same verdict as C1 != O.
template <class C>
ECG_D bool sm2pke_parse_c1(typename C::F::AffT& P, const uint8_t* rec, uint64_t len) {
  typedef typename C::F F;
  typedef typename F::FeT Fe;
  constexpr int NL = F::NL, FB = F::FB;
  static_assert(C::A_IS_MINUS3 == 1, "y^2 = x^3 - 3x + b");
  const uint32_t tag = len ? rec[0] : 0xFFu;
  const uint32_t c1len = sm2pke_c1_len(tag);
  if (c1len <= 1 || len < (uint64_t)c1len + 32) return false;
  Fe xc, b;
  load_be_bytes<NL, FB>(xc.v, rec + 1);
  if (!ltN<NL>(xc.v, C::P())) return false;
  F::from_canonical(P.x, xc);
  C::b_internal(b);
  if (tag == 4) {
    Fe yc;
    load_be_bytes<NL, FB>(yc.v, rec + 1 + FB);
    if (!ltN<NL>(yc.v, C::P())) return false;
    F::from_canonical(P.y, yc);
    return aff_on_curve<F, C::A_IS_MINUS3>(P, b);
  }
  Fe rhs, t, y, chk, yc;
  F::sqr(rhs, P.x);
  F::mul(rhs, rhs, P.x);
  F::mul_small(t, P.x, 3);
  F::sub(rhs, rhs, t);
  F::add(rhs, rhs, b);
  sqrt_candidate_generic<F, typename SqrtExp<C>::T>(y, rhs);
  F::sqr(chk, y);
  F::sub(chk, chk, rhs);
  if (!F::is_zero(chk)) return false;
  F::to_canonical(yc, y);
  if ((yc.v[0] & 1u) != (tag == 3 ? 1u : 0u)) F::neg(y, y);
  if (tag == 5) {  // compact: of y and p - y (the even root first), the smaller canonical value
    Fe ny, nyc;
    F::to_canonical(yc, y);
    F::neg(ny, y);
    F::to_canonical(nyc, ny);
    if (ltN<NL>(nyc.v, yc.v)) y = ny;
  }
  P.y = y;
  return true;
}

// a scalar record in [1, n - 1] (NonZeroScalar)
template <class C>
ECG_D bool sm2pke_load_nonzero_scalar(uint32_t* k, const uint8_t* p) {
  typedef typename C::F F;
  load_fe<F>(k, p);
  uint32_t any = 0;
#pragma unroll
  for (int i = 0; i < F::NL; i++) any |= k[i];
  return any != 0 && ltN<F::NL>(k, C::N());
}

// the variable-base inputs of one element: k, P as canonical records, or the stand-in (1, G) when !ok so that the
// launch stays uniform and its input checks stay quiet
template <class C>
ECG_D void sm2pke_store_inputs(uint8_t* k_out, uint8_t* pxy_out, size_t idx, uint32_t* k, typename C::F::AffT& P, bool ok) {
  typedef typename C::F F;
  constexpr int NL = F::NL, FB = F::FB;
  if (!ok) {
#pragma unroll
    for (int i = 0; i < NL; i++) k[i] = (i == 0);
    C::generator(P);
  }
  typename F::FeT xc, yc;
  F::to_canonical(xc, P.x);
  F::to_canonical(yc, P.y);
  store_fe<F>(k_out + FB * idx, k);
  store_fe<F>(pxy_out + 2 * FB * idx, xc.v);
  store_fe<F>(pxy_out + 2 * FB * idx + FB, yc.v);
}

}  // namespace ecg

// decryption front end: ciphertext i = cts[offsets[i] - cts_base ..), d = d32[i] -> (d, C1) for the variable-base kernel
template <class C>
ECG_KERNEL(128)
    sm2pke_dec_prep_kernel(const uint8_t* __restrict__ cts, const uint64_t* __restrict__ offsets, uint64_t cts_base, size_t n,
                           const uint8_t* __restrict__ d32, uint8_t* __restrict__ k_out, uint8_t* __restrict__ pxy_out,
                           uint8_t* __restrict__ ok_out) {
  size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n) return;
  typename C::F::AffT P;
  uint32_t d[C::F::NL];
  bool ok = ecg::sm2pke_parse_c1<C>(P, cts + (offsets[idx] - cts_base), offsets[idx + 1] - offsets[idx]);
  ok = ecg::sm2pke_load_nonzero_scalar<C>(d, d32 + C::F::FB * idx) && ok;
  ecg::sm2pke_store_inputs<C>(k_out, pxy_out, idx, d, P, ok);
  ok_out[idx] = ok ? 1 : 0;
}

// encryption front end: k in [1, n - 1] (NonZeroScalar), Pb = from_coordinates(x, y), a non-empty message (the
// reference's retry loop never ends on an empty one: its all-zero test over zero bytes is false)
template <class C>
ECG_KERNEL(128)
    sm2pke_enc_prep_kernel(const uint64_t* __restrict__ offsets, size_t n, const uint8_t* __restrict__ k32,
                           const uint8_t* __restrict__ pb_xy, uint8_t* __restrict__ k_out, uint8_t* __restrict__ pxy_out,
                           uint8_t* __restrict__ ok_out) {
  typedef typename C::F F;
  typedef typename F::FeT Fe;
  constexpr int NL = F::NL, FB = F::FB;
  size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n) return;
  uint32_t k[NL];
  bool ok = ecg::sm2pke_load_nonzero_scalar<C>(k, k32 + FB * idx) && offsets[idx + 1] > offsets[idx];
  typename F::AffT P;
  Fe xc, yc, b;
  load_fe<F>(xc.v, pb_xy + 2 * FB * idx);
  load_fe<F>(yc.v, pb_xy + 2 * FB * idx + FB);
  bool pok = ltN<NL>(xc.v, C::P()) && ltN<NL>(yc.v, C::P());
  F::from_canonical(P.x, xc);
  F::from_canonical(P.y, yc);
  C::b_internal(b);
  pok = pok && aff_on_curve<F, C::A_IS_MINUS3>(P, b);
  ok = ok && pok;
  ecg::sm2pke_store_inputs<C>(k_out, pxy_out, idx, k, P, ok);
  ok_out[idx] = ok ? 1 : 0;
}

// KDF, XOR, C3 and the record layout, one thread per record.  x2y2: [k]Pb or [d]C1 as 64-byte big-endian x || y records.
//   ENC: in = messages; record i goes to out + (offsets[i] - offsets[0]) + i * ovh as C1 || C3 || C2 (mode 0) or
//        C1 || C2 || C3 (mode 1), C1 = 02|03 || x (compressed) or 04 || x || y from c1xy; verdict 1, 2 (t all zero: the
//        caller draws another k) or 0 (refused by the front end); records with verdict != 1 are all zero.
//   DEC: in = ciphertexts; plaintext i goes to out + (offsets[i] - offsets[0]), pt_len[i] bytes, the rest of the record's
//        range zero; verdict 1 iff SM3(x2 || M' || y2) == C3 (compared without an early exit), else the range is zero.
template <bool ENC>
ECG_KERNEL(128)
    sm2pke_kdf_kernel(const uint8_t* __restrict__ in, const uint64_t* __restrict__ offsets, uint64_t in_base, size_t n, int mode,
                      int compressed, const uint8_t* __restrict__ x2y2, const uint8_t* __restrict__ c1xy, const uint8_t* __restrict__ ok,
                      uint8_t* __restrict__ out, uint8_t* __restrict__ verdict, uint64_t* __restrict__ pt_len) {
  size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n) return;
  const uint8_t* rec = in + (offsets[idx] - in_base);
  const uint64_t len = offsets[idx + 1] - offsets[idx];
  const uint32_t c1len = ENC ? (compressed ? 33u : 65u) : (len ? ecg::sm2pke_c1_len(rec[0]) : 0u);
  const uint64_t out_len = ENC ? len + c1len + 32 : len;
  uint8_t* dst = out + (offsets[idx] - offsets[0]) + (ENC ? idx * (uint64_t)(c1len + 32) : 0);
  if (!ok[idx]) {
#pragma unroll 1
    for (uint64_t i = 0; i < out_len; i++) dst[i] = 0;
    verdict[idx] = 0;
    if (!ENC) pt_len[idx] = 0;
    return;
  }
  const uint64_t L = ENC ? len : len - c1len - 32;  // message / C2 bytes
  const uint8_t* src = ENC ? rec : rec + c1len + (mode == 0 ? 32 : 0);      // M, or C2
  uint8_t* c2dst = ENC ? dst + c1len + (mode == 0 ? 32 : 0) : dst;           // C2, or M'
  // midstate of the KDF: one compression over the block x2 || y2
  uint32_t xy[16], mid[8];
  const uint8_t* pxy = x2y2 + 64 * idx;
#pragma unroll
  for (int i = 0; i < 16; i++)
    xy[i] = ((uint32_t)pxy[4 * i] << 24) | ((uint32_t)pxy[4 * i + 1] << 16) | ((uint32_t)pxy[4 * i + 2] << 8) | pxy[4 * i + 3];
  ecg::sm3_iv(mid);
  ecg::sm3_compress(mid, xy);
  // C3 stream: x2 first (32 bytes = half a block, so every 32-byte chunk of the message lands on a half-block boundary)
  ecg::Sm3Stream h;
  h.init();
#pragma unroll
  for (int i = 0; i < 8; i++) h.blk[i] = xy[i];
  h.fill = 32;
  h.total = 32;
  uint32_t tor = 0;  // OR of the key-stream bytes used (encrypting.rs:202: an all-zero t draws another k)
  const uint64_t chunks = (L + 31) / 32;
#pragma unroll 1
  for (uint64_t c = 0; c < chunks; c++) {
    uint32_t t[8], blk[16];
#pragma unroll
    for (int i = 0; i < 8; i++) t[i] = mid[i];
#pragma unroll
    for (int i = 0; i < 16; i++) blk[i] = 0;
    blk[0] = (uint32_t)(c + 1);  // BE32(j), then the padding of a 68-byte message
    blk[1] = 0x80000000u;
    blk[15] = (64 + 4) * 8;
    ecg::sm3_compress(t, blk);
    const uint64_t base = 32 * c;
    const uint32_t cnt = (uint32_t)(L - base < 32 ? L - base : 32);
#pragma unroll
    for (int b = 0; b < 32; b++) {
      if ((uint32_t)b < cnt) {
        const uint32_t tb = (t[b >> 2] >> (24 - 8 * (b & 3))) & 0xFFu;
        const uint32_t s = src[base + b];
        const uint32_t r = s ^ tb;
        tor |= tb;
        c2dst[base + b] = (uint8_t)r;
        h.put_noflush(ENC ? s : r);  // C3 hashes the plaintext: M (encryption), M' (decryption)
      }
    }
    if (h.fill == 64) h.flush_block();
  }
#pragma unroll 1
  for (int i = 0; i < 32; i++) h.put(pxy[32 + i]);
  uint32_t dg[8];
  h.finish(dg);
  if (ENC) {
    const bool good = tor != 0;
    if (good) {
      const uint8_t* pc = c1xy + 64 * idx;
      dst[0] = compressed ? (uint8_t)(2 | (pc[63] & 1)) : (uint8_t)4;
#pragma unroll 1
      for (uint32_t i = 0; i < c1len - 1; i++) dst[1 + i] = pc[i];
      uint8_t* c3 = mode == 0 ? dst + c1len : dst + c1len + L;
#pragma unroll
      for (int i = 0; i < 32; i++) c3[i] = (uint8_t)(dg[i >> 2] >> (24 - 8 * (i & 3)));
    } else {
#pragma unroll 1
      for (uint64_t i = 0; i < out_len; i++) dst[i] = 0;
    }
    verdict[idx] = good ? 1 : 2;
  } else {
    const uint8_t* c3 = mode == 0 ? rec + c1len : rec + c1len + L;
    uint32_t diff = 0;
#pragma unroll
    for (int i = 0; i < 32; i++) diff |= (uint32_t)c3[i] ^ ((dg[i >> 2] >> (24 - 8 * (i & 3))) & 0xFFu);
    const bool good = diff == 0;
#pragma unroll 1
    for (uint64_t i = good ? L : 0; i < out_len; i++) dst[i] = 0;
    verdict[idx] = good ? 1 : 0;
    pt_len[idx] = good ? L : 0;
  }
}
