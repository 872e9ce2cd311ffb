// ecg_sm3.cuh — SM3 (GB/T 32905-2016), the digest of SM2 public-key encryption (sm2/src/pke.rs:349-381, the KDF and C3;
// the reference takes it from the `sm3` crate).
//
//   compression: message expansion W[0..67] (W[j] = P1(W[j-16] ^ W[j-9] ^ (W[j-3] <<< 15)) ^ (W[j-13] <<< 7) ^ W[j-6]),
//   W'[j] = W[j] ^ W[j+4]; 64 rounds with FF / GG = XOR for j < 16 and majority / choice after, T_j <<< (j mod 32),
//   P0(X) = X ^ (X <<< 9) ^ (X <<< 17); the new state is the old one XOR the round output (not a sum, unlike SHA-2).
//   Padding and length field as SHA-256 (0x80, zeros, 64-bit big-endian bit count).
//
// The round loop is unrolled by 16 inside a loop over the four quarters, so the 16-word expansion window sits in
// registers with static indices and the code of one compression is 32 round bodies.  Host-compilable through ECG_D
// (tests/sim runs it).
#pragma once
#include <stddef.h>
#include <stdint.h>

#include "ecg_prim.cuh"

namespace ecg {

ECG_D uint32_t sm3_rotl(uint32_t x, int n) { return (n & 31) ? (x << (n & 31)) | (x >> (32 - (n & 31))) : x; }
ECG_D uint32_t sm3_p0(uint32_t x) { return x ^ sm3_rotl(x, 9) ^ sm3_rotl(x, 17); }
ECG_D uint32_t sm3_p1(uint32_t x) { return x ^ sm3_rotl(x, 15) ^ sm3_rotl(x, 23); }

ECG_D void sm3_iv(uint32_t* st) {
  const uint32_t iv[8] = {0x7380166fu, 0x4914b2b9u, 0x172442d7u, 0xda8a0600u, 0xa96f30bcu, 0x163138aau, 0xe38dee4du, 0xb0fb0e4eu};
#pragma unroll
  for (int i = 0; i < 8; i++) st[i] = iv[i];
}

// st = CF(st, block): block = 16 big-endian words.  `block` is not modified.
ECG_D void sm3_compress(uint32_t* st, const uint32_t* block) {
  uint32_t w[16];
#pragma unroll
  for (int i = 0; i < 16; i++) w[i] = block[i];
  uint32_t a = st[0], b = st[1], c = st[2], d = st[3], e = st[4], f = st[5], g = st[6], h = st[7];
  uint32_t tj = 0x79cc4519u;  // T_j <<< (j mod 32), rotated by one per round
#pragma unroll 1
  for (int q = 0; q < 4; q++) {
    if (q == 1) tj = sm3_rotl(0x7a879d8au, 16);
#pragma unroll
    for (int r = 0; r < 16; r++) {
      // W[j + 4] (j = 16 q + r) into the slot of W[j - 12], which is no longer needed
      if (q > 0 || r >= 12) {
        const uint32_t x = w[(r + 4) & 15] ^ w[(r + 11) & 15] ^ sm3_rotl(w[(r + 1) & 15], 15);  // W[j-12], W[j-5], W[j+1]
        w[(r + 4) & 15] = sm3_p1(x) ^ sm3_rotl(w[(r + 7) & 15], 7) ^ w[(r + 14) & 15];         // W[j-9], W[j-2]
      }
      const uint32_t wj = w[r & 15], wj4 = wj ^ w[(r + 4) & 15];
      const uint32_t a12 = sm3_rotl(a, 12);
      const uint32_t ss1 = sm3_rotl(a12 + e + tj, 7);
      const uint32_t ss2 = ss1 ^ a12;
      const uint32_t ff = q == 0 ? (a ^ b ^ c) : ((a & b) | (a & c) | (b & c));
      const uint32_t gg = q == 0 ? (e ^ f ^ g) : ((e & f) | (~e & g));
      const uint32_t tt1 = ff + d + ss2 + wj4;
      const uint32_t tt2 = gg + h + ss1 + wj;
      d = c;
      c = sm3_rotl(b, 9);
      b = a;
      a = tt1;
      h = g;
      g = sm3_rotl(f, 19);
      f = e;
      e = sm3_p0(tt2);
      tj = sm3_rotl(tj, 1);
    }
  }
  st[0] ^= a;
  st[1] ^= b;
  st[2] ^= c;
  st[3] ^= d;
  st[4] ^= e;
  st[5] ^= f;
  st[6] ^= g;
  st[7] ^= h;
}

// ---- streaming SM3 (byte-granular updates, as Sha256Stream in ecg_h2c.cuh) --------------------------------------
struct Sm3Stream {
  uint32_t st[8];
  uint32_t blk[16];
  uint32_t fill;   // bytes in blk
  uint64_t total;  // bytes absorbed
  ECG_D void init() {
    sm3_iv(st);
#pragma unroll
    for (int i = 0; i < 16; i++) blk[i] = 0;
    fill = 0;
    total = 0;
  }
  ECG_D void flush_block() {
    sm3_compress(st, blk);
#pragma unroll
    for (int i = 0; i < 16; i++) blk[i] = 0;
    fill = 0;
  }
  // one byte without the block check: the caller flushes when fill reaches 64
  ECG_D void put_noflush(uint32_t byte) {
    blk[fill >> 2] |= (byte & 0xFFu) << (24 - 8 * (fill & 3));
    fill++;
    total++;
  }
  ECG_D void put(uint32_t byte) {
    put_noflush(byte);
    if (fill == 64) flush_block();
  }
  ECG_D void update(const uint8_t* p, size_t len) {
#pragma unroll 1
    for (size_t i = 0; i < len; i++) put(p[i]);
  }
  ECG_D void finish(uint32_t* digest /* 8 big-endian words */) {
    const uint64_t bits = total * 8;
    put(0x80u);
    if (fill > 56) flush_block();
    blk[14] = (uint32_t)(bits >> 32);
    blk[15] = (uint32_t)bits;
    sm3_compress(st, blk);
#pragma unroll
    for (int i = 0; i < 8; i++) digest[i] = st[i];
  }
};

// SM3 of one message (tests / host simulation)
ECG_D void sm3_digest(uint8_t* out32, const uint8_t* msg, size_t len) {
  Sm3Stream h;
  h.init();
  h.update(msg, len);
  uint32_t dg[8];
  h.finish(dg);
#pragma unroll
  for (int i = 0; i < 32; i++) out32[i] = (uint8_t)(dg[i >> 2] >> (24 - 8 * (i & 3)));
}

}  // namespace ecg
