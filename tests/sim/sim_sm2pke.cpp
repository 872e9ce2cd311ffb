// tests/sim/sim_sm2pke.cpp — HOST SIMULATION of the SM2 public-key encryption kernels (test infrastructure only): the
// execution-model shim and the kernel launchers of sim.cpp, plus the SM3 / SM2 encryption headers, in a library of its own
// (libecgsim_sm2pke.so).  Never linked into libecgpu.so; never used as a fallback.
#include "sim.cpp"

#include "../../elliptic-curves_b200/csrc/ecg_sm2pke.cuh"

// SM3 of one message (ecg_sm3.cuh)
extern "C" int simk_sm3(const uint8_t* msg, size_t len, uint8_t* out32) {
  sm3_digest(out32, msg, len);
  return 0;
}

// ecg_sm2pke_decrypt_batch / ecg_sm2pke_encrypt_batch as ecgpu.cu chains them: front end -> variable-base [d]C1 or [k]Pb
// -> normalize -> (encryption: [k]G by the fixed-base table, or with table == nullptr by the variable-base routine with
// P = G, the ECG_FLAG_CONSTTIME path) -> KDF / C3 / record layout.  Returns the variable-base kernels' error flags
// (0: the front ends' stand-ins kept them quiet).
static uint32_t simk_sm2_varbase(size_t n, const uint8_t* k, const uint8_t* pxy, uint8_t* out_xy, uint8_t* out_inf) {
  typedef CurveSm2 C;
  size_t blocks = (n + SIM_BLOCK - 1) / SIM_BLOCK;
  std::vector<uint32_t> jac(24 * n + 24), gtab(blocks * SIM_BLOCK * (8 * 24));
  uint32_t status[2] = {0, 0xFFFFFFFFu};
  if (pxy)
    sim_launch(n, SIM_BLOCK, [&] { generic_varbase_kernel<C, SIM_BLOCK, 4>(k, pxy, nullptr, n, jac.data(), gtab.data(), status, 0); });
  else
    sim_launch(n, SIM_BLOCK, [&] { generic_varbase_kernel<C, SIM_BLOCK, 4, true>(k, nullptr, nullptr, n, jac.data(), gtab.data(), status, 0); });
  simk_normalize<C>(jac, n, out_xy, out_inf);
  return status[0];
}
extern "C" int simk_sm2pke_decrypt(size_t n, const uint8_t* cts, const uint64_t* offsets, const uint8_t* d32, int mode, uint8_t* out,
                                   uint64_t* pt_len, uint8_t* valid) {
  std::vector<uint8_t> vk(32 * n + 32), vp(64 * n + 64), vok(n + 1), vxy(64 * n + 64), vinf(n + 1);
  sim_launch(n, 128, [&] { sm2pke_dec_prep_kernel<CurveSm2>(cts, offsets, 0, n, d32, vk.data(), vp.data(), vok.data()); });
  uint32_t err = simk_sm2_varbase(n, vk.data(), vp.data(), vxy.data(), vinf.data());
  sim_launch(n, 128, [&] { sm2pke_kdf_kernel<false>(cts, offsets, 0, n, mode, 0, vxy.data(), nullptr, vok.data(), out, valid, pt_len); });
  return (int)err;
}
extern "C" int simk_sm2pke_encrypt(size_t n, const uint8_t* msgs, const uint64_t* offsets, const uint8_t* k32, const uint8_t* pb_xy, int mode,
                                   int compressed, const uint32_t* table, uint8_t* out, uint8_t* status) {
  std::vector<uint8_t> vk(32 * n + 32), vp(64 * n + 64), vok(n + 1), vxy(64 * n + 64), vinf(n + 1), c1xy(64 * n + 64), c1inf(n + 1);
  sim_launch(n, 128, [&] { sm2pke_enc_prep_kernel<CurveSm2>(offsets, n, k32, pb_xy, vk.data(), vp.data(), vok.data()); });
  uint32_t err = simk_sm2_varbase(n, vk.data(), vp.data(), vxy.data(), vinf.data());
  if (table) {
    std::vector<uint32_t> jac(24 * n + 24);
    uint32_t st[2] = {0, 0xFFFFFFFFu};
    sim_launch(n, 128, [&] { fixedbase_kernel<CurveSm2>(vk.data(), n, table, jac.data(), st, 0); });
    simk_normalize<CurveSm2>(jac, n, c1xy.data(), c1inf.data());
    err |= st[0];
  } else {
    err |= simk_sm2_varbase(n, vk.data(), nullptr, c1xy.data(), c1inf.data());
  }
  sim_launch(n, 128, [&] {
    sm2pke_kdf_kernel<true>(msgs, offsets, 0, n, mode, compressed, vxy.data(), c1xy.data(), vok.data(), out, status, nullptr);
  });
  return (int)err;
}
