// Shared epilogue helpers (bf16 packing, ReLU masks) and the plain-GEMM problems with which the unit tests validate
// the register-gather tcgen05 mainloop of igemm.cuh (K-major and MN-major descriptors) in isolation.
// The encoder itself runs on the TMA kernels: res_problems.cuh (convs) and tma_problems.cuh (fc layer).
#pragma once
#include "igemm.cuh"

namespace srl {

typedef __nv_bfloat16 bf16;

SRL_DEVINL uint4 ldg16(const void* p) { return __ldg(reinterpret_cast<const uint4*>(p)); }
SRL_DEVINL uint4 zero16() { return make_uint4(0, 0, 0, 0); }

SRL_DEVINL void store_bf16x16(bf16* dst, const float (&v)[16]) {
  uint4 a = make_uint4(pack_bf16x2(v[0], v[1]), pack_bf16x2(v[2], v[3]), pack_bf16x2(v[4], v[5]), pack_bf16x2(v[6], v[7]));
  uint4 b = make_uint4(pack_bf16x2(v[8], v[9]), pack_bf16x2(v[10], v[11]), pack_bf16x2(v[12], v[13]), pack_bf16x2(v[14], v[15]));
  reinterpret_cast<uint4*>(dst)[0] = a;
  reinterpret_cast<uint4*>(dst)[1] = b;
}
// v[j] *= (mask[j] > 0) for 16 bf16 mask values
SRL_DEVINL void relu_mask16(const bf16* mask, float (&v)[16]) {
  uint4 a = ldg16(mask), b = ldg16(mask + 8);
  const uint32_t w[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    if (!(bf16_lo(w[i]) > 0.f)) v[2 * i] = 0.f;
    if (!(bf16_hi(w[i]) > 0.f)) v[2 * i + 1] = 0.f;
  }
}

// same with the 32 mask bytes already in registers (prefetched before the accumulator was waited for)
SRL_DEVINL void relu_mask16_pre(const uint4 (&m)[2], float (&v)[16]) {
  const uint32_t w[8] = {m[0].x, m[0].y, m[0].z, m[0].w, m[1].x, m[1].y, m[1].z, m[1].w};
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    if (!(bf16_lo(w[i]) > 0.f)) v[2 * i] = 0.f;
    if (!(bf16_hi(w[i]) > 0.f)) v[2 * i + 1] = 0.f;
  }
}
SRL_DEVINL void ld_mask16(const bf16* mask, uint4 (&m)[2]) { m[0] = ldg16(mask); m[1] = ldg16(mask + 8); }

// ============================================================================================
// plain GEMM problems used by the unit tests to validate descriptors / pipeline in isolation
// ============================================================================================
struct TestGemmK {    // D[M][N] = A[M][K] * B[N][K]^T, K % 64 == 0, N % 64 == 0; grid = (ceil(M/128), N/64)
  static constexpr int BN = 64, STAGES = 3;
  static constexpr bool A_MN = false, B_MN = false;
  static constexpr int BIAS = 0, BIAS_N = 0;
  struct Params { const bf16* A; const bf16* B; float* D; int M, N, K; };
  typedef int RowA;
  typedef int RowB;
  SRL_DEVINL static int num_kblocks(const Params& p, int, int) { return p.K / 64; }
  SRL_DEVINL static RowA make_rowA(const Params& p, int tm, int, int srow) { const int m = tm * 128 + srow; return m < p.M ? m : -1; }
  SRL_DEVINL static RowB make_rowB(const Params&, int, int ty, int srow) { return ty * 64 + srow; }
  SRL_DEVINL static uint4 load_A(const Params& p, RowA m, int kb, int chunk) {
    return m < 0 ? zero16() : ldg16(p.A + (size_t)m * p.K + kb * 64 + chunk * 8);
  }
  SRL_DEVINL static uint4 load_B(const Params& p, RowB n, int kb, int chunk) { return ldg16(p.B + (size_t)n * p.K + kb * 64 + chunk * 8); }
  SRL_DEVINL static void epilogue16(const Params& p, int tm, int ty, int row, int c0, float (&v)[16]) {
    const int m = tm * 128 + row;
    if (m >= p.M) return;
#pragma unroll
    for (int j = 0; j < 16; ++j) p.D[(size_t)m * p.N + ty * 64 + c0 + j] = v[j];
  }
};
struct TestGemmMN {   // D[M][N] = At[K][M]^T * Bt[K][N], M % 128 == 0, N % 64 == 0, any K; grid = (M/128, N/64)
  static constexpr int BN = 64, STAGES = 3;
  static constexpr bool A_MN = true, B_MN = true;
  static constexpr int BIAS = 0, BIAS_N = 0;
  struct Params { const bf16* At; const bf16* Bt; float* D; int M, N, K; };
  typedef int RowA;
  typedef int RowB;
  SRL_DEVINL static int num_kblocks(const Params& p, int, int) { return (p.K + 63) / 64; }
  SRL_DEVINL static RowA make_rowA(const Params&, int, int, int srow) { return srow; }
  SRL_DEVINL static RowB make_rowB(const Params&, int, int, int srow) { return srow; }
  SRL_DEVINL static uint4 load_A(const Params& p, RowA srow, int kb, int chunk) {
    const int k = kb * 64 + (srow & 63);
    return k < p.K ? ldg16(p.At + (size_t)k * p.M + blockIdx.x * 128 + (srow >> 6) * 64 + chunk * 8) : zero16();
  }
  SRL_DEVINL static uint4 load_B(const Params& p, RowB srow, int kb, int chunk) {
    const int k = kb * 64 + srow;
    return k < p.K ? ldg16(p.Bt + (size_t)k * p.N + blockIdx.y * 64 + chunk * 8) : zero16();
  }
  SRL_DEVINL static void epilogue16(const Params& p, int tm, int ty, int row, int c0, float (&v)[16]) {
#pragma unroll
    for (int j = 0; j < 16; ++j) p.D[(size_t)(tm * 128 + row) * p.N + ty * 64 + c0 + j] = v[j];
  }
};

}  // namespace srl
