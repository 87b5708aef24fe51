// 2-layer LSTM core of AtariNet(use_lstm=True): forward over T1 = T+1 steps with done-resets and BPTT over the first T
// steps (reference: scalerl/algorithms/utils/atari_model.py:52-55,61-75,109-120; SURVEY.md §8 row a17).
//
//   gates_t = x_t Wih^T + b_ih + (m_t . h_{t-1}) Whh^T + b_hh ;  i,f,g,o ;  c_t = f (m_t . c_{t-1}) + i g ;  h_t = o tanh(c_t)
//
// Work split per layer:
//   * input projection of ALL steps in one tcgen05 GEMM  [T1*B x Hp] x [Hp x 4Hp]          (LGemmK)
//   * per step: recurrent tcgen05 GEMM [B x Hp] x [Hp x 4Hp] + one fused cell kernel     (sequential over t)
//   * BPTT per step: cell backward kernel + recurrent GEMM [B x 4Hp] x [4Hp x Hp]
//   * after the scan: dX (one GEMM), dWih / dWhh (two MN-major GEMMs over all T*B rows), bias gradients (column sums)
// H = 513 + A is padded to Hp (multiple of 64); the gate dimension is laid out [4][Hp] so every GEMM has K = Hp or 4Hp.
// All GEMM operands are bf16 (fp32 accumulate in TMEM); cell state, gate activations and gradients are fp32.
#include <stdio.h>
#include <new>
#include "tma_problems.cuh"
#include "kernels.h"
#include "../../include/scalerl_b200.h"

namespace srl {

// ------------------------------------------------------------------------------------------------ generic GEMM problems
struct LGemmK {
  static constexpr int KID = 34;
  static constexpr bool PREFETCH = false;      // C[c_row0 + m][n] = sum_k A[a_row0 + m][k] * B[n][k];  grid = (ceil(M/128), Npad/64)
  static constexpr int BN = 64, STAGES = 4, KROWS = 64;
  static constexpr bool A_MN = false, B_MN = false, ZERO_INIT = false;
  struct Params { SRL_TMAP a; SRL_TMAP b; float* C; int M, nkb, ldc, a_row0, c_row0; };
  SRL_DEVINL static void prefetch(const Params& p) { tma_prefetch_desc(&p.a); tma_prefetch_desc(&p.b); }
  SRL_DEVINL static int num_kblocks(const Params& p, int, int) { return p.nkb; }
  SRL_DEVINL static void issue(const Params& p, int tm, int ty, int kb, uint8_t* sA, uint8_t* sB, uint64_t* bar) {
    mbar_arrive_expect_tx(bar, 128 * 128 + 64 * 128);
    tma_load_2d(sA, &p.a, bar, kb * 64, p.a_row0 + tm * 128);
    tma_load_2d(sB, &p.b, bar, kb * 64, ty * 64);
  }
  SRL_DEVINL static void epilogue16(const Params& p, int tm, int ty, int row, int c0, float (&v)[16]) {
    const int m = tm * 128 + row;
    if (m >= p.M) return;
    float4* o = reinterpret_cast<float4*>(p.C + (size_t)(p.c_row0 + m) * p.ldc + ty * 64 + c0);
#pragma unroll
    for (int j = 0; j < 4; ++j) o[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
  }
};
struct LGemmMN {
  static constexpr int KID = 35;
  static constexpr bool PREFETCH = false;     // C[i][j] = sum_r A[r][i] * B[r][j]  (rows r = samples, MN-major operands); grid = (Ipad/128, Jpad/64)
  static constexpr int BN = 64, STAGES = 4, KROWS = 64;
  static constexpr bool A_MN = true, B_MN = true, ZERO_INIT = false;
  struct Params { SRL_TMAP a; SRL_TMAP b; float* C; int R, ldc; };
  SRL_DEVINL static void prefetch(const Params& p) { tma_prefetch_desc(&p.a); tma_prefetch_desc(&p.b); }
  SRL_DEVINL static int num_kblocks(const Params& p, int, int) { return (p.R + 63) >> 6; }
  SRL_DEVINL static void init_smem(const Params&, int, int, uint8_t*, int, int) {}
  SRL_DEVINL static void issue(const Params& p, int tm, int ty, int kb, uint8_t* sA, uint8_t* sB, uint64_t* bar) {
    mbar_arrive_expect_tx(bar, 3 * 64 * 128);
    tma_load_2d(sA, &p.a, bar, tm * 128, kb * 64);
    tma_load_2d(sA + KROWS * 128, &p.a, bar, tm * 128 + 64, kb * 64);
    tma_load_2d(sB, &p.b, bar, ty * 64, kb * 64);
  }
  SRL_DEVINL static void epilogue16(const Params& p, int tm, int ty, int row, int c0, float (&v)[16]) {
    float4* o = reinterpret_cast<float4*>(p.C + (size_t)(tm * 128 + row) * p.ldc + ty * 64 + c0);
#pragma unroll
    for (int j = 0; j < 4; ++j) o[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
  }
};

// ------------------------------------------------------------------------------------------------ element-wise kernels
SRL_DEVINL float sigmoidf_(float x) { return 1.0f / (1.0f + expf(-x)); }

// fp32 [rows][H] -> bf16 [rows][Hp] (zero padded)
__global__ void lstm_pad_bf16_kernel(const float* __restrict__ x, int rows, int H, int Hp, __nv_bfloat16* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)rows * Hp) return;
  const int r = (int)(i / Hp), j = (int)(i - (int64_t)r * Hp);
  out[i] = __float2bfloat16_rn(j < H ? x[(size_t)r * H + j] : 0.f);
}
// weights fp32 [4H][H] -> bf16 Wp [4Hp][Hp] (gate-major rows, zero padded) and its transpose WTp [Hp][4Hp]
__global__ void lstm_pack_w_kernel(const float* __restrict__ w, int H, int Hp, __nv_bfloat16* __restrict__ Wp, __nv_bfloat16* __restrict__ WTp) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int G = 4 * Hp;
  if (i >= (int64_t)G * Hp) return;
  const int row = (int)(i / Hp), k = (int)(i - (int64_t)row * Hp), q = row / Hp, j = row - q * Hp;
  const float v = (j < H && k < H) ? w[(size_t)(q * H + j) * H + k] : 0.f;
  const __nv_bfloat16 b = __float2bfloat16_rn(v);
  Wp[i] = b;
  WTp[(size_t)k * G + row] = b;
}
// state for step 0: hm[0] = m_0 . h_init (bf16, padded)
__global__ void lstm_init_hm_kernel(const float* __restrict__ h_init, const uint8_t* __restrict__ done, int B, int H, int Hp,
                                    __nv_bfloat16* __restrict__ hm0) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * Hp) return;
  const int b = i / Hp, j = i - b * Hp;
  const float m = done[b] ? 0.f : 1.f;
  hm0[i] = __float2bfloat16_rn(j < H ? m * h_init[(size_t)b * H + j] : 0.f);
}

// fused cell, one thread per (b, j): consumes gx[t], the recurrent product r, biases; writes gate activations, c_t, h_t (fp32),
// h_t (bf16, input of the next layer / wgrad operand) and hm[t+1] = m_{t+1} . h_t (bf16, next step's recurrent operand)
__global__ void lstm_cell_fwd_kernel(const float* __restrict__ gx, const float* __restrict__ r, const float* __restrict__ b_ih,
                                     const float* __restrict__ b_hh, const float* __restrict__ c_prev, const uint8_t* __restrict__ done_t,
                                     const uint8_t* __restrict__ done_next, int B, int H, int Hp, float* __restrict__ gates,
                                     float* __restrict__ c_out, float* __restrict__ h_out, __nv_bfloat16* __restrict__ h_bf,
                                     __nv_bfloat16* __restrict__ hm_next) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * Hp) return;
  const int b = i / Hp, j = i - b * Hp, G = 4 * Hp;
  float hv = 0.f, cv = 0.f, a[4] = {0.f, 0.f, 0.f, 0.f};
  if (j < H) {
    float pre[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) pre[q] = gx[(size_t)b * G + q * Hp + j] + r[(size_t)b * G + q * Hp + j] + b_ih[q * H + j] + b_hh[q * H + j];
    a[0] = sigmoidf_(pre[0]); a[1] = sigmoidf_(pre[1]); a[2] = tanhf(pre[2]); a[3] = sigmoidf_(pre[3]);
    const float cp = done_t[b] ? 0.f : c_prev[(size_t)b * Hp + j];
    cv = a[1] * cp + a[0] * a[2];
    hv = a[3] * tanhf(cv);
  }
#pragma unroll
  for (int q = 0; q < 4; ++q) gates[(size_t)b * G + q * Hp + j] = a[q];
  c_out[i] = cv;
  h_out[i] = hv;
  h_bf[i] = __float2bfloat16_rn(hv);
  if (hm_next) hm_next[i] = __float2bfloat16_rn(done_next[b] ? 0.f : hv);
}

// BPTT cell: dh = dh_out[t] + m_{t+1} . dhm_{t+1};  writes dgates (bf16) and the carried dc
__global__ void lstm_cell_bwd_kernel(const float* __restrict__ dh_out, const float* __restrict__ dhm_next, const uint8_t* __restrict__ done_next,
                                     const float* __restrict__ gates, const float* __restrict__ c_t, const float* __restrict__ c_prev,
                                     const uint8_t* __restrict__ done_t, float* __restrict__ dc_carry, int B, int H, int Hp,
                                     __nv_bfloat16* __restrict__ dgates) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * Hp) return;
  const int b = i / Hp, j = i - b * Hp, G = 4 * Hp;
  float d[4] = {0.f, 0.f, 0.f, 0.f};
  float dc_out = 0.f;
  if (j < H) {
    float dh = dh_out ? dh_out[i] : 0.f;
    if (dhm_next && !done_next[b]) dh += dhm_next[i];
    const float ig = gates[(size_t)b * G + j], fg = gates[(size_t)b * G + Hp + j], gg = gates[(size_t)b * G + 2 * Hp + j],
                og = gates[(size_t)b * G + 3 * Hp + j];
    const float tc = tanhf(c_t[i]);
    const float dct = dh * og * (1.f - tc * tc) + dc_carry[i];
    const float cp = done_t[b] ? 0.f : c_prev[i];
    d[0] = dct * gg * ig * (1.f - ig);
    d[1] = dct * cp * fg * (1.f - fg);
    d[2] = dct * ig * (1.f - gg * gg);
    d[3] = dh * tc * og * (1.f - og);
    dc_out = done_t[b] ? 0.f : dct * fg;     // flows into c_{t-1} through m_t
  }
  dc_carry[i] = dc_out;
#pragma unroll
  for (int q = 0; q < 4; ++q) dgates[(size_t)b * G + q * Hp + j] = __float2bfloat16_rn(d[q]);
}

// db[q*H + j] += sum_rows dgates[row][q*Hp + j]
__global__ void lstm_bias_grad_kernel(const __nv_bfloat16* __restrict__ dgates, int rows, int H, int Hp, int rows_per_block, float* __restrict__ db_ih,
                                      float* __restrict__ db_hh) {
  const int col = blockIdx.x * blockDim.x + threadIdx.x, G = 4 * Hp;
  if (col >= G) return;
  const int q = col / Hp, j = col - q * Hp;
  if (j >= H) return;
  const int r0 = blockIdx.y * rows_per_block, r1 = min(rows, r0 + rows_per_block);
  float s = 0.f;
  for (int r = r0; r < r1; ++r) s += __bfloat162float(dgates[(size_t)r * G + col]);
  atomicAdd(db_ih + q * H + j, s);
  atomicAdd(db_hh + q * H + j, s);
}
// padded fp32 [4Hp][Hp] -> PyTorch [4H][H] (accumulate)
__global__ void lstm_unpad_w_kernel(const float* __restrict__ src, int H, int Hp, float* __restrict__ dst) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)4 * H * H) return;
  const int row = (int)(i / H), k = (int)(i - (int64_t)row * H), q = row / H, j = row - q * H;
  dst[i] += src[(size_t)(q * Hp + j) * Hp + k];
}
// fp32 [rows][Hp] -> fp32 [rows][H]
__global__ void lstm_unpad_rows_kernel(const float* __restrict__ src, int rows, int H, int Hp, float* __restrict__ dst) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)rows * H) return;
  const int r = (int)(i / H), j = (int)(i - (int64_t)r * H);
  dst[i] = src[(size_t)r * Hp + j];
}

}  // namespace srl

using namespace srl;

// ------------------------------------------------------------------------------------------------ context
struct srl_lstm {
  int T1, B, H, Hp, G;
  const float* w[2][4];      // weight_ih, weight_hh, bias_ih, bias_hh (fp32, PyTorch layouts, caller-owned)
  float* g[2][4];            // gradients (same layouts), accumulated
  char* arena;
  // bf16 operands
  __nv_bfloat16 *xin[2];     // layer input rows [T1*B][Hp]        (xin[1] == hbf[0])
  __nv_bfloat16 *hm[2];      // m_t . h_{t-1} rows [T1*B][Hp]
  __nv_bfloat16 *hbf[2];     // h_t rows [T1*B][Hp]
  __nv_bfloat16 *Wih[2], *WihT[2], *Whh[2], *WhhT[2];
  __nv_bfloat16 *dgates[2];  // [T*B][G]
  // fp32
  float *gx, *r, *gates[2], *cseq[2], *hseq[2], *dc, *dhm, *dx, *dwpad;
  float *h_init, *c_init;    // [2][B][Hp] padded copies
  CUtensorMap m_xin[2], m_hm[2], m_hm64[2], m_xin64[2], m_Wih[2], m_Whh[2], m_WihT[2], m_WhhT[2], m_dg128[2], m_dg64[2];
};

static thread_local char g_lerr[256] = "";
extern "C" const char* srl_lstm_last_error(void) { return g_lerr; }
#define LCU(x, what) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { snprintf(g_lerr, sizeof(g_lerr), "%s: %s", what, cudaGetErrorString(e_)); return (int)e_; } } while (0)
#define LREQ(c, msg) do { if (!(c)) { snprintf(g_lerr, sizeof(g_lerr), "%s", msg); return SRL_EINVAL; } } while (0)

static bool map2(CUtensorMap* m, const void* base, uint64_t cols, uint64_t rows, uint32_t boxrows) {
  const uint64_t d[2] = {cols, rows}, s[1] = {cols};
  const uint32_t bx[2] = {64, boxrows};
  return make_map(m, base, 2, d, s, bx);
}

extern "C" int srl_lstm_create(int T1, int B, int H, const float* const* weights8, float* const* grads8, srl_lstm_t** out) {
  LREQ(T1 >= 2 && B >= 1 && H >= 1 && weights8 && grads8 && out, "lstm_create: bad argument");
  srl_lstm* L = new (std::nothrow) srl_lstm();
  LREQ(L, "out of memory");
  L->T1 = T1; L->B = B; L->H = H; L->Hp = (H + 63) / 64 * 64; L->G = 4 * L->Hp;
  for (int l = 0; l < 2; ++l) for (int k = 0; k < 4; ++k) { L->w[l][k] = weights8[l * 4 + k]; L->g[l][k] = grads8[l * 4 + k]; }
  const int64_t N1 = (int64_t)T1 * B, NB = (int64_t)(T1 - 1) * B, Hp = L->Hp, G = L->G;
  auto al = [](int64_t b) { return (b + 255) & ~int64_t(255); };
  int64_t total = 0;
  auto take = [&](int64_t bytes) { const int64_t o = total; total += al(bytes); return o; };
  int64_t o_xin0 = take(N1 * Hp * 2), o_hm[2], o_hbf[2], o_W[2][4], o_dg[2], o_gates[2], o_c[2], o_h[2];
  for (int l = 0; l < 2; ++l) {
    o_hm[l] = take(N1 * Hp * 2); o_hbf[l] = take(N1 * Hp * 2);
    for (int k = 0; k < 4; ++k) o_W[l][k] = take(G * Hp * 2);
    o_dg[l] = take(NB * G * 2); o_gates[l] = take(N1 * G * 4); o_c[l] = take(N1 * Hp * 4); o_h[l] = take(N1 * Hp * 4);
  }
  const int64_t o_gx = take(N1 * G * 4), o_r = take((int64_t)B * G * 4), o_dc = take((int64_t)B * Hp * 4), o_dhm = take((int64_t)B * Hp * 4),
                o_dx = take(NB * Hp * 4), o_dw = take(G * Hp * 4), o_hi = take(2 * (int64_t)B * Hp * 4), o_ci = take(2 * (int64_t)B * Hp * 4);
  if (cudaMalloc(&L->arena, total) != cudaSuccess || cudaMemset(L->arena, 0, total) != cudaSuccess) { delete L; LREQ(false, "lstm_create: cudaMalloc failed"); }
  char* a = L->arena;
  L->xin[0] = (__nv_bfloat16*)(a + o_xin0);
  for (int l = 0; l < 2; ++l) {
    L->hm[l] = (__nv_bfloat16*)(a + o_hm[l]); L->hbf[l] = (__nv_bfloat16*)(a + o_hbf[l]);
    L->Wih[l] = (__nv_bfloat16*)(a + o_W[l][0]); L->WihT[l] = (__nv_bfloat16*)(a + o_W[l][1]);
    L->Whh[l] = (__nv_bfloat16*)(a + o_W[l][2]); L->WhhT[l] = (__nv_bfloat16*)(a + o_W[l][3]);
    L->dgates[l] = (__nv_bfloat16*)(a + o_dg[l]); L->gates[l] = (float*)(a + o_gates[l]); L->cseq[l] = (float*)(a + o_c[l]); L->hseq[l] = (float*)(a + o_h[l]);
  }
  L->xin[1] = L->hbf[0];
  L->gx = (float*)(a + o_gx); L->r = (float*)(a + o_r); L->dc = (float*)(a + o_dc); L->dhm = (float*)(a + o_dhm); L->dx = (float*)(a + o_dx);
  L->dwpad = (float*)(a + o_dw); L->h_init = (float*)(a + o_hi); L->c_init = (float*)(a + o_ci);
  bool ok = true;
  for (int l = 0; l < 2 && ok; ++l) {
    ok = ok && map2(&L->m_xin[l], L->xin[l], Hp, N1, 128) && map2(&L->m_xin64[l], L->xin[l], Hp, NB, 64) && map2(&L->m_hm[l], L->hm[l], Hp, N1, 128) &&
         map2(&L->m_hm64[l], L->hm[l], Hp, NB, 64) && map2(&L->m_Wih[l], L->Wih[l], Hp, G, 64) && map2(&L->m_Whh[l], L->Whh[l], Hp, G, 64) &&
         map2(&L->m_WihT[l], L->WihT[l], G, Hp, 64) && map2(&L->m_WhhT[l], L->WhhT[l], G, Hp, 64) && map2(&L->m_dg128[l], L->dgates[l], G, NB, 128) &&
         map2(&L->m_dg64[l], L->dgates[l], G, NB, 64);
  }
  if (!ok) { cudaFree(L->arena); delete L; LREQ(false, "lstm_create: tensor map creation failed"); }
  *out = L;
  return 0;
}
extern "C" int srl_lstm_destroy(srl_lstm_t* L) { if (L) { cudaFree(L->arena); delete L; } return 0; }

static inline int cdiv_(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }

// core fp32 [T1*B][H], done u8 [T1*B], h0/c0 fp32 [2][B][H] -> out fp32 [T1*B][H], hT/cT fp32 [2][B][H] (may be NULL)
extern "C" int srl_lstm_forward(srl_lstm_t* L, const float* core, const uint8_t* done, const float* h0, const float* c0, float* out,
                                float* hT, float* cT, void* stream) {
  LREQ(L && core && done && h0 && c0 && out, "lstm_forward: NULL pointer");
  cudaStream_t st = (cudaStream_t)stream;
  const int T1 = L->T1, B = L->B, H = L->H, Hp = L->Hp, G = L->G;
  const int64_t N1 = (int64_t)T1 * B;
  lstm_pad_bf16_kernel<<<cdiv_(N1 * Hp, 256), 256, 0, st>>>(core, (int)N1, H, Hp, L->xin[0]);
  for (int l = 0; l < 2; ++l) {
    lstm_pack_w_kernel<<<cdiv_((int64_t)G * Hp, 256), 256, 0, st>>>(L->w[l][0], H, Hp, L->Wih[l], L->WihT[l]);
    lstm_pack_w_kernel<<<cdiv_((int64_t)G * Hp, 256), 256, 0, st>>>(L->w[l][1], H, Hp, L->Whh[l], L->WhhT[l]);
  }
  LCU(cudaGetLastError(), "lstm pack");
  const int cell_blocks = cdiv_((int64_t)B * Hp, 256);
  for (int l = 0; l < 2; ++l) {
    // padded copies of the initial state of this layer
    LCU(cudaMemcpy2DAsync(L->h_init + (size_t)l * B * Hp, Hp * 4, h0 + (size_t)l * B * H, H * 4, H * 4, B, cudaMemcpyDeviceToDevice, st), "h0 copy");
    LCU(cudaMemcpy2DAsync(L->c_init + (size_t)l * B * Hp, Hp * 4, c0 + (size_t)l * B * H, H * 4, H * 4, B, cudaMemcpyDeviceToDevice, st), "c0 copy");
    lstm_init_hm_kernel<<<cell_blocks, 256, 0, st>>>(h0 + (size_t)l * B * H, done, B, H, Hp, L->hm[l]);
    { LGemmK::Params q{L->m_xin[l], L->m_Wih[l], L->gx, (int)N1, Hp / 64, G, 0, 0};      // input projection of every step
      LCU(igemm_tma_launch<LGemmK>(q, dim3(cdiv_(N1, 128), G / 64), st), "lstm gx gemm"); }
    for (int t = 0; t < T1; ++t) {
      { LGemmK::Params q{L->m_hm[l], L->m_Whh[l], L->r, B, Hp / 64, G, t * B, 0};
        LCU(igemm_tma_launch<LGemmK>(q, dim3(cdiv_(B, 128), G / 64), st), "lstm recurrent gemm"); }
      const float* cprev = t == 0 ? L->c_init + (size_t)l * B * Hp : L->cseq[l] + (size_t)(t - 1) * B * Hp;
      lstm_cell_fwd_kernel<<<cell_blocks, 256, 0, st>>>(
          L->gx + (size_t)t * B * G, L->r, L->w[l][2], L->w[l][3], cprev, done + (size_t)t * B, t + 1 < T1 ? done + (size_t)(t + 1) * B : nullptr, B, H, Hp,
          L->gates[l] + (size_t)t * B * G, L->cseq[l] + (size_t)t * B * Hp, L->hseq[l] + (size_t)t * B * Hp, L->hbf[l] + (size_t)t * B * Hp,
          t + 1 < T1 ? L->hm[l] + (size_t)(t + 1) * B * Hp : nullptr);
    }
    LCU(cudaGetLastError(), "lstm cell");
  }
  lstm_unpad_rows_kernel<<<cdiv_(N1 * H, 256), 256, 0, st>>>(L->hseq[1], (int)N1, H, Hp, out);
  for (int l = 0; l < 2; ++l) {
    if (hT) LCU(cudaMemcpy2DAsync(hT + (size_t)l * B * H, H * 4, L->hseq[l] + (size_t)(T1 - 1) * B * Hp, Hp * 4, H * 4, B, cudaMemcpyDeviceToDevice, st), "hT");
    if (cT) LCU(cudaMemcpy2DAsync(cT + (size_t)l * B * H, H * 4, L->cseq[l] + (size_t)(T1 - 1) * B * Hp, Hp * 4, H * 4, B, cudaMemcpyDeviceToDevice, st), "cT");
  }
  LCU(cudaGetLastError(), "lstm forward");
  return 0;
}

// dout fp32 [T*B][H] (gradient w.r.t. the LSTM output of steps 0..T-1) -> dcore fp32 [T*B][H]; weight/bias gradients are
// ACCUMULATED into the grads8 buffers given at creation.  Must follow srl_lstm_forward on the same inputs.
extern "C" int srl_lstm_backward(srl_lstm_t* L, const float* dout, const uint8_t* done, float* dcore, void* stream) {
  LREQ(L && dout && done && dcore, "lstm_backward: NULL pointer");
  cudaStream_t st = (cudaStream_t)stream;
  const int T = L->T1 - 1, B = L->B, H = L->H, Hp = L->Hp, G = L->G;
  const int64_t NB = (int64_t)T * B;
  const int cell_blocks = cdiv_((int64_t)B * Hp, 256);
  // dh_out of the top layer, padded to Hp (reuse dx as the padded buffer)
  LCU(cudaMemsetAsync(L->dx, 0, NB * Hp * 4, st), "zero dx");
  LCU(cudaMemcpy2DAsync(L->dx, Hp * 4, dout, H * 4, H * 4, NB, cudaMemcpyDeviceToDevice, st), "pad dout");
  for (int l = 1; l >= 0; --l) {
    LCU(cudaMemsetAsync(L->dc, 0, (size_t)B * Hp * 4, st), "zero dc");
    for (int t = T - 1; t >= 0; --t) {
      const float* cprev = t == 0 ? L->c_init + (size_t)l * B * Hp : L->cseq[l] + (size_t)(t - 1) * B * Hp;
      lstm_cell_bwd_kernel<<<cell_blocks, 256, 0, st>>>(
          L->dx + (size_t)t * B * Hp, t + 1 < T ? L->dhm : nullptr, done + (size_t)(t + 1) * B, L->gates[l] + (size_t)t * B * G,
          L->cseq[l] + (size_t)t * B * Hp, cprev, done + (size_t)t * B, L->dc, B, H, Hp, L->dgates[l] + (size_t)t * B * G);
      if (t > 0) {   // dhm_t = dgates_t . Whh  (gradient w.r.t. m_t . h_{t-1})
        LGemmK::Params q{L->m_dg128[l], L->m_WhhT[l], L->dhm, B, G / 64, Hp, t * B, 0};
        LCU(igemm_tma_launch<LGemmK>(q, dim3(cdiv_(B, 128), Hp / 64), st), "lstm bwd recurrent gemm");
      }
    }
    LCU(cudaGetLastError(), "lstm cell bwd");
    // weight gradients over all T*B rows (MN-major operands), then un-pad + accumulate
    { LGemmMN::Params q{L->m_dg64[l], L->m_xin64[l], L->dwpad, (int)NB, Hp};
      LCU(igemm_tma_launch<LGemmMN>(q, dim3(G / 128, Hp / 64), st), "lstm dWih gemm");
      lstm_unpad_w_kernel<<<cdiv_((int64_t)4 * H * H, 256), 256, 0, st>>>(L->dwpad, H, Hp, L->g[l][0]); }
    { LGemmMN::Params q{L->m_dg64[l], L->m_hm64[l], L->dwpad, (int)NB, Hp};
      LCU(igemm_tma_launch<LGemmMN>(q, dim3(G / 128, Hp / 64), st), "lstm dWhh gemm");
      lstm_unpad_w_kernel<<<cdiv_((int64_t)4 * H * H, 256), 256, 0, st>>>(L->dwpad, H, Hp, L->g[l][1]); }
    { const int rpb = 64;
      lstm_bias_grad_kernel<<<dim3(cdiv_(G, 128), cdiv_(NB, rpb)), 128, 0, st>>>(L->dgates[l], (int)NB, H, Hp, rpb, L->g[l][2], L->g[l][3]); }
    // gradient w.r.t. this layer's input = dh_out of the layer below (or dcore)
    { LGemmK::Params q{L->m_dg128[l], L->m_WihT[l], L->dx, (int)NB, G / 64, Hp, 0, 0};
      LCU(igemm_tma_launch<LGemmK>(q, dim3(cdiv_(NB, 128), Hp / 64), st), "lstm dx gemm"); }
  }
  lstm_unpad_rows_kernel<<<cdiv_(NB * H, 256), 256, 0, st>>>(L->dx, (int)NB, H, Hp, dcore);
  LCU(cudaGetLastError(), "lstm backward");
  return 0;
}
