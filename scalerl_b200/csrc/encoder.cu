// Encoder forward / backward drivers: weight packing + the sequence of tcgen05 implicit-GEMM launches.
#include "encoder_problems.cuh"
#include "tma_problems.cuh"
#include "res_problems.cuh"
#include "kernels.h"
#include <initializer_list>

namespace srl {

// fp32 master parameters (PyTorch layouts) -> bf16 operand copies in the layouts the GEMMs consume.
// One launch, three block roles (fc.weight is 96 % of the elements and is written twice -- K-major for the forward GEMM, transposed
// for dgrad -- so both copies go through a shared-memory tile: coalesced fp32 reads, >= 128-byte contiguous bf16 writes):
//   blocks [0, 256)    wfk[j][hw*64 + c] = Wfc[j][c*49 + hw]        two rows j per block
//   blocks [256, 512)  wfd[hw*64 + c][j] = Wfc[j][c*49 + hw]        tile = 64 j x 2 c (98 consecutive source columns)
//   blocks [512, 800)  the conv weight copies (147,456 elements), two elements per thread
constexpr int PACK_BLOCKS_FK = 256, PACK_BLOCKS_FD = 256, PACK_BLOCKS_CONV = 288;
SRL_DEVINL void pack_store(bf16* __restrict__ out, bf16* __restrict__ out_lo, int64_t i, float v) {
  const bf16 hi = __float2bfloat16_rn(v);
  out[i] = hi;
  if (out_lo) out_lo[i] = __float2bfloat16_rn(v - __bfloat162float(hi));     // fp32-accurate mode: w = hi + lo to 16 significant bits
}
SRL_DEVINL void pack_store2(bf16* __restrict__ out, bf16* __restrict__ out_lo, int64_t i, float v0, float v1) {      // i even
  const bf16 h0 = __float2bfloat16_rn(v0), h1 = __float2bfloat16_rn(v1);
  *reinterpret_cast<uint32_t*>(out + i) = pack_bf16x2(v0, v1);
  if (out_lo) *reinterpret_cast<uint32_t*>(out_lo + i) = pack_bf16x2(v0 - __bfloat162float(h0), v1 - __bfloat162float(h1));
}
__global__ void __launch_bounds__(256) pack_weights_kernel(ParamPtrs p, bf16* __restrict__ out, bf16* __restrict__ out_lo, int skip_w1k) {
  pdl_wait(2);     // (not launched with the attribute: returns at once; names the kernel in the diagnostics timeline)
  __shared__ __align__(16) float tile[64 * 99];                 // role 1: two fc rows (2 x 3136); role 2: [64 j][99]
  const int t = threadIdx.x, b = blockIdx.x;
  if (b < PACK_BLOCKS_FK) {
    const float4* src = reinterpret_cast<const float4*>(p.wf + (size_t)(2 * b) * 3136);       // rows 2b, 2b+1: 1568 float4, all loads in flight
    float4 v[7];
#pragma unroll
    for (int u = 0; u < 7; ++u) { const int q = t + 256 * u; if (q < 1568) v[u] = __ldg(src + q); }
#pragma unroll
    for (int u = 0; u < 7; ++u) { const int q = t + 256 * u; if (q < 1568) *reinterpret_cast<float4*>(tile + 4 * q) = v[u]; }
    __syncthreads();
#pragma unroll 4
    for (int pp = t; pp < 2 * 1568; pp += 256) {   // output pair: row r, k = 2 pp' = hw*64 + c
      const int r = pp >= 1568, k = 2 * (pp - r * 1568), hw = k >> 6, c = k & 63;
      const float* row = tile + r * 3136;
      pack_store2(out, out_lo, WPack::WFK + (int64_t)(2 * b + r) * 3136 + k, row[c * 49 + hw], row[(c + 1) * 49 + hw]);
    }
  } else if (b < PACK_BLOCKS_FK + PACK_BLOCKS_FD) {
    const int bb = b - PACK_BLOCKS_FK, j0 = (bb & 7) * 64, c0 = (bb >> 3) * 2;
    // 64 rows x 49 float2 (98 consecutive source columns c0*49 .. c0*49+97), all 13 loads of a thread in flight together
    float2 v[13];
#pragma unroll
    for (int u = 0; u < 13; ++u) {
      const int q = t + 256 * u, jj = q / 49, e = q - jj * 49;
      if (q < 64 * 49) v[u] = __ldg(reinterpret_cast<const float2*>(p.wf + (size_t)(j0 + jj) * 3136 + c0 * 49 + 2 * e));
    }
#pragma unroll
    for (int u = 0; u < 13; ++u) {
      const int q = t + 256 * u, jj = q / 49, e = q - jj * 49;
      if (q < 64 * 49) { tile[jj * 99 + 2 * e] = v[u].x; tile[jj * 99 + 2 * e + 1] = v[u].y; }
    }
    __syncthreads();
    const int lane = t & 31, warp = t >> 5;
    for (int kk = warp; kk < 98; kk += 8) {      // source column kk = cc*49 + hw -> destination row hw*64 + c0 + cc
      const int cc = kk >= 49, hw = kk - cc * 49;
      pack_store2(out, out_lo, WPack::WFD + (int64_t)(hw * 64 + c0 + cc) * 512 + j0 + 2 * lane, tile[(2 * lane) * 99 + kk], tile[(2 * lane + 1) * 99 + kk]);
    }
  } else {
    const int bb = b - PACK_BLOCKS_FK - PACK_BLOCKS_FD;
    constexpr int64_t NCONV = WPack::WFK + (WPack::TOTAL - WPack::W3D);       // the copies before and after the two fc blocks
    for (int64_t n = (int64_t)bb * 256 + t; n < NCONV; n += (int64_t)PACK_BLOCKS_CONV * 256) {
      const int64_t i = n < WPack::WFK ? n : n - WPack::WFK + WPack::W3D;
      float v;
      if (i < WPack::W2K) {                       // w1k[co][(kh2*2+kw2)*64 + c*16 + dy*4 + dx] = W1[co][c][4kh2+dy][4kw2+dx]
        if (skip_w1k) continue;                   // written by obs_s2d_kernel's extra blocks inside a step
        const int e = (int)(i - WPack::W1K), co = e >> 8, k = e & 255, tap = k >> 6, q = k & 63;
        const int c = q >> 4, dy = (q >> 2) & 3, dx = q & 3, kh = 4 * (tap >> 1) + dy, kw = 4 * (tap & 1) + dx;
        v = p.w1[co * 256 + c * 64 + kh * 8 + kw];
      } else if (i < WPack::W3K) {                // w2k[co][(kh*4+kw)*32 + c]
        const int e = (int)(i - WPack::W2K), co = e >> 9, k = e & 511, tap = k >> 5, c = k & 31;
        v = p.w2[((co * 32 + c) << 4) + tap];
      } else if (i < WPack::WFK) {                // w3k[co][(kh*3+kw)*64 + c]
        const int e = (int)(i - WPack::W3K), co = e / 576, k = e - co * 576, tap = k >> 6, c = k & 63;
        v = p.w3[(co * 64 + c) * 9 + tap];
      } else if (i < WPack::W2D) {                // w3d[c][(kh*3+kw)*64 + co]
        const int e = (int)(i - WPack::W3D), c = e / 576, k = e - c * 576, tap = k >> 6, co = k & 63;
        v = p.w3[(co * 64 + c) * 9 + tap];
      } else {                                    // w2d[cls][c][(kh'*2+kw')*64 + co], kh = ph + 2kh', kw = pw + 2kw'
        const int e = (int)(i - WPack::W2D), cls = e >> 13, r = e & 8191, c = r >> 8, k = r & 255, tt = k >> 6, co = k & 63;
        const int kh = (cls >> 1) + 2 * (tt >> 1), kw = (cls & 1) + 2 * (tt & 1);
        v = p.w2[((co * 32 + c) << 4) + kh * 4 + kw];
      }
      pack_store(out, out_lo, i, v);
    }
  }
}

// u8 NCHW frames -> space-to-depth bf16 NHWC: xs[n][Y][X][c*16+dy*4+dx] = obs[n][c][4Y+dy][4X+dx]  (exact: u8 fits bf16).
// One block per frame: the 16 x 21 source rows (c,dy) are read coalesced (21 u32 each, all 84 B of loads of a thread in flight
// together) into shared memory, then each thread converts u32 (4 x dx) -> 4 bf16 and the block writes 21 x 21 x 128 B contiguously.
__global__ void __launch_bounds__(352) obs_s2d_kernel(const uint8_t* __restrict__ obs, bf16* __restrict__ xs, int frame_blocks,
                                                      const float* __restrict__ w1, bf16* __restrict__ w1k, bf16* __restrict__ w1k_lo) {
  pdl_wait(1);     // launched with programmatic stream serialization: see common.cuh
  pdl_launch();
  if ((int)blockIdx.x >= frame_blocks) {
    // extra blocks: conv1's K-major weight copy w1k[co][(kh2*2+kw2)*64 + c*16 + dy*4 + dx] = W1[co][c][4kh2+dy][4kw2+dx] -- conv1 is the next kernel
    // of the stream, so it never has to wait for pack_weights_kernel (which skips this copy when the step launches it)
    const int e = ((int)blockIdx.x - frame_blocks) * 352 + (int)threadIdx.x;
    if (e < 32 * 256 && w1k) {
      const int co = e >> 8, k = e & 255, tap = k >> 6, q = k & 63;
      const int c = q >> 4, dy = (q >> 2) & 3, dx = q & 3, kh = 4 * (tap >> 1) + dy, kw = 4 * (tap & 1) + dx;
      pack_store(w1k, w1k_lo, e, __ldg(w1 + co * 256 + c * 64 + kh * 8 + kw));
    }
    return;
  }
  __shared__ uint32_t tile[21][16][21];
  const int n = blockIdx.x;
  const int t = threadIdx.x;
  if (t < 336) {
    const int g = t / 21, X = t - g * 21;      // g = (c, dy)
    const uint8_t* src = obs + (size_t)n * 28224 + (g >> 2) * 7056 + (g & 3) * 84;
#pragma unroll
    for (int y = 0; y < 21; ++y) tile[y][g][X] = __ldg(reinterpret_cast<const uint32_t*>(src + y * 336) + X);
  }
  __syncthreads();
  if (t < 336) {
    const int X = t >> 4, g = t & 15;
#pragma unroll
    for (int y = 0; y < 21; ++y) {
      const uint32_t w = tile[y][g][X];
      const float f0 = __uint_as_float(__byte_perm(w, 0x4B000000u, 0x7540)) - 8388608.f;
      const float f1 = __uint_as_float(__byte_perm(w, 0x4B000000u, 0x7541)) - 8388608.f;
      const float f2 = __uint_as_float(__byte_perm(w, 0x4B000000u, 0x7542)) - 8388608.f;
      const float f3 = __uint_as_float(__byte_perm(w, 0x4B000000u, 0x7543)) - 8388608.f;
      *reinterpret_cast<uint2*>(xs + (((size_t)n * 21 + y) * 21 + X) * 64 + g * 4) = make_uint2(pack_bf16x2(f0, f1), pack_bf16x2(f2, f3));
    }
  }
}

// a3 [n][hw][c] (NHWC rows, what conv3 writes and fc forward / dgrad consume) -> a3t [n][c*49 + hw], fc.weight's own column order:
// with a3t as its B operand the fc weight-gradient GEMM produces 64 CONSECUTIVE columns of dW per row (16-byte stores) instead of 64
// stores 196 B apart.  One frame per block through shared memory, 16-byte reads, 4-byte writes; runs on the wgrad side stream.
__global__ void __launch_bounds__(256) a3_transpose_kernel(const bf16* __restrict__ a3, bf16* __restrict__ a3t) {
  pdl_wait(53);
  __shared__ __align__(16) uint16_t tile[49 * 66];        // row hw: 64 channels + 2 pad (132 B pitch: conflict-free column reads)
  const int n = blockIdx.x, t = threadIdx.x;
  const uint4* src = reinterpret_cast<const uint4*>(a3 + (size_t)n * 3136);
  for (int q = t; q < 392; q += 256) {                    // 392 x 16 B: row hw = q >> 3, channels 8 (q & 7) ..
    const uint4 v = __ldg(src + q);
    uint32_t* d = reinterpret_cast<uint32_t*>(tile + (q >> 3) * 66 + (q & 7) * 8);
    d[0] = v.x; d[1] = v.y; d[2] = v.z; d[3] = v.w;
  }
  __syncthreads();
  uint32_t* dst = reinterpret_cast<uint32_t*>(a3t + (size_t)n * 3136);
  for (int pp = t; pp < 1568; pp += 256) {                // output pair o = 2 pp = c*49 + hw
    const int o = 2 * pp, c0 = o / 49, h0 = o - c0 * 49, o1 = o + 1, c1 = o1 / 49, h1 = o1 - c1 * 49;
    dst[pp] = (uint32_t)tile[h0 * 66 + c0] | ((uint32_t)tile[h1 * 66 + c1] << 16);
  }
}
SRL_KSTAMP_SETTER(kstamp_set_encoder)

cudaError_t launch_a3_transpose(const bf16* a3, bf16* a3t, int frames, cudaStream_t st) {
  if (frames <= 0) return cudaSuccess;
  a3_transpose_kernel<<<frames, 256, 0, st>>>(a3, a3t);
  return cudaGetLastError();
}

cudaError_t launch_pack_weights(const ParamPtrs& p, bf16* wpack, cudaStream_t st, bf16* wpack_lo, bool skip_w1k) {
  pack_weights_kernel<<<PACK_BLOCKS_FK + PACK_BLOCKS_FD + PACK_BLOCKS_CONV, 256, 0, st>>>(p, wpack, wpack_lo, skip_w1k ? 1 : 0);
  return cudaGetLastError();
}

#define SRL_TRY(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) return e_; } while (0)

static inline int cdiv(int a, int b) { return (a + b - 1) / b; }

// ------------------------------------------------------------------------------------------------
// tensor maps
// ------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* f = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(f);
  }
  return fn;
}

// bf16 tensor, dims innermost-first, strides in ELEMENTS for dims 1..rank-1, SWIZZLE_128B, zero OOB fill
bool make_map(CUtensorMap* m, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_elems, const uint32_t* box,
              bool swizzle64) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) return false;
  cuuint64_t gd[5], gs[4];
  cuuint32_t bx[5], es[5];
  for (int i = 0; i < rank; ++i) { gd[i] = dims[i]; bx[i] = box[i]; es[i] = 1; }
  for (int i = 0; i + 1 < rank; ++i) gs[i] = strides_elems[i] * 2;
  return fn(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank, const_cast<void*>(base), gd, gs, bx, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
            swizzle64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

cudaError_t build_tma_maps(const EncoderBuffers& b, int NF, int NB, TmaMaps* M, const char** why) {
  const uint64_t nf = NF, nb = NB;
  bool ok = true;
  auto mk = [&](CUtensorMap* m, const void* base, int rank, std::initializer_list<uint64_t> dims, std::initializer_list<uint64_t> strides,
                std::initializer_list<uint32_t> box, const char* name) {
    if (!ok) return;
    uint64_t d[5], s[4]; uint32_t bx[5];
    int i = 0; for (auto v : dims) d[i++] = v;
    i = 0; for (auto v : strides) s[i++] = v;
    i = 0; for (auto v : box) bx[i++] = v;
    if (!make_map(m, base, rank, d, s, bx)) { ok = false; if (why) *why = name; }
  };
  auto rows = [&](CUtensorMap* m, const void* base, uint64_t nrows, uint32_t boxrows, const char* name) {
    mk(m, base, 2, {64, nrows}, {64}, {64, boxrows}, name);
  };
  rows(&M->xs_w, b.xs, nf * 441, RConv1Fwd::WROWS, "xs_w");
  rows(&M->a1p0_w, b.a1, nf * 100, RConv2Fwd::WROWS, "a1p0_w");
  rows(&M->a1p1_w, b.a1 + (size_t)nf * 100 * 64, nf * 100, RConv2Fwd::WROWS, "a1p1_w");
  rows(&M->a2_w, b.a2, nf * 81, RConv3Fwd::WROWS, "a2_w");
  rows(&M->da3g_w, b.da3, nb * 81, RConv3Dgrad::WROWS, "da3g_w");
  rows(&M->da3g_b, b.da3, nb * 81, 128, "da3g_b");
  rows(&M->da2g_w, b.da2, nb * 100, RConv2Dgrad::WROWS, "da2g_w");
  rows(&M->da2g_b, b.da2, nb * 100, 128, "da2g_b");
  { const uint64_t d[2] = {32, nb * 441}, st_[1] = {32}; const uint32_t bx[2] = {32, 128};      // da1g: 32-channel rows (64 B), SWIZZLE_64B
    if (ok && !make_map(&M->da1g_b, b.da1, 2, d, st_, bx, true)) { ok = false; if (why) *why = "da1g_b"; } }
  static_assert(RConv1Wgrad::WROWS == RConv1Fwd::WROWS && RConv2Wgrad::WROWS == RConv2Fwd::WROWS && RConv3Wgrad::WROWS == RConv3Fwd::WROWS,
                "forward and wgrad share the window maps");
  mk(&M->a3m128, b.a3, 2, {3136, nf}, {3136}, {64, 128}, "a3m128");
  mk(&M->a3m64, b.a3, 2, {3136, nf}, {3136}, {64, 64}, "a3m64");
  if (b.a3t) mk(&M->a3tm64, b.a3t, 2, {3136, nf}, {3136}, {64, 64}, "a3tm64");
  mk(&M->dhm128, b.dh, 2, {512, nb}, {512}, {64, 128}, "dhm128");
  mk(&M->dhm64, b.dh, 2, {512, nb}, {512}, {64, 64}, "dhm64");
  const bf16* w = b.wpack;
  mk(&M->w1k, w + WPack::W1K, 2, {256, 32}, {256}, {64, 32}, "w1k");
  mk(&M->w2k, w + WPack::W2K, 2, {512, 64}, {512}, {64, 64}, "w2k");
  mk(&M->w3k, w + WPack::W3K, 2, {576, 64}, {576}, {64, 64}, "w3k");
  mk(&M->wfk, w + WPack::WFK, 2, {3136, 512}, {3136}, {64, 64}, "wfk");
  mk(&M->wfd, w + WPack::WFD, 2, {512, 3136}, {512}, {64, 64}, "wfd");
  mk(&M->w3d, w + WPack::W3D, 2, {576, 64}, {576}, {64, 64}, "w3d");
  mk(&M->w2d, w + WPack::W2D, 2, {256, 128}, {256}, {64, 128}, "w2d");
  M->valid = ok;
  if (!ok && why && !*why) *why = "cuTensorMapEncodeTiled unavailable";
  return ok ? cudaSuccess : cudaErrorInvalidValue;
}

cudaError_t build_tma_maps_lo(const EncoderBuffers& b, int NF, int NB, TmaMapsLo* M, const char** why) {
  const uint64_t nf = NF, nb = NB;
  bool ok = true;
  auto mk = [&](CUtensorMap* m, const void* base, std::initializer_list<uint64_t> dims, std::initializer_list<uint64_t> strides,
                std::initializer_list<uint32_t> box, const char* name) {
    if (!ok) return;
    uint64_t d[5], s[4]; uint32_t bx[5];
    int i = 0; for (auto v : dims) d[i++] = v;
    i = 0; for (auto v : strides) s[i++] = v;
    i = 0; for (auto v : box) bx[i++] = v;
    if (!make_map(m, base, 2, d, s, bx)) { ok = false; if (why) *why = name; }
  };
  auto rows = [&](CUtensorMap* m, const void* base, uint64_t nrows, uint32_t boxrows, const char* name) { mk(m, base, {64, nrows}, {64}, {64, boxrows}, name); };
  rows(&M->a1p0_w, b.a1_lo, nf * 100, RConv2Fwd::WROWS, "a1p0_w_lo");
  rows(&M->a1p1_w, b.a1_lo + (size_t)nf * 100 * 64, nf * 100, RConv2Fwd::WROWS, "a1p1_w_lo");
  rows(&M->a2_w, b.a2_lo, nf * 81, RConv3Fwd::WROWS, "a2_w_lo");
  rows(&M->da3g_w, b.da3_lo, nb * 81, RConv3Dgrad::WROWS, "da3g_w_lo");
  rows(&M->da3g_b, b.da3_lo, nb * 81, 128, "da3g_b_lo");
  rows(&M->da2g_w, b.da2_lo, nb * 100, RConv2Dgrad::WROWS, "da2g_w_lo");
  rows(&M->da2g_b, b.da2_lo, nb * 100, 128, "da2g_b_lo");
  { const uint64_t d[2] = {32, nb * 441}, st_[1] = {32}; const uint32_t bx[2] = {32, 128};
    if (ok && !make_map(&M->da1g_b, b.da1_lo, 2, d, st_, bx, true)) { ok = false; if (why) *why = "da1g_b_lo"; } }
  mk(&M->a3m128, b.a3_lo, {3136, nf}, {3136}, {64, 128}, "a3m128_lo");
  mk(&M->a3m64, b.a3_lo, {3136, nf}, {3136}, {64, 64}, "a3m64_lo");
  mk(&M->dhm128, b.dh_lo, {512, nb}, {512}, {64, 128}, "dhm128_lo");
  mk(&M->dhm64, b.dh_lo, {512, nb}, {512}, {64, 64}, "dhm64_lo");
  const bf16* w = b.wpack_lo;
  mk(&M->w1k, w + WPack::W1K, {256, 32}, {256}, {64, 32}, "w1k_lo");
  mk(&M->w2k, w + WPack::W2K, {512, 64}, {512}, {64, 64}, "w2k_lo");
  mk(&M->w3k, w + WPack::W3K, {576, 64}, {576}, {64, 64}, "w3k_lo");
  mk(&M->wfk, w + WPack::WFK, {3136, 512}, {3136}, {64, 64}, "wfk_lo");
  mk(&M->wfd, w + WPack::WFD, {512, 3136}, {512}, {64, 64}, "wfd_lo");
  mk(&M->w3d, w + WPack::W3D, {576, 64}, {576}, {64, 64}, "w3d_lo");
  mk(&M->w2d, w + WPack::W2D, {256, 128}, {256}, {64, 128}, "w2d_lo");
  M->valid = ok;
  return ok ? cudaSuccess : cudaErrorInvalidValue;
}

static cudaError_t launch_s2d(const uint8_t* obs, int frames, bf16* xs, cudaStream_t st, const float* w1, bf16* w1k, bf16* w1k_lo) {
  constexpr int WB = (32 * 256 + 351) / 352;      // extra blocks that write conv1's weight copy
  SRL_TRY(launch_chain<PDL_SIMT>(obs_s2d_kernel, dim3(frames + WB), dim3(352), 0, st, obs, xs, frames, w1, w1k, w1k_lo));
  return cudaGetLastError();
}

// persistent CTAs of the resident-window kernels: one per SM
constexpr int kPersistentCtas = 148;
// persistent CTAs of the backward chain's resident-window kernels (conv3 / conv2 dgrad, conv1 wgrad): fewer than one per SM leaves SMs to the
// lower-priority side-stream wgrads while the chain runs.  132 of 148: measured -1.5 us per step at T=20, B=32 (148: 0.1607, 132: 0.1591, 120: 0.1629 ms)
constexpr int kBwdCtas = 132;
// CTAs of the conv3 / conv2 weight-gradient kernels (side streams)
constexpr int kSideWgradCtas = 64;

// workspace [tap-block][row][co] -> PyTorch-layout conv weight gradients (plain stores), and re-zero what was read
__global__ void __launch_bounds__(256) conv_wgrad_finalize_kernel(float* __restrict__ ws, float* __restrict__ g1, float* __restrict__ g2,
                                                                  float* __restrict__ g3) {
  pdl_wait(51);    // launched with programmatic stream serialization: see common.cuh
  pdl_launch();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < 36864) {                       // dW3[co][c][tap] = ws3[tap>>1][(tap&1)*64 + c][co]
    const int co = i / 576, r = i - co * 576, c = r / 9, tap = r - c * 9;
    float* q = ws + WS_W3 + ((tap >> 1) * 128 + (tap & 1) * 64 + c) * 64 + co;
    g3[i] = *q; *q = 0.f;        // self-cleaning: the workspace is zero again for the next step
  } else if (i < 36864 + 32768) {        // dW2[co][c][kh][kw] = ws2[kh][kw*32 + c][co]
    const int e = i - 36864, co = e >> 9, r = e & 511, c = r >> 4, kh = (r >> 2) & 3, kw = r & 3;
    float* q = ws + WS_W2 + (kh * 128 + kw * 32 + c) * 64 + co;
    g2[e] = *q; *q = 0.f;
  } else if (i < 36864 + 32768 + 8192) { // dW1[co][c][kh][kw] = ws1[kh>>2][(kw>>2)*64 + c*16 + (kh&3)*4 + (kw&3)][co] / 255
    const int e = i - 36864 - 32768, co = e >> 8, k = e & 255, c = k >> 6, kh = (k >> 3) & 7, kw = k & 7;
    float* q = ws + WS_W1 + ((kh >> 2) * 128 + (kw >> 2) * 64 + c * 16 + (kh & 3) * 4 + (kw & 3)) * 32 + co;
    g1[e] = *q * (1.0f / 255.0f); *q = 0.f;
  }
}

cudaError_t encoder_forward(const uint8_t* obs, int frames, const ParamPtrs& p, const EncoderBuffers& buf, const TmaMaps& maps, int mode,
                            cudaStream_t st, const Profiler& pf, cudaEvent_t wait_before_conv1, const TmaMapsLo* lo) {
  if (frames <= 0) return cudaSuccess;
  if ((mode != 0 && mode != 1) || !maps.valid) return cudaErrorInvalidValue;
  const int sp = mode;                                    // 1: fp32-accurate split operands
  TmaMapsLo dummy;                                        // bf16 mode: the low maps are never touched by the kernels
  if (sp && (!lo || !lo->valid)) return cudaErrorInvalidValue;
  const TmaMapsLo& L = sp ? *lo : dummy;
  pf.b(PS_S2D); SRL_TRY(launch_s2d(obs, frames, buf.xs, st, p.w1, buf.wpack + WPack::W1K, sp ? buf.wpack_lo + WPack::W1K : nullptr)); pf.e(PS_S2D);
  { RConv1Fwd::Params q{maps.xs_w, maps.w1k, L.w1k, p.b1, buf.a1, buf.a1_lo, frames, buf.NF};
    pf.b(PS_CONV1_FWD); SRL_TRY(res_fwd_launch<RConv1Fwd>(q, cdiv(frames * 441, 128), 2 * kPersistentCtas, st, sp)); pf.e(PS_CONV1_FWD); }
  if (wait_before_conv1) SRL_TRY(cudaStreamWaitEvent(st, wait_before_conv1, 0));      // conv1's weight copy comes from the frame-conversion kernel; conv2 is the first reader of the re-packed copies
  { RConv2Fwd::Params q{maps.a1p0_w, maps.a1p1_w, maps.w2k, L.a1p0_w, L.a1p1_w, L.w2k, p.b2, buf.a2, buf.a2_lo, frames};
    pf.b(PS_CONV2_FWD); SRL_TRY(res_fwd_launch<RConv2Fwd>(q, cdiv(frames * 100, 128), kPersistentCtas, st, sp)); pf.e(PS_CONV2_FWD); }
  { RConv3Fwd::Params q{maps.a2_w, maps.w3k, L.a2_w, L.w3k, p.b3, buf.a3, buf.a3_lo, frames};
    pf.b(PS_CONV3_FWD); SRL_TRY(res_fwd_launch<RConv3Fwd>(q, cdiv(frames * 81, 128), kPersistentCtas, st, sp)); pf.e(PS_CONV3_FWD); }
  { TFcFwd::Params q{maps.a3m128, maps.wfk, L.a3m128, L.wfk, buf.hpart, frames};
    static_assert(TFcFwd::SPLITS == FC_SPLITS, "split count");
    pf.b(PS_FC_FWD);
    if (sp) SRL_TRY((igemm_tma_launch<TFcFwd, 1>(q, dim3(cdiv(frames, 128), 8 * FC_SPLITS), st)));
    else SRL_TRY((igemm_tma_launch<TFcFwd, 0>(q, dim3(cdiv(frames, 128), 8 * FC_SPLITS), st)));
    pf.e(PS_FC_FWD); }
  return cudaSuccess;
}

cudaError_t encoder_backward(const uint8_t* obs, int frames, const EncoderBuffers& buf, const ParamPtrs& g, const TmaMaps& maps, int mode,
                             cudaStream_t st, const Profiler& pf, const SideStream& ss, int phase, const TmaMapsLo* lo) {
  (void)obs;
  if (frames <= 0) return cudaSuccess;
  if ((mode != 0 && mode != 1) || !maps.valid) return cudaErrorInvalidValue;
  const int sp = mode;
  TmaMapsLo dummy;
  if (sp && (!lo || !lo->valid)) return cudaErrorInvalidValue;
  const TmaMapsLo& L = sp ? *lo : dummy;
  const bool do_fc = phase != 1, do_conv = phase != 0;
  // The wgrad GEMMs only feed the optimizer: each runs on its own side stream beside the dgrad chain
  // (dh -> da3 -> da2 -> da1) and beside each other.  With per-kernel profiling on everything stays on `st`.
  const bool fork = ss.side != nullptr && !pf.on;
  cudaStream_t s1 = fork ? ss.side : st, s2 = fork ? ss.side2 : st, s3 = fork ? ss.side3 : st;
  Profiler p1 = pf, p2 = pf, p3 = pf; p1.st = s1; p2.st = s2; p3.st = s3;
  if (do_fc) {
    if (fork) { SRL_TRY(cudaEventRecord(ss.ev[0], st)); SRL_TRY(cudaStreamWaitEvent(s1, ss.ev[0], 0)); }
    { const bool native = !sp && buf.a3t != nullptr;          // bf16 mode: B operand = a3 transposed into fc.weight's column order, 256-column tiles
      p1.b(PS_FC_WGRAD);
      if (native) {
        if (!buf.a3t_ready) SRL_TRY(launch_a3_transpose(buf.a3, buf.a3t, frames, s1));
        TFcWgradN::Params q{maps.dhm64, maps.a3tm64, g.wf, g.bf, frames};
        SRL_TRY((igemm_tma_launch<TFcWgradN, 0>(q, dim3(1, 4 * (TFcWgradN::NCT + 1)), s1)));
      } else {
        TFcWgrad::Params q{maps.dhm64, maps.a3m64, L.dhm64, L.a3m64, g.wf, g.bf, frames};
        if (sp) SRL_TRY((igemm_tma_launch<TFcWgrad, 1>(q, dim3(1, 4 * 50), s1))); else SRL_TRY((igemm_tma_launch<TFcWgrad, 0>(q, dim3(1, 4 * 50), s1)));
      }
      buf.a3t_ready = false;
      p1.e(PS_FC_WGRAD); }
    { TFcDgrad::Params q{maps.dhm128, maps.wfd, L.dhm128, L.wfd, buf.a3, buf.da3, buf.da3_lo, frames};
      pf.b(PS_FC_DGRAD);
      if (sp) SRL_TRY((igemm_tma_launch<TFcDgrad, 1>(q, dim3(cdiv(frames, 128), 49), st))); else SRL_TRY((igemm_tma_launch<TFcDgrad, 0>(q, dim3(cdiv(frames, 128), 49), st)));
      pf.e(PS_FC_DGRAD); }
    if (fork) { SRL_TRY(cudaEventRecord(ss.ev[4], s1)); }
    if (fork && !do_conv) { SRL_TRY(cudaStreamWaitEvent(st, ss.ev[4], 0)); }
  }
  if (!do_conv) return cudaSuccess;
  if (fork) { SRL_TRY(cudaEventRecord(ss.ev[1], st)); SRL_TRY(cudaStreamWaitEvent(s2, ss.ev[1], 0)); }
  { RConv3Wgrad::Params q{maps.a2_w, maps.da3g_b, L.a2_w, L.da3g_b, buf.wgrad_ws + WS_W3, g.b3, frames * 81, 0};
    p2.b(PS_CONV3_WGRAD); SRL_TRY(res_wgrad_launch<RConv3Wgrad>(q, kSideWgradCtas, s2, sp)); p2.e(PS_CONV3_WGRAD); }
  { RConv3Dgrad::Params q{maps.da3g_w, maps.w3d, L.da3g_w, L.w3d, buf.a2, buf.da2, buf.da2_lo, frames};
    pf.b(PS_CONV3_DGRAD); SRL_TRY(res_fwd_launch<RConv3Dgrad>(q, cdiv(frames * 81, 128), kBwdCtas, st, sp)); pf.e(PS_CONV3_DGRAD); }
  if (fork) { SRL_TRY(cudaEventRecord(ss.ev[2], st)); SRL_TRY(cudaStreamWaitEvent(s3, ss.ev[2], 0)); }
  { RConv2Wgrad::Params q{maps.a1p0_w, maps.a1p1_w, maps.da2g_b, L.a1p0_w, L.a1p1_w, L.da2g_b, buf.wgrad_ws + WS_W2, g.b2, frames * 100, 0};
    p3.b(PS_CONV2_WGRAD); SRL_TRY(res_wgrad_launch<RConv2Wgrad>(q, kSideWgradCtas, s3, sp)); p3.e(PS_CONV2_WGRAD); }
  { RConv2Dgrad::Params q{maps.da2g_w, maps.w2d, L.da2g_w, L.w2d, buf.a1, buf.da1, buf.da1_lo, frames, buf.NF};
    pf.b(PS_CONV2_DGRAD); SRL_TRY(res_fwd_launch<RConv2Dgrad>(q, cdiv(frames * 100, 128), kBwdCtas, st, sp)); pf.e(PS_CONV2_DGRAD); }
  { RConv1Wgrad::Params q{maps.xs_w, maps.da1g_b, L.da1g_b, buf.wgrad_ws + WS_W1, g.b1, frames * 441, 0};
    pf.b(PS_CONV1_WGRAD); SRL_TRY(res_wgrad_launch<RConv1Wgrad>(q, kBwdCtas, st, sp)); pf.e(PS_CONV1_WGRAD); }
  if (fork) {      // join: fc wgrad (phase 2 only: phase 1 was joined by the caller of phase 0), conv3 wgrad, conv2 wgrad
    if (do_fc) { SRL_TRY(cudaStreamWaitEvent(st, ss.ev[4], 0)); }
    SRL_TRY(cudaEventRecord(ss.ev[3], s2)); SRL_TRY(cudaStreamWaitEvent(st, ss.ev[3], 0));
    SRL_TRY(cudaEventRecord(ss.ev[7], s3)); SRL_TRY(cudaStreamWaitEvent(st, ss.ev[7], 0));
  }
  pf.b(PS_WGRAD_FINALIZE);
  SRL_TRY(launch_chain<PDL_SIMT>(conv_wgrad_finalize_kernel, dim3((36864 + 32768 + 8192 + 255) / 256), dim3(256), 0, st, buf.wgrad_ws, g.w1, g.w2, g.w3));
  SRL_TRY(cudaGetLastError());
  pf.e(PS_WGRAD_FINALIZE);
  return cudaSuccess;
}

}  // namespace srl
