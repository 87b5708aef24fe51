// Internal launch prototypes shared by the .cu translation units (not part of the C ABI).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>

namespace srl {

// per-kernel CUDA-event bracketing (bench.py's roofline numbers): slots of one learner step
enum ProfSlot { PS_S2D = 0, PS_CONV1_FWD, PS_CONV2_FWD, PS_CONV3_FWD, PS_FC_FWD, PS_HEAD_FWD, PS_TAIL, PS_ZERO_GRADS, PS_HEAD_BWD,
                PS_FC_WGRAD, PS_FC_DGRAD, PS_CONV3_WGRAD, PS_CONV3_DGRAD, PS_CONV2_WGRAD, PS_CONV2_DGRAD, PS_CONV1_WGRAD,
                PS_WGRAD_FINALIZE, PS_GRAD_NORM, PS_OPTIMIZER, PS_PACK, PS_COUNT };
struct Profiler {
  bool on = false;
  cudaEvent_t* ev = nullptr;   // 2 * PS_COUNT events
  cudaStream_t st = nullptr;
  void b(int slot) const { if (on) cudaEventRecord(ev[2 * slot], st); }
  void e(int slot) const { if (on) cudaEventRecord(ev[2 * slot + 1], st); }
};
// second stream + fork/join events: the wgrad GEMMs run beside the dgrad chain (also under stream capture)
// ---- programmatic dependent launch (see common.cuh) ----------------------------------------------------------
// pdl_active(): SRL_PDL != 0 (default on) and not switched off by the caller (per-kernel profiling records events between
// the kernels, which would serialise them anyway).
bool pdl_active();
void pdl_set_active(bool on);      // per calling thread: every C-ABI entry point sets it for the launches it makes
int pdl_skip_mask();      // SRL_PDL_MASK diagnostic: bit t set = kernels of class t launch without the attribute
enum { PDL_SIMT = 0, PDL_IGEMM = 1, PDL_RESFWD = 2, PDL_RESWGRAD = 3 };
template <int TAG, class... KA, class... A>
inline cudaError_t launch_chain(void (*kernel)(KA...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, A... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = (pdl_active() && !((pdl_skip_mask() >> TAG) & 1)) ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, args...);
}

// Per-DEVICE once flags (a process may drive several GPUs: function attributes and occupancy are per device).
struct PerDeviceOnce {
  bool done[64] = {};
  // returns the current device ordinal, or -1 on error; *first = true when this device has not been marked yet
  int device(bool* first) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) { *first = true; return -1; }
    *first = !done[dev];
    return dev;
  }
  void mark(int dev) { if (dev >= 0 && dev < 64) done[dev] = true; }
};
template <class K>
inline cudaError_t ensure_max_dynamic_smem(PerDeviceOnce& once, K kernel, int bytes) {
  bool first;
  const int dev = once.device(&first);
  if (!first) return cudaSuccess;
  cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e == cudaSuccess) once.mark(dev);
  return e;
}

void kstamp_set_encoder(unsigned long long*); void kstamp_set_vtrace(unsigned long long*); void kstamp_set_heads(unsigned long long*);   // diagnostics build (common.cuh)

struct SideStream {
  cudaStream_t side = nullptr;      // fc wgrad, weight re-pack
  cudaStream_t side2 = nullptr;     // conv3 wgrad
  cudaStream_t side3 = nullptr;     // conv2 wgrad
  cudaStream_t pack = nullptr;      // weight re-pack + gradient memset at the start of a step: HIGHEST priority (conv2 waits for it), unlike the wgrad streams
  cudaEvent_t ev[12] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
};

// conv weight-gradient workspace (fp32, the wgrad kernels' native [tap-block][row][co] order; res_problems.cuh), float offsets:
constexpr int WS_W3 = 0;                       // [5 acc][128 rows][64 co]   (tap 9 half unused)
constexpr int WS_W2 = WS_W3 + 5 * 128 * 64;    // [4 kh][128 rows][64 co]
constexpr int WS_W1 = WS_W2 + 4 * 128 * 64;    // [2 kh2][128 rows][32 co]
constexpr int WS_TOTAL = WS_W1 + 2 * 128 * 32;

// ---- vtrace.cu
cudaError_t launch_vtrace_iw(const float* log_rhos, const float* discounts, const float* rewards, const float* values,
                             const float* bootstrap, int T, int B, float clip_rho, float clip_pg, float* vs, float* pg, int variant,
                             cudaStream_t st);
cudaError_t launch_vtrace_logits(const float* bl, const float* tl, const int64_t* actions, const float* discounts, const float* rewards,
                                 const float* values, const float* bootstrap, int T, int B, int A, float clip_rho, float clip_pg,
                                 float* vs, float* pg, float* lr, float* balp, float* talp, cudaStream_t st);
cudaError_t launch_policy_rows_fwd(const float* logits, const int64_t* actions, int64_t N, int A, float* logp, float* ent, cudaStream_t st);
cudaError_t launch_policy_rows_bwd(const float* logits, const int64_t* actions, const float* w_logp, const float* w_ent, int64_t N, int A,
                                   float* dlogits, cudaStream_t st);
cudaError_t launch_sample_actions(const float* logits, const float* u, int64_t N, int A, int64_t* actions, cudaStream_t st);
cudaError_t launch_reduce_sum(const float* x, int64_t n, int square, float scale, float* out, cudaStream_t st);
bool column_step_supported(int T, int B, int A);
cudaError_t launch_column_step(const float* hpart, int nsplit, const float* bfc, float* h, const float* reward, const int64_t* action,
                               const uint8_t* done, const float* bl, const float* Wp, const float* bp, const float* Wb, const float* bb,
                               int T, int B, int A, float discounting, int clip_reward, float clip_rho, float clip_pg,
                               float baseline_cost, float entropy_cost, float* logits, float* baseline, float* vs, float* pg,
                               float* dlogits, float* dbaseline, __nv_bfloat16* dh, float* losses, float* scratch, cudaStream_t st,
                               __nv_bfloat16* dh_lo = nullptr);
cudaError_t launch_impala_tail(const float* bl, const float* tl, const float* baseline, const int64_t* action, const float* reward,
                               const uint8_t* done, int T, int B, int A, float discounting, int clip_reward, float clip_rho,
                               float clip_pg, float baseline_cost, float entropy_cost, float* vs, float* pg, float* dlogits,
                               float* dbaseline, float* losses, float* scratch, cudaStream_t st);

// ---- heads_optim.cu
// hpart: FC_SPLITS split-K partials [s][N][512] of the fc layer; writes h = relu(sum_s hpart + bfc) and the head outputs
cudaError_t launch_head_fwd(const float* hpart, int nsplit, const float* bfc, float* h, const float* reward, const int64_t* action,
                            const float* Wp, const float* bp, const float* Wb, const float* bb, int N, int A, float* logits,
                            float* baseline, cudaStream_t st);
cudaError_t launch_head_bwd(const float* dlogits, const float* dbaseline, const float* h, const float* reward, const int64_t* action,
                            const float* Wp, const float* Wb, int N, int A, __nv_bfloat16* dh, float* gWp, float* gbp, float* gWb,
                            float* gbb, cudaStream_t st, cudaStream_t st_wgrad, bool do_dh = true, __nv_bfloat16* dh_lo = nullptr);
cudaError_t launch_core_build(const float* hpart, int nsplit, const float* bfc, const float* reward, const int64_t* action, int N, int A, float* h,
                              float* core, cudaStream_t st);
cudaError_t launch_head_dense_fwd(const float* X, const float* Wp, const float* bp, const float* Wb, const float* bb, int N, int A, float* logits,
                                  float* baseline, cudaStream_t st);
cudaError_t launch_head_dense_bwd(const float* X, const float* dlogits, const float* dbaseline, const float* Wp, const float* Wb, int N, int A,
                                  float* dX, float* gWp, float* gbp, float* gWb, float* gbb, cudaStream_t st);
cudaError_t launch_dcore_to_dh(const float* dcore, const float* h, int N, int A, __nv_bfloat16* dh, cudaStream_t st);
cudaError_t launch_unpack_slots(const uint8_t* staging, int64_t slot_bytes, const int64_t* off6, int T, int B, int A, uint8_t* obs, float* reward,
                                uint8_t* done, int64_t* action, float* logits, float* episode_return, cudaStream_t st);
cudaError_t launch_clip_optim(int optimizer, float* p, float* g, float* s0, float* s1, int64_t n, float max_norm, float* coef,
                              float* scratch, float lr, float a, float b, float eps, int step, int* dstep, cudaStream_t st);
struct DpPeers { float* g[8]; float* rs[8]; unsigned* ctl[8]; int rank, world; float* mc_g; };      // peer-mapped gradient buffers / control blocks; mc_g: NVLS multicast address of the gradient buffers (or null)
cudaError_t launch_dp_clip_optim(int optimizer, float* p, float* g, float* s0, float* s1, int64_t n, float max_norm, float* coef,
                                 float* scratch, float lr, float a, float b, float eps, int step, int* dstep, const DpPeers& P,
                                 cudaStream_t st);
cudaError_t launch_snapshot_if_finite(float* dst, const float* src, int64_t n, const float* losses, cudaStream_t st);
cudaError_t launch_grad_norm(const float* g, int64_t n, float max_norm, float* coef, float* scratch, cudaStream_t st);
cudaError_t launch_rmsprop(float* p, const float* g, float* v, int64_t n, const float* coef, float lr, float alpha, float eps,
                           cudaStream_t st);
cudaError_t launch_adam(float* p, const float* g, float* m, float* v, int64_t n, const float* coef, float lr, float b1, float b2, float eps,
                        int step, int* dstep, cudaStream_t st);

// ---- encoder.cu
// packed bf16 operand copies of the conv/fc weights (element offsets into one buffer)
struct WPack {
  static constexpr int64_t W1K = 0;                       // [32][256]            k = (kh2,kw2,c,dy,dx), kh=4kh2+dy, kw=4kw2+dx
  static constexpr int64_t W2K = W1K + 32 * 256;          // [64][512]            k = (kh,kw,c)
  static constexpr int64_t W3K = W2K + 64 * 512;          // [64][576]            k = (kh,kw,c)
  static constexpr int64_t WFK = W3K + 64 * 576;          // [512][3136]          k = (hw,c)
  static constexpr int64_t WFD = WFK + 512 * 3136;        // [3136][512]          row = (hw,c), k = j
  static constexpr int64_t W3D = WFD + 3136 * 512;        // [64 c][576]          k = (kh,kw,co)
  static constexpr int64_t W2D = W3D + 64 * 576;          // [4 cls][32 c][256]   k = (kh',kw',co)
  static constexpr int64_t TOTAL = W2D + 4 * 32 * 256;
};
// pointers to the fp32 master tensors inside the flat parameter (or gradient) buffer
struct ParamPtrs {
  float *w1, *b1, *w2, *b2, *w3, *b3, *wf, *bf, *wp, *bp, *wb, *bb;
};
constexpr int FC_SPLITS = 4;
struct EncoderBuffers {   // row layouts: see res_problems.cuh
  __nv_bfloat16* xs;                    // space-to-depth bf16 copy of the u8 frames [NF*441][64], 64 = (c,dy,dx)
  __nv_bfloat16 *a1, *a2, *a3;          // a1 [2 planes][NF*100][64], a2 [NF*81][64], a3 [NF*49][64]
  mutable bool a3t_ready = false;       // the transpose below was already launched for this step (early, under the column kernel: api.cu encode_impl)
  __nv_bfloat16* a3t = nullptr;         // [NF][64*49]: a3 of the learning frames in fc.weight's own column order (c,h,w) -- fc wgrad's B operand (bf16 mode)
  float* hpart;                         // [FC_SPLITS][NF][512] split-K partials of the fc layer
  float* h;                             // [NF][512] fc output (post-ReLU), fp32
  __nv_bfloat16 *dh, *da3, *da2, *da1;  // dh [NB][512]; da3g [NB*81][64], da2g [NB*100][64], da1g [NB*441][32] (grid layouts, zero-padded)
  __nv_bfloat16* wpack;
  float* wgrad_ws;                      // conv weight-gradient accumulation workspace (res_problems.cuh: WS_TOTAL floats)
  int NF;                               // frames the forward buffers were sized for (plane stride of a1)
  // fp32-accurate operand mode (srl_config_t.precision = 1): the "low" twin bf16(v - bf16(v)) of every operand tensor above
  // (same layouts; nullptr in the bf16 mode).  xs has none: u8 frames are exact in bf16.
  __nv_bfloat16 *a1_lo = nullptr, *a2_lo = nullptr, *a3_lo = nullptr, *dh_lo = nullptr, *da3_lo = nullptr, *da2_lo = nullptr, *da1_lo = nullptr,
                *wpack_lo = nullptr;
};
// tensor maps of the TMA kernels (built once per learner context: every operand buffer is fixed).
// Activations are [rows][64] bf16; "w" = window box (128 + max tap shift rows), "b" = 128-row box.
struct TmaMaps {
  alignas(64) CUtensorMap xs_w, a1p0_w, a1p1_w, a2_w, da3g_w, da3g_b, da2g_w, da2g_b, da1g_b;      // conv layers (res_problems.cuh)
  alignas(64) CUtensorMap a3m128, a3m64, dhm128, dhm64;                                            // fc layer (tma_problems.cuh)
  alignas(64) CUtensorMap a3tm64;                                                                  // a3 in fc.weight's native column order (c,h,w): fc wgrad's B operand
  alignas(64) CUtensorMap w1k, w2k, w3k, wfk, wfd, w3d, w2d;
  bool valid = false;
};
struct TmaMapsLo {      // the same maps over the low tensors (built only in the fp32-accurate mode)
  alignas(64) CUtensorMap a1p0_w, a1p1_w, a2_w, da3g_w, da3g_b, da2g_w, da2g_b, da1g_b, a3m128, a3m64, dhm128, dhm64;
  alignas(64) CUtensorMap w1k, w2k, w3k, wfk, wfd, w3d, w2d;
  bool valid = false;
};
// bf16 tensor map, dims innermost-first, strides in ELEMENTS for dims 1..rank-1, SWIZZLE_128B, zero OOB fill (encoder.cu)
bool make_map(CUtensorMap* m, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_elems, const uint32_t* box, bool swizzle64 = false);
// returns cudaSuccess or an error; `why` gets a message on failure
cudaError_t build_tma_maps(const EncoderBuffers& buf, int NF, int NB, TmaMaps* maps, const char** why);
cudaError_t build_tma_maps_lo(const EncoderBuffers& buf, int NF, int NB, TmaMapsLo* maps, const char** why);
// wpack_lo != nullptr: also the low copies bf16(w - bf16(w)) in the same layouts
cudaError_t launch_a3_transpose(const __nv_bfloat16* a3, __nv_bfloat16* a3t, int frames, cudaStream_t st);
cudaError_t launch_pack_weights(const ParamPtrs& p, __nv_bfloat16* wpack, cudaStream_t st, __nv_bfloat16* wpack_lo = nullptr, bool skip_w1k = false);
// wait_before_conv1: optional event (weight re-pack running on the side stream) that conv1 must wait for
// mode: 0 = bf16 operands, 1 = fp32-accurate split operands (maps_lo must be valid)
cudaError_t encoder_forward(const uint8_t* obs, int frames, const ParamPtrs& p, const EncoderBuffers& buf, const TmaMaps& maps, int mode,
                            cudaStream_t st, const Profiler& pf, cudaEvent_t wait_before_conv1, const TmaMapsLo* maps_lo = nullptr);
// backward for the first `frames` frames given buf.dh; accumulates into the (pre-zeroed) gradient tensors in `g`
// phase: 0 = fc layer only (fc.weight / fc.bias gradients complete and joined to `st` on return: 95 % of the gradient
//        bytes, ready for an early all-reduce), 1 = conv layers only, 2 = both
cudaError_t encoder_backward(const uint8_t* obs, int frames, const EncoderBuffers& buf, const ParamPtrs& g, const TmaMaps& maps, int mode,
                             cudaStream_t st, const Profiler& pf, const SideStream& ss, int phase, const TmaMapsLo* maps_lo = nullptr);
cudaError_t test_shift(const void* A, const void* B, float* D, int shift, int mn_major, int bo_mode, cudaStream_t st);
cudaError_t test_poison_smem(cudaStream_t st);
cudaError_t test_mma_rate(int N, int shift, int reps, int issuers, long long* out, cudaStream_t st);
cudaError_t test_pdl(int* flag, int* out, int nblk, unsigned delay_ns, cudaStream_t st);
cudaError_t test_gemm(const void* A, const void* B, float* D, int M, int N, int K, bool mn_major, bool simt, cudaStream_t st);

}  // namespace srl
