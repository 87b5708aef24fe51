// extern "C" entry points (include/scalerl_b200.h).  Argument checking + the learner context that owns
// the activation workspaces and sequences the kernels of one learner step on the caller's stream.
#include <stdio.h>
#include <string.h>
#include <stdarg.h>
#include <new>

#include "../../include/scalerl_b200.h"
#include "kernels.h"

using namespace srl;

static thread_local char g_err[512] = "";

static int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}
static int cuda_fail(cudaError_t e, const char* what) {
  snprintf(g_err, sizeof(g_err), "%s: %s (%s)", what, cudaGetErrorName(e), cudaGetErrorString(e));
  return (int)e;
}
#define CU(x, what) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) return cuda_fail(e_, what); } while (0)
#define REQ(c, ...) do { if (!(c)) return fail(SRL_EINVAL, __VA_ARGS__); } while (0)

extern "C" const char* srl_last_error(void) { return g_err; }
extern "C" int srl_version(void) { return 100; }

// ------------------------------------------------------------------------------------------------
// stand-alone ops
// ------------------------------------------------------------------------------------------------
extern "C" int srl_vtrace_from_importance_weights(const float* log_rhos, const float* discounts, const float* rewards,
                                                  const float* values, const float* bootstrap_value, int T, int B,
                                                  float clip_rho, float clip_pg, float* vs, float* pg, int variant, void* stream) {
  REQ(T >= 0 && B >= 0, "vtrace: negative shape T=%d B=%d", T, B);
  if (T == 0 || B == 0) return 0;
  REQ(log_rhos && discounts && rewards && values && bootstrap_value && vs && pg, "vtrace: NULL pointer");
  CU(launch_vtrace_iw(log_rhos, discounts, rewards, values, bootstrap_value, T, B, clip_rho, clip_pg, vs, pg, variant,
                      (cudaStream_t)stream), "vtrace_from_importance_weights");
  return 0;
}

extern "C" int srl_vtrace_from_logits(const float* bl, const float* tl, const int64_t* actions, const float* discounts,
                                      const float* rewards, const float* values, const float* bootstrap_value, int T, int B, int A,
                                      float clip_rho, float clip_pg, float* vs, float* pg, float* log_rhos, float* balp, float* talp,
                                      void* stream) {
  REQ(T >= 0 && B >= 0 && A >= 1, "vtrace_from_logits: bad shape T=%d B=%d A=%d", T, B, A);
  if (T == 0 || B == 0) return 0;
  REQ(bl && tl && actions && discounts && rewards && values && bootstrap_value && vs && pg, "vtrace_from_logits: NULL pointer");
  CU(launch_vtrace_logits(bl, tl, actions, discounts, rewards, values, bootstrap_value, T, B, A, clip_rho, clip_pg, vs, pg, log_rhos,
                          balp, talp, (cudaStream_t)stream), "vtrace_from_logits");
  return 0;
}

extern "C" int srl_impala_loss_and_head_grads(const float* bl, const float* tl, const float* baseline, const int64_t* action,
                                              const float* reward, const uint8_t* done, int T, int B, int A, float discounting,
                                              int reward_clip_abs_one, float clip_rho, float clip_pg, float baseline_cost,
                                              float entropy_cost, float* vs, float* pg, float* dlogits, float* dbaseline, float* losses,
                                              float* scratch, void* stream) {
  REQ(T >= 1 && B >= 1 && A >= 1, "impala_loss: bad shape T=%d B=%d A=%d", T, B, A);
  REQ(bl && tl && baseline && action && reward && done && dlogits && dbaseline && losses && scratch, "impala_loss: NULL pointer");
  CU(launch_impala_tail(bl, tl, baseline, action, reward, done, T, B, A, discounting, reward_clip_abs_one, clip_rho, clip_pg,
                        baseline_cost, entropy_cost, vs, pg, dlogits, dbaseline, losses, scratch, (cudaStream_t)stream), "impala_tail");
  return 0;
}

extern "C" int srl_policy_rows_forward(const float* logits, const int64_t* actions, int64_t N, int A, float* logp, float* ent, void* stream) {
  REQ(N >= 0 && A >= 1, "policy_rows_forward: bad shape N=%lld A=%d", (long long)N, A);
  if (N == 0) return 0;
  REQ(logits && (logp || ent) && (!logp || actions), "policy_rows_forward: NULL pointer");
  CU(launch_policy_rows_fwd(logits, actions, N, A, logp, ent, (cudaStream_t)stream), "policy_rows_forward");
  return 0;
}
extern "C" int srl_policy_rows_backward(const float* logits, const int64_t* actions, const float* w_logp, const float* w_ent, int64_t N, int A,
                                        float* dlogits, void* stream) {
  REQ(N >= 0 && A >= 1, "policy_rows_backward: bad shape N=%lld A=%d", (long long)N, A);
  if (N == 0) return 0;
  REQ(logits && dlogits && (!w_logp || actions), "policy_rows_backward: NULL pointer");
  CU(launch_policy_rows_bwd(logits, actions, w_logp, w_ent, N, A, dlogits, (cudaStream_t)stream), "policy_rows_backward");
  return 0;
}
extern "C" int srl_sample_actions(const float* logits, const float* uniforms, int64_t N, int A, int64_t* actions, void* stream) {
  REQ(N >= 0 && A >= 1, "sample_actions: bad shape N=%lld A=%d", (long long)N, A);
  if (N == 0) return 0;
  REQ(logits && actions, "sample_actions: NULL pointer");
  CU(launch_sample_actions(logits, uniforms, N, A, actions, (cudaStream_t)stream), "sample_actions");
  return 0;
}
extern "C" int srl_reduce_sum(const float* x, int64_t n, int square, float scale, float* out, void* stream) {
  REQ(n >= 0 && out && (x || n == 0), "reduce_sum: bad argument");
  CU(launch_reduce_sum(x, n, square, scale, out, (cudaStream_t)stream), "reduce_sum");
  return 0;
}

extern "C" int srl_unpack_slots(const uint8_t* staging, int64_t slot_bytes, const int64_t* offsets6_host, int T, int B, int A, uint8_t* obs,
                                float* reward, uint8_t* done, int64_t* action, float* policy_logits, float* episode_return, void* stream) {
  REQ(staging && offsets6_host && obs && reward && done && action && policy_logits, "unpack_slots: NULL pointer");
  REQ(T >= 1 && B >= 1 && A >= 1 && A <= 32 && slot_bytes > 0, "unpack_slots: bad shape");
  REQ((slot_bytes & 15) == 0 && (offsets6_host[0] & 15) == 0 && (reinterpret_cast<uintptr_t>(staging) & 15) == 0 &&
      (reinterpret_cast<uintptr_t>(obs) & 15) == 0, "unpack_slots: obs record and buffers must be 16-byte aligned");
  CU(launch_unpack_slots(staging, slot_bytes, offsets6_host, T, B, A, obs, reward, done, action, policy_logits, episode_return,
                         (cudaStream_t)stream), "unpack_slots");
  return 0;
}

extern "C" int srl_grad_norm_clip_coef(const float* grads, int64_t n, float max_norm, float* coef, float* scratch, void* stream) {
  REQ(grads && coef && scratch && n >= 0, "grad_norm: bad argument");
  REQ((reinterpret_cast<uintptr_t>(grads) & 15) == 0, "grad_norm: grads must be 16-byte aligned");
  CU(launch_grad_norm(grads, n, max_norm, coef, scratch, (cudaStream_t)stream), "grad_norm");
  return 0;
}
extern "C" int srl_rmsprop_step(float* params, const float* grads, float* square_avg, int64_t n, const float* coef, float lr, float alpha,
                                float eps, void* stream) {
  REQ(params && grads && square_avg && n >= 0, "rmsprop: bad argument");
  REQ(((reinterpret_cast<uintptr_t>(params) | reinterpret_cast<uintptr_t>(grads) | reinterpret_cast<uintptr_t>(square_avg)) & 15) == 0,
      "rmsprop: buffers must be 16-byte aligned");
  CU(launch_rmsprop(params, grads, square_avg, n, coef, lr, alpha, eps, (cudaStream_t)stream), "rmsprop");
  return 0;
}
extern "C" int srl_adam_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, int64_t n, const float* coef, float lr,
                             float beta1, float beta2, float eps, int step, void* stream) {
  REQ(params && grads && exp_avg && exp_avg_sq && n >= 0 && step >= 1, "adam: bad argument");
  CU(launch_adam(params, grads, exp_avg, exp_avg_sq, n, coef, lr, beta1, beta2, eps, step, nullptr, (cudaStream_t)stream), "adam");
  return 0;
}

// ------------------------------------------------------------------------------------------------
// parameter layout
// ------------------------------------------------------------------------------------------------
// Flat buffer order: every small tensor first (conv1..3, fc.bias, heads), fc.weight LAST.  The small block is one
// contiguous range (one memset, one late all-reduce); fc.weight (95 % of the bytes) is final early in the backward pass
// and can be all-reduced while the conv layers are still back-propagating.  off/cnt are indexed in state_dict order.
static int64_t layout_ex(int A, int use_lstm, int64_t* off, int64_t* cnt) {
  const int64_t core = 513 + A;
  const int64_t counts[20] = {32 * 256, 32, 64 * 512, 64, 64 * 576, 64, 512 * 3136, 512, A * core, A, core, 1,
                              4 * core * core, 4 * core * core, 4 * core, 4 * core, 4 * core * core, 4 * core * core, 4 * core, 4 * core};
  const int order[20] = {0, 1, 2, 3, 4, 5, 7, 8, 9, 10, 11, 6, 12, 13, 14, 15, 16, 17, 18, 19};
  int64_t o = 0;
  const int n = use_lstm ? 20 : 12;
  for (int k = 0; k < 20; ++k) {
    const int i = order[k];
    if (k >= n) { if (off) off[i] = o; if (cnt) cnt[i] = 0; continue; }
    if (off) off[i] = o;
    if (cnt) cnt[i] = counts[i];
    o += (counts[i] + 3) & ~int64_t(3);
  }
  return o;
}
static int64_t layout(int A, int64_t* off, int64_t* cnt) {
  int64_t o20[20], c20[20];
  const int64_t total = layout_ex(A, 0, o20, c20);
  for (int i = 0; i < 12; ++i) { if (off) off[i] = o20[i]; if (cnt) cnt[i] = c20[i]; }
  return total;
}
extern "C" int64_t srl_param_layout(int A, int64_t* offsets, int64_t* counts) { return layout(A, offsets, counts); }
extern "C" int64_t srl_param_layout_ex(int A, int use_lstm, int64_t* offsets20, int64_t* counts20) { return layout_ex(A, use_lstm, offsets20, counts20); }

static ParamPtrs make_ptrs(float* base, int A) {
  int64_t off[12];
  layout(A, off, nullptr);
  ParamPtrs p;
  p.w1 = base + off[0]; p.b1 = base + off[1]; p.w2 = base + off[2]; p.b2 = base + off[3]; p.w3 = base + off[4]; p.b3 = base + off[5];
  p.wf = base + off[6]; p.bf = base + off[7]; p.wp = base + off[8]; p.bp = base + off[9]; p.wb = base + off[10]; p.bb = base + off[11];
  return p;
}

// ------------------------------------------------------------------------------------------------
// learner context
// ------------------------------------------------------------------------------------------------
struct srl_learner {
  srl_config_t cfg;
  float *params, *grads, *opt0, *opt1;
  int64_t nparams;
  ParamPtrs P, G;
  EncoderBuffers buf;
  float *logits, *baseline;       // [NF][A], [NF]
  float *dlogits, *dbaseline;     // [NB][A], [NB]
  float *scratch;                 // reductions (tail + grad norm)
  float *coef;                    // {norm, clip coef}
  char* arena;
  int64_t arena_bytes;
  int step;                       // optimizer step count (Adam bias correction)
  bool have_fwd;
  TmaMaps maps;                   // tensor maps of the TMA mainloop
  TmaMapsLo maps_lo;              // ... over the low operand tensors (precision = 1 only)
  char* lo_arena;
  SideStream ss;                  // wgrad side stream + fork/join events
  int* dstep;                     // device-side optimizer step count (graph-replay safe Adam bias correction)
  srl_lstm_t* lstm;               // use_lstm: the 2-layer LSTM core (csrc/lstm.cu) working on views of params/grads
  float *core, *lstm_out, *dout, *dcore;   // [NF][H], [NF][H], [NB][H], [NB][H]
  char* lstm_arena;
  int64_t lstm_off0, lstm_len;    // LSTM gradient range inside the flat buffer
  bool column_fusion;             // heads + V-trace/loss + dh in one column kernel (SRL_NO_COLUMN_FUSION / srl_learner_set_option)
  Profiler pf;                    // per-kernel event bracketing (off by default)
  cudaEvent_t events[2 * PS_COUNT];
  bool slot_used[PS_COUNT];
};

static const char* kSlotNames[PS_COUNT] = {"obs_s2d", "conv1_fwd", "conv2_fwd", "conv3_fwd", "fc_fwd", "head_fwd", "vtrace_loss_tail",
                                           "zero_grads", "head_bwd", "fc_wgrad", "fc_dgrad", "conv3_wgrad", "conv3_dgrad", "conv2_wgrad",
                                           "conv2_dgrad", "conv1_wgrad", "conv_wgrad_finalize", "grad_norm", "optimizer", "pack_weights"};

static int check_cfg(const srl_config_t* c) {
  REQ(c, "config is NULL");
  REQ(c->T >= 1 && c->B >= 1, "config: T=%d B=%d must be >= 1", c->T, c->B);
  REQ(c->A >= 1 && c->A <= 31, "config: A=%d must be in [1,31] (one warp lane per action plus one for the baseline)", c->A);
  REQ((int64_t)(c->T + 1) * c->B <= 65536, "config: (T+1)*B=%lld frames per GPU exceeds 65536", (long long)(c->T + 1) * c->B);
  REQ(c->optimizer == 0 || c->optimizer == 1, "config: optimizer must be 0 (rmsprop) or 1 (adam)");
  REQ(c->use_lstm == 0 || c->use_lstm == 1, "config: use_lstm must be 0 or 1");
  REQ(c->precision == 0 || c->precision == 1, "config: precision must be 0 (bf16 operands) or 1 (fp32-accurate split operands)");
  REQ(!(c->precision == 1 && c->use_lstm), "config: the fp32-accurate operand mode covers the non-LSTM learner only");
  return 0;
}

extern "C" int srl_learner_create(const srl_config_t* cfg, float* params, float* grads, float* opt0, float* opt1, srl_learner_t** out) {
  int rc = check_cfg(cfg);
  if (rc) return rc;
  REQ(params && grads && opt0 && out, "learner_create: NULL buffer");
  REQ(cfg->optimizer == 0 || opt1, "learner_create: Adam needs opt_state1");
  REQ(((reinterpret_cast<uintptr_t>(params) | reinterpret_cast<uintptr_t>(grads) | reinterpret_cast<uintptr_t>(opt0) |
        reinterpret_cast<uintptr_t>(opt1)) & 15) == 0, "learner_create: flat buffers must be 16-byte aligned");
  srl_learner* L = new (std::nothrow) srl_learner();
  REQ(L, "out of host memory");
  L->cfg = *cfg; L->params = params; L->grads = grads; L->opt0 = opt0; L->opt1 = opt1;
  L->nparams = layout_ex(cfg->A, cfg->use_lstm, nullptr, nullptr);
  L->lo_arena = nullptr;
  L->lstm = nullptr; L->lstm_arena = nullptr; L->core = L->lstm_out = L->dout = L->dcore = nullptr; L->lstm_off0 = L->lstm_len = 0;
  L->P = make_ptrs(params, cfg->A);
  L->G = make_ptrs(grads, cfg->A);
  L->step = 0; L->have_fwd = false;
  { const char* nf = getenv("SRL_NO_COLUMN_FUSION"); L->column_fusion = !(nf && atoi(nf) != 0); }   // read once, at creation
  for (int i = 0; i < 2 * PS_COUNT; ++i) L->events[i] = nullptr;
  for (int i = 0; i < PS_COUNT; ++i) L->slot_used[i] = false;
  const int64_t NF = (int64_t)(cfg->T + 1) * cfg->B, NB = (int64_t)cfg->T * cfg->B, A = cfg->A;
  // carve one arena (256-byte aligned pieces)
  int64_t sizes[24]; int k = 0;
  auto al = [](int64_t b) { return (b + 255) & ~int64_t(255); };
  sizes[k++] = al(NF * 441 * 64 * 2);   // xs
  sizes[k++] = al((int64_t)FC_SPLITS * NF * 512 * 4);   // hpart
  sizes[k++] = al(NF * 400 * 32 * 2);   // a1
  sizes[k++] = al(NF * 81 * 64 * 2);    // a2
  sizes[k++] = al(NF * 49 * 64 * 2);    // a3
  sizes[k++] = al(NF * 512 * 4);        // h
  sizes[k++] = al(NB * 512 * 2);        // dh
  sizes[k++] = al(NB * 81 * 64 * 2);    // da3g (9x9 grid)
  sizes[k++] = al(NB * 100 * 64 * 2);   // da2g (10x10 grid)
  sizes[k++] = al(NB * 441 * 32 * 2);   // da1g (21x21 grid, 32 channels)
  sizes[k++] = al(WPack::TOTAL * 2);    // wpack
  sizes[k++] = al(NF * A * 4);          // logits
  sizes[k++] = al(NF * 4);              // baseline
  sizes[k++] = al(NB * A * 4);          // dlogits
  sizes[k++] = al(NB * 4);              // dbaseline
  sizes[k++] = al(4096 * 4);            // scratch
  sizes[k++] = al(16);                  // coef
  sizes[k++] = al(16);                  // dstep
  sizes[k++] = al(81920 * 4);           // conv wgrad workspace (res_problems.cuh WS_TOTAL = 81920 floats)
  sizes[k++] = al(NF * 3136 * 2);       // a3t
  int64_t total = 0;
  for (int i = 0; i < k; ++i) total += sizes[i];
  cudaError_t e = cudaMalloc(&L->arena, total);
  if (e != cudaSuccess) { delete L; return cuda_fail(e, "learner_create: cudaMalloc workspace"); }
  e = cudaMemset(L->arena, 0, total);
  if (e != cudaSuccess) { cudaFree(L->arena); delete L; return cuda_fail(e, "learner_create: cudaMemset"); }
  L->arena_bytes = total;
  char* q = L->arena; int i = 0;
  L->buf.xs = (__nv_bfloat16*)q; q += sizes[i++];
  L->buf.hpart = (float*)q; q += sizes[i++];
  L->buf.a1 = (__nv_bfloat16*)q; q += sizes[i++];
  L->buf.a2 = (__nv_bfloat16*)q; q += sizes[i++];
  L->buf.a3 = (__nv_bfloat16*)q; q += sizes[i++];
  L->buf.h = (float*)q; q += sizes[i++];
  L->buf.dh = (__nv_bfloat16*)q; q += sizes[i++];
  L->buf.da3 = (__nv_bfloat16*)q; q += sizes[i++];
  L->buf.da2 = (__nv_bfloat16*)q; q += sizes[i++];
  L->buf.da1 = (__nv_bfloat16*)q; q += sizes[i++];
  L->buf.wpack = (__nv_bfloat16*)q; q += sizes[i++];
  L->buf.NF = (int)NF;
  L->logits = (float*)q; q += sizes[i++];
  L->baseline = (float*)q; q += sizes[i++];
  L->dlogits = (float*)q; q += sizes[i++];
  L->dbaseline = (float*)q; q += sizes[i++];
  L->scratch = (float*)q; q += sizes[i++];
  L->coef = (float*)q; q += sizes[i++];
  L->dstep = (int*)q; q += sizes[i++];
  L->buf.wgrad_ws = (float*)q; q += sizes[i++];
  L->buf.a3t = (__nv_bfloat16*)q; q += sizes[i++];
  if (cudaStreamCreateWithFlags(&L->ss.side, cudaStreamNonBlocking) != cudaSuccess ||
      cudaStreamCreateWithFlags(&L->ss.side2, cudaStreamNonBlocking) != cudaSuccess ||
      cudaStreamCreateWithFlags(&L->ss.side3, cudaStreamNonBlocking) != cudaSuccess) L->ss.side = nullptr;
  {
    // the re-pack stream sits one level BELOW the greatest priority (which the learner's capture stream uses for the main chain) and above the
    // wgrad streams (default = least): its short blocks fill the slots the frame conversion leaves free without delaying it
    int lo = 0, hi = 0;       // (numerically lowest = greatest priority)
    if (L->ss.side && (cudaDeviceGetStreamPriorityRange(&lo, &hi) != cudaSuccess ||
                       cudaStreamCreateWithPriority(&L->ss.pack, cudaStreamNonBlocking, hi + 1 > lo ? lo : hi + 1) != cudaSuccess)) L->ss.side = nullptr;
  }
  for (int e2 = 0; e2 < 12 && L->ss.side; ++e2)
    if (cudaEventCreateWithFlags(&L->ss.ev[e2], cudaEventDisableTiming) != cudaSuccess) { L->ss.side = nullptr; }
  cudaGetLastError();
  if (cfg->precision == 1) {      // low twins of every bf16 operand tensor (same layouts), zero-initialised like the originals
    const int64_t lo_sizes[8] = {al(NF * 400 * 32 * 2), al(NF * 81 * 64 * 2), al(NF * 49 * 64 * 2), al(NB * 512 * 2), al(NB * 81 * 64 * 2),
                                 al(NB * 100 * 64 * 2), al(NB * 441 * 32 * 2), al(WPack::TOTAL * 2)};
    int64_t lo_total = 0;
    for (int j = 0; j < 8; ++j) lo_total += lo_sizes[j];
    if (cudaMalloc(&L->lo_arena, lo_total) != cudaSuccess || cudaMemset(L->lo_arena, 0, lo_total) != cudaSuccess) {
      if (L->lo_arena) cudaFree(L->lo_arena);
      cudaFree(L->arena); delete L;
      return fail(SRL_ESTATE, "learner_create: cudaMalloc of the low operand tensors failed");
    }
    L->arena_bytes += lo_total;
    char* ql = L->lo_arena; int j = 0;
    L->buf.a1_lo = (__nv_bfloat16*)ql; ql += lo_sizes[j++];
    L->buf.a2_lo = (__nv_bfloat16*)ql; ql += lo_sizes[j++];
    L->buf.a3_lo = (__nv_bfloat16*)ql; ql += lo_sizes[j++];
    L->buf.dh_lo = (__nv_bfloat16*)ql; ql += lo_sizes[j++];
    L->buf.da3_lo = (__nv_bfloat16*)ql; ql += lo_sizes[j++];
    L->buf.da2_lo = (__nv_bfloat16*)ql; ql += lo_sizes[j++];
    L->buf.da1_lo = (__nv_bfloat16*)ql; ql += lo_sizes[j++];
    L->buf.wpack_lo = (__nv_bfloat16*)ql; ql += lo_sizes[j++];
  }
  {
    const char* why = nullptr;
    if (build_tma_maps(L->buf, (int)NF, (int)NB, &L->maps, &why) != cudaSuccess ||
        (cfg->precision == 1 && build_tma_maps_lo(L->buf, (int)NF, (int)NB, &L->maps_lo, &why) != cudaSuccess)) {
      if (L->lo_arena) cudaFree(L->lo_arena);
      cudaFree(L->arena);
      delete L;
      return fail(SRL_ESTATE, "learner_create: building TMA tensor map '%s' failed (driver without cuTensorMapEncodeTiled?)", why ? why : "?");
    }
  }
  if (cfg->use_lstm) {
    int64_t off[20], cnt[20];
    const int64_t total_p = layout_ex(cfg->A, 1, off, cnt);
    const int H = 513 + cfg->A;
    const float* wp[8]; float* gp[8];
    for (int i = 0; i < 8; ++i) { wp[i] = params + off[12 + i]; gp[i] = grads + off[12 + i]; }
    L->lstm_off0 = off[12]; L->lstm_len = total_p - off[12];
    const int64_t bytes = ((NF + NF + NB + NB) * (int64_t)H * 4 + 1024);
    bool ok = cudaMalloc(&L->lstm_arena, bytes) == cudaSuccess && cudaMemset(L->lstm_arena, 0, bytes) == cudaSuccess;
    if (ok) {
      float* q2 = (float*)L->lstm_arena;
      L->core = q2; q2 += NF * H; L->lstm_out = q2; q2 += NF * H; L->dout = q2; q2 += NB * H; L->dcore = q2;
      ok = srl_lstm_create(cfg->T + 1, cfg->B, H, wp, gp, &L->lstm) == 0;
    }
    if (!ok) {
      if (L->lstm_arena) cudaFree(L->lstm_arena);
      cudaFree(L->arena);
      delete L;
      return fail(SRL_ESTATE, "learner_create: LSTM core allocation failed: %s", srl_lstm_last_error());
    }
  }
  *out = L;
  return 0;
}

extern "C" int srl_learner_destroy(srl_learner_t* L) {
  if (!L) return 0;
  for (int i = 0; i < 2 * PS_COUNT; ++i) if (L->events[i]) cudaEventDestroy(L->events[i]);
  for (int i = 0; i < 12; ++i) if (L->ss.ev[i]) cudaEventDestroy(L->ss.ev[i]);
  if (L->ss.side) cudaStreamDestroy(L->ss.side);
  if (L->ss.side2) cudaStreamDestroy(L->ss.side2);
  if (L->ss.side3) cudaStreamDestroy(L->ss.side3);
  if (L->ss.pack) cudaStreamDestroy(L->ss.pack);
  if (L->lstm) srl_lstm_destroy(L->lstm);
  if (L->lstm_arena) cudaFree(L->lstm_arena);
  if (L->lo_arena) cudaFree(L->lo_arena);
  cudaFree(L->arena);
  delete L;
  return 0;
}
extern "C" int srl_debug_kernel_timeline(void* buffer) {
#ifdef SRL_KSTAMP
  kstamp_set_encoder((unsigned long long*)buffer); kstamp_set_vtrace((unsigned long long*)buffer); kstamp_set_heads((unsigned long long*)buffer);
  cudaError_t e = cudaDeviceSynchronize();
  return e == cudaSuccess ? 0 : cuda_fail(e, "debug_kernel_timeline");
#else
  (void)buffer;
  return fail(SRL_ESTATE, "debug_kernel_timeline: this library was not built with SRL_DEFINES=SRL_KSTAMP");
#endif
}

extern "C" int64_t srl_learner_workspace_bytes(const srl_learner_t* L) { return L ? L->arena_bytes : 0; }

extern "C" int srl_learner_set_config(srl_learner_t* L, const srl_config_t* cfg) {
  REQ(L, "learner is NULL");
  int rc = check_cfg(cfg);
  if (rc) return rc;
  REQ(cfg->T == L->cfg.T && cfg->B == L->cfg.B && cfg->A == L->cfg.A && cfg->optimizer == L->cfg.optimizer &&
      cfg->precision == L->cfg.precision && cfg->use_lstm == L->cfg.use_lstm, "set_config: T/B/A/optimizer/precision/use_lstm are fixed at creation");
  L->cfg = *cfg;
  return 0;
}

extern "C" int srl_learner_set_option(srl_learner_t* L, const char* name, int value) {
  REQ(L && name, "set_option: NULL argument");
  if (strcmp(name, "column_fusion") == 0) { L->column_fusion = value != 0; return 0; }
  return fail(SRL_EINVAL, "set_option: unknown option '%s'", name);
}

extern "C" int srl_learner_set_step(srl_learner_t* L, int64_t step, void* stream) {
  REQ(L && step >= 0 && step < (int64_t(1) << 31), "set_step: bad argument");
  L->step = (int)step;
  const int v = (int)step;       // the device counter drives Adam's bias correction under graph replay
  CU(cudaMemcpyAsync(L->dstep, &v, sizeof(int), cudaMemcpyHostToDevice, (cudaStream_t)stream), "set_step");
  CU(cudaStreamSynchronize((cudaStream_t)stream), "set_step");      // `v` is a stack variable
  return 0;
}
extern "C" int64_t srl_learner_get_step(srl_learner_t* L, void* stream) {
  if (!L) return -1;
  int v = 0;
  if (cudaMemcpyAsync(&v, L->dstep, sizeof(int), cudaMemcpyDeviceToHost, (cudaStream_t)stream) != cudaSuccess) return -1;
  if (cudaStreamSynchronize((cudaStream_t)stream) != cudaSuccess) return -1;
  return v;
}

extern "C" int srl_learner_pack_weights(srl_learner_t* L, void* stream) {
  REQ(L, "learner is NULL");
  CU(launch_pack_weights(L->P, L->buf.wpack, (cudaStream_t)stream, L->buf.wpack_lo), "pack_weights");
  return 0;
}

namespace srl {
static thread_local bool g_pdl_on = true;      // per calling thread: two learners driven from two threads do not race on it
bool pdl_active() {
  static const bool env_on = [] { const char* e = getenv("SRL_PDL"); return !e || atoi(e) != 0; }();
  return env_on && g_pdl_on;
}
void pdl_set_active(bool on) { g_pdl_on = on; }
int pdl_skip_mask() {
  static const int m = [] { const char* e = getenv("SRL_PDL_MASK"); return e ? atoi(e) : 0; }();
  return m;
}
}  // namespace srl

static int encode_impl(srl_learner* L, const uint8_t* obs, int frames, cudaStream_t st, bool zero_small_grads = false) {
  // zero_small_grads: true when called from the learner step (forward + backward)
  L->pf.st = st;
  pdl_set_active(!L->pf.on);
  // The bf16 operand copies are re-derived from the fp32 master weights at the START of every forward (not at the end
  // of the optimizer step): the pack kernel runs on the side stream underneath the frame conversion.
  cudaEvent_t packed = nullptr;
  if (L->ss.side && !L->pf.on) {
    CU(cudaEventRecord(L->ss.ev[5], st), "fork pack");
    CU(cudaStreamWaitEvent(L->ss.pack, L->ss.ev[5], 0), "fork pack");
    if (zero_small_grads) {   // the accumulated gradient segments (everything before fc.weight) are cleared under the frame conversion
      int64_t off[12], cnt[12];
      layout(L->cfg.A, off, cnt);
      CU(cudaMemsetAsync(L->grads, 0, off[6] * sizeof(float), L->ss.pack), "zero small grads");
    }
    CU(launch_pack_weights(L->P, L->buf.wpack, L->ss.pack, L->buf.wpack_lo, true), "pack_weights");
    CU(cudaEventRecord(L->ss.ev[6], L->ss.pack), "join pack");
    packed = L->ss.ev[6];
  } else {
    if (zero_small_grads) {
      int64_t off[12], cnt[12];
      layout(L->cfg.A, off, cnt);
      L->pf.b(PS_ZERO_GRADS);
      CU(cudaMemsetAsync(L->grads, 0, off[6] * sizeof(float), st), "zero small grads");
      L->pf.e(PS_ZERO_GRADS);
    }
    L->pf.b(PS_PACK);
    CU(launch_pack_weights(L->P, L->buf.wpack, st, L->buf.wpack_lo, true), "pack_weights");
    L->pf.e(PS_PACK);
  }
  CU(encoder_forward(obs, frames, L->P, L->buf, L->maps, L->cfg.precision, st, L->pf, packed, &L->maps_lo), "encoder_forward");
  // learner step (bf16 mode): a3 -> fc.weight column order for the fc weight-gradient GEMM, on the wgrad side stream right after the fc forward,
  // i.e. under the column kernel (32 CTAs, the GPU is otherwise idle) instead of in the crowded backward phase
  L->buf.a3t_ready = false;
  if (zero_small_grads && L->ss.side && !L->pf.on && L->cfg.precision == 0 && L->buf.a3t && !L->cfg.use_lstm) {
    CU(cudaEventRecord(L->ss.ev[10], st), "fork a3 transpose");
    CU(cudaStreamWaitEvent(L->ss.side, L->ss.ev[10], 0), "fork a3 transpose");
    CU(launch_a3_transpose(L->buf.a3, L->buf.a3t, L->cfg.T * L->cfg.B, L->ss.side), "a3_transpose");
    L->buf.a3t_ready = true;
  }
  return 0;
}

static int forward_impl(srl_learner* L, const uint8_t* obs, const float* reward, const int64_t* action, int frames, float* logits,
                        float* baseline, cudaStream_t st, bool zero_small_grads = false) {
  REQ(!L->cfg.use_lstm, "this learner was created with use_lstm=1: call the *_lstm entry points");
  int rc = encode_impl(L, obs, frames, st, zero_small_grads);
  if (rc) return rc;
  L->pf.b(PS_HEAD_FWD);
  CU(launch_head_fwd(L->buf.hpart, FC_SPLITS, L->P.bf, L->buf.h, reward, action, L->P.wp, L->P.bp, L->P.wb, L->P.bb, frames, L->cfg.A,
                     logits, baseline, st), "head_fwd");
  L->pf.e(PS_HEAD_FWD);
  return 0;
}

extern "C" int srl_learner_forward(srl_learner_t* L, const uint8_t* obs, const float* reward, const int64_t* action, int rows,
                                   float* policy_logits, float* baseline, void* stream) {
  REQ(L && obs && reward && action && policy_logits && baseline, "learner_forward: NULL pointer");
  REQ(rows >= 1 && rows <= L->cfg.T + 1, "learner_forward: rows=%d must be in [1, T+1=%d]", rows, L->cfg.T + 1);
  REQ((reinterpret_cast<uintptr_t>(obs) & 3) == 0, "learner_forward: obs must be 4-byte aligned");
  return forward_impl(L, obs, reward, action, rows * L->cfg.B, policy_logits, baseline, (cudaStream_t)stream);
}

static int fb_begin(srl_learner* L, const uint8_t* obs, const float* reward, const uint8_t* done, const int64_t* action,
                    const float* behavior_logits, float* losses, float* vs, float* pg_advantages, cudaStream_t st, int phase) {
  const srl_config_t& c = L->cfg;
  const int NF = (c.T + 1) * c.B, NB = c.T * c.B;
  // heads + V-trace/losses + dh: one fused column kernel when its shared-memory footprint fits, else three kernels
  const bool fused = L->column_fusion && column_step_supported(c.T, c.B, c.A);
  int rc;
  if (fused) {
    REQ(!L->cfg.use_lstm, "this learner was created with use_lstm=1: call the *_lstm entry points");
    rc = encode_impl(L, obs, NF, st, true);
    if (rc) return rc;
    L->pf.b(PS_TAIL);
    CU(launch_column_step(L->buf.hpart, FC_SPLITS, L->P.bf, L->buf.h, reward, action, done, behavior_logits, L->P.wp, L->P.bp, L->P.wb,
                          L->P.bb, c.T, c.B, c.A, c.discounting, c.reward_clip_abs_one, c.clip_rho_threshold, c.clip_pg_rho_threshold,
                          c.baseline_cost, c.entropy_cost, L->logits, L->baseline, vs, pg_advantages, L->dlogits, L->dbaseline, L->buf.dh,
                          losses, L->scratch, st, L->buf.dh_lo), "column_step");
    L->pf.e(PS_TAIL);
  } else {
    rc = forward_impl(L, obs, reward, action, NF, L->logits, L->baseline, st, true);
    if (rc) return rc;
    L->pf.b(PS_TAIL);
    CU(launch_impala_tail(behavior_logits, L->logits, L->baseline, action, reward, done, c.T, c.B, c.A, c.discounting,
                          c.reward_clip_abs_one, c.clip_rho_threshold, c.clip_pg_rho_threshold, c.baseline_cost, c.entropy_cost, vs,
                          pg_advantages, L->dlogits, L->dbaseline, losses, L->scratch, st), "impala_tail");
    L->pf.e(PS_TAIL);
  }
  L->pf.b(PS_HEAD_BWD);
  {
    const bool fork = L->ss.side != nullptr && !L->pf.on;
    cudaStream_t sw = fork ? L->ss.side : st;
    if (fork) { CU(cudaEventRecord(L->ss.ev[8], st), "fork head wgrad"); CU(cudaStreamWaitEvent(sw, L->ss.ev[8], 0), "fork head wgrad"); }
    CU(launch_head_bwd(L->dlogits, L->dbaseline, L->buf.h, reward, action, L->P.wp, L->P.wb, NB, c.A, L->buf.dh, L->G.wp, L->G.bp, L->G.wb,
                       L->G.bb, st, sw, !fused, L->buf.dh_lo), "head_bwd");      // side stream `side` is joined by encoder_backward (after the fc wgrad)
  }
  L->pf.e(PS_HEAD_BWD);
  CU(encoder_backward(obs, NB, L->buf, L->G, L->maps, c.precision, st, L->pf, L->ss, phase, &L->maps_lo), "encoder_backward");
  L->have_fwd = true;
  return 0;
}

extern "C" int srl_learner_forward_backward(srl_learner_t* L, const uint8_t* obs, const float* reward, const uint8_t* done,
                                            const int64_t* action, const float* behavior_logits, float* losses, float* vs,
                                            float* pg_advantages, void* stream) {
  REQ(L && obs && reward && done && action && behavior_logits && losses, "learner_forward_backward: NULL pointer");
  REQ((reinterpret_cast<uintptr_t>(obs) & 3) == 0, "learner_forward_backward: obs must be 4-byte aligned");
  return fb_begin(L, obs, reward, done, action, behavior_logits, losses, vs, pg_advantages, (cudaStream_t)stream, 2);
}

extern "C" int srl_learner_forward_backward_begin(srl_learner_t* L, const uint8_t* obs, const float* reward, const uint8_t* done,
                                                  const int64_t* action, const float* behavior_logits, float* losses, float* vs,
                                                  float* pg_advantages, void* stream) {
  REQ(L && obs && reward && done && action && behavior_logits && losses, "learner_forward_backward_begin: NULL pointer");
  REQ((reinterpret_cast<uintptr_t>(obs) & 3) == 0, "learner_forward_backward_begin: obs must be 4-byte aligned");
  return fb_begin(L, obs, reward, done, action, behavior_logits, losses, vs, pg_advantages, (cudaStream_t)stream, 0);
}

extern "C" int srl_learner_backward_finish(srl_learner_t* L, const uint8_t* obs, void* stream) {
  REQ(L && obs, "learner_backward_finish: NULL pointer");
  REQ(L->have_fwd, "learner_backward_finish: call srl_learner_forward_backward_begin first");
  const srl_config_t& c = L->cfg;
  L->pf.st = (cudaStream_t)stream;
  pdl_set_active(!L->pf.on);
  CU(encoder_backward(obs, c.T * c.B, L->buf, L->G, L->maps, c.precision, (cudaStream_t)stream, L->pf, L->ss, 1, &L->maps_lo), "encoder_backward");
  return 0;
}

static int forward_lstm_impl(srl_learner* L, const uint8_t* obs, const float* reward, const uint8_t* done, const int64_t* action,
                             const float* h0, const float* c0, float* logits, float* baseline, float* hT, float* cT, cudaStream_t st) {
  REQ(L->cfg.use_lstm && L->lstm, "this learner was created with use_lstm=0");
  const srl_config_t& c = L->cfg;
  const int NF = (c.T + 1) * c.B;
  int rc = encode_impl(L, obs, NF, st);
  if (rc) return rc;
  CU(launch_core_build(L->buf.hpart, FC_SPLITS, L->P.bf, reward, action, NF, c.A, L->buf.h, L->core, st), "core_build");
  rc = srl_lstm_forward(L->lstm, L->core, done, h0, c0, L->lstm_out, hT, cT, st);
  if (rc) return fail(rc, "lstm_forward: %s", srl_lstm_last_error());
  CU(launch_head_dense_fwd(L->lstm_out, L->P.wp, L->P.bp, L->P.wb, L->P.bb, NF, c.A, logits, baseline, st), "head_dense_fwd");
  return 0;
}

extern "C" int srl_learner_forward_lstm(srl_learner_t* L, const uint8_t* obs, const float* reward, const uint8_t* done, const int64_t* action,
                                        const float* h0, const float* c0, float* policy_logits, float* baseline, float* hT, float* cT,
                                        void* stream) {
  REQ(L && obs && reward && done && action && h0 && c0 && policy_logits && baseline, "learner_forward_lstm: NULL pointer");
  return forward_lstm_impl(L, obs, reward, done, action, h0, c0, policy_logits, baseline, hT, cT, (cudaStream_t)stream);
}

extern "C" int srl_learner_forward_backward_lstm(srl_learner_t* L, const uint8_t* obs, const float* reward, const uint8_t* done,
                                                 const int64_t* action, const float* behavior_logits, const float* h0, const float* c0,
                                                 float* losses, float* vs, float* pg_advantages, void* stream) {
  REQ(L && obs && reward && done && action && behavior_logits && h0 && c0 && losses, "learner_forward_backward_lstm: NULL pointer");
  cudaStream_t st = (cudaStream_t)stream;
  const srl_config_t& c = L->cfg;
  const int NB = c.T * c.B;
  int rc = forward_lstm_impl(L, obs, reward, done, action, h0, c0, L->logits, L->baseline, nullptr, nullptr, st);
  if (rc) return rc;
  CU(launch_impala_tail(behavior_logits, L->logits, L->baseline, action, reward, done, c.T, c.B, c.A, c.discounting, c.reward_clip_abs_one,
                        c.clip_rho_threshold, c.clip_pg_rho_threshold, c.baseline_cost, c.entropy_cost, vs, pg_advantages, L->dlogits,
                        L->dbaseline, losses, L->scratch, st), "impala_tail");
  {
    int64_t off[12], cnt[12];
    layout(c.A, off, cnt);
    CU(cudaMemsetAsync(L->grads, 0, off[6] * sizeof(float), st), "zero small grads");
    CU(cudaMemsetAsync(L->grads + L->lstm_off0, 0, L->lstm_len * sizeof(float), st), "zero lstm grads");
  }
  CU(launch_head_dense_bwd(L->lstm_out, L->dlogits, L->dbaseline, L->P.wp, L->P.wb, NB, c.A, L->dout, L->G.wp, L->G.bp, L->G.wb, L->G.bb, st),
     "head_dense_bwd");
  rc = srl_lstm_backward(L->lstm, L->dout, done, L->dcore, st);
  if (rc) return fail(rc, "lstm_backward: %s", srl_lstm_last_error());
  CU(launch_dcore_to_dh(L->dcore, L->buf.h, NB, c.A, L->buf.dh, st), "dcore_to_dh");
  CU(encoder_backward(obs, NB, L->buf, L->G, L->maps, c.precision, st, L->pf, L->ss, 2, &L->maps_lo), "encoder_backward");
  L->have_fwd = true;
  return 0;
}

extern "C" int srl_learner_apply_gradients(srl_learner_t* L, float* grad_norm_out, void* stream) {
  REQ(L, "learner is NULL");
  cudaStream_t st = (cudaStream_t)stream;
  const srl_config_t& c = L->cfg;
  L->pf.st = st;
  L->step += 1;
  // clip_grad_norm_ + optimizer in one cooperative kernel (profile slot: optimizer)
  L->pf.b(PS_OPTIMIZER);
  if (c.optimizer == 0) {
    CU(launch_clip_optim(0, L->params, L->grads, L->opt0, nullptr, L->nparams, c.max_grad_norm, L->coef, L->scratch + 2048, c.learning_rate,
                         c.alpha, 0.f, c.epsilon, L->step, L->dstep, st), "clip+rmsprop");
  } else {
    CU(launch_clip_optim(1, L->params, L->grads, L->opt0, L->opt1, L->nparams, c.max_grad_norm, L->coef, L->scratch + 2048, c.learning_rate,
                         c.adam_beta1, c.adam_beta2, c.adam_eps, L->step, L->dstep, st), "clip+adam");
  }
  L->pf.e(PS_OPTIMIZER);
  if (grad_norm_out) CU(cudaMemcpyAsync(grad_norm_out, L->coef, 2 * sizeof(float), cudaMemcpyDeviceToDevice, st), "copy coef");
  return 0;
}

extern "C" int srl_learner_apply_gradients_dp(srl_learner_t* L, const srl_dp_peers_t* peers, float* grad_norm_out, void* stream) {
  REQ(L && peers, "apply_gradients_dp: NULL argument");
  REQ(peers->world >= 2 && peers->world <= 8 && peers->rank >= 0 && peers->rank < peers->world, "apply_gradients_dp: world=%d rank=%d",
      peers->world, peers->rank);
  REQ(peers->grads[peers->rank] == (void*)L->grads, "apply_gradients_dp: grads[rank] must be the learner's gradient buffer");
  cudaStream_t st = (cudaStream_t)stream;
  const srl_config_t& c = L->cfg;
  DpPeers P;
  for (int i = 0; i < 8; ++i) {
    P.g[i] = i < peers->world ? (float*)peers->grads[i] : nullptr;
    P.ctl[i] = i < peers->world ? (unsigned*)peers->ctl[i] : nullptr;
    P.rs[i] = i < peers->world ? (float*)peers->exchange[i] : nullptr;
    REQ(i >= peers->world || (P.g[i] && P.ctl[i] && P.rs[i]), "apply_gradients_dp: NULL peer pointer %d", i);
  }
  P.rank = peers->rank; P.world = peers->world; P.mc_g = (float*)peers->grads_multicast;
  L->pf.st = st;
  L->step += 1;
  L->pf.b(PS_OPTIMIZER);
  if (c.optimizer == 0) {
    CU(launch_dp_clip_optim(0, L->params, L->grads, L->opt0, nullptr, L->nparams, c.max_grad_norm, L->coef, L->scratch + 2048,
                            c.learning_rate, c.alpha, 0.f, c.epsilon, L->step, L->dstep, P, st), "dp clip+rmsprop");
  } else {
    CU(launch_dp_clip_optim(1, L->params, L->grads, L->opt0, L->opt1, L->nparams, c.max_grad_norm, L->coef, L->scratch + 2048,
                            c.learning_rate, c.adam_beta1, c.adam_beta2, c.adam_eps, L->step, L->dstep, P, st), "dp clip+adam");
  }
  L->pf.e(PS_OPTIMIZER);
  if (grad_norm_out) CU(cudaMemcpyAsync(grad_norm_out, L->coef, 2 * sizeof(float), cudaMemcpyDeviceToDevice, st), "copy coef");
  return 0;
}

extern "C" int srl_learner_set_profiling(srl_learner_t* L, int enable) {
  REQ(L, "learner is NULL");
  if (enable && !L->events[0])
    for (int i = 0; i < 2 * PS_COUNT; ++i) CU(cudaEventCreate(&L->events[i]), "cudaEventCreate");
  L->pf.on = enable != 0;
  L->pf.ev = L->events;
  return 0;
}
extern "C" int srl_profile_slot_count(void) { return PS_COUNT; }
extern "C" const char* srl_profile_slot_name(int slot) { return (slot >= 0 && slot < PS_COUNT) ? kSlotNames[slot] : ""; }
extern "C" int srl_learner_profile_collect(srl_learner_t* L, float* ms_out_host) {
  REQ(L && ms_out_host, "profile_collect: NULL argument");
  REQ(L->pf.on, "profile_collect: profiling is off");
  for (int i = 0; i < PS_COUNT; ++i) {
    float ms = 0.f;
    cudaError_t e = cudaEventSynchronize(L->events[2 * i + 1]);
    if (e == cudaSuccess) e = cudaEventElapsedTime(&ms, L->events[2 * i], L->events[2 * i + 1]);
    if (e != cudaSuccess) { cudaGetLastError(); ms = -1.f; }   // slot not recorded in the last step
    ms_out_host[i] = ms;
  }
  return 0;
}

extern "C" int srl_learner_snapshot_params(srl_learner_t* L, float* dst, const float* losses, void* stream) {
  REQ(L && dst, "snapshot_params: NULL argument");
  REQ((reinterpret_cast<uintptr_t>(dst) & 15) == 0, "snapshot_params: dst must be 16-byte aligned");
  CU(launch_snapshot_if_finite(dst, L->params, L->nparams, losses, (cudaStream_t)stream), "snapshot_params");
  return 0;
}

// Pinning of caller-owned HOST memory (the shared-memory trajectory ring, the actors' shared parameter tensors) so that the
// copy engine reads / writes it directly.  A stale registration left by a freed mapping at the same address (or a second tensor
// on an already pinned page) is replaced instead of failing, and no sticky error is left behind for the next CUDA call.
extern "C" int srl_host_register(void* ptr_host, int64_t bytes) {
  REQ(ptr_host && bytes > 0, "host_register: bad argument");
  cudaError_t e = cudaHostRegister(ptr_host, (size_t)bytes, cudaHostRegisterDefault);
  if (e == cudaErrorHostMemoryAlreadyRegistered) {
    cudaGetLastError();
    cudaHostUnregister(ptr_host);
    cudaGetLastError();
    e = cudaHostRegister(ptr_host, (size_t)bytes, cudaHostRegisterDefault);
    if (e == cudaErrorHostMemoryAlreadyRegistered) { cudaGetLastError(); return 0; }     // part of a larger live registration: fine
  }
  if (e != cudaSuccess) { cudaGetLastError(); return cuda_fail(e, "cudaHostRegister"); }
  return 0;
}
extern "C" int srl_host_unregister(void* ptr_host) {
  REQ(ptr_host, "host_unregister: NULL");
  cudaError_t e = cudaHostUnregister(ptr_host);
  cudaGetLastError();
  return (e == cudaSuccess || e == cudaErrorHostMemoryNotRegistered) ? 0 : cuda_fail(e, "cudaHostUnregister");
}

extern "C" int srl_memcpy_d2d(void* dst, const void* src, int64_t bytes, void* stream) {
  REQ(dst && src && bytes >= 0, "memcpy_d2d: bad argument");
  CU(cudaMemcpyAsync(dst, src, (size_t)bytes, cudaMemcpyDeviceToDevice, (cudaStream_t)stream), "memcpy_d2d");
  return 0;
}

extern "C" int srl_learner_debug_buffer(srl_learner_t* L, const char* name, void** ptr, int64_t* count) {
  REQ(L && name && ptr && count, "debug_buffer: NULL argument");
  const int64_t NF = (int64_t)(L->cfg.T + 1) * L->cfg.B, NB = (int64_t)L->cfg.T * L->cfg.B, A = L->cfg.A;
  struct { const char* n; void* p; int64_t c; } tab[] = {
      {"xs", L->buf.xs, NF * 441 * 64}, {"a1", L->buf.a1, NF * 400 * 32}, {"a2", L->buf.a2, NF * 81 * 64}, {"a3", L->buf.a3, NF * 49 * 64}, {"a3t", L->buf.a3t, NF * 49 * 64}, {"h", L->buf.h, NF * 512},
      {"logits", L->logits, NF * A}, {"baseline", L->baseline, NF}, {"dlogits", L->dlogits, NB * A}, {"dbaseline", L->dbaseline, NB},
      {"dh", L->buf.dh, NB * 512}, {"da3", L->buf.da3, NB * 81 * 64}, {"da2", L->buf.da2, NB * 100 * 64},
      {"da1", L->buf.da1, NB * 441 * 32}, {"wpack", L->buf.wpack, WPack::TOTAL},
      {"a1_lo", L->buf.a1_lo, NF * 400 * 32}, {"a2_lo", L->buf.a2_lo, NF * 81 * 64}, {"a3_lo", L->buf.a3_lo, NF * 49 * 64},
      {"dh_lo", L->buf.dh_lo, NB * 512}, {"da3_lo", L->buf.da3_lo, NB * 81 * 64}, {"da2_lo", L->buf.da2_lo, NB * 100 * 64},
      {"da1_lo", L->buf.da1_lo, NB * 441 * 32}, {"wpack_lo", L->buf.wpack_lo, WPack::TOTAL}};
  for (auto& t : tab)
    if (strcmp(t.n, name) == 0) {
      if (!t.p) return fail(SRL_ESTATE, "debug_buffer: '%s' exists only in the fp32-accurate operand mode (precision = 1)", name);
      *ptr = t.p; *count = t.c; return 0;
    }
  return fail(SRL_EINVAL, "debug_buffer: unknown buffer '%s'", name);
}
