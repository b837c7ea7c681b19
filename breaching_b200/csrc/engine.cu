// The iteration engine: owns the device-resident state of one trial and executes the four sweeps of the layer
// program plus objective, priors and the fused optimiser step, captured once as a CUDA graph and replayed with
// no host synchronisation inside the loop (the reference needs three host syncs per iteration,
// optimization_based_attack.py:119,131,135).  C ABI in include/breaching_b200.h.
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <limits>
#include <string>
#include <vector>

#include "../../include/breaching_b200.h"
#include "common.cuh"
#include "igemm.cuh"
#include "layers.cuh"
#include "tokens.cuh"
#include "objective.cuh"
#include "augment.cuh"

namespace bre {
void set_pdl(bool on);
static thread_local std::string g_last_error;
void set_error(const std::string& msg) { g_last_error = msg; }
static int g_pdl = -1;
bool use_pdl() {
  if (g_pdl < 0) {
    const char* e = getenv("BRE_PDL");
    g_pdl = e ? (atoi(e) != 0) : 1;
  }
  return g_pdl != 0;
}
void set_pdl(bool on) { g_pdl = on ? 1 : 0; }
static thread_local bool g_serialize_once = false;
void serialize_next_launch() { g_serialize_once = true; }
bool consume_serialize_once() { const bool r = g_serialize_once; g_serialize_once = false; return r; }
}  // namespace bre

using namespace bre;

namespace {

struct TensorBuf {
  bre_tensor_desc desc;
  long long numel = 0;
  float *val = nullptr, *d = nullptr, *tval = nullptr, *td = nullptr;
};
struct ParamInfo {
  bre_param_desc desc;
  long long off = 0;
};
struct BnBuf {
  int C = 0;
  float *rm = nullptr, *rv = nullptr, *scale = nullptr, *shift = nullptr, *inv = nullptr, *nrm = nullptr;
  float *di_mean = nullptr, *di_var = nullptr, *di_cm = nullptr, *di_cv = nullptr;
  // train-mode BN reuses di_mean / di_var for the batch statistics and di_cm / di_cv for the tangent-forward means; the
  // tangent-backward means live here
  float *tb1 = nullptr, *tb2 = nullptr;
};

#define BRE_TRY(call)            \
  do {                           \
    int _rc = (call);            \
    if (_rc != 0) return _rc;    \
  } while (0)
#define BRE_LAUNCH(call)         \
  do {                           \
    int _rc = (call);            \
    if (_rc != 0) return _rc;    \
    ++launch_count;              \
  } while (0)

template <typename T>
int dev_alloc(T** p, long long n) {
  if (n <= 0) n = 1;
  BRE_CUDA_CHECK(cudaMalloc((void**)p, (size_t)n * sizeof(T)));
  BRE_CUDA_CHECK(cudaMemset(*p, 0, (size_t)n * sizeof(T)));
  return 0;
}

}  // namespace

struct bre_engine {
  int device = 0;
  cudaStream_t stream = nullptr;
  std::vector<TensorBuf> t;
  std::vector<bre_op_desc> ops;
  std::vector<ParamInfo> params;
  std::vector<BnBuf> bn;           // indexed by op.bn_buffer
  std::vector<int*> pool_idx;      // per op (maxpool only)
  int logits = -1;
  bre_attack_cfg cfg;
  std::vector<void*> allocs;

  long long P_pad = 0, max_param = 0, max_tensor = 0;
  float *W = nullptr, *g = nullptr, *G = nullptr, *V = nullptr, *stage = nullptr, *chunk_w = nullptr;
  // TF32-rounded shadows of the parameter and direction arenas: what the tcgen05 GEMMs read (the masters stay fp32: a local
  // SGD step or an adjoint update is far below one TF32 ulp of the weights).  See tf32_rna in common.cuh.
  float *Wt = nullptr, *Vt = nullptr;
  std::vector<float*> ms_Wt;
  bool tc_round_env = [] { const char* e = getenv("BRE_TC_ROUND"); return e ? atoi(e) != 0 : true; }();
  bool tc_round() const { return gemm_backend == 1 && tc_round_env; }
  float *p = nullptr, *loss_n = nullptr;
  long long* labels = nullptr;
  // token-sequence programs (compiler.compile_transformer): rows = batch * seq_len, next-token loss over rows
  int seq_len = 0;
  std::vector<float*> tok_a, tok_b;   // per op: LayerNorm (mean, inv) per row | attention probabilities P and their tangent P'
  float* soft_q = nullptr;        // class-probability targets [N, C] (joint-optimisation attacks), null = index labels
  float* soft_q_buf = nullptr;    // owned storage behind soft_q
  float* label_grad = nullptr;    // d(objective)/d(soft_q) of the last evaluation
  int n_labels = 0;
  // token models: the vocabulary may be padded to the GEMM tile width -- logits-shaped tensors then have td(logits).C columns of
  // which the first `logits_valid` are real classes (0 = all of them); label-shaped tensors are dense [rows, classes]
  int logits_valid = 0;
  int classes() const { return logits_valid > 0 ? logits_valid : td(logits).C; }
  // joint data + label optimisation on the device (optimization_with_label_attack.py:89-143): the label logits are a second
  // leaf [rows, classes] with their own optimiser state and best-so-far copy
  bool joint = false;
  float *ell = nullptr, *ell_m = nullptr, *ell_v = nullptr, *ell_best = nullptr;
  long long n_ell = 0;
  // candidate state
  long long nx = 0;
  int xN = 0, xC = 0, xH = 0, xW = 0;
  float *x = nullptr, *gradx = nullptr, *gradx_task = nullptr, *m = nullptr, *v = nullptr, *best = nullptr;
  float *history = nullptr, *lr_table = nullptr, *lo = nullptr, *hi = nullptr;
  int n_lr = 0, lr_cap = 0;
  Scalars* sc = nullptr;
  // scratch
  float* ws = nullptr;
  int ws_tiles = 0;
  int* gemm_counters = nullptr;
  float* red_partials = nullptr;
  int* red_counters = nullptr;
  double* dpartials = nullptr;
  int* dcounter = nullptr;
  DiLayer* di_layers_dev = nullptr;
  int n_di = 0;
  float* feat_measured = nullptr;
  long long feat_numel = 0;
  int feat_op = -1;
  // side stream: weight gradients are off the critical path of the backward sweep (they only feed the matching
  // reduction), so they run concurrently with the dgrad chain; the side stream has its own split-K / reduction scratch
  cudaStream_t side = nullptr;
  std::vector<cudaEvent_t> ev_fork;
  cudaEvent_t ev_join = nullptr;
  bool overlap_wgrad = true;
  // BN + residual + ReLU (and its tangent) in the epilogue of the producing tcgen05 fprop.  Off by default: measured on the
  // B200 it removes 32 of 201 launches per config-2 iteration and is still 1.5 % slower (the split-K epilogue's extra global
  // loads cost more than the PDL-overlapped element-wise kernels they replace).  BRE_FUSE_BNACT=1 / option "fuse_bnact".
  bool fuse_bnact = [] { const char* e = getenv("BRE_FUSE_BNACT"); return e ? atoi(e) != 0 : false; }();
  float* ws2 = nullptr;
  int* gemm_counters2 = nullptr;
  float* red_partials2 = nullptr;
  int* red_counters2 = nullptr;
  // FedAvg / multi-step local updates (objectives.py:48-72): K forward+backward passes at W_0 .. W_{K-1}, the matched
  // quantity is W_K - W_0; the adjoint is carried back over the steps with Hessian-vector products (tangent wgrads).
  struct StepBufs {
    std::vector<float*> val, d;
    std::vector<int*> idx;
    std::vector<float*> bn_scale, bn_shift;
    float* p = nullptr; float* loss_n = nullptr; long long* labels = nullptr;
  };
  int ms_steps = 0;                 // 0 = single gradient (objectives.py:40-46)
  float ms_lr = 0.f;
  std::vector<float*> ms_W;         // K + 1 parameter arenas, ms_W[0] = W
  std::vector<StepBufs> ms_bufs;    // per-step saved state (step 0 = the default buffers)
  std::vector<long long> ms_offset; // element offset of each step's candidate slice
  float* ms_D = nullptr;            // W_K - W_0
  float* gradx_step = nullptr;      // tangent input gradient of one step (program batch)
  float* W0 = nullptr;
  struct BnPrep { int gamma_off, beta_off, C; const float* inv; const float* nrm; float* scale; float* shift; };
  std::vector<BnPrep*> ms_bnprep_dev;  // per step (k >= 1): device table for the batched BN-constant refresh
  int n_bn_layers = 0;
  bool want_tangent_G = false;
  // column path of the candidate-fed convolution on the tensor-core back end (stem_cols.cu)
  int stem_op = -1, stem_Kp = 0;
  float *xcol = nullptr, *dcol = nullptr, *Wcol = nullptr, *Vcol = nullptr, *Gcol = nullptr;
  bool stem_cols_env = [] { const char* e = getenv("BRE_STEM_COLS"); return e ? atoi(e) != 0 : true; }();
  bool use_stem_cols(size_t i) { return gemm_backend == 1 && stem_cols_env && (int)i == stem_op && !is_precise(i); }
  GemmArgs stem_geom(const bre_op_desc& op) const {   // the layer as a 1x1 convolution over xcol [N, Ho, Wo, Kp]
    GemmArgs a;
    memset(&a, 0, sizeof(a));
    const bre_tensor_desc& to = td(op.tout);
    a.g = ConvGeom{to.N, to.H, to.W, stem_Kp, to.H, to.W, to.C, 1, 1, 1, 0};
    a.x_sN = (long long)to.H * to.W * stem_Kp; a.x_sP = stem_Kp; a.x_sC = 1;
    a.nsrc = 1;
    a.ws = ws; a.counters = gemm_counters; a.ws_tiles = ws_tiles; a.splits = 0;
    return a;
  }
  int stem_unfold(const bre_op_desc& op) {            // candidate -> xcol
    const bre_tensor_desc &ti = td(op.tin), &to = td(op.tout);
    BRE_LAUNCH(launch_stem_im2col(t[0].val, xcol, ti.N, ti.C, ti.H, ti.W, to.H, to.W, op.R, op.S, op.stride, op.pad, stem_Kp, tc_round(), stream));
    return 0;
  }
  int stem_pad(const float* src, float* dst, const bre_op_desc& op, cudaStream_t st) {
    BRE_LAUNCH(launch_stem_pad_rows(src, dst, td(op.tout).C, op.R * op.S * td(op.tin).C, stem_Kp, false, tc_round(), st));
    return 0;
  }
  int stem_fold(const bre_op_desc& op, float* grad_out) {   // dcol -> NCHW candidate gradient
    const bre_tensor_desc &ti = td(op.tin), &to = td(op.tout);
    BRE_LAUNCH(launch_stem_col2im(dcol, grad_out, ti.N, ti.C, ti.H, ti.W, to.H, to.W, op.R, op.S, op.stride, op.pad, stem_Kp, stream));
    return 0;
  }
  // precision knob of the tensor-core back end: the first `precise_first` and last `precise_last` conv / linear layers (program
  // order) run on the fp32 kernels with unrounded operands -- for badly conditioned cases (config 3: random-init ResNet-50 whose
  // BN-statistics prior differences amplify TF32 rounding, see DESIGN.md) at the price of those layers' tensor-core speed
  int precise_first = [] { const char* e = getenv("BRE_PRECISE_FIRST"); return e ? atoi(e) : 0; }();
  int precise_last = [] { const char* e = getenv("BRE_PRECISE_LAST"); return e ? atoi(e) : 0; }();
  mutable std::vector<char> precise_op;
  bool is_precise(size_t i) const {
    if (precise_op.size() != ops.size()) {
      precise_op.assign(ops.size(), 0);
      std::vector<int> gemm_ops_idx;
      for (size_t j = 0; j < ops.size(); ++j) if (ops[j].kind == BRE_OP_CONV || ops[j].kind == BRE_OP_LINEAR) gemm_ops_idx.push_back((int)j);
      const int n = (int)gemm_ops_idx.size();
      for (int j = 0; j < n; ++j) if (j < precise_first || j >= n - precise_last) precise_op[gemm_ops_idx[j]] = 1;
    }
    return gemm_backend == 1 && precise_op[i] != 0;
  }
  // candidate augmentations (augment.cu; optimization_based_attack.py:149-153): the model and the priors see view(x); the
  // gradient is pulled back through the transposed view (differentiable mode) or x itself is replaced by its view (the
  // reference's non-differentiable mode, which assigns candidate.data)
  bool aug_on = false, aug_diff = false;
  AugPlan aug;
  AugDraws* aug_draws = nullptr;
  float *x_aug = nullptr, *gradx_aug = nullptr, *aug_tmp = nullptr, *cj_scale = nullptr, *cj_shift = nullptr;
  float* input_x() const { return aug_on && aug_diff ? x_aug : x; }          // what the first layer and the priors read
  float* input_grad() const { return aug_on && aug_diff ? gradx_aug : gradx; }
  void bind_input() { t[0].val = input_x(); t[0].td = input_grad(); }
  int augment_forward() {
    BRE_LAUNCH(launch_aug_draw(aug, sc, aug_draws, xN, stream));
    BRE_LAUNCH(launch_aug_view(x, x_aug, xN, xC, xH, xW, aug, aug_draws, stream));
    if (!aug_diff) BRE_CUDA_CHECK(cudaMemcpyAsync(x, x_aug, nx * sizeof(float), cudaMemcpyDeviceToDevice, stream));
    return 0;
  }
  int augment_pull() {   // gradx <- view^T (gradx_aug + task_regularization * gradx_task)
    if (need_task_grad()) BRE_LAUNCH(launch_axpy(gradx_task, gradx_aug, cfg.task_regularization, nx, stream));
    BRE_LAUNCH(launch_aug_pull(gradx_aug, aug_tmp, gradx, xN, xC, xH, xW, aug, aug_draws, stream));
    return 0;
  }
  bool task_grad_folded() const { return aug_on && aug_diff; }   // the task-gradient term already sits inside gradx
  // deferred finalisation of the BN parameter gradients (layers.cu bn_grad_finalize_kernel): per-layer partial regions + table
  bool defer_bn_env = [] { const char* e = getenv("BRE_DEFER_BN"); return e ? atoi(e) != 0 : true; }();
  std::vector<float*> bn_partials;      // per op (BNACT with eval-mode BN), null otherwise
  BnGradSlot* bn_slots_dev = nullptr;
  int bn_slots = 0, bn_slot_blocks = 0;
  bool bn_slots_built = false;
  int build_bn_slots() {
    if (bn_slots_built) return 0;
    bn_slots_built = true;
    if (!defer_bn_env) return 0;
    std::vector<BnGradSlot> table;
    bn_partials.assign(ops.size(), nullptr);
    int blocks = 0;
    for (size_t i = 0; i < ops.size(); ++i) {
      const bre_op_desc& op = ops[i];
      if (op.kind != BRE_OP_BNACT || !op.has_bn || op.bn_train) continue;
      const bre_tensor_desc& to = td(op.tout);
      int slabs = 0, Cpad = 0;
      bnact_bwd_plan((long long)to.N * to.H * to.W, to.C, &slabs, &Cpad);
      float* buf = nullptr;
      BRE_TRY(alloc(&buf, (long long)slabs * Cpad * 2));
      bn_partials[i] = buf;
      table.push_back(BnGradSlot{buf, slabs, Cpad, to.C, blocks, nullptr, nullptr});   // gradient pointers: filled per sweep (G arena is fixed)
      table.back().g_gamma = Gp(op.gamma); table.back().g_beta = Gp(op.beta);
      blocks += (to.C + 31) / 32;     // bn_grad_finalize_kernel: one block per 32 channels
    }
    bn_slots = (int)table.size(); bn_slot_blocks = blocks;
    if (bn_slots == 0) return 0;
    BRE_TRY(alloc(&bn_slots_dev, (long long)table.size()));
    BRE_CUDA_CHECK(cudaMemcpy(bn_slots_dev, table.data(), table.size() * sizeof(BnGradSlot), cudaMemcpyHostToDevice));
    return 0;
  }
  // execution
  bool use_graph = true;
  int gemm_backend = 0;  // 0 = SIMT fp32, 1 = tcgen05 TF32 where supported
  cudaGraphExec_t exec = nullptr;
  bool graph_ready = false;
  int launch_count = 0, launches_per_iter = 0;
  bool model_loaded = false, targets_loaded = false, trial_begun = false;

  template <typename T>
  int alloc(T** ptr, long long n) {
    int rc = dev_alloc(ptr, n);
    if (rc == 0) allocs.push_back((void*)*ptr);
    return rc;
  }

  const bre_tensor_desc& td(int i) const { return t[i].desc; }
  float* Wp(int idx) const { return W + params[idx].off; }
  float* Gp(int idx) const { return G + params[idx].off; }
  float* Vp(int idx) const { return V + params[idx].off; }
  // conv / linear weights as GEMM operands: the TF32-rounded shadow for the layers the tcgen05 back end covers, the fp32
  // master for the layers that run on the SIMT kernels (so that a network with no eligible layer is bit-identical on both
  // back ends)
  size_t op_index(const bre_op_desc& op) const { return (size_t)(&op - ops.data()); }
  const float* Wg(const bre_op_desc& op) { return (round_val(op.tin) && !is_precise(op_index(op)) ? Wt : W) + params[op.w].off; }
  const float* Vg(const bre_op_desc& op) { return (round_val(op.tin) && !is_precise(op_index(op)) ? Vt : V) + params[op.w].off; }
  int refresh_Vt() {
    if (tc_round()) BRE_LAUNCH(launch_round_tf32(V, Vt, P_pad, stream));
    return 0;
  }
  // per-chunk routing of the direction write (launch_make_v): 1 = TF32 shadow only for the weights of tensor-core layers (the
  // GEMMs read Vt, nothing reads their fp32 direction in single-step mode), 0 = fp32 only for everything else (BN / bias
  // vectors, layers on the fp32 kernels, the stem weight that stem_pad rounds itself)
  unsigned char* chunk_mode = nullptr;
  bool chunk_mode_ready = false;
  int build_chunk_modes() {
    if (chunk_mode_ready || !tc_round()) return 0;
    std::vector<unsigned char> host((size_t)(P_pad / kChunk), 0);
    for (const bre_op_desc& op : ops) {
      if ((op.kind != BRE_OP_CONV && op.kind != BRE_OP_LINEAR) || !round_val(op.tin) || is_precise(op_index(op))) continue;
      const long long c0 = params[op.w].off / kChunk, c1 = c0 + (params[op.w].desc.numel + kChunk - 1) / kChunk;
      for (long long c = c0; c < c1; ++c) host[(size_t)c] = 1;
    }
    if (!chunk_mode) BRE_TRY(alloc(&chunk_mode, P_pad / kChunk));
    // (host vector -> pageable copy: performed before the copy call returns; no kernel of the captured iteration depends on
    // stream order here because the first launch that reads it follows in the same stream)
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    cudaStreamIsCapturing(stream, &cs);
    if (cs != cudaStreamCaptureStatusNone) { set_error("chunk modes must be built before graph capture"); return BRE_ERR_STATE; }
    BRE_CUDA_CHECK(cudaMemcpy(chunk_mode, host.data(), host.size(), cudaMemcpyHostToDevice));
    chunk_mode_ready = true;
    return 0;
  }
  // Which activation tensors are operands of a tensor-core GEMM: inputs (value / tangent) and output deltas of the
  // convolutions the tcgen05 back end covers.  Only those are stored TF32-rounded; layers that run on the fp32 SIMT kernels
  // (3-channel stem, narrow test networks, the classifier head) keep full fp32 operands.
  std::vector<char> rnd_val, rnd_d;
  void compute_round_flags() {
    rnd_val.assign(t.size(), 0);
    rnd_d.assign(t.size(), 0);
    for (size_t oi = 0; oi < ops.size(); ++oi) {
      const bre_op_desc& op = ops[oi];
      if (op.kind != BRE_OP_CONV && op.kind != BRE_OP_LINEAR) continue;
      if (is_precise(oi)) continue;
      GemmArgs a = conv_geom(op);
      a.act[0] = t[op.tin].val; a.wgt[0] = Wp(op.w); a.out = t[op.tout].val;
      bool any = false;
      for (int mode = 0; mode < 3; ++mode) { a.mode = mode; any = any || igemm_tc_supported(a); }
      if (any) { rnd_val[op.tin] = 1; rnd_d[op.tout] = 1; }
    }
    if (stem_op >= 0 && stem_cols_env && !is_precise((size_t)stem_op)) rnd_d[ops[stem_op].tout] = 1;   // deltas of the stem output feed its column GEMMs
  }
  bool round_val(int tensor) { if (rnd_val.size() != t.size()) compute_round_flags(); return tc_round() && rnd_val[tensor]; }
  bool round_d(int tensor) { if (rnd_d.size() != t.size()) compute_round_flags(); return tc_round() && rnd_d[tensor]; }

  // ---- GEMM argument assembly -----------------------------------------------------------------
  GemmArgs conv_geom(const bre_op_desc& op) const {
    GemmArgs a;
    memset(&a, 0, sizeof(a));
    const bre_tensor_desc &ti = td(op.tin), &to = td(op.tout);
    ConvGeom& g = a.g;
    if (op.kind == BRE_OP_LINEAR) {
      g.N = ti.N; g.H = 1; g.W = 1; g.Ci = ti.C * ti.H * ti.W; g.Ho = 1; g.Wo = 1; g.Co = to.C;
      g.R = 1; g.S = 1; g.stride = 1; g.pad = 0;
      a.x_sN = g.Ci; a.x_sP = g.Ci; a.x_sC = 1;
    } else {
      g.N = ti.N; g.H = ti.H; g.W = ti.W; g.Ci = ti.C; g.Ho = to.H; g.Wo = to.W; g.Co = to.C;
      g.R = op.R; g.S = op.S; g.stride = op.stride; g.pad = op.pad;
      if (op.tin == 0) { a.x_sN = (long long)ti.C * ti.H * ti.W; a.x_sP = 1; a.x_sC = ti.H * ti.W; }   // NCHW candidate
      else { a.x_sN = (long long)ti.H * ti.W * ti.C; a.x_sP = ti.C; a.x_sC = 1; }                         // NHWC internal
    }
    a.nsrc = 1;
    a.ws = ws; a.counters = gemm_counters; a.ws_tiles = ws_tiles; a.splits = 0;
    a.force_fp32 = is_precise(op_index(op)) ? 1 : 0;
    return a;
  }
  int gemm(const GemmArgs& a) { return gemm_on(a, stream); }
  // Weight operands the tensor-core kernels may load ahead of griddepcontrol.wait: the model weights (and their TF32 shadow /
  // column copy) of a single-step user never change during a run; the direction v and its shadow are final once the serialised
  // launch after make_v has started (evaluate()).  FedAvg users (ms_steps > 0) rewrite W_k and v inside the iteration: none.
  bool weight_prefetch = [] { const char* e = getenv("BRE_TC_WPREFETCH"); return e ? atoi(e) != 0 : true; }();
  bool v_settled = false;
  bool inside(const float* p, const float* base, long long n) const { return base != nullptr && p >= base && p < base + n; }
  unsigned static_weights(const GemmArgs& a) const {
    if (!weight_prefetch || ms_steps > 0 || a.mode == GEMM_WGRAD) return 0u;
    unsigned mask = 0;
    for (int s = 0; s < a.nsrc; ++s) {
      const float* p = a.wgt[s];
      const bool model = inside(p, W, P_pad) || inside(p, Wt, P_pad) || (Wcol != nullptr && p == Wcol);
      const bool direction = v_settled && (inside(p, V, P_pad) || inside(p, Vt, P_pad));
      if (model || direction) mask |= 1u << s;
    }
    return mask;
  }
  // gemm_on's choice of the tcgen05 kernel (the only one that applies an epilogue)
  bool runs_on_tc(const GemmArgs& a) const {
    return !linear_tall_supported(a) && !linear_small_preferred(a) && gemm_backend == 1 && !a.force_fp32 && igemm_tc_supported(a);
  }
  int gemm_on(const GemmArgs& a, cudaStream_t st) {
    if (linear_tall_supported(a)) return launch_linear_tall(a, st);
    if (linear_small_preferred(a)) return launch_linear_small(a, st);
    if (runs_on_tc(a)) {
      GemmArgs b = a;
      b.wgt_static = static_weights(a);
      return launch_igemm_tc(b, st);
    }
    return launch_igemm_simt(a, st);
  }

  // The BN/residual/ReLU op that directly follows conv `i` and reads its output can run in the GEMM epilogue, when the GEMM runs
  // on the tcgen05 kernel (a precise layer runs on the fp32 kernel, which has no epilogue).
  bool fuses_with_next(size_t i, const GemmArgs& a) const {
    if (!fuse_bnact || i + 1 >= ops.size()) return false;
    const bre_op_desc& nx = ops[i + 1];
    return nx.kind == BRE_OP_BNACT && nx.tin == ops[i].tout && !nx.bn_train && runs_on_tc(a);
  }
  int consumers_of(int tensor) const {
    int n = 0;
    for (const bre_op_desc& o : ops) n += (o.tin == tensor) + (o.res == tensor);
    return n;
  }

  // common part of the train-mode BN argument block of op (rules in layers.cuh)
  BnTrainArgs bn_train_args(const bre_op_desc& op) {
    const bre_tensor_desc& to = td(op.tout);
    const BnBuf& b = bn[op.bn_buffer];
    BnTrainArgs a;
    memset(&a, 0, sizeof(a));
    a.P = (long long)to.N * to.H * to.W; a.C = to.C; a.relu = op.relu != 0;
    a.in = t[op.tin].val; a.out = t[op.tout].val;
    a.inv = b.inv; a.nrm = b.nrm; a.scale = b.scale;
    a.v_gamma = Vp(op.gamma); a.v_beta = Vp(op.beta);
    a.sum_du = Gp(op.beta); a.sum_duxh = Gp(op.gamma);
    a.m1 = b.di_cm; a.m2 = b.di_cv; a.b1 = b.tb1; a.b2 = b.tb2;
    a.dout = t[op.tout].d; a.tdout = t[op.tout].td; a.xd = t[op.tin].tval;
    return a;
  }

  BnConsts bn_consts(const bre_op_desc& op) const {
    BnConsts c{nullptr, nullptr, nullptr, nullptr};
    if (op.has_bn) { const BnBuf& b = bn[op.bn_buffer]; c = BnConsts{b.scale, b.shift, b.inv, b.nrm}; }
    return c;
  }
  PoolGeom pool_geom(const bre_op_desc& op) const {
    const bre_tensor_desc &ti = td(op.tin), &to = td(op.tout);
    return PoolGeom{ti.N, ti.H, ti.W, ti.C, to.H, to.W, op.R, op.stride, op.pad};
  }
  bool need_task_grad() const { return cfg.task_regularization != 0.f; }
  float value_task_reg() const { return cfg.objective_excludes_task ? 0.f : cfg.task_regularization; }

  // ---- sweeps ---------------------------------------------------------------------------------------
  int sweep_forward() {
    for (size_t i = 0; i < ops.size(); ++i) {
      const bre_op_desc& op = ops[i];
      const bre_tensor_desc& to = td(op.tout);
      const long long Pout = (long long)to.N * to.H * to.W;
      switch (op.kind) {
        case BRE_OP_CONV:
        case BRE_OP_LINEAR: {
          GemmArgs a = conv_geom(op);
          a.mode = GEMM_FPROP;
          a.act[0] = t[op.tin].val; a.wgt[0] = Wg(op);
          if (use_stem_cols(i)) {
            BRE_TRY(stem_unfold(op));
            if (ms_steps > 0) BRE_TRY(stem_pad(Wp(op.w), Wcol, op, stream));   // W_k changes per local step
            a = stem_geom(op);
            a.mode = GEMM_FPROP;
            a.act[0] = xcol; a.wgt[0] = Wcol;
          }
          a.bias = op.b >= 0 ? Wp(op.b) : nullptr;
          a.out = t[op.tout].val;
          if (fuses_with_next(i, a)) {
            const bre_op_desc& nx = ops[i + 1];
            const BnConsts c = bn_consts(nx);
            a.epi.kind = 1; a.epi.has_bn = nx.has_bn != 0; a.epi.relu = nx.relu != 0; a.epi.round_out = round_val(nx.tout);
            a.epi.out2 = t[nx.tout].val; a.epi.res = nx.res >= 0 ? t[nx.res].val : nullptr;
            a.epi.scale = c.scale; a.epi.shift = c.shift;
            ++i;   // the BNACT op ran in the epilogue
          }
          BRE_LAUNCH(gemm(a));
          break;
        }
        case BRE_OP_BNACT:
          if (op.has_bn && op.bn_train) {   // batch statistics of this forward -> the per-channel constants the kernels read
            BnBuf& b = bn[op.bn_buffer];
            BRE_LAUNCH(launch_channel_stats(t[op.tin].val, Pout, to.C, b.di_mean, b.di_var, red_partials, red_counters, stream));
            BRE_LAUNCH(launch_bn_train_prepare(b.di_mean, b.di_var, Wp(op.gamma), Wp(op.beta), op.eps, to.C, b.scale, b.shift, b.inv,
                                               b.nrm, stream));
          }
          BRE_LAUNCH(launch_bnact_fwd(t[op.tin].val, op.res >= 0 ? t[op.res].val : nullptr, t[op.tout].val, Pout, to.C,
                                      op.has_bn != 0, op.relu != 0, bn_consts(op), round_val(op.tout), stream));
          break;
        case BRE_OP_MAXPOOL:
          BRE_LAUNCH(launch_maxpool_fwd(t[op.tin].val, t[op.tout].val, pool_idx[i], pool_geom(op), stream));
          break;
        case BRE_OP_AVGPOOL: {
          const bre_tensor_desc& ti = td(op.tin);
          BRE_LAUNCH(launch_avgpool_fwd(t[op.tin].val, t[op.tout].val, ti.N, ti.H * ti.W, ti.C, stream));
          break;
        }
        case BRE_OP_POSADD:
          BRE_LAUNCH(launch_token_posadd(t[op.tin].val, Wp(op.w), t[op.tout].val, to.N, to.C, op.S, stream));
          break;
        case BRE_OP_LAYERNORM:
          BRE_LAUNCH(launch_token_layernorm(0, t[op.tin].val, nullptr, nullptr, nullptr, Wp(op.gamma), Wp(op.beta), nullptr, nullptr, op.eps,
                                            to.N, to.C, tok_a[i], t[op.tout].val, 0, stream));
          break;
        case BRE_OP_ATTENTION:
          BRE_LAUNCH(launch_token_attention(0, t[op.tin].val, nullptr, nullptr, nullptr, to.N / op.S, op.S, op.R, to.C / op.R, tok_a[i], tok_b[i],
                                            t[op.tout].val, 0, stream));
          break;
        default: set_error("unknown op kind"); return BRE_ERR_INVALID;
      }
    }
    const bre_tensor_desc& lt = td(logits);
    if (seq_len > 0) {   // next-token loss over rows with class-probability targets (joint attacker on a causal language model)
      if (soft_q == nullptr) { set_error("token programs need soft labels (bre_engine_load_soft_labels)"); return BRE_ERR_STATE; }
      BRE_LAUNCH(launch_token_ce_fwd(t[logits].val, soft_q, lt.N, classes(), lt.C, seq_len, p, loss_n, t[logits].d, stream));
      BRE_LAUNCH(launch_loss_mean(loss_n, lt.N, sc, stream));
      return 0;
    }
    if (classes() != lt.C) { set_error("padded class dimension is only supported for token programs"); return BRE_ERR_UNSUPPORTED; }
    BRE_LAUNCH(launch_ce_fwd(t[logits].val, labels, soft_q, lt.N, lt.C, p, loss_n, t[logits].d, stream));
    BRE_LAUNCH(launch_loss_mean(loss_n, lt.N, sc, stream));
    return 0;
  }

  int sweep_backward() {
    bool forked = false, deferred_bn = false;
    for (int i = (int)ops.size() - 1; i >= 0; --i) {
      const bre_op_desc& op = ops[i];
      const bre_tensor_desc& to = td(op.tout);
      const long long Pout = (long long)to.N * to.H * to.W;
      switch (op.kind) {
        case BRE_OP_CONV:
        case BRE_OP_LINEAR: {
          const bool cols = use_stem_cols((size_t)i);
          GemmArgs a = cols ? stem_geom(op) : conv_geom(op);
          a.mode = GEMM_WGRAD;
          a.act[0] = cols ? xcol : t[op.tin].val; a.wgt[0] = t[op.tout].d; a.out = cols ? Gcol : Gp(op.w);
          const int Kraw = op.R * op.S * td(op.tin).C;
          if (overlap_wgrad && side != nullptr) {
            BRE_CUDA_CHECK(cudaEventRecord(ev_fork[i], stream));
            BRE_CUDA_CHECK(cudaStreamWaitEvent(side, ev_fork[i], 0));
            a.ws = ws2; a.counters = gemm_counters2;
            BRE_LAUNCH(gemm_on(a, side));
            if (cols) BRE_LAUNCH(launch_stem_pad_rows(Gcol, Gp(op.w), to.C, Kraw, stem_Kp, true, false, side));
            if (op.b >= 0) BRE_LAUNCH(launch_channel_sum(t[op.tout].d, Pout, to.C, Gp(op.b), red_partials2, red_counters2, side));
            forked = true;
          } else {
            BRE_LAUNCH(gemm(a));
            if (cols) BRE_LAUNCH(launch_stem_pad_rows(Gcol, Gp(op.w), to.C, Kraw, stem_Kp, true, false, stream));
            if (op.b >= 0) BRE_LAUNCH(launch_channel_sum(t[op.tout].d, Pout, to.C, Gp(op.b), red_partials, red_counters, stream));
          }
          if (op.tin != 0 || need_task_grad()) {
            GemmArgs b = cols ? stem_geom(op) : conv_geom(op);
            b.mode = GEMM_DGRAD;
            b.act[0] = t[op.tout].d; b.wgt[0] = cols ? Wcol : Wg(op);
            b.out = cols ? dcol : (op.tin == 0 ? gradx_task : t[op.tin].d);
            b.accumulate = op.tin == 0 ? 0 : op.acc_in;
            BRE_LAUNCH(gemm(b));
            if (cols) BRE_TRY(stem_fold(op, gradx_task));
          }
          break;
        }
        case BRE_OP_BNACT: {
          BnActBwdArgs a;
          a.P = Pout; a.C = to.C; a.has_bn = op.has_bn != 0; a.relu = op.relu != 0; a.bn = bn_consts(op);
          a.in = t[op.tin].val; a.out = t[op.tout].val; a.dout = t[op.tout].d;
          a.din = t[op.tin].d; a.acc_in = op.acc_in != 0; a.round_din = round_d(op.tin);
          a.dres = op.res >= 0 ? t[op.res].d : nullptr; a.acc_res = op.acc_res != 0;
          a.g_gamma = op.has_bn ? Gp(op.gamma) : nullptr; a.g_beta = op.has_bn ? Gp(op.beta) : nullptr;
          a.partials = red_partials; a.counters = red_counters; a.defer = 0;
          if (op.has_bn && !op.bn_train && !bn_partials.empty() && bn_partials[i] != nullptr) { a.partials = bn_partials[i]; a.defer = 1; deferred_bn = true; }
          // (splitting this op into an element-wise kernel on the main stream and the gamma / beta reductions on the side
          // stream was measured: config 2 unchanged, configs 1 and 3 3-5 % slower -- the side stream is already full)
          if (op.has_bn && op.bn_train) {
            // pass 1: sum(du), sum(du xh) (= the gamma / beta gradients) and the residual delta; pass 2: dx needs those sums
            BnActBwdArgs r = a;
            r.din = nullptr;
            BRE_LAUNCH(launch_bnact_bwd(r, stream));
            BnTrainArgs ta = bn_train_args(op);
            ta.dst = t[op.tin].d; ta.acc = op.acc_in != 0; ta.round_out = round_d(op.tin);
            BRE_LAUNCH(launch_bn_train_bwd(ta, stream));
            break;
          }
          BRE_LAUNCH(launch_bnact_bwd(a, stream));
          break;
        }
        case BRE_OP_MAXPOOL:
          BRE_LAUNCH(launch_maxpool_bwd(t[op.tout].d, pool_idx[i], t[op.tin].d, op.acc_in != 0, pool_geom(op), stream));
          break;
        case BRE_OP_AVGPOOL: {
          const bre_tensor_desc& ti = td(op.tin);
          BRE_LAUNCH(launch_avgpool_bwd(t[op.tout].d, t[op.tin].d, op.acc_in != 0, ti.N, ti.H * ti.W, ti.C, stream));
          break;
        }
        case BRE_OP_POSADD:      // gradient of the positional table (the candidate's own first-backward delta is not needed)
          BRE_LAUNCH(launch_token_pos_grad(t[op.tout].d, Gp(op.w), to.N, to.C, op.S, stream));
          break;
        case BRE_OP_LAYERNORM:
          BRE_LAUNCH(launch_token_ln_param_grad(t[op.tin].val, t[op.tout].d, tok_a[i], to.N, to.C, Gp(op.gamma), Gp(op.beta), stream));
          BRE_LAUNCH(launch_token_layernorm(1, t[op.tin].val, t[op.tout].d, nullptr, nullptr, Wp(op.gamma), Wp(op.beta), nullptr, nullptr, op.eps,
                                            to.N, to.C, tok_a[i], t[op.tin].d, op.acc_in != 0, stream));
          break;
        case BRE_OP_ATTENTION:
          BRE_LAUNCH(launch_token_attention(1, t[op.tin].val, t[op.tout].d, nullptr, nullptr, to.N / op.S, op.S, op.R, to.C / op.R, tok_a[i],
                                            tok_b[i], t[op.tin].d, op.acc_in != 0, stream));
          break;
        default: break;
      }
    }
    if (deferred_bn) BRE_LAUNCH(launch_bn_grad_finalize(bn_slots_dev, bn_slots, bn_slot_blocks, stream));   // gamma / beta gradients of all layers
    if (forked) {
      BRE_CUDA_CHECK(cudaEventRecord(ev_join, side));
      BRE_CUDA_CHECK(cudaStreamWaitEvent(stream, ev_join, 0));
    }
    return 0;
  }

  int reduce_objective(int objective, float scale, float mask_value, bool finalize) {
    const float mv = objective == BRE_OBJ_MASKED_COSINE ? mask_value : -1.f;
    BRE_LAUNCH(launch_match_reduce(G, g, chunk_w, P_pad, mv, objective, scale, cfg.tag_scale, cfg.angular_fudge, finalize, sc,
                                   dpartials, dcounter, stream));
    return 0;
  }

  int sweep_tangent_forward() {
    for (size_t i = 0; i < ops.size(); ++i) {
      const bre_op_desc& op = ops[i];
      const bre_tensor_desc& to = td(op.tout);
      const long long Pout = (long long)to.N * to.H * to.W;
      switch (op.kind) {
        case BRE_OP_CONV:
        case BRE_OP_LINEAR: {
          GemmArgs a = conv_geom(op);
          a.mode = GEMM_FPROP;
          if (use_stem_cols(i)) {
            if (ms_steps > 0) { BRE_TRY(stem_unfold(op)); BRE_TRY(stem_pad(Wp(op.w), Wcol, op, stream)); }   // this step's slice / weights
            BRE_TRY(stem_pad(Vp(op.w), Vcol, op, stream));
            a = stem_geom(op);
            a.mode = GEMM_FPROP;
            a.act[0] = xcol; a.wgt[0] = Vcol;
          } else if (op.tin == 0) {  // tangent of the candidate is zero: only the v-term
            a.act[0] = t[op.tin].val; a.wgt[0] = Vg(op);
          } else {
            a.nsrc = 2;
            a.act[0] = t[op.tin].tval; a.wgt[0] = Wg(op);
            a.act[1] = t[op.tin].val; a.wgt[1] = Vg(op);
          }
          a.bias = op.b >= 0 ? Vp(op.b) : nullptr;
          a.out = t[op.tout].tval;
          if (fuses_with_next(i, a)) {
            const bre_op_desc& nx = ops[i + 1];
            const BnConsts c = bn_consts(nx);
            a.epi.kind = 2; a.epi.has_bn = nx.has_bn != 0; a.epi.relu = nx.relu != 0; a.epi.round_out = round_val(nx.tout);
            a.epi.out2 = t[nx.tout].tval; a.epi.res = nx.res >= 0 ? t[nx.res].tval : nullptr;
            a.epi.scale = c.scale; a.epi.inv = c.inv; a.epi.nrm = c.nrm;
            a.epi.v_gamma = nx.has_bn ? Vp(nx.gamma) : nullptr; a.epi.v_beta = nx.has_bn ? Vp(nx.beta) : nullptr;
            a.epi.pre = t[nx.tin].val; a.epi.post = t[nx.tout].val;
            // nobody else reads the pre-BN tangent, unless the tangent gamma-gradient of a FedAvg step does (sweep_tangent_backward)
            if (consumers_of(op.tout) == 1 && !want_tangent_G) a.out = nullptr;
            ++i;
          }
          BRE_LAUNCH(gemm(a));
          break;
        }
        case BRE_OP_BNACT: {
          if (op.has_bn && op.bn_train) {
            BnBuf& b = bn[op.bn_buffer];
            BnTrainArgs ta = bn_train_args(op);
            BRE_LAUNCH(launch_bn_train_tan_stats(ta, b.di_cm, b.di_cv, red_partials, red_counters, stream));
            ta.tres = op.res >= 0 ? t[op.res].tval : nullptr;
            ta.dst = t[op.tout].tval; ta.round_out = round_val(op.tout);
            BRE_LAUNCH(launch_bn_train_tan_fwd(ta, stream));
            break;
          }
          BnActTanFwdArgs a;
          a.P = Pout; a.C = to.C; a.has_bn = op.has_bn != 0; a.relu = op.relu != 0; a.bn = bn_consts(op);
          a.in = t[op.tin].val; a.out = t[op.tout].val;
          a.tin = t[op.tin].tval; a.tres = op.res >= 0 ? t[op.res].tval : nullptr;
          a.v_gamma = op.has_bn ? Vp(op.gamma) : nullptr; a.v_beta = op.has_bn ? Vp(op.beta) : nullptr;
          a.tout = t[op.tout].tval; a.round_out = round_val(op.tout);
          BRE_LAUNCH(launch_bnact_tan_fwd(a, stream));
          break;
        }
        case BRE_OP_MAXPOOL:
          BRE_LAUNCH(launch_maxpool_gather(t[op.tin].tval, pool_idx[i], t[op.tout].tval, pool_geom(op), stream));
          break;
        case BRE_OP_AVGPOOL: {
          const bre_tensor_desc& ti = td(op.tin);
          BRE_LAUNCH(launch_avgpool_fwd(t[op.tin].tval, t[op.tout].tval, ti.N, ti.H * ti.W, ti.C, stream));
          break;
        }
        case BRE_OP_POSADD:      // the candidate's tangent is zero: only the direction component of the positional table
          BRE_LAUNCH(launch_token_posadd(nullptr, Vp(op.w), t[op.tout].tval, to.N, to.C, op.S, stream));
          break;
        case BRE_OP_LAYERNORM:
          BRE_LAUNCH(launch_token_layernorm(2, t[op.tin].val, t[op.tin].tval, nullptr, nullptr, Wp(op.gamma), Wp(op.beta), Vp(op.gamma),
                                            Vp(op.beta), op.eps, to.N, to.C, tok_a[i], t[op.tout].tval, 0, stream));
          break;
        case BRE_OP_ATTENTION:
          BRE_LAUNCH(launch_token_attention(2, t[op.tin].val, t[op.tin].tval, nullptr, nullptr, to.N / op.S, op.S, op.R, to.C / op.R, tok_a[i],
                                            tok_b[i], t[op.tout].tval, 0, stream));
          break;
        default: break;
      }
    }
    return 0;
  }

  // DeepInversion statistics of every BN input of this forward pass: one batched launch pair (layers.cu) + per-layer finalisation
  StatSlot* di_stat_slots = nullptr;
  double* di_layer_values = nullptr;
  int di_stat_blocks = 0, di_stat_groups = 0;
  bool di_batched = false, di_tables_built = false;
  int build_di_tables() {
    if (di_tables_built) return 0;
    di_tables_built = true;
    if (cfg.di_scale <= 0.f || n_di == 0) return 0;
    BRE_TRY(alloc(&di_layer_values, n_di));
    static const bool env = [] { const char* e = getenv("BRE_DI_BATCHED"); return e ? atoi(e) != 0 : true; }();
    if (!env || ms_steps > 0) return 0;
    std::vector<StatSlot> table;
    int blocks = 0, groups = 0;
    // one launch covers every BN input: ~16 blocks per SM in total, dealt to the tensors in proportion to their size
    double all_elems = 0.0;
    for (const bre_op_desc& op : ops)
      if (op.kind == BRE_OP_BNACT && op.has_bn) { const bre_tensor_desc& ti = td(op.tin); all_elems += (double)ti.N * ti.H * ti.W * ti.C; }
    for (const bre_op_desc& op : ops) {
      if (op.kind != BRE_OP_BNACT || !op.has_bn) continue;
      const bre_tensor_desc& ti = td(op.tin);
      StatSlot sl;
      memset(&sl, 0, sizeof(sl));
      const double share = (double)ti.N * ti.H * ti.W * ti.C / all_elems;
      long long target = (long long)(share * 16.0 * kNumSMs + 0.5);
      if (target < 4) target = 4;
      if (!channel_stats_plan((long long)ti.N * ti.H * ti.W, ti.C, &sl, target)) return 0;   // odd channel count somewhere: per-layer kernels
      BnBuf& b = bn[op.bn_buffer];
      sl.x = t[op.tin].val; sl.mean = b.di_mean; sl.var = b.di_var;
      BRE_TRY(alloc(&sl.partials, (long long)sl.slabs * sl.Cpad * 2));
      sl.first_block = blocks; sl.first_group = groups;
      blocks += sl.cg * sl.slabs; groups += (ti.C + 255) / 256;
      table.push_back(sl);
    }
    if (table.empty()) return 0;
    BRE_TRY(alloc(&di_stat_slots, (long long)table.size()));
    BRE_CUDA_CHECK(cudaMemcpy(di_stat_slots, table.data(), table.size() * sizeof(StatSlot), cudaMemcpyHostToDevice));
    di_stat_blocks = blocks; di_stat_groups = groups; di_batched = true;
    return 0;
  }
  int deep_inversion_stats() {
    if (cfg.di_scale <= 0.f || n_di == 0) return 0;
    if (di_batched) {
      BRE_LAUNCH(launch_channel_stats_batched(di_stat_slots, n_di, di_stat_blocks, di_stat_groups, stream));
    } else {
      for (size_t i = 0; i < ops.size(); ++i) {
        const bre_op_desc& op = ops[i];
        if (op.kind != BRE_OP_BNACT || !op.has_bn) continue;
        const bre_tensor_desc& ti = td(op.tin);
        BnBuf& b = bn[op.bn_buffer];
        BRE_LAUNCH(launch_channel_stats(t[op.tin].val, (long long)ti.N * ti.H * ti.W, ti.C, b.di_mean, b.di_var, red_partials,
                                        red_counters, stream));
      }
    }
    BRE_LAUNCH(launch_di_finalize(di_layers_dev, n_di, di_layer_values, sc, stream));
    return 0;
  }

  int sweep_tangent_backward() {
    bool forked = false;
    const bre_tensor_desc& lt = td(logits);
    if (seq_len > 0) BRE_LAUNCH(launch_token_ce_tan_bwd(p, t[logits].tval, lt.N, classes(), lt.C, seq_len, t[logits].td, stream));
    else BRE_LAUNCH(launch_ce_tan_bwd(p, t[logits].tval, lt.N, lt.C, t[logits].td, stream));
    const bool di = cfg.di_scale > 0.f && n_di > 0;
    for (int i = (int)ops.size() - 1; i >= 0; --i) {
      const bre_op_desc& op = ops[i];
      const bre_tensor_desc& to = td(op.tout);
      const long long Pout = (long long)to.N * to.H * to.W;
      switch (op.kind) {
        case BRE_OP_CONV:
        case BRE_OP_LINEAR: {
          const bool cols = use_stem_cols((size_t)i);
          GemmArgs a = cols ? stem_geom(op) : conv_geom(op);
          a.mode = GEMM_DGRAD;
          a.nsrc = 2;
          a.act[0] = t[op.tout].td; a.wgt[0] = cols ? Wcol : Wg(op);
          a.act[1] = t[op.tout].d; a.wgt[1] = cols ? Vcol : Vg(op);
          a.out = cols ? dcol : (op.tin == 0 ? t[0].td : t[op.tin].td);
          a.accumulate = op.tin == 0 ? 0 : op.acc_in;
          BRE_LAUNCH(gemm(a));
          if (cols) BRE_TRY(stem_fold(op, t[0].td));
          if (want_tangent_G) {
            // tangent of the weight gradient: wgrad(a, delta_dot) + wgrad(a_dot, delta)   (a_dot = 0 for the candidate)
            GemmArgs w = cols ? stem_geom(op) : conv_geom(op);
            w.mode = GEMM_WGRAD;
            w.act[0] = cols ? xcol : t[op.tin].val; w.wgt[0] = t[op.tout].td;
            if (op.tin != 0) { w.nsrc = 2; w.act[1] = t[op.tin].tval; w.wgt[1] = t[op.tout].d; }
            w.out = cols ? Gcol : Gp(op.w);
            cudaStream_t wst = stream;
            if (overlap_wgrad && side != nullptr) {
              BRE_CUDA_CHECK(cudaEventRecord(ev_fork[i], stream));
              BRE_CUDA_CHECK(cudaStreamWaitEvent(side, ev_fork[i], 0));
              w.ws = ws2; w.counters = gemm_counters2;
              wst = side;
              forked = true;
            }
            BRE_LAUNCH(gemm_on(w, wst));
            if (cols) BRE_LAUNCH(launch_stem_pad_rows(Gcol, Gp(op.w), to.C, op.R * op.S * td(op.tin).C, stem_Kp, true, false, wst));
            if (op.b >= 0)
              BRE_LAUNCH(launch_channel_sum(t[op.tout].td, Pout, to.C, Gp(op.b), wst == side ? red_partials2 : red_partials,
                                            wst == side ? red_counters2 : red_counters, wst));
          }
          if ((int)i == feat_op && cfg.feat_scale > 0.f && feat_measured != nullptr)
            BRE_LAUNCH(launch_feature_reg(t[op.tin].val, feat_measured, t[op.tin].td, feat_numel, cfg.feat_scale, sc, stream));
          break;
        }
        case BRE_OP_BNACT: {
          if (op.has_bn && op.bn_train) {
            BnBuf& b = bn[op.bn_buffer];
            BnTrainArgs ta = bn_train_args(op);
            BRE_LAUNCH(launch_bn_train_tanbwd_stats(ta, b.tb1, b.tb2, red_partials, red_counters, stream));
            ta.dst = t[op.tin].td; ta.acc = op.acc_in != 0; ta.round_out = round_d(op.tin);
            ta.dres = op.res >= 0 ? t[op.res].td : nullptr; ta.acc_res = op.acc_res != 0;
            BRE_LAUNCH(launch_bn_train_tan_bwd(ta, stream));
            break;
          }
          BnActTanBwdArgs a;
          a.P = Pout; a.C = to.C; a.has_bn = op.has_bn != 0; a.relu = op.relu != 0; a.bn = bn_consts(op);
          a.in = t[op.tin].val; a.out = t[op.tout].val; a.tdout = t[op.tout].td; a.dout = t[op.tout].d;
          a.v_gamma = op.has_bn ? Vp(op.gamma) : nullptr;
          a.di_cm = a.di_cv = a.di_mean = nullptr;
          if (di && op.has_bn) { const BnBuf& b = bn[op.bn_buffer]; a.di_cm = b.di_cm; a.di_cv = b.di_cv; a.di_mean = b.di_mean; }
          a.tdin = t[op.tin].td; a.acc_in = op.acc_in != 0; a.round_din = round_d(op.tin);
          a.tdres = op.res >= 0 ? t[op.res].td : nullptr; a.acc_res = op.acc_res != 0;
          a.tin = nullptr; a.tg_gamma = a.tg_beta = nullptr; a.partials = red_partials; a.counters = red_counters;
          if (want_tangent_G && op.has_bn) { a.tin = t[op.tin].tval; a.tg_gamma = Gp(op.gamma); a.tg_beta = Gp(op.beta); }
          BRE_LAUNCH(launch_bnact_tan_bwd(a, stream));
          break;
        }
        case BRE_OP_MAXPOOL:
          BRE_LAUNCH(launch_maxpool_bwd(t[op.tout].td, pool_idx[i], t[op.tin].td, op.acc_in != 0, pool_geom(op), stream));
          break;
        case BRE_OP_AVGPOOL: {
          const bre_tensor_desc& ti = td(op.tin);
          BRE_LAUNCH(launch_avgpool_bwd(t[op.tout].td, t[op.tin].td, op.acc_in != 0, ti.N, ti.H * ti.W, ti.C, stream));
          break;
        }
        case BRE_OP_POSADD:      // d objective / d candidate = tangent delta of the embedded sequence
          BRE_CUDA_CHECK(cudaMemcpyAsync(t[0].td, t[op.tout].td, (size_t)to.N * to.C * sizeof(float), cudaMemcpyDeviceToDevice, stream));
          break;
        case BRE_OP_LAYERNORM:
          BRE_LAUNCH(launch_token_layernorm(3, t[op.tin].val, t[op.tout].td, t[op.tout].d, t[op.tin].tval, Wp(op.gamma), Wp(op.beta),
                                            Vp(op.gamma), nullptr, op.eps, to.N, to.C, tok_a[i], t[op.tin].td, op.acc_in != 0, stream));
          break;
        case BRE_OP_ATTENTION:
          BRE_LAUNCH(launch_token_attention(3, t[op.tin].val, t[op.tout].td, t[op.tout].d, t[op.tin].tval, to.N / op.S, op.S, op.R, to.C / op.R,
                                            tok_a[i], tok_b[i], t[op.tin].td, op.acc_in != 0, stream));
          break;
        default: break;
      }
    }
    if (forked) {
      BRE_CUDA_CHECK(cudaEventRecord(ev_join, side));
      BRE_CUDA_CHECK(cudaStreamWaitEvent(stream, ev_join, 0));
    }
    return 0;
  }

  // ---- multi-step (FedAvg) ------------------------------------------------------------------------------------
  void bind_step(int k) {
    const StepBufs& b = ms_bufs[k];
    for (size_t i = 1; i < t.size(); ++i) { t[i].val = b.val[i]; t[i].d = b.d[i]; }
    pool_idx = b.idx;
    p = b.p; loss_n = b.loss_n; labels = b.labels;
    W = ms_W[k]; Wt = ms_Wt[k];
    for (int j = 0; j < n_bn_layers; ++j) { bn[j].scale = b.bn_scale[j]; bn[j].shift = b.bn_shift[j]; }
    t[0].val = x + ms_offset[k];
    t[0].td = gradx_step;
  }
  int refresh_bn_constants(int k);   // defined below (needs a kernel)

  int multistep_forward() {
    for (int k = 0; k < ms_steps; ++k) {
      bind_step(k);
      if (k > 0) BRE_TRY(refresh_bn_constants(k));
      BRE_TRY(sweep_forward());
      BRE_TRY(sweep_backward());
      // W_{k+1} = W_k - lr * grad (:63-66).  The matched "gradient" W_K - W_0 (:69) is accumulated directly,
      // D_{k+1} = D_k - lr * grad, instead of being formed as a difference of two nearly equal parameter vectors.
      BRE_LAUNCH(launch_axpby(ms_W[k], G, -ms_lr, ms_W[k + 1], P_pad, stream));
      if (tc_round()) BRE_LAUNCH(launch_round_tf32(ms_W[k + 1], ms_Wt[k + 1], P_pad, stream));
      if (k == 0) BRE_CUDA_CHECK(cudaMemsetAsync(ms_D, 0, P_pad * sizeof(float), stream));
      BRE_LAUNCH(launch_axpby(ms_D, G, -ms_lr, ms_D, P_pad, stream));
    }
    return 0;
  }

  int evaluate_multistep() {
    BRE_CUDA_CHECK(cudaMemsetAsync(gradx, 0, nx * sizeof(float), stream));
    BRE_TRY(multistep_forward());
    const float mv = cfg.objective == BRE_OBJ_MASKED_COSINE ? cfg.mask_value : -1.f;
    BRE_LAUNCH(launch_match_reduce(ms_D, g, chunk_w, P_pad, mv, cfg.objective, cfg.obj_scale, cfg.tag_scale, cfg.angular_fudge, true, sc,
                                   dpartials, dcounter, stream));
    BRE_LAUNCH(launch_make_v(ms_D, g, chunk_w, V, P_pad, mv, sc, stream));          // adjoint of W_K
    BRE_TRY(refresh_Vt());
    const long long nstep = t[0].numel;
    for (int k = ms_steps - 1; k >= 0; --k) {
      bind_step(k);
      want_tangent_G = k > 0;
      BRE_TRY(sweep_tangent_forward());
      const int rc = sweep_tangent_backward();
      want_tangent_G = false;
      if (rc != 0) return rc;
      // d Phi / d x_k = -lr * d/d eps grad_x L(x_k, W_{k-1} + eps u_k)
      BRE_LAUNCH(launch_axpy(gradx_step, gradx + ms_offset[k], -ms_lr, nstep, stream));
      if (k > 0) {
        BRE_LAUNCH(launch_axpby(V, G, -ms_lr, V, P_pad, stream));                     // u_{k-1} = u_k - lr * H_k u_k
        BRE_TRY(refresh_Vt());
      }
    }
    bind_step(0);
    BRE_TRY(priors());
    return 0;
  }

  int priors() {
    const bool image_terms = cfg.tv_scale != 0.f || cfg.norm_scale != 0.f;
    if (!image_terms) {
      if (cfg.orthogonality != 0)
        BRE_LAUNCH(launch_orthogonality(input_x(), input_grad(), xN, (long long)xC * xH * xW, true, sc, dpartials, dcounter, stream));
      return 0;
    }
    if (xC != 3) {   // TV on non-RGB candidates is rejected at creation (the reference's grouped conv raises as well)
      BRE_LAUNCH(launch_norm_prior(input_x(), input_grad(), nx, cfg.norm_scale, cfg.norm_p, 1, sc, dpartials, dcounter, stream));
      if (cfg.orthogonality != 0)
        BRE_LAUNCH(launch_orthogonality(input_x(), input_grad(), xN, (long long)xC * xH * xW, false, sc, dpartials, dcounter, stream));
      return 0;
    }
    PriorArgs a;
    a.x = input_x(); a.grad = input_grad(); a.N = xN; a.H = xH; a.W = xW; a.accumulate = 1;
    a.tv_scale = cfg.tv_scale; a.p = cfg.tv_inner_exp; a.q = cfg.tv_outer_exp; a.eps = cfg.tv_eps;
    a.double_opponents = cfg.tv_double_opponents; a.norm_scale = cfg.norm_scale; a.norm_p = cfg.norm_p;
    BRE_LAUNCH(launch_image_priors(a, sc, dpartials, dcounter, stream));
    if (cfg.orthogonality != 0)
      BRE_LAUNCH(launch_orthogonality(input_x(), input_grad(), xN, (long long)xC * xH * xW, false, sc, dpartials, dcounter, stream));
    return 0;
  }

  // objective + its gradient w.r.t. the candidate (closure body, optimization_based_attack.py:146-165)
  int evaluate() {
    if (ms_steps > 0) return evaluate_multistep();
    if (aug_on) BRE_TRY(augment_forward());
    BRE_TRY(sweep_forward());
    BRE_TRY(sweep_backward());
    BRE_TRY(reduce_objective(cfg.objective, cfg.obj_scale, cfg.mask_value, true));
    // direction v and (tensor-core back end) its TF32 shadow in one pass; chunks of tensor-core conv weights get the shadow only
    BRE_TRY(build_chunk_modes());
    BRE_LAUNCH(launch_make_v(G, g, chunk_w, V, P_pad, cfg.objective == BRE_OBJ_MASKED_COSINE ? cfg.mask_value : -1.f, sc, stream,
                             tc_round() ? Vt : nullptr, tc_round() ? chunk_mode : nullptr));
    serialize_next_launch();   // v is complete and visible before anything of the tangent sweeps starts
    v_settled = true;
    BRE_TRY(sweep_tangent_forward());
    BRE_TRY(deep_inversion_stats());
    BRE_TRY(sweep_tangent_backward());
    v_settled = false;
    BRE_TRY(priors());
    if (aug_on && aug_diff) BRE_TRY(augment_pull());
    return 0;
  }

  StepArgs step_args() const {
    StepArgs a;
    a.x = x; a.m = m; a.v = v; a.best = best; a.grad = gradx; a.grad_task = (need_task_grad() && !task_grad_folded()) ? gradx_task : nullptr;
    a.lr_table = lr_table; a.n_lr = n_lr; a.lo = lo; a.hi = hi; a.n = nx; a.C = xC; a.HW = xH * xW; a.cfg = cfg;
    return a;
  }

  int label_gradient_on_device() {   // d(objective)/d(label logits) of the evaluation that just ran -> label_grad
    const bre_tensor_desc& lt = td(logits);
    if (seq_len > 0)
      BRE_LAUNCH(launch_token_label_grad(t[logits].val, p, t[logits].tval, lt.N, classes(), lt.C, seq_len, cfg.task_regularization, label_grad, stream));
    else
      BRE_LAUNCH(launch_ce_label_grad(t[logits].val, p, t[logits].tval, lt.N, lt.C, cfg.task_regularization, label_grad, stream));
    BRE_LAUNCH(launch_softmax_chain(soft_q_buf, label_grad, lt.N, classes(), stream));
    return 0;
  }

  // one iteration of the joint attacker: both leaves post-processed separately (:164-186), one optimiser steps both (:108),
  // box projection on the data only (:111-114), best-so-far of both on the pre-step objective (:115-118)
  int iteration_joint() {
    const bre_tensor_desc& lt = td(logits);
    BRE_LAUNCH(launch_row_softmax(ell, soft_q_buf, lt.N, classes(), stream));
    soft_q = soft_q_buf;
    BRE_TRY(evaluate());
    BRE_TRY(label_gradient_on_device());
    StepArgs a = step_args();
    if (cfg.grad_clip >= 0.f) BRE_LAUNCH(launch_grad_norm(a, sc, dpartials, dcounter, stream));
    BRE_LAUNCH(launch_pixel_step(a, sc, stream));
    StepArgs b = a;
    b.x = ell; b.m = ell_m; b.v = ell_v; b.best = ell_best; b.grad = label_grad; b.grad_task = nullptr;
    b.n = n_ell; b.C = 1; b.HW = 1; b.cfg.boxed = 0; b.cfg.noise_seed = cfg.noise_seed + 0x9E3779B97F4A7C15ull;
    if (cfg.grad_clip >= 0.f) BRE_LAUNCH(launch_grad_norm(b, sc, dpartials, dcounter, stream));
    BRE_LAUNCH(launch_pixel_step(b, sc, stream));
    BRE_LAUNCH(launch_commit(sc, history, lr_cap, value_task_reg(), stream));
    return 0;
  }

  int iteration() {
    if (joint) return iteration_joint();
    BRE_TRY(evaluate());
    StepArgs a = step_args();
    if (cfg.grad_clip >= 0.f) BRE_LAUNCH(launch_grad_norm(a, sc, dpartials, dcounter, stream));
    BRE_LAUNCH(launch_pixel_step(a, sc, stream));
    BRE_LAUNCH(launch_commit(sc, history, lr_cap, value_task_reg(), stream));
    return 0;
  }
};

namespace {
__global__ void bn_refresh_kernel(const bre_engine::BnPrep* table, const float* W) {
  pdl_prologue();
  const bre_engine::BnPrep e = table[blockIdx.x];
  for (int c = threadIdx.x; c < e.C; c += blockDim.x) {
    const float gmm = W[e.gamma_off + c];
    e.scale[c] = gmm * e.inv[c];
    e.shift[c] = fmaf(gmm, e.nrm[c], W[e.beta_off + c]);
  }
}
}  // namespace

int bre_engine::refresh_bn_constants(int k) {
  if (n_bn_layers == 0) return 0;
  BRE_KLAUNCH(bn_refresh_kernel, n_bn_layers, 128, 0, stream, (const BnPrep*)ms_bnprep_dev[k], (const float*)ms_W[k]);
  ++launch_count;
  return 0;
}

// ======================================================================================================
// C ABI
// ======================================================================================================
extern "C" {

const char* bre_last_error(void) { return bre::g_last_error.c_str(); }
const char* bre_version(void) { return "breaching_b200 0.1.0 (sm_100a)"; }

int bre_engine_create(const bre_tensor_desc* tensors, int32_t n_tensors, const bre_op_desc* ops, int32_t n_ops,
                      const bre_param_desc* params, int32_t n_params, int32_t logits_tensor, const bre_attack_cfg* cfg,
                      int32_t device, bre_engine** out) {
  if (!tensors || !ops || !params || !cfg || !out || n_tensors < 2 || n_ops < 1) { set_error("bre_engine_create: bad arguments"); return BRE_ERR_INVALID; }
  BRE_CUDA_CHECK(cudaSetDevice(device));
  bre_engine* e = new bre_engine();
  e->device = device;
  e->cfg = *cfg;
  e->logits = logits_tensor;
  e->ops.assign(ops, ops + n_ops);
  auto fail = [&](int rc) { bre_engine_destroy(e); return rc; };
  if (cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking) != cudaSuccess) { set_error("stream creation failed"); return fail(BRE_ERR_CUDA); }

  // ---- validate the program -------------------------------------------------------------------
  int consumers0 = 0;
  int n_bn = 0;
  for (int i = 0; i < n_ops; ++i) {
    const bre_op_desc& op = ops[i];
    if (op.tin < 0 || op.tin >= n_tensors || op.tout <= 0 || op.tout >= n_tensors || op.res >= n_tensors) { set_error("op tensor id out of range"); return fail(BRE_ERR_INVALID); }
    if (op.tin == 0 || op.res == 0) {
      ++consumers0;
      if (op.res == 0 || (op.kind != BRE_OP_CONV && op.kind != BRE_OP_LINEAR && op.kind != BRE_OP_POSADD)) { set_error("the candidate must feed exactly one conv/linear/posadd layer"); return fail(BRE_ERR_UNSUPPORTED); }
    }
    if (op.kind == BRE_OP_BNACT && op.has_bn) n_bn = op.bn_buffer + 1 > n_bn ? op.bn_buffer + 1 : n_bn;
    if ((op.kind == BRE_OP_CONV || op.kind == BRE_OP_LINEAR) && (op.w < 0 || op.w >= n_params)) { set_error("conv/linear without weight"); return fail(BRE_ERR_INVALID); }
    if (op.kind == BRE_OP_LINEAR) e->feat_op = i;
  }
  if (consumers0 != 1) { set_error("the candidate must feed exactly one layer"); return fail(BRE_ERR_UNSUPPORTED); }
  if (cfg->tv_scale != 0.f && tensors[0].C != 3) {
    // regularizers.py:109-128 builds a grouped 3x3 convolution for 3 colour channels; on anything else it raises
    set_error("total_variation needs a 3-channel image candidate");
    return fail(BRE_ERR_UNSUPPORTED);
  }
  if (tensors[logits_tensor].H * tensors[logits_tensor].W != 1) { set_error("logits must be [N, classes]"); return fail(BRE_ERR_INVALID); }

  // ---- parameter arenas -------------------------------------------------------------------------
  long long off = 0;
  e->params.resize(n_params);
  for (int i = 0; i < n_params; ++i) {
    e->params[i].desc = params[i];
    e->params[i].off = off;
    // perm NONE: d0 = allocated element count when larger than numel (zero tail: rows of a padded vocabulary)
    const long long alloc_n = (params[i].perm == BRE_PERM_NONE && params[i].d0 > params[i].numel) ? params[i].d0 : params[i].numel;
    off += ((alloc_n + kChunk - 1) / kChunk) * kChunk;
    if (params[i].numel > e->max_param) e->max_param = params[i].numel;
  }
  e->P_pad = off;
  int rc = 0;
  rc |= e->alloc(&e->W, off); rc |= e->alloc(&e->g, off); rc |= e->alloc(&e->G, off); rc |= e->alloc(&e->V, off);
  rc |= e->alloc(&e->Wt, off); rc |= e->alloc(&e->Vt, off);
  rc |= e->alloc(&e->chunk_w, off / kChunk);
  // ---- activations ---------------------------------------------------------------------------------
  e->t.resize(n_tensors);
  int maxC = 1;
  for (int i = 0; i < n_tensors; ++i) {
    e->t[i].desc = tensors[i];
    e->t[i].numel = (long long)tensors[i].N * tensors[i].C * tensors[i].H * tensors[i].W;
    if (e->t[i].numel > e->max_tensor) e->max_tensor = e->t[i].numel;
    if (tensors[i].C > maxC) maxC = tensors[i].C;
    if (i == 0) continue;
    rc |= e->alloc(&e->t[i].val, e->t[i].numel); rc |= e->alloc(&e->t[i].d, e->t[i].numel);
    rc |= e->alloc(&e->t[i].tval, e->t[i].numel); rc |= e->alloc(&e->t[i].td, e->t[i].numel);
  }
  rc |= e->alloc(&e->stage, e->max_param > e->max_tensor ? e->max_param : e->max_tensor);
  const bre_tensor_desc& x0 = tensors[0];
  e->xN = x0.N; e->xC = x0.C; e->xH = x0.H; e->xW = x0.W; e->nx = e->t[0].numel;
  rc |= e->alloc(&e->x, e->nx); rc |= e->alloc(&e->gradx, e->nx); rc |= e->alloc(&e->gradx_task, e->nx);
  rc |= e->alloc(&e->m, e->nx); rc |= e->alloc(&e->v, e->nx); rc |= e->alloc(&e->best, e->nx);
  rc |= e->alloc(&e->lo, x0.C); rc |= e->alloc(&e->hi, x0.C);
  e->t[0].val = e->x; e->t[0].d = e->gradx_task; e->t[0].td = e->gradx; e->t[0].tval = nullptr;
  const bre_tensor_desc& lt = tensors[logits_tensor];
  rc |= e->alloc(&e->p, (long long)lt.N * lt.C); rc |= e->alloc(&e->loss_n, lt.N); rc |= e->alloc(&e->labels, lt.N);
  e->n_labels = lt.N;
  rc |= e->alloc(&e->sc, 1);
  // ---- per-op buffers --------------------------------------------------------------------------------
  e->pool_idx.assign(n_ops, nullptr);
  e->tok_a.assign(n_ops, nullptr);
  e->tok_b.assign(n_ops, nullptr);
  for (int i = 0; i < n_ops; ++i) {
    const bre_op_desc& op = ops[i];
    if (op.kind == BRE_OP_LAYERNORM) rc |= e->alloc(&e->tok_a[i], 2LL * tensors[op.tin].N);
    if (op.kind == BRE_OP_ATTENTION || op.kind == BRE_OP_POSADD) {
      if (op.S < 1 || tensors[op.tin].N % op.S != 0) { set_error("token op: rows must be a multiple of seq_len"); return fail(BRE_ERR_INVALID); }
      e->seq_len = op.S;
    }
    if (op.kind == BRE_OP_ATTENTION) {
      const long long np = (long long)(tensors[op.tin].N / op.S) * op.R * op.S * op.S;
      rc |= e->alloc(&e->tok_a[i], np);
      rc |= e->alloc(&e->tok_b[i], np);
    }
  }
  e->bn.resize(n_bn);
  for (int i = 0; i < n_ops; ++i) {
    const bre_op_desc& op = ops[i];
    if (op.kind == BRE_OP_MAXPOOL) rc |= e->alloc(&e->pool_idx[i], e->t[op.tout].numel);
    if (op.kind == BRE_OP_BNACT && op.has_bn) {
      BnBuf& b = e->bn[op.bn_buffer];
      b.C = tensors[op.tout].C;
      float** ptrs[] = {&b.rm, &b.rv, &b.scale, &b.shift, &b.inv, &b.nrm, &b.di_mean, &b.di_var, &b.di_cm, &b.di_cv, &b.tb1, &b.tb2};
      for (float** pp : ptrs) rc |= e->alloc(pp, b.C);
    }
  }
  // ---- column path of the candidate-fed convolution (tensor-core back end; stem_cols.cu) -------------------------------------
  for (int i = 0; i < n_ops; ++i) {
    const bre_op_desc& op = ops[i];
    if (op.kind == BRE_OP_CONV && op.tin == 0 && tensors[0].C <= 4 && tensors[op.tout].C % 64 == 0 && op.R * op.S <= 64) {
      e->stem_op = i;
      e->stem_Kp = ((op.R * op.S * tensors[0].C + 63) / 64) * 64;
      const long long M = (long long)tensors[op.tout].N * tensors[op.tout].H * tensors[op.tout].W;
      rc |= e->alloc(&e->xcol, M * e->stem_Kp); rc |= e->alloc(&e->dcol, M * e->stem_Kp);
      rc |= e->alloc(&e->Wcol, (long long)tensors[op.tout].C * e->stem_Kp); rc |= e->alloc(&e->Vcol, (long long)tensors[op.tout].C * e->stem_Kp);
      rc |= e->alloc(&e->Gcol, (long long)tensors[op.tout].C * e->stem_Kp);
    }
  }
  // ---- side stream for the weight-gradient GEMMs ----------------------------------------------------------
  if (cudaStreamCreateWithFlags(&e->side, cudaStreamNonBlocking) != cudaSuccess) { set_error("stream creation failed"); return fail(BRE_ERR_CUDA); }
  e->ev_fork.assign(n_ops, nullptr);
  for (int i = 0; i < n_ops; ++i)
    if ((ops[i].kind == BRE_OP_CONV || ops[i].kind == BRE_OP_LINEAR) &&
        cudaEventCreateWithFlags(&e->ev_fork[i], cudaEventDisableTiming) != cudaSuccess) { set_error("event creation failed"); return fail(BRE_ERR_CUDA); }
  if (cudaEventCreateWithFlags(&e->ev_join, cudaEventDisableTiming) != cudaSuccess) { set_error("event creation failed"); return fail(BRE_ERR_CUDA); }
  // ---- scratch ---------------------------------------------------------------------------------------
  e->ws_tiles = 1024;
  rc |= e->alloc(&e->ws, (long long)e->ws_tiles * IG_BM * IG_BN);
  rc |= e->alloc(&e->gemm_counters, 1 << 16);
  long long redp = (long long)(16384 > 2 * maxC + 64 ? 16384 : 2 * maxC + 64) * 2 * 2;
  if (redp < kSlabPartialFloats) redp = kSlabPartialFloats;
  rc |= e->alloc(&e->red_partials, redp);
  rc |= e->alloc(&e->red_counters, maxC / 32 + 8);
  rc |= e->alloc(&e->ws2, (long long)e->ws_tiles * IG_BM * IG_BN);
  rc |= e->alloc(&e->gemm_counters2, 1 << 16);
  rc |= e->alloc(&e->red_partials2, redp);
  rc |= e->alloc(&e->red_counters2, maxC / 32 + 8);
  long long tv_blocks = (long long)((x0.W + 31) / 32) * ((x0.H + 7) / 8) * x0.N;
  long long dp = tv_blocks * 2 > kMatchMaxBlocks * 5 ? tv_blocks * 2 : kMatchMaxBlocks * 5;
  if (dp < kNumSMs * 8) dp = kNumSMs * 8;
  rc |= e->alloc(&e->dpartials, dp);
  rc |= e->alloc(&e->dcounter, 4);
  if (rc != 0) return fail(BRE_ERR_CUDA);
  // DeepInversion layer table
  bool any_bn_train = false;
  for (int i = 0; i < n_ops; ++i) any_bn_train = any_bn_train || (ops[i].kind == BRE_OP_BNACT && ops[i].has_bn && ops[i].bn_train);
  if (any_bn_train && (cfg->di_scale > 0.f || cfg->feat_scale > 0.f)) {
    set_error("DeepInversion / feature priors need running statistics: not available with train-mode BatchNorm");
    return fail(BRE_ERR_UNSUPPORTED);
  }
  if (cfg->di_scale > 0.f && n_bn > 0) {
    std::vector<DiLayer> layers;
    bool first = true;
    for (int i = 0; i < n_ops; ++i) {
      const bre_op_desc& op = ops[i];
      if (op.kind != BRE_OP_BNACT || !op.has_bn) continue;
      const BnBuf& b = e->bn[op.bn_buffer];
      const bre_tensor_desc& ti = tensors[op.tin];
      DiLayer L{b.di_mean, b.di_var, b.rm, b.rv, b.di_cm, b.di_cv, b.C, (float)((long long)ti.N * ti.H * ti.W),
                cfg->di_scale * (first ? cfg->di_first_bn_multiplier : 1.f)};
      first = false;
      layers.push_back(L);
    }
    e->n_di = (int)layers.size();
    if (e->alloc(&e->di_layers_dev, (long long)layers.size()) != 0) return fail(BRE_ERR_CUDA);
    if (cudaMemcpy(e->di_layers_dev, layers.data(), layers.size() * sizeof(DiLayer), cudaMemcpyHostToDevice) != cudaSuccess) { set_error("DI table upload failed"); return fail(BRE_ERR_CUDA); }
  }
  // default box = unbounded; chunk weights = 1
  {
    std::vector<float> ones((size_t)(off / kChunk), 1.f);
    if (!ones.empty() && cudaMemcpy(e->chunk_w, ones.data(), ones.size() * sizeof(float), cudaMemcpyHostToDevice) != cudaSuccess) { set_error("chunk weight upload failed"); return fail(BRE_ERR_CUDA); }
  }
  *out = e;
  return BRE_OK;
}

void bre_engine_destroy(bre_engine* e) {
  if (!e) return;
  cudaSetDevice(e->device);
  if (e->stream) cudaStreamSynchronize(e->stream);
  if (e->side) cudaStreamSynchronize(e->side);
  if (e->exec) cudaGraphExecDestroy(e->exec);
  for (cudaEvent_t ev : e->ev_fork) if (ev) cudaEventDestroy(ev);
  if (e->ev_join) cudaEventDestroy(e->ev_join);
  if (e->side) cudaStreamDestroy(e->side);
  for (void* p : e->allocs) cudaFree(p);
  if (e->stream) cudaStreamDestroy(e->stream);
  delete e;
}

static int load_list(bre_engine* e, const float* const* ptrs, int32_t n, float* arena) {
  if (n != (int)e->params.size()) { set_error("parameter count mismatch"); return BRE_ERR_INVALID; }
  for (int i = 0; i < n; ++i) {
    const ParamInfo& pi = e->params[i];
    if (!ptrs[i]) { set_error("null parameter pointer"); return BRE_ERR_INVALID; }
    if (pi.desc.perm == BRE_PERM_NONE) {
      BRE_CUDA_CHECK(cudaMemcpyAsync(arena + pi.off, ptrs[i], pi.desc.numel * sizeof(float), cudaMemcpyDefault, e->stream));
    } else {
      BRE_CUDA_CHECK(cudaMemcpyAsync(e->stage, ptrs[i], pi.desc.numel * sizeof(float), cudaMemcpyDefault, e->stream));
      BRE_TRY(launch_permute(e->stage, arena + pi.off, pi.desc.d0, pi.desc.d1, pi.desc.d2, false, e->stream));
    }
  }
  return 0;
}

int bre_engine_load_model(bre_engine* e, const float* const* params, int32_t n_params, const float* const* bn_mean,
                          const float* const* bn_var, int32_t n_bn) {
  if (!e || !params) { set_error("bre_engine_load_model: bad arguments"); return BRE_ERR_INVALID; }
  BRE_CUDA_CHECK(cudaSetDevice(e->device));
  if (n_bn != (int)e->bn.size()) { set_error("BN buffer count mismatch"); return BRE_ERR_INVALID; }
  BRE_TRY(load_list(e, params, n_params, e->W));
  for (int j = 0; j < n_bn; ++j) {
    BnBuf& b = e->bn[j];
    BRE_CUDA_CHECK(cudaMemcpyAsync(b.rm, bn_mean[j], b.C * sizeof(float), cudaMemcpyDefault, e->stream));
    BRE_CUDA_CHECK(cudaMemcpyAsync(b.rv, bn_var[j], b.C * sizeof(float), cudaMemcpyDefault, e->stream));
  }
  for (const bre_op_desc& op : e->ops) {
    if (op.kind != BRE_OP_BNACT || !op.has_bn) continue;
    BnBuf& b = e->bn[op.bn_buffer];
    BRE_TRY(launch_bn_prepare(e->Wp(op.gamma), e->Wp(op.beta), b.rm, b.rv, op.eps, b.C, b.scale, b.shift, b.inv, b.nrm, e->stream));
  }
  BRE_CUDA_CHECK(cudaStreamSynchronize(e->stream));
  BRE_TRY(launch_round_tf32(e->W, e->Wt, e->P_pad, e->stream));   // GEMM-operand shadow (used by the tcgen05 back end)
  if (e->stem_op >= 0) {   // zero-padded [Co][Kp] copy of the stem weight (TF32-rounded like Wt when the tensor-core back end rounds)
    const bre_op_desc& op = e->ops[e->stem_op];
    BRE_TRY(launch_stem_pad_rows(e->Wp(op.w), e->Wcol, e->td(op.tout).C, op.R * op.S * e->td(op.tin).C, e->stem_Kp, false, e->tc_round_env, e->stream));
  }
  e->model_loaded = true;
  return BRE_OK;
}

int bre_engine_load_targets(bre_engine* e, const float* const* grads, int32_t n_params, const float* tensor_weights,
                            const int64_t* labels, int32_t n_labels, const float* mean, const float* stdv, int32_t n_channels) {
  if (!e || !grads || !labels) { set_error("bre_engine_load_targets: bad arguments"); return BRE_ERR_INVALID; }
  BRE_CUDA_CHECK(cudaSetDevice(e->device));
  if (n_labels != e->n_labels) { set_error("label count must equal the batch size"); return BRE_ERR_INVALID; }
  BRE_TRY(load_list(e, grads, n_params, e->g));
  BRE_CUDA_CHECK(cudaMemcpyAsync(e->labels, labels, n_labels * sizeof(int64_t), cudaMemcpyDefault, e->stream));
  std::vector<float> cw((size_t)(e->P_pad / kChunk), 1.f);
  if (tensor_weights) {
    std::vector<float> tw(n_params);
    BRE_CUDA_CHECK(cudaMemcpy(tw.data(), tensor_weights, n_params * sizeof(float), cudaMemcpyDefault));
    for (int i = 0; i < n_params; ++i) {
      const long long c0 = e->params[i].off / kChunk, c1 = c0 + (e->params[i].desc.numel + kChunk - 1) / kChunk;
      for (long long c = c0; c < c1; ++c) cw[(size_t)c] = tw[i];
    }
  }
  if (!cw.empty()) BRE_CUDA_CHECK(cudaMemcpyAsync(e->chunk_w, cw.data(), cw.size() * sizeof(float), cudaMemcpyHostToDevice, e->stream));
  std::vector<float> lo(e->xC, -std::numeric_limits<float>::infinity()), hi(e->xC, std::numeric_limits<float>::infinity());
  if (mean && stdv) {
    if (n_channels != e->xC) { set_error("mean/std channel count mismatch"); return BRE_ERR_INVALID; }
    std::vector<float> mh(n_channels), sh(n_channels);
    BRE_CUDA_CHECK(cudaMemcpy(mh.data(), mean, n_channels * sizeof(float), cudaMemcpyDefault));
    BRE_CUDA_CHECK(cudaMemcpy(sh.data(), stdv, n_channels * sizeof(float), cudaMemcpyDefault));
    for (int c = 0; c < n_channels; ++c) { lo[c] = -mh[c] / sh[c]; hi[c] = (1.f - mh[c]) / sh[c]; }  // base_attack.py:117-118 box
  } else {
    for (int c = 0; c < e->xC; ++c) { lo[c] = -0.f / 1.f; hi[c] = 1.f; }  // dm = 0, ds = 1 (base_attack.py:57)
  }
  BRE_CUDA_CHECK(cudaMemcpyAsync(e->lo, lo.data(), lo.size() * sizeof(float), cudaMemcpyHostToDevice, e->stream));
  BRE_CUDA_CHECK(cudaMemcpyAsync(e->hi, hi.data(), hi.size() * sizeof(float), cudaMemcpyHostToDevice, e->stream));
  BRE_CUDA_CHECK(cudaStreamSynchronize(e->stream));
  e->targets_loaded = true;
  return BRE_OK;
}

int bre_engine_load_feature_targets(bre_engine* e, const float* measured, int64_t numel) {
  if (!e || !measured || e->feat_op < 0) { set_error("bre_engine_load_feature_targets: no linear layer / bad arguments"); return BRE_ERR_INVALID; }
  BRE_CUDA_CHECK(cudaSetDevice(e->device));
  const long long expect = e->t[e->ops[e->feat_op].tin].numel;
  if (numel != expect) { set_error("feature target size mismatch"); return BRE_ERR_INVALID; }
  if (!e->feat_measured) BRE_TRY(e->alloc(&e->feat_measured, numel));
  e->feat_numel = numel;
  BRE_CUDA_CHECK(cudaMemcpy(e->feat_measured, measured, numel * sizeof(float), cudaMemcpyDefault));
  e->graph_ready = false;
  return BRE_OK;
}

int bre_engine_load_soft_labels(bre_engine* e, const float* probabilities, int64_t numel) {
  if (!e) return BRE_ERR_INVALID;
  BRE_CUDA_CHECK(cudaSetDevice(e->device));
  e->graph_ready = false;
  if (probabilities == nullptr) { e->soft_q = nullptr; return BRE_OK; }   // back to index labels
  const bre_tensor_desc& lt = e->td(e->logits);
  if (numel != (int64_t)lt.N * e->classes()) { set_error("bre_engine_load_soft_labels: expected N x classes probabilities"); return BRE_ERR_INVALID; }
  if (e->ms_steps > 0) { set_error("soft labels are not supported together with local steps"); return BRE_ERR_UNSUPPORTED; }
  if (!e->soft_q_buf) { BRE_TRY(e->alloc(&e->soft_q_buf, numel)); BRE_TRY(e->alloc(&e->label_grad, numel)); }
  BRE_CUDA_CHECK(cudaMemcpyAsync(e->soft_q_buf, probabilities, numel * sizeof(float), cudaMemcpyDefault, e->stream));
  e->soft_q = e->soft_q_buf;
  return BRE_OK;
}

int bre_engine_set_labels(bre_engine* e, const int64_t* labels, int32_t n_labels) {
  if (!e || !labels) return BRE_ERR_INVALID;
  BRE_CUDA_CHECK(cudaSetDevice(e->device));
  if (n_labels != e->td(e->logits).N) { set_error("bre_engine_set_labels: one label per row of the logits expected"); return BRE_ERR_INVALID; }
  BRE_CUDA_CHECK(cudaMemcpyAsync(e->labels, labels, n_labels * sizeof(int64_t), cudaMemcpyDefault, e->stream));
  return BRE_OK;
}

int bre_engine_label_gradient(bre_engine* e, float* grad_out) {
  if (!e || !grad_out) return BRE_ERR_INVALID;
  if (!e->soft_q) { set_error("bre_engine_label_gradient: no soft labels loaded"); return BRE_ERR_STATE; }
  BRE_CUDA_CHECK(cudaSetDevice(e->device));
  const bre_tensor_desc& lt = e->td(e->logits);
  if (e->seq_len > 0)
    BRE_TRY(launch_token_label_grad(e->t[e->logits].val, e->p, e->t[e->logits].tval, lt.N, e->classes(), lt.C, e->seq_len,
                                    e->cfg.task_regularization, e->label_grad, e->stream));
  else
    BRE_TRY(launch_ce_label_grad(e->t[e->logits].val, e->p, e->t[e->logits].tval, lt.N, lt.C, e->cfg.task_regularization, e->label_grad,
                                 e->stream));
  BRE_CUDA_CHECK(cudaMemcpyAsync(grad_out, e->label_grad, (size_t)lt.N * e->classes() * sizeof(float), cudaMemcpyDefault, e->stream));
  BRE_CUDA_CHECK(cudaStreamSynchronize(e->stream));
  return BRE_OK;
}

int bre_engine_set_local_steps(bre_engine* e, int32_t total_images, int32_t steps, float lr, const int64_t* labels) {
  if (!e || steps < 1 || total_images < 1 || !labels) { set_error("bre_engine_set_local_steps: bad arguments"); return BRE_ERR_INVALID; }
  if (!e->model_loaded) { set_error("load the model first"); return BRE_ERR_STATE; }
  if (e->ms_steps > 0) { set_error("local steps already configured"); return BRE_ERR_STATE; }
  for (const bre_op_desc& o : e->ops)
    if (o.kind == BRE_OP_BNACT && o.has_bn && o.bn_train) { set_error("multi-step updates with train-mode BatchNorm are not implemented"); return BRE_ERR_UNSUPPORTED; }
  if (e->cfg.task_regularization != 0.f || e->cfg.di_scale > 0.f || e->cfg.feat_scale > 0.f) {
    set_error("task regularisation / DeepInversion / feature priors are not implemented for multi-step updates "
              "(the reference crashes on the latter two, SURVEY.md section 0 fact 9)");
    return BRE_ERR_UNSUPPORTED;
  }
  BRE_CUDA_CHECK(cudaSetDevice(e->device));
  const int dps = e->t[0].desc.N;
  const long long per_image = (long long)e->xC * e->xH * e->xW;
  e->ms_offset.resize(steps);
  int seen = 0;
  for (int k = 0; k < steps; ++k) {               // objectives.py:56-58
    if (seen + dps > total_images) { set_error("a local step would read a ragged candidate slice (unsupported)"); return BRE_ERR_UNSUPPORTED; }
    e->ms_offset[k] = seen * per_image;
    seen = (seen + dps) % total_images;
  }
  // candidate-sized state for all images
  e->xN = total_images;
  e->nx = total_images * per_image;
  int rc = 0;
  rc |= e->alloc(&e->x, e->nx); rc |= e->alloc(&e->gradx, e->nx); rc |= e->alloc(&e->gradx_task, e->nx);
  rc |= e->alloc(&e->m, e->nx); rc |= e->alloc(&e->v, e->nx); rc |= e->alloc(&e->best, e->nx);
  rc |= e->alloc(&e->gradx_step, e->t[0].numel);
  rc |= e->alloc(&e->ms_D, e->P_pad);
  e->ms_W.assign(steps + 1, nullptr);
  e->ms_W[0] = e->W;
  e->ms_Wt.assign(steps + 1, nullptr);
  e->ms_Wt[0] = e->Wt;
  e->W0 = e->W;
  for (int k = 1; k <= steps; ++k) { rc |= e->alloc(&e->ms_W[k], e->P_pad); rc |= e->alloc(&e->ms_Wt[k], e->P_pad); }
  e->ms_bufs.resize(steps);
  e->n_bn_layers = (int)e->bn.size();
  e->ms_bnprep_dev.assign(steps, nullptr);
  const int nlab = e->n_labels;
  for (int k = 0; k < steps; ++k) {
    bre_engine::StepBufs& b = e->ms_bufs[k];
    b.val.assign(e->t.size(), nullptr); b.d.assign(e->t.size(), nullptr); b.idx.assign(e->ops.size(), nullptr);
    b.bn_scale.assign(e->bn.size(), nullptr); b.bn_shift.assign(e->bn.size(), nullptr);
    if (k == 0) {
      for (size_t i = 1; i < e->t.size(); ++i) { b.val[i] = e->t[i].val; b.d[i] = e->t[i].d; }
      b.idx = e->pool_idx; b.p = e->p; b.loss_n = e->loss_n; b.labels = e->labels;
      for (size_t j = 0; j < e->bn.size(); ++j) { b.bn_scale[j] = e->bn[j].scale; b.bn_shift[j] = e->bn[j].shift; }
    } else {
      for (size_t i = 1; i < e->t.size(); ++i) { rc |= e->alloc(&b.val[i], e->t[i].numel); rc |= e->alloc(&b.d[i], e->t[i].numel); }
      for (size_t i = 0; i < e->ops.size(); ++i)
        if (e->ops[i].kind == BRE_OP_MAXPOOL) rc |= e->alloc(&b.idx[i], e->t[e->ops[i].tout].numel);
      const bre_tensor_desc& lt = e->t[e->logits].desc;
      rc |= e->alloc(&b.p, (long long)lt.N * lt.C); rc |= e->alloc(&b.loss_n, lt.N); rc |= e->alloc(&b.labels, lt.N);
      for (size_t j = 0; j < e->bn.size(); ++j) { rc |= e->alloc(&b.bn_scale[j], e->bn[j].C); rc |= e->alloc(&b.bn_shift[j], e->bn[j].C); }
      std::vector<bre_engine::BnPrep> table;
      for (const bre_op_desc& op : e->ops) {
        if (op.kind != BRE_OP_BNACT || !op.has_bn) continue;
        const BnBuf& bb = e->bn[op.bn_buffer];
        table.push_back({(int)e->params[op.gamma].off, (int)e->params[op.beta].off, bb.C, bb.inv, bb.nrm, b.bn_scale[op.bn_buffer],
                         b.bn_shift[op.bn_buffer]});
      }
      rc |= e->alloc(&e->ms_bnprep_dev[k], (long long)table.size());
      if (rc == 0 && !table.empty())
        BRE_CUDA_CHECK(cudaMemcpy(e->ms_bnprep_dev[k], table.data(), table.size() * sizeof(bre_engine::BnPrep), cudaMemcpyHostToDevice));
    }
    if (rc != 0) return BRE_ERR_CUDA;
    BRE_CUDA_CHECK(cudaMemcpy(b.labels, labels + (long long)k * nlab, nlab * sizeof(int64_t), cudaMemcpyDefault));
  }
  e->ms_steps = steps;
  e->ms_lr = lr;
  e->bind_step(0);
  e->graph_ready = false;
  return BRE_OK;
}

static int reset_trial_state(bre_engine* e) {
  Scalars h;
  memset(&h, 0, sizeof(h));
  h.fmin = std::numeric_limits<double>::infinity();
  BRE_CUDA_CHECK(cudaMemcpyAsync(e->sc, &h, sizeof(h), cudaMemcpyHostToDevice, e->stream));
  BRE_CUDA_CHECK(cudaStreamSynchronize(e->stream));  // `h` is a stack object
  return 0;
}

int bre_engine_begin_trial(bre_engine* e, const float* candidate, const float* lr_table, int32_t n_lr) {
  if (!e || !candidate || !lr_table || n_lr <= 0) { set_error("bre_engine_begin_trial: bad arguments"); return BRE_ERR_INVALID; }
  if (!e->model_loaded || !e->targets_loaded) { set_error("load model and targets before beginning a trial"); return BRE_ERR_STATE; }
  BRE_CUDA_CHECK(cudaSetDevice(e->device));
  if (n_lr > e->lr_cap) {
    // (re)allocate schedule + history; device pointers baked into a captured graph change -> recapture
    BRE_TRY(e->alloc(&e->lr_table, n_lr));
    BRE_TRY(e->alloc(&e->history, n_lr));
    e->lr_cap = n_lr;
    e->graph_ready = false;
  }
  if (n_lr != e->n_lr) e->graph_ready = false;
  e->n_lr = n_lr;
  BRE_CUDA_CHECK(cudaMemcpyAsync(e->lr_table, lr_table, n_lr * sizeof(float), cudaMemcpyDefault, e->stream));
  BRE_CUDA_CHECK(cudaMemcpyAsync(e->x, candidate, e->nx * sizeof(float), cudaMemcpyDefault, e->stream));
  BRE_CUDA_CHECK(cudaMemcpyAsync(e->best, e->x, e->nx * sizeof(float), cudaMemcpyDeviceToDevice, e->stream));
  BRE_CUDA_CHECK(cudaMemsetAsync(e->m, 0, e->nx * sizeof(float), e->stream));
  BRE_CUDA_CHECK(cudaMemsetAsync(e->v, 0, e->nx * sizeof(float), e->stream));
  BRE_TRY(reset_trial_state(e));
  if (e->joint) { e->joint = false; e->graph_ready = false; }
  e->trial_begun = true;
  return BRE_OK;
}

int bre_engine_begin_joint_trial(bre_engine* e, const float* candidate, const float* label_logits, int64_t n_label_elems,
                                 const float* lr_table, int32_t n_lr) {
  if (!e || !label_logits) { set_error("bre_engine_begin_joint_trial: bad arguments"); return BRE_ERR_INVALID; }
  const bre_tensor_desc& lt = e->td(e->logits);
  if (n_label_elems != (int64_t)lt.N * e->classes()) { set_error("bre_engine_begin_joint_trial: expected N x classes label logits"); return BRE_ERR_INVALID; }
  if (e->ms_steps > 0) { set_error("joint optimisation is not supported together with local steps"); return BRE_ERR_UNSUPPORTED; }
  BRE_TRY(bre_engine_begin_trial(e, candidate, lr_table, n_lr));
  BRE_CUDA_CHECK(cudaSetDevice(e->device));
  if (!e->soft_q_buf) { BRE_TRY(e->alloc(&e->soft_q_buf, n_label_elems)); BRE_TRY(e->alloc(&e->label_grad, n_label_elems)); }
  if (!e->ell) {
    BRE_TRY(e->alloc(&e->ell, n_label_elems)); BRE_TRY(e->alloc(&e->ell_m, n_label_elems));
    BRE_TRY(e->alloc(&e->ell_v, n_label_elems)); BRE_TRY(e->alloc(&e->ell_best, n_label_elems));
    e->n_ell = n_label_elems;
  }
  BRE_CUDA_CHECK(cudaMemcpyAsync(e->ell, label_logits, n_label_elems * sizeof(float), cudaMemcpyDefault, e->stream));
  BRE_CUDA_CHECK(cudaMemcpyAsync(e->ell_best, e->ell, n_label_elems * sizeof(float), cudaMemcpyDeviceToDevice, e->stream));
  BRE_CUDA_CHECK(cudaMemsetAsync(e->ell_m, 0, n_label_elems * sizeof(float), e->stream));
  BRE_CUDA_CHECK(cudaMemsetAsync(e->ell_v, 0, n_label_elems * sizeof(float), e->stream));
  BRE_CUDA_CHECK(cudaStreamSynchronize(e->stream));
  e->soft_q = e->soft_q_buf;
  e->joint = true;
  e->graph_ready = false;
  return BRE_OK;
}

int bre_engine_get_joint_labels(bre_engine* e, int32_t best, float* out) {
  if (!e || !out || !e->ell) { set_error("bre_engine_get_joint_labels: no joint trial"); return BRE_ERR_STATE; }
  BRE_CUDA_CHECK(cudaSetDevice(e->device));
  BRE_CUDA_CHECK(cudaMemcpyAsync(out, best ? e->ell_best : e->ell, e->n_ell * sizeof(float), cudaMemcpyDefault, e->stream));
  BRE_CUDA_CHECK(cudaStreamSynchronize(e->stream));
  return BRE_OK;
}

int bre_engine_run(bre_engine* e, int32_t n_iters) {
  if (!e || n_iters < 0) { set_error("bre_engine_run: bad arguments"); return BRE_ERR_INVALID; }
  if (!e->trial_begun) { set_error("bre_engine_begin_trial must be called first"); return BRE_ERR_STATE; }
  BRE_CUDA_CHECK(cudaSetDevice(e->device));
  if (!e->use_graph) {
    BRE_TRY(e->build_chunk_modes());
    BRE_TRY(e->build_bn_slots());
    BRE_TRY(e->build_di_tables());
    for (int i = 0; i < n_iters; ++i) { e->launch_count = 0; BRE_TRY(e->iteration()); e->launches_per_iter = e->launch_count; }
    return BRE_OK;
  }
  if (!e->graph_ready) {
    BRE_TRY(e->build_chunk_modes());   // host -> device tables: must exist before the capture starts
    BRE_TRY(e->build_bn_slots());
    BRE_TRY(e->build_di_tables());
    if (e->exec) { cudaGraphExecDestroy(e->exec); e->exec = nullptr; }
    cudaGraph_t graph = nullptr;
    BRE_CUDA_CHECK(cudaStreamBeginCapture(e->stream, cudaStreamCaptureModeThreadLocal));
    e->launch_count = 0;
    const int rc = e->iteration();
    cudaError_t err = cudaStreamEndCapture(e->stream, &graph);
    if (rc != 0) { if (graph) cudaGraphDestroy(graph); return rc; }
    if (err != cudaSuccess) { set_error(std::string("graph capture failed: ") + cudaGetErrorString(err)); return BRE_ERR_CUDA; }
    e->launches_per_iter = e->launch_count;
    err = cudaGraphInstantiate(&e->exec, graph, 0);
    cudaGraphDestroy(graph);
    if (err != cudaSuccess) { set_error(std::string("graph instantiation failed: ") + cudaGetErrorString(err)); return BRE_ERR_CUDA; }
    e->graph_ready = true;
  }
  for (int i = 0; i < n_iters; ++i) BRE_CUDA_CHECK(cudaGraphLaunch(e->exec, e->stream));
  return BRE_OK;
}

int bre_engine_run_timed(bre_engine* e, int32_t n_iters, float* ms_out) {
  if (!e || !ms_out) return BRE_ERR_INVALID;
  BRE_CUDA_CHECK(cudaSetDevice(e->device));
  cudaEvent_t ev0, ev1;
  BRE_CUDA_CHECK(cudaEventCreate(&ev0));
  BRE_CUDA_CHECK(cudaEventCreate(&ev1));
  BRE_CUDA_CHECK(cudaStreamSynchronize(e->stream));
  BRE_CUDA_CHECK(cudaEventRecord(ev0, e->stream));
  int rc = bre_engine_run(e, n_iters);
  if (rc == 0 && cudaEventRecord(ev1, e->stream) != cudaSuccess) rc = BRE_ERR_CUDA;
  if (rc == 0 && cudaEventSynchronize(ev1) != cudaSuccess) rc = BRE_ERR_CUDA;
  if (rc == 0 && cudaEventElapsedTime(ms_out, ev0, ev1) != cudaSuccess) rc = BRE_ERR_CUDA;
  cudaEventDestroy(ev0);
  cudaEventDestroy(ev1);
  if (rc == BRE_ERR_CUDA) set_error("timed run failed");
  return rc;
}

int bre_engine_sync(bre_engine* e) {
  if (!e) return BRE_ERR_INVALID;
  BRE_CUDA_CHECK(cudaSetDevice(e->device));
  BRE_CUDA_CHECK(cudaStreamSynchronize(e->stream));
  return BRE_OK;
}

static int read_scalars(bre_engine* e, Scalars* h) {
  BRE_CUDA_CHECK(cudaSetDevice(e->device));
  BRE_CUDA_CHECK(cudaMemcpyAsync(h, e->sc, sizeof(Scalars), cudaMemcpyDeviceToHost, e->stream));
  BRE_CUDA_CHECK(cudaStreamSynchronize(e->stream));
  return 0;
}

int bre_engine_status(bre_engine* e, int32_t* iters_recorded, int32_t* stopped, double* min_objective, double* last_task_loss) {
  if (!e) return BRE_ERR_INVALID;
  Scalars h;
  BRE_TRY(read_scalars(e, &h));
  if (iters_recorded) *iters_recorded = h.recorded;
  if (stopped) *stopped = h.stopped;
  if (min_objective) *min_objective = h.fmin;
  if (last_task_loss) *last_task_loss = h.task_loss;
  return BRE_OK;
}

int bre_engine_read_history(bre_engine* e, float* out_host, int32_t n) {
  if (!e || !out_host || n < 0 || n > e->lr_cap) { set_error("bre_engine_read_history: bad arguments"); return BRE_ERR_INVALID; }
  BRE_CUDA_CHECK(cudaSetDevice(e->device));
  BRE_CUDA_CHECK(cudaMemcpyAsync(out_host, e->history, n * sizeof(float), cudaMemcpyDeviceToHost, e->stream));
  BRE_CUDA_CHECK(cudaStreamSynchronize(e->stream));
  return BRE_OK;
}

static int copy_out(bre_engine* e, const float* src, float* out) {
  if (!e || !out) return BRE_ERR_INVALID;
  BRE_CUDA_CHECK(cudaSetDevice(e->device));
  BRE_CUDA_CHECK(cudaMemcpyAsync(out, src, e->nx * sizeof(float), cudaMemcpyDefault, e->stream));
  BRE_CUDA_CHECK(cudaStreamSynchronize(e->stream));
  return BRE_OK;
}
int bre_engine_get_best(bre_engine* e, float* out) { return copy_out(e, e ? e->best : nullptr, out); }
int bre_engine_get_candidate(bre_engine* e, float* out) { return copy_out(e, e ? e->x : nullptr, out); }

int bre_engine_score(bre_engine* e, const float* candidate, int32_t scoring, double* out_score) {
  if (!e || !candidate || !out_score) return BRE_ERR_INVALID;
  if (scoring != BRE_OBJ_EUCLIDEAN && scoring != BRE_OBJ_COSINE) { set_error("scoring must be euclidean or cosine-similarity"); return BRE_ERR_UNSUPPORTED; }
  if (!e->model_loaded || !e->targets_loaded) { set_error("load model and targets first"); return BRE_ERR_STATE; }
  BRE_CUDA_CHECK(cudaSetDevice(e->device));
  BRE_CUDA_CHECK(cudaMemcpyAsync(e->x, candidate, e->nx * sizeof(float), cudaMemcpyDefault, e->stream));
  if (e->ms_steps > 0) {
    BRE_TRY(e->multistep_forward());
    BRE_TRY(launch_match_reduce(e->ms_D, e->g, e->chunk_w, e->P_pad, -1.f, scoring, 1.0f, e->cfg.tag_scale, e->cfg.angular_fudge, true,
                                e->sc, e->dpartials, e->dcounter, e->stream));
    e->bind_step(0);
  } else {
    e->t[0].val = e->x;                 // scores are taken on the candidate itself, not on an augmented view (:191-204)
    int rc = e->sweep_forward();
    if (rc == 0) rc = e->sweep_backward();
    e->bind_input();
    if (rc != 0) return rc;
    BRE_TRY(e->reduce_objective(scoring, 1.0f, -1.f, true));
  }
  Scalars h;
  BRE_TRY(read_scalars(e, &h));
  const double s = (double)(float)h.match;
  *out_score = isfinite(s) ? s : std::numeric_limits<double>::infinity();
  return BRE_OK;
}

int bre_engine_objective_and_gradient(bre_engine* e, const float* candidate, double* objective, float* grad_out) {
  if (!e || !candidate) return BRE_ERR_INVALID;
  if (!e->model_loaded || !e->targets_loaded) { set_error("load model and targets first"); return BRE_ERR_STATE; }
  BRE_CUDA_CHECK(cudaSetDevice(e->device));
  BRE_CUDA_CHECK(cudaMemcpyAsync(e->x, candidate, e->nx * sizeof(float), cudaMemcpyDefault, e->stream));
  e->launch_count = 0;
  BRE_TRY(e->build_chunk_modes());
  BRE_TRY(e->build_bn_slots());
  BRE_TRY(e->build_di_tables());
  BRE_TRY(e->evaluate());
  if (e->need_task_grad() && !e->task_grad_folded()) BRE_TRY(launch_axpy(e->gradx_task, e->gradx, e->cfg.task_regularization, e->nx, e->stream));
  Scalars h;
  BRE_TRY(read_scalars(e, &h));
  if (objective) {
    double phi = h.match + h.tv + h.norm + h.di + h.feat;
    if (e->value_task_reg() != 0.f) phi += (double)e->value_task_reg() * h.task_loss;
    *objective = phi;
  }
  if (grad_out) BRE_TRY(copy_out(e, e->gradx, grad_out));
  return BRE_OK;
}

// ---- user-side update production (cases/users.py:148-169) and plain forward (analysis/analysis.py:66-69) ------------------
int bre_engine_forward(bre_engine* e, const float* data, float* logits_out) {
  if (!e || !data || !logits_out) { set_error("bre_engine_forward: bad arguments"); return BRE_ERR_INVALID; }
  if (!e->model_loaded) { set_error("load the model first"); return BRE_ERR_STATE; }
  if (e->ms_steps > 0) { set_error("bre_engine_forward: not available on a multi-step engine"); return BRE_ERR_UNSUPPORTED; }
  BRE_CUDA_CHECK(cudaSetDevice(e->device));
  BRE_CUDA_CHECK(cudaMemcpyAsync(e->x, data, e->nx * sizeof(float), cudaMemcpyDefault, e->stream));
  float* keep_q = e->soft_q;
  if (e->seq_len > 0 && e->soft_q == nullptr) {   // the token loss needs targets; forward-only callers have none
    const bre_tensor_desc& lt = e->td(e->logits);
    if (!e->soft_q_buf) { BRE_TRY(e->alloc(&e->soft_q_buf, (long long)lt.N * lt.C)); BRE_TRY(e->alloc(&e->label_grad, (long long)lt.N * lt.C)); }
    e->soft_q = e->soft_q_buf;
  }
  const int rc = e->sweep_forward();
  e->soft_q = keep_q;
  if (rc != 0) return rc;
  const bre_tensor_desc& lt = e->td(e->logits);
  BRE_CUDA_CHECK(cudaMemcpyAsync(logits_out, e->t[e->logits].val, (size_t)lt.N * lt.C * sizeof(float), cudaMemcpyDefault, e->stream));
  BRE_CUDA_CHECK(cudaStreamSynchronize(e->stream));
  return BRE_OK;
}

int bre_engine_param_gradients(bre_engine* e, const float* data, const int64_t* labels, int32_t n_labels, float* const* grads_out,
                               int32_t n_params, double* loss_out) {
  if (!e || !data || !labels || !grads_out) { set_error("bre_engine_param_gradients: bad arguments"); return BRE_ERR_INVALID; }
  if (!e->model_loaded) { set_error("load the model first"); return BRE_ERR_STATE; }
  if (e->ms_steps > 0 || e->seq_len > 0) { set_error("bre_engine_param_gradients: single-step vision programs only"); return BRE_ERR_UNSUPPORTED; }
  if (n_labels != e->n_labels || n_params != (int)e->params.size()) { set_error("bre_engine_param_gradients: label / parameter count mismatch"); return BRE_ERR_INVALID; }
  BRE_CUDA_CHECK(cudaSetDevice(e->device));
  BRE_CUDA_CHECK(cudaMemcpyAsync(e->x, data, e->nx * sizeof(float), cudaMemcpyDefault, e->stream));
  BRE_CUDA_CHECK(cudaMemcpyAsync(e->labels, labels, n_labels * sizeof(int64_t), cudaMemcpyDefault, e->stream));
  float* keep_q = e->soft_q;
  e->soft_q = nullptr;                         // index labels (users.py:152)
  int rc = e->sweep_forward();
  if (rc == 0) rc = e->sweep_backward();
  e->soft_q = keep_q;
  if (rc != 0) return rc;
  for (int i = 0; i < n_params; ++i) {
    const ParamInfo& pi = e->params[i];
    if (!grads_out[i]) { set_error("null output pointer"); return BRE_ERR_INVALID; }
    const float* src = e->G + pi.off;
    if (pi.desc.perm != BRE_PERM_NONE) {       // back to torch's OIHW / CHW-column layout
      BRE_TRY(launch_permute(src, e->stage, pi.desc.d0, pi.desc.d1, pi.desc.d2, true, e->stream));
      src = e->stage;
    }
    BRE_CUDA_CHECK(cudaMemcpyAsync(grads_out[i], src, pi.desc.numel * sizeof(float), cudaMemcpyDefault, e->stream));
  }
  Scalars h;
  BRE_TRY(read_scalars(e, &h));
  if (loss_out) *loss_out = h.task_loss;
  return BRE_OK;
}

int bre_engine_bn_batch_stats(bre_engine* e, int32_t bn_index, float* mean_out, float* var_out) {
  if (!e || !mean_out || !var_out || bn_index < 0 || bn_index >= (int)e->bn.size()) { set_error("bre_engine_bn_batch_stats: bad arguments"); return BRE_ERR_INVALID; }
  bool train = false;
  for (const bre_op_desc& op : e->ops) train = train || (op.kind == BRE_OP_BNACT && op.has_bn && op.bn_buffer == bn_index && op.bn_train);
  if (!train) { set_error("bre_engine_bn_batch_stats: this layer normalises with running statistics"); return BRE_ERR_STATE; }
  BRE_CUDA_CHECK(cudaSetDevice(e->device));
  const BnBuf& b = e->bn[bn_index];
  BRE_CUDA_CHECK(cudaMemcpyAsync(mean_out, b.di_mean, b.C * sizeof(float), cudaMemcpyDefault, e->stream));
  BRE_CUDA_CHECK(cudaMemcpyAsync(var_out, b.di_var, b.C * sizeof(float), cudaMemcpyDefault, e->stream));
  BRE_CUDA_CHECK(cudaStreamSynchronize(e->stream));
  return BRE_OK;
}

int bre_engine_set_augmentations(bre_engine* e, int32_t n_steps, const int32_t* kinds, const float* params, int32_t cs_enabled, float cs_shift,
                                 int32_t cs_circular, const float* cj_scale, const float* cj_shift, int32_t differentiable, uint64_t seed) {
  if (!e || n_steps < 0 || n_steps > AUG_MAX_STEPS || (n_steps > 0 && (!kinds || !params))) { set_error("bre_engine_set_augmentations: bad arguments"); return BRE_ERR_INVALID; }
  if (e->ms_steps > 0) { set_error("augmentations are not supported together with local steps"); return BRE_ERR_UNSUPPORTED; }
  if (e->xN > AUG_MAX_BATCH) { set_error("augmentations: batch too large"); return BRE_ERR_UNSUPPORTED; }
  BRE_CUDA_CHECK(cudaSetDevice(e->device));
  e->graph_ready = false;
  const bool any = n_steps > 0 || cs_enabled || cj_scale != nullptr;
  memset(&e->aug, 0, sizeof(e->aug));
  e->aug_on = any;
  e->aug_diff = any && differentiable != 0;
  if (any) {
    for (int s = 0; s < n_steps; ++s) {
      if (kinds[s] != AUG_SHIFT && kinds[s] != AUG_FLIP) { set_error("unknown augmentation step"); return BRE_ERR_INVALID; }
      e->aug.kind[s] = kinds[s]; e->aug.p0[s] = params[s];
    }
    e->aug.n_steps = n_steps; e->aug.cs_enabled = cs_enabled; e->aug.cs_shift = cs_shift; e->aug.cs_circular = cs_circular; e->aug.seed = seed;
    if (cs_enabled && e->xH != e->xW) { set_error("continuous_shift needs square images (the reference builds an S x S grid from shape[2])"); return BRE_ERR_UNSUPPORTED; }
    if (!e->x_aug) {
      BRE_TRY(e->alloc(&e->x_aug, e->nx)); BRE_TRY(e->alloc(&e->gradx_aug, e->nx)); BRE_TRY(e->alloc(&e->aug_tmp, e->nx));
      BRE_TRY(e->alloc(&e->aug_draws, 1));
      BRE_TRY(e->alloc(&e->cj_scale, (long long)e->xN * e->xC)); BRE_TRY(e->alloc(&e->cj_shift, (long long)e->xN * e->xC));
    }
    if (cj_scale != nullptr) {
      if (!cj_shift) { set_error("colour scale and shift go together"); return BRE_ERR_INVALID; }
      BRE_CUDA_CHECK(cudaMemcpyAsync(e->cj_scale, cj_scale, (size_t)e->xN * e->xC * sizeof(float), cudaMemcpyDefault, e->stream));
      BRE_CUDA_CHECK(cudaMemcpyAsync(e->cj_shift, cj_shift, (size_t)e->xN * e->xC * sizeof(float), cudaMemcpyDefault, e->stream));
      BRE_CUDA_CHECK(cudaStreamSynchronize(e->stream));
      e->aug.cj_scale = e->cj_scale; e->aug.cj_shift = e->cj_shift;
    }
  }
  e->bind_input();
  return BRE_OK;
}

int bre_engine_last_augmentation(bre_engine* e, int32_t* o1, int32_t* o2, float* sx, float* sy) {
  if (!e || !e->aug_draws) { set_error("bre_engine_last_augmentation: no augmentations configured"); return BRE_ERR_STATE; }
  BRE_CUDA_CHECK(cudaSetDevice(e->device));
  AugDraws h;
  BRE_CUDA_CHECK(cudaMemcpyAsync(&h, e->aug_draws, sizeof(h), cudaMemcpyDeviceToHost, e->stream));
  BRE_CUDA_CHECK(cudaStreamSynchronize(e->stream));
  for (int s = 0; s < AUG_MAX_STEPS; ++s) { if (o1) o1[s] = h.o1[s]; if (o2) o2[s] = h.o2[s]; }
  for (int n = 0; n < e->xN && n < AUG_MAX_BATCH; ++n) { if (sx) sx[n] = h.sx[n]; if (sy) sy[n] = h.sy[n]; }
  return BRE_OK;
}

int bre_engine_last_terms(bre_engine* e, double* terms6) {
  if (!e || !terms6) return BRE_ERR_INVALID;
  Scalars h;
  BRE_TRY(read_scalars(e, &h));
  terms6[0] = h.match; terms6[1] = h.task_loss; terms6[2] = h.tv; terms6[3] = h.norm; terms6[4] = h.di; terms6[5] = h.feat;
  return BRE_OK;
}

int bre_engine_debug_param(bre_engine* e, int32_t which, int32_t index, float* out_host) {
  if (!e || !out_host || index < 0 || index >= (int)e->params.size() || which < 0 || which > 3) return BRE_ERR_INVALID;
  BRE_CUDA_CHECK(cudaSetDevice(e->device));
  const float* arenas[4] = {e->G, e->V, e->W, e->g};
  const ParamInfo& pi = e->params[index];
  const float* src = arenas[which] + pi.off;
  if (pi.desc.perm != BRE_PERM_NONE) {
    BRE_TRY(launch_permute(src, e->stage, pi.desc.d0, pi.desc.d1, pi.desc.d2, true, e->stream));
    src = e->stage;
  }
  BRE_CUDA_CHECK(cudaMemcpyAsync(out_host, src, pi.desc.numel * sizeof(float), cudaMemcpyDeviceToHost, e->stream));
  BRE_CUDA_CHECK(cudaStreamSynchronize(e->stream));
  return BRE_OK;
}

int bre_engine_debug_tensor(bre_engine* e, int32_t which, int32_t tensor, float* out_host) {
  if (!e || !out_host || tensor < 0 || tensor >= (int)e->t.size() || which < 0 || which > 3) return BRE_ERR_INVALID;
  BRE_CUDA_CHECK(cudaSetDevice(e->device));
  const TensorBuf& tb = e->t[tensor];
  const float* bufs[4] = {tb.val, tb.d, tb.tval, tb.td};
  const float* src = bufs[which];
  if (!src) { set_error("tensor has no such buffer"); return BRE_ERR_INVALID; }
  if (tensor != 0) {
    BRE_TRY(launch_permute(src, e->stage, tb.desc.N, tb.desc.C, tb.desc.H * tb.desc.W, true, e->stream));
    src = e->stage;
  }
  BRE_CUDA_CHECK(cudaMemcpyAsync(out_host, src, tb.numel * sizeof(float), cudaMemcpyDeviceToHost, e->stream));
  BRE_CUDA_CHECK(cudaStreamSynchronize(e->stream));
  return BRE_OK;
}

int bre_engine_launches_per_iteration(bre_engine* e, int32_t* out) {
  if (!e || !out) return BRE_ERR_INVALID;
  *out = e->launches_per_iter;
  return BRE_OK;
}

int bre_engine_set_option(bre_engine* e, const char* name, int64_t value) {
  if (!e || !name) return BRE_ERR_INVALID;
  const std::string n(name);
  if (n == "use_graph") { e->use_graph = value != 0; e->graph_ready = false; return BRE_OK; }
  if (n == "pdl") { bre::set_pdl(value != 0); e->graph_ready = false; return BRE_OK; }
  if (n == "overlap_wgrad") { e->overlap_wgrad = value != 0; e->graph_ready = false; return BRE_OK; }
  if (n == "fuse_bnact") { e->fuse_bnact = value != 0; e->graph_ready = false; return BRE_OK; }
  if (n == "precise_first" || n == "precise_last") {
    (n == "precise_first" ? e->precise_first : e->precise_last) = (int)value;
    e->precise_op.clear(); e->rnd_val.clear(); e->rnd_d.clear(); e->chunk_mode_ready = false; e->graph_ready = false;
    return BRE_OK;
  }
  if (n == "logits_valid") {
    if (value < 1 || value > e->td(e->logits).C) { set_error("logits_valid must be in [1, logits columns]"); return BRE_ERR_INVALID; }
    if (e->soft_q_buf != nullptr) { set_error("logits_valid must be set before soft labels are loaded"); return BRE_ERR_STATE; }
    e->logits_valid = (int)value; e->graph_ready = false; return BRE_OK;
  }
  if (n == "gemm_backend") {
    if (value != 0 && value != 1) { set_error("gemm_backend must be 0 (simt) or 1 (tcgen05)"); return BRE_ERR_INVALID; }
    e->gemm_backend = (int)value; e->graph_ready = false; e->chunk_mode_ready = false; return BRE_OK;
  }
  set_error("unknown option " + n);
  return BRE_ERR_INVALID;
}

// ---- stand-alone kernels --------------------------------------------------------------------------
int bre_match_reduce(const float* G, const float* g, const float* chunk_weights, int64_t n, float mask_value,
                     double* sums5_host, void* stream) {
  if (!G || !g || n <= 0) { set_error("bre_match_reduce: bad arguments"); return BRE_ERR_INVALID; }
  cudaStream_t s = (cudaStream_t)stream;
  static thread_local Scalars* sc = nullptr;
  static thread_local double* partials = nullptr;
  static thread_local int* counter = nullptr;
  if (!sc) {
    BRE_TRY(dev_alloc(&sc, 1));
    BRE_TRY(dev_alloc(&partials, (long long)kMatchMaxBlocks * 5));
    BRE_TRY(dev_alloc(&counter, 1));
  }
  BRE_TRY(launch_match_reduce(G, g, chunk_weights, n, mask_value, BRE_OBJ_COSINE, 1.f, 0.f, 0.f, false, sc, partials, counter, s));
  if (sums5_host == nullptr) return BRE_OK;  // launch only (lets callers time / graph-capture the bare kernel)
  Scalars h;
  BRE_CUDA_CHECK(cudaMemcpyAsync(&h, sc, sizeof(h), cudaMemcpyDeviceToHost, s));
  BRE_CUDA_CHECK(cudaStreamSynchronize(s));
  sums5_host[0] = h.dot; sums5_host[1] = h.nG; sums5_host[2] = h.ng; sums5_host[3] = h.sq; sums5_host[4] = h.l1w;
  return BRE_OK;
}

int bre_total_variation(const float* x, float* grad, int32_t N, int32_t H, int32_t W, float scale, float inner_exp,
                        float outer_exp, float eps, int32_t double_opponents, int32_t accumulate, double* value_host,
                        void* stream) {
  if (!x || !grad || N <= 0 || H <= 0 || W <= 0) { set_error("bre_total_variation: bad arguments (x: [N, 3, H, W], three colour channels)"); return BRE_ERR_INVALID; }
  cudaStream_t s = (cudaStream_t)stream;
  Scalars* sc = nullptr; double* partials = nullptr; int* counter = nullptr;
  const long long blocks = (long long)((W + 31) / 32) * ((H + 7) / 8) * N;
  BRE_TRY(dev_alloc(&sc, 1)); BRE_TRY(dev_alloc(&partials, blocks * 2)); BRE_TRY(dev_alloc(&counter, 1));
  PriorArgs a;
  a.x = x; a.grad = grad; a.N = N; a.H = H; a.W = W; a.accumulate = accumulate; a.tv_scale = scale; a.p = inner_exp;
  a.q = outer_exp; a.eps = eps; a.double_opponents = double_opponents; a.norm_scale = 0.f; a.norm_p = 2.f;
  int rc = launch_image_priors(a, sc, partials, counter, s);
  Scalars h;
  if (rc == 0 && cudaMemcpyAsync(&h, sc, sizeof(h), cudaMemcpyDeviceToHost, s) != cudaSuccess) rc = BRE_ERR_CUDA;
  if (rc == 0 && cudaStreamSynchronize(s) != cudaSuccess) rc = BRE_ERR_CUDA;
  cudaFree(sc); cudaFree(partials); cudaFree(counter);
  if (rc == 0 && value_host) *value_host = h.tv;
  return rc;
}

int bre_conv_gemm(int32_t mode, int32_t backend, const float* a, const float* w, const float* a2, const float* w2, float* out,
                  int32_t N, int32_t H, int32_t W, int32_t Ci, int32_t Co, int32_t R, int32_t S, int32_t stride, int32_t pad,
                  void* stream) {
  if (!a || !w || !out || mode < 0 || mode > 2) { set_error("bre_conv_gemm: bad arguments"); return BRE_ERR_INVALID; }
  cudaStream_t s = (cudaStream_t)stream;
  GemmArgs g;
  memset(&g, 0, sizeof(g));
  g.mode = mode;
  g.g = ConvGeom{N, H, W, Ci, (H + 2 * pad - R) / stride + 1, (W + 2 * pad - S) / stride + 1, Co, R, S, stride, pad};
  g.nsrc = (a2 && w2) ? 2 : 1;
  g.act[0] = a; g.wgt[0] = w; g.act[1] = a2; g.wgt[1] = w2;
  g.x_sN = (long long)H * W * Ci; g.x_sP = Ci; g.x_sC = 1;
  g.out = out;
  static thread_local float* ws = nullptr;
  static thread_local int* counters = nullptr;
  if (!ws) { BRE_TRY(dev_alloc(&ws, 1024LL * IG_BM * IG_BN)); BRE_TRY(dev_alloc(&counters, 1 << 16)); }
  g.ws = ws; g.counters = counters; g.ws_tiles = 1024;
  if (linear_tall_supported(g)) return launch_linear_tall(g, s) == 0 ? BRE_OK : BRE_ERR_CUDA;   // the engine's dispatch rule (gemm_on)
  if (backend == 1) {
    if (!igemm_tc_supported(g)) { set_error("tcgen05 back end does not cover this shape"); return BRE_ERR_UNSUPPORTED; }
    return launch_igemm_tc(g, s);
  }
  if (backend == 2 && linear_small_preferred(g)) return launch_linear_small(g, s) == 0 ? BRE_OK : BRE_ERR_CUDA;
  if (backend == 2 && igemm_tc_supported(g)) return launch_igemm_tc(g, s);  // the engine's own dispatch rule
  return launch_igemm_simt(g, s);
}

}  // extern "C"
