// C ABI of libmpg_b200.so (include/mpg_b200.h): handle, weight packing, launches.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <vector>

#include "mlp_kernels.cuh"
#include "model_kernels.cuh"
#include "tc_rollout.cuh"
#include "replay.cuh"

using namespace mpg;

namespace {

struct NetStore {
  float* flat = nullptr;   // Keras order W1|b1|W2|b2|..|WL|bL|Wout|bout (natural layouts)
  float* W1p = nullptr;
  float* Wp = nullptr;     // [L - 1][H][H]: the hidden -> hidden kernels W2..WL, packed columns (none at L = 1)
  float* WTp = nullptr;    // [L - 1][H][H]: their transposes, packed columns
  DevBuf<float> adam_m, adam_v;   // Adam moments (allocated on the first optimiser step)
  int in_dim = 0, out_dim = 0;
  bool set = false;
};

thread_local char g_create_err[512] = "";

// watchdog record of the mbarrier waits (tc_common.cuh: g_wait_dbg): pinned, mapped host memory, one per process and device
unsigned long long* g_wait_host = nullptr;
bool wait_dbg_init() {
  if (g_wait_host) return true;
  unsigned long long* h = nullptr; unsigned long long* d = nullptr;
  if (cudaHostAlloc((void**)&h, 256, cudaHostAllocMapped) != cudaSuccess) { cudaGetLastError(); return false; }
  memset(h, 0, 256);
  // this unit's copy (the dW kernel) and that of each activation's unit (the rollout kernels)
  if (cudaHostGetDevicePointer((void**)&d, h, 0) != cudaSuccess || !tc::wait_dbg_attach(d)
      || !mlp_kernels(tc::H, MPG_ACT_ELU).attach_watchdog(d) || !mlp_kernels(tc::H, MPG_ACT_RELU).attach_watchdog(d)
      || !mlp_kernels(tc::H, MPG_ACT_TANH).attach_watchdog(d)) {
    cudaGetLastError(); cudaFreeHost(h); return false;
  }
  g_wait_host = h;
  return true;
}

}  // namespace

struct mpg_ctx {
  mpg_config cfg;
  int device = 0, sms = 0, S = 0;
  NetStore nets[MPG_NUM_NETS];
  float* ckpt = nullptr;
  float* partial = nullptr;
  float* loss_partial = nullptr;
  float* stats_part = nullptr;   // [MPG_MAX_LIST_LONG][RED_BLOCKS][2]
  float* red_part = nullptr;     // [2][RED_BLOCKS] partial sums of the two-stage reductions (squared error, gradient norm)
  DevBuf<float> qtmp, qtmp2;     // [rows] Q values of the evaluations and of the tensor-core regression pass
  size_t partial_stride = 0;
  size_t ws_bytes = 0;
  uint64_t launches = 0;
  int backend = MPG_BACKEND_FFMA;
  int act = MPG_ACT_ELU;                  // hidden activation of every net (MPG_ACT_*)
  int layers = 2;                         // hidden layers of every net (1..MAX_LAYERS)
  int timing = 0, timed = 0;
  int long_n = -1;                        // list of mpg_set_rollout_list (n_list = MPG_LIST_FROM_HANDLE); -1: never set
  int32_t long_list[MPG_MAX_LIST_LONG];
  float long_w[MPG_MAX_LIST_LONG];
  DevBuf<FarStep> far_steps;             // the list at steps >= STEP_TAB of the last long-horizon rollout
  long long* prof = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  cudaStream_t aux = nullptr;             // side stream: weight-gradient GEMMs of finished waves run under the tail wave
  cudaEvent_t ev_wave = nullptr, ev_aux = nullptr;
  int tail_overlap = 1;
  char err[512];
  TcState tc;
};

namespace {

int fail(mpg_ctx* ctx, int code, const char* fmt, const char* detail = "") {
  char* dst = ctx ? ctx->err : g_create_err;
  snprintf(dst, 512, fmt, detail);
  return code;
}

#define CUDA_OK(ctx, expr)                                                              \
  do {                                                                                  \
    cudaError_t e__ = (expr);                                                           \
    if (e__ != cudaSuccess) return fail(ctx, MPG_ERR_CUDA, #expr ": %s", cudaGetErrorString(e__)); \
  } while (0)

// flat parameter layout of one net of this handle
GradLayout layout(const mpg_ctx* c, const NetStore& n) { return GradLayout(n.in_dim, n.out_dim, c->cfg.hidden, c->layers); }

NetDev net_dev(const mpg_ctx* c, int net) {
  const NetStore& n = c->nets[net];
  const GradLayout L = layout(c, n);
  const size_t hh = (size_t)c->cfg.hidden * c->cfg.hidden;
  NetDev d;
  memset(&d, 0, sizeof(d));
  d.W1p = n.W1p; d.b1 = n.flat + L.ob1;
  for (int l = 2; l <= c->layers; ++l) {
    d.Wp[l - 2] = n.Wp + (l - 2) * hh; d.WTp[l - 2] = n.WTp + (l - 2) * hh; d.b[l - 2] = n.flat + L.ob(l);
  }
  d.Wout = n.flat + L.oWout; d.bout = n.flat + L.obout; d.W1 = n.flat + L.oW1;
  d.in_dim = n.in_dim; d.out_dim = n.out_dim; d.layers = c->layers;
  return d;
}

template <int H>
__global__ void pack_kernel(const float* __restrict__ flat, int in_dim, int out_dim, int layers, float* __restrict__ W1p,
                            float* __restrict__ Wp, float* __restrict__ WTp) {
  const GradLayout L(in_dim, out_dim, H, layers);
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= H * H) return;
  // natural column c of row k -> packed column packed_col<H>(c) (mlp_tile.cuh: rowgemm reads through the same map)
  const int k = idx / H, c = idx % H, o = k * H + packed_col<H>(c);
  for (int l = 2; l <= layers; ++l) {
    const size_t img = (size_t)(l - 2) * H * H;
    Wp[img + o] = flat[L.oW(l) + k * H + c];
    WTp[img + o] = flat[L.oW(l) + c * H + k];   // WT[n=k][col c] = W[c][k]
  }
  if (k < in_dim) W1p[o] = flat[L.oW1 + k * H + c];
}

__global__ void adam_kernel(float* __restrict__ w, float* __restrict__ m, float* __restrict__ v, const float* __restrict__ g,
                            int n, float lr_t, float b1, float b2, float eps) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float gi = g[i];
  const float mi = b1 * m[i] + (1.f - b1) * gi;
  const float vi = b2 * v[i] + (1.f - b2) * gi * gi;
  m[i] = mi; v[i] = vi;
  w[i] -= lr_t * mi / (sqrtf(vi) + eps);
}

// loss_sum = sum_i 0.5 (q_i - target_i)^2: RED_BLOCKS fixed slices, then their partial sums in index order
__global__ void sq_err_partial_kernel(const float* __restrict__ q, const float* __restrict__ target, int n, float* __restrict__ part) {
  const int per = (n + RED_BLOCKS - 1) / RED_BLOCKS, lo = blockIdx.x * per, hi = min(n, lo + per);
  float s = 0.f;
  for (int i = lo + threadIdx.x; i < hi; i += blockDim.x) { const float d = q[i] - target[i]; s = fmaf(0.5f * d, d, s); }
  s = block_sum(s);
  if (threadIdx.x == 0) part[blockIdx.x] = s;
}
__global__ void sum_partials_kernel(const float* __restrict__ part, float* __restrict__ out) {
  out[0] = sum_in_order<RED_BLOCKS>(part);
}

__global__ void polyak_kernel(float* __restrict__ dst, const float* __restrict__ src, int n, float tau) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = tau * src[i] + (1.f - tau) * dst[i];
}

__global__ void reduce_partials_kernel(const float* __restrict__ partial, size_t stride, int nparts, int n,
                                       float* __restrict__ out, const float* __restrict__ loss_partial,
                                       float* __restrict__ loss_out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) {
    float s = 0.f;
    for (int c = 0; c < nparts; ++c) s += partial[(size_t)c * stride + i];
    out[i] = s;
  }
  if (loss_out && blockIdx.x == 0 && threadIdx.x == 0) {
    float s = 0.f;
    for (int c = 0; c < nparts; ++c) s += loss_partial[c];
    loss_out[0] = s;
  }
}

// tf.clip_by_global_norm in two stages (a single block needed 45 us for a 68K-float net: latency bound): RED_BLOCKS blocks
// sum the squares of fixed slices, then every block adds the partial sums in index order and scales its slice.
__global__ void sumsq_partial_kernel(const float* __restrict__ g, int n, float* __restrict__ part) {
  const int per = (n + RED_BLOCKS - 1) / RED_BLOCKS, lo = blockIdx.x * per, hi = min(n, lo + per);
  float s = 0.f;
  for (int i = lo + threadIdx.x; i < hi; i += blockDim.x) s = fmaf(g[i], g[i], s);
  s = block_sum(s);
  if (threadIdx.x == 0) part[blockIdx.x] = s;
}
__global__ void clip_apply_kernel(float* __restrict__ g, int n, float clip, const float* __restrict__ part,
                                  float* __restrict__ norm_out) {
  const float norm = sqrtf(sum_in_order<RED_BLOCKS>(part));
  const float scale = clip * fminf(1.f / norm, 1.f / clip);   // tf.clip_by_global_norm
  const int per = (n + RED_BLOCKS - 1) / RED_BLOCKS, lo = blockIdx.x * per, hi = min(n, lo + per);
  if (scale != 1.f)
    for (int i = lo + threadIdx.x; i < hi; i += blockDim.x) g[i] *= scale;
  if (blockIdx.x == 0 && threadIdx.x == 0 && norm_out) norm_out[0] = norm;
}

// returns (n_list, M*rows) -> tile mean (n_list, rows) and/or sums over rows of mean, mean^2.
// Two stages so that 64K-row batches do not serialise on one block: grid (n_list, RED_BLOCKS) partial sums of fixed
// slices, then one thread per k adds the RED_BLOCKS partials in index order.
__global__ void returns_stats_kernel(const float* __restrict__ ret, int n_list, int rows, int M,
                                     float* __restrict__ mean_out, float* __restrict__ part) {
  const int k = blockIdx.x, blk = blockIdx.y;
  const int per = (rows + RED_BLOCKS - 1) / RED_BLOCKS, lo = blk * per, hi = min(rows, lo + per);
  float s[2] = {0.f, 0.f};
  for (int i = lo + threadIdx.x; i < hi; i += blockDim.x) {
    float m = 0.f;
    for (int t = 0; t < M; ++t) m += ret[(size_t)k * M * rows + (size_t)t * rows + i];
    m /= (float)M;
    if (mean_out) mean_out[(size_t)k * rows + i] = m;
    s[0] += m; s[1] = fmaf(m, m, s[1]);
  }
  block_sum(s);
  if (threadIdx.x == 0 && part) { part[(k * RED_BLOCKS + blk) * 2] = s[0]; part[(k * RED_BLOCKS + blk) * 2 + 1] = s[1]; }
}
__global__ void returns_stats_final_kernel(const float* __restrict__ part, int n_list, float* __restrict__ stats_out) {
  const int k = threadIdx.x;
  if (k >= n_list) return;
  const float* pk = part + k * RED_BLOCKS * 2;
  stats_out[k] = sum_in_order<RED_BLOCKS>(pk, 2); stats_out[n_list + k] = sum_in_order<RED_BLOCKS>(pk + 1, 2);
}

__global__ void philox_noise_kernel(unsigned long long seed, long long global_rows, long long row_offset, int rows,
                                    int M, int horizon, float* __restrict__ out) {
  const int MB = rows * M;
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)horizon * MB) return;
  const int t = (int)(idx / MB), grow = (int)(idx % MB);
  const unsigned long long nr = (unsigned long long)(grow / rows) * global_rows + row_offset + (grow % rows);
  out[idx] = philox_normal(seed, nr, (uint32_t)t);
}

int check_net(mpg_ctx* ctx, int net) {
  if (net < 0 || net >= MPG_NUM_NETS) return fail(ctx, MPG_ERR_ARG, "bad net id%s");
  if (!ctx->nets[net].set) return fail(ctx, MPG_ERR_STATE, "weights of a required net were never set%s");
  return MPG_OK;
}

int fill_rollout_args(mpg_ctx* ctx, const mpg_rollout_params* p, RolloutArgs& a) {
  const mpg_config& c = ctx->cfg;
  const bool from_handle = p->n_list == MPG_LIST_FROM_HANDLE;
  if (p->rows <= 0 || p->M <= 0 || p->horizon < 0 || (!from_handle && (p->n_list < 0 || p->n_list > MPG_MAX_LIST)))
    return fail(ctx, MPG_ERR_ARG, "bad rollout params%s");
  if (from_handle && ctx->long_n < 0)
    return fail(ctx, MPG_ERR_STATE, "n_list = MPG_LIST_FROM_HANDLE but mpg_set_rollout_list was never called%s");
  if ((long long)p->rows * p->M > c.max_rows || p->horizon > c.max_horizon)
    return fail(ctx, MPG_ERR_ARG, "rollout exceeds the capacity given to mpg_create (max_rows / max_horizon)%s");
  const int n_list = from_handle ? ctx->long_n : p->n_list;
  const int32_t* list = from_handle ? ctx->long_list : p->list;
  const float* list_w = from_handle ? ctx->long_w : p->list_w;
  for (int k = 0; k < n_list; ++k)
    if (list[k] < 0 || list[k] > p->horizon) return fail(ctx, MPG_ERR_ARG, "rollout index outside [0, horizon]%s");
  memset(&a, 0, sizeof(a));
  a.obs_dim = c.obs_dim; a.act_dim = c.act_dim; a.nfd = c.num_future_data; a.policy_out_tanh = c.policy_out_tanh;
  a.action_range = c.action_range;
  for (int i = 0; i < MPG_MAX_OBS; ++i) a.obs_scale[i] = c.obs_scale[i];
  a.rew_scale = c.rew_scale; a.rew_shift = c.rew_shift; a.gamma = c.gamma;
  a.rows = p->rows; a.M = p->M; a.horizon = p->horizon; a.n_list = n_list;
  for (int k = 0; k < n_list; ++k) { a.list[k] = list[k]; a.list_w[k] = list_w[k]; }
  a.full_bptt = p->full_bptt;
  a.has_q = p->q_net >= 0;
  a.global_rows = p->global_rows > 0 ? p->global_rows : p->rows;
  a.row_offset = p->row_offset;
  a.seed = p->noise_seed;
  int rc = check_net(ctx, p->policy_net);
  if (rc) return rc;
  a.pol = net_dev(ctx, p->policy_net);
  if (a.has_q) {
    rc = check_net(ctx, p->q_net);
    if (rc) return rc;
    a.q = net_dev(ctx, p->q_net);
  }
  a.ckpt = ctx->ckpt;
  a.partial = ctx->partial;
  a.partial_stride = (long long)ctx->partial_stride;
  return MPG_OK;
}

// the list at steps [STEP_TAB, horizon] (StepTab serves the steps below from shared memory)
__global__ void far_steps_kernel(const __grid_constant__ RolloutArgs a, FarStep* __restrict__ out) {
  const int t = STEP_TAB + blockIdx.x * blockDim.x + threadIdx.x;
  if (t <= a.horizon) out[t - STEP_TAB] = list_step(a.list, a.list_w, a.n_list, t);
}

// a.far_steps for a horizon that reaches past the shared-memory step tables; nothing to do for shorter ones
int prepare_far_steps(mpg_ctx* ctx, RolloutArgs& a, cudaStream_t st) {
  a.far_steps = nullptr;
  if (a.horizon < STEP_TAB) return MPG_OK;
  const size_t n = (size_t)(a.horizon + 1 - STEP_TAB);
  CUDA_OK(ctx, ctx->far_steps.grow(n));
  far_steps_kernel<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(a, ctx->far_steps.p);
  ctx->launches++;
  CUDA_OK(ctx, cudaGetLastError());
  a.far_steps = ctx->far_steps.p;
  return MPG_OK;
}

// the Q scratch (ctx->qtmp, ctx->qtmp2) for `rows` rows
int q_scratch(mpg_ctx* ctx, int rows) {
  if (ctx->qtmp.grow(rows) != cudaSuccess || ctx->qtmp2.grow(rows) != cudaSuccess)
    return fail(ctx, MPG_ERR_CUDA, "cudaMalloc of the Q scratch failed%s");
  return MPG_OK;
}

// a rollout of horizon 0 over `rows` rows: the policy's action (or the given one) and, with q_net >= 0, the Q value of
// that action as the returns row of the one-entry list {0}
mpg_rollout_params horizon0_params(int rows, int policy_net, int q_net) {
  mpg_rollout_params p;
  memset(&p, 0, sizeof(p));
  p.rows = rows; p.M = 1; p.horizon = 0;
  p.n_list = q_net >= 0 ? 1 : 0; p.list[0] = 0; p.list_w[0] = 1.f;
  p.q_net = q_net; p.policy_net = policy_net;
  return p;
}

// dW2 = sum over (row, step) of h1^T delta2 is the only contraction of the path whose K is the batch.  With K in the
// millions the rounding of the operands averages out, so the records of LARGE policy-gradient contractions keep only the hi
// plane of h1 (11 bits) and delta2 (8 bits) and the dW kernel issues one product instead of three: half the record
// traffic, and the side-stream GEMMs fit under the tail wave (+14 % state-steps/s at 65,536 rows).  Emulated on the CPU
// oracle (DESIGN 4.3) and measured: the added gradient error is ~1e-5 at K = 262,144 (rows x recorded steps) and falls
// with 1/sqrt(K); below that the full hi + lo records are kept (at K = 16..256 x 26 hi-only records miss the 1e-4 bar).
// The rounding error is ~1.1e-3 of the root-sum-square of the terms, so relative to the gradient it grows with the
// cancellation in the sum (worst case, a gradient that is pure sampling noise: 1.1e-3 of that noise): the Q regression
// never uses it, and MPG_REC_HI_ONLY=0 keeps full records everywhere (=1 forces hi-only, for tests).  The same flag makes
// dW3 = sum h2^T delta3 -- the other contraction over the batch -- take only the hi plane of h2 (tc_gemm.cuh: d3_issue).
int rec_hi_only(const mpg_ctx* ctx, long long contraction_rows) {
  (void)ctx;
  const char* e = getenv("MPG_REC_HI_ONLY");
  if (e && (e[0] == '0' || e[0] == '1')) return e[0] == '1';
  return contraction_rows >= 262144 ? 1 : 0;
}

// grad_out = the sum of the first nparts partial gradients of net (and *loss_out = that of the partial losses, when given)
void launch_reduce(const mpg_ctx* ctx, int net, int nparts, float* grad_out, float* loss_out, cudaStream_t st) {
  const int n = layout(ctx, ctx->nets[net]).total;
  reduce_partials_kernel<<<(n + 255) / 256, 256, 0, st>>>(ctx->partial, ctx->partial_stride, nparts, n, grad_out,
                                                          ctx->loss_partial, loss_out);
}

// tensor-core rollout kernel of the handle's activation; cudaErrorNotSupported: there is none (backward on the real env)
template <bool BWD>
cudaError_t tc_launch_rollout(int env, int act, const tc::TcArgs& a, int grid, cudaStream_t st) {
  if (!mlp_kernels(tc::H, act).tc_rollout(env, BWD, a, grid, st)) return cudaErrorNotSupported;
  return cudaGetLastError();
}

// the arguments of the tensor-core rollout kernel that every launch shares: the rollout and the nets' weight images
tc::TcArgs tc_args(const mpg_ctx* ctx, const RolloutArgs& a, int policy_net, int q_net) {
  tc::TcArgs ta;
  memset(&ta, 0, sizeof(ta));
  ta.r = a;
  ta.pol = tc_net(ctx->tc, policy_net, ctx->nets[policy_net].flat, a.pol.in_dim, a.pol.out_dim);
  if (a.has_q) ta.q = tc_net(ctx->tc, q_net, ctx->nets[q_net].flat, a.q.in_dim, a.q.out_dim);
  ta.act_ckpt = ctx->tc.act_ckpt.p;
  return ta;
}

// weight gradient of the dW operand store records of tiles [tile0, tile0 + tiles) into the partial gradients from row
// part_row on: tc_dw_kernel, two CTAs per record, at most the even number of the `sms` SMs it may use
void launch_dw(const mpg_ctx* ctx, const tc::TcArgs& ta, int tile0, int tiles, int part_row, int sms, cudaStream_t st) {
  tc::DwArgs da;
  da.store = ctx->tc.store.p + (size_t)tile0 * ta.store_steps * tc::SLOT_BYTES;
  da.nrecords = tiles * ta.store_steps;
  da.in_dim = ta.pol.in_dim; da.out_dim = ta.pol.out_dim;
  da.partial = ctx->partial + (size_t)part_row * ctx->partial_stride; da.partial_stride = (long long)ctx->partial_stride;
  da.hi_only = ta.rec_hi_only;
  const int grid = 2 * da.nrecords < sms ? 2 * da.nrecords : (sms & ~1);
  tc::tc_dw_kernel<<<grid, tc::DW_THREADS, tc::DW_SMEM, st>>>(da);
}

template <bool BWD>
int launch_rollout(mpg_ctx* ctx, const RolloutArgs& a, int grid, cudaStream_t st, int env) {
  if (ctx->timing) cudaEventRecord(ctx->ev0, st);
  if (!mlp_kernels(ctx->cfg.hidden, ctx->act).rollout(env, BWD, a, grid, st))
    return fail(ctx, MPG_ERR_UNSUPPORTED, "the real environment is forward only%s");
  if (ctx->timing) { cudaEventRecord(ctx->ev1, st); ctx->timed = 1; }
  ctx->launches++;
  CUDA_OK(ctx, cudaGetLastError());
  return MPG_OK;
}

}  // namespace

extern "C" {

const char* mpg_last_error(const mpg_ctx* ctx) { return ctx ? ctx->err : g_create_err; }
size_t mpg_workspace_bytes(const mpg_ctx* ctx) { return ctx->ws_bytes; }
int mpg_num_sms(const mpg_ctx* ctx) { return ctx->sms; }
int mpg_state_dim(const mpg_ctx* ctx) { return ctx->S; }
uint64_t mpg_launch_count(const mpg_ctx* ctx) { return ctx->launches; }

int mpg_get_backend(const mpg_ctx* ctx) { return ctx->backend; }
int mpg_set_backend(mpg_ctx* ctx, int backend) {
  if (!ctx || (backend != MPG_BACKEND_FFMA && backend != MPG_BACKEND_TC)) return fail(ctx, MPG_ERR_ARG, "bad backend%s");
  if (backend == MPG_BACKEND_TC && !ctx->tc.ready) {
    if (ctx->layers != 2) {
      char n[16];
      snprintf(n, sizeof(n), "%d", ctx->layers);
      return fail(ctx, MPG_ERR_UNSUPPORTED,
                  "tensor-core backend does not cover this configuration (it needs hidden = 256 and 2 hidden layers; "
                  "this handle has %s)", n);
    }
    return fail(ctx, MPG_ERR_UNSUPPORTED,
                "tensor-core backend does not cover this configuration (it needs hidden = 256 and obs_dim + act_dim <= 15)%s");
  }
  ctx->backend = backend;
  return MPG_OK;
}

int mpg_get_activation(const mpg_ctx* ctx) { return ctx->act; }
int mpg_set_activation(mpg_ctx* ctx, int act) {
  if (!ctx || (act != MPG_ACT_ELU && act != MPG_ACT_RELU && act != MPG_ACT_TANH)) return fail(ctx, MPG_ERR_ARG, "bad activation%s");
  ctx->act = act;
  return MPG_OK;
}

// {flag, site, block, thread, parity} of the mbarrier wait that timed out (flag == 0: none); see tc_common.cuh
int mpg_wait_debug(unsigned long long out[32]) {
  if (!out) return MPG_ERR_ARG;
  for (int i = 0; i < 32; ++i) out[i] = g_wait_host ? ((volatile unsigned long long*)g_wait_host)[i] : 0ull;
  return MPG_OK;
}

#ifdef MPG_DEBUG_PROBES
int mpg_set_profile_buffer(mpg_ctx* ctx, long long* buf) {
  if (!ctx) return MPG_ERR_ARG;
  ctx->prof = buf;
  return MPG_OK;
}
#endif
int mpg_set_timing(mpg_ctx* ctx, int enabled) {
  if (!ctx) return MPG_ERR_ARG;
  if (enabled && !ctx->ev0) {
    CUDA_OK(ctx, cudaEventCreate(&ctx->ev0));
    CUDA_OK(ctx, cudaEventCreate(&ctx->ev1));
  }
  ctx->timing = enabled ? 1 : 0;
  ctx->timed = 0;
  return MPG_OK;
}
float mpg_kernel_ms(mpg_ctx* ctx) {
  if (!ctx || !ctx->timed) return -1.f;
  float ms = -1.f;
  if (cudaEventSynchronize(ctx->ev1) != cudaSuccess || cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1) != cudaSuccess) return -1.f;
  return ms;
}

#ifdef MPG_DEBUG_PROBES
int mpg_tc_selftest(mpg_ctx* ctx, int kind, const float* X, const float* W, float* Z, int repeats, void* stream) {
  if (!ctx || !X || !W || !Z || kind < 0 || kind > 5 || repeats < 1) return fail(ctx, MPG_ERR_ARG, "bad argument to mpg_tc_selftest%s");
  CUDA_OK(ctx, tc_selftest(ctx->tc, kind, X, W, Z, repeats, (cudaStream_t)stream));
  ctx->launches += 2;
  return MPG_OK;
}
#endif

int mpg_param_count(const mpg_ctx* ctx, int net) {
  if (net < 0 || net >= MPG_NUM_NETS) return -1;
  return layout(ctx, ctx->nets[net]).total;
}

int mpg_hidden_layers(const mpg_ctx* ctx) { return ctx->layers; }

int mpg_create(const mpg_config* cfg, mpg_ctx** out) { return mpg_create_layers(cfg, 2, out); }

int mpg_create_layers(const mpg_config* cfg, int hidden_layers, mpg_ctx** out) {
  if (!cfg || !out) return fail(nullptr, MPG_ERR_ARG, "null argument%s");
  *out = nullptr;
  if (hidden_layers < 1 || hidden_layers > MAX_LAYERS)
    return fail(nullptr, MPG_ERR_UNSUPPORTED, "hidden_layers must be 1, 2 or 3; deeper nets are not supported%s");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return fail(nullptr, MPG_ERR_CUDA, "no CUDA device: mpg_b200 has no CPU fallback%s");
  if (cfg->hidden != 64 && cfg->hidden != 128 && cfg->hidden != 256)
    return fail(nullptr, MPG_ERR_UNSUPPORTED, "hidden must be 64, 128 or 256; other widths are not built%s");
  if (cfg->env < 0 || cfg->env > 3) return fail(nullptr, MPG_ERR_ARG, "unknown env%s");
  static const int SD[4] = {6, 4, 6, 8}, AD[4] = {2, 1, 1, 2};
  if (cfg->act_dim != AD[cfg->env]) return fail(nullptr, MPG_ERR_ARG, "act_dim does not match env%s");
  const int want_obs = (cfg->env == 0 || cfg->env == 3) ? 6 + cfg->num_future_data : (cfg->env == 1 ? 4 : 11);
  if (cfg->obs_dim != want_obs || cfg->obs_dim > MPG_MAX_OBS) return fail(nullptr, MPG_ERR_ARG, "obs_dim does not match env%s");
  if (cfg->max_rows <= 0 || cfg->max_horizon < 0) return fail(nullptr, MPG_ERR_ARG, "bad capacity%s");
  mpg_ctx* c = new (std::nothrow) mpg_ctx();
  if (!c) return fail(nullptr, MPG_ERR_ARG, "out of host memory%s");
  c->cfg = *cfg;
  c->layers = hidden_layers;
  c->err[0] = 0;
  c->S = SD[cfg->env];
  cudaDeviceProp prop;
  if (cudaGetDevice(&c->device) != cudaSuccess || cudaGetDeviceProperties(&prop, c->device) != cudaSuccess) {
    delete c;
    return fail(nullptr, MPG_ERR_CUDA, "cudaGetDeviceProperties failed%s");
  }
  c->sms = prop.multiProcessorCount;
  if (prop.major < 10) {
    delete c;
    return fail(nullptr, MPG_ERR_UNSUPPORTED, "built for sm_100a (B200) only%s");
  }
  auto alloc = [&](float** p, size_t n) -> bool {
    if (cudaMalloc(p, n * sizeof(float)) != cudaSuccess) return false;
    c->ws_bytes += n * sizeof(float);
    return true;
  };
  bool ok = true;
  size_t maxP = 0;
  for (int n = 0; n < MPG_NUM_NETS && ok; ++n) {
    NetStore& ns = c->nets[n];
    const bool is_pol = (n == MPG_NET_POLICY || n == MPG_NET_POLICY_TARGET);
    ns.in_dim = is_pol ? cfg->obs_dim : cfg->obs_dim + cfg->act_dim;
    ns.out_dim = is_pol ? 2 * cfg->act_dim : 1;
    const GradLayout L = layout(c, ns);
    const size_t hw = (size_t)cfg->hidden;
    maxP = L.total > (int)maxP ? L.total : maxP;
    const size_t himg = (size_t)(hidden_layers - 1) * hw * hw;
    ok = ok && alloc(&ns.flat, L.total) && alloc(&ns.W1p, MAX_IN * hw)
         && (himg == 0 || (alloc(&ns.Wp, himg) && alloc(&ns.WTp, himg)));
  }
  c->partial_stride = (maxP + 3) & ~size_t(3);
  ok = ok && alloc(&c->ckpt, (size_t)(cfg->max_horizon + 1) * cfg->max_rows * c->S)
       && alloc(&c->partial, (size_t)2 * c->sms * c->partial_stride) && alloc(&c->loss_partial, c->sms)
       && alloc(&c->stats_part, (size_t)MPG_MAX_LIST_LONG * RED_BLOCKS * 2) && alloc(&c->red_part, 2 * RED_BLOCKS);
  if (ok) ok = tc_init(c->tc, c->cfg, hidden_layers, c->sms, c->ws_bytes);
  if (ok && c->tc.ready) {   // the tensor-core evaluations up to max_rows rows: their Q scratch is there from the start
    ok = q_scratch(c, cfg->max_rows) == MPG_OK;
    c->ws_bytes += 2 * (size_t)cfg->max_rows * sizeof(float);
  }
  wait_dbg_init();   // best effort: without it a timed-out wait still traps, only the record is missing
  if (!ok) {
    cudaError_t e = cudaGetLastError();   // a grow-only buffer has already taken its error off the record
    snprintf(g_create_err, 512, "cudaMalloc of the workspace failed: %s",
             cudaGetErrorString(e != cudaSuccess ? e : cudaErrorMemoryAllocation));
    mpg_destroy(c);
    return MPG_ERR_CUDA;
  }
  cudaError_t e = cudaSuccess;
  for (const int act : {MPG_ACT_ELU, MPG_ACT_RELU, MPG_ACT_TANH})   // the activation can change on the handle later
    if (e == cudaSuccess) e = mlp_kernels(cfg->hidden, act).set_smem();
  if (e != cudaSuccess) {
    snprintf(g_create_err, 512, "cudaFuncSetAttribute (max dynamic shared memory of the MLP kernels): %s", cudaGetErrorString(e));
    mpg_destroy(c);
    return MPG_ERR_CUDA;
  }
  if (cudaStreamCreateWithFlags(&c->aux, cudaStreamNonBlocking) != cudaSuccess
      || cudaEventCreateWithFlags(&c->ev_wave, cudaEventDisableTiming) != cudaSuccess
      || cudaEventCreateWithFlags(&c->ev_aux, cudaEventDisableTiming) != cudaSuccess) {
    snprintf(g_create_err, 512, "side stream / event creation failed: %s", cudaGetErrorString(cudaGetLastError()));
    mpg_destroy(c);
    return MPG_ERR_CUDA;
  }
  // default backend: the tensor-core path wherever it covers the configuration, else fp32 FFMA
  c->backend = c->tc.ready ? MPG_BACKEND_TC : MPG_BACKEND_FFMA;
  const char* be = getenv("MPG_B200_BACKEND");
  if (be && !strcmp(be, "ffma")) c->backend = MPG_BACKEND_FFMA;
  const char* ov = getenv("MPG_TAIL_OVERLAP");
  c->tail_overlap = !(ov && ov[0] == '0');
  *out = c;
  return MPG_OK;
}

void mpg_destroy(mpg_ctx* c) {
  if (!c) return;
  for (int n = 0; n < MPG_NUM_NETS; ++n) {
    cudaFree(c->nets[n].flat); cudaFree(c->nets[n].W1p); cudaFree(c->nets[n].Wp); cudaFree(c->nets[n].WTp);
    c->nets[n].adam_m.release(); c->nets[n].adam_v.release();
  }
  cudaFree(c->ckpt); cudaFree(c->partial); cudaFree(c->loss_partial); cudaFree(c->stats_part); cudaFree(c->red_part);
  c->qtmp.release(); c->qtmp2.release(); c->far_steps.release();
  if (c->ev0) { cudaEventDestroy(c->ev0); cudaEventDestroy(c->ev1); }
  if (c->aux) { cudaStreamSynchronize(c->aux); cudaStreamDestroy(c->aux); }
  if (c->ev_wave) cudaEventDestroy(c->ev_wave);
  if (c->ev_aux) cudaEventDestroy(c->ev_aux);
  tc_destroy(c->tc);
  delete c;
}

// FFMA weight images (W1p, Wp, WTp) of one net from its flat natural weights
static void launch_pack(mpg_ctx* ctx, const NetStore& ns, cudaStream_t st) {
  const int hw = ctx->cfg.hidden, grid = (hw * hw + 255) / 256;   // mpg_create admits 64, 128 and 256
  const int L = ctx->layers;
  switch (hw) {
    case 64: pack_kernel<64><<<grid, 256, 0, st>>>(ns.flat, ns.in_dim, ns.out_dim, L, ns.W1p, ns.Wp, ns.WTp); break;
    case 128: pack_kernel<128><<<grid, 256, 0, st>>>(ns.flat, ns.in_dim, ns.out_dim, L, ns.W1p, ns.Wp, ns.WTp); break;
    default: pack_kernel<256><<<grid, 256, 0, st>>>(ns.flat, ns.in_dim, ns.out_dim, L, ns.W1p, ns.Wp, ns.WTp); break;
  }
  ctx->launches++;
}

// flat offset and size of the i-th of the 2 (L + 1) weight arrays W1, b1, W2, b2, .., WL, bL, Wout, bout of a net
static void weight_array(const mpg_ctx* ctx, const NetStore& ns, int i, int& off, int& cnt) {
  const GradLayout L = layout(ctx, ns);
  const int hw = ctx->cfg.hidden, l = i / 2 + 1;
  if (l == 1) { off = i ? L.ob1 : L.oW1; cnt = i ? hw : ns.in_dim * hw; }
  else if (l <= ctx->layers) { off = i & 1 ? L.ob(l) : L.oW(l); cnt = i & 1 ? hw : hw * hw; }
  else { off = i & 1 ? L.obout : L.oWout; cnt = i & 1 ? ns.out_dim : hw * ns.out_dim; }
}

int mpg_set_weights(mpg_ctx* ctx, int net, const float* const w[], void* stream) {
  if (!ctx || net < 0 || net >= MPG_NUM_NETS || !w) return fail(ctx, MPG_ERR_ARG, "bad argument to mpg_set_weights%s");
  cudaStream_t st = (cudaStream_t)stream;
  NetStore& ns = ctx->nets[net];
  for (int i = 0; i < 2 * (ctx->layers + 1); ++i) {
    if (!w[i]) return fail(ctx, MPG_ERR_ARG, "null weight pointer%s");
    int off, cnt;
    weight_array(ctx, ns, i, off, cnt);
    CUDA_OK(ctx, cudaMemcpyAsync(ns.flat + off, w[i], cnt * sizeof(float), cudaMemcpyDefault, st));
  }
  launch_pack(ctx, ns, st);
  CUDA_OK(ctx, cudaGetLastError());
  ns.set = true;
  return tc_pack_weights(ctx->tc, net, ns.flat, ns.in_dim, ns.out_dim, st) ? MPG_OK
                                                                           : fail(ctx, MPG_ERR_CUDA, "tc weight pack failed%s");
}

static int repack(mpg_ctx* ctx, int net, cudaStream_t st) {
  NetStore& ns = ctx->nets[net];
  launch_pack(ctx, ns, st);
  CUDA_OK(ctx, cudaGetLastError());
  return tc_pack_weights(ctx->tc, net, ns.flat, ns.in_dim, ns.out_dim, st) ? MPG_OK
                                                                           : fail(ctx, MPG_ERR_CUDA, "tc weight pack failed%s");
}

static int adam_alloc(mpg_ctx* ctx, NetStore& ns, int n, cudaStream_t st) {
  if (ns.adam_v.n >= (size_t)n) return MPG_OK;
  CUDA_OK(ctx, ns.adam_m.grow(n));
  CUDA_OK(ctx, ns.adam_v.grow(n));
  CUDA_OK(ctx, cudaMemsetAsync(ns.adam_m.p, 0, n * sizeof(float), st));
  CUDA_OK(ctx, cudaMemsetAsync(ns.adam_v.p, 0, n * sizeof(float), st));
  return MPG_OK;
}

int mpg_adam_step(mpg_ctx* ctx, int net, const float* grad, float lr, int64_t step, float beta1, float beta2, float eps,
                  void* stream) {
  if (!ctx || !grad || step < 1) return fail(ctx, MPG_ERR_ARG, "bad argument to mpg_adam_step%s");
  int rc = check_net(ctx, net);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  NetStore& ns = ctx->nets[net];
  const int n = layout(ctx, ns).total;
  if ((rc = adam_alloc(ctx, ns, n, st))) return rc;
  const double t = (double)step;
  const float lr_t = (float)((double)lr * sqrt(1.0 - pow((double)beta2, t)) / (1.0 - pow((double)beta1, t)));
  adam_kernel<<<(n + 255) / 256, 256, 0, st>>>(ns.flat, ns.adam_m.p, ns.adam_v.p, grad, n, lr_t, beta1, beta2, eps);
  ctx->launches++;
  CUDA_OK(ctx, cudaGetLastError());
  return repack(ctx, net, st);
}

int mpg_get_adam_state(mpg_ctx* ctx, int net, float* m, float* v, void* stream) {
  if (!ctx || !m || !v) return fail(ctx, MPG_ERR_ARG, "bad argument to mpg_get_adam_state%s");
  int rc = check_net(ctx, net);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  NetStore& ns = ctx->nets[net];
  const int n = layout(ctx, ns).total;
  if ((rc = adam_alloc(ctx, ns, n, st))) return rc;
  CUDA_OK(ctx, cudaMemcpyAsync(m, ns.adam_m.p, n * sizeof(float), cudaMemcpyDeviceToDevice, st));
  CUDA_OK(ctx, cudaMemcpyAsync(v, ns.adam_v.p, n * sizeof(float), cudaMemcpyDeviceToDevice, st));
  return MPG_OK;
}

int mpg_set_adam_state(mpg_ctx* ctx, int net, const float* m, const float* v, void* stream) {
  if (!ctx || !m || !v) return fail(ctx, MPG_ERR_ARG, "bad argument to mpg_set_adam_state%s");
  int rc = check_net(ctx, net);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  NetStore& ns = ctx->nets[net];
  const int n = layout(ctx, ns).total;
  if ((rc = adam_alloc(ctx, ns, n, st))) return rc;
  CUDA_OK(ctx, cudaMemcpyAsync(ns.adam_m.p, m, n * sizeof(float), cudaMemcpyDeviceToDevice, st));
  CUDA_OK(ctx, cudaMemcpyAsync(ns.adam_v.p, v, n * sizeof(float), cudaMemcpyDeviceToDevice, st));
  return MPG_OK;
}

int mpg_polyak_update(mpg_ctx* ctx, int src_net, int dst_net, float tau, void* stream) {
  int rc = check_net(ctx, src_net);
  if (!rc) rc = check_net(ctx, dst_net);
  if (rc) return rc;
  NetStore &a = ctx->nets[src_net], &d = ctx->nets[dst_net];
  if (a.in_dim != d.in_dim || a.out_dim != d.out_dim) return fail(ctx, MPG_ERR_ARG, "polyak: nets differ in shape%s");
  cudaStream_t st = (cudaStream_t)stream;
  const int n = layout(ctx, a).total;
  polyak_kernel<<<(n + 255) / 256, 256, 0, st>>>(d.flat, a.flat, n, tau);
  ctx->launches++;
  CUDA_OK(ctx, cudaGetLastError());
  return repack(ctx, dst_net, st);
}

int mpg_get_weights(mpg_ctx* ctx, int net, float* const w[], void* stream) {
  int rc = check_net(ctx, net);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  NetStore& ns = ctx->nets[net];
  for (int i = 0; i < 2 * (ctx->layers + 1); ++i) {
    int off, cnt;
    weight_array(ctx, ns, i, off, cnt);
    CUDA_OK(ctx, cudaMemcpyAsync(w[i], ns.flat + off, cnt * sizeof(float), cudaMemcpyDefault, st));
  }
  return MPG_OK;
}

int mpg_set_rollout_list(mpg_ctx* ctx, int n, const int32_t* list_host, const float* list_w_host) {
  if (!ctx || n < 0 || (n > 0 && (!list_host || !list_w_host))) return fail(ctx, MPG_ERR_ARG, "bad argument to mpg_set_rollout_list%s");
  if (n > MPG_MAX_LIST_LONG) return fail(ctx, MPG_ERR_ARG, "rollout list too long: at most 64 (MPG_MAX_LIST_LONG) entries%s");
  for (int k = 0; k < n; ++k) { ctx->long_list[k] = list_host[k]; ctx->long_w[k] = list_w_host[k]; }
  ctx->long_n = n;
  return MPG_OK;
}

int mpg_policy_grad(mpg_ctx* ctx, const mpg_rollout_params* p, const float* obs, const float* noise, float* grad_out,
                    float* returns_out, void* stream) {
  if (!ctx || !p || !obs || !grad_out) return fail(ctx, MPG_ERR_ARG, "null argument to mpg_policy_grad%s");
  if (p->real_env || ctx->cfg.env == MPG_ENV_PATH_TRACKING_REAL) return fail(ctx, MPG_ERR_UNSUPPORTED, "the real environment is forward only%s");
  cudaStream_t st = (cudaStream_t)stream;
  RolloutArgs a;
  int rc = fill_rollout_args(ctx, p, a);
  if (rc) return rc;
  a.obs = obs; a.noise = noise; a.returns_out = returns_out;
  a.noise_mode = noise ? 1 : (p->use_philox ? 2 : 0);
  if ((rc = prepare_far_steps(ctx, a, st))) return rc;
  const int MB = p->rows * p->M;
  if (ctx->backend == MPG_BACKEND_TC) {
    // tensor-core path: fused rollout + BPTT (dX chain), then the split-K weight-gradient GEMMs
    const int ntiles = (MB + tc::ACT_ROWS - 1) / tc::ACT_ROWS;
    const int grid = ntiles < ctx->sms ? ntiles : ctx->sms;
    if (ctx->tc.act_ckpt.grow((size_t)a.n_list * MB * MAX_A) != cudaSuccess)
      return fail(ctx, MPG_ERR_CUDA, "cudaMalloc of the action checkpoints failed%s");
    tc::TcArgs ta = tc_args(ctx, a, p->policy_net, p->q_net);
    ta.store_steps = p->full_bptt ? p->horizon + 1 : 1;
    const size_t need = (size_t)ntiles * ta.store_steps * tc::SLOT_BYTES;
    if (ctx->tc.store.grow(need) != cudaSuccess) return fail(ctx, MPG_ERR_CUDA, "cudaMalloc of the dW operand store failed%s");
    ta.store = ctx->tc.store.p;
    ta.rec_hi_only = rec_hi_only(ctx, (long long)MB * ta.store_steps);
    if (ctx->tc.h2store.grow((size_t)ntiles * (p->horizon + 1) * 2 * tc::ACT_SPLIT) != cudaSuccess)
      return fail(ctx, MPG_ERR_CUDA, "cudaMalloc of the h2 image store failed%s");
    ta.h2store = ctx->tc.h2store.p;
    ta.z_ckpt = ctx->tc.z_ckpt;
    ta.prof = ctx->prof;
    // Wave-tail overlap: with ntiles = w * sms + tail the last wave leaves sms - tail SMs idle.  The full waves and
    // the tail wave are two launches; the weight-gradient GEMMs of the full waves (HBM-bound) run on the side
    // stream on exactly the SMs the tail wave does not use.  Partial rows [0, sms): full waves, [sms, 2 sms): tail.
    const int tail = ntiles % ctx->sms, full = ntiles - tail;
    // The side-stream GEMMs get only the SMs the tail wave leaves idle: worth it when that is a good part of the GPU (their
    // work grows with the number of full waves); with a nearly full tail wave they would crawl on a handful of SMs, so
    // the weight-gradient GEMMs then run on all SMs after the rollout.
    const bool split = ctx->tail_overlap && ctx->aux && full > 0 && tail > 0 && !ctx->prof
                       && (long long)(ctx->sms - tail) * 4 >= (long long)(full / ctx->sms) * ctx->sms / 2;
    CUDA_OK(ctx, cudaMemsetAsync(ctx->partial, 0, (size_t)(split ? 2 : 1) * ctx->sms * ctx->partial_stride * sizeof(float), st));
    if (ctx->timing) cudaEventRecord(ctx->ev0, st);
    if (!split) {
      CUDA_OK(ctx, tc_launch_rollout<true>(ctx->cfg.env, ctx->act, ta, grid, st));
      if (ctx->timing) { cudaEventRecord(ctx->ev1, st); ctx->timed = 1; }
      launch_dw(ctx, ta, 0, ntiles, 0, ctx->sms, st);
      launch_reduce(ctx, p->policy_net, ctx->sms, grad_out, nullptr, st);
      ctx->launches += 3;
    } else {
      ta.tile0 = 0; ta.tile1 = full;
      CUDA_OK(ctx, tc_launch_rollout<true>(ctx->cfg.env, ctx->act, ta, ctx->sms, st));
      CUDA_OK(ctx, cudaEventRecord(ctx->ev_wave, st));
      tc::TcArgs tb = ta;
      tb.tile0 = full; tb.tile1 = ntiles;
      tb.r.partial = ctx->partial + (size_t)ctx->sms * ctx->partial_stride;
      CUDA_OK(ctx, tc_launch_rollout<true>(ctx->cfg.env, ctx->act, tb, tail, st));
      if (ctx->timing) { cudaEventRecord(ctx->ev1, st); ctx->timed = 1; }
      CUDA_OK(ctx, cudaStreamWaitEvent(ctx->aux, ctx->ev_wave, 0));
      launch_dw(ctx, ta, 0, full, 0, ctx->sms - tail, ctx->aux);   // full waves: >= sms records, all of the idle SMs
      CUDA_OK(ctx, cudaEventRecord(ctx->ev_aux, ctx->aux));
      launch_dw(ctx, ta, full, tail, ctx->sms, ctx->sms, st);
      CUDA_OK(ctx, cudaStreamWaitEvent(st, ctx->ev_aux, 0));
      launch_reduce(ctx, p->policy_net, 2 * ctx->sms, grad_out, nullptr, st);
      ctx->launches += 5;
    }
    CUDA_OK(ctx, cudaGetLastError());
    return MPG_OK;
  }
  const int ntiles = (MB + TILE_R - 1) / TILE_R;
  const int grid = ntiles < ctx->sms ? ntiles : ctx->sms;
  CUDA_OK(ctx, cudaMemsetAsync(ctx->partial, 0, (size_t)grid * ctx->partial_stride * sizeof(float), st));
  rc = launch_rollout<true>(ctx, a, grid, st, ctx->cfg.env);
  if (rc) return rc;
  launch_reduce(ctx, p->policy_net, grid, grad_out, nullptr, st);
  ctx->launches++;
  CUDA_OK(ctx, cudaGetLastError());
  return MPG_OK;
}

int mpg_rollout_forward(mpg_ctx* ctx, const mpg_rollout_params* p, const float* obs, const float* start_actions,
                        const float* noise, float* returns_out, float* traj_obs, float* traj_rew, float* traj_act,
                        void* stream) {
  if (!ctx || !p || !obs) return fail(ctx, MPG_ERR_ARG, "null argument to mpg_rollout_forward%s");
  cudaStream_t st = (cudaStream_t)stream;
  RolloutArgs a;
  int rc = fill_rollout_args(ctx, p, a);
  if (rc) return rc;
  a.obs = obs; a.noise = noise; a.returns_out = returns_out;
  a.start_actions = start_actions; a.use_start_actions = start_actions != nullptr;
  a.traj_obs = traj_obs; a.traj_rew = traj_rew; a.traj_act = traj_act;
  a.noise_mode = noise ? 1 : (p->use_philox ? 2 : 0);
  if ((rc = prepare_far_steps(ctx, a, st))) return rc;
  const int MB = p->rows * p->M;
  int env = ctx->cfg.env;
  if (p->real_env) {
    if (ctx->cfg.env != MPG_ENV_PATH_TRACKING && ctx->cfg.env != MPG_ENV_PATH_TRACKING_REAL)
      return fail(ctx, MPG_ERR_UNSUPPORTED, "real_env rollouts exist for PathTracking only (the pendulum ground truth is mujoco)%s");
    env = MPG_ENV_PATH_TRACKING_REAL;
  }
  if (ctx->backend == MPG_BACKEND_TC) {
    const int ntiles = (MB + tc::ACT_ROWS - 1) / tc::ACT_ROWS;
    const int grid = ntiles < ctx->sms ? ntiles : ctx->sms;
    const tc::TcArgs ta = tc_args(ctx, a, p->policy_net, p->q_net);
    if (ctx->timing) cudaEventRecord(ctx->ev0, st);
    CUDA_OK(ctx, tc_launch_rollout<false>(env, ctx->act, ta, grid, st));
    if (ctx->timing) { cudaEventRecord(ctx->ev1, st); ctx->timed = 1; }
    ctx->launches++;
    return MPG_OK;
  }
  const int ntiles = (MB + TILE_R - 1) / TILE_R;
  const int grid = ntiles < ctx->sms ? ntiles : ctx->sms;
  return launch_rollout<false>(ctx, a, grid, st, env);
}

int mpg_returns_stats(mpg_ctx* ctx, const float* returns, int n_list, int rows, int M, float* out, void* stream) {
  if (!ctx || !returns || !out || n_list <= 0) return fail(ctx, MPG_ERR_ARG, "bad argument to mpg_returns_stats%s");
  if (n_list > MPG_MAX_LIST_LONG) return fail(ctx, MPG_ERR_ARG, "n_list too large: at most 64 (MPG_MAX_LIST_LONG)%s");
  returns_stats_kernel<<<dim3(n_list, RED_BLOCKS), 256, 0, (cudaStream_t)stream>>>(returns, n_list, rows, M, nullptr, ctx->stats_part);
  returns_stats_final_kernel<<<1, MPG_MAX_LIST_LONG, 0, (cudaStream_t)stream>>>(ctx->stats_part, n_list, out);
  ctx->launches += 2;
  CUDA_OK(ctx, cudaGetLastError());
  return MPG_OK;
}

int mpg_returns_tile_mean(mpg_ctx* ctx, const float* returns, int n_list, int rows, int M, float* out, void* stream) {
  if (!ctx || !returns || !out || n_list <= 0) return fail(ctx, MPG_ERR_ARG, "bad argument to mpg_returns_tile_mean%s");
  returns_stats_kernel<<<dim3(n_list, RED_BLOCKS), 256, 0, (cudaStream_t)stream>>>(returns, n_list, rows, M, out, nullptr);
  ctx->launches++;
  CUDA_OK(ctx, cudaGetLastError());
  return MPG_OK;
}

int mpg_q_grad(mpg_ctx* ctx, int net, int rows, int64_t global_rows, const float* obs, const float* act,
               const float* target, float* grad_out, float* loss_sum_out, void* stream) {
  if (!ctx || !obs || !act || !target || !grad_out || rows <= 0) return fail(ctx, MPG_ERR_ARG, "bad argument to mpg_q_grad%s");
  int rc = check_net(ctx, net);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  if (ctx->backend == MPG_BACKEND_TC && rows <= ctx->cfg.max_rows) {
    // tensor-core path: the rollout kernel in regression mode (horizon 0, given actions) + the dW kernel
    const mpg_config& c = ctx->cfg;
    // policy_net = net: unused in regression mode (actions are given, the policy part is skipped); fixes the gradient layout
    mpg_rollout_params p = horizon0_params(rows, net, net);
    p.full_bptt = 1;
    p.global_rows = global_rows;
    RolloutArgs a;
    if ((rc = fill_rollout_args(ctx, &p, a)) || (rc = q_scratch(ctx, rows))) return rc;
    a.use_start_actions = 1; a.start_actions = act; a.obs = obs; a.returns_out = ctx->qtmp.p;
    if (ctx->tc.act_ckpt.grow((size_t)rows * MAX_A) != cudaSuccess)
      return fail(ctx, MPG_ERR_CUDA, "cudaMalloc of the action checkpoints failed%s");
    tc::TcArgs ta = tc_args(ctx, a, net, net);
    ta.q_regress = 1; ta.q_target = target; ta.q_inv_rows = 1.f / (float)a.global_rows;
    const int ntiles = (rows + tc::ACT_ROWS - 1) / tc::ACT_ROWS;
    const int grid = ntiles < ctx->sms ? ntiles : ctx->sms;
    ta.store_steps = 1;
    if (ctx->tc.store.grow((size_t)ntiles * tc::SLOT_BYTES) != cudaSuccess)
      return fail(ctx, MPG_ERR_CUDA, "cudaMalloc of the dW operand store failed%s");
    ta.store = ctx->tc.store.p;
    // full hi + lo records always: a regression residual can be pure zero-mean noise (converged critic), the sum over the rows
    // then cancels to ~1/sqrt(rows) of its terms and the 2^-9 rounding of hi-only records would not average out relative
    // to it (measured 1.4e-3 at 262,144 rows); this GEMM is 0.04 ms, there is nothing to gain
    ta.rec_hi_only = 0;
    CUDA_OK(ctx, cudaMemsetAsync(ctx->partial, 0, (size_t)ctx->sms * ctx->partial_stride * sizeof(float), st));
    CUDA_OK(ctx, tc_launch_rollout<true>(c.env, ctx->act, ta, grid, st));
    launch_dw(ctx, ta, 0, ntiles, 0, ctx->sms, st);
    launch_reduce(ctx, net, ctx->sms, grad_out, nullptr, st);
    if (loss_sum_out) {
      sq_err_partial_kernel<<<RED_BLOCKS, 256, 0, st>>>(ctx->qtmp.p, target, rows, ctx->red_part);
      sum_partials_kernel<<<1, 1, 0, st>>>(ctx->red_part, loss_sum_out);
    }
    ctx->launches += 5;
    CUDA_OK(ctx, cudaGetLastError());
    return MPG_OK;
  }
  QGradArgs a;
  memset(&a, 0, sizeof(a));
  a.obs_dim = ctx->cfg.obs_dim; a.act_dim = ctx->cfg.act_dim; a.rows = rows;
  for (int i = 0; i < MPG_MAX_OBS; ++i) a.obs_scale[i] = ctx->cfg.obs_scale[i];
  a.inv_global_rows = 1.f / (float)(global_rows > 0 ? global_rows : rows);
  a.obs = obs; a.act = act; a.target = target;
  a.partial = ctx->partial; a.loss_partial = ctx->loss_partial; a.partial_stride = (long long)ctx->partial_stride;
  a.q = net_dev(ctx, net);
  const int ntiles = (rows + TILE_R - 1) / TILE_R;
  const int grid = ntiles < ctx->sms ? ntiles : ctx->sms;
  CUDA_OK(ctx, cudaMemsetAsync(ctx->partial, 0, (size_t)grid * ctx->partial_stride * sizeof(float), st));
  mlp_kernels(ctx->cfg.hidden, ctx->act).q_grad(a, grid, st);
  launch_reduce(ctx, net, grid, grad_out, loss_sum_out, st);
  ctx->launches += 2;
  CUDA_OK(ctx, cudaGetLastError());
  return MPG_OK;
}

// the FFMA evaluation kernel over a replay batch: with q_net < 0 the actions pi_policy(sigma obs) into out, else
// Q_q(sigma obs, a) into out and, with q2_net >= 0, Q_q2(sigma obs, a) into out2, a = act or pi_policy(sigma obs)
static int ffma_eval(mpg_ctx* ctx, int policy_net, int rows, const float* obs, const float* act, int q_net, float* out,
                     int q2_net, float* out2, void* stream) {
  const mpg_config& c = ctx->cfg;
  EvalArgs a;
  memset(&a, 0, sizeof(a));
  a.mode = q_net >= 0 ? 1 : 0; a.obs_dim = c.obs_dim; a.act_dim = c.act_dim; a.rows = rows;
  a.policy_out_tanh = c.policy_out_tanh; a.action_range = c.action_range;
  for (int i = 0; i < MPG_MAX_OBS; ++i) a.obs_scale[i] = c.obs_scale[i];
  a.obs = obs; a.act = act; a.out = out;
  if (!act) a.pol = net_dev(ctx, policy_net);
  if (q_net >= 0) a.q = net_dev(ctx, q_net);
  if (q2_net >= 0) { a.q2 = net_dev(ctx, q2_net); a.out2 = out2; }
  const int ntiles = (rows + TILE_R - 1) / TILE_R;
  const int grid = ntiles < ctx->sms ? ntiles : ctx->sms;
  mlp_kernels(c.hidden, ctx->act).eval(a, grid, (cudaStream_t)stream);
  ctx->launches++;
  CUDA_OK(ctx, cudaGetLastError());
  return MPG_OK;
}

static bool tc_eval_ok(const mpg_ctx* ctx, int rows) {
  return ctx->backend == MPG_BACKEND_TC && ctx->tc.ready && rows <= ctx->cfg.max_rows;
}

// tensor-core evaluation of Q(sigma obs, a), a = given actions or pi(sigma obs): the forward rollout kernel with horizon 0
// (one policy forward + one Q forward per row) -- 0.07 ms per 65,536 rows instead of 0.4 ms per MLP on the FFMA tile
// engine.  Like every rollout, its step 0 feeds the nets sigma * obs as given, the same input eval_kernel reads.
static int tc_q_eval(mpg_ctx* ctx, int q_net, int policy_net, int rows, const float* obs, const float* actions, float* out,
                     void* stream) {
  const mpg_rollout_params p = horizon0_params(rows, policy_net, q_net);
  return mpg_rollout_forward(ctx, &p, obs, actions, nullptr, out, nullptr, nullptr, nullptr, stream);
}

// Q_q(sigma obs, a) into out and, with q2_net >= 0, Q_q2(sigma obs, a) into out2, a = act or pi_policy(sigma obs): the
// evaluations of the target, TD-error and bootstrap entry points, on tensor cores where the handle runs them and the batch
// fits its capacity, else on the FFMA kernel (both Q nets in one launch)
static int eval_q(mpg_ctx* ctx, int policy_net, int rows, const float* obs, const float* act, int q_net, float* out,
                  int q2_net, float* out2, void* stream) {
  if (!tc_eval_ok(ctx, rows)) return ffma_eval(ctx, policy_net, rows, obs, act, q_net, out, q2_net, out2, stream);
  int rc = tc_q_eval(ctx, q_net, policy_net, rows, obs, act, out, stream);
  if (!rc && q2_net >= 0) rc = tc_q_eval(ctx, q2_net, policy_net, rows, obs, act, out2, stream);
  return rc;
}

// out = (base + shift) scale + coef min(q1, q2) - sub, q2 and sub optional: the arithmetic of the Q target
// (mpg_learner.py:126-134, 147-152), the TD error (136-144) and the n-step bootstrap (153-169)
__global__ void affine_q_kernel(int n, const float* __restrict__ base, float shift, float scale, float coef,
                                const float* __restrict__ q1, const float* __restrict__ q2, const float* __restrict__ sub,
                                float* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float q = q2 ? fminf(q1[i], q2[i]) : q1[i];
  out[i] = (base[i] + shift) * scale + coef * q - (sub ? sub[i] : 0.f);
}
static int affine_q(mpg_ctx* ctx, int rows, const float* base, float shift, float scale, float coef, const float* q2,
                    const float* sub, float* out, void* stream) {
  affine_q_kernel<<<(rows + 255) / 256, 256, 0, (cudaStream_t)stream>>>(rows, base, shift, scale, coef, ctx->qtmp.p, q2, sub, out);
  ctx->launches++;
  CUDA_OK(ctx, cudaGetLastError());
  return MPG_OK;
}

int mpg_policy_forward(mpg_ctx* ctx, int net, int rows, const float* obs, float* act_out, void* stream) {
  if (!ctx || !obs || !act_out || rows <= 0) return fail(ctx, MPG_ERR_ARG, "bad argument to mpg_policy_forward%s");
  int rc = check_net(ctx, net);
  if (rc) return rc;
  if (tc_eval_ok(ctx, rows) && (net == MPG_NET_POLICY || net == MPG_NET_POLICY_TARGET)) {
    // tensor-core forward kernel, horizon 0, no Q: the action of step 0 is the output (traj_act)
    const mpg_rollout_params p = horizon0_params(rows, net, -1);
    return mpg_rollout_forward(ctx, &p, obs, nullptr, nullptr, nullptr, nullptr, nullptr, act_out, stream);
  }
  return ffma_eval(ctx, net, rows, obs, nullptr, -1, act_out, -1, nullptr, stream);
}

int mpg_q_forward(mpg_ctx* ctx, int net, int rows, const float* obs, const float* act, float* q_out, void* stream) {
  if (!ctx || !obs || !act || !q_out || rows <= 0) return fail(ctx, MPG_ERR_ARG, "bad argument to mpg_q_forward%s");
  int rc = check_net(ctx, net);
  if (rc) return rc;
  if (tc_eval_ok(ctx, rows) && net != MPG_NET_POLICY && net != MPG_NET_POLICY_TARGET && ctx->nets[MPG_NET_POLICY].set)
    return tc_q_eval(ctx, net, MPG_NET_POLICY, rows, obs, act, q_out, stream);
  return ffma_eval(ctx, -1, rows, obs, act, net, q_out, -1, nullptr, stream);
}

int mpg_q_target(mpg_ctx* ctx, int double_q, int rows, const float* rew, const float* obs_tp1, float* target_out,
                 void* stream) {
  if (!ctx || !rew || !obs_tp1 || !target_out || rows <= 0) return fail(ctx, MPG_ERR_ARG, "bad argument to mpg_q_target%s");
  int rc = check_net(ctx, MPG_NET_POLICY_TARGET);
  if (!rc) rc = check_net(ctx, MPG_NET_Q1_TARGET);
  if (!rc && double_q) rc = check_net(ctx, MPG_NET_Q2_TARGET);
  if (!rc) rc = q_scratch(ctx, rows);
  if (!rc) rc = eval_q(ctx, MPG_NET_POLICY_TARGET, rows, obs_tp1, nullptr, MPG_NET_Q1_TARGET, ctx->qtmp.p,
                       double_q ? MPG_NET_Q2_TARGET : -1, ctx->qtmp2.p, stream);
  if (rc) return rc;
  const mpg_config& c = ctx->cfg;
  return affine_q(ctx, rows, rew, c.rew_shift, c.rew_scale, c.gamma, double_q ? ctx->qtmp2.p : nullptr, nullptr,
                  target_out, stream);
}

int mpg_q_bootstrap(mpg_ctx* ctx, int rows, const float* base, float coef, const float* obs, float* out, void* stream) {
  if (!ctx || !base || !obs || !out || rows <= 0) return fail(ctx, MPG_ERR_ARG, "bad argument to mpg_q_bootstrap%s");
  int rc = check_net(ctx, MPG_NET_POLICY_TARGET);
  if (!rc) rc = check_net(ctx, MPG_NET_Q1_TARGET);
  if (!rc) rc = q_scratch(ctx, rows);
  if (!rc) rc = eval_q(ctx, MPG_NET_POLICY_TARGET, rows, obs, nullptr, MPG_NET_Q1_TARGET, ctx->qtmp.p, -1, nullptr, stream);
  if (rc) return rc;
  return affine_q(ctx, rows, base, 0.f, 1.f, coef, nullptr, nullptr, out, stream);
}

int mpg_td_error(mpg_ctx* ctx, int rows, const float* obs, const float* act, const float* rew, const float* obs_tp1,
                 float* td_out, void* stream) {
  if (!ctx || !obs || !act || !rew || !obs_tp1 || !td_out || rows <= 0) return fail(ctx, MPG_ERR_ARG, "bad argument to mpg_td_error%s");
  int rc = check_net(ctx, MPG_NET_POLICY_TARGET);
  if (!rc) rc = check_net(ctx, MPG_NET_Q1_TARGET);
  if (!rc) rc = check_net(ctx, MPG_NET_Q1);
  if (!rc) rc = q_scratch(ctx, rows);
  if (!rc) rc = eval_q(ctx, MPG_NET_POLICY_TARGET, rows, obs_tp1, nullptr, MPG_NET_Q1_TARGET, ctx->qtmp.p, -1, nullptr, stream);
  // the policy does not enter Q1(sigma obs, act); the tensor-core kernel takes the online policy's weight images
  if (!rc) rc = eval_q(ctx, MPG_NET_POLICY, rows, obs, act, MPG_NET_Q1, ctx->qtmp2.p, -1, nullptr, stream);
  if (rc) return rc;
  const mpg_config& c = ctx->cfg;
  return affine_q(ctx, rows, rew, c.rew_shift, c.rew_scale, c.gamma, nullptr, ctx->qtmp2.p, td_out, stream);
}

int mpg_model_reset(mpg_ctx* ctx, int rows, const float* obs, float* state_out, void* stream) {
  if (!ctx || !obs || !state_out || rows <= 0) return fail(ctx, MPG_ERR_ARG, "bad argument to mpg_model_reset%s");
  cudaStream_t st = (cudaStream_t)stream;
  with_env(ctx->cfg.env, false, [&](auto env, auto) {
    model_reset_kernel<decltype(env)::value><<<(rows + 127) / 128, 128, 0, st>>>(rows, ctx->cfg.obs_dim, obs, state_out);
  });
  ctx->launches++;
  CUDA_OK(ctx, cudaGetLastError());
  return MPG_OK;
}

int mpg_model_step(mpg_ctx* ctx, int rows, const float* state_in, const float* action, const float* eps,
                   float* state_out, float* obs_out, float* rew_out, void* stream) {
  if (!ctx || !state_in || !action || !state_out || rows <= 0) return fail(ctx, MPG_ERR_ARG, "bad argument to mpg_model_step%s");
  cudaStream_t st = (cudaStream_t)stream;
  with_env(ctx->cfg.env, false, [&](auto env, auto) {
    model_step_kernel<decltype(env)::value><<<(rows + 127) / 128, 128, 0, st>>>(
        rows, ctx->cfg.obs_dim, ctx->cfg.num_future_data, state_in, action, eps, state_out, obs_out, rew_out);
  });
  ctx->launches++;
  CUDA_OK(ctx, cudaGetLastError());
  return MPG_OK;
}

int mpg_model_step_bwd(mpg_ctx* ctx, int rows, const float* state_in, const float* action, const float* eps,
                       const float* g_obs_out, const float* g_rew_out, const float* g_state_out, float* g_state_in,
                       float* g_action, void* stream) {
  if (!ctx || !state_in || !action || !g_state_in || !g_action || rows <= 0)
    return fail(ctx, MPG_ERR_ARG, "bad argument to mpg_model_step_bwd%s");
  cudaStream_t st = (cudaStream_t)stream;
  if (!with_env(ctx->cfg.env, true, [&](auto env, auto) {
        model_step_bwd_kernel<decltype(env)::value><<<(rows + 127) / 128, 128, 0, st>>>(
            rows, ctx->cfg.obs_dim, ctx->cfg.num_future_data, state_in, action, eps, g_obs_out, g_rew_out, g_state_out,
            g_state_in, g_action);
      }))
    return fail(ctx, MPG_ERR_UNSUPPORTED, "the real environment is forward only%s");
  ctx->launches++;
  CUDA_OK(ctx, cudaGetLastError());
  return MPG_OK;
}

int mpg_env_step(mpg_ctx* ctx, int rows, const float* state_in, const float* action, float* state_out, float* obs_out,
                 float* rew_out, int32_t* done_out, void* stream) {
  if (!ctx || !state_in || !action || !state_out || rows <= 0) return fail(ctx, MPG_ERR_ARG, "bad argument to mpg_env_step%s");
  if (ctx->cfg.env != MPG_ENV_PATH_TRACKING_REAL) return fail(ctx, MPG_ERR_STATE, "mpg_env_step needs a handle created with MPG_ENV_PATH_TRACKING_REAL%s");
  env_step_kernel<<<(rows + 127) / 128, 128, 0, (cudaStream_t)stream>>>(rows, ctx->cfg.obs_dim, ctx->cfg.num_future_data, state_in,
                                                                        action, state_out, obs_out, rew_out, done_out);
  ctx->launches++;
  CUDA_OK(ctx, cudaGetLastError());
  return MPG_OK;
}

int mpg_env_sample(mpg_ctx* ctx, int policy_net, int agents, int steps, float explore_sigma, const float* explore_noise,
                   const float* reset_obs, float* state, float* obs, float* out_obs, float* out_act, float* out_rew,
                   float* out_obs_tp1, float* out_done, void* stream) {
  if (!ctx || !state || !obs || !out_obs || !out_act || !out_rew || !out_obs_tp1 || !out_done || agents <= 0
      || steps <= 0)
    return fail(ctx, MPG_ERR_ARG, "bad argument to mpg_env_sample%s");
  if (ctx->cfg.env != MPG_ENV_PATH_TRACKING)
    return fail(ctx, MPG_ERR_UNSUPPORTED, "mpg_env_sample: the fused sampler is built for the PathTracking policy handle%s");
  int rc = check_net(ctx, policy_net);
  if (rc) return rc;
  SampleArgs a;
  memset(&a, 0, sizeof(a));
  a.agents = agents; a.steps = steps; a.obs_dim = ctx->cfg.obs_dim; a.act_dim = ctx->cfg.act_dim;
  a.nfd = ctx->cfg.num_future_data; a.policy_out_tanh = ctx->cfg.policy_out_tanh; a.action_range = ctx->cfg.action_range;
  a.sigma = explore_sigma;
  for (int i = 0; i < MPG_MAX_OBS; ++i) a.obs_scale[i] = ctx->cfg.obs_scale[i];
  a.explore_noise = explore_noise; a.reset_obs = reset_obs; a.state = state; a.obs = obs;
  a.out_obs = out_obs; a.out_act = out_act; a.out_rew = out_rew; a.out_obs_tp1 = out_obs_tp1; a.out_done = out_done;
  a.net = net_dev(ctx, policy_net);
  mlp_kernels(ctx->cfg.hidden, ctx->act).env_sample(a, (agents + TILE_R - 1) / TILE_R, (cudaStream_t)stream);
  ctx->launches++;
  CUDA_OK(ctx, cudaGetLastError());
  return MPG_OK;
}

int mpg_compute_rewards(mpg_ctx* ctx, int rows, const float* state, const float* scaled_action, float* rew_out,
                        void* stream) {
  if (!ctx || !state || !rew_out || rows <= 0) return fail(ctx, MPG_ERR_ARG, "bad argument to mpg_compute_rewards%s");
  if ((ctx->cfg.env == MPG_ENV_PATH_TRACKING || ctx->cfg.env == MPG_ENV_PATH_TRACKING_REAL) && !scaled_action)
    return fail(ctx, MPG_ERR_ARG, "PathTracking rewards need actions%s");
  cudaStream_t st = (cudaStream_t)stream;
  with_env(ctx->cfg.env, false, [&](auto env, auto) {
    rewards_kernel<decltype(env)::value><<<(rows + 127) / 128, 128, 0, st>>>(rows, state, scaled_action, rew_out);
  });
  ctx->launches++;
  CUDA_OK(ctx, cudaGetLastError());
  return MPG_OK;
}

int mpg_clip_global_norm(mpg_ctx* ctx, float* grad, int n, float clip, float* norm_out, void* stream) {
  if (!ctx || !grad || n <= 0 || !(clip > 0.f)) return fail(ctx, MPG_ERR_ARG, "bad argument to mpg_clip_global_norm%s");
  sumsq_partial_kernel<<<RED_BLOCKS, 256, 0, (cudaStream_t)stream>>>(grad, n, ctx->red_part + RED_BLOCKS);
  clip_apply_kernel<<<RED_BLOCKS, 256, 0, (cudaStream_t)stream>>>(grad, n, clip, ctx->red_part + RED_BLOCKS, norm_out);
  ctx->launches += 2;
  CUDA_OK(ctx, cudaGetLastError());
  return MPG_OK;
}

int mpg_philox_noise(mpg_ctx* ctx, const mpg_rollout_params* p, float* out, void* stream) {
  if (!ctx || !p || !out) return fail(ctx, MPG_ERR_ARG, "bad argument to mpg_philox_noise%s");
  const long long total = (long long)p->horizon * p->rows * p->M;
  if (total <= 0) return MPG_OK;
  const long long gr = p->global_rows > 0 ? p->global_rows : p->rows;
  philox_noise_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(p->noise_seed, gr, p->row_offset,
                                                                                        p->rows, p->M, p->horizon, out);
  ctx->launches++;
  CUDA_OK(ctx, cudaGetLastError());
  return MPG_OK;
}

}  // extern "C"

// =====================================================================================================
// prioritized replay
// =====================================================================================================
struct mpg_replay {
  int capacity = 0, maxsize = 0, obs_dim = 0, act_dim = 0, size = 0, next_idx = 0;   // capacity: power of two of the trees (it_capacity); maxsize: ring size
  double alpha = 0.6, beta = 0.4;
  float *obs = nullptr, *act = nullptr, *rew = nullptr, *obs1 = nullptr, *done = nullptr;
  double *sum_tree = nullptr, *min_tree = nullptr, *max_prio = nullptr;
  int* owner = nullptr;
  char err[256];
};

namespace {
thread_local char g_replay_err[256] = "";
int rfail(mpg_replay* rb, int code, const char* msg) {
  snprintf(rb ? rb->err : g_replay_err, 256, "%s", msg);
  return code;
}
#define RB_CUDA(rb, expr)                                                          \
  do {                                                                             \
    cudaError_t e__ = (expr);                                                      \
    if (e__ != cudaSuccess) return rfail(rb, MPG_ERR_CUDA, cudaGetErrorString(e__)); \
  } while (0)

int rebuild_tree(mpg_replay* rb, cudaStream_t st) {
  int first = rb->capacity / 2;
  for (; first > 512; first >>= 1) replay_level_kernel<<<(first + 255) / 256, 256, 0, st>>>(first, rb->sum_tree, rb->min_tree);
  if (first >= 1) replay_top_kernel<<<1, 512, 0, st>>>(first, rb->sum_tree, rb->min_tree);
  RB_CUDA(rb, cudaGetLastError());
  return MPG_OK;
}
}  // namespace

extern "C" {

const char* mpg_replay_last_error(const mpg_replay* rb) { return rb ? rb->err : g_replay_err; }
int mpg_replay_size(const mpg_replay* rb) { return rb ? rb->size : -1; }

int mpg_replay_create(int capacity, int obs_dim, int act_dim, double alpha, double beta, mpg_replay** out) {
  if (!out || capacity <= 0 || obs_dim <= 0 || act_dim <= 0 || !(alpha > 0)) return rfail(nullptr, MPG_ERR_ARG, "bad replay config (alpha must be > 0)");
  *out = nullptr;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return rfail(nullptr, MPG_ERR_CUDA, "no CUDA device: mpg_b200 has no CPU fallback");
  mpg_replay* rb = new (std::nothrow) mpg_replay();
  if (!rb) return rfail(nullptr, MPG_ERR_ARG, "out of host memory");
  rb->err[0] = 0;
  int cap = 1;
  while (cap < capacity) cap *= 2;                       // it_capacity (buffer.py:119-121)
  rb->capacity = cap; rb->maxsize = capacity; rb->obs_dim = obs_dim; rb->act_dim = act_dim; rb->alpha = alpha; rb->beta = beta;
  bool ok = cudaMalloc(&rb->obs, (size_t)cap * obs_dim * 4) == cudaSuccess && cudaMalloc(&rb->obs1, (size_t)cap * obs_dim * 4) == cudaSuccess
            && cudaMalloc(&rb->act, (size_t)cap * act_dim * 4) == cudaSuccess && cudaMalloc(&rb->rew, (size_t)cap * 4) == cudaSuccess
            && cudaMalloc(&rb->done, (size_t)cap * 4) == cudaSuccess && cudaMalloc(&rb->sum_tree, (size_t)2 * cap * 8) == cudaSuccess
            && cudaMalloc(&rb->min_tree, (size_t)2 * cap * 8) == cudaSuccess && cudaMalloc(&rb->max_prio, 8) == cudaSuccess
            && cudaMalloc(&rb->owner, (size_t)cap * 4) == cudaSuccess;
  if (!ok) { mpg_replay_destroy(rb); return rfail(nullptr, MPG_ERR_CUDA, "cudaMalloc of the replay storage failed"); }
  cudaMemset(rb->sum_tree, 0, (size_t)2 * cap * 8);
  std::vector<double> inf((size_t)2 * cap, INFINITY);     // neutral element of the min tree
  cudaMemcpy(rb->min_tree, inf.data(), inf.size() * 8, cudaMemcpyHostToDevice);
  const double one = 1.0;                                 // _max_priority = 1.0 (buffer.py:125)
  cudaMemcpy(rb->max_prio, &one, 8, cudaMemcpyHostToDevice);
  cudaMemset(rb->owner, 0xFF, (size_t)cap * 4);
  *out = rb;
  return MPG_OK;
}

void mpg_replay_destroy(mpg_replay* rb) {
  if (!rb) return;
  cudaFree(rb->obs); cudaFree(rb->obs1); cudaFree(rb->act); cudaFree(rb->rew); cudaFree(rb->done);
  cudaFree(rb->sum_tree); cudaFree(rb->min_tree); cudaFree(rb->max_prio); cudaFree(rb->owner);
  delete rb;
}

int mpg_replay_add(mpg_replay* rb, int n, const float* obs, const float* act, const float* rew, const float* obs_tp1,
                   const float* done, const float* priorities, void* stream) {
  if (!rb || n <= 0 || !obs || !act || !rew || !obs_tp1) return rfail(rb, MPG_ERR_ARG, "bad argument to mpg_replay_add");
  if (n > rb->maxsize) return rfail(rb, MPG_ERR_ARG, "more transitions than the buffer capacity in one add");
  cudaStream_t st = (cudaStream_t)stream;
  replay_write_kernel<<<(n + 127) / 128, 128, 0, st>>>(n, rb->capacity, rb->maxsize, rb->next_idx, rb->obs_dim, rb->act_dim, obs, act, rew,
                                                        obs_tp1, done, priorities, rb->max_prio, rb->alpha, rb->obs, rb->act,
                                                        rb->rew, rb->obs1, rb->done, rb->sum_tree, rb->min_tree);
  rb->next_idx = (rb->next_idx + n) % rb->maxsize;                       // storage wraps at _maxsize (buffer.py:52-60)
  rb->size = rb->size + n < rb->maxsize ? rb->size + n : rb->maxsize;
  return rebuild_tree(rb, st);
}

int mpg_replay_sample(mpg_replay* rb, int n, const float* u, int32_t* idx_out, float* weights_out, float* obs_out,
                      float* act_out, float* rew_out, float* obs_tp1_out, float* done_out, void* stream) {
  if (!rb || n <= 0 || !u || !idx_out || !obs_out || !act_out || !rew_out || !obs_tp1_out || !done_out)
    return rfail(rb, MPG_ERR_ARG, "bad argument to mpg_replay_sample");
  if (rb->size == 0) return rfail(rb, MPG_ERR_STATE, "sampling from an empty replay buffer");
  replay_sample_kernel<<<(n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(
      n, rb->capacity, rb->size, rb->obs_dim, rb->act_dim, rb->beta, u, rb->sum_tree, rb->min_tree, rb->obs, rb->act, rb->rew,
      rb->obs1, rb->done, idx_out, weights_out, obs_out, act_out, rew_out, obs_tp1_out, done_out);
  RB_CUDA(rb, cudaGetLastError());
  return MPG_OK;
}

int mpg_replay_update_priorities(mpg_replay* rb, int n, const int32_t* idx, const float* priorities, void* stream) {
  if (!rb || n <= 0 || !idx || !priorities) return rfail(rb, MPG_ERR_ARG, "bad argument to mpg_replay_update_priorities");
  cudaStream_t st = (cudaStream_t)stream;
  const int g = (n + 127) / 128;
  replay_owner_kernel<<<g, 128, 0, st>>>(n, idx, rb->owner);
  replay_set_prio_kernel<<<g, 128, 0, st>>>(n, rb->capacity, idx, priorities, rb->alpha, rb->owner, rb->sum_tree, rb->min_tree);
  replay_owner_reset_kernel<<<g, 128, 0, st>>>(n, idx, rb->owner);
  replay_max_prio_kernel<<<1, 256, 0, st>>>(n, priorities, rb->max_prio);
  return rebuild_tree(rb, st);
}

int mpg_replay_tree_stats(mpg_replay* rb, double* sum_out, double* min_out, double* max_priority_out, void* stream) {
  if (!rb) return MPG_ERR_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  if (sum_out) RB_CUDA(rb, cudaMemcpyAsync(sum_out, rb->sum_tree + 1, 8, cudaMemcpyDeviceToHost, st));
  if (min_out) RB_CUDA(rb, cudaMemcpyAsync(min_out, rb->min_tree + 1, 8, cudaMemcpyDeviceToHost, st));
  if (max_priority_out) RB_CUDA(rb, cudaMemcpyAsync(max_priority_out, rb->max_prio, 8, cudaMemcpyDeviceToHost, st));
  RB_CUDA(rb, cudaStreamSynchronize(st));
  return MPG_OK;
}

}  // extern "C"
