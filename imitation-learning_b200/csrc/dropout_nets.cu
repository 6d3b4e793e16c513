// Networks with dropout (models.py:48-69 with input_dropout / dropout > 0) and the two algorithms that use them:
//   RED  (models.py:252-284, training.py:68-75): predictor / target embedding networks, regression of the predictor onto the frozen random target,
//        kernel-median bandwidth, reward exp(-sigma mean((pred - target)^2));
//   DRIL (models.py:104-120): a dropout policy trained by behavioural cloning; reward = +-1 by the variance of pi(a|s) over a 5-member MC-dropout ensemble.
// Dropout sits BEFORE the activation (Linear -> Dropout -> activation, models.py:54-61) and on the input. Masks are explicit inputs, pre-scaled
// {0, 1 / (1 - p)} (il_fill_dropout_mask draws them on the device; tests inject them), so every call is deterministic and graph-capturable.
// The MLP passes are programs over the replica-batched grouped GEMMs with small element-wise kernels for the mask / activation steps.
#include "mlp.cuh"

namespace {

unsigned dblocks(int64_t n) { return (unsigned)((n + 255) / 256); }

struct DropMasks {
  const float* in;                      // [G, n, dims[0]] or nullptr
  const float* hid[IL_MAX_LAYERS];      // [G, n, dims[l + 1]] for hidden layer l, or nullptr
};

// out[g, i, k] = X[g, i / rep, k] * (mask ? mask[g, i, k] : 1)   (contiguous [G, n, K]; rep = row repetition of the source, DRIL ensemble)
__global__ void input_mask_kernel(const float* __restrict__ X, int64_t x_gs, int ldx, int rep, const float* __restrict__ mask, float* __restrict__ out, int G, int n, int K) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (int64_t)G * n * K) return;
  const int k = (int)(t % K);
  const int64_t gi = t / K;
  const int g = (int)(gi / n), i = (int)(gi % n);
  const float v = X[(int64_t)g * x_gs + (int64_t)(i / rep) * ldx + k];
  out[t] = mask ? v * mask[t] : v;
}
// y = act(z * mask) in place
__global__ void dropout_act_kernel(float* __restrict__ z, const float* __restrict__ mask, int64_t n, int act) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n) z[t] = act_apply(mask ? z[t] * mask[t] : z[t], act);
}
// t = t * act'(y) * mask in place (y = activation output)
__global__ void dropout_bwd_kernel(float* __restrict__ t_, const float* __restrict__ y, const float* __restrict__ mask, int64_t n, int act) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n) t_[t] = t_[t] * act_grad_from_output(y[t], act) * (mask ? mask[t] : 1.f);
}
// Bernoulli(1 - p) / (1 - p) from Philox4x32-10
__global__ void dropout_mask_kernel(float* __restrict__ out, int64_t n, float p, uint64_t seed, uint64_t stream_id, const uint64_t* __restrict__ counter) {
  const int64_t i4 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i4 * 4 >= n) return;
  const uint64_t c = (counter ? *counter : 0ull) + (uint64_t)i4;
  const uint4 r = philox4x32_10(make_uint4((uint32_t)c, (uint32_t)(c >> 32), (uint32_t)stream_id, (uint32_t)(stream_id >> 32)), make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
  const float keep = 1.f / (1.f - p);
  const uint32_t bits[4] = {r.x, r.y, r.z, r.w};
  for (int e = 0; e < 4; ++e)
    if (i4 * 4 + e < n) out[i4 * 4 + e] = u32_to_unit(bits[e]) >= p ? keep : 0.f;
}

// forward: hid[l] = act((x_l W_l^T + b_l) * mask_l), out = x_{L-1} W_L^T + b_L. X must already carry the input mask (see input_mask_kernel).
int mlp_forward_dropout(il_handle* h, const il_mlp* m, int G, int n, MatView X, const DropMasks& mk, const MlpActs& acts, float* out, int64_t out_gs, int ld_out, cudaStream_t st) {
  const MlpOffsets o = mlp_offsets(m->dims, m->n_layers);
  const int L = m->n_layers;
  for (int l = 0; l < L; ++l) {
    GemmArgs a{};
    if (l == 0) { a.A = X.ptr; a.a_gs = X.gs; a.a_gdiv = X.gdiv; a.lda = X.ld; }
    else { a.A = acts.hid[l - 1]; a.a_gs = (int64_t)n * m->dims[l]; a.a_gdiv = 1; a.lda = m->dims[l]; }
    a.a_kmajor = 1;
    a.B = m->params + o.w[l]; a.b_gs = m->stride; a.b_gdiv = 1; a.ldb = m->dims[l]; a.b_kmajor = 1;
    a.bias = m->params + o.b[l]; a.bias_gs = m->stride; a.act = -1;
    if (l == L - 1) { a.C = out; a.c_gs = out_gs; a.ldc = ld_out; }
    else { a.C = acts.hid[l]; a.c_gs = (int64_t)n * m->dims[l + 1]; a.ldc = m->dims[l + 1]; }
    a.M = n; a.N = m->dims[l + 1]; a.K = m->dims[l]; a.G = G;
    IL_TRY(launch_gemm(h, a, st));
    if (l < L - 1) {
      const int64_t cnt = (int64_t)G * n * m->dims[l + 1];
      IL_LAUNCH(h, dropout_act_kernel, dblocks(cnt), 256, 0, st, acts.hid[l], mk.hid[l], cnt, m->activation);
    }
  }
  return 0;
}

// backward from dOut (gradient at the linear head); grads in the flat parameter layout
int mlp_backward_dropout(il_handle* h, const il_mlp* m, int G, int n, MatView X, const DropMasks& mk, const MlpActs& acts, MatView dOut, float* grads, int64_t grad_stride, float* tmpA,
                         float* tmpB, cudaStream_t st) {
  const MlpOffsets o = mlp_offsets(m->dims, m->n_layers);
  const int L = m->n_layers;
  MatView dZ = dOut;
  float* next_tmp = tmpA;
  for (int l = L - 1; l >= 0; --l) {
    MatView Xin = l == 0 ? X : MatView{acts.hid[l - 1], (int64_t)n * m->dims[l], 1, m->dims[l]};
    {
      GemmArgs a{};
      a.A = dZ.ptr; a.a_gs = dZ.gs; a.a_gdiv = dZ.gdiv; a.lda = dZ.ld; a.a_kmajor = 0;
      a.B = Xin.ptr; a.b_gs = Xin.gs; a.b_gdiv = Xin.gdiv; a.ldb = Xin.ld; a.b_kmajor = 0;
      a.C = grads + o.w[l]; a.c_gs = grad_stride; a.ldc = m->dims[l]; a.act = -1;
      a.colsum = grads + o.b[l]; a.colsum_gs = grad_stride;
      a.M = m->dims[l + 1]; a.N = m->dims[l]; a.K = n; a.G = G;
      IL_TRY(launch_gemm(h, a, st));
    }
    if (l > 0) {
      GemmArgs a{};
      a.A = dZ.ptr; a.a_gs = dZ.gs; a.a_gdiv = dZ.gdiv; a.lda = dZ.ld; a.a_kmajor = 1;
      a.B = m->params + o.w[l]; a.b_gs = m->stride; a.b_gdiv = 1; a.ldb = m->dims[l]; a.b_kmajor = 0;
      a.C = next_tmp; a.c_gs = (int64_t)n * m->dims[l]; a.ldc = m->dims[l]; a.act = -1;
      a.M = n; a.N = m->dims[l]; a.K = m->dims[l + 1]; a.G = G;
      IL_TRY(launch_gemm(h, a, st));
      const int64_t cnt = (int64_t)G * n * m->dims[l];
      IL_LAUNCH(h, dropout_bwd_kernel, dblocks(cnt), 256, 0, st, next_tmp, acts.hid[l - 1], mk.hid[l - 1], cnt, m->activation);
      dZ = MatView{next_tmp, (int64_t)n * m->dims[l], 1, m->dims[l]};
      next_tmp = next_tmp == tmpA ? tmpB : tmpA;
    }
  }
  return 0;
}

struct Carve {
  char* p;
  int64_t used;
  float* take(int64_t floats) {
    float* r = p ? reinterpret_cast<float*>(p + used) : nullptr;
    used += il_align_up(floats * 4, 256);
    return r;
  }
};
void acts_carve(Carve& c, const il_mlp* m, int G, int n, MlpActs* a) {
  for (int l = 0; l < IL_MAX_LAYERS; ++l) a->hid[l] = nullptr;
  for (int l = 0; l + 1 < m->n_layers; ++l) a->hid[l] = c.take((int64_t)G * n * m->dims[l + 1]);
}
int hidden_max(const il_mlp* m) {
  int d = 1;
  for (int l = 1; l < m->n_layers; ++l) d = m->dims[l] > d ? m->dims[l] : d;
  return d;
}

// ---- RED ----------------------------------------------------------------------------------------------------------------------
// d = pred - targ;  loss[r] = mean_b w_b mean_j d^2;  dpred = 2 w_b d / (din B). One CTA per replica.
__global__ void __launch_bounds__(256) red_loss_kernel(const float* __restrict__ pred, const float* __restrict__ targ, const float* __restrict__ rows, int64_t rs, int row, int off_weight,
                                                       float* __restrict__ dpred, float* __restrict__ out_loss, int B, int din) {
  __shared__ float red[32];
  const int r = blockIdx.x;
  float loss = 0.f;
  for (int i = threadIdx.x; i < B * din; i += blockDim.x) {
    const int b = i / din;
    const float w = rows[(int64_t)r * rs + (int64_t)b * row + off_weight];
    const int64_t idx = (int64_t)r * B * din + i;
    const float d = pred[idx] - targ[idx];
    loss += w * d * d;
    dpred[idx] = 2.f * w * d / ((float)din * (float)B);
  }
  loss = block_sum(loss, red);
  if (threadIdx.x == 0 && out_loss) out_loss[r] = loss / ((float)din * (float)B);
}
// reward[r, b] = exp(-sigma[r] * mean_j (pred - targ)^2)   (models.py:282-284)
__global__ void red_reward_kernel(const float* __restrict__ pred, const float* __restrict__ targ, const float* __restrict__ sigma, float* __restrict__ reward, int64_t reward_rs, int reward_ld,
                                  int R, int B, int din) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (int64_t)R * B) return;
  const int r = (int)(t / B), b = (int)(t % B);
  float s = 0.f;
  for (int j = 0; j < din; ++j) { const float d = pred[t * din + j] - targ[t * din + j]; s = fmaf(d, d, s); }
  reward[(int64_t)r * reward_rs + (int64_t)b * reward_ld] = expf(-sigma[r] * (s / (float)din));
}
// D[r, i, j] = mean_k (pred[r, i, k] - targ[r, j, k])^2   (_squared_distance, models.py:25-28)
__global__ void red_pairwise_kernel(const float* __restrict__ pred, const float* __restrict__ targ, float* __restrict__ D, int R, int B, int din) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (int64_t)R * B * B) return;
  const int j = (int)(t % B);
  const int64_t ri = t / B;
  const int r = (int)(ri / B);
  const float* a = pred + ri * din;
  const float* b = targ + ((int64_t)r * B + j) * din;
  float s = 0.f;
  for (int k = 0; k < din; ++k) { const float d = a[k] - b[k]; s += d * d; }
  D[t] = s / (float)din;
}
// sigma[r] = 1 / (lower median of the n non-negative values of D[r]) (torch.median semantics): bit-pattern bisection on the k-th smallest. One CTA per replica.
__global__ void __launch_bounds__(256) red_median_kernel(const float* __restrict__ D, int64_t n, float* __restrict__ sigma) {
  __shared__ float red[32];
  const float* d = D + (int64_t)blockIdx.x * n;
  const int64_t k = (n - 1) / 2;  // 0-based rank of the lower median
  uint32_t lo = 0u, hi = 0x7f800000u;  // non-negative finite floats order like their bit patterns
  while (lo < hi) {
    const uint32_t mid = lo + (hi - lo) / 2;
    float cnt = 0.f;
    for (int64_t i = threadIdx.x; i < n; i += blockDim.x) cnt += __float_as_uint(d[i]) <= mid ? 1.f : 0.f;
    cnt = block_sum(cnt, red);
    if ((int64_t)cnt >= k + 1) hi = mid; else lo = mid + 1;
  }
  if (threadIdx.x == 0) sigma[blockIdx.x] = 1.f / __uint_as_float(lo);
}

struct RedWs {
  float *xin, *pred, *targ, *dpred, *tmpA, *tmpB, *grads, *dist;
  MlpActs pacts, tacts;
  int64_t bytes;
};
RedWs red_layout(const il_red* d, int R, int B, char* base, bool with_dist) {
  RedWs w{};
  Carve c{base, 0};
  const int din = d->predictor.dims[0], hm = hidden_max(&d->predictor);
  w.xin = c.take((int64_t)R * B * din);
  acts_carve(c, &d->predictor, R, B, &w.pacts);
  acts_carve(c, &d->target, R, B, &w.tacts);
  w.pred = c.take((int64_t)R * B * din); w.targ = c.take((int64_t)R * B * din); w.dpred = c.take((int64_t)R * B * din);
  w.tmpA = c.take((int64_t)R * B * hm); w.tmpB = c.take((int64_t)R * B * hm);
  w.grads = c.take((int64_t)R * d->predictor.stride);
  w.dist = with_dist ? c.take((int64_t)R * B * B) : nullptr;
  w.bytes = c.used;
  return w;
}
int red_validate(const il_red* d, const il_batch* b, const char* what) {
  IL_CHECK(d && b && b->rows, "%s: null argument", what);
  IL_TRY(mlp_validate(&d->predictor, what));
  IL_TRY(mlp_validate(&d->target, what));
  const int din = d->state_only ? b->S : b->S + b->A;
  IL_CHECK(d->predictor.dims[0] == din && d->predictor.dims[d->predictor.n_layers] == din && d->target.dims[0] == din && d->target.dims[d->target.n_layers] == din,
           "%s: embedding networks must map %d -> %d", what, din, din);
  IL_CHECK(b->row == row_layout(b->S, b->A).len, "%s: bad row length", what);
  return 0;
}
// prediction (with the given masks) and target for the rows of `b`
int red_forward(il_handle* h, const il_red* d, int R, const il_batch* b, const DropMasks& mk, RedWs& w, cudaStream_t st) {
  const int B = b->B, din = d->predictor.dims[0];
  MatView X{b->rows, b->replica_stride, 1, b->row};
  if (mk.in) {
    IL_LAUNCH(h, input_mask_kernel, dblocks((int64_t)R * B * din), 256, 0, st, b->rows, b->replica_stride, b->row, 1, mk.in, w.xin, R, B, din);
    IL_TRY(mlp_forward_dropout(h, &d->predictor, R, B, MatView{w.xin, (int64_t)B * din, 1, din}, mk, w.pacts, w.pred, (int64_t)B * din, din, st));
  } else {
    IL_TRY(mlp_forward_dropout(h, &d->predictor, R, B, X, mk, w.pacts, w.pred, (int64_t)B * din, din, st));
  }
  DropMasks none{};
  return mlp_forward_dropout(h, &d->target, R, B, X, none, w.tacts, w.targ, (int64_t)B * din, din, st);
}
DropMasks masks_of(const float* in, const float* const* hid) {
  DropMasks m{};
  m.in = in;
  for (int l = 0; l < IL_MAX_LAYERS; ++l) m.hid[l] = hid ? hid[l] : nullptr;
  return m;
}

// ---- DRIL -----------------------------------------------------------------------------------------------------------------------
// reward[r, b] = +1 if var_e exp(log_prob[r, b * E + e]) <= q else -1   (unbiased variance over the ensemble, models.py:104-120)
__global__ void dril_reward_kernel(const float* __restrict__ log_prob, int R, int B, int E, const float* __restrict__ q, int q_shared, float* __restrict__ reward, int64_t reward_rs, int reward_ld,
                                   float* __restrict__ variance) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (int64_t)R * B) return;
  const int r = (int)(t / B), b = (int)(t % B);
  float mean = 0.f;
  for (int e = 0; e < E; ++e) mean += expf(log_prob[t * E + e]);
  mean /= (float)E;
  float var = 0.f;
  for (int e = 0; e < E; ++e) { const float d = expf(log_prob[t * E + e]) - mean; var = fmaf(d, d, var); }
  var /= (float)(E - 1);
  if (variance) variance[t] = var;
  if (reward) reward[(int64_t)r * reward_rs + (int64_t)b * reward_ld] = var <= q[q_shared ? 0 : r] ? 1.f : -1.f;
}

}  // namespace

extern "C" int il_fill_dropout_mask(il_handle* h, float* out, int64_t n, float p, uint64_t seed, uint64_t stream_id, const uint64_t* counter, void* stream) {
  IL_CHECK(h && out && n > 0 && p >= 0.f && p < 1.f, "il_fill_dropout_mask: bad argument (p = %f)", (double)p);
  IL_LAUNCH(h, dropout_mask_kernel, dblocks((n + 3) / 4), 256, 0, (cudaStream_t)stream, out, n, p, seed, stream_id, counter);
  return 0;
}

extern "C" int64_t il_red_workspace_bytes(const il_red* d, int R, int B) {
  if (!d || R <= 0 || B <= 0) return -1;
  return red_layout(d, R, B, nullptr, true).bytes;
}

extern "C" int il_red_update(il_handle* h, const il_red_update_args* a, void* stream) {
  IL_CHECK(h && a, "il_red_update: null argument");
  cudaStream_t st = (cudaStream_t)stream;
  const il_red* d = &a->disc;
  IL_TRY(red_validate(d, &a->batch, "il_red_update"));
  const int R = a->R, B = a->batch.B, din = d->predictor.dims[0];
  IL_CHECK(R > 0 && a->opt.m && a->opt.v && a->opt.step && a->workspace && a->workspace_bytes >= il_red_workspace_bytes(d, R, B), "il_red_update: bad optimiser state / workspace");
  RedWs w = red_layout(d, R, B, static_cast<char*>(a->workspace), true);
  const DropMasks mk = masks_of(a->mask_in, a->mask_hid);
  const RowLayout RL = row_layout(a->batch.S, a->batch.A);
  IL_TRY(launch_tick(h, a->opt.step, nullptr, nullptr, st));
  IL_TRY(red_forward(h, d, R, &a->batch, mk, w, st));
  IL_LAUNCH(h, red_loss_kernel, R, 256, 0, st, w.pred, w.targ, a->batch.rows, a->batch.replica_stride, a->batch.row, RL.weight, w.dpred, a->out_loss, B, din);
  IL_CUDA(cudaMemsetAsync(w.grads, 0, (size_t)R * d->predictor.stride * 4, st));
  const MatView X = mk.in ? MatView{w.xin, (int64_t)B * din, 1, din} : MatView{a->batch.rows, a->batch.replica_stride, 1, a->batch.row};
  IL_TRY(mlp_backward_dropout(h, &d->predictor, R, B, X, mk, w.pacts, MatView{w.dpred, (int64_t)B * din, 1, din}, w.grads, d->predictor.stride, w.tmpA, w.tmpB, st));
  il_adam opt = a->opt;
  opt.replica_floats = d->predictor.stride;
  return launch_adam(h, d->predictor.params, w.grads, &opt, (int64_t)R * d->predictor.stride, st);
}

extern "C" int il_red_sigma(il_handle* h, const il_red* d, int R, const il_batch* batch, const float* mask_in, const float* const* mask_hid, void* workspace, int64_t workspace_bytes,
                            void* stream) {
  IL_CHECK(h && d && d->sigma && workspace, "il_red_sigma: null argument");
  cudaStream_t st = (cudaStream_t)stream;
  IL_TRY(red_validate(d, batch, "il_red_sigma"));
  const int B = batch->B, din = d->predictor.dims[0];
  IL_CHECK(workspace_bytes >= il_red_workspace_bytes(d, R, B), "il_red_sigma: workspace too small");
  RedWs w = red_layout(d, R, B, static_cast<char*>(workspace), true);
  IL_TRY(red_forward(h, d, R, batch, masks_of(mask_in, mask_hid), w, st));
  IL_LAUNCH(h, red_pairwise_kernel, dblocks((int64_t)R * B * B), 256, 0, st, w.pred, w.targ, w.dist, R, B, din);
  IL_LAUNCH(h, red_median_kernel, R, 256, 0, st, w.dist, (int64_t)B * B, d->sigma);
  return 0;
}

extern "C" int il_red_reward(il_handle* h, const il_red* d, int R, const il_batch* batch, float* reward, int64_t reward_rs, int reward_ld, void* workspace, int64_t workspace_bytes,
                             void* stream) {
  IL_CHECK(h && d && d->sigma && reward && workspace, "il_red_reward: null argument");
  cudaStream_t st = (cudaStream_t)stream;
  IL_TRY(red_validate(d, batch, "il_red_reward"));
  const int B = batch->B, din = d->predictor.dims[0];
  IL_CHECK(workspace_bytes >= il_red_workspace_bytes(d, R, B), "il_red_reward: workspace too small");
  RedWs w = red_layout(d, R, B, static_cast<char*>(workspace), true);
  DropMasks none{};  // eval mode (train.py:147): no dropout
  IL_TRY(red_forward(h, d, R, batch, none, w, st));
  IL_LAUNCH(h, red_reward_kernel, dblocks((int64_t)R * B), 256, 0, st, w.pred, w.targ, d->sigma, reward, reward_rs, reward_ld, R, B, din);
  return 0;
}

// ---- dropout SoftActor (DRIL) ------------------------------------------------------------------------------------------------------
namespace {
struct ActWs {
  float *xin, *given, *head, *dhead, *row_loss, *tmpA, *tmpB, *grads;
  MlpActs acts;
  int64_t bytes;
};
ActWs actor_layout(const il_mlp* m, int R, int n, char* base, bool with_grad) {
  ActWs w{};
  Carve c{base, 0};
  const int S = m->dims[0], out = m->dims[m->n_layers], hm = hidden_max(m);
  w.xin = c.take((int64_t)R * n * S);
  w.given = c.take((int64_t)R * n * (out / 2));
  acts_carve(c, m, R, n, &w.acts);
  w.head = c.take((int64_t)R * n * out);
  if (with_grad) {
    w.dhead = c.take((int64_t)R * n * out); w.row_loss = c.take((int64_t)R * n);
    w.tmpA = c.take((int64_t)R * n * hm); w.tmpB = c.take((int64_t)R * n * hm);
    w.grads = c.take((int64_t)R * m->stride);
  }
  w.bytes = c.used;
  return w;
}
}  // namespace

extern "C" int64_t il_actor_dropout_workspace_bytes(const il_mlp* actor, int R, int n) { return actor ? actor_layout(actor, R, n, nullptr, true).bytes : -1; }

// log pi(given_action | state) of R dropout policies on n rows each; rows of `states` / `given_action` are repeated `repeat` times (n = repeat * source rows).
extern "C" int il_actor_log_prob_dropout(il_handle* h, const il_mlp* actor, int R, int n, int repeat, const float* states, int64_t states_rs, int ld_states, const float* given_action,
                                         const float* mask_in, const float* const* mask_hid, float* log_prob, void* workspace, int64_t workspace_bytes, void* stream) {
  IL_CHECK(h && states && given_action && log_prob && workspace && R > 0 && n > 0 && repeat >= 1 && n % repeat == 0, "il_actor_log_prob_dropout: bad argument");
  IL_TRY(mlp_validate(actor, "il_actor_log_prob_dropout"));
  IL_CHECK(workspace_bytes >= il_actor_dropout_workspace_bytes(actor, R, n), "il_actor_log_prob_dropout: workspace too small");
  cudaStream_t st = (cudaStream_t)stream;
  const int S = actor->dims[0], out = actor->dims[actor->n_layers], A = out / 2;
  ActWs w = actor_layout(actor, R, n, static_cast<char*>(workspace), true);
  const DropMasks mk = masks_of(mask_in, mask_hid);
  IL_LAUNCH(h, input_mask_kernel, dblocks((int64_t)R * n * S), 256, 0, st, states, states_rs, ld_states, repeat, mask_in, w.xin, R, n, S);
  IL_LAUNCH(h, input_mask_kernel, dblocks((int64_t)R * n * A), 256, 0, st, given_action, (int64_t)(n / repeat) * A, A, repeat, nullptr, w.given, R, n, A);
  IL_TRY(mlp_forward_dropout(h, actor, R, n, MatView{w.xin, (int64_t)n * S, 1, S}, mk, w.acts, w.head, (int64_t)n * out, out, st));
  HeadFwdArgs ha{};
  ha.head = w.head; ha.given = w.given; ha.log_prob = log_prob; ha.R = R; ha.n = n; ha.A = A;
  return launch_actor_head(h, ha, st);
}

extern "C" int il_dril_reward(il_handle* h, const float* log_prob, int R, int B, int ensemble, const float* q, int q_shared, float* reward, int64_t reward_rs, int reward_ld,
                              float* variance, void* stream) {
  IL_CHECK(h && log_prob && R > 0 && B > 0 && ensemble >= 2 && (reward == nullptr || q != nullptr), "il_dril_reward: bad argument");
  IL_LAUNCH(h, dril_reward_kernel, dblocks((int64_t)R * B), 256, 0, (cudaStream_t)stream, log_prob, R, B, ensemble, q, q_shared, reward, reward_rs, reward_ld, variance);
  return 0;
}

// behavioural_cloning_update of a dropout policy (train.py:120: DRIL's ensemble pretraining): il_bc_update with explicit masks
int bc_head_backward_launch(il_handle* h, const float* head, const il_batch* batch, float* dhead, float* row_loss, int R, cudaStream_t st);
int bc_row_mean_launch(il_handle* h, const float* row_loss, float* out_loss, int R, int B, cudaStream_t st);

extern "C" int il_bc_update_dropout(il_handle* h, const il_bc_args* a, const float* mask_in, const float* const* mask_hid, void* stream) {
  IL_CHECK(h && a, "il_bc_update_dropout: null argument");
  cudaStream_t st = (cudaStream_t)stream;
  const int R = a->R, B = a->batch.B, S = a->batch.S, A = a->batch.A;
  IL_TRY(mlp_validate(&a->actor, "il_bc_update_dropout"));
  IL_CHECK(R > 0 && B > 0 && a->actor.dims[0] == S && a->actor.dims[a->actor.n_layers] == 2 * A, "il_bc_update_dropout: actor dims do not match the batch");
  IL_CHECK(a->batch.rows && a->batch.row == row_layout(S, A).len && a->workspace && a->workspace_bytes >= il_actor_dropout_workspace_bytes(&a->actor, R, B), "il_bc_update_dropout: bad batch / workspace");
  ActWs w = actor_layout(&a->actor, R, B, static_cast<char*>(a->workspace), true);
  const DropMasks mk = masks_of(mask_in, mask_hid);
  const int out = 2 * A;
  IL_TRY(launch_tick(h, a->opt.step, nullptr, nullptr, st));
  MatView X{a->batch.rows, a->batch.replica_stride, 1, a->batch.row};
  if (mask_in) {
    IL_LAUNCH(h, input_mask_kernel, dblocks((int64_t)R * B * S), 256, 0, st, a->batch.rows, a->batch.replica_stride, a->batch.row, 1, mask_in, w.xin, R, B, S);
    X = MatView{w.xin, (int64_t)B * S, 1, S};
  }
  IL_TRY(mlp_forward_dropout(h, &a->actor, R, B, X, mk, w.acts, w.head, (int64_t)B * out, out, st));
  IL_TRY(bc_head_backward_launch(h, w.head, &a->batch, w.dhead, a->out_loss ? w.row_loss : nullptr, R, st));
  if (a->out_loss) IL_TRY(bc_row_mean_launch(h, w.row_loss, a->out_loss, R, B, st));
  IL_CUDA(cudaMemsetAsync(w.grads, 0, (size_t)R * a->actor.stride * 4, st));
  IL_TRY(mlp_backward_dropout(h, &a->actor, R, B, X, mk, w.acts, MatView{w.dhead, (int64_t)B * out, 1, out}, w.grads, a->actor.stride, w.tmpA, w.tmpB, st));
  il_adam opt = a->opt;
  opt.replica_floats = a->actor.stride;
  return launch_adam(h, a->actor.params, w.grads, &opt, (int64_t)R * a->actor.stride, st);
}
