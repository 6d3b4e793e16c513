// sac_update (training.py:14-54) for R independent replicas as one stream-ordered program of grouped GEMMs
// and small fused elementwise kernels. Order of operations follows SURVEY.md §3.2 exactly: target from the
// OLD critic/actor, critic AdamW step, actor loss through the UPDATED critic, temperature loss with the alpha
// captured at entry, polyak last.
#include "mlp.cuh"

namespace {

struct AbsView {  // absorbing[r, b] = ptr[r * rs + b * ld] (nullptr -> 0)
  const float* ptr;
  int64_t rs;
  int ld;
};
__device__ __forceinline__ float abs_at(const AbsView& v, int r, int b) { return v.ptr ? __ldg(v.ptr + (int64_t)r * v.rs + (int64_t)b * v.ld) : 0.f; }

// training.py:24-25: y = r + (1 - terminal) * discount * (min(Q1', Q2') - (1 - absorbing) * alpha * log_pi')
__global__ void sac_target_kernel(const float* __restrict__ qt, const float* __restrict__ lp_next, const float* __restrict__ log_alpha, const float* __restrict__ rows,
                                  int64_t rs, int row, int off_reward, int off_terminal, AbsView av, float discount, const float* __restrict__ discount_r,
                                  float* __restrict__ y, int R, int B) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)R * B) return;
  const int r = (int)(i / B), b = (int)(i % B);
  if (discount_r) discount = discount_r[r];
  const float alpha = expf(__ldg(log_alpha + r));
  const float* tr = rows + (int64_t)r * rs + (int64_t)b * row;
  const float q = fminf(qt[((int64_t)2 * r) * B + b], qt[((int64_t)2 * r + 1) * B + b]);
  const float ent = __fmul_rn(__fmul_rn(__fsub_rn(1.f, abs_at(av, r, b)), alpha), lp_next[i]);
  const float tv = __fsub_rn(q, ent);
  y[i] = __fadd_rn(tr[off_reward], __fmul_rn(__fmul_rn(__fsub_rn(1.f, tr[off_terminal]), discount), tv));
}

// training.py:26-27 + backward of value_loss w.r.t. Q1, Q2. One block per replica.
__global__ void sac_critic_lossgrad_kernel(const float* __restrict__ q, const float* __restrict__ y, const float* __restrict__ rows, int64_t rs, int row, int off_weight,
                                           float* __restrict__ dq, float* __restrict__ out_q, float* __restrict__ out_losses, int B) {
  __shared__ float red[32];
  const int r = blockIdx.x;
  const float invB = 1.f / (float)B;
  float l1 = 0.f, l2 = 0.f;
  for (int b = threadIdx.x; b < B; b += blockDim.x) {
    const float w = rows[(int64_t)r * rs + (int64_t)b * row + off_weight];
    const float yy = y[(int64_t)r * B + b];
    const float q1 = q[((int64_t)2 * r) * B + b], q2 = q[((int64_t)2 * r + 1) * B + b];
    const float d1 = __fsub_rn(q1, yy), d2 = __fsub_rn(q2, yy);
    l1 += w * d1 * d1;
    l2 += w * d2 * d2;
    const float c = __fmul_rn(invB, w);
    dq[((int64_t)2 * r) * B + b] = __fmul_rn(c, __fmul_rn(2.f, d1));
    dq[((int64_t)2 * r + 1) * B + b] = __fmul_rn(c, __fmul_rn(2.f, d2));
    if (out_q) out_q[(int64_t)r * B + b] = fminf(q1, q2);
  }
  l1 = block_sum(l1, red);
  l2 = block_sum(l2, red);
  if (threadIdx.x == 0 && out_losses) out_losses[r * 3 + 0] = l1 * invB + l2 * invB;
}

// training.py:37-38: policy_loss = mean(w (1 - abs) alpha log_pi - min(Q1, Q2)); gradient w.r.t. Q1, Q2. One block per replica.
__global__ void sac_actor_loss_kernel(const float* __restrict__ q, const float* __restrict__ lp_new, const float* __restrict__ log_alpha, const float* __restrict__ rows,
                                      int64_t rs, int row, int off_weight, AbsView av, float* __restrict__ dq, float* __restrict__ out_losses, int B) {
  __shared__ float red[32];
  const int r = blockIdx.x;
  const float invB = 1.f / (float)B;
  const float alpha = expf(__ldg(log_alpha + r));
  float loss = 0.f;
  for (int b = threadIdx.x; b < B; b += blockDim.x) {
    const float w = rows[(int64_t)r * rs + (int64_t)b * row + off_weight];
    const float q1 = q[((int64_t)2 * r) * B + b], q2 = q[((int64_t)2 * r + 1) * B + b];
    const float g1 = q1 < q2 ? 1.f : (q1 == q2 ? 0.5f : 0.f);  // torch.minimum backward: ties split evenly
    dq[((int64_t)2 * r) * B + b] = -invB * g1;
    dq[((int64_t)2 * r + 1) * B + b] = -invB * (1.f - g1);
    loss += w * (1.f - abs_at(av, r, b)) * alpha * lp_new[(int64_t)r * B + b] - fminf(q1, q2);
  }
  loss = block_sum(loss, red);
  if (threadIdx.x == 0 && out_losses) out_losses[r * 3 + 1] = loss * invB;
}

// Backward of the tanh-Gaussian head w.r.t. the raw actor output (mean | log-std), rsample path (training.py:34-38).
//  dL/dx_j   = dL/da_j (1 - a_j^2) + c * 2 a_j          (c = w (1 - abs) alpha / B; d log_pi / d x_j = 2 tanh x_j)
//  dL/dmu_j  = dL/dx_j ;  dL/dlogstd_j = [dL/dx_j * std_j eps_j - c] * 1[-20 <= raw <= 2]
__global__ void sac_head_backward_kernel(const float* __restrict__ head, const float* __restrict__ eps, const float* __restrict__ xnew, int d, int S,
                                         const float* __restrict__ dxa, const float* __restrict__ log_alpha, const float* __restrict__ rows, int64_t rs, int row,
                                         int off_weight, AbsView av, float* __restrict__ dhead, int R, int B, int A) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)R * B) return;
  const int r = (int)(i / B), b = (int)(i % B);
  const float alpha = expf(__ldg(log_alpha + r));
  const float w = rows[(int64_t)r * rs + (int64_t)b * row + off_weight];
  const float c = w * (1.f - abs_at(av, r, b)) * alpha / (float)B;
  const float* hd = head + i * 2 * A;
  const float* a_row = xnew + i * d + S;
  const float* g1 = dxa + (((int64_t)2 * r) * B + b) * A;
  const float* g2 = dxa + (((int64_t)2 * r + 1) * B + b) * A;
  for (int j = 0; j < A; ++j) {
    const float raw = hd[A + j];
    const bool in_range = raw >= -20.f && raw <= 2.f;
    const float sd = expf(fminf(fmaxf(raw, -20.f), 2.f));
    const float a = a_row[j];
    const float dx = (g1[j] + g2[j]) * (1.f - a * a) + c * 2.f * a;
    dhead[i * 2 * A + j] = dx;
    dhead[i * 2 * A + A + j] = in_range ? dx * (sd * eps[i * A + j]) - c : 0.f;
  }
}

// training.py:45-49: temperature loss with the entry alpha, gradient w.r.t. log_alpha, Adam step (train.py:66). One block per replica.
__global__ void sac_alpha_kernel(float* __restrict__ log_alpha, const float* __restrict__ lp_new, const float* __restrict__ rows, int64_t rs, int row, int off_weight,
                                 AbsView av, float entropy_target, const float* __restrict__ entropy_target_r, float* __restrict__ m, float* __restrict__ v,
                                 const int64_t* __restrict__ step, double lr, double beta1, double beta2, double eps, double wd, const double* __restrict__ lr_r,
                                 const double* __restrict__ wd_r, float* __restrict__ out_losses, int B) {
  __shared__ float red[32];
  const int r = blockIdx.x;
  if (entropy_target_r) entropy_target = entropy_target_r[r];
  if (lr_r) lr = lr_r[r];
  if (wd_r) wd = wd_r[r];
  float s = 0.f;
  for (int b = threadIdx.x; b < B; b += blockDim.x) {
    const float w = rows[(int64_t)r * rs + (int64_t)b * row + off_weight];
    s += w * (1.f - abs_at(av, r, b)) * (lp_new[(int64_t)r * B + b] + entropy_target);
  }
  s = block_sum(s, red);
  if (threadIdx.x == 0) {
    float p = log_alpha[r];
    const float alpha = expf(p);
    const float g = -alpha * s / (float)B;  // d/dlog_alpha of -mean(w (1-abs) alpha (log_pi + H)) ; equals the loss value
    if (out_losses) out_losses[r * 3 + 2] = g;
    const double t = (double)*step;
    const float step_size = (float)(lr / (1.0 - pow(beta1, t))), bc2_sqrt = (float)sqrt(1.0 - pow(beta2, t));
    float mi = m[r], vi = v[r];
    if (wd != 0.0) p = __fmul_rn(p, (float)(1.0 - lr * wd));
    mi = __fadd_rn(mi, __fmul_rn((float)(1.0 - beta1), __fsub_rn(g, mi)));
    vi = __fadd_rn(__fmul_rn(vi, (float)beta2), __fmul_rn(__fmul_rn((float)(1.0 - beta2), g), g));
    const float denom = __fadd_rn(__fdiv_rn(sqrtf(vi), bc2_sqrt), (float)eps);
    p = __fadd_rn(p, __fmul_rn(-step_size, __fdiv_rn(mi, denom)));
    log_alpha[r] = p; m[r] = mi; v[r] = vi;
  }
}

// behavioural cloning (training.py:57-64): d(-w log pi(a|s) / B) / d(mean, log-std) for a given (clamped) expert action.
__global__ void bc_head_backward_kernel(const float* __restrict__ head, const float* __restrict__ rows, int64_t rs, int row, int off_action, int off_weight,
                                        float* __restrict__ dhead, float* __restrict__ row_loss, int R, int B, int A) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)R * B) return;
  const int r = (int)(i / B), b = (int)(i % B);
  const float* tr = rows + (int64_t)r * rs + (int64_t)b * row;
  const float w = tr[off_weight], c = -w / (float)B;
  const float A_LO = (float)(-1.0 + 1e-6), A_HI = (float)(1.0 - 1e-6), LOG_SQRT_2PI = 0.91893853320467274178f, LOG2 = 0.69314718055994530942f;
  const float* hd = head + i * 2 * A;
  float lp = 0.f, ladj = 0.f;
  for (int j = 0; j < A; ++j) {
    const float raw = hd[A + j];
    const bool in_range = raw >= -20.f && raw <= 2.f;
    const float ls = fminf(fmaxf(raw, -20.f), 2.f), sd = expf(ls), var = sd * sd;
    const float x = atanhf(fminf(fmaxf(tr[off_action + j], A_LO), A_HI));  // training.py:59, models.py:98
    const float diff = x - hd[j];
    lp += -(diff * diff) / (2.f * var) - logf(sd) - LOG_SQRT_2PI;
    ladj += 2.f * (LOG2 - x - softplusf(-2.f * x));
    dhead[i * 2 * A + j] = c * diff / var;
    dhead[i * 2 * A + A + j] = in_range ? c * (diff * diff / var - 1.f) : 0.f;
  }
  if (row_loss) row_loss[i] = -w * ((0.f - ladj) + lp);
}

__global__ void row_mean_kernel(const float* __restrict__ x, float* __restrict__ out, int B) {
  __shared__ float red[32];
  float s = 0.f;
  for (int b = threadIdx.x; b < B; b += blockDim.x) s += x[(int64_t)blockIdx.x * B + b];
  s = block_sum(s, red);
  if (threadIdx.x == 0) out[blockIdx.x] = s / (float)B;
}

struct SacWs {
  MlpActs actor_acts, critic_acts;
  float *head, *q, *xn, *y, *lp_next, *dq, *dxa, *dhead, *tmpA, *tmpB, *g_actor, *g_critic;
  int64_t bytes;
};

int64_t carve(char*& p, int64_t floats) {
  const int64_t b = il_align_up(floats * 4, 256);
  p += b;
  return b;
}

SacWs sac_layout(const il_sac_args* a, char* base) {
  SacWs w{};
  const int R = a->R, B = a->batch.B, A = a->batch.A, d = a->batch.S + a->batch.A;
  char* p = base;
  p = mlp_acts_carve(&a->actor, R, B, p, &w.actor_acts);
  p = mlp_acts_carve(&a->critic, 2 * R, B, p, &w.critic_acts);
  auto take = [&](int64_t floats) { float* r = reinterpret_cast<float*>(p); carve(p, floats); return r; };
  w.head = take((int64_t)R * B * 2 * A);
  w.q = take((int64_t)2 * R * B);
  w.xn = take((int64_t)R * B * d);
  w.y = take((int64_t)R * B);
  w.lp_next = take((int64_t)R * B);
  w.dq = take((int64_t)2 * R * B);
  w.dxa = take((int64_t)2 * R * B * A);
  w.dhead = take((int64_t)R * B * 2 * A);
  int hmax = mlp_max_hidden(&a->critic);
  if (mlp_max_hidden(&a->actor) > hmax) hmax = mlp_max_hidden(&a->actor);
  w.tmpA = take((int64_t)2 * R * B * hmax);
  w.tmpB = take((int64_t)2 * R * B * hmax);
  w.g_actor = take((int64_t)R * a->actor.stride);
  w.g_critic = take((int64_t)2 * R * a->critic.stride);
  w.bytes = p - base;
  return w;
}

}  // namespace

extern "C" int64_t il_sac_workspace_bytes(const il_sac_args* a) {
  if (!a) return -1;
  return sac_layout(a, nullptr).bytes;
}

extern "C" int il_sac_update(il_handle* h, const il_sac_args* a, void* stream) {
  IL_CHECK(h && a, "il_sac_update: null argument");
  cudaStream_t st = (cudaStream_t)stream;
  const int R = a->R, B = a->batch.B, S = a->batch.S, A = a->batch.A, d = S + A;
  IL_CHECK(R > 0 && B > 0 && S > 0 && A > 0, "il_sac_update: R=%d B=%d S=%d A=%d", R, B, S, A);
  IL_TRY(mlp_validate(&a->actor, "il_sac_update(actor)"));
  IL_TRY(mlp_validate(&a->critic, "il_sac_update(critic)"));
  IL_TRY(mlp_validate(&a->target, "il_sac_update(target)"));
  IL_CHECK(a->actor.dims[0] == S && a->actor.dims[a->actor.n_layers] == 2 * A, "il_sac_update: actor dims do not match S=%d A=%d", S, A);
  IL_CHECK(a->critic.dims[0] == d && a->critic.dims[a->critic.n_layers] == 1, "il_sac_update: critic dims do not match S+A=%d", d);
  IL_CHECK(a->target.n_layers == a->critic.n_layers && a->target.stride == a->critic.stride, "il_sac_update: target/critic layout mismatch");
  const RowLayout L = row_layout(S, A);
  IL_CHECK(a->batch.row == L.len, "il_sac_update: batch row length %d != %d", a->batch.row, L.len);
  IL_CHECK(a->batch.rows && a->log_alpha && a->eps_next && a->eps_new && a->workspace, "il_sac_update: null buffer");
  IL_CHECK(a->workspace_bytes >= il_sac_workspace_bytes(a), "il_sac_update: workspace too small (%lld < %lld)", (long long)a->workspace_bytes,
           (long long)il_sac_workspace_bytes(a));
  SacWs w = sac_layout(a, static_cast<char*>(a->workspace));
  const float* rows = a->batch.rows;
  const int64_t rs = a->batch.replica_stride;
  const int row = L.len;
  AbsView av{nullptr, 0, 0};
  if (a->absorbing) av = AbsView{a->absorbing, (int64_t)B, 1};
  else if (a->absorbing_from_state) av = AbsView{rows + L.state + (S - 1), rs, row};
  const unsigned ew = (unsigned)(((int64_t)R * B + 127) / 128);

  IL_TRY(launch_tick(h, a->actor_opt.step, a->critic_opt.step, a->alpha_opt.step, st));

  // (1) a' ~ pi(.|s'), log pi(a'|s')  [training.py:20-23]
  IL_TRY(mlp_forward(h, &a->actor, R, B, MatView{rows + L.next_state, rs, 1, row}, w.actor_acts, w.head, (int64_t)B * 2 * A, 2 * A, st, /*keep_hidden=*/false));
  {
    HeadFwdArgs ha{};
    ha.head = w.head; ha.eps = a->eps_next;
    ha.action = w.xn + S; ha.action_rs = (int64_t)B * d; ha.ld_action = d;
    ha.zero_mask = av.ptr; ha.zero_mask_rs = av.rs; ha.zero_mask_ld = av.ld;
    ha.log_prob = w.lp_next;
    ha.copy_src = rows + L.next_state; ha.copy_rs = rs; ha.copy_ld = row; ha.copy_cols = S;
    ha.R = R; ha.n = B; ha.A = A;
    IL_TRY(launch_actor_head(h, ha, st));
  }
  // (2) target critics on (s', a') and the Bellman target  [training.py:24-25]
  IL_TRY(mlp_forward(h, &a->target, 2 * R, B, MatView{w.xn, (int64_t)B * d, 2, d}, w.critic_acts, w.q, (int64_t)B, 1, st, /*keep_hidden=*/false));
  IL_LAUNCH(h, sac_target_kernel, ew, 128, 0, st, w.q, w.lp_next, a->log_alpha, rows, rs, row, L.reward, L.terminal, av, a->discount, a->discount_r, w.y, R, B);
  // (3) critic loss, backward, AdamW  [training.py:26-31]
  IL_TRY(mlp_forward(h, &a->critic, 2 * R, B, MatView{rows + L.state, rs, 2, row}, w.critic_acts, w.q, (int64_t)B, 1, st));
  IL_LAUNCH(h, sac_critic_lossgrad_kernel, R, 256, 0, st, w.q, w.y, rows, rs, row, L.weight, w.dq, a->out_q_values, a->out_losses, B);
  IL_TRY(mlp_backward(h, &a->critic, 2 * R, B, MatView{rows + L.state, rs, 2, row}, w.critic_acts, MatView{w.dq, (int64_t)B, 1, 1}, w.g_critic, a->critic.stride, nullptr, 0,
                      0, 0, 0, w.tmpA, w.tmpB, st));
  // polyak (training.py:52) is fused into the critic AdamW pass: the critic parameters do not change again inside this
  // update and the target is not read again, so the result equals the reference's end-of-update target step
  il_adam critic_opt = a->critic_opt, actor_opt = a->actor_opt;  // per-replica hyperparameters: replica r owns its twin (2 nets) / its actor
  critic_opt.replica_floats = 2 * a->critic.stride;
  actor_opt.replica_floats = a->actor.stride;
  IL_TRY(launch_adam(h, a->critic.params, w.g_critic, &critic_opt, (int64_t)2 * R * a->critic.stride, st, a->target.params, a->polyak_factor, a->polyak_r));
  // (4) actor loss through the UPDATED critic  [training.py:34-42]
  IL_TRY(mlp_forward(h, &a->actor, R, B, MatView{rows + L.state, rs, 1, row}, w.actor_acts, w.head, (int64_t)B * 2 * A, 2 * A, st));
  {
    HeadFwdArgs ha{};
    ha.head = w.head; ha.eps = a->eps_new;
    ha.action = w.xn + S; ha.action_rs = (int64_t)B * d; ha.ld_action = d;
    ha.log_prob = a->out_log_probs ? a->out_log_probs : w.lp_next;
    ha.copy_src = rows + L.state; ha.copy_rs = rs; ha.copy_ld = row; ha.copy_cols = S;
    ha.R = R; ha.n = B; ha.A = A;
    IL_TRY(launch_actor_head(h, ha, st));
  }
  const float* lp_new = a->out_log_probs ? a->out_log_probs : w.lp_next;
  // only the action gradient of Q(s, pi(s)) is needed (no critic parameter gradients): the hidden layers are kept as ReLU sign bits where the kernels allow
  IL_TRY(mlp_forward(h, &a->critic, 2 * R, B, MatView{w.xn, (int64_t)B * d, 2, d}, w.critic_acts, w.q, (int64_t)B, 1, st, MLP_KEEP_MASKS));
  IL_LAUNCH(h, sac_actor_loss_kernel, R, 256, 0, st, w.q, lp_new, a->log_alpha, rows, rs, row, L.weight, av, w.dq, a->out_losses, B);
  IL_TRY(mlp_backward(h, &a->critic, 2 * R, B, MatView{w.xn, (int64_t)B * d, 2, d}, w.critic_acts, MatView{w.dq, (int64_t)B, 1, 1}, nullptr, 0, w.dxa, (int64_t)B * A, A, S,
                      A, w.tmpA, w.tmpB, st));
  IL_LAUNCH(h, sac_head_backward_kernel, ew, 128, 0, st, w.head, a->eps_new, w.xn, d, S, w.dxa, a->log_alpha, rows, rs, row, L.weight, av, w.dhead, R, B, A);
  IL_TRY(mlp_backward(h, &a->actor, R, B, MatView{rows + L.state, rs, 1, row}, w.actor_acts, MatView{w.dhead, (int64_t)B * 2 * A, 1, 2 * A}, w.g_actor, a->actor.stride,
                      nullptr, 0, 0, 0, 0, w.tmpA, w.tmpB, st));
  IL_TRY(launch_adam(h, a->actor.params, w.g_actor, &actor_opt, (int64_t)R * a->actor.stride, st));
  // (5) temperature  [training.py:45-49]
  IL_LAUNCH(h, sac_alpha_kernel, R, 256, 0, st, a->log_alpha, lp_new, rows, rs, row, L.weight, av, a->entropy_target, a->entropy_target_r, a->alpha_opt.m, a->alpha_opt.v,
            a->alpha_opt.step, a->alpha_opt.lr, a->alpha_opt.beta1, a->alpha_opt.beta2, a->alpha_opt.eps, a->alpha_opt.weight_decay, a->alpha_opt.lr_r, a->alpha_opt.weight_decay_r,
            a->out_losses, B);
  return 0;  // (6) polyak [training.py:52]: done inside the critic AdamW kernel above
}

// ---- behavioural_cloning_update (training.py:57-64) --------------------------------------------------------------------
namespace {
struct BcWs {
  MlpActs acts;
  float *head, *dhead, *row_loss, *tmpA, *tmpB, *grads;
  int64_t bytes;
};
BcWs bc_layout(const il_bc_args* a, char* base) {
  BcWs w{};
  const int R = a->R, B = a->batch.B, A = a->batch.A;
  char* p = mlp_acts_carve(&a->actor, R, B, base, &w.acts);
  auto take = [&](int64_t floats) { float* r = reinterpret_cast<float*>(p); carve(p, floats); return r; };
  w.head = take((int64_t)R * B * 2 * A);
  w.dhead = take((int64_t)R * B * 2 * A);
  w.row_loss = take((int64_t)R * B);
  const int hmax = mlp_max_hidden(&a->actor);
  w.tmpA = take((int64_t)R * B * hmax);
  w.tmpB = take((int64_t)R * B * hmax);
  w.grads = take((int64_t)R * a->actor.stride);
  w.bytes = p - base;
  return w;
}
}  // namespace

// launchers shared with the dropout-policy variant (dropout_nets.cu)
int bc_head_backward_launch(il_handle* h, const float* head, const il_batch* batch, float* dhead, float* row_loss, int R, cudaStream_t st) {
  const RowLayout L = row_layout(batch->S, batch->A);
  IL_LAUNCH(h, bc_head_backward_kernel, (unsigned)(((int64_t)R * batch->B + 127) / 128), 128, 0, st, head, batch->rows, batch->replica_stride, L.len, L.action, L.weight, dhead, row_loss, R,
            batch->B, batch->A);
  return 0;
}
int bc_row_mean_launch(il_handle* h, const float* row_loss, float* out_loss, int R, int B, cudaStream_t st) {
  IL_LAUNCH(h, row_mean_kernel, R, 256, 0, st, row_loss, out_loss, B);
  return 0;
}

extern "C" int64_t il_bc_workspace_bytes(const il_bc_args* a) { return a ? bc_layout(a, nullptr).bytes : -1; }

extern "C" int il_bc_update(il_handle* h, const il_bc_args* a, void* stream) {
  IL_CHECK(h && a, "il_bc_update: null argument");
  cudaStream_t st = (cudaStream_t)stream;
  const int R = a->R, B = a->batch.B, S = a->batch.S, A = a->batch.A;
  IL_TRY(mlp_validate(&a->actor, "il_bc_update(actor)"));
  IL_CHECK(R > 0 && B > 0 && a->actor.dims[0] == S && a->actor.dims[a->actor.n_layers] == 2 * A, "il_bc_update: actor dims do not match the batch");
  const RowLayout L = row_layout(S, A);
  IL_CHECK(a->batch.rows && a->batch.row == L.len && a->workspace && a->workspace_bytes >= il_bc_workspace_bytes(a), "il_bc_update: bad batch / workspace");
  BcWs w = bc_layout(a, static_cast<char*>(a->workspace));
  const MatView X{a->batch.rows + L.state, a->batch.replica_stride, 1, L.len};
  IL_TRY(launch_tick(h, a->opt.step, nullptr, nullptr, st));
  IL_TRY(mlp_forward(h, &a->actor, R, B, X, w.acts, w.head, (int64_t)B * 2 * A, 2 * A, st));
  IL_LAUNCH(h, bc_head_backward_kernel, (unsigned)(((int64_t)R * B + 127) / 128), 128, 0, st, w.head, a->batch.rows, a->batch.replica_stride, L.len, L.action, L.weight, w.dhead,
            a->out_loss ? w.row_loss : nullptr, R, B, A);
  if (a->out_loss) IL_LAUNCH(h, row_mean_kernel, R, 256, 0, st, w.row_loss, a->out_loss, B);
  IL_TRY(mlp_backward(h, &a->actor, R, B, X, w.acts, MatView{w.dhead, (int64_t)B * 2 * A, 1, 2 * A}, w.grads, a->actor.stride, nullptr, 0, 0, 0, 0, w.tmpA, w.tmpB, st));
  il_adam opt = a->opt;
  opt.replica_floats = a->actor.stride;
  return launch_adam(h, a->actor.params, w.grads, &opt, (int64_t)R * a->actor.stride, st);
}
