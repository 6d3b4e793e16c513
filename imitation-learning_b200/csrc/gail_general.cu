// General GAILDiscriminator (models.py:152-180) and adversarial_imitation_update (training.py:85-134) for the configurations the
// fused one-CTA-per-replica kernel (gail.cu) does not cover: reward shaping (linear g + MLP h, f = g(s,a) + (1-t)(gamma h(s') - h(s))),
// subtract_log_policy, depth > 1, tanh / sigmoid activations. Written as a stream-ordered PROGRAM over the replica-batched primitives
// (grouped GEMMs + MLP forward / backward of mlp.cu) plus small element-wise kernels:
//   * every evaluation of a net is one spectral-norm ACCESS (torch parametrization semantics: a train-mode access runs one power
//     iteration in place, then W_eff = W / (u^T W v) with u, v constants) — g is accessed once per discriminator forward, h twice
//     (h(s') then h(s), models.py:174), each with its own (u, v, sigma);
//   * the gradient penalty (training.py:117-127) is the explicit double backward of |d f / d(s, a)|^2 through the MLPs:
//       delta_{L-1} = kappa W_L * s'(y_{L-1}),  delta_l = (delta_{l+1} W_{l+1}) * s'(y_l),  g_x = delta_1 W_1        (input gradient)
//       then, with gbar = dP/dg_x:  dW_1 += delta_1^T gbar,  dbar_1 = gbar W_1^T,  ubar_l = dbar_l * s'(y_l),
//       dW_{l+1} += delta_{l+1}^T ubar_l,  dbar_{l+1} = ubar_l W_{l+1}^T,  and through s'(z_l):  zbar_l = dbar_l * u_l * s''(y_l)
//       back-propagated like an ordinary loss gradient (zero for relu);
//   * gradients w.r.t. W_eff are projected through each access: dW = (G - <G, W_eff> u v^T) / sigma (SURVEY §8a a12).
#include "mlp.cuh"

namespace {

// IL_DEBUG_SYNC=1: synchronise after every stage of the program and name the stage that failed (diagnostics only; not capturable)
#define GX_STAGE(h, st, ...)                                                                          \
  do {                                                                                                \
    if ((h)->debug_sync) {                                                                            \
      cudaError_t _e = cudaStreamSynchronize(st);                                                     \
      if (_e != cudaSuccess) {                                                                        \
        char _where[160];                                                                             \
        snprintf(_where, sizeof(_where), __VA_ARGS__);                                                \
        IL_FAIL("gailx stage '%s' failed: %s", _where, cudaGetErrorString(_e));                       \
      }                                                                                               \
    }                                                                                                 \
  } while (0)

constexpr int GX_MAX_EVALS = 9;

__device__ __forceinline__ float act_grad2_from_output(float y, int act) {  // second derivative of the activation through its output
  if (act == IL_ACT_RELU) return 0.f;
  if (act == IL_ACT_TANH) return -2.f * y * (1.f - y * y);
  return y * (1.f - y) * (1.f - 2.f * y);
}

struct SnLayout {  // offsets of the per-layer u / v vectors inside the concatenated buffers
  int uo[IL_MAX_LAYERS], vo[IL_MAX_LAYERS], u_total, v_total;
};
__host__ __device__ inline SnLayout sn_layout(const int32_t* dims, int L) {
  SnLayout s;
  int u = 0, v = 0;
  for (int l = 0; l < L; ++l) { s.uo[l] = u; s.vo[l] = v; u += dims[l + 1]; v += dims[l]; }
  s.u_total = u; s.v_total = v;
  return s;
}

// One spectral-norm access of every layer of R nets. One CTA per replica. eff receives W / sigma (or W without spectral norm)
// and the biases; snap receives per layer [u | v | sigma] of THIS access (layout: u_total + v_total + L floats).
struct SnAccessParams {
  il_mlp net, eff;
  float *u, *v;      // persistent buffers (nullptr: no spectral norm)
  int u_stride, v_stride;
  float* snap;
  int snap_stride, training;
};
__global__ void __launch_bounds__(256) sn_access_kernel(const SnAccessParams p) {
  __shared__ float red[32];
  extern __shared__ float sm[];  // tvec [max(out, in)]
  const int r = blockIdx.x, tid = threadIdx.x, L = p.net.n_layers;
  int u_total = 0, v_total = 0;
  for (int l = 0; l < L; ++l) { u_total += p.net.dims[l + 1]; v_total += p.net.dims[l]; }
  const float* prm = p.net.params + (int64_t)r * p.net.stride;
  float* eff = p.eff.params + (int64_t)r * p.eff.stride;
  float* snap = p.snap + (int64_t)r * p.snap_stride;
  int off = 0, uo = 0, vo = 0;  // running offsets of layer l: parameters (mlp_offsets rule), u, v
  for (int l = 0; l < L; ++l) {
    const int od = p.net.dims[l + 1], in = p.net.dims[l];
    const int w_off = off, b_off = (off + od * in + 3) / 4 * 4;
    off = (b_off + od + 3) / 4 * 4;
    const float* W = prm + w_off;
    float sigma = 1.f;
    if (p.u) {
      float* u = p.u + (int64_t)r * p.u_stride + uo;
      float* v = p.v + (int64_t)r * p.v_stride + vo;
      __syncthreads();
      if (p.training) {  // u <- normalize(W v), v <- normalize(W^T u)  (eps 1e-12)
        for (int i = tid; i < od; i += 256) { float s = 0.f; for (int j = 0; j < in; ++j) s = fmaf(W[i * in + j], v[j], s); sm[i] = s; }
        __syncthreads();
        float nn = 0.f;
        for (int i = tid; i < od; i += 256) nn = fmaf(sm[i], sm[i], nn);
        nn = fmaxf(sqrtf(block_sum(nn, red)), 1e-12f);
        for (int i = tid; i < od; i += 256) u[i] = sm[i] / nn;
        __syncthreads();
        for (int j = tid; j < in; j += 256) { float s = 0.f; for (int i = 0; i < od; ++i) s = fmaf(W[i * in + j], u[i], s); sm[j] = s; }
        __syncthreads();
        nn = 0.f;
        for (int j = tid; j < in; j += 256) nn = fmaf(sm[j], sm[j], nn);
        nn = fmaxf(sqrtf(block_sum(nn, red)), 1e-12f);
        for (int j = tid; j < in; j += 256) v[j] = sm[j] / nn;
        __syncthreads();
      }
      float s = 0.f;  // sigma = u . (W v)
      for (int i = tid; i < od; i += 256) { float t = 0.f; for (int j = 0; j < in; ++j) t = fmaf(W[i * in + j], v[j], t); s = fmaf(u[i], t, s); }
      sigma = block_sum(s, red);
      for (int i = tid; i < od; i += 256) snap[uo + i] = u[i];
      for (int j = tid; j < in; j += 256) snap[u_total + vo + j] = v[j];
    }
    if (tid == 0) snap[u_total + v_total + l] = sigma;
    for (int i = tid; i < od * in; i += 256) eff[w_off + i] = W[i] / sigma;
    for (int i = tid; i < od; i += 256) eff[b_off + i] = prm[b_off + i];
    uo += od; vo += in;
  }
}

// dL/dW_orig += (G - <G, W_eff> u v^T) / sigma per layer; biases add directly. One CTA per replica.
struct SnProjectParams {
  il_mlp eff;
  const float* g_eff;   // [R, eff.stride] gradient w.r.t. the effective parameters
  const float* snap;
  int snap_stride, has_sn;
  float* g_out;         // flat gradient buffer, this net's slice: element (r, i) at g_out + r * out_stride + i
  int64_t out_stride;
};
__global__ void __launch_bounds__(256) sn_project_kernel(const SnProjectParams p) {
  __shared__ float red[32];
  const int r = blockIdx.x, tid = threadIdx.x, L = p.eff.n_layers;
  int u_total = 0, v_total = 0;
  for (int l = 0; l < L; ++l) { u_total += p.eff.dims[l + 1]; v_total += p.eff.dims[l]; }
  const float* eff = p.eff.params + (int64_t)r * p.eff.stride;
  const float* G = p.g_eff + (int64_t)r * p.eff.stride;
  const float* snap = p.snap + (int64_t)r * p.snap_stride;
  float* out = p.g_out + (int64_t)r * p.out_stride;
  int off = 0, uo = 0, vo = 0;
  for (int l = 0; l < L; ++l) {
    const int od = p.eff.dims[l + 1], in = p.eff.dims[l];
    const int w_off = off, b_off = (off + od * in + 3) / 4 * 4;
    off = (b_off + od + 3) / 4 * 4;
    if (p.has_sn) {
      float s = 0.f;
      for (int i = tid; i < od * in; i += 256) s = fmaf(G[w_off + i], eff[w_off + i], s);
      const float inner = block_sum(s, red), sigma = snap[u_total + v_total + l];
      for (int i = tid; i < od * in; i += 256) out[w_off + i] += (G[w_off + i] - inner * snap[uo + i / in] * snap[u_total + vo + i % in]) / sigma;
    } else {
      for (int i = tid; i < od * in; i += 256) out[w_off + i] += G[w_off + i];
    }
    for (int i = tid; i < od; i += 256) out[b_off + i] += G[b_off + i];
    uo += od; vo += in;
  }
}

// training.py:79-81 on every field of the packed rows: out = eps * expert + (1 - eps) * policy
__global__ void mix_batch_kernel(const float* __restrict__ ex, int64_t ex_rs, const float* __restrict__ po, int64_t po_rs, const float* __restrict__ eps, float* __restrict__ out,
                                 int64_t out_rs, int R, int B, int row) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (int64_t)R * B * row) return;
  const int j = (int)(t % row);
  const int64_t rb = t / row;
  const int r = (int)(rb / B), b = (int)(rb % B);
  const float e = eps[rb];
  out[(int64_t)r * out_rs + (int64_t)b * row + j] = __fadd_rn(__fmul_rn(e, ex[(int64_t)r * ex_rs + (int64_t)b * row + j]), __fmul_rn(__fsub_rn(1.f, e), po[(int64_t)r * po_rs + (int64_t)b * row + j]));
}

struct PassView {        // one discriminator forward (models.py:172-175) on a batch
  const float* rows;     // packed rows (terminals, weights read from here)
  int64_t rs;
  const float* og;       // [R, B] g output
  const float* ohn;      // [R, B] h(next_state) output (nullptr without shaping)
  const float* ohs;      // [R, B] h(state)
  const float* logp;     // [R, B] log pi(a | s) (nullptr unless subtract_log_policy)
  const float* eps;      // [R, B] mixup epsilon (Mixup pass)
  float* dg;             // [R, B] out: dLoss / d g-output;  dhn, dhs likewise
  float* dhn;
  float* dhs;
  int kind;              // 0 policy, 1 expert, 2 mixup
};
struct LossParams {
  PassView pass[2];
  int n_pass, B, row, off_terminal, off_weight, loss_function, shaping;
  float discount, entropy_bonus, pos_class_prior, nonnegative_margin;
  float* out_losses;     // [R, 2]
  const float* discount_r;       // [R] or nullptr (il_gailx.discount_r)
  const float* entropy_bonus_r;  // [R] or nullptr
};
__device__ __forceinline__ float pass_logit(const PassView& v, const LossParams& p, int r, int b, float* one_minus_t) {
  const int64_t i = (int64_t)r * p.B + b;
  float f = v.og[i];
  float omt = 1.f;
  if (p.shaping) {
    omt = 1.f - v.rows[(int64_t)r * v.rs + (int64_t)b * p.row + p.off_terminal];
    const float discount = p.discount_r ? p.discount_r[r] : p.discount;
    f = f + omt * (discount * v.ohn[i] - v.ohs[i]);  // models.py:174
  }
  if (v.logp) f = f - v.logp[i];                      // models.py:175
  *one_minus_t = omt;
  return f;
}
// training.py:94-114,130-132: loss value and d loss / d logits for every pass, then the output gradients of g, h(s'), h(s). One CTA per replica.
__global__ void __launch_bounds__(256) gailx_loss_kernel(const LossParams p) {
  __shared__ float red[32];
  const int r = blockIdx.x, B = p.B;
  const float invB = 1.f / (float)B;
  const float discount = p.discount_r ? p.discount_r[r] : p.discount, entropy_bonus = p.entropy_bonus_r ? p.entropy_bonus_r[r] : p.entropy_bonus;
  float pu_gate = 1.f;
  if (p.loss_function == IL_LOSS_PUGAIL) {  // the clamp of training.py:102 needs the batch scalar first
    float sp = 0.f, se = 0.f;
    for (int b = threadIdx.x; b < B; b += blockDim.x) {
      float omt;
      const float fp = pass_logit(p.pass[0], p, r, b, &omt), fe = pass_logit(p.pass[1], p, r, b, &omt);
      sp += p.pass[0].rows[(int64_t)r * p.pass[0].rs + (int64_t)b * p.row + p.off_weight] * softplusf(fp);
      se += p.pass[1].rows[(int64_t)r * p.pass[1].rs + (int64_t)b * p.row + p.off_weight] * softplusf(fe);
    }
    sp = block_sum(sp, red);
    se = block_sum(se, red);
    pu_gate = (p.pos_class_prior * (se * invB) - sp * invB) >= -p.nonnegative_margin ? 1.f : 0.f;
  }
  float loss = 0.f;
  for (int k = 0; k < p.n_pass; ++k) {
    const PassView& v = p.pass[k];
    for (int b = threadIdx.x; b < B; b += blockDim.x) {
      float omt;
      const float f = pass_logit(v, p, r, b, &omt), sg = sigmoidf(f);
      const float w = v.rows[(int64_t)r * v.rs + (int64_t)b * p.row + p.off_weight];
      float df;
      if (v.kind == 2) {
        const float e = v.eps[(int64_t)r * B + b];
        df = w * (sg - e) * invB;
        loss += e * w * softplusf(-f) + (1.f - e) * w * softplusf(f);
      } else if (p.loss_function == IL_LOSS_BCE) {
        df = v.kind == 1 ? w * (sg - 1.f) * invB : w * sg * invB;
        loss += v.kind == 1 ? w * softplusf(-f) : w * softplusf(f);
      } else {
        const float pr = p.pos_class_prior;
        df = v.kind == 1 ? pr * w * (sg - 1.f) * invB + pu_gate * pr * w * sg * invB : -pu_gate * w * sg * invB;
        loss += v.kind == 1 ? pr * w * softplusf(-f) + pu_gate * pr * w * softplusf(f) : -pu_gate * w * softplusf(f);
      }
      if (entropy_bonus > 0.f) df += entropy_bonus * w * f * sg * (1.f - sg) * invB;
      const int64_t i = (int64_t)r * B + b;
      v.dg[i] = df;
      if (p.shaping) { v.dhn[i] = df * omt * discount; v.dhs[i] = -df * omt; }
    }
  }
  loss = block_sum(loss, red);
  if (threadIdx.x == 0 && p.out_losses) p.out_losses[r * 2 + 0] = loss * invB;
}

// ---- gradient penalty element-wise pieces -------------------------------------------------------------------------------------
// kappa[r, b] of a net evaluation: 1 (g) or -(1 - terminal) (h(state)); terminals read from the mixed rows
struct Kappa {
  const float* rows;  // nullptr -> 1
  int64_t rs;
  int row, off_terminal;
};
__device__ __forceinline__ float kappa_at(const Kappa& k, int r, int b) { return k.rows ? -(1.f - k.rows[(int64_t)r * k.rs + (int64_t)b * k.row + k.off_terminal]) : 1.f; }

// top of the delta chain: U[b, j] = kappa_b W_L[j],  D = U * s'(Y)
__global__ void gp_top_kernel(const float* __restrict__ wl, int64_t w_gs, Kappa kp, const float* __restrict__ Y, float* __restrict__ U, float* __restrict__ D, int R, int B, int H, int act) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (int64_t)R * B * H) return;
  const int j = (int)(t % H);
  const int64_t rb = t / H;
  const int r = (int)(rb / B), b = (int)(rb % B);
  const float u = kappa_at(kp, r, b) * wl[(int64_t)r * w_gs + j];
  U[t] = u;
  D[t] = u * act_grad_from_output(Y[t], act);
}
__global__ void gp_mask_kernel(const float* __restrict__ U, const float* __restrict__ Y, float* __restrict__ D, int64_t n, int act) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n) D[t] = U[t] * act_grad_from_output(Y[t], act);
}
// linear net (L == 1): g_x[b, j] (+)= kappa_b W_1[j]
__global__ void gp_linear_gx_kernel(const float* __restrict__ w1, int64_t w_gs, Kappa kp, float* __restrict__ gin, int ld, int R, int B, int din, int accumulate) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (int64_t)R * B * din) return;
  const int j = (int)(t % din);
  const int64_t rb = t / din;
  const int r = (int)(rb / B), b = (int)(rb % B);
  const float v = kappa_at(kp, r, b) * w1[(int64_t)r * w_gs + j];
  float* dst = gin + rb * ld + j;
  *dst = accumulate ? *dst + v : v;
}
// P_b = lambda w_b |g_in|^2;  gbar = 2 lambda w_b / B * g_in (in place);  loss = mean(P). One CTA per replica.
__global__ void __launch_bounds__(256) gp_penalty_kernel(float* __restrict__ gin, int ld, int cols, const float* __restrict__ rows, int64_t rs, int row, int off_weight, float lambda,
                                                         const float* __restrict__ lambda_r, float* __restrict__ out_losses, int B) {
  __shared__ float red[32];
  const int r = blockIdx.x;
  if (lambda_r) lambda = lambda_r[r];
  float loss = 0.f;
  for (int b = threadIdx.x; b < B; b += blockDim.x) {
    float* g = gin + ((int64_t)r * B + b) * ld;
    const float w = rows[(int64_t)r * rs + (int64_t)b * row + off_weight];
    float pen = 0.f;
    for (int j = 0; j < cols; ++j) pen = fmaf(g[j], g[j], pen);
    loss += lambda * w * pen;
    const float c = 2.f * lambda * w / (float)B;
    for (int j = 0; j < cols; ++j) g[j] *= c;
  }
  loss = block_sum(loss, red);
  if (threadIdx.x == 0 && out_losses) out_losses[r * 2 + 1] = loss / (float)B;
}
// Ubar = Dbar * s'(Y);  Zgp = Dbar * U * s''(Y)
__global__ void gp_second_kernel(const float* __restrict__ Dbar, const float* __restrict__ U, const float* __restrict__ Y, float* __restrict__ Ubar, float* __restrict__ Zgp, int64_t n, int act) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  const float y = Y[t], d = Dbar[t];
  Ubar[t] = d * act_grad_from_output(y, act);
  Zgp[t] = d * U[t] * act_grad2_from_output(y, act);
}
// out[r, j] = sum_b kappa_b X[r, b, j]  (gradient of the last-layer weight row, or of a linear net's weight). One CTA per (replica, 256 columns).
__global__ void __launch_bounds__(256) gp_kappa_colsum_kernel(const float* __restrict__ X, int ld, Kappa kp, float* __restrict__ out, int64_t out_gs, int B, int cols) {
  const int r = blockIdx.y, j = blockIdx.x * 256 + threadIdx.x;
  if (j >= cols) return;
  float s = 0.f;
  for (int b = 0; b < B; ++b) s = fmaf(kappa_at(kp, r, b), X[((int64_t)r * B + b) * ld + j], s);
  out[(int64_t)r * out_gs + j] = s;
}
__global__ void add_kernel(float* __restrict__ a, const float* __restrict__ b, int64_t n) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t < n) a[t] += b[t];
}
// models.py:177-180 on combined logits
__global__ void gailx_reward_kernel(PassView v, LossParams p, int reward_function, float* __restrict__ reward, int64_t reward_rs, int reward_ld, float* __restrict__ logits, int R) {
  const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (int64_t)R * p.B) return;
  const int r = (int)(t / p.B), b = (int)(t % p.B);
  float omt;
  const float f = pass_logit(v, p, r, b, &omt);
  if (logits) logits[t] = f;
  if (reward) {
    const float D = sigmoidf(f);
    float hh = reward_function == IL_REWARD_GAIL ? -log1pf(-D + 1e-6f) : logf(D + 1e-6f) - log1pf(-D + 1e-6f);
    if (reward_function == IL_REWARD_FAIRL) hh = expf(hh) * -hh;
    reward[(int64_t)r * reward_rs + (int64_t)b * reward_ld] = hh;
  }
}

// ---- host-side program ----------------------------------------------------------------------------------------------------------
struct Carver {
  char* p;
  int64_t used;
  float* take(int64_t floats) {
    float* r = p ? reinterpret_cast<float*>(p + used) : nullptr;
    used += il_align_up(floats * 4, 256);
    return r;
  }
};

struct NetEval {        // one spectral-norm access + forward of one net on one input view
  const il_mlp* net;
  float *u, *v;
  int u_stride, v_stride;
  il_mlp eff;           // effective parameters of this access (workspace), same layout as the net
  float* snap;
  int snap_stride;
  MlpActs acts;
  float* out;           // [R, B]
  float* dout;          // [R, B] output gradient (loss passes)
  float* g_eff;         // [R, net stride]
  MatView X;
  int din;
  float* g_out;         // this net's slice of the flat gradient buffer
};

int snap_floats(const il_mlp* m) {
  const SnLayout s = sn_layout(m->dims, m->n_layers);
  return (s.u_total + s.v_total + m->n_layers + 3) / 4 * 4;
}
int max_dim(const il_mlp* m) {
  int d = 1;
  for (int l = 0; l <= m->n_layers; ++l) d = m->dims[l] > d ? m->dims[l] : d;
  return d;
}

void eval_carve(Carver& c, NetEval& e, const il_mlp* net, float* u, float* v, int us, int vs, int R, int B, bool need_grad) {
  e.net = net; e.u = u; e.v = v; e.u_stride = us; e.v_stride = vs;
  e.eff = *net;
  e.eff.params = c.take((int64_t)R * net->stride);
  e.snap_stride = snap_floats(net);
  e.snap = c.take((int64_t)R * e.snap_stride);
  for (int l = 0; l < IL_MAX_LAYERS; ++l) e.acts.hid[l] = nullptr;
  for (int l = 0; l + 1 < net->n_layers; ++l) e.acts.hid[l] = c.take((int64_t)R * B * net->dims[l + 1]);
  e.out = c.take((int64_t)R * B);
  e.dout = need_grad ? c.take((int64_t)R * B) : nullptr;
  e.g_eff = need_grad ? c.take((int64_t)R * net->stride) : nullptr;
  e.din = net->dims[0];
}

int eval_access(il_handle* h, NetEval& e, int R, int training, cudaStream_t st) {
  SnAccessParams p;
  p.net = *e.net; p.eff = e.eff; p.u = e.u; p.v = e.v; p.u_stride = e.u_stride; p.v_stride = e.v_stride; p.snap = e.snap; p.snap_stride = e.snap_stride; p.training = training;
  IL_LAUNCH(h, sn_access_kernel, R, 256, (size_t)max_dim(e.net) * 4, st, p);
  return 0;
}
int eval_forward(il_handle* h, NetEval& e, int R, int B, cudaStream_t st) { return mlp_forward(h, &e.eff, R, B, e.X, e.acts, e.out, (int64_t)B, 1, st); }
int eval_project(il_handle* h, NetEval& e, int R, int64_t out_stride, cudaStream_t st) {
  IL_CHECK(e.eff.params && e.g_eff && e.snap && e.g_out, "gailx: internal: projecting an evaluation without gradient storage (eff=%p g_eff=%p snap=%p out=%p)", (void*)e.eff.params,
           (void*)e.g_eff, (void*)e.snap, (void*)e.g_out);
  SnProjectParams p;
  p.eff = e.eff; p.g_eff = e.g_eff; p.snap = e.snap; p.snap_stride = e.snap_stride; p.has_sn = e.u != nullptr; p.g_out = e.g_out; p.out_stride = out_stride;
  IL_LAUNCH(h, sn_project_kernel, R, 256, 0, st, p);
  return 0;
}

struct GpBufs {  // per hidden layer: U (pre-mask back signal), D (delta), Dbar, Ubar, Zgp; plus scratch
  float *U[IL_MAX_LAYERS], *D[IL_MAX_LAYERS], *Dbar[IL_MAX_LAYERS], *Ubar[IL_MAX_LAYERS], *Zgp[IL_MAX_LAYERS], *T;
};
void gp_carve(Carver& c, GpBufs& g, int R, int B, int hmax, int n_hidden) {
  for (int l = 0; l < IL_MAX_LAYERS; ++l) g.U[l] = g.D[l] = g.Dbar[l] = g.Ubar[l] = g.Zgp[l] = nullptr;
  for (int l = 0; l < n_hidden; ++l) {
    g.U[l] = c.take((int64_t)R * B * hmax); g.D[l] = c.take((int64_t)R * B * hmax); g.Dbar[l] = c.take((int64_t)R * B * hmax);
    g.Ubar[l] = c.take((int64_t)R * B * hmax); g.Zgp[l] = c.take((int64_t)R * B * hmax);
  }
  g.T = c.take((int64_t)R * B * hmax);
}

GemmArgs gemm(int M, int N, int K, int G, const float* A, int64_t a_gs, int lda, int a_km, const float* Bm, int64_t b_gs, int ldb, int b_km, float* C, int64_t c_gs, int ldc) {
  GemmArgs a{};
  a.A = A; a.a_gs = a_gs; a.a_gdiv = 1; a.lda = lda; a.a_kmajor = a_km;
  a.B = Bm; a.b_gs = b_gs; a.b_gdiv = 1; a.ldb = ldb; a.b_kmajor = b_km;
  a.C = C; a.c_gs = c_gs; a.ldc = ldc; a.act = -1;
  a.M = M; a.N = N; a.K = K; a.G = G;
  return a;
}
unsigned blocks(int64_t n) { return (unsigned)((n + 255) / 256); }

// Input gradient of one net evaluation (forward already done): writes / accumulates g_x into gin[:, :, 0:din] and keeps the delta chain in gb.
int gp_input_gradient(il_handle* h, NetEval& e, const Kappa& kp, GpBufs& gb, float* gin, int ld_gin, int accumulate, int R, int B, cudaStream_t st) {
  const il_mlp& m = e.eff;
  const int L = m.n_layers, act = m.activation;
  const MlpOffsets o = mlp_offsets(m.dims, L);
  if (L == 1) {
    IL_LAUNCH(h, gp_linear_gx_kernel, blocks((int64_t)R * B * e.din), 256, 0, st, m.params + o.w[0], m.stride, kp, gin, ld_gin, R, B, e.din, accumulate);
    return 0;
  }
  const int Ht = m.dims[L - 1];
  IL_LAUNCH(h, gp_top_kernel, blocks((int64_t)R * B * Ht), 256, 0, st, m.params + o.w[L - 1], m.stride, kp, e.acts.hid[L - 2], gb.U[L - 2], gb.D[L - 2], R, B, Ht, act);
  for (int l = L - 2; l >= 1; --l) {  // U_l = D_{l+1} W_{l+1};  D_l = U_l * s'(Y_l)   (hidden layer l has index l - 1 in the buffers)
    const int Hu = m.dims[l + 1], Hl = m.dims[l];
    IL_TRY(launch_gemm(h, gemm(B, Hl, Hu, R, gb.D[l], (int64_t)B * Hu, Hu, 1, m.params + o.w[l], m.stride, Hl, 0, gb.U[l - 1], (int64_t)B * Hl, Hl), st));
    IL_LAUNCH(h, gp_mask_kernel, blocks((int64_t)R * B * Hl), 256, 0, st, gb.U[l - 1], e.acts.hid[l - 1], gb.D[l - 1], (int64_t)R * B * Hl, act);
  }
  GemmArgs a = gemm(B, e.din, m.dims[1], R, gb.D[0], (int64_t)B * m.dims[1], m.dims[1], 1, m.params + o.w[0], m.stride, m.dims[0], 0, gin, (int64_t)B * ld_gin, ld_gin);
  a.accumulate = accumulate;
  return launch_gemm(h, a, st);
}

// Double backward of the penalty through one net evaluation: gbar [R, B, ld] (first din columns) -> e.g_eff (overwritten).
int gp_double_backward(il_handle* h, NetEval& e, const Kappa& kp, GpBufs& gb, const float* gbar, int ld, int R, int B, cudaStream_t st) {
  const il_mlp& m = e.eff;
  const int L = m.n_layers, act = m.activation;
  const MlpOffsets o = mlp_offsets(m.dims, L);
  IL_CUDA(cudaMemsetAsync(e.g_eff, 0, (size_t)R * m.stride * 4, st));
  if (L == 1) {  // g_x = kappa_b W_1: dW_1[j] = sum_b kappa_b gbar[b, j]
    IL_LAUNCH(h, gp_kappa_colsum_kernel, dim3((e.din + 255) / 256, R), 256, 0, st, gbar, ld, kp, e.g_eff + o.w[0], m.stride, B, e.din);
    return 0;
  }
  const int H1 = m.dims[1];
  // dW_1 = D_1^T gbar ;  Dbar_1 = gbar W_1^T
  IL_TRY(launch_gemm(h, gemm(H1, e.din, B, R, gb.D[0], (int64_t)B * H1, H1, 0, gbar, (int64_t)B * ld, ld, 0, e.g_eff + o.w[0], m.stride, m.dims[0]), st));
  IL_TRY(launch_gemm(h, gemm(B, H1, e.din, R, gbar, (int64_t)B * ld, ld, 1, m.params + o.w[0], m.stride, m.dims[0], 1, gb.Dbar[0], (int64_t)B * H1, H1), st));
  for (int l = 1; l <= L - 1; ++l) {
    const int Hl = m.dims[l];
    IL_LAUNCH(h, gp_second_kernel, blocks((int64_t)R * B * Hl), 256, 0, st, gb.Dbar[l - 1], gb.U[l - 1], e.acts.hid[l - 1], gb.Ubar[l - 1], gb.Zgp[l - 1], (int64_t)R * B * Hl, act);
    if (l < L - 1) {  // dW_{l+1} = D_{l+1}^T Ubar_l ;  Dbar_{l+1} = Ubar_l W_{l+1}^T
      const int Hu = m.dims[l + 1];
      IL_TRY(launch_gemm(h, gemm(Hu, Hl, B, R, gb.D[l], (int64_t)B * Hu, Hu, 0, gb.Ubar[l - 1], (int64_t)B * Hl, Hl, 0, e.g_eff + o.w[l], m.stride, Hl), st));
      IL_TRY(launch_gemm(h, gemm(B, Hu, Hl, R, gb.Ubar[l - 1], (int64_t)B * Hl, Hl, 1, m.params + o.w[l], m.stride, Hl, 1, gb.Dbar[l], (int64_t)B * Hu, Hu), st));
    } else {  // u_{L-1} = kappa_b W_L: dW_L[j] = sum_b kappa_b Ubar[b, j]
      IL_LAUNCH(h, gp_kappa_colsum_kernel, dim3((Hl + 255) / 256, R), 256, 0, st, gb.Ubar[l - 1], Hl, kp, e.g_eff + o.w[L - 1], m.stride, B, Hl);
    }
  }
  if (act == IL_ACT_RELU) return 0;  // s'' = 0: nothing flows through the pre-activations
  // ordinary backward of zbar_l = Zgp_l (+ what arrives from above): dW_l += zbar_l^T Y_{l-1}, db_l = colsum(zbar_l), zbar_{l-1} += (zbar_l W_l) * s'(Y_{l-1})
  float* zbar = gb.Zgp[L - 2];
  for (int l = L - 1; l >= 1; --l) {
    const int Hl = m.dims[l], Hin = m.dims[l - 1];
    GemmArgs a = l == 1 ? gemm(Hl, Hin, B, R, zbar, (int64_t)B * Hl, Hl, 0, e.X.ptr, e.X.gs, e.X.ld, 0, e.g_eff + o.w[0], m.stride, Hin)
                        : gemm(Hl, Hin, B, R, zbar, (int64_t)B * Hl, Hl, 0, e.acts.hid[l - 2], (int64_t)B * Hin, Hin, 0, e.g_eff + o.w[l - 1], m.stride, Hin);
    if (l == 1) a.b_gdiv = e.X.gdiv;
    a.accumulate = 1;
    a.colsum = e.g_eff + o.b[l - 1]; a.colsum_gs = m.stride;
    IL_TRY(launch_gemm(h, a, st));
    if (l > 1) {
      GemmArgs d = gemm(B, Hin, Hl, R, zbar, (int64_t)B * Hl, Hl, 1, m.params + o.w[l - 1], m.stride, Hin, 0, gb.T, (int64_t)B * Hin, Hin);
      d.mask = e.acts.hid[l - 2]; d.mask_gs = (int64_t)B * Hin; d.ldmask = Hin; d.mask_act = act;
      IL_TRY(launch_gemm(h, d, st));
      IL_LAUNCH(h, add_kernel, blocks((int64_t)R * B * Hin), 256, 0, st, gb.Zgp[l - 2], gb.T, (int64_t)R * B * Hin);
      zbar = gb.Zgp[l - 2];
    }
  }
  return 0;
}

int validate_disc(const il_gailx* d, const il_batch* b, const char* what) {
  IL_CHECK(d && d->g.params, "%s: null discriminator", what);
  IL_TRY(mlp_validate(&d->g, what));
  const int din = d->state_only ? b->S : b->S + b->A;
  IL_CHECK(d->g.dims[0] == din && d->g.dims[d->g.n_layers] == 1, "%s: g dims do not match the input width %d", what, din);
  if (d->h.n_layers > 0) {
    IL_TRY(mlp_validate(&d->h, what));
    IL_CHECK(d->g.n_layers == 1, "%s: with reward shaping g is a single linear layer (models.py:158)", what);
    IL_CHECK(d->h.dims[0] == b->S && d->h.dims[d->h.n_layers] == 1 && d->h.activation == d->g.activation, "%s: h dims do not match the state size %d", what, b->S);
    IL_CHECK((d->h_u == nullptr) == (d->g_u == nullptr), "%s: spectral norm must cover both g and h", what);
  }
  IL_CHECK((d->g_u == nullptr) == (d->g_v == nullptr), "%s: spectral-norm buffers must both be set or both be null", what);
  IL_CHECK(b->row == row_layout(b->S, b->A).len && b->rows, "%s: bad batch", what);
  return 0;
}

struct UpdLayout {
  NetEval ev[GX_MAX_EVALS];
  int n_ev;
  float* mix_rows[2];   // mixup batch, gradient-penalty batch
  float* gin;           // [R, B, S + A]
  float* g_flat;        // [R, params stride] gradient w.r.t. the original parameters
  float *tmpA, *tmpB;   // ping-pong scratch of the MLP backward program
  GpBufs gb;
  int64_t bytes;
};

// evaluation slots: pass k (loss passes first, then the GP pass) x {g, h(s'), h(s)}
void upd_layout(const il_gailx_update_args* a, char* base, UpdLayout* L) {
  Carver c{base, 0};
  const il_gailx& d = a->disc;
  const int R = a->R, B = a->policy.B, S = a->policy.S, A = a->policy.A, row = a->policy.row;
  const bool shaping = d.h.n_layers > 0, gp = a->grad_penalty > 0.f, mixup = a->loss_function == IL_LOSS_MIXUP;
  const int n_loss_pass = mixup ? 1 : 2;
  L->n_ev = 0;
  for (int k = 0; k < n_loss_pass + (gp ? 1 : 0); ++k) {
    const bool is_gp = k == n_loss_pass;
    eval_carve(c, L->ev[L->n_ev++], &d.g, d.g_u, d.g_v, d.g_u_stride, d.g_v_stride, R, B, true);
    if (shaping) {
      eval_carve(c, L->ev[L->n_ev++], &d.h, d.h_u, d.h_v, d.h_u_stride, d.h_v_stride, R, B, !is_gp);  // h(s'): forward only in the GP pass (its input is not differentiated)
      eval_carve(c, L->ev[L->n_ev++], &d.h, d.h_u, d.h_v, d.h_u_stride, d.h_v_stride, R, B, true);
    }
  }
  L->mix_rows[0] = mixup ? c.take((int64_t)R * B * row) : nullptr;
  L->mix_rows[1] = gp ? c.take((int64_t)R * B * row) : nullptr;
  L->gin = gp ? c.take((int64_t)R * B * (S + A)) : nullptr;
  L->g_flat = c.take(a->params_floats);
  int hmax = 1, nh = 0;
  const il_mlp* nets[2] = {&d.g, &d.h};
  for (const il_mlp* m : nets) {
    if (m->n_layers == 0) continue;
    for (int l = 1; l < m->n_layers; ++l) hmax = m->dims[l] > hmax ? m->dims[l] : hmax;
    nh = m->n_layers - 1 > nh ? m->n_layers - 1 : nh;
  }
  L->tmpA = c.take((int64_t)R * B * hmax);
  L->tmpB = c.take((int64_t)R * B * hmax);
  if (gp) gp_carve(c, L->gb, R, B, hmax, nh);
  L->bytes = c.used;
}

}  // namespace

extern "C" int il_gail_mix_batch(il_handle* h, const il_batch* expert, const il_batch* policy, const float* eps, int R, const il_batch* out, void* stream) {
  IL_CHECK(h && expert && policy && eps && out && R > 0, "il_gail_mix_batch: bad argument");
  IL_CHECK(expert->row == policy->row && out->row == policy->row && expert->B == policy->B && out->B == policy->B && expert->rows && policy->rows && out->rows, "il_gail_mix_batch: shape mismatch");
  const int64_t n = (int64_t)R * policy->B * policy->row;
  IL_LAUNCH(h, mix_batch_kernel, blocks(n), 256, 0, (cudaStream_t)stream, expert->rows, expert->replica_stride, policy->rows, policy->replica_stride, eps, out->rows, out->replica_stride, R,
            policy->B, policy->row);
  return 0;
}

extern "C" int64_t il_gailx_workspace_bytes(const il_gailx_update_args* a) {
  if (!a) return -1;
  UpdLayout L;
  upd_layout(a, nullptr, &L);
  return L.bytes;
}

extern "C" int il_gailx_update(il_handle* h, const il_gailx_update_args* a, void* stream) {
  IL_CHECK(h && a, "il_gailx_update: null argument");
  cudaStream_t st = (cudaStream_t)stream;
  const il_gailx& d = a->disc;
  IL_TRY(validate_disc(&d, &a->policy, "il_gailx_update"));
  const int R = a->R, B = a->policy.B, S = a->policy.S, A = a->policy.A, row = a->policy.row;
  const RowLayout RL = row_layout(S, A);
  IL_CHECK(R > 0 && a->expert.rows && a->expert.B == B && a->expert.S == S && a->expert.A == A, "il_gailx_update: policy / expert batch mismatch");
  IL_CHECK(a->opt.m && a->opt.v && a->opt.step && a->params_floats > 0, "il_gailx_update: null optimiser state");
  IL_CHECK(a->loss_function >= 0 && a->loss_function <= 2, "il_gailx_update: bad loss function %d", a->loss_function);
  const bool shaping = d.h.n_layers > 0, gp = a->grad_penalty > 0.f, mixup = a->loss_function == IL_LOSS_MIXUP, sublp = d.subtract_log_policy != 0;
  IL_CHECK(!(gp && !a->eps_gp) && !(mixup && !a->eps_mix), "il_gailx_update: missing eps_gp / eps_mix");
  IL_CHECK(!(gp && d.state_only), "il_gailx_update: grad_penalty with a state-only discriminator is undefined in the reference (autograd.grad on the unused action, training.py:125)");
  IL_CHECK(!sublp || (mixup ? a->logp_mix != nullptr : (a->logp_policy && a->logp_expert)), "il_gailx_update: subtract_log_policy needs the log-policy inputs");
  IL_CHECK(a->workspace && a->workspace_bytes >= il_gailx_workspace_bytes(a), "il_gailx_update: workspace too small");
  UpdLayout L;
  upd_layout(a, static_cast<char*>(a->workspace), &L);
  const int64_t pstride = a->params_floats / R;
  IL_CHECK(pstride * R == a->params_floats && d.g.stride == pstride && (!shaping || d.h.stride == pstride), "il_gailx_update: g / h must live in one flat [R, stride] parameter buffer");
  IL_CUDA(cudaMemsetAsync(L.g_flat, 0, (size_t)a->params_floats * 4, st));
  IL_TRY(launch_tick(h, a->opt.step, nullptr, nullptr, st));

  const int per_pass = shaping ? 3 : 1, n_loss_pass = mixup ? 1 : 2;
  const int64_t h_off = shaping ? d.h.params - d.g.params : 0;
  // ---- batches of the passes ------------------------------------------------------------------------------------------------
  const float* pass_rows[3]; int64_t pass_rs[3];
  if (mixup) {
    il_batch ob = a->policy; ob.rows = L.mix_rows[0]; ob.replica_stride = (int64_t)B * row;
    IL_TRY(il_gail_mix_batch(h, &a->expert, &a->policy, a->eps_mix, R, &ob, stream));
    pass_rows[0] = L.mix_rows[0]; pass_rs[0] = (int64_t)B * row;
  } else {
    pass_rows[0] = a->policy.rows; pass_rs[0] = a->policy.replica_stride;
    pass_rows[1] = a->expert.rows; pass_rs[1] = a->expert.replica_stride;
  }
  if (gp) {
    il_batch ob = a->policy; ob.rows = L.mix_rows[1]; ob.replica_stride = (int64_t)B * row;
    IL_TRY(il_gail_mix_batch(h, &a->expert, &a->policy, a->eps_gp, R, &ob, stream));
    pass_rows[n_loss_pass] = L.mix_rows[1]; pass_rs[n_loss_pass] = (int64_t)B * row;
  }
  // ---- forwards in the reference's order: per pass g, h(s'), h(s); each one spectral-norm access --------------------------------
  for (int k = 0; k < n_loss_pass + (gp ? 1 : 0); ++k) {
    const bool is_gp = k == n_loss_pass;
    for (int j = 0; j < per_pass; ++j) {
      NetEval& e = L.ev[k * per_pass + j];
      const int col0 = j == 1 ? RL.next_state : RL.state;
      e.X = MatView{pass_rows[k] + col0, pass_rs[k], 1, row};
      e.g_out = L.g_flat + (j == 0 ? 0 : h_off);
      IL_TRY(eval_access(h, e, R, a->training, st));
      GX_STAGE(h, st, "access pass %d net %d", k, j);
      if (is_gp && j == 1) continue;  // h(s') of the GP pass: the access (power iteration) happens, its value and gradient are never used
      IL_TRY(eval_forward(h, e, R, B, st));
      GX_STAGE(h, st, "forward pass %d net %d", k, j);
    }
  }
  // ---- loss, d loss / d outputs -------------------------------------------------------------------------------------------------
  LossParams lp{};
  lp.n_pass = n_loss_pass; lp.B = B; lp.row = row; lp.off_terminal = RL.terminal; lp.off_weight = RL.weight; lp.loss_function = a->loss_function; lp.shaping = shaping;
  lp.discount = d.discount; lp.entropy_bonus = a->entropy_bonus; lp.pos_class_prior = a->pos_class_prior; lp.nonnegative_margin = a->nonnegative_margin; lp.out_losses = a->out_losses;
  lp.discount_r = d.discount_r; lp.entropy_bonus_r = a->entropy_bonus_r;
  for (int k = 0; k < n_loss_pass; ++k) {
    PassView& v = lp.pass[k];
    NetEval* e = &L.ev[k * per_pass];
    v.rows = pass_rows[k]; v.rs = pass_rs[k];
    v.og = e[0].out; v.dg = e[0].dout;
    if (shaping) { v.ohn = e[1].out; v.ohs = e[2].out; v.dhn = e[1].dout; v.dhs = e[2].dout; }
    v.logp = sublp ? (mixup ? a->logp_mix : (k == 0 ? a->logp_policy : a->logp_expert)) : nullptr;
    v.eps = mixup ? a->eps_mix : nullptr;
    v.kind = mixup ? 2 : k;
  }
  IL_LAUNCH(h, gailx_loss_kernel, R, 256, 0, st, lp);
  GX_STAGE(h, st, "loss");
  // ---- backward of the loss passes, projected through each access ----------------------------------------------------------------
  for (int k = 0; k < n_loss_pass; ++k)
    for (int j = 0; j < per_pass; ++j) {
      NetEval& e = L.ev[k * per_pass + j];
      IL_TRY(mlp_backward(h, &e.eff, R, B, e.X, e.acts, MatView{e.dout, (int64_t)B, 1, 1}, e.g_eff, e.eff.stride, nullptr, 0, 0, 0, 0, L.tmpA, L.tmpB, st));
      GX_STAGE(h, st, "backward pass %d net %d", k, j);
      IL_TRY(eval_project(h, e, R, pstride, st));
      GX_STAGE(h, st, "project pass %d net %d (eff %p g_eff %p out %p ws %p + %lld)", k, j, (void*)e.eff.params, (void*)e.g_eff, (void*)e.g_out, a->workspace, (long long)a->workspace_bytes);
    }
  // ---- gradient penalty ------------------------------------------------------------------------------------------------------------
  if (gp) {
    NetEval* e = &L.ev[n_loss_pass * per_pass];
    const Kappa one{nullptr, 0, 0, 0}, kh{pass_rows[n_loss_pass], pass_rs[n_loss_pass], row, RL.terminal};
    const int ld = S + A;
    IL_CUDA(cudaMemsetAsync(L.gin, 0, (size_t)R * B * ld * 4, st));
    // The penalty couples the nets through |g_x(g) + g_x(h)|^2, so both input gradients come first. Only one net has a delta chain to
    // keep for the double backward: with reward shaping g is linear (no chain) and h owns the scratch; without shaping there is only g.
    IL_TRY(gp_input_gradient(h, e[0], one, L.gb, L.gin, ld, 0, R, B, st));
    if (shaping) IL_TRY(gp_input_gradient(h, e[2], kh, L.gb, L.gin, ld, 1, R, B, st));
    IL_LAUNCH(h, gp_penalty_kernel, R, 256, 0, st, L.gin, ld, ld, pass_rows[n_loss_pass], pass_rs[n_loss_pass], row, RL.weight, a->grad_penalty, a->grad_penalty_r, a->out_losses,
              B);
    GX_STAGE(h, st, "gp input gradients + penalty");
    if (shaping) {
      IL_TRY(gp_double_backward(h, e[2], kh, L.gb, L.gin, ld, R, B, st));
      GX_STAGE(h, st, "gp double backward h");
      IL_TRY(eval_project(h, e[2], R, pstride, st));
      GX_STAGE(h, st, "gp project h");
    }
    IL_TRY(gp_double_backward(h, e[0], one, L.gb, L.gin, ld, R, B, st));
    GX_STAGE(h, st, "gp double backward g");
    IL_TRY(eval_project(h, e[0], R, pstride, st));
    GX_STAGE(h, st, "gp project g");
  }
  // ---- AdamW over the flat parameter buffer (train.py:84) ------------------------------------------------------------------------
  il_adam opt = a->opt;
  opt.replica_floats = pstride;
  return launch_adam(h, d.g.params, L.g_flat, &opt, a->params_floats, st);
}

extern "C" int64_t il_gailx_reward_workspace_bytes(const il_gailx* d, int R, int B) {
  if (!d || R <= 0 || B <= 0) return -1;
  Carver c{nullptr, 0};
  NetEval e;
  eval_carve(c, e, &d->g, nullptr, nullptr, 0, 0, R, B, false);
  if (d->h.n_layers > 0) { eval_carve(c, e, &d->h, nullptr, nullptr, 0, 0, R, B, false); eval_carve(c, e, &d->h, nullptr, nullptr, 0, 0, R, B, false); }
  return c.used;
}

extern "C" int il_gailx_reward(il_handle* h, const il_gailx* d, int R, const il_batch* batch, const float* log_policy, float* reward, int64_t reward_rs, int reward_ld, float* logits,
                               void* workspace, int64_t workspace_bytes, void* stream) {
  IL_CHECK(h && d && batch && R > 0 && workspace, "il_gailx_reward: bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  IL_TRY(validate_disc(d, batch, "il_gailx_reward"));
  IL_CHECK(workspace_bytes >= il_gailx_reward_workspace_bytes(d, R, batch->B), "il_gailx_reward: workspace too small");
  IL_CHECK(!d->subtract_log_policy || log_policy, "il_gailx_reward: subtract_log_policy needs log_policy");
  const int B = batch->B, row = batch->row;
  const RowLayout RL = row_layout(batch->S, batch->A);
  const bool shaping = d->h.n_layers > 0;
  Carver c{static_cast<char*>(workspace), 0};
  NetEval ev[3];
  eval_carve(c, ev[0], &d->g, d->g_u, d->g_v, d->g_u_stride, d->g_v_stride, R, B, false);
  if (shaping) {
    eval_carve(c, ev[1], &d->h, d->h_u, d->h_v, d->h_u_stride, d->h_v_stride, R, B, false);
    eval_carve(c, ev[2], &d->h, d->h_u, d->h_v, d->h_u_stride, d->h_v_stride, R, B, false);
  }
  for (int j = 0; j < (shaping ? 3 : 1); ++j) {  // eval mode (train.py:180,194): no power iteration, sigma from the stored (u, v)
    ev[j].X = MatView{batch->rows + (j == 1 ? RL.next_state : RL.state), batch->replica_stride, 1, row};
    IL_TRY(eval_access(h, ev[j], R, 0, st));
    IL_TRY(eval_forward(h, ev[j], R, B, st));
  }
  LossParams lp{};
  lp.B = B; lp.row = row; lp.off_terminal = RL.terminal; lp.off_weight = RL.weight; lp.shaping = shaping; lp.discount = d->discount; lp.discount_r = d->discount_r;
  PassView v{};
  v.rows = batch->rows; v.rs = batch->replica_stride; v.og = ev[0].out;
  if (shaping) { v.ohn = ev[1].out; v.ohs = ev[2].out; }
  v.logp = d->subtract_log_policy ? log_policy : nullptr;
  IL_LAUNCH(h, gailx_reward_kernel, blocks((int64_t)R * B), 256, 0, st, v, lp, d->reward_function, reward, reward_rs, reward_ld, logits, R);
  return 0;
}
