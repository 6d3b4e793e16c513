// GAILDiscriminator (models.py:152-180, depth-1 `g` network, optional spectral norm) — one CTA per replica.
//   il_gail_update : adversarial_imitation_update (training.py:85-134): BCE / PUGAIL / Mixup loss, gradient
//                    penalty (closed-form double backward for a one-hidden-layer net, SURVEY.md §8a a13),
//                    entropy bonus, spectral-norm power iterations per train-mode forward (a12) and their
//                    backward projection, AdamW — everything in shared memory, parameters touched once.
//   il_gail_reward : eval-mode forward + reward (models.py:177-180).
#include "common.cuh"

namespace {

constexpr int THREADS = 256;
enum PassKind { PASS_POLICY = 0, PASS_EXPERT = 1, PASS_MIX = 2 };

struct GailDims {
  int S, A, d, H, B, row, ldx, ldz, RB, HD;
};

struct GailSmem {
  float *W1, *W1e, *G1, *b1, *w2, *w2e, *G2, *gb1, *G2k, *gb1k, *u1, *v1, *v2, *tvec, *slots, *X, *Z, *GX, *DF, *CO, *red, *scal, *part;
};

__host__ __device__ inline int gail_slot_floats(int H, int d) { return 2 * H + d + 4; }  // u1[H] v1[d] v2[H] + sigma1 sigma2 u2 pad

__host__ __device__ inline int64_t gail_carve(const GailDims& g, float* base, GailSmem* s) {
  int64_t o = 0;
  auto take = [&](int n) { float* p = base ? base + o : nullptr; o += (n + 3) / 4 * 4; return p; };
  GailSmem t;
  t.W1 = take(g.HD); t.W1e = take(g.HD); t.G1 = take(g.HD);
  t.b1 = take(g.H); t.w2 = take(g.H); t.w2e = take(g.H); t.G2 = take(g.H); t.gb1 = take(g.H); t.G2k = take(g.H); t.gb1k = take(g.H);
  t.u1 = take(g.H); t.v1 = take(g.d); t.v2 = take(g.H); t.tvec = take(g.H > g.d ? g.H : g.d);
  t.slots = take(3 * gail_slot_floats(g.H, g.d));
  t.X = take(g.RB * g.ldx); t.Z = take(g.RB * g.ldz); t.GX = take(g.RB * g.ldx); t.DF = take(g.RB); t.CO = take(g.RB);
  t.red = take(32); t.scal = take(32); t.part = take(2 * THREADS);  // per-thread partial sums of the row-split reductions
  if (s) *s = t;
  return o * 4;
}

__host__ inline GailDims gail_dims(int S, int A, int H, int B, int state_only, int RB) {
  GailDims g;
  g.S = S; g.A = A; g.d = state_only ? S : S + A; g.H = H; g.B = B; g.row = row_layout(S, A).len;
  g.ldx = g.d | 1; g.ldz = H | 1; g.RB = RB; g.HD = (H * g.d + 3) / 4 * 4;
  return g;
}

struct GailUpdParams {
  il_gail_update_args a;
  GailDims g;
  int64_t off_w1, off_b1, off_w2, off_b2;
};
struct GailRewParams {
  il_gail disc;
  il_batch batch;
  GailDims g;
  int64_t off_w1, off_b1, off_w2, off_b2;
  float* reward; int64_t reward_rs; int reward_ld;
  float* logits;
};

__device__ __forceinline__ float bsum(float v, float* red) { return block_sum(v, red); }

// W v for a [H, d] matrix in shared memory -> out[H]
__device__ void matvec(const float* W, const float* v, float* out, int H, int d) {
  for (int h = threadIdx.x; h < H; h += blockDim.x) {
    float s = 0.f;
    for (int j = 0; j < d; ++j) s = fmaf(W[h * d + j], v[j], s);
    out[h] = s;
  }
}
__device__ void matvec_t(const float* W, const float* u, float* out, int H, int d) {
  for (int j = threadIdx.x; j < d; j += blockDim.x) {
    float s = 0.f;
    for (int h = 0; h < H; ++h) s = fmaf(W[h * d + j], u[h], s);
    out[j] = s;
  }
}
__device__ float sq_norm(const float* x, int n, float* red) {
  float s = 0.f;
  for (int i = threadIdx.x; i < n; i += blockDim.x) s = fmaf(x[i], x[i], s);
  return bsum(s, red);
}

// torch _SpectralNorm: (training) u <- normalize(W v), v <- normalize(W^T u); sigma = u . (W v).
__device__ float spectral_sigma(const float* W, float* u, float* v, float* tvec, float* red, int H, int d, bool training) {
  if (training) {
    matvec(W, v, tvec, H, d);
    __syncthreads();
    float dn = fmaxf(sqrtf(sq_norm(tvec, H, red)), 1e-12f);
    for (int h = threadIdx.x; h < H; h += blockDim.x) u[h] = tvec[h] / dn;
    __syncthreads();
    matvec_t(W, u, tvec, H, d);
    __syncthreads();
    dn = fmaxf(sqrtf(sq_norm(tvec, d, red)), 1e-12f);
    for (int j = threadIdx.x; j < d; j += blockDim.x) v[j] = tvec[j] / dn;
    __syncthreads();
  }
  matvec(W, v, tvec, H, d);
  __syncthreads();
  float s = 0.f;
  for (int h = threadIdx.x; h < H; h += blockDim.x) s = fmaf(u[h], tvec[h], s);
  s = bsum(s, red);
  return s;
}

// Loads rows [b0, b0 + nb) of a pass into X (features) and CO (sample weight w); DF receives the mixing epsilon.
__device__ void load_rows(const GailDims& g, const float* pol, const float* exp_, const float* eps, int kind, int b0, int nb, float* X, float* CO, float* DF) {
  const RowLayout L = row_layout(g.S, g.A);
  for (int idx = threadIdx.x; idx < nb * g.d; idx += blockDim.x) {
    const int b = idx / g.d, j = idx % g.d;
    const int64_t ro = (int64_t)(b0 + b) * g.row + j;  // state | action are adjacent at the row start
    float v;
    if (kind == PASS_POLICY) v = pol[ro];
    else if (kind == PASS_EXPERT) v = exp_[ro];
    else {
      const float e = eps[b0 + b];
      v = __fadd_rn(__fmul_rn(e, exp_[ro]), __fmul_rn(__fsub_rn(1.f, e), pol[ro]));  // training.py:81
    }
    X[b * g.ldx + j] = v;
  }
  for (int b = threadIdx.x; b < nb; b += blockDim.x) {
    const int64_t wo = (int64_t)(b0 + b) * g.row + L.weight;
    float w, e = 0.f;
    if (kind == PASS_POLICY) w = pol[wo];
    else if (kind == PASS_EXPERT) w = exp_[wo];
    else {
      e = eps[b0 + b];
      w = __fadd_rn(__fmul_rn(e, exp_[wo]), __fmul_rn(__fsub_rn(1.f, e), pol[wo]));
    }
    CO[b] = w;
    DF[b] = e;
  }
}

// hidden = relu(W1e x + b1) into Z; logits f into FO (one warp per row).
__device__ void forward_chunk(const GailDims& g, const GailSmem& s, int nb, float b2, float* FO) {
  const int H = g.H, d = g.d;
  for (int p = threadIdx.x; p < nb * H; p += blockDim.x) {
    const int b = p % nb, h = p / nb;
    float z = s.b1[h];
    const float* wr = s.W1e + h * d;
    const float* xr = s.X + b * g.ldx;
    for (int j = 0; j < d; ++j) z = fmaf(wr[j], xr[j], z);
    s.Z[b * g.ldz + h] = fmaxf(z, 0.f);
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  for (int b = warp; b < nb; b += nw) {
    float f = 0.f;
    for (int h = lane; h < H; h += 32) f = fmaf(s.w2e[h], s.Z[b * g.ldz + h], f);
    f = warp_sum(f);
    if (lane == 0) FO[b] = f + b2;
  }
  __syncthreads();
}

template <int NE>
__global__ void __launch_bounds__(THREADS) gail_update_kernel(const GailUpdParams p) {
  extern __shared__ __align__(16) float sm[];
  const GailDims g = p.g;
  GailSmem s;
  gail_carve(g, sm, &s);
  const il_gail_update_args& a = p.a;
  const int r = blockIdx.x, tid = threadIdx.x;
  const int H = g.H, d = g.d, B = g.B;
  float* prm = a.disc.g.params + (int64_t)r * a.disc.g.stride;
  const bool sn = a.disc.u != nullptr;
  const float* pol = a.policy.rows + (int64_t)r * a.policy.replica_stride;
  const float* exp_ = a.expert.rows + (int64_t)r * a.expert.replica_stride;
  const float* eps_gp = a.eps_gp ? a.eps_gp + (int64_t)r * B : nullptr;
  const float* eps_mix = a.eps_mix ? a.eps_mix + (int64_t)r * B : nullptr;
  const float invB = 1.f / (float)B;
  // this replica's hyperparameters (per-replica arrays, else the scalars); the gradient-penalty pass runs where grad_penalty > 0
  const float grad_penalty = a.grad_penalty_r ? a.grad_penalty_r[r] : a.grad_penalty, entropy_bonus = a.entropy_bonus_r ? a.entropy_bonus_r[r] : a.entropy_bonus;
  const double lr = a.opt.lr_r ? a.opt.lr_r[r] : a.opt.lr, wd = a.opt.weight_decay_r ? a.opt.weight_decay_r[r] : a.opt.weight_decay;

  // ---- load parameters / buffers -------------------------------------------------------------------------
  for (int i = tid; i < H * d; i += THREADS) { s.W1[i] = prm[p.off_w1 + i]; s.G1[i] = 0.f; }
  for (int h = tid; h < H; h += THREADS) {
    s.b1[h] = prm[p.off_b1 + h]; s.w2[h] = prm[p.off_w2 + h]; s.G2[h] = 0.f; s.gb1[h] = 0.f;
    if (sn) { s.u1[h] = a.disc.u[(int64_t)r * a.disc.u_stride + h]; s.v2[h] = a.disc.v[(int64_t)r * a.disc.v_stride + d + h]; }
  }
  if (sn) for (int j = tid; j < d; j += THREADS) s.v1[j] = a.disc.v[(int64_t)r * a.disc.v_stride + j];
  const float b2 = prm[p.off_b2];
  float u2 = sn ? a.disc.u[(int64_t)r * a.disc.u_stride + H] : 1.f;
  __syncthreads();

  // ---- pass schedule (training.py:94-127): [policy, expert] or [mixup], then the gradient-penalty mix -----
  int kinds[3], n_pass = 0;
  const float* pass_eps[3] = {nullptr, nullptr, nullptr};
  int gp_pass = -1;
  if (a.loss_function == IL_LOSS_MIXUP) { kinds[n_pass] = PASS_MIX; pass_eps[n_pass++] = eps_mix; }
  else { kinds[n_pass++] = PASS_POLICY; kinds[n_pass++] = PASS_EXPERT; }
  if (grad_penalty > 0.f) { gp_pass = n_pass; kinds[n_pass] = PASS_MIX; pass_eps[n_pass++] = eps_gp; }

  // ---- phase 1: one power iteration per layer per train-mode forward; remember (u, v, sigma) of each ------
  const int SF = gail_slot_floats(H, d);
  for (int k = 0; k < n_pass; ++k) {
    float* slot = s.slots + k * SF;
    float sig1 = 1.f, sig2 = 1.f;
    if (sn) {
      sig1 = spectral_sigma(s.W1, s.u1, s.v1, s.tvec, s.red, H, d, a.training != 0);
      // layer 2 is a [1, H] matrix: u2 scalar, v2 [H]
      float t = 0.f;
      if (a.training) {
        for (int h = tid; h < H; h += THREADS) t = fmaf(s.w2[h], s.v2[h], t);
        t = bsum(t, s.red);
        u2 = t / fmaxf(fabsf(t), 1e-12f);
        for (int h = tid; h < H; h += THREADS) s.tvec[h] = s.w2[h] * u2;
        __syncthreads();
        const float dn = fmaxf(sqrtf(sq_norm(s.tvec, H, s.red)), 1e-12f);
        for (int h = tid; h < H; h += THREADS) s.v2[h] = s.tvec[h] / dn;
        __syncthreads();
      }
      t = 0.f;
      for (int h = tid; h < H; h += THREADS) t = fmaf(s.w2[h], s.v2[h], t);
      sig2 = u2 * bsum(t, s.red);
    }
    for (int h = tid; h < H; h += THREADS) { slot[h] = s.u1[h]; slot[H + d + h] = s.v2[h]; }
    for (int j = tid; j < d; j += THREADS) slot[H + j] = s.v1[j];
    if (tid == 0) { slot[2 * H + d] = sig1; slot[2 * H + d + 1] = sig2; slot[2 * H + d + 2] = u2; }
    __syncthreads();
  }

  // ---- phase 2 (PUGAIL only): the clamp of training.py:102 needs the batch scalar before any gradient ------
  float pu_gate = 1.f;
  float loss_bce = 0.f, loss_gp = 0.f;
  if (a.loss_function == IL_LOSS_PUGAIL) {
    float sums[2] = {0.f, 0.f};  // sum w_p softplus(f_p), sum w_e softplus(f_e)
    for (int k = 0; k < 2; ++k) {
      const float* slot = s.slots + k * SF;
      const float sig1 = slot[2 * H + d], sig2 = slot[2 * H + d + 1];
      for (int i = tid; i < H * d; i += THREADS) s.W1e[i] = s.W1[i] / sig1;
      for (int h = tid; h < H; h += THREADS) s.w2e[h] = s.w2[h] / sig2;
      __syncthreads();
      float part = 0.f;
      for (int b0 = 0; b0 < B; b0 += g.RB) {
        const int nb = min(g.RB, B - b0);
        load_rows(g, pol, exp_, nullptr, kinds[k], b0, nb, s.X, s.CO, s.DF);
        __syncthreads();
        forward_chunk(g, s, nb, b2, s.DF);
        for (int b = tid; b < nb; b += THREADS) part += s.CO[b] * softplusf(s.DF[b]);
        __syncthreads();
      }
      sums[k] = bsum(part, s.red);
    }
    const float inner = a.pos_class_prior * (sums[1] * invB) - sums[0] * invB;
    pu_gate = inner >= -a.nonnegative_margin ? 1.f : 0.f;  // torch.clamp(min=) passes gradient where x >= min
  }

  // ---- phase 3: forward + backward per pass, projected through that pass's spectral norm --------------------
  float g1k[NE];
  float gb2 = 0.f;
  for (int k = 0; k < n_pass; ++k) {
    const float* slot = s.slots + k * SF;
    const float sig1 = slot[2 * H + d], sig2 = slot[2 * H + d + 1], u2k = slot[2 * H + d + 2];
    const int kind = kinds[k];
    const bool is_gp = (k == gp_pass);
    for (int i = tid; i < H * d; i += THREADS) s.W1e[i] = s.W1[i] / sig1;
    for (int h = tid; h < H; h += THREADS) { s.w2e[h] = s.w2[h] / sig2; s.G2k[h] = 0.f; s.gb1k[h] = 0.f; }
#pragma unroll
    for (int i = 0; i < NE; ++i) g1k[i] = 0.f;
    float gb2k = 0.f, loss_part = 0.f;
    __syncthreads();
    for (int b0 = 0; b0 < B; b0 += g.RB) {
      const int nb = min(g.RB, B - b0);
      load_rows(g, pol, exp_, pass_eps[k], kind, b0, nb, s.X, s.CO, s.DF);
      __syncthreads();
      if (!is_gp) {
        // DF holds eps (mixup) on entry; forward writes logits into GX[0..nb) scratch first
        forward_chunk(g, s, nb, b2, s.GX);
        for (int b = tid; b < nb; b += THREADS) {
          const float f = s.GX[b], w = s.CO[b], sg = sigmoidf(f);
          float df;
          if (a.loss_function == IL_LOSS_MIXUP) {  // training.py:112
            const float e = s.DF[b];
            df = w * (sg - e) * invB;
            loss_part += e * w * softplusf(-f) + (1.f - e) * w * softplusf(f);
          } else if (a.loss_function == IL_LOSS_BCE) {  // training.py:98-99
            df = kind == PASS_EXPERT ? w * (sg - 1.f) * invB : w * sg * invB;
            loss_part += kind == PASS_EXPERT ? w * softplusf(-f) : w * softplusf(f);
          } else {  // PUGAIL, training.py:101-102
            const float pr = a.pos_class_prior;
            df = kind == PASS_EXPERT ? pr * w * (sg - 1.f) * invB + pu_gate * pr * w * sg * invB : -pu_gate * w * sg * invB;
            loss_part += kind == PASS_EXPERT ? pr * w * softplusf(-f) + pu_gate * pr * w * softplusf(f) : -pu_gate * w * softplusf(f);
          }
          if (entropy_bonus > 0.f) df += entropy_bonus * w * f * sg * (1.f - sg) * invB;  // training.py:130-132
          s.DF[b] = df;
          gb2k += df;
        }
        __syncthreads();
        // dL/dw2e[h] += sum_b df_b hidden[b,h];  dz[b,h] = df_b w2e[h] 1[hidden>0] (in place);  dL/db1[h] += sum_b dz[b,h]
        // all 256 threads: hidden unit h = tid % H, row slice = tid / H of the chunk; partials combined in a fixed order
        {
          const int parts = H <= THREADS ? THREADS / H : 1, hh = tid % H, part = tid / H;
          float acc2 = 0.f, accb = 0.f;
          if (part < parts) {
            const float w2h = s.w2e[hh];
            const int per = (nb + parts - 1) / parts, b_lo = part * per, b_hi = min(nb, b_lo + per);
            for (int b = b_lo; b < b_hi; ++b) {
              const float hv = s.Z[b * g.ldz + hh], df = s.DF[b];
              acc2 = fmaf(df, hv, acc2);
              const float dz = hv > 0.f ? df * w2h : 0.f;
              s.Z[b * g.ldz + hh] = dz;
              accb += dz;
            }
          }
          s.part[tid] = acc2;
          s.part[THREADS + tid] = accb;
          __syncthreads();
          for (int h = tid; h < H; h += THREADS) {
            float a2 = 0.f, ab = 0.f;
            for (int q = 0; q < parts; ++q) { a2 += s.part[q * H + h]; ab += s.part[THREADS + q * H + h]; }
            s.G2k[h] += a2;
            s.gb1k[h] += ab;
          }
        }
        __syncthreads();
        // dL/dW1e[h, j] += sum_b dz[b,h] x[b,j]
#pragma unroll
        for (int i = 0; i < NE; ++i) {
          const int e = tid + i * THREADS;
          if (e < H * d) {
            const int h = e / d, j = e % d;
            float acc = g1k[i];
            for (int b = 0; b < nb; ++b) acc = fmaf(s.Z[b * g.ldz + h], s.X[b * g.ldx + j], acc);
            g1k[i] = acc;
          }
        }
        __syncthreads();
      } else {
        // gradient penalty (training.py:117-127): g_x = W1e^T (m . w2e); loss = mean(lambda w_m |g_x|^2)
        forward_chunk(g, s, nb, b2, s.DF);  // Z = hidden (mask source); logits unused
        for (int q = tid; q < nb * d; q += THREADS) {
          const int b = q / d, j = q % d;
          float acc = 0.f;
          for (int h = 0; h < H; ++h) acc = fmaf(s.Z[b * g.ldz + h] > 0.f ? s.w2e[h] : 0.f, s.W1e[h * d + j], acc);
          s.GX[b * g.ldx + j] = acc;
        }
        __syncthreads();
        for (int b = tid; b < nb; b += THREADS) {
          float pen = 0.f;
          for (int j = 0; j < d; ++j) pen = fmaf(s.GX[b * g.ldx + j], s.GX[b * g.ldx + j], pen);
          const float wm = s.CO[b];
          loss_part += grad_penalty * wm * pen;
          s.DF[b] = 2.f * grad_penalty * wm * invB;  // coef_b
        }
        __syncthreads();
        // dL/dw2e[h] += sum_b coef_b m[b,h] (W1e g_b)[h]
        {
          const int parts = H <= THREADS ? THREADS / H : 1, hh = tid % H, part = tid / H;
          float acc2 = 0.f;
          if (part < parts) {
            const float* wr = s.W1e + hh * d;
            const int per = (nb + parts - 1) / parts, b_lo = part * per, b_hi = min(nb, b_lo + per);
            for (int b = b_lo; b < b_hi; ++b) {
              if (s.Z[b * g.ldz + hh] > 0.f) {
                float t = 0.f;
                for (int j = 0; j < d; ++j) t = fmaf(wr[j], s.GX[b * g.ldx + j], t);
                acc2 = fmaf(s.DF[b], t, acc2);
              }
            }
          }
          s.part[tid] = acc2;
          __syncthreads();
          for (int h = tid; h < H; h += THREADS) {
            float a2 = 0.f;
            for (int q = 0; q < parts; ++q) a2 += s.part[q * H + h];
            s.G2k[h] += a2;
          }
        }
        // dL/dW1e[h, j] += sum_b coef_b (m[b,h] w2e[h]) g_b[j]
#pragma unroll
        for (int i = 0; i < NE; ++i) {
          const int e = tid + i * THREADS;
          if (e < H * d) {
            const int h = e / d, j = e % d;
            const float w2h = s.w2e[h];
            float acc = g1k[i];
            for (int b = 0; b < nb; ++b) acc = fmaf(s.Z[b * g.ldz + h] > 0.f ? s.DF[b] * w2h : 0.f, s.GX[b * g.ldx + j], acc);
            g1k[i] = acc;
          }
        }
        __syncthreads();
      }
    }
    // ---- spectral-norm backward: dL/dW = (G - <G, W_eff> u v^T) / sigma (SURVEY §8a a12), accumulate over passes
    float inner1 = 0.f, inner2 = 0.f;
    if (sn) {
#pragma unroll
      for (int i = 0; i < NE; ++i) {
        const int e = tid + i * THREADS;
        if (e < H * d) inner1 = fmaf(g1k[i], s.W1e[e], inner1);
      }
      inner1 = bsum(inner1, s.red);
      for (int h = tid; h < H; h += THREADS) inner2 = fmaf(s.G2k[h], s.w2e[h], inner2);
      inner2 = bsum(inner2, s.red);
    }
#pragma unroll
    for (int i = 0; i < NE; ++i) {
      const int e = tid + i * THREADS;
      if (e < H * d) {
        const int h = e / d, j = e % d;
        s.G1[e] += sn ? (g1k[i] - inner1 * slot[h] * slot[H + j]) / sig1 : g1k[i];
      }
    }
    for (int h = tid; h < H; h += THREADS) {
      s.G2[h] += sn ? (s.G2k[h] - inner2 * u2k * slot[H + d + h]) / sig2 : s.G2k[h];
      s.gb1[h] += s.gb1k[h];
    }
    gb2k = bsum(gb2k, s.red);
    gb2 += gb2k;
    loss_part = bsum(loss_part, s.red);
    if (is_gp) loss_gp = loss_part * invB; else loss_bce += loss_part * invB;
    __syncthreads();
  }
  if (tid == 0 && a.out_losses) { a.out_losses[r * 2 + 0] = loss_bce; a.out_losses[r * 2 + 1] = loss_gp; }

  // ---- AdamW (train.py:84; torch _single_tensor_adam) -----------------------------------------------------------
  if (tid == 0) {
    const double t = (double)*a.opt.step;
    s.scal[0] = (float)(lr / (1.0 - pow(a.opt.beta1, t)));
    s.scal[1] = (float)sqrt(1.0 - pow(a.opt.beta2, t));
  }
  __syncthreads();
  const float step_size = s.scal[0], bc2_sqrt = s.scal[1];
  const float decay = (float)(1.0 - lr * wd), w1 = (float)(1.0 - a.opt.beta1), w2c = (float)(1.0 - a.opt.beta2), beta2 = (float)a.opt.beta2,
              eps = (float)a.opt.eps;
  const bool has_wd = wd != 0.0;
  float* am = a.opt.m + (int64_t)r * a.disc.g.stride;
  float* avv = a.opt.v + (int64_t)r * a.disc.g.stride;
  auto adam = [&](int64_t off, float grad) {
    float pi = prm[off], mi = am[off], vi = avv[off];
    if (has_wd) pi = __fmul_rn(pi, decay);
    mi = __fadd_rn(mi, __fmul_rn(w1, __fsub_rn(grad, mi)));
    vi = __fadd_rn(__fmul_rn(vi, beta2), __fmul_rn(__fmul_rn(w2c, grad), grad));
    const float denom = __fadd_rn(__fdiv_rn(sqrtf(vi), bc2_sqrt), eps);
    pi = __fadd_rn(pi, __fmul_rn(-step_size, __fdiv_rn(mi, denom)));
    prm[off] = pi; am[off] = mi; avv[off] = vi;
  };
  for (int i = tid; i < H * d; i += THREADS) adam(p.off_w1 + i, s.G1[i]);
  for (int h = tid; h < H; h += THREADS) { adam(p.off_b1 + h, s.gb1[h]); adam(p.off_w2 + h, s.G2[h]); }
  if (tid == 0) adam(p.off_b2, gb2);
  if (sn) {  // persist the power-iteration state (in-place buffers of the parametrization)
    for (int h = tid; h < H; h += THREADS) { a.disc.u[(int64_t)r * a.disc.u_stride + h] = s.u1[h]; a.disc.v[(int64_t)r * a.disc.v_stride + d + h] = s.v2[h]; }
    for (int j = tid; j < d; j += THREADS) a.disc.v[(int64_t)r * a.disc.v_stride + j] = s.v1[j];
    if (tid == 0) a.disc.u[(int64_t)r * a.disc.u_stride + H] = u2;
  }
}


// ---- register-tiled variant of the update (d <= 32, H in {32, 64, 128}) -------------------------------------------------------------
// Same mathematics and phase order as gail_update_kernel; the three GEMM-shaped inner loops per pass run on 4 x 4 register tiles
// with 128-bit shared-memory operand loads (the first kernel issues two shared loads per FMA and is bound by the shared-memory pipe:
// 0.77 ms at R = 1024 = 3.9 TFLOP/s). Chunk of RB rows resident in shared memory; 2 CTAs per SM.
struct TSmem {
  float *W1, *G1, *W1e, *W1eT, *G1k, *b1, *w2, *w2e, *G2, *gb1, *G2k, *gb1k, *u1, *v1, *v2, *tvec, *slots, *X, *Z, *GX, *F, *DF, *CO, *red, *scal, *part;
};
struct TDims { int S, A, d, DP, H, B, row, RB, LDZ, HD; };
__host__ __device__ inline int64_t tiled_carve(const TDims& g, float* base, TSmem* s) {
  int64_t o = 0;
  auto take = [&](int n) { float* p = base ? base + o : nullptr; o += (n + 3) / 4 * 4; return p; };
  TSmem t;
  t.W1 = take(g.HD); t.G1 = take(g.HD); t.W1e = take(g.H * g.DP); t.W1eT = take(g.DP * g.H); t.G1k = take(g.H * g.DP);
  t.b1 = take(g.H); t.w2 = take(g.H); t.w2e = take(g.H); t.G2 = take(g.H); t.gb1 = take(g.H); t.G2k = take(g.H); t.gb1k = take(g.H);
  t.u1 = take(g.H); t.v1 = take(g.d); t.v2 = take(g.H); t.tvec = take(g.H > g.d ? g.H : g.d);
  t.slots = take(3 * gail_slot_floats(g.H, g.d));
  t.X = take(g.RB * g.DP); t.Z = take(g.RB * g.LDZ); t.GX = take(g.RB * g.DP);
  t.F = take(g.RB); t.DF = take(g.RB); t.CO = take(g.RB);
  t.red = take(32); t.scal = take(32); t.part = take(4 * THREADS);
  if (s) *s = t;
  return o * 4;
}
struct GailTiledParams {
  il_gail_update_args a;
  TDims g;
  int64_t off_w1, off_b1, off_w2, off_b2;
};

// Loads rows [b0, b0 + nb) into X [RB][DP] (zero padded columns / rows); CO = sample weight, DF = mixing epsilon.
__device__ void tiled_load_rows(const TDims& g, const float* pol, const float* exp_, const float* eps, int kind, int b0, int nb, float* X, float* CO, float* DF) {
  const RowLayout L = row_layout(g.S, g.A);
  const int nq = g.DP >> 2;  // 128-bit chunks per row (packed rows are 16-byte aligned with a stride that is a multiple of 4 floats)
  for (int idx = threadIdx.x; idx < g.RB * nq; idx += blockDim.x) {
    const int b = idx / nq, q = idx % nq;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (b < nb) {
      const int64_t ro = (int64_t)(b0 + b) * g.row + 4 * q;
      if (kind == PASS_POLICY) v = __ldg(reinterpret_cast<const float4*>(pol + ro));
      else if (kind == PASS_EXPERT) v = __ldg(reinterpret_cast<const float4*>(exp_ + ro));
      else {
        const float e = __ldg(eps + b0 + b), f = __fsub_rn(1.f, e);
        const float4 x = __ldg(reinterpret_cast<const float4*>(exp_ + ro)), y = __ldg(reinterpret_cast<const float4*>(pol + ro));
        v = make_float4(__fadd_rn(__fmul_rn(e, x.x), __fmul_rn(f, y.x)), __fadd_rn(__fmul_rn(e, x.y), __fmul_rn(f, y.y)), __fadd_rn(__fmul_rn(e, x.z), __fmul_rn(f, y.z)),
                        __fadd_rn(__fmul_rn(e, x.w), __fmul_rn(f, y.w)));
      }
      const int j = 4 * q;  // columns beyond d (the rest of the packed row) are not discriminator inputs
      if (j + 1 >= g.d) v.y = 0.f;
      if (j + 2 >= g.d) v.z = 0.f;
      if (j + 3 >= g.d) v.w = 0.f;
      if (j >= g.d) v.x = 0.f;
    }
    *reinterpret_cast<float4*>(X + b * g.DP + 4 * q) = v;
  }
  for (int b = threadIdx.x; b < g.RB; b += blockDim.x) {
    float w = 0.f, e = 0.f;
    if (b < nb) {
      const int64_t wo = (int64_t)(b0 + b) * g.row + L.weight;
      if (kind == PASS_POLICY) w = pol[wo];
      else if (kind == PASS_EXPERT) w = exp_[wo];
      else {
        e = eps[b0 + b];
        w = __fadd_rn(__fmul_rn(e, exp_[wo]), __fmul_rn(__fsub_rn(1.f, e), pol[wo]));
      }
    }
    CO[b] = w;
    DF[b] = e;
  }
}

// acc[4 b][4 h] = bias[h] + sum_j IN[b][j] * WT[j][h] on 4 x 4 register tiles, handed to `epi(tb, th, acc)`; lanes run over the h-tiles
// (operand rows broadcast). Tile t = tid + m * 256 keeps th = t % (H / 4) fixed per thread (256 is a multiple of H / 4).
template <typename Epi>
__device__ __forceinline__ void tiled_rows_times_wt(const TDims& g, const float* IN, const float* WT, const float* bias, Epi epi) {
  const int nth = g.H >> 2, ntb = g.RB >> 2;
  for (int t = threadIdx.x; t < nth * ntb; t += blockDim.x) {
    const int th = t % nth, tb = t / nth;
    float acc[4][4];
    const float4 bv = bias ? *reinterpret_cast<const float4*>(bias + 4 * th) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int i = 0; i < 4; ++i) { acc[i][0] = bv.x; acc[i][1] = bv.y; acc[i][2] = bv.z; acc[i][3] = bv.w; }
    const float* xr = IN + (4 * tb) * g.DP;
    for (int j4 = 0; j4 < g.DP; j4 += 4) {
      float4 x[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) x[i] = *reinterpret_cast<const float4*>(xr + i * g.DP + j4);
#pragma unroll
      for (int jj = 0; jj < 4; ++jj) {
        const float4 w = *reinterpret_cast<const float4*>(WT + (j4 + jj) * g.H + 4 * th);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float xv = jj == 0 ? x[i].x : (jj == 1 ? x[i].y : (jj == 2 ? x[i].z : x[i].w));
          acc[i][0] = fmaf(xv, w.x, acc[i][0]); acc[i][1] = fmaf(xv, w.y, acc[i][1]); acc[i][2] = fmaf(xv, w.z, acc[i][2]); acc[i][3] = fmaf(xv, w.w, acc[i][3]);
        }
      }
    }
    epi(tb, th, acc);
  }
}
// hidden = relu(W1e x + b1) stored to Z [RB][LDZ]
__device__ __forceinline__ void tiled_hidden(const TDims& g, const float* X, const float* W1eT, const float* b1, float* Z) {
  tiled_rows_times_wt(g, X, W1eT, b1, [&](int tb, int th, float (&acc)[4][4]) {
#pragma unroll
    for (int i = 0; i < 4; ++i)
      *reinterpret_cast<float4*>(Z + (4 * tb + i) * g.LDZ + 4 * th) = make_float4(fmaxf(acc[i][0], 0.f), fmaxf(acc[i][1], 0.f), fmaxf(acc[i][2], 0.f), fmaxf(acc[i][3], 0.f));
  });
}

// The same, plus the logit of every row FO[b] = w2e . hidden[b] + b2 from the tiles in registers: each thread dots its 4 hidden units with w2e, the
// H / 4 lanes that share a row block reduce with xor shuffles (the tile loop's trip count is warp-uniform: H / 4 * RB / 4 is a multiple of 32).
__device__ __forceinline__ void tiled_hidden_logits(const TDims& g, const float* X, const float* W1eT, const float* b1, float* Z, const float* w2e, float b2, float* FO) {
  const int nth = g.H >> 2;
  tiled_rows_times_wt(g, X, W1eT, b1, [&](int tb, int th, float (&acc)[4][4]) {
    const float4 w = *reinterpret_cast<const float4*>(w2e + 4 * th);
    float f[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float4 z = make_float4(fmaxf(acc[i][0], 0.f), fmaxf(acc[i][1], 0.f), fmaxf(acc[i][2], 0.f), fmaxf(acc[i][3], 0.f));
      *reinterpret_cast<float4*>(Z + (4 * tb + i) * g.LDZ + 4 * th) = z;
      f[i] = fmaf(z.w, w.w, fmaf(z.z, w.z, fmaf(z.y, w.y, z.x * w.x)));
    }
    for (int o = nth >> 1; o > 0; o >>= 1) {
#pragma unroll
      for (int i = 0; i < 4; ++i) f[i] += __shfl_xor_sync(0xffffffffu, f[i], o);
    }
    if (th == 0) *reinterpret_cast<float4*>(FO + 4 * tb) = make_float4(f[0] + b2, f[1] + b2, f[2] + b2, f[3] + b2);
  });
}
// acc[4 h][4 j] += sum over this thread's rows of  DZ(b, 4 th + k) * IN[b][4 tj + c]   (weight-gradient shape [H][DP], K = rows split 4 ways
// over lane groups: lane = th_low + 8 * ks). DZ(b, h) is produced by `dz` from Z / per-row coefficients.
// Slot q of a thread covers tile (warp * 8 + lane % 8) + 64 q; ks = (lane / 8) is the row group.
struct TileMap { int th, tj, active; };
__device__ __forceinline__ TileMap tiled_wgrad_map(const TDims& g, int q) {
  TileMap m;
  const int nth = g.H >> 2, ntj = g.DP >> 2;
  const int tile = (threadIdx.x >> 5) * 8 + (threadIdx.x & 7) + 64 * q;
  m.active = tile < nth * ntj;
  const int tc = m.active ? tile : 0;
  m.th = tc % nth; m.tj = tc / nth;
  return m;
}

template <int NT>
__global__ void __launch_bounds__(THREADS, 2) gail_update_tiled_kernel(const GailTiledParams p) {
  extern __shared__ __align__(16) float sm[];
  const TDims g = p.g;
  TSmem s;
  tiled_carve(g, sm, &s);
  const il_gail_update_args& a = p.a;
  const int r = blockIdx.x, tid = threadIdx.x;
  const int H = g.H, d = g.d, B = g.B, DP = g.DP, LDZ = g.LDZ;
  float* prm = a.disc.g.params + (int64_t)r * a.disc.g.stride;
  const bool sn = a.disc.u != nullptr;
  const float* pol = a.policy.rows + (int64_t)r * a.policy.replica_stride;
  const float* exp_ = a.expert.rows + (int64_t)r * a.expert.replica_stride;
  const float* eps_gp = a.eps_gp ? a.eps_gp + (int64_t)r * B : nullptr;
  const float* eps_mix = a.eps_mix ? a.eps_mix + (int64_t)r * B : nullptr;
  const float invB = 1.f / (float)B;
  // this replica's hyperparameters (per-replica arrays, else the scalars); the gradient-penalty pass runs where grad_penalty > 0
  const float grad_penalty = a.grad_penalty_r ? a.grad_penalty_r[r] : a.grad_penalty, entropy_bonus = a.entropy_bonus_r ? a.entropy_bonus_r[r] : a.entropy_bonus;
  const double lr = a.opt.lr_r ? a.opt.lr_r[r] : a.opt.lr, wd = a.opt.weight_decay_r ? a.opt.weight_decay_r[r] : a.opt.weight_decay;

  for (int i = tid; i < H * d; i += THREADS) { s.W1[i] = prm[p.off_w1 + i]; s.G1[i] = 0.f; }
  for (int h = tid; h < H; h += THREADS) {
    s.b1[h] = prm[p.off_b1 + h]; s.w2[h] = prm[p.off_w2 + h]; s.G2[h] = 0.f; s.gb1[h] = 0.f;
    if (sn) { s.u1[h] = a.disc.u[(int64_t)r * a.disc.u_stride + h]; s.v2[h] = a.disc.v[(int64_t)r * a.disc.v_stride + d + h]; }
  }
  if (sn) for (int j = tid; j < d; j += THREADS) s.v1[j] = a.disc.v[(int64_t)r * a.disc.v_stride + j];
  const float b2 = prm[p.off_b2];
  float u2 = sn ? a.disc.u[(int64_t)r * a.disc.u_stride + H] : 1.f;
  __syncthreads();

  int kinds[3], n_pass = 0;
  const float* pass_eps[3] = {nullptr, nullptr, nullptr};
  int gp_pass = -1;
  if (a.loss_function == IL_LOSS_MIXUP) { kinds[n_pass] = PASS_MIX; pass_eps[n_pass++] = eps_mix; }
  else { kinds[n_pass++] = PASS_POLICY; kinds[n_pass++] = PASS_EXPERT; }
  if (grad_penalty > 0.f) { gp_pass = n_pass; kinds[n_pass] = PASS_MIX; pass_eps[n_pass++] = eps_gp; }

  // ---- phase 1: power iterations (identical to gail_update_kernel) -------------------------------------------------------------
  const int SF = gail_slot_floats(H, d);
  for (int k = 0; k < n_pass; ++k) {
    float* slot = s.slots + k * SF;
    float sig1 = 1.f, sig2 = 1.f;
    if (sn) {
      sig1 = spectral_sigma(s.W1, s.u1, s.v1, s.tvec, s.red, H, d, a.training != 0);
      float t = 0.f;
      if (a.training) {
        for (int h = tid; h < H; h += THREADS) t = fmaf(s.w2[h], s.v2[h], t);
        t = bsum(t, s.red);
        u2 = t / fmaxf(fabsf(t), 1e-12f);
        for (int h = tid; h < H; h += THREADS) s.tvec[h] = s.w2[h] * u2;
        __syncthreads();
        const float dn = fmaxf(sqrtf(sq_norm(s.tvec, H, s.red)), 1e-12f);
        for (int h = tid; h < H; h += THREADS) s.v2[h] = s.tvec[h] / dn;
        __syncthreads();
      }
      t = 0.f;
      for (int h = tid; h < H; h += THREADS) t = fmaf(s.w2[h], s.v2[h], t);
      sig2 = u2 * bsum(t, s.red);
    }
    for (int h = tid; h < H; h += THREADS) { slot[h] = s.u1[h]; slot[H + d + h] = s.v2[h]; }
    for (int j = tid; j < d; j += THREADS) slot[H + j] = s.v1[j];
    if (tid == 0) { slot[2 * H + d] = sig1; slot[2 * H + d + 1] = sig2; slot[2 * H + d + 2] = u2; }
    __syncthreads();
  }

  auto set_effective = [&](const float* slot) {  // W1e [H][DP] and its transpose [DP][H], zero padded; w2e
    const float sig1 = slot[2 * H + d], sig2 = slot[2 * H + d + 1];
    for (int i = tid; i < H * DP; i += THREADS) {
      const int h = i / DP, j = i % DP;
      const float v = j < d ? s.W1[h * d + j] / sig1 : 0.f;
      s.W1e[i] = v;
      s.W1eT[j * H + h] = v;
    }
    for (int h = tid; h < H; h += THREADS) s.w2e[h] = s.w2[h] / sig2;
  };
  // ---- phase 2 (PUGAIL): batch scalar of the clamp ---------------------------------------------------------------------------------
  float pu_gate = 1.f, loss_bce = 0.f, loss_gp = 0.f;
  if (a.loss_function == IL_LOSS_PUGAIL) {
    float sums[2] = {0.f, 0.f};
    for (int k = 0; k < 2; ++k) {
      set_effective(s.slots + k * SF);
      __syncthreads();
      float part = 0.f;
      for (int b0 = 0; b0 < B; b0 += g.RB) {
        const int nb = min(g.RB, B - b0);
        tiled_load_rows(g, pol, exp_, nullptr, kinds[k], b0, nb, s.X, s.CO, s.DF);
        __syncthreads();
        tiled_hidden_logits(g, s.X, s.W1eT, s.b1, s.Z, s.w2e, b2, s.F);
        __syncthreads();
        for (int b = tid; b < nb; b += THREADS) part += s.CO[b] * softplusf(s.F[b]);
        __syncthreads();
      }
      sums[k] = bsum(part, s.red);
    }
    pu_gate = (a.pos_class_prior * (sums[1] * invB) - sums[0] * invB) >= -a.nonnegative_margin ? 1.f : 0.f;
  }

  // ---- phase 3: forward + backward per pass ---------------------------------------------------------------------------------------
  TileMap wm[NT];
#pragma unroll
  for (int q = 0; q < NT; ++q) wm[q] = tiled_wgrad_map(g, q);
  const int wks = (tid >> 3) & 3;  // row group of this lane in the weight-gradient tiles
  const int parts = THREADS / H, hh = tid % H, part = tid / H;  // column-sum helpers: hidden unit hh, row slice `part`
  float gb2 = 0.f;
  for (int k = 0; k < n_pass; ++k) {
    const float* slot = s.slots + k * SF;
    const float sig1 = slot[2 * H + d], sig2 = slot[2 * H + d + 1], u2k = slot[2 * H + d + 2];
    const int kind = kinds[k];
    const bool is_gp = (k == gp_pass);
    set_effective(slot);
    for (int h = tid; h < H; h += THREADS) { s.G2k[h] = 0.f; s.gb1k[h] = 0.f; }
    float wacc[NT][4][4];  // this thread's tiles of dL/dW1e, summed over its rows of every chunk
#pragma unroll
    for (int q = 0; q < NT; ++q)
#pragma unroll
      for (int i = 0; i < 4; ++i) wacc[q][i][0] = wacc[q][i][1] = wacc[q][i][2] = wacc[q][i][3] = 0.f;
    float gb2k = 0.f, loss_part = 0.f;
    __syncthreads();
    float4 w2t[NT];
#pragma unroll
    for (int q = 0; q < NT; ++q) w2t[q] = *reinterpret_cast<const float4*>(s.w2e + 4 * wm[q].th);
    // wacc[q] += sum over this lane's rows of  (coef_b * 1[hidden > 0] * w2e)[b, 4 th + i] * IN[b][4 tj + c]
    auto wgrad = [&](const float* IN, int nb) {
#pragma unroll
      for (int q = 0; q < NT; ++q) {
        if (!wm[q].active) continue;
        for (int b = wks; b < nb; b += 4) {
          const float4 z = *reinterpret_cast<const float4*>(s.Z + b * LDZ + 4 * wm[q].th);
          const float4 x = *reinterpret_cast<const float4*>(IN + b * DP + 4 * wm[q].tj);
          const float cf = s.DF[b];
          const float dz[4] = {z.x > 0.f ? cf * w2t[q].x : 0.f, z.y > 0.f ? cf * w2t[q].y : 0.f, z.z > 0.f ? cf * w2t[q].z : 0.f, z.w > 0.f ? cf * w2t[q].w : 0.f};
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            wacc[q][i][0] = fmaf(dz[i], x.x, wacc[q][i][0]); wacc[q][i][1] = fmaf(dz[i], x.y, wacc[q][i][1]);
            wacc[q][i][2] = fmaf(dz[i], x.z, wacc[q][i][2]); wacc[q][i][3] = fmaf(dz[i], x.w, wacc[q][i][3]);
          }
        }
      }
    };
    for (int b0 = 0; b0 < B; b0 += g.RB) {
      const int nb = min(g.RB, B - b0);
      tiled_load_rows(g, pol, exp_, pass_eps[k], kind, b0, nb, s.X, s.CO, s.DF);
      __syncthreads();
      if (is_gp) tiled_hidden(g, s.X, s.W1eT, s.b1, s.Z);  // hidden = relu(W1e x + b1)
      else tiled_hidden_logits(g, s.X, s.W1eT, s.b1, s.Z, s.w2e, b2, s.F);  // + logits
      __syncthreads();
      if (!is_gp) {
        for (int b = tid; b < g.RB; b += THREADS) {
          float df = 0.f;
          if (b < nb) {
            const float f = s.F[b], w = s.CO[b], sg = sigmoidf(f);
            if (a.loss_function == IL_LOSS_MIXUP) {
              const float e = s.DF[b];
              df = w * (sg - e) * invB;
              loss_part += e * w * softplusf(-f) + (1.f - e) * w * softplusf(f);
            } else if (a.loss_function == IL_LOSS_BCE) {
              df = kind == PASS_EXPERT ? w * (sg - 1.f) * invB : w * sg * invB;
              loss_part += kind == PASS_EXPERT ? w * softplusf(-f) : w * softplusf(f);
            } else {
              const float pr = a.pos_class_prior;
              df = kind == PASS_EXPERT ? pr * w * (sg - 1.f) * invB + pu_gate * pr * w * sg * invB : -pu_gate * w * sg * invB;
              loss_part += kind == PASS_EXPERT ? pr * w * softplusf(-f) + pu_gate * pr * w * softplusf(f) : -pu_gate * w * softplusf(f);
            }
            if (entropy_bonus > 0.f) df += entropy_bonus * w * f * sg * (1.f - sg) * invB;
            gb2k += df;
          }
          s.DF[b] = df;  // padded rows: 0
        }
        __syncthreads();
        // dL/dw2e[h] += sum_b df_b hidden[b,h];  dL/db1[h] += sum_b dz[b,h], dz = df_b w2e[h] 1[hidden > 0]
        {
          float acc2 = 0.f, accb = 0.f;
          if (part < parts) {
            const float w2h = s.w2e[hh];
            const int per = (nb + parts - 1) / parts, b_lo = part * per, b_hi = min(nb, b_lo + per);
            for (int b = b_lo; b < b_hi; ++b) {
              const float hv = s.Z[b * LDZ + hh], df = s.DF[b];
              acc2 = fmaf(df, hv, acc2);
              accb += hv > 0.f ? df * w2h : 0.f;
            }
          }
          s.part[tid] = acc2;
          s.part[THREADS + tid] = accb;
          __syncthreads();
          for (int h = tid; h < H; h += THREADS) {
            float a2 = 0.f, ab = 0.f;
            for (int q = 0; q < parts; ++q) { a2 += s.part[q * H + h]; ab += s.part[THREADS + q * H + h]; }
            s.G2k[h] += a2;
            s.gb1k[h] += ab;
          }
        }
        wgrad(s.X, nb);  // dL/dW1e[h, j] += sum_b dz[b,h] x[b,j]   (dz formed on the fly from the hidden tile)
        __syncthreads();
      } else {
        // gradient penalty: g_x[b][j] = sum_h q[b][h] W1e[h][j], q = 1[hidden > 0] w2e[h]; 4 x 4 tiles, h split over 4 lane groups
        {
          const int ntj = DP >> 2, ntiles = (g.RB >> 2) * ntj, l8 = tid & 7, ks = (tid >> 3) & 3;
          for (int base = (tid >> 5) * 8; base < ntiles; base += (THREADS / 32) * 8) {  // warp-uniform trip count (full-mask shuffles inside)
            const bool valid = base + l8 < ntiles;
            const int tile = valid ? base + l8 : 0, tj = tile % ntj, tb = tile / ntj;
            float acc[4][4];
#pragma unroll
            for (int i = 0; i < 4; ++i) acc[i][0] = acc[i][1] = acc[i][2] = acc[i][3] = 0.f;
            for (int h = ks; h < H; h += 4) {
              const float4 w = *reinterpret_cast<const float4*>(s.W1e + h * DP + 4 * tj);
              const float w2h = s.w2e[h];
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                const float q = s.Z[(4 * tb + i) * LDZ + h] > 0.f ? w2h : 0.f;
                acc[i][0] = fmaf(q, w.x, acc[i][0]); acc[i][1] = fmaf(q, w.y, acc[i][1]); acc[i][2] = fmaf(q, w.z, acc[i][2]); acc[i][3] = fmaf(q, w.w, acc[i][3]);
              }
            }
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
              for (int c = 0; c < 4; ++c) {
                float v = acc[i][c];
                v += __shfl_xor_sync(0xffffffffu, v, 8);
                v += __shfl_xor_sync(0xffffffffu, v, 16);
                acc[i][c] = v;
              }
            if (valid && ks == 0) {
#pragma unroll
              for (int i = 0; i < 4; ++i) *reinterpret_cast<float4*>(s.GX + (4 * tb + i) * DP + 4 * tj) = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
            }
          }
        }
        __syncthreads();
        for (int b = tid; b < g.RB; b += THREADS) {
          float coef = 0.f;
          if (b < nb) {
            float pen = 0.f;
            for (int j = 0; j < d; ++j) pen = fmaf(s.GX[b * DP + j], s.GX[b * DP + j], pen);
            const float wmix = s.CO[b];
            loss_part += grad_penalty * wmix * pen;
            coef = 2.f * grad_penalty * wmix * invB;
          }
          s.DF[b] = coef;
        }
        __syncthreads();
        // dL/dw2e[h] += sum_b coef_b m[b,h] (W1e g_b)[h]: the product is formed tile by tile and reduced in registers (th is fixed per thread)
        {
          float a2[4] = {0.f, 0.f, 0.f, 0.f};
          tiled_rows_times_wt(g, s.GX, s.W1eT, nullptr, [&](int tb, int th, float (&acc)[4][4]) {
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const float4 z = *reinterpret_cast<const float4*>(s.Z + (4 * tb + i) * LDZ + 4 * th);
              const float cf = s.DF[4 * tb + i];  // 0 on padded rows
              a2[0] = fmaf(z.x > 0.f ? cf : 0.f, acc[i][0], a2[0]); a2[1] = fmaf(z.y > 0.f ? cf : 0.f, acc[i][1], a2[1]);
              a2[2] = fmaf(z.z > 0.f ? cf : 0.f, acc[i][2], a2[2]); a2[3] = fmaf(z.w > 0.f ? cf : 0.f, acc[i][3], a2[3]);
            }
          });
          *reinterpret_cast<float4*>(s.part + 4 * tid) = make_float4(a2[0], a2[1], a2[2], a2[3]);
          __syncthreads();
          const int nth = H >> 2;
          for (int h = tid; h < H; h += THREADS) {
            float t2 = 0.f;
            for (int q = h >> 2; q < THREADS; q += nth) t2 += s.part[4 * q + (h & 3)];  // threads whose tile column block is h / 4
            s.G2k[h] += t2;
          }
          __syncthreads();
        }
        wgrad(s.GX, nb);  // dL/dW1e[h, j] += sum_b coef_b (m[b,h] w2e[h]) g_b[j]
        __syncthreads();
      }
    }
    // gather the weight-gradient tiles: sum over the 4 row groups, then G1k [H][DP] in shared memory
#pragma unroll
    for (int q = 0; q < NT; ++q) {
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          float v = wacc[q][i][c];
          v += __shfl_xor_sync(0xffffffffu, v, 8);
          v += __shfl_xor_sync(0xffffffffu, v, 16);
          wacc[q][i][c] = v;
        }
      if (wm[q].active && wks == 0) {
#pragma unroll
        for (int i = 0; i < 4; ++i) *reinterpret_cast<float4*>(s.G1k + (4 * wm[q].th + i) * DP + 4 * wm[q].tj) = make_float4(wacc[q][i][0], wacc[q][i][1], wacc[q][i][2], wacc[q][i][3]);
      }
    }
    __syncthreads();
    // ---- spectral-norm backward: dL/dW = (G - <G, W_eff> u v^T) / sigma, accumulated over the passes
    float inner1 = 0.f, inner2 = 0.f;
    if (sn) {
      for (int e = tid; e < H * d; e += THREADS) inner1 = fmaf(s.G1k[(e / d) * DP + e % d], s.W1e[(e / d) * DP + e % d], inner1);
      inner1 = bsum(inner1, s.red);
      for (int h = tid; h < H; h += THREADS) inner2 = fmaf(s.G2k[h], s.w2e[h], inner2);
      inner2 = bsum(inner2, s.red);
    }
    for (int e = tid; e < H * d; e += THREADS) {
      const int h = e / d, j = e % d;
      const float gk = s.G1k[h * DP + j];
      s.G1[e] += sn ? (gk - inner1 * slot[h] * slot[H + j]) / sig1 : gk;
    }
    for (int h = tid; h < H; h += THREADS) {
      s.G2[h] += sn ? (s.G2k[h] - inner2 * u2k * slot[H + d + h]) / sig2 : s.G2k[h];
      s.gb1[h] += s.gb1k[h];
    }
    gb2k = bsum(gb2k, s.red);
    gb2 += gb2k;
    loss_part = bsum(loss_part, s.red);
    if (is_gp) loss_gp = loss_part * invB; else loss_bce += loss_part * invB;
    __syncthreads();
  }
  if (tid == 0 && a.out_losses) { a.out_losses[r * 2 + 0] = loss_bce; a.out_losses[r * 2 + 1] = loss_gp; }

  // ---- AdamW (train.py:84; torch _single_tensor_adam) -----------------------------------------------------------
  if (tid == 0) {
    const double t = (double)*a.opt.step;
    s.scal[0] = (float)(lr / (1.0 - pow(a.opt.beta1, t)));
    s.scal[1] = (float)sqrt(1.0 - pow(a.opt.beta2, t));
  }
  __syncthreads();
  const float step_size = s.scal[0], bc2_sqrt = s.scal[1];
  const float decay = (float)(1.0 - lr * wd), w1c = (float)(1.0 - a.opt.beta1), w2c = (float)(1.0 - a.opt.beta2), beta2 = (float)a.opt.beta2,
              eps = (float)a.opt.eps;
  const bool has_wd = wd != 0.0;
  float* am = a.opt.m + (int64_t)r * a.disc.g.stride;
  float* avv = a.opt.v + (int64_t)r * a.disc.g.stride;
  auto adam = [&](int64_t off, float grad) {
    float pi = prm[off], mi = am[off], vi = avv[off];
    if (has_wd) pi = __fmul_rn(pi, decay);
    mi = __fadd_rn(mi, __fmul_rn(w1c, __fsub_rn(grad, mi)));
    vi = __fadd_rn(__fmul_rn(vi, beta2), __fmul_rn(__fmul_rn(w2c, grad), grad));
    const float denom = __fadd_rn(__fdiv_rn(sqrtf(vi), bc2_sqrt), eps);
    pi = __fadd_rn(pi, __fmul_rn(-step_size, __fdiv_rn(mi, denom)));
    prm[off] = pi; am[off] = mi; avv[off] = vi;
  };
  for (int i = tid; i < H * d; i += THREADS) adam(p.off_w1 + i, s.G1[i]);
  for (int h = tid; h < H; h += THREADS) { adam(p.off_b1 + h, s.gb1[h]); adam(p.off_w2 + h, s.G2[h]); }
  if (tid == 0) adam(p.off_b2, gb2);
  if (sn) {
    for (int h = tid; h < H; h += THREADS) { a.disc.u[(int64_t)r * a.disc.u_stride + h] = s.u1[h]; a.disc.v[(int64_t)r * a.disc.v_stride + d + h] = s.v2[h]; }
    for (int j = tid; j < d; j += THREADS) a.disc.v[(int64_t)r * a.disc.v_stride + j] = s.v1[j];
    if (tid == 0) a.disc.u[(int64_t)r * a.disc.u_stride + H] = u2;
  }
}

__global__ void __launch_bounds__(THREADS) gail_reward_kernel(const GailRewParams p) {
  extern __shared__ __align__(16) float sm[];
  const GailDims g = p.g;
  GailSmem s;
  gail_carve(g, sm, &s);
  const int r = blockIdx.x, tid = threadIdx.x, H = g.H, d = g.d, B = g.B;
  const float* prm = p.disc.g.params + (int64_t)r * p.disc.g.stride;
  const bool sn = p.disc.u != nullptr;
  for (int i = tid; i < H * d; i += THREADS) s.W1[i] = prm[p.off_w1 + i];
  for (int h = tid; h < H; h += THREADS) {
    s.b1[h] = prm[p.off_b1 + h]; s.w2[h] = prm[p.off_w2 + h];
    if (sn) { s.u1[h] = p.disc.u[(int64_t)r * p.disc.u_stride + h]; s.v2[h] = p.disc.v[(int64_t)r * p.disc.v_stride + d + h]; }
  }
  if (sn) for (int j = tid; j < d; j += THREADS) s.v1[j] = p.disc.v[(int64_t)r * p.disc.v_stride + j];
  const float b2 = prm[p.off_b2];
  __syncthreads();
  float sig1 = 1.f, sig2 = 1.f;
  if (sn) {  // eval mode: no power iteration, sigma from the stored (u, v) (train.py:180,194)
    sig1 = spectral_sigma(s.W1, s.u1, s.v1, s.tvec, s.red, H, d, false);
    float t = 0.f;
    for (int h = tid; h < H; h += THREADS) t = fmaf(s.w2[h], s.v2[h], t);
    sig2 = p.disc.u[(int64_t)r * p.disc.u_stride + H] * bsum(t, s.red);
  }
  for (int i = tid; i < H * d; i += THREADS) s.W1e[i] = s.W1[i] / sig1;
  for (int h = tid; h < H; h += THREADS) s.w2e[h] = s.w2[h] / sig2;
  __syncthreads();
  const float* rows = p.batch.rows + (int64_t)r * p.batch.replica_stride;
  for (int b0 = 0; b0 < B; b0 += g.RB) {
    const int nb = min(g.RB, B - b0);
    load_rows(g, rows, rows, nullptr, PASS_POLICY, b0, nb, s.X, s.CO, s.DF);
    __syncthreads();
    forward_chunk(g, s, nb, b2, s.DF);
    for (int b = tid; b < nb; b += THREADS) {
      const float f = s.DF[b];
      if (p.logits) p.logits[(int64_t)r * B + b0 + b] = f;
      if (p.reward) {  // models.py:177-180
        const float D = sigmoidf(f);
        float hh = p.disc.reward_function == IL_REWARD_GAIL ? -log1pf(-D + 1e-6f) : logf(D + 1e-6f) - log1pf(-D + 1e-6f);
        if (p.disc.reward_function == IL_REWARD_FAIRL) hh = expf(hh) * -hh;
        p.reward[(int64_t)r * p.reward_rs + (int64_t)(b0 + b) * p.reward_ld] = hh;
      }
    }
    __syncthreads();
  }
}

// predict_reward on the register-tiled forward (same helpers as gail_update_tiled_kernel): ~30 KB of shared memory instead of the update kernel's carve-up, so
// several replicas share an SM (the first kernel ran one CTA per SM with two shared loads per FMA: 112 us per step for 39 MB of input).
struct GailRewTiledParams { GailRewParams r; TDims g; };
__host__ __device__ inline int64_t reward_tiled_floats(const TDims& g) {
  auto r4 = [](int n) { return (n + 3) / 4 * 4; };
  return r4(g.HD) + r4(g.DP * g.H) + 6 * r4(g.H) + r4(g.d) + r4(g.H > g.d ? g.H : g.d) + r4(g.RB * g.DP) + r4(g.RB * g.LDZ) + 3 * r4(g.RB) + 32;
}
__global__ void __launch_bounds__(THREADS, 3) gail_reward_tiled_kernel(const GailRewTiledParams tp) {
  extern __shared__ __align__(16) float sm[];
  const GailRewParams& p = tp.r;
  const TDims g = tp.g;
  const int r = blockIdx.x, tid = threadIdx.x, H = g.H, d = g.d, B = g.B, DP = g.DP;
  int64_t o = 0;
  auto take = [&](int n) { float* q = sm + o; o += (n + 3) / 4 * 4; return q; };
  float *W1 = take(g.HD), *W1eT = take(DP * H), *b1 = take(H), *w2 = take(H), *w2e = take(H), *u1 = take(H), *v2 = take(H), *spare = take(H), *v1 = take(d), *tvec = take(H > d ? H : d);
  float *X = take(g.RB * DP), *Z = take(g.RB * g.LDZ), *F = take(g.RB), *CO = take(g.RB), *DF = take(g.RB), *red = take(32);
  (void)spare;
  const float* prm = p.disc.g.params + (int64_t)r * p.disc.g.stride;
  const bool sn = p.disc.u != nullptr;
  for (int i = tid; i < H * d; i += THREADS) W1[i] = prm[p.off_w1 + i];
  for (int h = tid; h < H; h += THREADS) {
    b1[h] = prm[p.off_b1 + h]; w2[h] = prm[p.off_w2 + h];
    if (sn) { u1[h] = p.disc.u[(int64_t)r * p.disc.u_stride + h]; v2[h] = p.disc.v[(int64_t)r * p.disc.v_stride + d + h]; }
  }
  if (sn) for (int j = tid; j < d; j += THREADS) v1[j] = p.disc.v[(int64_t)r * p.disc.v_stride + j];
  const float b2 = prm[p.off_b2];
  __syncthreads();
  float sig1 = 1.f, sig2 = 1.f;
  if (sn) {  // eval mode: no power iteration, sigma from the stored (u, v) (train.py:180,194)
    sig1 = spectral_sigma(W1, u1, v1, tvec, red, H, d, false);
    float t = 0.f;
    for (int h = tid; h < H; h += THREADS) t = fmaf(w2[h], v2[h], t);
    sig2 = p.disc.u[(int64_t)r * p.disc.u_stride + H] * bsum(t, red);
  }
  for (int i = tid; i < H * DP; i += THREADS) {
    const int h = i / DP, j = i % DP;
    W1eT[j * H + h] = j < d ? W1[h * d + j] / sig1 : 0.f;
  }
  for (int h = tid; h < H; h += THREADS) w2e[h] = w2[h] / sig2;
  __syncthreads();
  const float* rows = p.batch.rows + (int64_t)r * p.batch.replica_stride;
  for (int b0 = 0; b0 < B; b0 += g.RB) {
    const int nb = min(g.RB, B - b0);
    tiled_load_rows(g, rows, rows, nullptr, PASS_POLICY, b0, nb, X, CO, DF);
    __syncthreads();
    tiled_hidden_logits(g, X, W1eT, b1, Z, w2e, b2, F);
    __syncthreads();
    for (int b = tid; b < nb; b += THREADS) {
      const float f = F[b];
      if (p.logits) p.logits[(int64_t)r * B + b0 + b] = f;
      if (p.reward) {  // models.py:177-180
        const float D = sigmoidf(f);
        float hh = p.disc.reward_function == IL_REWARD_GAIL ? -log1pf(-D + 1e-6f) : logf(D + 1e-6f) - log1pf(-D + 1e-6f);
        if (p.disc.reward_function == IL_REWARD_FAIRL) hh = expf(hh) * -hh;
        p.reward[(int64_t)r * p.reward_rs + (int64_t)(b0 + b) * p.reward_ld] = hh;
      }
    }
  }
}

__global__ void gail_tick_kernel(int64_t* s) { *s += 1; }

int gail_setup(const il_gail* disc, const il_batch* batch, GailDims* g, int64_t* smem, int64_t off[4], const char* what) {
  IL_CHECK(disc && disc->g.params, "%s: null discriminator", what);
  IL_CHECK(disc->g.n_layers == 2 && disc->g.dims[2] == 1, "%s: only the depth-1 discriminator (GAIL.yaml:10-13) is supported by this kernel (n_layers=%d)", what, disc->g.n_layers);
  IL_CHECK(disc->g.activation == IL_ACT_RELU, "%s: only relu discriminators are supported", what);
  const int d = disc->state_only ? batch->S : batch->S + batch->A;
  IL_CHECK(disc->g.dims[0] == d, "%s: discriminator input %d != %d", what, disc->g.dims[0], d);
  const int H = disc->g.dims[1];
  IL_CHECK(H * d <= 64 * THREADS, "%s: hidden*input = %d exceeds the kernel limit %d", what, H * d, 64 * THREADS);
  IL_CHECK(H <= THREADS, "%s: hidden size %d exceeds the kernel limit %d", what, H, THREADS);
  IL_CHECK((disc->u == nullptr) == (disc->v == nullptr), "%s: spectral-norm buffers must both be set or both be null", what);
  if (disc->u) IL_CHECK(disc->u_stride >= H + 1 && disc->v_stride >= d + H, "%s: spectral-norm buffer strides too small", what);
  int RB = 64;
  for (;;) {
    *g = gail_dims(batch->S, batch->A, H, batch->B, disc->state_only, RB);
    *smem = gail_carve(*g, nullptr, nullptr);
    if (*smem <= 220 * 1024 || RB == 8) break;
    RB /= 2;
  }
  IL_CHECK(*smem <= 220 * 1024, "%s: discriminator %dx%d does not fit in shared memory", what, H, d);
  const MlpOffsets o = mlp_offsets(disc->g.dims, 2);
  off[0] = o.w[0]; off[1] = o.b[0]; off[2] = o.w[1]; off[3] = o.b[1];
  return 0;
}

}  // namespace

extern "C" int64_t il_gail_workspace_bytes(const il_gail_update_args*) { return 0; }

extern "C" int il_gail_update(il_handle* h, const il_gail_update_args* a, void* stream) {
  IL_CHECK(h && a, "il_gail_update: null argument");
  IL_CHECK(a->R > 0 && a->policy.rows && a->expert.rows, "il_gail_update: bad batches");
  IL_CHECK(a->policy.B == a->expert.B && a->policy.S == a->expert.S && a->policy.A == a->expert.A, "il_gail_update: policy/expert batch shape mismatch");
  IL_CHECK(a->policy.row == row_layout(a->policy.S, a->policy.A).len && a->expert.row == a->policy.row, "il_gail_update: bad row length");
  IL_CHECK(a->opt.m && a->opt.v && a->opt.step, "il_gail_update: null optimiser state");
  IL_CHECK(a->loss_function >= 0 && a->loss_function <= 2, "il_gail_update: bad loss function %d", a->loss_function);
  IL_CHECK(!((a->grad_penalty > 0.f || a->grad_penalty_r) && !a->eps_gp), "il_gail_update: grad_penalty > 0 (or grad_penalty_r) needs eps_gp");
  IL_CHECK(!(a->loss_function == IL_LOSS_MIXUP && !a->eps_mix), "il_gail_update: Mixup needs eps_mix");
  GailUpdParams p;
  p.a = *a;
  int64_t smem, off[4];
  IL_TRY(gail_setup(&a->disc, &a->policy, &p.g, &smem, off, "il_gail_update"));
  p.off_w1 = off[0]; p.off_b1 = off[1]; p.off_w2 = off[2]; p.off_b2 = off[3];
  cudaStream_t st = (cudaStream_t)stream;
  IL_LAUNCH(h, gail_tick_kernel, 1, 1, 0, st, a->opt.step);
  const int tiled_tiles = (p.g.H / 4) * ((p.g.d + 3) / 4);
  if (h->gail_tiled && p.g.d <= 32 && (p.g.H == 32 || p.g.H == 64 || p.g.H == 128) && a->policy.B % 4 == 0 && tiled_tiles <= 256 && p.g.row % 4 == 0) {
    GailTiledParams tp;
    tp.a = *a;
    TDims& t = tp.g;
    t.S = p.g.S; t.A = p.g.A; t.d = p.g.d; t.DP = (p.g.d + 3) / 4 * 4; t.H = p.g.H; t.B = p.g.B; t.row = p.g.row; t.LDZ = p.g.H + 4; t.HD = (p.g.H * p.g.d + 3) / 4 * 4;
    t.RB = a->policy.B < 128 ? (a->policy.B + 15) / 16 * 16 : 128;  // multiple of 16: the tile loops (H / 4 x RB / 4 tiles) have warp-uniform trip counts
    tp.off_w1 = off[0]; tp.off_b1 = off[1]; tp.off_w2 = off[2]; tp.off_b2 = off[3];
    int64_t tsm = tiled_carve(t, nullptr, nullptr);
    while (tsm > 110 * 1024 && t.RB > 32) {  // wider nets: shorter row chunks keep two CTAs per SM
      t.RB /= 2;
      tsm = tiled_carve(t, nullptr, nullptr);
    }
    IL_CHECK(tsm <= 110 * 1024, "il_gail_update: tiled kernel shared memory %lld", (long long)tsm);
    if (tiled_tiles <= 64) IL_LAUNCH(h, gail_update_tiled_kernel<1>, a->R, THREADS, (size_t)tsm, st, tp);
    else if (tiled_tiles <= 128) IL_LAUNCH(h, gail_update_tiled_kernel<2>, a->R, THREADS, (size_t)tsm, st, tp);
    else IL_LAUNCH(h, gail_update_tiled_kernel<4>, a->R, THREADS, (size_t)tsm, st, tp);
    return 0;
  }
  const int ne = (p.g.H * p.g.d + THREADS - 1) / THREADS;
#define GAIL_LAUNCH(NE) IL_LAUNCH(h, gail_update_kernel<NE>, a->R, THREADS, (size_t)smem, st, p)
  if (ne <= 4) GAIL_LAUNCH(4);
  else if (ne <= 16) GAIL_LAUNCH(16);
  else if (ne <= 32) GAIL_LAUNCH(32);
  else GAIL_LAUNCH(64);
#undef GAIL_LAUNCH
  return 0;
}

extern "C" int il_gail_reward(il_handle* h, const il_gail* disc, int R, const il_batch* batch, float* reward, int64_t reward_rs, int reward_ld, float* logits, void* stream) {
  IL_CHECK(h && disc && batch && batch->rows && R > 0, "il_gail_reward: bad argument");
  IL_CHECK(batch->row == row_layout(batch->S, batch->A).len, "il_gail_reward: bad row length");
  GailRewParams p;
  p.disc = *disc; p.batch = *batch;
  int64_t smem, off[4];
  IL_TRY(gail_setup(disc, batch, &p.g, &smem, off, "il_gail_reward"));
  p.off_w1 = off[0]; p.off_b1 = off[1]; p.off_w2 = off[2]; p.off_b2 = off[3];
  p.reward = reward; p.reward_rs = reward_rs; p.reward_ld = reward_ld; p.logits = logits;
  if (h->gail_tiled && p.g.d <= 32 && (p.g.H == 32 || p.g.H == 64 || p.g.H == 128) && p.g.row % 4 == 0) {
    GailRewTiledParams tp;
    tp.r = p;
    TDims& t = tp.g;
    t.S = p.g.S; t.A = p.g.A; t.d = p.g.d; t.DP = (p.g.d + 3) / 4 * 4; t.H = p.g.H; t.B = p.g.B; t.row = p.g.row; t.LDZ = p.g.H + 4; t.HD = (p.g.H * p.g.d + 3) / 4 * 4;
    t.RB = batch->B < 64 ? (batch->B + 15) / 16 * 16 : 64;
    const int64_t tsm = reward_tiled_floats(t) * 4;
    if (tsm <= 72 * 1024) {
      IL_LAUNCH(h, gail_reward_tiled_kernel, R, THREADS, (size_t)tsm, (cudaStream_t)stream, tp);
      return 0;
    }
  }
  IL_LAUNCH(h, gail_reward_kernel, R, THREADS, (size_t)smem, (cudaStream_t)stream, p);
  return 0;
}

// Opt in to > 48 KB dynamic shared memory once (not inside a stream capture).
int gail_init() {
  IL_CUDA(cudaFuncSetAttribute(gail_update_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
  IL_CUDA(cudaFuncSetAttribute(gail_update_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
  IL_CUDA(cudaFuncSetAttribute(gail_update_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
  IL_CUDA(cudaFuncSetAttribute(gail_update_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
  IL_CUDA(cudaFuncSetAttribute(gail_reward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
  IL_CUDA(cudaFuncSetAttribute(gail_reward_tiled_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 72 * 1024));
  IL_CUDA(cudaFuncSetAttribute(gail_update_tiled_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 110 * 1024));
  IL_CUDA(cudaFuncSetAttribute(gail_update_tiled_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 110 * 1024));
  IL_CUDA(cudaFuncSetAttribute(gail_update_tiled_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 110 * 1024));
  return 0;
}
