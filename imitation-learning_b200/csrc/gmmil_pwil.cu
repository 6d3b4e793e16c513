// GMMILDiscriminator.predict_reward (models.py:183-201, helpers :25-44) and PWILDiscriminator
// (models.py:216-249) for R replicas. Neither materialises the reference's [n1, n2, d] tensor.
#include "common.cuh"

#include <math.h>

namespace {

constexpr int GT = 256;  // threads; also rows of the "i" tile handled per CTA
constexpr int TJ = 32;   // rows of the "j" tile staged in shared memory

struct GmmilParams {
  il_batch pol, exp_;
  int d;               // feature width (S or S + A)
  const float* gamma;  // [R, 2]
  float* reward; int64_t reward_rs; int reward_ld;
  float* dist;         // optional [R, B, B] output of pairwise distances (bandwidth pass)
  int dist_expert_self;  // 1: distances expert-expert instead of policy-expert
};

// reward_i = wn_i * ( sum_j (K1+K2)(x_i, e_j) wen_j - sum_j (K1+K2)(x_i, x_j) wn_j ),  D = mean_k (x_ik - y_jk)^2
__global__ void __launch_bounds__(GT) gmmil_kernel(const GmmilParams p) {
  extern __shared__ __align__(16) float sm[];
  const int r = blockIdx.y, i0 = blockIdx.x * GT, tid = threadIdx.x;
  const int B = p.pol.B, d = p.d, ld = d | 1, row = p.pol.row;
  const RowLayout L = row_layout(p.pol.S, p.pol.A);
  float* Xi = sm;               // [GT, ld]
  float* Yj = Xi + GT * ld;     // [TJ, ld]
  float* wj = Yj + TJ * ld;     // [TJ]
  float* red = wj + TJ;         // [32]
  const float* prow = p.pol.rows + (int64_t)r * p.pol.replica_stride;
  const float* erow = p.exp_.rows + (int64_t)r * p.exp_.replica_stride;
  const bool dist_only = p.dist != nullptr;
  const float* irow = (dist_only && p.dist_expert_self) ? erow : prow;
  // normalisers (models.py:197)
  float ws = 0.f, es = 0.f;
  for (int b = tid; b < B; b += GT) { ws += prow[(int64_t)b * row + L.weight]; es += erow[(int64_t)b * row + L.weight]; }
  ws = block_sum(ws, red);
  es = block_sum(es, red);
  const int ni = min(GT, B - i0);
  for (int idx = tid; idx < ni * d; idx += GT) Xi[(idx / d) * ld + idx % d] = irow[(int64_t)(i0 + idx / d) * row + idx % d];
  const float g1 = dist_only ? 0.f : p.gamma[r * 2 + 0], g2 = dist_only ? 0.f : p.gamma[r * 2 + 1];
  const float inv_d = 1.f / (float)d;
  float acc = 0.f;
  const int n_src = dist_only ? 1 : 2;  // 0: expert rows (similarity), 1: policy rows (self-similarity)
  for (int src = 0; src < n_src; ++src) {
    const float* jrow = src == 0 ? erow : prow;
    const float wnorm = src == 0 ? es : ws;
    float part = 0.f;
    for (int j0 = 0; j0 < B; j0 += TJ) {
      const int nj = min(TJ, B - j0);
      __syncthreads();
      for (int idx = tid; idx < nj * d; idx += GT) Yj[(idx / d) * ld + idx % d] = jrow[(int64_t)(j0 + idx / d) * row + idx % d];
      for (int j = tid; j < nj; j += GT) wj[j] = jrow[(int64_t)(j0 + j) * row + L.weight] / wnorm;
      __syncthreads();
      if (tid < ni) {
        const float* xi = Xi + tid * ld;
        for (int j = 0; j < nj; ++j) {
          const float* yj = Yj + j * ld;
          float s = 0.f;
          for (int k = 0; k < d; ++k) {
            const float df = xi[k] - yj[k];
            s = fmaf(df, df, s);
          }
          const float D = s * inv_d;  // models.py:28 (mean over features)
          if (dist_only) p.dist[((int64_t)r * B + i0 + tid) * B + j0 + j] = D;
          else part = fmaf(expf(-g1 * D) + expf(-g2 * D), wj[j], part);
        }
      }
    }
    acc += src == 0 ? part : -part;
  }
  if (!dist_only && tid < ni) {
    const float wn = prow[(int64_t)(i0 + tid) * row + L.weight] / ws;
    p.reward[(int64_t)r * p.reward_rs + (int64_t)(i0 + tid) * p.reward_ld] = wn * acc;
  }
}

// models.py:40-44 weighted median of the [B, B] distance matrix with weights outer(w_row, w_col):
// smallest element x with sum_{x_ij <= x} w_i w_j >= 0.5 * sum w_i w_j. Binary search over the (non-negative)
// float bit patterns; one CTA per replica. out[r] = 1 / (median + 1e-8) (models.py:194-195).
__global__ void __launch_bounds__(256) weighted_median_kernel(const float* __restrict__ dist, const float* __restrict__ rows_i, int64_t rs_i, const float* __restrict__ rows_j,
                                                               int64_t rs_j, int row, int off_w, int B, float* __restrict__ gamma_out, int gamma_col) {
  __shared__ double redd[32];
  __shared__ unsigned int s_lo, s_hi;
  const int r = blockIdx.x, tid = threadIdx.x;
  const float* D = dist + (int64_t)r * B * B;
  const float* wi = rows_i + (int64_t)r * rs_i + off_w;
  const float* wjp = rows_j + (int64_t)r * rs_j + off_w;
  auto bsumd = [&](double v) {
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    __syncthreads();
    if ((tid & 31) == 0) redd[tid >> 5] = v;
    __syncthreads();
    double t = 0.0;
    for (int w = 0; w < 8; ++w) t += redd[w];
    return t;
  };
  double tot = 0.0;
  for (int64_t e = tid; e < (int64_t)B * B; e += 256) tot += (double)wi[(e / B) * row] * (double)wjp[(e % B) * row];
  tot = bsumd(tot);
  if (tid == 0) { s_lo = 0u; s_hi = 0x7f800000u; }
  __syncthreads();
  for (int it = 0; it < 32; ++it) {
    const unsigned lo = s_lo, hi = s_hi;
    if (lo >= hi) break;
    const unsigned mid = lo + (hi - lo) / 2;
    double c = 0.0;
    for (int64_t e = tid; e < (int64_t)B * B; e += 256)
      if (__float_as_uint(D[e]) <= mid) c += (double)wi[(e / B) * row] * (double)wjp[(e % B) * row];
    c = bsumd(c);
    if (tid == 0) {
      if (c >= 0.5 * tot) s_hi = mid; else s_lo = mid + 1;
    }
    __syncthreads();
  }
  if (tid == 0) gamma_out[r * 2 + gamma_col] = (float)(1.0 / ((double)__uint_as_float(s_hi) + 1e-8));
}

int gmmil_launch(il_handle* h, int R, const il_batch* pol, const il_batch* exp_, int state_only, const float* gamma, float* reward, int64_t reward_rs, int reward_ld, float* dist,
                 int expert_self, cudaStream_t st) {
  IL_CHECK(pol && exp_ && pol->rows && exp_->rows && R > 0, "gmmil: bad batches");
  IL_CHECK(pol->B == exp_->B && pol->S == exp_->S && pol->A == exp_->A && pol->row == exp_->row, "gmmil: policy/expert batch shape mismatch");
  IL_CHECK(pol->row == row_layout(pol->S, pol->A).len, "gmmil: bad row length");
  GmmilParams p;
  p.pol = *pol; p.exp_ = *exp_; p.d = state_only ? pol->S : pol->S + pol->A;
  p.gamma = gamma; p.reward = reward; p.reward_rs = reward_rs; p.reward_ld = reward_ld; p.dist = dist; p.dist_expert_self = expert_self;
  const int ld = p.d | 1;
  const size_t smem = (size_t)(GT * ld + TJ * ld + TJ + 32) * 4;
  IL_CHECK(smem <= 220 * 1024, "gmmil: feature width %d too large", p.d);
  dim3 grid((pol->B + GT - 1) / GT, R);
  IL_LAUNCH(h, gmmil_kernel, grid, GT, smem, st, p);
  return 0;
}

// ---- PWIL ----------------------------------------------------------------------------------------------------
// One CTA per replica. weights[r, i] < 0 marks a consumed (deleted, models.py:244) atom.
__global__ void __launch_bounds__(256) pwil_reward_kernel(const il_pwil p, int R, const float* __restrict__ state, const float* __restrict__ action, float* __restrict__ reward,
                                                          const int32_t* __restrict__ active) {
  extern __shared__ __align__(16) float sm[];
  __shared__ float s_val[8];
  __shared__ int s_idx[8];
  __shared__ int s_best;
  const int r = blockIdx.x, tid = threadIdx.x;
  if (active && !active[r]) return;
  const int N = p.N, d = p.d;
  float* dists = sm;         // [N]
  float* atom = dists + N;   // [d]
  float* w = p.weights + (int64_t)r * N;
  for (int k = tid; k < d; k += 256) {
    const float raw = k < p.S ? state[(int64_t)r * p.S + k] : action[(int64_t)r * p.A + (k - p.S)];
    atom[k] = p.scale[k] * (raw + p.offset[k]);  // models.py:234
  }
  __syncthreads();
  for (int i = tid; i < N; i += 256) {  // models.py:236
    float s = 0.f;
    if (w[i] >= 0.f) {
      const float* a = p.atoms + (int64_t)i * d;
      for (int k = 0; k < d; ++k) {
        const float df = a[k] - atom[k];
        s = fmaf(df, df, s);
      }
      s = sqrtf(s);
    } else {
      s = INFINITY;
    }
    dists[i] = s;
  }
  __syncthreads();
  double weight = 1.0 / (double)p.time_horizon - 1e-6, cost = 0.0;  // models.py:235 (Python floats)
  while (weight > 0.0) {
    // block argmin, first occurrence on ties (torch.argmin)
    float bv = INFINITY;
    int bi = 0x7fffffff;
    for (int i = tid; i < N; i += 256) {
      const float v = dists[i];
      if (v < bv) { bv = v; bi = i; }
    }
    for (int o = 16; o > 0; o >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
      const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
      if (ov < bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
    }
    if ((tid & 31) == 0) { s_val[tid >> 5] = bv; s_idx[tid >> 5] = bi; }
    __syncthreads();
    if (tid == 0) {
      for (int q = 1; q < 8; ++q)
        if (s_val[q] < bv || (s_val[q] == bv && s_idx[q] < bi)) { bv = s_val[q]; bi = s_idx[q]; }
      s_best = bi;
    }
    __syncthreads();
    const int best = s_best;
    if (best == 0x7fffffff || !(dists[best] < INFINITY)) break;  // no expert atoms left
    const double ew = (double)w[best], dd = (double)dists[best];
    __syncthreads();
    if (weight >= ew) {  // models.py:241-244
      cost += ew * dd;
      weight -= ew;
      if (tid == 0) { w[best] = -1.f; dists[best] = INFINITY; }
    } else {  // models.py:246-248
      cost += weight * dd;
      if (tid == 0) w[best] = (float)((double)w[best] - weight);
      weight = 0.0;
    }
    __syncthreads();
  }
  if (tid == 0) {  // models.py:249
    const float scale = p.reward_scale_r ? p.reward_scale_r[r] : p.reward_scale, bandwidth = p.reward_bandwidth_r ? p.reward_bandwidth_r[r] : p.reward_bandwidth;
    reward[r] = (float)((double)scale * exp(-(double)bandwidth * cost));
  }
}

__global__ void pwil_reset_kernel(float* __restrict__ weights, int N, int R, const int32_t* __restrict__ mask) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)R * N) return;
  if (mask && !mask[i / N]) return;
  weights[i] = 1.f / (float)N;  // models.py:230
}

}  // namespace

extern "C" int64_t il_gmmil_workspace_bytes(int R, int B) { return (int64_t)R * B * B * 4; }

extern "C" int il_gmmil_bandwidth(il_handle* h, int R, const il_batch* policy, const il_batch* expert, int state_only, float* gamma, void* workspace, int64_t workspace_bytes,
                                  void* stream) {
  IL_CHECK(h && gamma && workspace, "il_gmmil_bandwidth: null argument");
  IL_CHECK(policy && workspace_bytes >= il_gmmil_workspace_bytes(R, policy->B), "il_gmmil_bandwidth: workspace too small");
  cudaStream_t st = (cudaStream_t)stream;
  float* dist = static_cast<float*>(workspace);
  const RowLayout L = row_layout(policy->S, policy->A);
  IL_TRY(gmmil_launch(h, R, policy, expert, state_only, nullptr, nullptr, 0, 0, dist, 0, st));
  IL_LAUNCH(h, weighted_median_kernel, R, 256, 0, st, dist, policy->rows, policy->replica_stride, expert->rows, expert->replica_stride, policy->row, L.weight, policy->B, gamma, 0);
  IL_TRY(gmmil_launch(h, R, policy, expert, state_only, nullptr, nullptr, 0, 0, dist, 1, st));
  IL_LAUNCH(h, weighted_median_kernel, R, 256, 0, st, dist, expert->rows, expert->replica_stride, expert->rows, expert->replica_stride, policy->row, L.weight, policy->B, gamma, 1);
  return 0;
}

extern "C" int il_gmmil_reward(il_handle* h, int R, const il_batch* policy, const il_batch* expert, int state_only, const float* gamma, float* reward, int64_t reward_rs,
                               int reward_ld, void* stream) {
  IL_CHECK(h && gamma && reward, "il_gmmil_reward: null argument");
  return gmmil_launch(h, R, policy, expert, state_only, gamma, reward, reward_rs, reward_ld, nullptr, 0, (cudaStream_t)stream);
}

extern "C" int il_pwil_reset(il_handle* h, const il_pwil* p, int R, const int32_t* mask, void* stream) {
  IL_CHECK(h && p && p->weights && p->N > 0 && R > 0, "il_pwil_reset: bad argument");
  IL_LAUNCH(h, pwil_reset_kernel, (unsigned)(((int64_t)R * p->N + 255) / 256), 256, 0, (cudaStream_t)stream, p->weights, p->N, R, mask);
  return 0;
}

extern "C" int il_pwil_reward(il_handle* h, const il_pwil* p, int R, const float* state, const float* action, float* reward, const int32_t* active, void* stream) {
  IL_CHECK(h && p && p->atoms && p->scale && p->offset && p->weights && state && reward && R > 0, "il_pwil_reward: bad argument");
  IL_CHECK(p->state_only || action, "il_pwil_reward: null action");
  IL_CHECK(p->d == (p->state_only ? p->S : p->S + p->A), "il_pwil_reward: atom width %d inconsistent with S=%d A=%d", p->d, p->S, p->A);
  const size_t smem = (size_t)(p->N + p->d) * 4;
  IL_CHECK(smem <= 220 * 1024, "il_pwil_reward: %d expert atoms do not fit in shared memory", p->N);
  IL_LAUNCH(h, pwil_reward_kernel, R, 256, smem, (cudaStream_t)stream, *p, R, state, action, reward, active);
  return 0;
}

int gmmil_pwil_init() {
  IL_CUDA(cudaFuncSetAttribute(gmmil_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
  IL_CUDA(cudaFuncSetAttribute(pwil_reward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
  return 0;
}
