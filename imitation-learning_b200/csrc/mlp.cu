// Replica-batched MLP programs + SoftActor / TwinCritic entry points + Adam / polyak kernels.
#include "mlp.cuh"

#include <math.h>

constexpr int HB_MAXN = 8;
struct HeadBwdArgs {
  const float* dout; int64_t dout_gs; int dout_gdiv, ld_dout;   // [n, Nh]
  const float* w; int64_t w_gs;                                 // W_L [Nh, H] row-major
  const float* y; int64_t y_gs;                                 // Y [n, H]
  float* dz; int64_t dz_gs;                                     // out [n, H]
  float* dw; float* db; float* db_prev; int64_t g_gs;           // gradient slices (group stride g_gs): dW_L [Nh, H], db_L [Nh], db_{L-1} [H]
  int n, H, Nh;
};
int launch_head_backward(il_handle* h, const HeadBwdArgs& a, int G, cudaStream_t stream);
int launch_head_dx_bits(il_handle* h, const HeadBwdArgs& a, const uint32_t* bits, int64_t bits_gs, int G, cudaStream_t stream);

int mlp_validate(const il_mlp* m, const char* what) {
  IL_CHECK(m != nullptr && m->params != nullptr, "%s: null mlp", what);
  IL_CHECK(m->n_layers >= 1 && m->n_layers <= IL_MAX_LAYERS, "%s: n_layers %d out of range", what, m->n_layers);
  IL_CHECK(m->activation >= 0 && m->activation <= 2, "%s: bad activation %d", what, m->activation);
  for (int l = 0; l <= m->n_layers; ++l) IL_CHECK(m->dims[l] > 0, "%s: dims[%d] = %d", what, l, m->dims[l]);
  const MlpOffsets o = mlp_offsets(m->dims, m->n_layers);
  IL_CHECK(m->stride >= o.total - 31 && m->stride % 4 == 0, "%s: stride %lld too small / unaligned for %lld parameters", what, (long long)m->stride, (long long)o.total);
  IL_CHECK((reinterpret_cast<uintptr_t>(m->params) & 15) == 0, "%s: params not 16-byte aligned", what);
  return 0;
}

int mlp_max_hidden(const il_mlp* m) {
  int mx = 1;
  for (int l = 1; l <= m->n_layers; ++l) mx = m->dims[l] > mx ? m->dims[l] : mx;
  return mx;
}

static int64_t mlp_bits_bytes(const il_mlp* m, int G, int n, int l) {  // sign-bit words of hidden layer l (0 when the width is not a multiple of 32)
  return m->dims[l + 1] % 32 == 0 ? il_align_up((int64_t)G * n * (m->dims[l + 1] / 32) * 4, 256) : 0;
}

int64_t mlp_acts_bytes(const il_mlp* m, int G, int n) {
  int64_t b = 0;
  for (int l = 0; l + 1 < m->n_layers; ++l) b += il_align_up((int64_t)G * n * m->dims[l + 1] * 4, 256) + mlp_bits_bytes(m, G, n, l);
  return b;
}

char* mlp_acts_carve(const il_mlp* m, int G, int n, char* ws, MlpActs* acts) {
  for (int l = 0; l < IL_MAX_LAYERS; ++l) { acts->hid[l] = nullptr; acts->bits[l] = nullptr; acts->bits_valid[l] = false; }
  for (int l = 0; l + 1 < m->n_layers; ++l) {
    acts->hid[l] = reinterpret_cast<float*>(ws);
    ws += il_align_up((int64_t)G * n * m->dims[l + 1] * 4, 256);
    if (mlp_bits_bytes(m, G, n, l)) {
      acts->bits[l] = reinterpret_cast<uint32_t*>(ws);
      ws += mlp_bits_bytes(m, G, n, l);
    }
  }
  return ws;
}

int mlp_forward(il_handle* h, const il_mlp* m, int G, int n, MatView X, MlpActs& acts, float* out, int64_t out_gs, int ld_out, cudaStream_t stream, int keep) {
  const MlpOffsets o = mlp_offsets(m->dims, m->n_layers);
  const int L = m->n_layers;
  const bool keep_hidden = keep != MLP_KEEP_NONE;
  const bool want_bits = h->mask_bits && keep_hidden && m->activation == IL_ACT_RELU;
  for (int l = 0; l < IL_MAX_LAYERS; ++l) acts.bits_valid[l] = false;
  auto layer_args = [&](int l) {
    GemmArgs a{};
    if (l == 0) { a.A = X.ptr; a.a_gs = X.gs; a.a_gdiv = X.gdiv; a.lda = X.ld; }
    else { a.A = acts.hid[l - 1]; a.a_gs = (int64_t)n * m->dims[l]; a.a_gdiv = 1; a.lda = m->dims[l]; }
    a.a_kmajor = 1;
    a.B = m->params + o.w[l]; a.b_gs = m->stride; a.b_gdiv = 1; a.ldb = m->dims[l]; a.b_kmajor = 1;
    a.bias = m->params + o.b[l]; a.bias_gs = m->stride;
    if (l == L - 1) { a.C = out; a.c_gs = out_gs; a.ldc = ld_out; a.act = -1; }
    else { a.C = acts.hid[l]; a.c_gs = (int64_t)n * m->dims[l + 1]; a.ldc = m->dims[l + 1]; a.act = m->activation; }
    a.M = n; a.N = m->dims[l + 1]; a.K = m->dims[l]; a.G = G;
    return a;
  };
  // the last hidden layer runs on the tensor-core engine with the final linear layer (N <= 8) fused into its epilogue
  const bool head_shape = L >= 2 && m->activation == IL_ACT_RELU && ld_out == m->dims[L] && out_gs == (int64_t)n * m->dims[L];
  for (int l = 0; l < L; ++l) {
    if (head_shape && l == L - 2) {
      GemmArgs a = layer_args(l);
      if (tc_head_fusable(h, a, m->dims[L])) {
        // MLP_KEEP_MASKS: an input-gradient pass needs the last hidden layer only as its ReLU mask -> sign bits (1/32 of the bytes) instead of the fp32 tile
        const bool bits = want_bits && keep == MLP_KEEP_MASKS && acts.bits[l] && m->dims[L] <= HB_MAXN;
        if (bits) { a.bits_out = acts.bits[l]; a.bits_out_gs = (int64_t)n * (m->dims[l + 1] / 32); acts.bits_valid[l] = true; }
        IL_TRY(launch_tc_gemm_head(h, a, m->params + o.w[L - 1], m->params + o.b[L - 1], m->stride, m->dims[L], out, out_gs, keep_hidden && !bits ? 1 : 0, stream));
        return 0;
      }
    }
    if (head_shape && l == 0 && L == 3) {
      // depth-2 nets (every actor / critic of the reference, conf/train_config.yaml:28-35): the first layer (K0 = state or
      // state + action columns) is computed inside the producers of the second layer's tensor-core launch, so its output
      // is written to HBM only when a backward pass needs it — and never read back by the forward pass
      GemmArgs a1 = layer_args(1);
      a1.A = nullptr; a1.a_gs = 0; a1.a_gdiv = 1; a1.lda = m->dims[1];
      if (tc_head_fusable(h, a1, m->dims[L]) && tc_l1_fusable(h, a1, m->dims[0])) {
        TcFuseL1 f{};
        f.x = X.ptr; f.x_gs = X.gs; f.x_gdiv = X.gdiv; f.x_ld = X.ld; f.x_k = m->dims[0];
        f.w1 = m->params + o.w[0]; f.b1 = m->params + o.b[0]; f.gs = m->stride;
        f.store = keep_hidden ? acts.hid[0] : nullptr; f.store_gs = (int64_t)n * m->dims[1];
        IL_TRY(launch_tc_gemm_head(h, a1, m->params + o.w[L - 1], m->params + o.b[L - 1], m->stride, m->dims[L], out, out_gs, keep_hidden ? 1 : 0, stream, &f));
        return 0;
      }
    }
    GemmArgs a = layer_args(l);
    if (want_bits && l + 1 < L && acts.bits[l] && gemm_first_layer_emits_bits(h, a)) {  // the mask of the next layer's input-gradient product
      a.bits_out = acts.bits[l]; a.bits_out_gs = (int64_t)n * (m->dims[l + 1] / 32);
      acts.bits_valid[l] = true;
    }
    IL_TRY(launch_gemm(h, a, stream));
  }
  return 0;
}

static bool head_backward_eligible(const il_mlp* m, int n, int64_t grad_stride) {
  const int L = m->n_layers, H = m->dims[L - 1], Nh = m->dims[L];
  return m->activation == IL_ACT_RELU && Nh <= HB_MAXN && H % 4 == 0 && n <= 1024 && grad_stride % 4 == 0 && m->stride % 4 == 0;
}

int mlp_backward(il_handle* h, const il_mlp* m, int G, int n, MatView X, const MlpActs& acts, MatView dOut, float* grads, int64_t grad_stride,
                 float* dX, int64_t dx_gs, int ld_dx, int dx_col0, int dx_cols, float* tmpA, float* tmpB, cudaStream_t stream) {
  const MlpOffsets o = mlp_offsets(m->dims, m->n_layers);
  const int L = m->n_layers;
  MatView dZ = dOut;  // gradient w.r.t. the pre-activation output of layer l
  float* next_tmp = tmpA;
  bool bias_done = false;  // db of the current layer already produced by the fused head kernel
  for (int l = L - 1; l >= 0; --l) {
    MatView Xin = l == 0 ? X : MatView{acts.hid[l - 1], (int64_t)n * m->dims[l], 1, m->dims[l]};
    if (l == L - 1 && l > 0 && grads && h->head_fused && head_backward_eligible(m, n, grad_stride)) {
      // head: dZ_{L-2}, dW_L, db_L and db_{L-1} in one pass over the last hidden activation
      HeadBwdArgs a{};
      a.dout = dZ.ptr; a.dout_gs = dZ.gs; a.dout_gdiv = dZ.gdiv; a.ld_dout = dZ.ld;
      a.w = m->params + o.w[l]; a.w_gs = m->stride;
      a.y = acts.hid[l - 1]; a.y_gs = (int64_t)n * m->dims[l];
      a.dz = next_tmp; a.dz_gs = (int64_t)n * m->dims[l];
      a.dw = grads + o.w[l]; a.db = grads + o.b[l]; a.db_prev = grads + o.b[l - 1]; a.g_gs = grad_stride;
      a.n = n; a.H = m->dims[l]; a.Nh = m->dims[l + 1];
      IL_TRY(launch_head_backward(h, a, G, stream));
      dZ = MatView{next_tmp, (int64_t)n * m->dims[l], 1, m->dims[l]};
      next_tmp = next_tmp == tmpA ? tmpB : tmpA;
      bias_done = true;
      continue;
    }
    if (l == L - 1 && l > 0 && !grads && acts.bits_valid[l - 1] && m->dims[l + 1] <= HB_MAXN) {
      // input-gradient pass: dZ_{L-2} = (dOut W_L) * 1[hidden > 0] straight from the sign-bit words (the hidden tile itself was never stored)
      HeadBwdArgs a{};
      a.dout = dZ.ptr; a.dout_gs = dZ.gs; a.dout_gdiv = dZ.gdiv; a.ld_dout = dZ.ld;
      a.w = m->params + o.w[l]; a.w_gs = m->stride;
      a.dz = next_tmp; a.dz_gs = (int64_t)n * m->dims[l];
      a.n = n; a.H = m->dims[l]; a.Nh = m->dims[l + 1];
      IL_TRY(launch_head_dx_bits(h, a, acts.bits[l - 1], (int64_t)n * (m->dims[l] / 32), G, stream));
      dZ = MatView{next_tmp, (int64_t)n * m->dims[l], 1, m->dims[l]};
      next_tmp = next_tmp == tmpA ? tmpB : tmpA;
      continue;
    }
    if (grads) {  // dW_l[o, i] = sum_b dZ[b, o] * Xin[b, i];  db_l[o] = sum_b dZ[b, o]
      GemmArgs a{};
      a.A = dZ.ptr; a.a_gs = dZ.gs; a.a_gdiv = dZ.gdiv; a.lda = dZ.ld; a.a_kmajor = 0;
      a.B = Xin.ptr; a.b_gs = Xin.gs; a.b_gdiv = Xin.gdiv; a.ldb = Xin.ld; a.b_kmajor = 0;
      a.C = grads + o.w[l]; a.c_gs = grad_stride; a.ldc = m->dims[l]; a.act = -1;
      if (!bias_done) { a.colsum = grads + o.b[l]; a.colsum_gs = grad_stride; }
      bias_done = false;
      a.M = m->dims[l + 1]; a.N = m->dims[l]; a.K = n; a.G = G;
      IL_TRY(launch_gemm(h, a, stream));
    }
    if (l > 0) {  // dZ_{l-1}[b, i] = (sum_o dZ[b, o] * W_l[o, i]) * act'(hid_{l-1}[b, i])
      GemmArgs a{};
      a.A = dZ.ptr; a.a_gs = dZ.gs; a.a_gdiv = dZ.gdiv; a.lda = dZ.ld; a.a_kmajor = 1;
      a.B = m->params + o.w[l]; a.b_gs = m->stride; a.b_gdiv = 1; a.ldb = m->dims[l]; a.b_kmajor = 0;
      a.C = next_tmp; a.c_gs = (int64_t)n * m->dims[l]; a.ldc = m->dims[l]; a.act = -1;
      a.mask_act = m->activation;
      a.M = n; a.N = m->dims[l]; a.K = m->dims[l + 1]; a.G = G;
      if (acts.bits_valid[l - 1] && m->activation == IL_ACT_RELU && gemm_uses_tc(h, a)) {  // ReLU mask from the sign-bit words: 8 KB instead of 256 KB per 256 x 256 tile
        a.mask_bits = acts.bits[l - 1]; a.mask_bits_gs = (int64_t)n * (m->dims[l] / 32);
        if (h->mask_bits >= 2 && l == 1 && !grads && dX && ld_dx == dx_cols && dx_gs == (int64_t)n * dx_cols && tc_dx_head_fusable(h, a, dx_cols)) {
          // input-gradient pass: dZ_0 is only an intermediate of dX = dZ_0 W_1[:, cols] — the thin product runs in the epilogue on the masked rows, dZ_0 is never stored
          a.C = nullptr;
          IL_TRY(launch_tc_gemm_dx_head(h, a, m->params + o.w[0] + dx_col0, m->stride, m->dims[0], dx_cols, dX, dx_gs, stream));
          return 0;
        }
      } else {
        a.mask = acts.hid[l - 1]; a.mask_gs = (int64_t)n * m->dims[l]; a.ldmask = m->dims[l];
      }
      IL_TRY(launch_gemm(h, a, stream));
      dZ = MatView{next_tmp, (int64_t)n * m->dims[l], 1, m->dims[l]};
      next_tmp = next_tmp == tmpA ? tmpB : tmpA;
    } else if (dX) {  // gradient w.r.t. a column slice of the input
      GemmArgs a{};
      a.A = dZ.ptr; a.a_gs = dZ.gs; a.a_gdiv = dZ.gdiv; a.lda = dZ.ld; a.a_kmajor = 1;
      a.B = m->params + o.w[0] + dx_col0; a.b_gs = m->stride; a.b_gdiv = 1; a.ldb = m->dims[0]; a.b_kmajor = 0;
      a.C = dX; a.c_gs = dx_gs; a.ldc = ld_dx; a.act = -1;
      a.M = n; a.N = dx_cols; a.K = m->dims[1]; a.G = G;
      IL_TRY(launch_gemm(h, a, stream));
    }
  }
  return 0;
}

// ---- tanh-Gaussian head (models.py:90-102; torch TransformedDistribution / TanhTransform arithmetic) -------
namespace {

__global__ void actor_head_kernel(const HeadFwdArgs p) {
  const int64_t row = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (row >= (int64_t)p.R * p.n) return;
  const int r = (int)(row / p.n), i = (int)(row % p.n);
  const int A = p.A;
  const float* hd = p.head + row * 2 * A;
  float* act_row = p.action ? p.action + (int64_t)r * p.action_rs + (int64_t)i * p.ld_action : nullptr;
  if (p.copy_src && act_row) {
    const float* src = p.copy_src + (int64_t)r * p.copy_rs + (int64_t)i * p.copy_ld;
    for (int j = 0; j < p.copy_cols; ++j) act_row[j - p.copy_cols] = __ldg(src + j);
  }
  const float keep = p.zero_mask ? 1.f - __ldg(p.zero_mask + (int64_t)r * p.zero_mask_rs + (int64_t)i * p.zero_mask_ld) : 1.f;
  const float LOG_SQRT_2PI = 0.91893853320467274178f, LOG2 = 0.69314718055994530942f;
  const float A_LO = (float)(-1.0 + 1e-6), A_HI = (float)(1.0 - 1e-6);
  float sum_ladj = 0.f, sum_nlp = 0.f;
  const bool want_lp = p.log_prob != nullptr && (p.eps != nullptr || p.given != nullptr);
  for (int j = 0; j < A; ++j) {
    const float mu = hd[j];
    const float ls = fminf(fmaxf(hd[A + j], -20.f), 2.f);  // models.py:92
    if (p.mean) p.mean[row * A + j] = mu;
    if (p.log_std) p.log_std[row * A + j] = ls;
    float x, a;
    const float sd = expf(ls);
    if (p.given) {  // models.py:97-99: clamp, atanh
      a = fminf(fmaxf(p.given[row * A + j], A_LO), A_HI);
      x = atanhf(a);
    } else if (p.eps) {  // Normal.sample / rsample: loc + eps * scale
      x = __fadd_rn(mu, __fmul_rn(sd, p.eps[row * A + j]));
      a = tanhf(x);
    } else {  // models.py:101-102
      x = mu;
      a = tanhf(mu);
    }
    if (act_row && !p.given) act_row[j] = keep * a;
    if (want_lp) {
      const float var = __fmul_rn(sd, sd);
      const float diff = __fsub_rn(x, mu);
      float nlp = __fdiv_rn(-__fmul_rn(diff, diff), __fmul_rn(2.f, var));
      nlp = __fsub_rn(__fsub_rn(nlp, logf(sd)), LOG_SQRT_2PI);
      const float ladj = __fmul_rn(2.f, __fsub_rn(__fsub_rn(LOG2, x), softplusf(__fmul_rn(-2.f, x))));
      sum_nlp += nlp;
      sum_ladj += ladj;
    }
  }
  if (want_lp) p.log_prob[row] = __fadd_rn(__fsub_rn(0.f, sum_ladj), sum_nlp);
}

// Whole-MLP forward for a few rows per net (rollout: n = 1 per replica, train.py:152; batched evaluation: n = episodes):
// one CTA per (net, block of NR rows); activations ping-pong in shared memory, every weight row is streamed once per CTA
// with coalesced 128-bit loads (one warp per output unit) — a GEMV that is bound by reading the parameters.
struct SmallFwdArgs {
  il_mlp m;
  MlpOffsets o;
  const float* X;
  int64_t x_gs;
  int x_gdiv, ldx, n, maxd;
  float* out;  // [G, n, dims[L]]; tanh_first = A > 0: [G, n, A] = tanh of the first A outputs (the greedy action, models.py:101-102)
  int tanh_first;
};
template <int NR>
__global__ void __launch_bounds__(256) mlp_small_forward_kernel(const SmallFwdArgs p) {
  extern __shared__ __align__(16) float sm[];
  const int g = blockIdx.x, r0 = blockIdx.y * NR, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int nr = min(NR, p.n - r0), L = p.m.n_layers, maxd = p.maxd;
  float* bufs[2] = {sm, sm + NR * maxd};
  const float* X = p.X + (int64_t)(g / p.x_gdiv) * p.x_gs;
  for (int idx = tid; idx < NR * p.m.dims[0]; idx += 256) {
    const int r = idx / p.m.dims[0], k = idx % p.m.dims[0];
    bufs[0][r * maxd + k] = r < nr ? __ldg(X + (int64_t)(r0 + r) * p.ldx + k) : 0.f;
  }
  const float* prm = p.m.params + (int64_t)g * p.m.stride;
  __syncthreads();
  for (int l = 0; l < L; ++l) {
    const int in = p.m.dims[l], od = p.m.dims[l + 1];
    const float* W = prm + p.o.w[l];
    const float* bias = prm + p.o.b[l];
    const float* xin = bufs[l & 1];
    float* xout = bufs[(l + 1) & 1];
    const bool vec = (in % 4 == 0) && (p.m.stride % 4 == 0);
    if (NR == 1 && vec && in <= 16) {
      // single row, thin layer (the state input of the rollout, train.py:152): one output unit per thread, its whole weight row in flight at once
      for (int o = tid; o < od; o += 256) {
        const float4* wr = reinterpret_cast<const float4*>(W + (int64_t)o * in);
        float4 w4[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) w4[q] = 4 * q < in ? __ldg(wr + q) : make_float4(0.f, 0.f, 0.f, 0.f);
        float v = __ldg(bias + o);
#pragma unroll
        for (int q = 0; q < 4; ++q)
          if (4 * q < in) {
            const float4 x4 = *reinterpret_cast<const float4*>(xin + 4 * q);
            v = fmaf(w4[q].x, x4.x, fmaf(w4[q].y, x4.y, fmaf(w4[q].z, x4.z, fmaf(w4[q].w, x4.w, v))));
          }
        if (l < L - 1) v = act_apply(v, p.m.activation);
        xout[o] = v;
      }
      __syncthreads();
      continue;
    }
    if (NR == 1 && vec && in % 128 == 0 && in <= 256) {
      // single row, wide layer: the kernel is a pure weight stream and its layers are dependent phases, so what matters is how many bytes each warp
      // has in flight per round trip: EIGHT weight rows (8 output units, 16 x 128-bit loads per lane) are issued together and reduced together
      // (ncu on the 4-rows-per-round version: 2.4 TB/s, long-scoreboard bound: 16 dependent load rounds per warp for a 256 x 256 layer, now 4)
      const int kv = in >> 7;
      float4 x4[2];
#pragma unroll
      for (int v = 0; v < 2; ++v) x4[v] = v < kv ? *reinterpret_cast<const float4*>(xin + v * 128 + lane * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
      for (int o0 = warp * 8; o0 < od; o0 += 64) {
        float4 w4[8][2];
#pragma unroll
        for (int u = 0; u < 8; ++u)
#pragma unroll
          for (int v = 0; v < 2; ++v)
            w4[u][v] = (o0 + u < od && v < kv) ? __ldg(reinterpret_cast<const float4*>(W + (int64_t)(o0 + u) * in + v * 128 + lane * 4)) : make_float4(0.f, 0.f, 0.f, 0.f);
        float a8[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          float t = 0.f;
#pragma unroll
          for (int v = 0; v < 2; ++v) t = fmaf(w4[u][v].x, x4[v].x, fmaf(w4[u][v].y, x4[v].y, fmaf(w4[u][v].z, x4[v].z, fmaf(w4[u][v].w, x4[v].w, t))));
          a8[u] = warp_sum(t);
        }
        if (lane < 8 && o0 + lane < od) {
          float v = a8[0];
#pragma unroll
          for (int u = 1; u < 8; ++u) v = lane == u ? a8[u] : v;
          v += __ldg(bias + o0 + lane);
          if (l < L - 1) v = act_apply(v, p.m.activation);
          xout[o0 + lane] = v;
        }
      }
      __syncthreads();
      continue;
    }
    if (NR == 1 && vec) {
      // single row, other widths: every warp keeps FOUR weight rows in flight (4 output units per iteration, 128-bit loads) and reduces them together
      for (int o0 = warp * 4; o0 < od; o0 += 32) {
        float a4[4] = {0.f, 0.f, 0.f, 0.f};
        for (int k = lane * 4; k < in; k += 128) {
          const float4 x4 = *reinterpret_cast<const float4*>(xin + k);
          float4 w4[4];
#pragma unroll
          for (int u = 0; u < 4; ++u) w4[u] = o0 + u < od ? __ldg(reinterpret_cast<const float4*>(W + (int64_t)(o0 + u) * in + k)) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
          for (int u = 0; u < 4; ++u) a4[u] = fmaf(w4[u].x, x4.x, fmaf(w4[u].y, x4.y, fmaf(w4[u].z, x4.z, fmaf(w4[u].w, x4.w, a4[u]))));
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) a4[u] = warp_sum(a4[u]);
        if (lane < 4 && o0 + lane < od) {
          float v = (lane == 0 ? a4[0] : lane == 1 ? a4[1] : lane == 2 ? a4[2] : a4[3]) + __ldg(bias + o0 + lane);
          if (l < L - 1) v = act_apply(v, p.m.activation);
          xout[o0 + lane] = v;
        }
      }
      __syncthreads();
      continue;
    }
    for (int o = warp; o < od; o += 8) {
      float acc[NR];
#pragma unroll
      for (int r = 0; r < NR; ++r) acc[r] = 0.f;
      const float* wr = W + (int64_t)o * in;
      if (vec) {
        for (int k = lane * 4; k < in; k += 128) {
          const float4 w4 = __ldg(reinterpret_cast<const float4*>(wr + k));
#pragma unroll
          for (int r = 0; r < NR; ++r) {
            const float4 x4 = *reinterpret_cast<const float4*>(xin + r * maxd + k);
            acc[r] = fmaf(w4.x, x4.x, fmaf(w4.y, x4.y, fmaf(w4.z, x4.z, fmaf(w4.w, x4.w, acc[r]))));
          }
        }
      } else {
        for (int k = lane; k < in; k += 32) {
          const float w = __ldg(wr + k);
#pragma unroll
          for (int r = 0; r < NR; ++r) acc[r] = fmaf(w, xin[r * maxd + k], acc[r]);
        }
      }
#pragma unroll
      for (int r = 0; r < NR; ++r) acc[r] = warp_sum(acc[r]);
      if (lane == 0) {
        const float b = __ldg(bias + o);
#pragma unroll
        for (int r = 0; r < NR; ++r) {
          float v = acc[r] + b;
          if (l < L - 1) v = act_apply(v, p.m.activation);
          xout[r * maxd + o] = v;
        }
      }
    }
    __syncthreads();
  }
  const int od = p.m.dims[L];
  const float* fin = bufs[L & 1];
  if (p.tanh_first > 0) {
    const int A = p.tanh_first;
    for (int idx = tid; idx < nr * A; idx += 256) {
      const int r = idx / A, o = idx % A;
      p.out[((int64_t)g * p.n + r0 + r) * A + o] = tanhf(fin[r * maxd + o]);
    }
    return;
  }
  for (int idx = tid; idx < nr * od; idx += 256) {
    const int r = idx / od, o = idx % od;
    p.out[((int64_t)g * p.n + r0 + r) * od + o] = fin[r * maxd + o];
  }
}

// Per-replica hyperparameters of one AdamW launch (il_adam.lr_r / weight_decay_r, il_sac_args.polyak_r). The PR kernel variants build a
// table of every replica's float step size, decay and polyak pair in shared memory once per CTA (the double expressions of the scalar path)
// and look it up per 4-float chunk: replica_floats is a multiple of 4, so a chunk never straddles two replicas.
struct AdamRep {
  const double* lr;
  const double* wd;
  const float* tau;
  int64_t rf;                         // floats per replica
  double inv_rf;
  int nrep;
};
constexpr int ADAM_MAX_REPLICAS = 4096; // shared-memory table: 16 B per replica
__device__ __forceinline__ int adam_replica(int64_t i, const AdamRep& r) {  // i / rf without a 64-bit division
  int64_t q = (int64_t)((double)i * r.inv_rf);
  if (q * r.rf > i) --q;
  else if ((q + 1) * r.rf <= i) ++q;
  return (int)q;
}
__device__ __forceinline__ void adam_fill_table(float4* tab, const AdamRep& r, double bc1, double lr, double wd, float tau) {
  for (int k = threadIdx.x; k < r.nrep; k += blockDim.x) {
    const double l = r.lr ? r.lr[k] : lr, w = r.wd ? r.wd[k] : wd;
    const float t = r.tau ? r.tau[k] : tau;
    tab[k] = make_float4((float)(l / bc1), (float)(1.0 - l * w), t, (float)(1.0 - (double)t));
  }
}

template <bool PR>
__global__ void adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v, const int64_t* __restrict__ step,
                            double lr, double beta1_d, double beta2_d, double eps_d, double wd, int64_t n, float* __restrict__ target, float tau, float one_minus_tau,
                            const AdamRep rep) {
  extern __shared__ float4 adam_tab[];  // PR: [nrep] (step size, decay, tau, 1 - tau)
  __shared__ float s_step_size, s_bc2_sqrt;
  if (threadIdx.x == 0) {  // torch _single_tensor_adam: Python-double scalars, then cast to the tensor dtype
    const double t = (double)*step;
    const double bc1 = 1.0 - pow(beta1_d, t), bc2 = 1.0 - pow(beta2_d, t);
    s_step_size = (float)(lr / bc1);
    s_bc2_sqrt = (float)sqrt(bc2);
  }
  if (PR) adam_fill_table(adam_tab, rep, 1.0 - pow(beta1_d, (double)*step), lr, wd, tau);
  __syncthreads();
  float step_size = s_step_size, decay = (float)(1.0 - lr * wd);
  const float bc2_sqrt = s_bc2_sqrt, w1 = (float)(1.0 - beta1_d), w2 = (float)(1.0 - beta2_d);
  const float beta2 = (float)beta2_d, eps = (float)eps_d;
  bool has_wd = wd != 0.0;
  auto upd = [&](float& pi, float& mi, float& vi, float gi) {
    if (has_wd) pi = __fmul_rn(pi, decay);                                     // param.mul_(1 - lr * weight_decay)
    mi = __fadd_rn(mi, __fmul_rn(w1, __fsub_rn(gi, mi)));                      // exp_avg.lerp_(grad, 1 - beta1)
    vi = __fadd_rn(__fmul_rn(vi, beta2), __fmul_rn(__fmul_rn(w2, gi), gi));    // exp_avg_sq.mul_(beta2).addcmul_(grad, grad, value=1 - beta2)
    const float denom = __fadd_rn(__fdiv_rn(sqrtf(vi), bc2_sqrt), eps);        // (exp_avg_sq.sqrt() / bias_correction2_sqrt).add_(eps)
    pi = __fadd_rn(pi, __fmul_rn(-step_size, __fdiv_rn(mi, denom)));           // param.addcdiv_(exp_avg, denom, value=-step_size)
  };
  auto use_replica = [&](int64_t i) {  // decay == 1 is the scalar path's "weight_decay == 0": both leave the parameter unchanged
    const float4 e = adam_tab[adam_replica(i, rep)];
    step_size = e.x; decay = e.y; has_wd = e.y != 1.f; tau = e.z; one_minus_tau = e.w;
  };
  // n is a multiple of 4 and all buffers are 16-byte aligned (flat parameter layout): 128-bit streams
  const int64_t n4 = n >> 2;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
    if (PR) use_replica(i << 2);
    float4 pv = reinterpret_cast<float4*>(p)[i], mv = reinterpret_cast<float4*>(m)[i], vv = reinterpret_cast<float4*>(v)[i];
    const float4 gv = reinterpret_cast<const float4*>(g)[i];
    upd(pv.x, mv.x, vv.x, gv.x); upd(pv.y, mv.y, vv.y, gv.y); upd(pv.z, mv.z, vv.z, gv.z); upd(pv.w, mv.w, vv.w, gv.w);
    reinterpret_cast<float4*>(p)[i] = pv; reinterpret_cast<float4*>(m)[i] = mv; reinterpret_cast<float4*>(v)[i] = vv;
    if (target) {  // fused update_target_network (models.py:81)
      float4 tv = reinterpret_cast<float4*>(target)[i];
      tv.x = __fadd_rn(__fmul_rn(tv.x, tau), __fmul_rn(one_minus_tau, pv.x)); tv.y = __fadd_rn(__fmul_rn(tv.y, tau), __fmul_rn(one_minus_tau, pv.y));
      tv.z = __fadd_rn(__fmul_rn(tv.z, tau), __fmul_rn(one_minus_tau, pv.z)); tv.w = __fadd_rn(__fmul_rn(tv.w, tau), __fmul_rn(one_minus_tau, pv.w));
      reinterpret_cast<float4*>(target)[i] = tv;
    }
  }
  for (int64_t i = (n4 << 2) + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {  // tail (< 4 elements)
    if (PR) use_replica(i);
    float pi = p[i], mi = m[i], vi = v[i];
    upd(pi, mi, vi, g[i]);
    p[i] = pi; m[i] = mi; v[i] = vi;
    if (target) target[i] = __fadd_rn(__fmul_rn(target[i], tau), __fmul_rn(one_minus_tau, pi));
  }
}

// Same update with TMA staging: persistent CTAs stream 8 KB tiles of every operand into shared memory with 1-D bulk copies
// (cp.async.bulk ... mbarrier::complete_tx, issued by one thread), update in place, and write the results back with bulk stores —
// the LSU only sees shared-memory traffic, global traffic is 128-byte-line bulk transfers on the copy engine path. Double buffered.
constexpr int ADAM_STREAMS = 5;                 // p, g, m, v, target
constexpr int ADAM_CONSUMERS = 256;             // threads 0..255 compute; warp 8 (one elected lane) drives the copy engine
template <int TILE, int STAGES> constexpr int adam_tma_smem() { return STAGES * ADAM_STREAMS * TILE * 4 + 2 * STAGES * 8 + 64; }  // + 16 B per replica (PR)
__device__ __forceinline__ void adam_mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred q;\n\t"
      "ADAM_WAIT:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 q, [%0], %1;\n\t"
      "@q bra ADAM_DONE;\n\t"
      "bra ADAM_WAIT;\n\t"
      "ADAM_DONE:\n\t}" ::"r"(bar), "r"(parity) : "memory");
}
// TILE floats per operand per stage, STAGES-deep ring. Warp-specialised: the copy thread keeps STAGES - 1 tiles of loads in flight and turns
// every computed stage into bulk stores; the 256 compute threads only ever wait on "stage full" and signal "stage computed" (no CTA-wide barrier
// in the loop).
template <int TILE, int STAGES, bool PR>
__global__ void __launch_bounds__(ADAM_CONSUMERS + 32) adam_tma_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v,
                                                                      const int64_t* __restrict__ step, double lr, double beta1_d, double beta2_d, double eps_d, double wd, int64_t n,
                                                                      float* __restrict__ target, float tau, float one_minus_tau, const AdamRep rep) {
  extern __shared__ __align__(128) uint8_t adam_smem[];
  float* buf = reinterpret_cast<float*>(adam_smem);                                  // [stage][stream][TILE]
  const uint32_t smem0 = (uint32_t)__cvta_generic_to_shared(buf);
  const uint32_t full0 = smem0 + (uint32_t)(STAGES * ADAM_STREAMS * TILE * 4), done0 = full0 + 8u * STAGES;  // full[stage] (tx bytes), done[stage] (256 compute threads)
  __shared__ float s_step_size, s_bc2_sqrt;
  const int tid = threadIdx.x;
  if (tid == 0) {
    const double t = (double)*step;
    s_step_size = (float)(lr / (1.0 - pow(beta1_d, t)));
    s_bc2_sqrt = (float)sqrt(1.0 - pow(beta2_d, t));
    for (int s_ = 0; s_ < STAGES; ++s_) {
      asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(full0 + 8u * s_));
      asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(done0 + 8u * s_), "r"(ADAM_CONSUMERS));
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  float4* tab = reinterpret_cast<float4*>(adam_smem + adam_tma_smem<TILE, STAGES>());  // PR: [nrep] behind the ring and the barriers
  if (PR) adam_fill_table(tab, rep, 1.0 - pow(beta1_d, (double)*step), lr, wd, tau);
  __syncthreads();
  const int64_t n_tiles = (n + TILE - 1) / TILE;
  const int n_streams = target ? 5 : 4;
  auto tile_floats = [&](int64_t tile) { const int64_t left = n - tile * TILE; return (int)(left < TILE ? left : TILE); };
  const int64_t my_tiles = blockIdx.x < n_tiles ? (n_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
  if (tid >= ADAM_CONSUMERS) {  // ---- copy warp ----
    if (tid != ADAM_CONSUMERS) return;
    auto issue_loads = [&](int64_t k) {
      const int64_t tile = blockIdx.x + k * gridDim.x;
      const int stage = (int)(k % STAGES);
      const uint32_t bytes = (uint32_t)tile_floats(tile) * 4u, bar = full0 + 8u * stage;
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes * (uint32_t)n_streams) : "memory");
      const float* src[5] = {p, g, m, v, target};
      for (int q = 0; q < n_streams; ++q)
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem0 + (uint32_t)((stage * ADAM_STREAMS + q) * TILE * 4)),
                     "l"(src[q] + tile * TILE), "r"(bytes), "r"(bar) : "memory");
    };
    for (int64_t k = 0; k < STAGES - 1 && k < my_tiles; ++k) issue_loads(k);
    for (int64_t k = 0; k < my_tiles; ++k) {
      const int stage = (int)(k % STAGES);
      const int64_t tile = blockIdx.x + k * gridDim.x;
      if (k + STAGES - 1 < my_tiles) {  // tile k + STAGES - 1 goes into the stage of tile k - 1: its stores (the last committed group) must have left shared memory
        if (k > 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
        issue_loads(k + STAGES - 1);
      }
      adam_mbar_wait(done0 + 8u * stage, (uint32_t)((k / STAGES) & 1));  // stage computed (each compute thread fenced its writes to the async proxy before arriving)
      const uint32_t bytes = (uint32_t)tile_floats(tile) * 4u;
      float* dst[5] = {p, nullptr, m, v, target};
      for (int q = 0; q < n_streams; ++q) {
        if (!dst[q]) continue;
        asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst[q] + tile * TILE), "r"(smem0 + (uint32_t)((stage * ADAM_STREAMS + q) * TILE * 4)), "r"(bytes)
                     : "memory");
      }
      asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    }
    asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");  // all stores complete before the CTA (and its shared memory) goes away
    return;
  }
  // ---- compute threads ----
  float step_size = s_step_size, decay = (float)(1.0 - lr * wd);
  const float bc2_sqrt = s_bc2_sqrt, w1 = (float)(1.0 - beta1_d), w2 = (float)(1.0 - beta2_d), beta2 = (float)beta2_d, eps = (float)eps_d;
  bool has_wd = wd != 0.0;
  auto upd = [&](float& pi, float& mi, float& vi, float gi) {
    if (has_wd) pi = __fmul_rn(pi, decay);
    mi = __fadd_rn(mi, __fmul_rn(w1, __fsub_rn(gi, mi)));
    vi = __fadd_rn(__fmul_rn(vi, beta2), __fmul_rn(__fmul_rn(w2, gi), gi));
    const float denom = __fadd_rn(__fdiv_rn(sqrtf(vi), bc2_sqrt), eps);
    pi = __fadd_rn(pi, __fmul_rn(-step_size, __fdiv_rn(mi, denom)));
  };
  for (int64_t k = 0; k < my_tiles; ++k) {
    const int stage = (int)(k % STAGES);
    const int64_t tile = blockIdx.x + k * gridDim.x;
    adam_mbar_wait(full0 + 8u * stage, (uint32_t)((k / STAGES) & 1));
    const int nf4 = tile_floats(tile) >> 2;
    float4* sp = reinterpret_cast<float4*>(buf + (stage * ADAM_STREAMS + 0) * TILE);
    const float4* sg = reinterpret_cast<const float4*>(buf + (stage * ADAM_STREAMS + 1) * TILE);
    float4* smm = reinterpret_cast<float4*>(buf + (stage * ADAM_STREAMS + 2) * TILE);
    float4* sv = reinterpret_cast<float4*>(buf + (stage * ADAM_STREAMS + 3) * TILE);
    float4* stg = reinterpret_cast<float4*>(buf + (stage * ADAM_STREAMS + 4) * TILE);
    for (int i = tid; i < nf4; i += ADAM_CONSUMERS) {
      if (PR) {
        const float4 e = tab[adam_replica(tile * TILE + 4 * i, rep)];
        step_size = e.x; decay = e.y; has_wd = e.y != 1.f; tau = e.z; one_minus_tau = e.w;
      }
      float4 pv = sp[i], mv = smm[i], vv = sv[i];
      const float4 gv = sg[i];
      upd(pv.x, mv.x, vv.x, gv.x); upd(pv.y, mv.y, vv.y, gv.y); upd(pv.z, mv.z, vv.z, gv.z); upd(pv.w, mv.w, vv.w, gv.w);
      sp[i] = pv; smm[i] = mv; sv[i] = vv;
      if (target) {  // fused update_target_network (models.py:81)
        float4 tv = stg[i];
        tv.x = __fadd_rn(__fmul_rn(tv.x, tau), __fmul_rn(one_minus_tau, pv.x)); tv.y = __fadd_rn(__fmul_rn(tv.y, tau), __fmul_rn(one_minus_tau, pv.y));
        tv.z = __fadd_rn(__fmul_rn(tv.z, tau), __fmul_rn(one_minus_tau, pv.z)); tv.w = __fadd_rn(__fmul_rn(tv.w, tau), __fmul_rn(one_minus_tau, pv.w));
        stg[i] = tv;
      }
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy writes -> visible to the bulk-copy engine
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(done0 + 8u * stage) : "memory");
  }
}

template <int TILE, int STAGES>
static int launch_adam_tma(il_handle* h, int ctas_per_sm, float* params, const float* grads, const il_adam* opt, int64_t n, cudaStream_t stream, float* polyak_target, float polyak_factor,
                           const AdamRep& rep) {
  static bool attr_set = false;
  if (!attr_set) {
    IL_CUDA(cudaFuncSetAttribute(adam_tma_kernel<TILE, STAGES, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, adam_tma_smem<TILE, STAGES>()));
    IL_CUDA(cudaFuncSetAttribute(adam_tma_kernel<TILE, STAGES, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, adam_tma_smem<TILE, STAGES>() + 16 * ADAM_MAX_REPLICAS));
    attr_set = true;
  }
  if (rep.nrep) IL_LAUNCH(h, (adam_tma_kernel<TILE, STAGES, true>), h->sm_count * ctas_per_sm, ADAM_CONSUMERS + 32, (size_t)(adam_tma_smem<TILE, STAGES>() + 16 * rep.nrep), stream, params, grads,
                          opt->m, opt->v, opt->step, opt->lr, opt->beta1, opt->beta2, opt->eps, opt->weight_decay, n, polyak_target, polyak_factor, (float)(1.0 - (double)polyak_factor), rep);
  else IL_LAUNCH(h, (adam_tma_kernel<TILE, STAGES, false>), h->sm_count * ctas_per_sm, ADAM_CONSUMERS + 32, (adam_tma_smem<TILE, STAGES>()), stream, params, grads, opt->m, opt->v, opt->step, opt->lr,
                 opt->beta1, opt->beta2, opt->eps, opt->weight_decay, n, polyak_target, polyak_factor, (float)(1.0 - (double)polyak_factor), rep);
  return 0;
}
constexpr int ADAM_TMA_MIN_TILES = 4096;        // floats per CTA-iteration below which the plain kernel is used


// ---- fused backward of the linear head + last hidden activation (one pass over the hidden output) -----------------------------------
// For the last layer out = Y W_L^T + b_L (N_h <= 8 units) with Y = relu(Z) [n, H]:
//   dZ[b, o]   = (sum_j dOut[b, j] W_L[j, o]) * 1[Y[b, o] > 0]        (was: K-thin GEMM with mask epilogue, reads Y, writes dZ)
//   dW_L[j, o] = sum_b dOut[b, j] Y[b, o],  db_L[j] = sum_b dOut[b, j]  (was: streaming TN kernel, reads Y again)
//   db_{L-1}[o] = sum_b dZ[b, o]                                        (was: column-sum kernel, reads dZ again)
// One CTA per (net, 256 hidden columns) streams Y once and writes dZ once; thread = 4 columns x every 4th row, W_L columns in registers,
// cross-row-group reduction through shared memory in a fixed order (deterministic).
template <int NH>  // compile-time bound on the head width (1: critic, HB_MAXN: actor) — the weight / gradient register tiles and the FMA count scale with it
__global__ void __launch_bounds__(256, 2) head_backward_kernel(const HeadBwdArgs p) {
  extern __shared__ __align__(16) float hb_sm[];   // dOut [n][HB_MAXN] (zero padded), then the reduction scratch [4][HB_MAXN * 4 + 4][64]
  const int g = blockIdx.y, n0 = blockIdx.x * 256, tid = threadIdx.x, tc = tid & 63, tr = tid >> 6, col = n0 + tc * 4;
  float* dos = hb_sm;
  float* red = hb_sm + p.n * HB_MAXN;
  const float* dout = p.dout + (int64_t)(g / p.dout_gdiv) * p.dout_gs;
  const bool active = col < p.H;
  const float* Y = p.y + (int64_t)g * p.y_gs + col;
  float4 yv[4], yn[4];
  auto fetch = [&](float4 (&dst)[4], int b0) {  // rows b0, b0 + 4, b0 + 8, b0 + 12
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int b = b0 + 4 * u;
      dst[u] = (active && b < p.n) ? __ldg(reinterpret_cast<const float4*>(Y + (int64_t)b * p.H)) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  };
  fetch(yv, tr);  // in flight while dOut is staged
  for (int i = tid; i < p.n * HB_MAXN; i += 256) {
    const int b = i / HB_MAXN, j = i % HB_MAXN;
    dos[i] = j < p.Nh ? __ldg(dout + (int64_t)b * p.ld_dout + j) : 0.f;
  }
  float4 w[NH];
#pragma unroll
  for (int j = 0; j < NH; ++j) w[j] = (active && j < p.Nh) ? __ldg(reinterpret_cast<const float4*>(p.w + (int64_t)g * p.w_gs + (int64_t)j * p.H + col)) : make_float4(0.f, 0.f, 0.f, 0.f);
  __syncthreads();
  float4 dw[NH], cs = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
  for (int j = 0; j < NH; ++j) dw[j] = make_float4(0.f, 0.f, 0.f, 0.f);
  if (active) {
    float* DZ = p.dz + (int64_t)g * p.dz_gs + col;
    for (int b0 = tr; b0 < p.n; b0 += 16) {
      fetch(yn, b0 + 16);  // the next 4 rows are in flight while these 4 are consumed
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int b = b0 + 4 * u;
        if (b >= p.n) continue;
        float dj[NH];
        if (NH == 1) dj[0] = dos[b * HB_MAXN];
        else {
          const float4 d0 = *reinterpret_cast<const float4*>(dos + b * HB_MAXN), d1 = *reinterpret_cast<const float4*>(dos + b * HB_MAXN + 4);
          const float t[8] = {d0.x, d0.y, d0.z, d0.w, d1.x, d1.y, d1.z, d1.w};
#pragma unroll
          for (int j = 0; j < NH; ++j) dj[j] = t[j];
        }
        float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int j = 0; j < NH; ++j) {
          z.x = fmaf(dj[j], w[j].x, z.x); z.y = fmaf(dj[j], w[j].y, z.y); z.z = fmaf(dj[j], w[j].z, z.z); z.w = fmaf(dj[j], w[j].w, z.w);
          dw[j].x = fmaf(dj[j], yv[u].x, dw[j].x); dw[j].y = fmaf(dj[j], yv[u].y, dw[j].y); dw[j].z = fmaf(dj[j], yv[u].z, dw[j].z); dw[j].w = fmaf(dj[j], yv[u].w, dw[j].w);
        }
        z.x = yv[u].x > 0.f ? z.x : 0.f; z.y = yv[u].y > 0.f ? z.y : 0.f; z.z = yv[u].z > 0.f ? z.z : 0.f; z.w = yv[u].w > 0.f ? z.w : 0.f;
        cs.x += z.x; cs.y += z.y; cs.z += z.z; cs.w += z.w;
        *reinterpret_cast<float4*>(DZ + (int64_t)b * p.H) = z;
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) yv[u] = yn[u];
    }
  }
  // reduce the 4 row groups: red[tr][slot][tc] (slot = j for dW_L rows, HB_MAXN for the column sum), float4 per entry
  float4* r4 = reinterpret_cast<float4*>(red);
#pragma unroll
  for (int j = 0; j < NH; ++j) r4[(tr * (HB_MAXN + 1) + j) * 64 + tc] = dw[j];
  r4[(tr * (HB_MAXN + 1) + HB_MAXN) * 64 + tc] = cs;
  __syncthreads();
  if (tr == 0 && active) {
#pragma unroll
    for (int j = 0; j <= HB_MAXN; ++j) {
      if ((j < NH && j < p.Nh) || j == HB_MAXN) {
        float4 a = r4[(0 * (HB_MAXN + 1) + j) * 64 + tc];
#pragma unroll
        for (int q = 1; q < 4; ++q) {
          const float4 t = r4[(q * (HB_MAXN + 1) + j) * 64 + tc];
          a.x += t.x; a.y += t.y; a.z += t.z; a.w += t.w;
        }
        float* dst = j == HB_MAXN ? p.db_prev + (int64_t)g * p.g_gs + col : p.dw + (int64_t)g * p.g_gs + (int64_t)j * p.H + col;
        *reinterpret_cast<float4*>(dst) = a;
      }
    }
  }
  if (blockIdx.x == 0 && tid < p.Nh) {  // db_L[j] = sum_b dOut[b, j]
    float sacc = 0.f;
    for (int b = 0; b < p.n; ++b) sacc += dos[b * HB_MAXN + tid];
    p.db[(int64_t)g * p.g_gs + tid] = sacc;
  }
}

__global__ void tick_kernel(int64_t* s0, int64_t* s1, int64_t* s2) {
  if (s0) *s0 += 1;
  if (s1) *s1 += 1;
  if (s2) *s2 += 1;
}

__global__ void polyak_kernel(float* __restrict__ t, const float* __restrict__ o, int64_t n, float tau, float one_minus_tau) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    t[i] = __fadd_rn(__fmul_rn(t[i], tau), __fmul_rn(one_minus_tau, o[i]));  // models.py:81: mul_(tau).add_((1 - tau) * param)
}

// q1/q2 split of the twin output [2R, n] -> q1 [R, n], q2 [R, n]
__global__ void split_twin_kernel(const float* __restrict__ q, float* __restrict__ q1, float* __restrict__ q2, int R, int n) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (int64_t)R * n) return;
  const int r = (int)(i / n), b = (int)(i % n);
  if (q1) q1[i] = q[((int64_t)2 * r) * n + b];
  if (q2) q2[i] = q[((int64_t)2 * r + 1) * n + b];
}

// X[r, i, :] = cat(state[r, i, :S], action[r, i, :A])   (models.py:20-21)
__global__ void concat_kernel(const float* __restrict__ s, int64_t s_rs, int ld_s, int S, const float* __restrict__ a, int64_t a_rs, int ld_a, int A,
                              float* __restrict__ x, int R, int n) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int d = S + A;
  if (idx >= (int64_t)R * n * d) return;
  const int j = (int)(idx % d);
  const int64_t row = idx / d;
  const int r = (int)(row / n), i = (int)(row % n);
  x[idx] = j < S ? s[(int64_t)r * s_rs + (int64_t)i * ld_s + j] : a[(int64_t)r * a_rs + (int64_t)i * ld_a + (j - S)];
}

inline int ew_blocks(int64_t n, int threads, int sm_count) {
  int64_t b = (n + threads - 1) / threads;
  const int64_t cap = (int64_t)sm_count * 16;
  return (int)(b < 1 ? 1 : (b > cap ? cap : b));
}

}  // namespace

int launch_actor_head(il_handle* h, const HeadFwdArgs& a, cudaStream_t stream) {
  const int64_t rows = (int64_t)a.R * a.n;
  IL_LAUNCH(h, actor_head_kernel, (unsigned)((rows + 127) / 128), 128, 0, stream, a);
  return 0;
}

int launch_adam(il_handle* h, float* params, const float* grads, const il_adam* opt, int64_t n, cudaStream_t stream, float* polyak_target, float polyak_factor, const float* polyak_r) {
  IL_CHECK(opt->m && opt->v && opt->step, "adam: null state");
  IL_CHECK(((reinterpret_cast<uintptr_t>(params) | reinterpret_cast<uintptr_t>(grads) | reinterpret_cast<uintptr_t>(opt->m) | reinterpret_cast<uintptr_t>(opt->v) |
             reinterpret_cast<uintptr_t>(polyak_target)) & 15) == 0, "adam: buffers must be 16-byte aligned");
  AdamRep rep{opt->lr_r, opt->weight_decay_r, polyak_target ? polyak_r : nullptr, opt->replica_floats, 0.0, 0};
  if (rep.lr || rep.wd || rep.tau) {  // per-replica hyperparameters: the PR variants (the default step keeps the scalar kernels)
    IL_CHECK(rep.rf > 0 && rep.rf % 4 == 0 && n % rep.rf == 0, "adam: per-replica hyperparameters need replica_floats (%lld) > 0, a multiple of 4 dividing n = %lld", (long long)rep.rf,
             (long long)n);
    rep.nrep = (int)(n / rep.rf);
    rep.inv_rf = 1.0 / (double)rep.rf;
    IL_CHECK(rep.nrep <= ADAM_MAX_REPLICAS, "adam: %d replicas with per-replica hyperparameters exceed %d", rep.nrep, ADAM_MAX_REPLICAS);
  }
  if (h->adam_tma && n % 4 == 0 && n >= (int64_t)ADAM_TMA_MIN_TILES * h->sm_count * 2) {  // large flat buffers: TMA-staged streaming variant
    // Isolated launches on the bench buffers (profiles/r2_adam_variants.jsonl; copy = 6.5-6.6 TB/s): every geometry is within 8 % of the copy rate, the
    // 1-CTA-per-SM ones (4096 x 2, 2048 x 4) are the fastest alone (6.55 TB/s) — but inside the step the 2-CTA-per-SM 2048 x 2 ring wins (6.49 vs 6.59
    // ms / step, A/B in one gpurun call): its CTAs co-reside with the tail of the previous kernel and the head of the next.
    const int variant = h->adam_tma;
    switch (variant) {  // (tile floats, stages, CTAs per SM): 20 B/float of shared memory per stage
      case 2: return launch_adam_tma<4096, 2>(h, 1, params, grads, opt, n, stream, polyak_target, polyak_factor, rep);
      case 3: return launch_adam_tma<2048, 3>(h, 1, params, grads, opt, n, stream, polyak_target, polyak_factor, rep);
      case 4: return launch_adam_tma<1024, 4>(h, 2, params, grads, opt, n, stream, polyak_target, polyak_factor, rep);
      case 5: return launch_adam_tma<1024, 3>(h, 3, params, grads, opt, n, stream, polyak_target, polyak_factor, rep);
      case 6: return launch_adam_tma<512, 4>(h, 4, params, grads, opt, n, stream, polyak_target, polyak_factor, rep);
      case 7: return launch_adam_tma<2048, 4>(h, 1, params, grads, opt, n, stream, polyak_target, polyak_factor, rep);
      default: return launch_adam_tma<2048, 2>(h, 2, params, grads, opt, n, stream, polyak_target, polyak_factor, rep);
    }
  }
  if (rep.nrep) {
    static bool attr_set = false;
    if (!attr_set) { IL_CUDA(cudaFuncSetAttribute(adam_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 16 * ADAM_MAX_REPLICAS)); attr_set = true; }
    IL_LAUNCH(h, adam_kernel<true>, ew_blocks(n / 4 + 1, 256, h->sm_count), 256, (size_t)16 * rep.nrep, stream, params, grads, opt->m, opt->v, opt->step, opt->lr, opt->beta1, opt->beta2,
              opt->eps, opt->weight_decay, n, polyak_target, polyak_factor, (float)(1.0 - (double)polyak_factor), rep);
    return 0;
  }
  IL_LAUNCH(h, adam_kernel<false>, ew_blocks(n / 4 + 1, 256, h->sm_count), 256, 0, stream, params, grads, opt->m, opt->v, opt->step, opt->lr, opt->beta1, opt->beta2, opt->eps,
            opt->weight_decay, n, polyak_target, polyak_factor, (float)(1.0 - (double)polyak_factor), rep);
  return 0;
}

namespace {
// Input-gradient pass through the linear head when the last hidden activation exists only as ReLU sign bits (MLP_KEEP_MASKS):
// dZ[b, o] = (sum_j dOut[b, j] W_L[j, o]) * bit(b, o). One CTA per (net, 256 hidden columns): thread = 4 columns x every 4th row, W_L columns in
// registers, 128-bit stores; reads 1/32 of what the fp32 mask would cost.
template <int NH, int U>  // NH: compile-time bound on the head width; U rows in flight per thread (all their word / dOut loads are issued before the first store)
__global__ void __launch_bounds__(256) head_dx_bits_kernel(const HeadBwdArgs p, const uint32_t* __restrict__ bits, int64_t bits_gs) {
  const int g = blockIdx.y, tid = threadIdx.x, tc = tid & 63, tr = tid >> 6, col = blockIdx.x * 256 + tc * 4;
  if (col >= p.H) return;
  const float* __restrict__ dout = p.dout + (int64_t)(g / p.dout_gdiv) * p.dout_gs;
  const uint32_t* __restrict__ bw = bits + (int64_t)g * bits_gs + (col >> 5);
  const int sh = col & 31, wpr = p.H >> 5;
  float4 w[NH];
#pragma unroll
  for (int j = 0; j < NH; ++j) w[j] = j < p.Nh ? __ldg(reinterpret_cast<const float4*>(p.w + (int64_t)g * p.w_gs + (int64_t)j * p.H + col)) : make_float4(0.f, 0.f, 0.f, 0.f);
  float* __restrict__ dz = p.dz + (int64_t)g * p.dz_gs + col;
  for (int b0 = tr; b0 < p.n; b0 += 4 * U) {
    uint32_t m[U];
    float d[U][NH];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int b = b0 + 4 * u;
      m[u] = b < p.n ? __ldg(bw + (int64_t)b * wpr) >> sh : 0u;
#pragma unroll
      for (int j = 0; j < NH; ++j) d[u][j] = (j < p.Nh && b < p.n) ? __ldg(dout + (int64_t)b * p.ld_dout + j) : 0.f;
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int b = b0 + 4 * u;
      if (b >= p.n) break;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int j = 0; j < NH; ++j)
        if (j < p.Nh) { v.x = fmaf(d[u][j], w[j].x, v.x); v.y = fmaf(d[u][j], w[j].y, v.y); v.z = fmaf(d[u][j], w[j].z, v.z); v.w = fmaf(d[u][j], w[j].w, v.w); }
      v.x = m[u] & 1u ? v.x : 0.f; v.y = m[u] & 2u ? v.y : 0.f; v.z = m[u] & 4u ? v.z : 0.f; v.w = m[u] & 8u ? v.w : 0.f;
      *reinterpret_cast<float4*>(dz + (int64_t)b * p.H) = v;
    }
  }
}
}  // namespace

int launch_head_dx_bits(il_handle* h, const HeadBwdArgs& a, const uint32_t* bits, int64_t bits_gs, int G, cudaStream_t stream) {
  IL_CHECK(a.H % 32 == 0 && a.Nh <= HB_MAXN && (reinterpret_cast<uintptr_t>(a.w) & 15) == 0 && a.w_gs % 4 == 0 && (reinterpret_cast<uintptr_t>(a.dz) & 15) == 0 && a.dz_gs % 4 == 0,
           "head_dx_bits: H=%d Nh=%d or unaligned buffers", a.H, a.Nh);
  if (a.Nh == 1) IL_LAUNCH(h, (head_dx_bits_kernel<1, 8>), dim3((a.H + 255) / 256, G), 256, 0, stream, a, bits, bits_gs);
  else IL_LAUNCH(h, (head_dx_bits_kernel<HB_MAXN, 4>), dim3((a.H + 255) / 256, G), 256, 0, stream, a, bits, bits_gs);
  return 0;
}

int launch_head_backward(il_handle* h, const HeadBwdArgs& a, int G, cudaStream_t stream) {
  const size_t smem = ((size_t)a.n * HB_MAXN + 4 * (HB_MAXN + 1) * 64 * 4) * sizeof(float);
  if (a.Nh == 1) IL_LAUNCH(h, head_backward_kernel<1>, dim3((a.H + 255) / 256, G), 256, smem, stream, a);
  else IL_LAUNCH(h, head_backward_kernel<HB_MAXN>, dim3((a.H + 255) / 256, G), 256, smem, stream, a);
  return 0;
}

int mlp_init() {
  IL_CUDA(cudaFuncSetAttribute(head_backward_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (1024 * HB_MAXN + 4 * (HB_MAXN + 1) * 64 * 4) * 4));
  IL_CUDA(cudaFuncSetAttribute(head_backward_kernel<HB_MAXN>, cudaFuncAttributeMaxDynamicSharedMemorySize, (1024 * HB_MAXN + 4 * (HB_MAXN + 1) * 64 * 4) * 4));
  return 0;
}

int launch_tick(il_handle* h, int64_t* s0, int64_t* s1, int64_t* s2, cudaStream_t stream) {
  IL_LAUNCH(h, tick_kernel, 1, 1, 0, stream, s0, s1, s2);
  return 0;
}

// n <= 32 rows per net: the fused whole-MLP kernel (parameter-bandwidth bound) instead of per-layer GEMMs.
int mlp_small_forward(il_handle* h, const il_mlp* m, int G, int n, MatView X, float* out, cudaStream_t stream, int tanh_first) {
  SmallFwdArgs a;
  a.m = *m; a.o = mlp_offsets(m->dims, m->n_layers);
  a.X = X.ptr; a.x_gs = X.gs; a.x_gdiv = X.gdiv; a.ldx = X.ld; a.n = n; a.out = out; a.tanh_first = tanh_first;
  int maxd = 4;
  for (int l = 0; l <= m->n_layers; ++l) maxd = m->dims[l] > maxd ? m->dims[l] : maxd;
  a.maxd = (maxd + 3) / 4 * 4;
  if (n == 1) {
    IL_LAUNCH(h, mlp_small_forward_kernel<1>, dim3(G, 1), 256, (size_t)2 * 1 * a.maxd * 4, stream, a);
  } else {
    IL_CHECK((size_t)2 * 8 * a.maxd * 4 <= 48 * 1024, "mlp_small_forward: layer width %d too large", maxd);
    IL_LAUNCH(h, mlp_small_forward_kernel<8>, dim3(G, (n + 7) / 8), 256, (size_t)2 * 8 * a.maxd * 4, stream, a);
  }
  return 0;
}

extern "C" int il_adam_step(il_handle* h, float* params, const float* grads, const il_adam* opt, int64_t n, void* stream) {
  IL_CHECK(h && params && grads && opt, "il_adam_step: null argument");
  IL_TRY(launch_tick(h, opt->step, nullptr, nullptr, (cudaStream_t)stream));
  return launch_adam(h, params, grads, opt, n, (cudaStream_t)stream);
}

extern "C" int il_adam_step_polyak(il_handle* h, float* params, const float* grads, const il_adam* opt, int64_t n, float* target, float polyak_factor, void* stream) {
  IL_CHECK(h && params && grads && opt && target, "il_adam_step_polyak: null argument");
  IL_TRY(launch_tick(h, opt->step, nullptr, nullptr, (cudaStream_t)stream));
  return launch_adam(h, params, grads, opt, n, (cudaStream_t)stream, target, polyak_factor);
}

extern "C" int il_polyak(il_handle* h, float* target, const float* online, int64_t n, float polyak_factor, void* stream) {
  IL_CHECK(h && target && online && n >= 0, "il_polyak: bad argument");
  if (n == 0) return 0;
  IL_LAUNCH(h, polyak_kernel, ew_blocks(n, 256, h->sm_count), 256, 0, (cudaStream_t)stream, target, online, n, polyak_factor, (float)(1.0 - (double)polyak_factor));
  return 0;
}

// ---- SoftActor ------------------------------------------------------------------------------------------------
extern "C" int64_t il_actor_workspace_bytes(const il_mlp* actor, int R, int n) {
  return mlp_acts_bytes(actor, R, n) + il_align_up((int64_t)R * n * actor->dims[actor->n_layers] * 4, 256);
}

extern "C" int il_actor_forward(il_handle* h, const il_mlp* actor, int R, int n, const float* states, int64_t states_rs, int ld_states, const float* eps,
                                const float* given_action, float* action, float* log_prob, float* mean, float* log_std, void* workspace, int64_t workspace_bytes,
                                void* stream) {
  IL_CHECK(h && states && workspace, "il_actor_forward: null argument");
  IL_TRY(mlp_validate(actor, "il_actor_forward"));
  IL_CHECK(R > 0 && n > 0, "il_actor_forward: R=%d n=%d", R, n);
  const int out = actor->dims[actor->n_layers];
  IL_CHECK(out % 2 == 0, "il_actor_forward: head size %d is not 2*A", out);
  IL_CHECK(workspace_bytes >= il_actor_workspace_bytes(actor, R, n), "il_actor_forward: workspace too small");
  MlpActs acts;
  char* ws = mlp_acts_carve(actor, R, n, static_cast<char*>(workspace), &acts);
  float* head = reinterpret_cast<float*>(ws);
  if (n <= 32) IL_TRY(mlp_small_forward(h, actor, R, n, MatView{states, states_rs, 1, ld_states}, head, (cudaStream_t)stream));
  else IL_TRY(mlp_forward(h, actor, R, n, MatView{states, states_rs, 1, ld_states}, acts, head, (int64_t)n * out, out, (cudaStream_t)stream, MLP_KEEP_NONE));
  HeadFwdArgs a{};
  a.head = head; a.eps = eps; a.given = given_action;
  a.action = action; a.action_rs = (int64_t)n * (out / 2); a.ld_action = out / 2;
  a.log_prob = log_prob; a.mean = mean; a.log_std = log_std;
  a.R = R; a.n = n; a.A = out / 2;
  return launch_actor_head(h, a, (cudaStream_t)stream);
}

// ---- TwinCritic -----------------------------------------------------------------------------------------------
extern "C" int64_t il_critic_workspace_bytes(const il_mlp* critic, int R, int n) {
  return mlp_acts_bytes(critic, 2 * R, n) + il_align_up((int64_t)R * n * critic->dims[0] * 4, 256) + il_align_up((int64_t)2 * R * n * 4, 256);
}

extern "C" int il_critic_forward(il_handle* h, const il_mlp* twin, int R, int n, int S, const float* states, int64_t states_rs, int ld_states, const float* actions,
                                 int64_t actions_rs, int ld_actions, float* q1, float* q2, void* workspace, int64_t workspace_bytes, void* stream) {
  IL_CHECK(h && states && actions && workspace, "il_critic_forward: null argument");
  IL_TRY(mlp_validate(twin, "il_critic_forward"));
  IL_CHECK(twin->dims[twin->n_layers] == 1, "il_critic_forward: critic head must have one output");
  IL_CHECK(workspace_bytes >= il_critic_workspace_bytes(twin, R, n), "il_critic_forward: workspace too small");
  cudaStream_t st = (cudaStream_t)stream;
  const int d = twin->dims[0];
  MlpActs acts;
  char* ws = mlp_acts_carve(twin, 2 * R, n, static_cast<char*>(workspace), &acts);
  float* X = reinterpret_cast<float*>(ws);
  ws += il_align_up((int64_t)R * n * d * 4, 256);
  float* q = reinterpret_cast<float*>(ws);
  const int A = d - S;
  IL_CHECK(S > 0 && A > 0, "il_critic_forward: S=%d with input width %d", S, d);
  const int64_t total = (int64_t)R * n * d;
  IL_LAUNCH(h, concat_kernel, (unsigned)((total + 255) / 256), 256, 0, st, states, states_rs, ld_states, S, actions, actions_rs, ld_actions, A, X, R, n);
  IL_TRY(mlp_forward(h, twin, 2 * R, n, MatView{X, (int64_t)n * d, 2, d}, acts, q, (int64_t)n, 1, st, MLP_KEEP_NONE));
  IL_LAUNCH(h, split_twin_kernel, (unsigned)(((int64_t)R * n + 255) / 256), 256, 0, st, q, q1, q2, R, n);
  return 0;
}
