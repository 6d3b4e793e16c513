// Library plumbing: handle, error reporting, layout queries, Philox fills.
#include "common.cuh"
#include <cstdlib>

thread_local char g_il_error[512] = "";
int gail_init();
int gmmil_pwil_init();
int gemm_init();
int mlp_init();

extern "C" const char* il_last_error(void) { return g_il_error; }
extern "C" int il_version(void) { return 102; }

extern "C" int il_create(int device, il_handle** out) {
  IL_CHECK(out != nullptr, "il_create: null out");
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0) IL_FAIL("il_create: no CUDA device (%s); this library has no CPU fallback", cudaGetErrorString(e));
  IL_CHECK(device >= 0 && device < count, "il_create: device %d out of range (%d devices)", device, count);
  cudaDeviceProp prop;
  IL_CUDA(cudaGetDeviceProperties(&prop, device));
  IL_CHECK(prop.major == 10, "il_create: device %d is sm_%d%d; this library is built for sm_100a (B200) only", device, prop.major, prop.minor);
  IL_CUDA(cudaSetDevice(device));
  IL_TRY(gail_init());
  IL_TRY(gmmil_pwil_init());
  IL_TRY(tc_gemm_init());
  IL_TRY(gemm_init());
  IL_TRY(mlp_init());
  il_handle* h = new il_handle();
  h->device = device;
  h->sm_count = prop.multiProcessorCount;
  h->gemm_mode = IL_GEMM_FP32;
  {
    const char* e = getenv("IL_TC_PAIRS");
    h->tc_pairs = (e && e[0] == '0') ? 0 : 1;
    h->tc_pair_groups = 0;
    const char* wt = getenv("IL_WIDE_TN");
    h->wide_tn = (wt && wt[0] == '0') ? 0 : 1;
    const char* ff = getenv("IL_FIRST_LAYER_FAST");
    h->first_layer_fast = ff ? atoi(ff) : 2;  // 0 generic K-thin kernel, 1 FFMA2 kernel with shared-memory weights, 2 register-resident weights (N == 256)
    const char* mb = getenv("IL_MASK_BITS");
    h->mask_bits = mb ? atoi(mb) : 2;  // 0: fp32 activations as masks; 1: sign-bit words; 2: + the input-gradient slice fused into the masked dX launch
    const char* hf = getenv("IL_HEAD_FUSED");
    h->head_fused = (hf && hf[0] == '0') ? 0 : 1;
    const char* ds = getenv("IL_DEBUG_SYNC");
    h->debug_sync = (ds && ds[0] == '1') ? 1 : 0;
    // AdamW with TMA staging (cp.async.bulk tiles through shared memory): bit-identical to the plain kernel, 7.309 -> 7.285 ms / step in an
    // A/B inside one gpurun call (profiles/README.md) -> on by default for the large flat buffers
    const char* at = getenv("IL_ADAM_TMA");
    h->adam_tma = at ? atoi(at) : 1;  // 0 plain kernel, 1 auto (ring geometry by stream count), 2..7 fixed geometries (scripts/adam_bench.py)
    const char* gt = getenv("IL_GAIL_TILED");
    h->gail_tiled = (gt && gt[0] == '0') ? 0 : 1;
    // first MLP layer computed inside the producers of the tcgen05 launch: measured 7.64 vs 7.59 ms / step against the separate
    // K-thin launch (the CUDA-core work makes the 13-warp CTA issue-bound, profiles/README.md) -> off by default, kept for A/B
    const char* fl = getenv("IL_TC_FUSE_L1");
    h->tc_fuse_l1 = (fl && fl[0] == '1') ? 1 : 0;
    const char* th = getenv("IL_THIN_HOIST");
    h->thin_hoist = (th && th[0] == '0') ? 0 : 1;  // default on: +2.3 % step throughput (A/B in one gpurun call, parity suite green both ways)
  }
  h->launches = 0;
  h->profiling = 0;
  h->profiled_bytes = 0.0;
  h->eval_graph = nullptr;
  h->build_stream = nullptr;
  *out = h;
  return 0;
}

extern "C" int il_destroy(il_handle* h) {
  if (h) il_eval_release(h);
  if (h && h->build_stream) cudaStreamDestroy(h->build_stream);
  delete h;
  return 0;
}

extern "C" int il_set_gemm_mode(il_handle* h, int mode) {
  IL_CHECK(h, "il_set_gemm_mode: null handle");
  IL_CHECK(mode >= IL_GEMM_FP32 && mode <= IL_GEMM_TF32, "il_set_gemm_mode: bad mode %d", mode);
  h->gemm_mode = mode;
  return 0;
}

extern "C" int64_t il_launch_count(il_handle* h) { return h ? h->launches : -1; }

extern "C" int il_set_option(il_handle* h, const char* name, int value) {
  IL_CHECK(h && name, "il_set_option: null argument");
  if (!strcmp(name, "tc_fuse_l1")) h->tc_fuse_l1 = value;
  else if (!strcmp(name, "gail_tiled")) h->gail_tiled = value;
  else if (!strcmp(name, "adam_tma")) h->adam_tma = value;
  else if (!strcmp(name, "head_fused")) h->head_fused = value;
  else if (!strcmp(name, "mask_bits")) h->mask_bits = value;
  else if (!strcmp(name, "first_layer_fast")) h->first_layer_fast = value;
  else if (!strcmp(name, "wide_tn")) h->wide_tn = value;
  else if (!strcmp(name, "tc_pairs")) { h->tc_pairs = value; h->tc_pair_groups = 0; }
  else if (!strcmp(name, "thin_hoist")) h->thin_hoist = value;
  else IL_FAIL("il_set_option: unknown option '%s'", name);
  return 0;
}

extern "C" int il_struct_sizes(int32_t* out) {
  out[0] = (int32_t)sizeof(il_mlp);
  out[1] = (int32_t)sizeof(il_adam);
  out[2] = (int32_t)sizeof(il_batch);
  out[3] = (int32_t)sizeof(il_replay);
  out[4] = (int32_t)sizeof(il_sac_args);
  out[5] = (int32_t)sizeof(il_gail);
  out[6] = (int32_t)sizeof(il_gail_update_args);
  out[7] = (int32_t)sizeof(il_pwil);
  out[8] = (int32_t)sizeof(il_env);
  out[9] = (int32_t)sizeof(il_bc_args);
  out[10] = (int32_t)sizeof(il_eval_args);
  out[11] = (int32_t)sizeof(il_gailx);
  out[12] = (int32_t)sizeof(il_gailx_update_args);
  out[13] = (int32_t)sizeof(il_red);
  out[14] = (int32_t)sizeof(il_red_update_args);
  return 0;
}

extern "C" int il_mlp_param_offsets(const int32_t* dims, int n_layers, int64_t* w_off, int64_t* b_off, int64_t* total) {
  IL_CHECK(dims && n_layers >= 1 && n_layers <= IL_MAX_LAYERS, "il_mlp_param_offsets: bad arguments");
  const MlpOffsets o = mlp_offsets(dims, n_layers);
  for (int l = 0; l < n_layers; ++l) {
    if (w_off) w_off[l] = o.w[l];
    if (b_off) b_off[l] = o.b[l];
  }
  if (total) *total = o.total;
  return 0;
}

extern "C" int il_row_layout(int S, int A, int32_t* off, int32_t* row_len) {
  IL_CHECK(S > 0 && A > 0, "il_row_layout: S=%d A=%d", S, A);
  const RowLayout L = row_layout(S, A);
  if (off) {
    off[0] = L.state; off[1] = L.action; off[2] = L.reward; off[3] = L.next_state;
    off[4] = L.terminal; off[5] = L.timeout; off[6] = L.weight; off[7] = L.step;
  }
  if (row_len) *row_len = L.len;
  return 0;
}

namespace {

// 4 outputs per Philox call; element i uses counter (base + i / 4), lane i % 4.
__global__ void fill_kernel(float* __restrict__ out, int64_t n, uint64_t seed, uint64_t stream_id, const uint64_t* __restrict__ counter, int normal) {
  const uint64_t base = counter ? *counter : 0ull;
  const uint2 key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
  for (int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; q * 4 < n; q += (int64_t)gridDim.x * blockDim.x) {
    const uint64_t c = base + (uint64_t)q;
    const uint4 r = philox4x32_10(make_uint4((uint32_t)c, (uint32_t)(c >> 32), (uint32_t)stream_id, (uint32_t)(stream_id >> 32)), key);
    float v[4];
    if (normal) {  // Box-Muller on two pairs
      const float u0 = 1.f - u32_to_unit(r.x), u1 = u32_to_unit(r.y), u2 = 1.f - u32_to_unit(r.z), u3 = u32_to_unit(r.w);
      const float r0 = sqrtf(-2.f * logf(u0)), r1 = sqrtf(-2.f * logf(u2));
      float s0, c0, s1, c1;
      sincospif(2.f * u1, &s0, &c0);
      sincospif(2.f * u3, &s1, &c1);
      v[0] = r0 * c0; v[1] = r0 * s0; v[2] = r1 * c1; v[3] = r1 * s1;
    } else {
      v[0] = u32_to_unit(r.x); v[1] = u32_to_unit(r.y); v[2] = u32_to_unit(r.z); v[3] = u32_to_unit(r.w);
    }
    for (int j = 0; j < 4; ++j)
      if (q * 4 + j < n) out[q * 4 + j] = v[j];
  }
}

__global__ void counter_add_kernel(uint64_t* c, uint64_t inc) { *c += inc; }

int fill(il_handle* h, float* out, int64_t n, uint64_t seed, uint64_t stream_id, const uint64_t* counter, void* stream, int normal) {
  IL_CHECK(h && out && n >= 0, "il_fill: bad argument");
  if (n == 0) return 0;
  int64_t blocks = (n / 4 + 255) / 256;
  if (blocks > (int64_t)h->sm_count * 16) blocks = (int64_t)h->sm_count * 16;
  if (blocks < 1) blocks = 1;
  IL_LAUNCH(h, fill_kernel, (unsigned)blocks, 256, 0, (cudaStream_t)stream, out, n, seed, stream_id, counter, normal);
  return 0;
}

}  // namespace

extern "C" int il_fill_normal(il_handle* h, float* out, int64_t n, uint64_t seed, uint64_t stream_id, const uint64_t* counter, void* stream) {
  return fill(h, out, n, seed, stream_id, counter, stream, 1);
}
extern "C" int il_fill_uniform(il_handle* h, float* out, int64_t n, uint64_t seed, uint64_t stream_id, const uint64_t* counter, void* stream) {
  return fill(h, out, n, seed, stream_id, counter, stream, 0);
}
extern "C" int il_counter_add(il_handle* h, uint64_t* counter, uint64_t inc, void* stream) {
  IL_CHECK(h && counter, "il_counter_add: null argument");
  IL_LAUNCH(h, counter_add_kernel, 1, 1, 0, (cudaStream_t)stream, counter, inc);
  return 0;
}
