// Replica-to-replica state copy (population-based training): replica r becomes a copy of replica src_of[r] in every listed buffer.
#include "common.cuh"

namespace {

constexpr int kThreads = 256;
constexpr int kUnroll = 8;
constexpr int64_t kChunkBytes = 16 * kThreads * kUnroll;  // one work item: 32 KB, 8 independent 16-byte loads in flight per thread

struct ReplicaCopyDesc {
  char* base[IL_REPLICA_COPY_MAX_BUFS];
  int64_t stride[IL_REPLICA_COPY_MAX_BUFS];
  int64_t bytes[IL_REPLICA_COPY_MAX_BUFS];
  int64_t first_chunk[IL_REPLICA_COPY_MAX_BUFS + 1];  // prefix sums of the per-replica chunk counts; first_chunk[nbufs] = chunks per replica
  int32_t vec16[IL_REPLICA_COPY_MAX_BUFS];           // base, stride and length all 16-byte aligned
  int32_t nbufs;
};

// Work item i = (replica i / chunks-per-replica, chunk i % chunks-per-replica), walked grid-stride by a fixed grid. Items of a replica that
// maps to itself are skipped after one read of the map, so one launch shape serves every map: a captured graph stays valid when the device
// map is rewritten between replays. Sources map to themselves (the caller's precondition), so no item reads bytes another item writes.
__global__ void __launch_bounds__(kThreads) replica_copy_kernel(const __grid_constant__ ReplicaCopyDesc d, const int32_t* __restrict__ src_of, int R) {
  const int64_t per = d.first_chunk[d.nbufs], items = per * R;
  for (int64_t i = blockIdx.x; i < items; i += gridDim.x) {
    const int r = (int)(i / per);
    const int s = __ldg(src_of + r);
    if (s == r) {  // jump to this CTA's last item of replica r; the loop increment then lands on its first item past it
      i += ((int64_t)(r + 1) * per - 1 - i) / gridDim.x * gridDim.x;
      continue;
    }
    const int64_t c = i % per;
    int b = 0;
    while (c >= d.first_chunk[b + 1]) ++b;
    const int64_t lo = (c - d.first_chunk[b]) * kChunkBytes, hi = min(d.bytes[b], lo + kChunkBytes);
    const char* src = d.base[b] + (int64_t)s * d.stride[b];
    char* dst = d.base[b] + (int64_t)r * d.stride[b];
    if (d.vec16[b]) {
      const int4* s4 = reinterpret_cast<const int4*>(src);
      int4* d4 = reinterpret_cast<int4*>(dst);
      int4 v[kUnroll];
#pragma unroll
      for (int k = 0; k < kUnroll; ++k) {
        const int64_t j = lo / 16 + (int64_t)k * kThreads + threadIdx.x;
        if (j * 16 < hi) v[k] = __ldcs(s4 + j);
      }
#pragma unroll
      for (int k = 0; k < kUnroll; ++k) {
        const int64_t j = lo / 16 + (int64_t)k * kThreads + threadIdx.x;
        if (j * 16 < hi) __stcs(d4 + j, v[k]);
      }
    } else {
      const int32_t* s1 = reinterpret_cast<const int32_t*>(src);
      int32_t* d1 = reinterpret_cast<int32_t*>(dst);
      for (int64_t j = lo / 4 + threadIdx.x; j * 4 < hi; j += kThreads) d1[j] = s1[j];
    }
  }
}

}  // namespace

extern "C" int il_replica_copy(il_handle* h, int nbufs, void* const* base, const int64_t* stride_bytes, const int64_t* bytes, int R, const int32_t* src_of,
                               void* stream) {
  IL_CHECK(h && base && stride_bytes && bytes && src_of, "il_replica_copy: null argument");
  IL_CHECK(nbufs >= 1 && nbufs <= IL_REPLICA_COPY_MAX_BUFS, "il_replica_copy: nbufs=%d outside [1, %d]", nbufs, IL_REPLICA_COPY_MAX_BUFS);
  IL_CHECK(R >= 1, "il_replica_copy: R=%d", R);
  IL_CHECK(((uintptr_t)src_of & 3) == 0, "il_replica_copy: src_of is not 4-byte aligned");
  ReplicaCopyDesc d;
  d.nbufs = nbufs;
  d.first_chunk[0] = 0;
  for (int b = 0; b < nbufs; ++b) {
    IL_CHECK(base[b] != nullptr, "il_replica_copy: buffer %d is null", b);
    IL_CHECK(bytes[b] >= 0 && bytes[b] <= stride_bytes[b], "il_replica_copy: buffer %d copies %lld bytes per replica with a stride of %lld bytes", b,
             (long long)bytes[b], (long long)stride_bytes[b]);
    IL_CHECK((((uintptr_t)base[b]) & 3) == 0 && (stride_bytes[b] & 3) == 0 && (bytes[b] & 3) == 0,
             "il_replica_copy: buffer %d is not 4-byte aligned (base %p, stride %lld, bytes %lld)", b, base[b], (long long)stride_bytes[b], (long long)bytes[b]);
    d.base[b] = (char*)base[b];
    d.stride[b] = stride_bytes[b];
    d.bytes[b] = bytes[b];
    d.vec16[b] = (((uintptr_t)base[b]) & 15) == 0 && (stride_bytes[b] & 15) == 0 && (bytes[b] & 15) == 0;
    d.first_chunk[b + 1] = d.first_chunk[b] + (bytes[b] + kChunkBytes - 1) / kChunkBytes;
  }
  const int64_t items = d.first_chunk[nbufs] * R;
  if (items == 0) return 0;
  const int64_t grid = items < (int64_t)h->sm_count * 8 ? items : (int64_t)h->sm_count * 8;
  IL_LAUNCH(h, replica_copy_kernel, (unsigned)grid, kThreads, 0, (cudaStream_t)stream, d, src_of, R);
  return 0;
}
