// K10 — minibatch gather out of a rollout stored as unique frame planes:
//     dst[j, y, x, c] = frames[index[perm[start + j], c], y, x]
// i.e. the [count, H, W, k] uint8 minibatch K2 (gather.cu) produces from the stacked column,
// bit for bit, while the rollout itself holds every 84x84 frame once instead of k times
// (runners/frame_stacks.py defines the format).
//
//   gather_frame_stacks_tma_kernel  k = 4, H*W % 16 == 0: persistent CTAs (one per SM).  An
//                                   elected thread issues the 4 plane copies of a sample
//                                   (cp.async.bulk global -> shared) into a stage of an mbarrier
//                                   ring; the CTA interleaves the planes into NHWC order in
//                                   shared memory with a PRMT 4x4 byte transpose; one
//                                   cp.async.bulk shared -> global writes the whole row.
//   gather_frame_stacks_kernel      any k, H, W: one thread per output pixel.
#include "common.cuh"

namespace derl {
namespace {

constexpr int kFsThreads = 256;
constexpr int kFsStages = 4;    // input ring: 4 samples (4 x 28 224 B at 84x84) in flight per SM
constexpr int kFsOutBufs = 2;   // output rows: one being written back while the next is built

inline size_t fs_smem_bytes(long long plane_bytes) {
  const size_t row = (size_t)(4 * plane_bytes);
  return row * (kFsStages + kFsOutBufs) + 8 * kFsStages;
}

// 4 words of 4 pixels each (one word per channel plane) -> the 4 pixels' NHWC words.
__device__ __forceinline__ uint4 interleave4(unsigned a0, unsigned a1, unsigned a2, unsigned a3) {
  const unsigned t0 = __byte_perm(a0, a1, 0x5140);  // a0.0 a1.0 a0.1 a1.1
  const unsigned t1 = __byte_perm(a0, a1, 0x7362);  // a0.2 a1.2 a0.3 a1.3
  const unsigned t2 = __byte_perm(a2, a3, 0x5140);
  const unsigned t3 = __byte_perm(a2, a3, 0x7362);
  return make_uint4(__byte_perm(t0, t2, 0x5410), __byte_perm(t0, t2, 0x7632),
                    __byte_perm(t1, t3, 0x5410), __byte_perm(t1, t3, 0x7632));
}

__global__ void __launch_bounds__(kFsThreads, 1)
gather_frame_stacks_tma_kernel(const uint8_t* __restrict__ frames, int plane_bytes,
                               const int4* __restrict__ index, const long long* __restrict__ perm,
                               long long start, long long count, uint8_t* __restrict__ dst) {
  extern __shared__ __align__(128) uint8_t smem[];
  const int row_bytes = 4 * plane_bytes;
  uint8_t* in_ring = smem;
  uint8_t* out_ring = smem + (size_t)kFsStages * row_bytes;
  uint64_t* full = reinterpret_cast<uint64_t*>(out_ring + (size_t)kFsOutBufs * row_bytes);
  const bool leader = threadIdx.x == 0;
  if (leader) {
#pragma unroll
    for (int s = 0; s < kFsStages; ++s) mbar_init(&full[s], 1);
    mbar_fence_init();
  }
  __syncthreads();

  // rows j = blockIdx.x + i * gridDim.x: neighbouring CTAs write neighbouring rows
  const long long first = blockIdx.x, step = gridDim.x;
  const long long mine = first < count ? (count - first + step - 1) / step : 0;
  auto sample_of = [&](long long i) -> long long { return __ldg(perm + start + first + i * step); };
  auto load = [&](long long i, int4 ids) {
    const int s = (int)(i % kFsStages);
    uint8_t* stage = in_ring + (size_t)s * row_bytes;
    mbar_expect_tx(&full[s], (uint32_t)row_bytes);
    const int plane[4] = {ids.x, ids.y, ids.z, ids.w};
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      bulk_g2s(stage + c * plane_bytes, frames + (long long)plane[c] * plane_bytes,
               (uint32_t)plane_bytes, &full[s]);
    }
  };

  // The leader keeps the plane ids of the sample it refills with next in registers, and the
  // permutation entry of the one after: the dependent perm -> index loads are issued a full row
  // ahead of their use, off the CTA's critical path.
  long long next_sample = 0;
  int4 next_ids = make_int4(0, 0, 0, 0);
  if (leader) {
    long long issued = 0;
    for (; issued < kFsStages && issued < mine; ++issued) load(issued, __ldg(index + sample_of(issued)));
    if (kFsStages < mine) next_sample = sample_of(kFsStages);
  }

  const int words = plane_bytes >> 2;   // 4-pixel words per plane
  for (long long i = 0; i < mine; ++i) {
    const int s = (int)(i % kFsStages);
    const int b = (int)(i % kFsOutBufs);
    if (leader) {
      if (i + kFsStages < mine) next_ids = __ldg(index + next_sample);
      if (i + kFsStages + 1 < mine) next_sample = sample_of(i + kFsStages + 1);
      bulk_wait_read<kFsOutBufs - 1>();   // the store that last used out buffer b has read it
    }
    __syncthreads();
    mbar_wait(&full[s], (uint32_t)((i / kFsStages) & 1));
    const unsigned* in = reinterpret_cast<const unsigned*>(in_ring + (size_t)s * row_bytes);
    uint4* out = reinterpret_cast<uint4*>(out_ring + (size_t)b * row_bytes);
    for (int w = threadIdx.x; w < words; w += kFsThreads) {
      out[w] = interleave4(in[w], in[words + w], in[2 * words + w], in[3 * words + w]);
    }
    fence_proxy_async_smem();
    __syncthreads();   // stage s fully read, out buffer b fully written
    if (leader) {
      const long long j = first + i * step;
      bulk_s2g(dst + j * row_bytes, out_ring + (size_t)b * row_bytes, (uint32_t)row_bytes);
      bulk_commit();
      if (i + kFsStages < mine) load(i + kFsStages, next_ids);
    }
  }
  if (leader) bulk_wait<0>();
}

__global__ void __launch_bounds__(256)
gather_frame_stacks_kernel(const uint8_t* __restrict__ frames, long long plane_bytes,
                           const int* __restrict__ index, int k,
                           const long long* __restrict__ perm, long long start, long long count,
                           uint8_t* __restrict__ dst) {
  const long long total = count * plane_bytes;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += stride) {
    const long long j = t / plane_bytes;
    const long long px = t - j * plane_bytes;
    const int* ids = index + __ldg(perm + start + j) * k;
    uint8_t* o = dst + t * k;
    for (int c = 0; c < k; ++c) o[c] = __ldg(frames + (long long)__ldg(ids + c) * plane_bytes + px);
  }
}

}  // namespace
}  // namespace derl

using namespace derl;

extern "C" int derl_b200_gather_frame_stacks(const void* frames, int64_t n_frames, int64_t height,
                                             int64_t width, const int32_t* index, int64_t n_samples,
                                             int64_t k, const int64_t* perm, int64_t start,
                                             int64_t count, void* dst, void* stream) {
  DERL_REQUIRE(frames && index && perm && dst, "gather_frame_stacks: null pointer");
  DERL_REQUIRE(n_frames >= 1 && n_samples >= 1 && height >= 1 && width >= 1 && k >= 1 &&
                   start >= 0 && count >= 0,
               "gather_frame_stacks: bad sizes (frames=%lld %lldx%lld samples=%lld k=%lld "
               "start=%lld count=%lld)",
               (long long)n_frames, (long long)height, (long long)width, (long long)n_samples,
               (long long)k, (long long)start, (long long)count);
  int rc = require_device();
  if (rc != DERL_OK) return rc;
  if (count == 0) return DERL_OK;
  cudaStream_t st = as_stream(stream);
  const long long plane_bytes = height * width;
  const long long* p = reinterpret_cast<const long long*>(perm);
  const uint8_t* src = reinterpret_cast<const uint8_t*>(frames);
  uint8_t* out = reinterpret_cast<uint8_t*>(dst);
  const size_t smem = fs_smem_bytes(plane_bytes);
  const bool aligned = (((uintptr_t)frames | (uintptr_t)dst | (uintptr_t)index) & 15) == 0;
  if (k == 4 && plane_bytes % 16 == 0 && aligned && smem <= 227 * 1024) {
    if (int rc_attr = ensure_dynamic_smem(
            reinterpret_cast<const void*>(gather_frame_stacks_tma_kernel), (int)smem)) {
      return rc_attr;
    }
    long long grid = sm_count();
    if (grid > count) grid = count;
    gather_frame_stacks_tma_kernel<<<(unsigned)grid, kFsThreads, smem, st>>>(
        src, (int)plane_bytes, reinterpret_cast<const int4*>(index), p, start, count, out);
    DERL_LAUNCH_CHECK("gather_frame_stacks_tma_kernel");
    return DERL_OK;
  }
  long long blocks = (count * plane_bytes + 255) / 256;
  const long long cap = (long long)sm_count() * 32;
  if (blocks > cap) blocks = cap;
  gather_frame_stacks_kernel<<<(unsigned)blocks, 256, 0, st>>>(src, plane_bytes, index, (int)k, p,
                                                               start, count, out);
  DERL_LAUNCH_CHECK("gather_frame_stacks_kernel");
  return DERL_OK;
}
