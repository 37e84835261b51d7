// K11 — one env step of frame-stack packing: FrameStackPacker.pack (runners/frame_stacks.py) on
// the device.  For the same sequence of steps it hands out the same plane ids and writes the same
// plane bytes, bit for bit:
//   channel k-1 of every stack is a new plane, id count + n;
//   for c = k-2 ... 0, channel c of env n reuses the id of channel c+1 of the same stack if their
//   bytes are equal, else the id of channel c+1 of env n's previous step if those bytes are
//   equal, else it is a new plane; the new planes of channel c take the next ids in env order.
//
// Three launches, no host synchronisation (the running plane count lives in device memory):
//   pack_diff4_kernel / pack_diff_kernel  one CTA per env: ORs per-channel "differs" bits for the
//        same-stack and previous-step tests over the whole stack, and writes channel k-1 into its
//        plane.  k = 4 fast path: 16-byte loads, a 32-bit word is one pixel's four channels, so
//        w ^ (w >> 8) and w ^ (p >> 8) test channels 0-2 at once; PRMT gathers byte 3.
//   pack_assign_kernel                    one CTA: per-channel block scans of the new-plane flags
//        hand out ids in the host's order, resolve each env's reuse chain, write the [N, k] ids,
//        list the new planes of channels < k-1, and advance the count (or set the overflow flag).
//   pack_copy4_kernel / pack_copy_kernel  copies the listed channels into their planes (PRMT byte
//        selects on the fast path).  On the usual stacking wrappers the list is empty.
#include "common.cuh"

namespace derl {
namespace {

constexpr int kPkThreads = 256;
constexpr int kAssignThreads = 1024;

// workspace: int64 {first listed plane id, listed planes}; uint2 flags [N]; int32 list [N*(k-1)]
constexpr size_t kPkHeaderBytes = 16;

inline size_t pack_workspace_bytes(long long n, long long k) {
  const size_t bytes = kPkHeaderBytes + 8 * (size_t)n + 4 * (size_t)n * (size_t)(k - 1);
  return (bytes + 15) & ~(size_t)15;
}

// differs-bytes word (bytes 0-2 relevant) -> bit c = channel c differs somewhere
__device__ __forceinline__ unsigned byte_bits3(unsigned x) {
  return ((x & 0xffu) != 0u) | (((x & 0xff00u) != 0u) << 1) | (((x & 0xff0000u) != 0u) << 2);
}

// byte c of each of the four words, in order
__device__ __forceinline__ unsigned select_bytes(uint4 v, unsigned sel) {
  return __byte_perm(__byte_perm(v.x, v.y, sel), __byte_perm(v.z, v.w, sel), 0x5410);
}

// OR of v over the block; valid in thread 0.  scratch: 32 words.
__device__ __forceinline__ unsigned block_or(unsigned v, unsigned* scratch) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  v = __reduce_or_sync(0xffffffffu, v);
  if (lane == 0) scratch[warp] = v;
  __syncthreads();
  if (warp == 0) {
    v = lane < (int)(blockDim.x >> 5) ? scratch[lane] : 0u;
    v = __reduce_or_sync(0xffffffffu, v);
  }
  return v;
}

// k = 4, H*W % 16 == 0, 16-byte aligned stacks and pool.  groups = H*W / 16 (16 pixels each).
template <bool kHasPrev>
__global__ void __launch_bounds__(kPkThreads)
pack_diff4_kernel(const uint4* __restrict__ cur, const uint4* __restrict__ prev, int groups,
                  int n_envs, uint8_t* __restrict__ pool, long long capacity,
                  const long long* __restrict__ state, uint2* __restrict__ flags) {
  __shared__ unsigned scratch[2][32];
  const int n = blockIdx.x;
  const long long count = state[0];
  const bool write = state[1] == 0 && count + n_envs <= capacity;
  const uint4* c = cur + (size_t)n * groups * 4;
  const uint4* p = kHasPrev ? prev + (size_t)n * groups * 4 : nullptr;
  uint4* plane = reinterpret_cast<uint4*>(pool) + (size_t)(count + n) * groups;
  unsigned same = 0u, back = 0u;
  for (int g = threadIdx.x; g < groups; g += kPkThreads) {
    uint4 v[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) v[i] = __ldg(c + 4 * g + i);
    if (kHasPrev) {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const uint4 q = __ldg(p + 4 * g + i);
        back |= (v[i].x ^ (q.x >> 8)) | (v[i].y ^ (q.y >> 8)) | (v[i].z ^ (q.z >> 8)) |
                (v[i].w ^ (q.w >> 8));
      }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      same |= (v[i].x ^ (v[i].x >> 8)) | (v[i].y ^ (v[i].y >> 8)) | (v[i].z ^ (v[i].z >> 8)) |
              (v[i].w ^ (v[i].w >> 8));
    }
    if (write) {
      plane[g] = make_uint4(select_bytes(v[0], 0x73), select_bytes(v[1], 0x73),
                            select_bytes(v[2], 0x73), select_bytes(v[3], 0x73));
    }
  }
  same = block_or(same, scratch[0]);
  if (kHasPrev) back = block_or(back, scratch[1]);
  if (threadIdx.x == 0) flags[n] = make_uint2(byte_bits3(same), kHasPrev ? byte_bits3(back) : 7u);
}

// any 1 <= k <= 32, any H x W: byte loads, one pixel per thread per iteration.
__global__ void __launch_bounds__(kPkThreads)
pack_diff_kernel(const uint8_t* __restrict__ cur, const uint8_t* __restrict__ prev,
                 long long plane_bytes, int k, int n_envs, uint8_t* __restrict__ pool,
                 long long capacity, const long long* __restrict__ state,
                 uint2* __restrict__ flags) {
  __shared__ unsigned scratch[2][32];
  const int n = blockIdx.x;
  const long long count = state[0];
  const bool write = state[1] == 0 && count + n_envs <= capacity;
  const uint8_t* c = cur + (size_t)n * plane_bytes * k;
  const uint8_t* p = prev != nullptr ? prev + (size_t)n * plane_bytes * k : nullptr;
  uint8_t* plane = pool + (size_t)(count + n) * plane_bytes;
  unsigned same = 0u, back = 0u;
  for (long long px = threadIdx.x; px < plane_bytes; px += kPkThreads) {
    const uint8_t* s = c + px * k;
    uint8_t next = s[k - 1];
    if (write) plane[px] = next;
    for (int ch = k - 2; ch >= 0; --ch) {
      const uint8_t b = s[ch];
      if (b != next) same |= 1u << ch;
      if (p != nullptr && b != p[px * k + ch + 1]) back |= 1u << ch;
      next = b;
    }
  }
  same = block_or(same, scratch[0]);
  back = block_or(back, scratch[1]);
  if (threadIdx.x == 0) {
    flags[n] = make_uint2(same, p != nullptr ? back : (unsigned)((1ull << (k - 1)) - 1));
  }
}

// Exclusive prefix of v over the block (thread order) and the block total.  scratch: 32 ints.
__device__ __forceinline__ int block_exclusive_scan(int v, int* scratch, int& total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int nwarps = blockDim.x >> 5;
  int x = v;
#pragma unroll
  for (int off = 1; off < 32; off <<= 1) {
    const int y = __shfl_up_sync(0xffffffffu, x, off);
    if (lane >= off) x += y;
  }
  if (lane == 31) scratch[warp] = x;
  __syncthreads();
  if (warp == 0) {
    int s = lane < nwarps ? scratch[lane] : 0;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
      const int y = __shfl_up_sync(0xffffffffu, s, off);
      if (lane >= off) s += y;
    }
    scratch[lane] = s;
  }
  __syncthreads();
  const int excl = x - v + (warp > 0 ? scratch[warp - 1] : 0);
  total = scratch[nwarps - 1];
  __syncthreads();   // scratch is reused by the next scan
  return excl;
}

__global__ void __launch_bounds__(kAssignThreads, 1)
pack_assign_kernel(const uint2* __restrict__ flags, const int* __restrict__ prev_ids, int n_envs,
                   int k, long long capacity, long long* __restrict__ state,
                   int* __restrict__ ids, long long* __restrict__ header, int* __restrict__ list) {
  __shared__ int scratch[32];
  const long long count = state[0];
  if (state[1] != 0) {   // an earlier step overflowed: the rollout is void, do nothing
    if (threadIdx.x == 0) header[1] = 0;
    return;
  }
  const int chunk = (n_envs + kAssignThreads - 1) / kAssignThreads;
  const int lo = min(n_envs, (int)threadIdx.x * chunk), hi = min(n_envs, lo + chunk);
  // run[c]: the id of this thread's first new plane of channel c
  long long run[32];
  long long next = count + n_envs;
  for (int ch = k - 2; ch >= 0; --ch) {
    int mine = 0;
    for (int n = lo; n < hi; ++n) {
      const uint2 f = flags[n];
      mine += (int)((f.x & f.y) >> ch & 1u);
    }
    int total;
    const int excl = block_exclusive_scan(mine, scratch, total);
    run[ch] = next + excl;
    next += total;
  }
  if (next > capacity) {
    if (threadIdx.x == 0) {
      state[1] = 1;
      header[1] = 0;
    }
    return;
  }
  const long long first = count + n_envs;
  for (int n = lo; n < hi; ++n) {
    const uint2 f = flags[n];
    int id = (int)(count + n);
    int* row = ids + (size_t)n * k;
    row[k - 1] = id;
    for (int ch = k - 2; ch >= 0; --ch) {
      if (f.x >> ch & 1u) {
        if (!(f.y >> ch & 1u)) {
          id = prev_ids[(size_t)n * k + ch + 1];
        } else {
          id = (int)run[ch]++;
          list[id - first] = n * k + ch;
        }
      }
      row[ch] = id;
    }
  }
  __syncthreads();   // every thread has read state[0]
  if (threadIdx.x == 0) {
    state[0] = next;
    header[0] = first;
    header[1] = next - first;
  }
}

__global__ void __launch_bounds__(kPkThreads)
pack_copy4_kernel(const uint4* __restrict__ stacks, int groups,
                  const long long* __restrict__ header, const int* __restrict__ list,
                  uint8_t* __restrict__ pool) {
  const long long first = header[0], listed = header[1];
  for (long long e = blockIdx.x; e < listed; e += gridDim.x) {
    const int nk = list[e];
    const int n = nk >> 2;
    const unsigned ch = (unsigned)(nk & 3);
    const unsigned sel = ch | ((ch + 4u) << 4);
    const uint4* s = stacks + (size_t)n * groups * 4;
    uint4* plane = reinterpret_cast<uint4*>(pool) + (size_t)(first + e) * groups;
    for (int g = threadIdx.x; g < groups; g += kPkThreads) {
      plane[g] = make_uint4(select_bytes(__ldg(s + 4 * g), sel),
                            select_bytes(__ldg(s + 4 * g + 1), sel),
                            select_bytes(__ldg(s + 4 * g + 2), sel),
                            select_bytes(__ldg(s + 4 * g + 3), sel));
    }
  }
}

__global__ void __launch_bounds__(kPkThreads)
pack_copy_kernel(const uint8_t* __restrict__ stacks, long long plane_bytes, int k,
                 const long long* __restrict__ header, const int* __restrict__ list,
                 uint8_t* __restrict__ pool) {
  const long long first = header[0], listed = header[1];
  for (long long e = blockIdx.x; e < listed; e += gridDim.x) {
    const int nk = list[e];
    const int n = nk / k, ch = nk - n * k;
    const uint8_t* s = stacks + (size_t)n * plane_bytes * k + ch;
    uint8_t* plane = pool + (size_t)(first + e) * plane_bytes;
    for (long long px = threadIdx.x; px < plane_bytes; px += kPkThreads) plane[px] = s[px * k];
  }
}

}  // namespace
}  // namespace derl

using namespace derl;

extern "C" size_t derl_b200_pack_frame_stacks_workspace_bytes(int64_t n, int64_t k) {
  if (n < 1 || k < 1 || k > 32) return 0;
  return pack_workspace_bytes(n, k);
}

extern "C" int derl_b200_pack_frame_stacks(const void* stacks, const void* prev_stacks,
                                           const int32_t* prev_ids, int64_t n, int64_t height,
                                           int64_t width, int64_t k, void* pool, int64_t capacity,
                                           int64_t* state, int32_t* ids, void* workspace,
                                           size_t workspace_bytes, void* stream) {
  DERL_REQUIRE(stacks && pool && state && ids && workspace, "pack_frame_stacks: null pointer");
  DERL_REQUIRE((prev_stacks == nullptr) == (prev_ids == nullptr),
               "pack_frame_stacks: prev_stacks and prev_ids must both be given or both be null");
  DERL_REQUIRE(k >= 1 && k <= 32, "pack_frame_stacks: k = %lld outside 1..32", (long long)k);
  DERL_REQUIRE(n >= 1 && height >= 1 && width >= 1 && capacity >= 1,
               "pack_frame_stacks: bad sizes (n=%lld %lldx%lld capacity=%lld)", (long long)n,
               (long long)height, (long long)width, (long long)capacity);
  DERL_REQUIRE(capacity <= INT32_MAX && n * k <= INT32_MAX,
               "pack_frame_stacks: int32 plane ids cannot address capacity=%lld n*k=%lld",
               (long long)capacity, (long long)(n * k));
  DERL_REQUIRE(workspace_bytes >= pack_workspace_bytes(n, k),
               "pack_frame_stacks: workspace of %zu bytes < %zu", workspace_bytes,
               pack_workspace_bytes(n, k));
  int rc = require_device();
  if (rc != DERL_OK) return rc;
  cudaStream_t st = as_stream(stream);
  const long long plane_bytes = height * width;
  long long* header = reinterpret_cast<long long*>(workspace);
  uint2* flags = reinterpret_cast<uint2*>(reinterpret_cast<uint8_t*>(workspace) + kPkHeaderBytes);
  int* list = reinterpret_cast<int*>(flags + n);
  const uint8_t* cur = reinterpret_cast<const uint8_t*>(stacks);
  const uint8_t* prev = reinterpret_cast<const uint8_t*>(prev_stacks);
  uint8_t* planes = reinterpret_cast<uint8_t*>(pool);
  long long* st64 = reinterpret_cast<long long*>(state);
  const bool fast = k == 4 && plane_bytes % 16 == 0 &&
                    (((uintptr_t)stacks | (uintptr_t)prev_stacks | (uintptr_t)pool) & 15) == 0;
  const int groups = (int)(plane_bytes / 16);
  if (fast && prev != nullptr) {
    pack_diff4_kernel<true><<<(unsigned)n, kPkThreads, 0, st>>>(
        reinterpret_cast<const uint4*>(cur), reinterpret_cast<const uint4*>(prev), groups, (int)n,
        planes, capacity, st64, flags);
  } else if (fast) {
    pack_diff4_kernel<false><<<(unsigned)n, kPkThreads, 0, st>>>(
        reinterpret_cast<const uint4*>(cur), nullptr, groups, (int)n, planes, capacity, st64,
        flags);
  } else {
    pack_diff_kernel<<<(unsigned)n, kPkThreads, 0, st>>>(cur, prev, plane_bytes, (int)k, (int)n,
                                                         planes, capacity, st64, flags);
  }
  DERL_LAUNCH_CHECK("pack_diff_kernel");
  pack_assign_kernel<<<1, kAssignThreads, 0, st>>>(flags, prev_ids, (int)n, (int)k, capacity,
                                                   st64, ids, header, list);
  DERL_LAUNCH_CHECK("pack_assign_kernel");
  if (k == 1) return DERL_OK;
  long long grid = (long long)sm_count() * 4;
  if (grid > n * (k - 1)) grid = n * (k - 1);
  if (fast) {
    pack_copy4_kernel<<<(unsigned)grid, kPkThreads, 0, st>>>(reinterpret_cast<const uint4*>(cur),
                                                             groups, header, list, planes);
  } else {
    pack_copy_kernel<<<(unsigned)grid, kPkThreads, 0, st>>>(cur, plane_bytes, (int)k, header, list,
                                                            planes);
  }
  DERL_LAUNCH_CHECK("pack_copy_kernel");
  return DERL_OK;
}
