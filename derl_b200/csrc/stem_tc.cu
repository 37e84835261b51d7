// K6t — the NatureCNN stem forward (conv 8x8 / 4 over uint8 [84,84,4] frames + bias + ReLU,
// derl/models.py:102-103,117-123) straight from the uint8 frames, on the 5th-generation tensor
// cores: tcgen05.mma kind::i8 with the accumulators in tensor memory.
// Number format: the frame operand is the raw uint8 bytes (exact, no float conversion); the
// weights are two signed 8-bit digit planes per output channel n: s = max|W[n]| / 127,
//   W ~= s (q1 + q2 / 254),  q1 = rint(W / s),  q2 = clamp(rint((W - s q1) * 254 / s), +-127),
// residual <= s / 508.  Both digit planes accumulate exactly in int32 (|acc| < 2^24); the fp32
// epilogue is y = relu(float(acc1 * 254 + acc2) * (s / 64770) + bias), every step separately
// rounded (tests/stem_model.py restates it bit for bit).  bf16 outputs are y rounded to nearest
// even.
//
// Operand formulation.  With the frame cut into 4x4-pixel blocks (space-to-depth(4): block
// (Y, X) = rows 4Y..4Y+3, columns 4X..4X+3, 64 bytes) the 8x8/4 convolution is a 2x2/1
// convolution over 21x21 blocks: for kernel quadrant (a, b) the output pixel (oy, ox) reads block
// (oy + a, ox + b).  One TMA tensor copy lands the frame in shared memory with its 84 image rows
// PERMUTED, row 4Y + i -> slot i * 21 + Y (tensor map {84 u32, 21 Y, 4 i, frames}, box = one
// frame): plane i then holds, for every block m' = 21 Y + X, the 16 bytes (j, c) of its image row
// i, as 16-byte units at address 16 m'.  That is exactly the canonical NO-SWIZZLE K-major UMMA
// operand — core matrix = 8 consecutive blocks x 16 bytes = 128 contiguous bytes, next 8 blocks
// at +128 B (SBO), the K-neighbour chunk (i + 1) at +7056 B (LBO) — and with pixels numbered
// m = 21 oy + ox (one junk column per output row) quadrant (a, b) is the same operand started
// 16 (21 a + b) bytes later.  No im2col, no byte transpose, no fragment loads: per frame the
// tensor core reads the landed bytes in 32 instructions
//     D[128 pixels x 64 (plane, channel)] += A[128 x 32 B] * W[64 x 32 B]
// (4 pixel tiles x 4 quadrants x 2 K-halves; ~1 k tensor cycles) issued by one thread.
// The 64 accumulator columns of a pixel (32 channels x 2 digit planes) sit in ONE tensor-memory
// lane, so the epilogue thread that owns the pixel recombines the planes, applies scale, /255,
// bias and ReLU and holds the pixel's 32 outputs — 128 bytes of fp32 written to a 128B-swizzled
// staging tile, or 64 bytes of bf16 to a 64B-swizzled one (16-byte stores, conflict-free) — that a
// TMA tensor store drains as two 200-pixel boxes per frame.
//
// Roles (576 threads, one persistent CTA per SM): warp 0 = TMA producer (frames, three
// buffers: HBM latency is ~a frame period, so loads run two frames ahead), warp 1 = MMA issuer + TMEM owner, warps 2-9 / 10-17 = two epilogue groups taking
// alternate frames (each owns one 256-column accumulator buffer and one staging tile), so that
// frame f+1's loads and MMAs and frame f's epilogue and frame f-1's store overlap.
#include <cuda.h>
#include <cuda_bf16.h>

#include "common.cuh"
#include "tcgen05.cuh"

namespace derl {
namespace {

constexpr int kImgBytes = 84 * 84 * 4;        // 28224
constexpr int kPlaneBytes = 21 * 336;         // 7056: one tap-row plane [21 Y][336 B]
constexpr int kFrameBuf = 29824;              // frame + over-read slack of the last pixel tile
constexpr int kOutC = 32, kPixPad = 420;      // padded pixel index m = 21 oy + ox, ox = 20 is junk
constexpr int kMTiles = 4;                    // 4 x 128 rows
constexpr int kWBytes = 16 * 64 * 16;         // [k16][n'][16 B]
constexpr int kStageBytes = 400 * 128;        // one frame's fp32 activation (bf16 uses half)
constexpr int kEpiWarps = 8;                  // warps per epilogue group: 4 lane quarters x 2 tile parities
constexpr int kThreads = (2 + 2 * kEpiWarps) * 32;   // 576
constexpr int kStages = 3;                    // frame buffers: loads run two frames ahead of the MMAs
constexpr uint32_t kTmemCols = 512;

struct TcSmem {   // byte offsets from a 1024-aligned base
  static constexpr int stage = 0;                              // [2][51200]
  static constexpr int frame = stage + 2 * kStageBytes;        // [kStages][29824]
  static constexpr int w = frame + kStages * kFrameBuf;        // 16384
  static constexpr int scale = w + kWBytes;                    // float[32]
  static constexpr int bias = scale + 128;                     // float[32]
  static constexpr int escale = bias + 128;                    // float[32]: s / (254 * 255)
  static constexpr int bars = escale + 128;                    // 2 * kStages + 4 mbarriers
  static constexpr int slot = bars + 128;                      // tmem base address
  static constexpr int bytes = slot + 16;
  static constexpr int alloc = bytes + 1024;                   // slack for the manual alignment
};
static_assert(TcSmem::frame % 128 == 0 && TcSmem::w % 128 == 0, "smem alignment");
static_assert(TcSmem::alloc <= 227 * 1024, "shared memory budget");

constexpr uint32_t kIdesc = umma_idesc_i8(128, 64, /*a u8*/ 0, /*b s8*/ 1, 0, 0);

__device__ __forceinline__ unsigned pack_bf16(float lo, float hi) {   // round to nearest even
  const __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<const unsigned*>(&v);
}

// kMask: also emit the ReLU mask words (K7t's input).  OT: float or __nv_bfloat16 output.
template <bool kMask, typename OT>
__global__ void __launch_bounds__(kThreads, 1)
stem_conv_relu_tc_kernel(const __grid_constant__ CUtensorMap tm_frames,
                         const __grid_constant__ CUtensorMap tm_out,
                         const long long* __restrict__ rows, const float* __restrict__ weight,
                         const float* __restrict__ bias, unsigned* __restrict__ mask_out,
                         long long batch, int out_block) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + (((raw_addr + 1023u) & ~1023u) - raw_addr);
  uint8_t* wsm = smem + TcSmem::w;
  float* ssm = reinterpret_cast<float*>(smem + TcSmem::scale);
  float* bsm = reinterpret_cast<float*>(smem + TcSmem::bias);
  float* esm = reinterpret_cast<float*>(smem + TcSmem::escale);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + TcSmem::bars);   // [kStages] TMA -> MMA
  uint64_t* empty = full + kStages;                                    // [kStages] MMA -> TMA
  uint64_t* tfull = full + 2 * kStages;                                // [2] MMA -> epilogue
  uint64_t* tempty = tfull + 2;                                        // [2] epilogue -> MMA
  uint32_t* slot = reinterpret_cast<uint32_t*>(smem + TcSmem::slot);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const long long first = blockIdx.x, stride = gridDim.x;

  if (tid == 0) {
    for (int i = 0; i < kStages; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tfull[i], 1);
      mbar_init(&tempty[i], kEpiWarps * 32);
    }
    mbar_fence_init();
    tma_prefetch_desc(&tm_frames);
    tma_prefetch_desc(&tm_out);
  }
  if (warp == 1) tmem_alloc(slot, kTmemCols);

  // ---- per-channel scales and the two digit planes of the weights, [k16][n'][16 B]:
  // k16 = (a * 2 + b) * 4 + i, n' = plane * 32 + channel, byte j * 4 + c  <->  W[n][c][4a+i][4b+j]
  for (int n = warp; n < kOutC; n += kThreads / 32) {
    float m = 0.f;
    for (int k = lane; k < 256; k += 32) m = fmaxf(m, fabsf(__ldg(weight + n * 256 + k)));
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, off));
    if (lane == 0) ssm[n] = m > 0.f ? m / 127.f : 1.f;
  }
  if (tid < kOutC) bsm[tid] = __ldg(bias + tid);
  __syncthreads();
  // epilogue scale s / (254 * 255): (q1 * 254 + q2) * that = (q1 + q2 / 254) * s / 255
  if (tid < kOutC) esm[tid] = ssm[tid] / 64770.f;
  for (int e = tid; e < 16 * kOutC; e += kThreads) {
    const int n = e & 31, k16 = e >> 5;
    const int q = k16 >> 2, i = k16 & 3, kh = 4 * (q >> 1) + i, kw0 = 4 * (q & 1);
    const float s = ssm[n], inv = 1.f / s;
    unsigned p1[4], p2[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      p1[j] = 0u;
      p2[j] = 0u;
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        const float w = __ldg(weight + ((n * 4 + c) * 8 + kh) * 8 + kw0 + j);
        const float q1 = rintf(w * inv);
        const float q2 = fminf(fmaxf(rintf((w - q1 * s) * 254.f * inv), -127.f), 127.f);
        p1[j] |= ((unsigned)(int)q1 & 0xffu) << (8 * c);
        p2[j] |= ((unsigned)(int)q2 & 0xffu) << (8 * c);
      }
    }
    *reinterpret_cast<uint4*>(wsm + k16 * 1024 + n * 16) = make_uint4(p1[0], p1[1], p1[2], p1[3]);
    *reinterpret_cast<uint4*>(wsm + k16 * 1024 + (32 + n) * 16) =
        make_uint4(p2[0], p2[1], p2[2], p2[3]);
  }
  fence_proxy_async_smem();     // generic-proxy writes of W -> visible to the tensor core
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem = *slot;

  if (warp == 0) {
    // ===================================================================== TMA producer
    if (lane == 0) {
      int it = 0;
      for (long long f = first; f < batch; f += stride, ++it) {
        const int b = it % kStages;
        mbar_wait(&empty[b], (unsigned)(((it / kStages) & 1) ^ 1));
        mbar_expect_tx(&full[b], kImgBytes);
        const long long src = rows ? __ldg(rows + f) : f;   // fused minibatch gather
        tma_load_4d(smem + TcSmem::frame + b * kFrameBuf, &tm_frames, 0, 0, 0, (int)src, &full[b]);
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ===================================================================== MMA issuer
    // The whole warp runs the control flow (waits, descriptor arithmetic: warp-uniform); one
    // elected lane issues the MMAs and the commits.
    const uint64_t w_desc = umma_desc(smem_u32(wsm), 1024, 128);
    int it = 0;
    for (long long f = first; f < batch; f += stride, ++it) {
      const int b = it % kStages, g = it & 1;
      const unsigned ph = (unsigned)((it >> 1) & 1);
      mbar_wait(&tempty[g], ph ^ 1u);     // the epilogue has drained this accumulator buffer
      mbar_wait(&full[b], (unsigned)((it / kStages) & 1));   // the frame has landed
      tcgen05_fence_after();
      // descriptors once per frame, advanced by adding to the start-address field (units of 16 B)
      const uint64_t a_frame = umma_desc(smem_u32(smem + TcSmem::frame + b * kFrameBuf),
                                         kPlaneBytes, 128);
      const uint32_t d0 = tmem + (uint32_t)(g * 256);
      if (elect_one_sync()) {
#pragma unroll
        for (int mt = 0; mt < kMTiles; ++mt) {
#pragma unroll
          for (int q = 0; q < 4; ++q) {
#pragma unroll
            for (int ip = 0; ip < 2; ++ip) {
              const uint64_t a_desc = a_frame + (uint64_t)((2 * ip * kPlaneBytes +
                                                            (21 * (q >> 1) + (q & 1)) * 16 + mt * 2048) >> 4);
              const uint64_t b_desc = w_desc + (uint64_t)(((q * 4 + 2 * ip) * 1024) >> 4);
              umma_i8(d0 + mt * 64, a_desc, b_desc, kIdesc, (q | ip) != 0);
            }
          }
        }
        umma_commit(&empty[b]);    // frame buffer may be refilled once these MMAs have read it
        umma_commit(&tfull[g]);    // accumulators complete
      }
      __syncwarp();
    }
  } else {
    // ===================================================================== epilogue groups
    // 16 warps = 2 groups (alternate frames) x 4 tensor-memory lane quarters x 2 tile parities.
    // A warp can only read the quarter (warp id % 4) of tensor memory; the two warps of a
    // quarter split the frame's four 128-pixel tiles between them.
    const int e = warp - 2;
    const int g = e / kEpiWarps;                        // group: frames with it % 2 == g
    const int wq = warp & 3;                            // tensor-memory lane quarter
    const int tp = (e % kEpiWarps) >> 2;                // tile parity
    const int gt = tid - (2 + kEpiWarps * g) * 32;      // thread index inside the group
    uint8_t* stage = smem + TcSmem::stage + g * kStageBytes;
    constexpr int kRow = 32 * sizeof(OT);               // staging bytes per pixel: 128 or 64
    int it = 0, mine = 0;
    for (long long f = first; f < batch; f += stride, ++it) {
      if ((it & 1) != g) continue;
      const unsigned ph = (unsigned)((it >> 1) & 1);
      // the previous store of this staging tile must have finished READING it
      if (gt == 0 && mine > 0) bulk_wait_read<0>();
      named_bar_sync(1 + g, kEpiWarps * 32);
      mbar_wait(&tfull[g], ph);
      tcgen05_fence_after();
#pragma unroll 1
      for (int mt = tp; mt < kMTiles; mt += 2) {
        const int m = mt * 128 + wq * 32 + lane;
        const uint32_t taddr = tmem + ((uint32_t)(wq * 32) << 16) + (uint32_t)(g * 256 + mt * 64);
        const int oy = m / 21, ox = m - oy * 21;
        const bool valid = m < kPixPad && ox < 20;
        int row = oy * 20 + ox;
        if (out_block == 2) row = (((oy >> 1) * 10 + (ox >> 1)) << 2) + ((oy & 1) << 1) + (ox & 1);
        unsigned bits = 0u;       // lane c ends up with channel c's bits of this warp's 32 pixels
        uint8_t* dst = stage + row * kRow;
        // TMA swizzle of 16-byte chunks: 128B rows -> chunk ^ (row & 7), 64B -> chunk ^ (row/2 & 3)
        const int sw = kRow == 128 ? row & 7 : (row >> 1) & 3;
        unsigned packed[4];       // bf16: the current 8-channel chunk
#pragma unroll
        for (int half = 0; half < 2; ++half) {   // 16 channels at a time: 32 live accumulator words
          uint32_t v1[16], v2[16];
          tmem_ld_32x16(taddr + 16 * half, v1);         // digit plane 1
          tmem_ld_32x16(taddr + 32 + 16 * half, v2);    // digit plane 2
          tmem_ld_wait();
#pragma unroll
          for (int c4 = 0; c4 < 4; ++c4) {
            const int ch0 = 16 * half + 4 * c4;
            const float4 e4 = *reinterpret_cast<const float4*>(esm + ch0);   // broadcast LDS.128
            const float4 b4 = *reinterpret_cast<const float4*>(bsm + ch0);
            const float es[4] = {e4.x, e4.y, e4.z, e4.w}, bs[4] = {b4.x, b4.y, b4.z, b4.w};
            float y[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              const int ch = ch0 + k;
              // exact: |q1 * 254 + q2| <= 256 * 255 * 127 * 255 < 2^31
              const int both = (int)v1[4 * c4 + k] * 254 + (int)v2[4 * c4 + k];
              float x = (float)both * es[k] + bs[k];
              x = fmaxf(x, 0.f);
              if (kMask) {
                const unsigned word = __ballot_sync(0xffffffffu, valid && x > 0.f);
                bits = lane == ch ? word : bits;
              }
              y[k] = x;
            }
            if constexpr (kRow == 128) {
              if (valid) {
                *reinterpret_cast<float4*>(dst + (((4 * half + c4) ^ sw) << 4)) =
                    make_float4(y[0], y[1], y[2], y[3]);
              }
            } else {
              packed[2 * (c4 & 1)] = pack_bf16(y[0], y[1]);
              packed[2 * (c4 & 1) + 1] = pack_bf16(y[2], y[3]);
              if (valid && (c4 & 1)) {
                *reinterpret_cast<uint4*>(dst + (((2 * half + (c4 >> 1)) ^ sw) << 4)) =
                    make_uint4(packed[0], packed[1], packed[2], packed[3]);
              }
            }
          }
        }
        // mask words [frame][tile of 32 padded pixels (14)][channel (32)]: one coalesced 128-byte
        // store per warp and tile; tiles 14, 15 (m >= 448) hold no pixel
        const int tile32 = mt * 4 + wq;
        if (kMask && tile32 < 14) mask_out[(f * 14 + tile32) * 32 + lane] = bits;
      }
      tcgen05_fence_before();
      mbar_arrive(&tempty[g]);               // accumulator buffer g may be overwritten
      fence_proxy_async_smem();              // staging writes -> visible to the TMA store
      named_bar_sync(1 + g, kEpiWarps * 32);
      if (gt == 0) {
        tma_store_2d(&tm_out, stage, 0, (int)(f * 400));
        tma_store_2d(&tm_out, stage + 200 * kRow, 0, (int)(f * 400 + 200));
        bulk_commit();
      }
      ++mine;
    }
    if (gt == 0) bulk_wait<0>();             // stores complete before the CTA retires its smem
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == 1) {
    tcgen05_fence_after();
    tmem_dealloc(tmem, kTmemCols);
  }
}

// ------------------------------------------------------------------ tensor maps (memoised per thread)
enum MapKind { kFramesMap, kOutF32Map, kOutBf16Map };
struct MapKey {
  const void* base;
  long long n;
  int kind;
  bool operator==(const MapKey& o) const { return base == o.base && n == o.n && kind == o.kind; }
};
constexpr int kMapSlots = 16;
struct MapCache {
  MapKey keys[kMapSlots];
  CUtensorMap maps[kMapSlots];
  int used = 0, next = 0;
};

bool cached_map(CUtensorMap* out, const MapKey& key, bool (*make)(CUtensorMap*, const MapKey&)) {
  static thread_local MapCache cache;
  for (int i = 0; i < cache.used; ++i) {
    if (cache.keys[i] == key) {
      *out = cache.maps[i];
      return true;
    }
  }
  if (!make(out, key)) return false;
  const int s = cache.used < kMapSlots ? cache.used++ : cache.next;
  cache.next = (s + 1) % kMapSlots;
  cache.keys[s] = key;
  cache.maps[s] = *out;
  return true;
}

// frames [n][84 rows][336 B] seen as {84 u32 (one image row), 21 Y (stride 4 rows), 4 i (stride
// 1 row), n frames}; box = one frame -> shared memory [i][Y][336 B].
bool make_frames_map(CUtensorMap* map, const MapKey& key) {
  TmapEncodeFn enc = tmap_encode_fn();
  if (enc == nullptr) return false;
  cuuint64_t dims[4] = {84, 21, 4, (cuuint64_t)key.n};
  cuuint64_t strides[3] = {4 * 336, 336, (cuuint64_t)kImgBytes};
  cuuint32_t box[4] = {84, 21, 4, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  return enc(map, CU_TENSOR_MAP_DATA_TYPE_UINT32, 4, const_cast<void*>(key.base), dims, strides,
             box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
             CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// out [n * 400 rows][32 channels] of fp32 (128 B rows, 128B swizzle) or bf16 (64 B rows, 64B
// swizzle); box = 200 rows (the staging tile's layout).
bool make_out_map(CUtensorMap* map, const MapKey& key) {
  TmapEncodeFn enc = tmap_encode_fn();
  if (enc == nullptr) return false;
  const bool bf16 = key.kind == kOutBf16Map;
  cuuint64_t dims[2] = {32, (cuuint64_t)key.n * 400};
  cuuint64_t strides[1] = {bf16 ? 64u : 128u};
  cuuint32_t box[2] = {32, 200};
  cuuint32_t estr[2] = {1, 1};
  return enc(map, bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2,
             const_cast<void*>(key.base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
             bf16 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B,
             CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// With rows the frames array is the gather source, whose length the caller may not know: the map
// is built for 2^30 frames (the indices are trusted, as in every gather of this library).
int launch_stem_tc(const uint8_t* frames, const long long* rows, long long batch,
                   const float* weight, const float* bias, void* out, int out_dtype,
                   unsigned* mask_out, int out_block, cudaStream_t st) {
  const bool bf16 = out_dtype == DERL_DTYPE_BF16;
  CUtensorMap tm_frames, tm_out;
  if (!cached_map(&tm_frames, MapKey{frames, rows ? (1ll << 30) : batch, kFramesMap},
                  make_frames_map) ||
      !cached_map(&tm_out, MapKey{out, batch, bf16 ? kOutBf16Map : kOutF32Map}, make_out_map)) {
    set_error("stem_conv_relu: cuTensorMapEncodeTiled failed (batch %lld)", batch);
    return DERL_E_CUDA;
  }
  auto kern = bf16                ? stem_conv_relu_tc_kernel<false, __nv_bfloat16>
              : mask_out != nullptr ? stem_conv_relu_tc_kernel<true, float>
                                    : stem_conv_relu_tc_kernel<false, float>;
  if (int rc = ensure_dynamic_smem(reinterpret_cast<const void*>(kern), TcSmem::alloc)) return rc;
  long long grid = sm_count();
  if (grid > batch) grid = batch;
  kern<<<(unsigned)grid, kThreads, TcSmem::alloc, st>>>(tm_frames, tm_out, rows, weight, bias,
                                                        mask_out, batch, out_block);
  DERL_LAUNCH_CHECK("stem_conv_relu_tc_kernel");
  return DERL_OK;
}

}  // namespace

bool stem_tc_available() { return tmap_encode_fn() != nullptr; }

}  // namespace derl

using namespace derl;

extern "C" int derl_b200_stem_conv_relu(const uint8_t* frames, const int64_t* rows, int64_t batch,
                                        const float* weight, const float* bias, void* out,
                                        int out_dtype, int out_block, void* stream) {
  DERL_REQUIRE(out_block == 1 || out_block == 2, "stem_conv_relu: out_block must be 1 or 2");
  DERL_REQUIRE(frames && weight && bias && out && batch >= 0, "stem_conv_relu: bad arguments");
  DERL_REQUIRE(out_dtype == DERL_DTYPE_F32 || out_dtype == DERL_DTYPE_BF16,
               "stem_conv_relu: out_dtype must be DERL_DTYPE_F32 or DERL_DTYPE_BF16");
  DERL_REQUIRE(((uintptr_t)frames & 15) == 0 && ((uintptr_t)out & 15) == 0,
               "stem_conv_relu: frames and out must be 16-byte aligned");
  DERL_REQUIRE(batch * 400 < (1ll << 31), "stem_conv_relu: batch too large");
  int rc = require_device();
  if (rc != DERL_OK) return rc;
  if (batch == 0) return DERL_OK;
  DERL_REQUIRE(stem_tc_available(), "stem_conv_relu: cuTensorMapEncodeTiled is unavailable");
  return launch_stem_tc(frames, reinterpret_cast<const long long*>(rows), batch, weight, bias, out,
                        out_dtype, nullptr, out_block, as_stream(stream));
}

extern "C" int derl_b200_stem_conv_relu_mask(const uint8_t* frames, const int64_t* rows,
                                             int64_t batch, const float* weight, const float* bias,
                                             float* out, uint32_t* relu_mask, int out_block,
                                             void* stream) {
  DERL_REQUIRE(out_block == 1 || out_block == 2, "stem_conv_relu_mask: out_block must be 1 or 2");
  DERL_REQUIRE(frames && weight && bias && out && relu_mask && batch >= 0,
               "stem_conv_relu_mask: bad arguments");
  DERL_REQUIRE(((uintptr_t)frames & 15) == 0 && ((uintptr_t)out & 127) == 0 &&
                   ((uintptr_t)relu_mask & 15) == 0,
               "stem_conv_relu_mask: frames / mask must be 16-byte, out 128-byte aligned");
  DERL_REQUIRE(batch * 400 < (1ll << 31), "stem_conv_relu_mask: batch too large");
  int rc = require_device();
  if (rc != DERL_OK) return rc;
  if (batch == 0) return DERL_OK;
  DERL_REQUIRE(stem_tc_available(), "stem_conv_relu_mask: cuTensorMapEncodeTiled is unavailable");
  return launch_stem_tc(frames, reinterpret_cast<const long long*>(rows), batch, weight, bias, out,
                        DERL_DTYPE_F32, relu_mask, out_block, as_stream(stream));
}
