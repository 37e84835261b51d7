// K7t — backward of the NatureCNN stem (ReLU mask, bias gradient, weight gradient of
// nn.Conv2d(4, 32, 8, 4) + ReLU, derl/models.py:102-103) straight from the uint8 frames, on
// tcgen05.mma kind::i8 with the accumulators in tensor memory:
//     g[p, n]     = relu_mask[p, n] ? grad_out[p, n] : 0                      (400 pixels x 32)
//     dbias[n]   += sum_p g[p, n]
//     dW[n, c, 4a+i, 4b+j] += (1/255) * sum_{oy,ox} x[4(oy+a)+i, 4(ox+b)+j, c] * g[(oy,ox), n]
// Number format: the frame operand is the raw uint8 bytes (exact); the masked gradient is
// quantised per (frame, channel) into two signed 8-bit digit planes (block floating point):
// s = max_p |g[p, n]| / 127, g ~= s (q1 + q2 / 254), residual <= s / 508.  The int32 accumulation
// of a frame is exact; the per-frame tiles are scaled into fp32 running sums per CTA, and a second
// small kernel sums the CTA partials in a fixed order (float64), so the result is deterministic.
//
// Operand formulation:
//   * the frame lands by ONE TMA tensor copy in the row-permuted layout of K6t (plane i = image
//     rows 4Y + i: for every 4x4-pixel block m' = 21 Y + X its 16 bytes (j, c) at 16 m').  Read
//     as an MN-MAJOR no-swizzle UMMA operand that is A[tap = 16 i + 4 j + c][k = block m'] — core
//     matrix = 8 blocks x 16 tap bytes = 128 contiguous bytes, next 8 blocks +128 B (LBO), next
//     16 taps +7056 B (SBO) — and kernel quadrant (a, b) is the same operand started
//     16 (21 a + b) bytes later: no byte transpose, no fragment loads;
//   * the reduction index is the padded pixel number m = 21 oy + ox (one junk column per output
//     row, digits 0 there), so the quantiser writes the digits K-major, 16 consecutive m per
//     16-byte unit: Gq[m / 16][plane * 32 + channel][16] — the canonical K-major operand
//     (LBO 1024, SBO 128) with one 16-byte store per (group, channel, plane);
//   * per frame 4 quadrants x 14 K-steps of  D_q[64 taps x 64 (plane, channel)] += A * Gq^T
//     (M = 64, N = 64, K = 32), issued by one thread; an accumulator row (a tap) holds both digit
//     planes of all 32 channels, so the thread that owns it recombines and scales them;
//   * the ReLU mask arrives as 1 bit per activation (written by K6t with warp ballots, one word
//     per (32 padded pixels, channel)), not as the fp32 tensor.
// Per frame HBM reads: 28 224 (frame) + 51 200 (gradient) + 1 792 (mask) = 81 KB.
//
// Roles (576 threads, one persistent CTA per SM): warps 0-15 are workers — quantise frame f+1,
// then fold frame f's accumulators into their running sums (worker w owns quadrant w / 4 and the
// tensor-memory lane quarter w % 4 = tap row i) — warp 16 = TMA producer (frames, gradient tiles
// and mask words all double buffered), warp 17 = MMA issuer + TMEM owner.  MMAs of frame f
// overlap the quantisation of f+1.
#include <cuda.h>

#include "common.cuh"
#include "tcgen05.cuh"

namespace derl {
namespace {

constexpr int kImgBytes = 84 * 84 * 4;
constexpr int kPlaneBytes = 21 * 336;          // 7056
constexpr int kFrameBuf = 29824;               // frame + over-read slack (last K-step, last quadrant)
constexpr int kCh = 32, kPix = 400, kPixPad = 420;
constexpr int kKSteps = 14;                    // 448 padded pixels / 32
constexpr int kGroups = 28;                    // 16-pixel groups (k16 units); 27 hold pixels
constexpr int kGqBytes = kGroups * 64 * 16;    // 28672
constexpr int kGradBytes = kPix * kCh * 4;     // 51200
constexpr int kMaskBytes = 14 * 32 * 4;        // 1792: [tile of 32 padded pixels][channel] words
constexpr int kWorkers = 16, kWorkerThreads = kWorkers * 32;
constexpr int kThreads = kWorkerThreads + 64;
constexpr int kPartial = 4 * 64 * kCh;
constexpr uint32_t kTmemCols = 512;

constexpr int kGradBuf = kGradBytes + kMaskBytes;   // gradient tile + mask words, one buffer
struct BtSmem {   // byte offsets from a 128-aligned base
  static constexpr int frame = 0;                              // [2][29824]
  static constexpr int grad = frame + 2 * kFrameBuf;           // [2][51200 tile | 1792 mask]
  static constexpr int gq = grad + 2 * kGradBuf;               // [2][28672]
  static constexpr int red = gq + 2 * kGqBytes;                // float [2][16][32]
  static constexpr int scale = red + 2 * kWorkers * kCh * 4;   // float [2][32]
  static constexpr int table = scale + 2 * kCh * 4;            // unsigned [28 * 16] pixel table
  static constexpr int bars = table + 28 * 16 * 4;             // 16 mbarriers
  static constexpr int slot = bars + 16 * 8;
  static constexpr int bytes = slot + 16;
  static constexpr int alloc = bytes + 128;
};
static_assert(BtSmem::grad % 128 == 0 && kGradBuf % 128 == 0 && BtSmem::gq % 128 == 0 &&
                  BtSmem::bars % 8 == 0, "smem alignment");
static_assert(BtSmem::alloc <= 227 * 1024, "shared memory budget");

// A = frame taps (u8, MN-major), B = gradient digits (s8, K-major), D = int32 [64 x 64]
constexpr uint32_t kIdesc = umma_idesc_i8(64, 64, /*a u8*/ 0, /*b s8*/ 1, /*a MN-major*/ 1, 0);

// Two-digit quantisation of x in [-127, 127]: q1 = rint(x), q2 = rint((x - q1) * 254) (|q2| <= 127
// because |x - q1| <= 1/2 exactly).  Rounding by the 1.5 * 2^23 trick keeps the conversion pipe
// idle; the digits are the low bytes of the biased sums.
__device__ __forceinline__ void quantise2(float x, unsigned* b1, unsigned* b2) {
  const float m1 = x + 12582912.f;
  *b1 = __float_as_uint(m1);
  *b2 = __float_as_uint(__fmaf_rn(x - (m1 - 12582912.f), 254.f, 12582912.f));
}
__device__ __forceinline__ unsigned pack4b(unsigned a, unsigned b, unsigned c, unsigned d) {
  return __byte_perm(__byte_perm(a, b, 0x0040), __byte_perm(c, d, 0x0040), 0x5410);
}

__global__ void __launch_bounds__(kThreads, 1)
stem_bwd_tc_kernel(const __grid_constant__ CUtensorMap tm_frames, const long long* __restrict__ rows,
                   const float* __restrict__ grad_out, const unsigned* __restrict__ mask,
                   float* __restrict__ partial_w, float* __restrict__ partial_b, long long batch,
                   int blocked) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + (((raw_addr + 127u) & ~127u) - raw_addr);
  unsigned* table = reinterpret_cast<unsigned*>(smem + BtSmem::table);
  uint8_t* gq = smem + BtSmem::gq;
  float* red = reinterpret_cast<float*>(smem + BtSmem::red);
  float* scale = reinterpret_cast<float*>(smem + BtSmem::scale);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + BtSmem::bars);
  uint64_t* frame_full = bars;          // [2] TMA -> MMA
  uint64_t* frame_empty = bars + 2;     // [2] MMA -> TMA
  uint64_t* gq_full = bars + 4;         // [2] workers -> MMA (16 warp arrivals)
  uint64_t* gq_empty = bars + 6;        // [2] MMA -> workers
  uint64_t* tfull = bars + 8;           // [2] MMA -> workers
  uint64_t* tempty = bars + 10;         // [2] workers -> MMA (16 warp arrivals)
  uint64_t* grad_full = bars + 12;      // [2] TMA -> workers
  uint64_t* grad_empty = bars + 14;     // [2] workers -> TMA (16 warp arrivals)
  uint32_t* slot = reinterpret_cast<uint32_t*>(smem + BtSmem::slot);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const long long first = blockIdx.x, stride = gridDim.x;
  const int nframes = (int)((batch - first + stride - 1) / stride);

  if (tid == 0) {
    for (int i = 0; i < 2; ++i) {
      mbar_init(&frame_full[i], 1);
      mbar_init(&frame_empty[i], 1);
      mbar_init(&gq_full[i], kWorkers);
      mbar_init(&gq_empty[i], 1);
      mbar_init(&tfull[i], 1);
      mbar_init(&tempty[i], kWorkers);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&grad_full[i], 1);
      mbar_init(&grad_empty[i], kWorkers);
    }
    mbar_fence_init();
    tma_prefetch_desc(&tm_frames);
  }
  if (warp == kWorkers + 1) tmem_alloc(slot, kTmemCols);
  // digit buffers start as zeros: group 27 and the tail of group 26 are never written again
  for (int i = tid; i < 2 * kGqBytes / 16; i += kThreads) {
    reinterpret_cast<uint4*>(gq)[i] = make_uint4(0u, 0u, 0u, 0u);
  }
  // padded pixel m = 21 oy + ox -> float offset of its row in the gradient tile (plain or
  // space-to-depth(2) order).  The junk column and the tail point at row 0: their mask bits are 0.
  for (int m = tid; m < kGroups * 16; m += kThreads) {
    const int oy = m / 21, ox = m - oy * 21;
    unsigned entry = 0u;
    if (m < kPixPad && ox < 20) {
      const int row = blocked ? ((((oy >> 1) * 10 + (ox >> 1)) << 2) + ((oy & 1) << 1) + (ox & 1))
                              : oy * 20 + ox;
      entry = (unsigned)(row * kCh);
    }
    table[m] = entry;
  }
  fence_proxy_async_smem();
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem = *slot;

  if (warp == kWorkers) {
    // ===================================================================== TMA producer
    if (lane == 0) {
      for (int it = 0; it < nframes; ++it) {
        const long long f = first + (long long)it * stride;
        const int b = it & 1;
        // gradient tile first: its buffer was released when the workers copied tile it-2 to
        // registers, long before the MMAs of frame it-2 let go of the frame buffer — issuing in
        // this order gives the 53 KB a whole frame period to arrive (the other order made the
        // quantiser wait on HBM latency every frame: 27 % of the stall samples)
        mbar_wait(&grad_empty[b], (unsigned)(((it >> 1) & 1) ^ 1));
        mbar_expect_tx(&grad_full[b], kGradBytes + kMaskBytes);
        uint8_t* gbuf = smem + BtSmem::grad + b * kGradBuf;
        bulk_g2s(gbuf, grad_out + f * (kPix * kCh), kGradBytes, &grad_full[b]);
        bulk_g2s(gbuf + kGradBytes, mask + f * (kMaskBytes / 4), kMaskBytes, &grad_full[b]);
        mbar_wait(&frame_empty[b], (unsigned)(((it >> 1) & 1) ^ 1));
        mbar_expect_tx(&frame_full[b], kImgBytes);
        const long long src = rows ? __ldg(rows + f) : f;
        tma_load_4d(smem + BtSmem::frame + b * kFrameBuf, &tm_frames, 0, 0, 0, (int)src,
                    &frame_full[b]);
      }
    }
    __syncwarp();
  } else if (warp == kWorkers + 1) {
    // ===================================================================== MMA issuer
    // The whole warp runs the control flow (waits, descriptor arithmetic: warp-uniform, so it
    // lives in uniform registers); one elected lane issues the MMAs and the commits.
    for (int it = 0; it < nframes; ++it) {
      const int b = it & 1;
      const unsigned ph = (unsigned)((it >> 1) & 1);
      mbar_wait(&tempty[b], ph ^ 1u);
      mbar_wait(&frame_full[b], ph);
      mbar_wait(&gq_full[b], ph);
      tcgen05_fence_after();
      // Descriptors are built once per frame and advanced by adding to the 14-bit start-address
      // field (units of 16 B; shared-memory addresses stay below 2^18, so no carry leaves the
      // field): ~4 instructions per MMA instead of ~14 — with the full descriptor arithmetic per
      // MMA in a single divergent thread its issue rate, not the tensor pipe, set the frame time
      // (ncu: workers 34 % of their samples on the accumulator barrier, tensor pipe 32 % active).
      const uint64_t a_frame = umma_desc(smem_u32(smem + BtSmem::frame + b * kFrameBuf),
                                         /*lbo: next 8 blocks*/ 128, /*sbo: next 16 taps*/ kPlaneBytes);
      const uint64_t g_desc = umma_desc(smem_u32(gq + b * kGqBytes), 1024, 128);
      const uint32_t d0 = tmem + (uint32_t)(b * 256);
      if (elect_one_sync()) {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const uint64_t a_desc = a_frame + (uint64_t)(21 * (q >> 1) + (q & 1));   // 16 (21a + b) B
#pragma unroll
          for (int ks = 0; ks < kKSteps; ++ks) {
            umma_i8(d0 + q * 64, a_desc + (uint64_t)(ks * 32), g_desc + (uint64_t)(ks * 128), kIdesc,
                    ks != 0);
          }
        }
        umma_commit(&frame_empty[b]);
        umma_commit(&gq_empty[b]);
        umma_commit(&tfull[b]);
      }
      __syncwarp();
    }
  } else {
    // ===================================================================== workers
    const int ch = lane;                       // quantiser role: one channel per lane
    const int quad = warp >> 2, quarter = warp & 3;   // accumulator role
    float wsum[16];   // [row select][rep][h]: rows t/4 (+8), channels 8 rep + 2 (t % 4) + h
#pragma unroll
    for (int k = 0; k < 16; ++k) wsum[k] = 0.f;
    float bsum = 0.f;

    auto quantise_frame = [&](int it) {
      const int b = it & 1;
      float v[2][16];
      const float* grad_sm = reinterpret_cast<const float*>(smem + BtSmem::grad + b * kGradBuf);
      const unsigned* mask_sm = reinterpret_cast<const unsigned*>(
          smem + BtSmem::grad + b * kGradBuf + kGradBytes);
      mbar_wait(&grad_full[b], (unsigned)((it >> 1) & 1));
      float vmax = 0.f, vsum = 0.f;
#pragma unroll
      for (int k = 0; k < 2; ++k) {
        const int group = warp + kWorkers * k;      // warp-uniform; groups >= 27 hold no pixel
        if (group < kGroups - 1) {
          // this channel's ReLU bits of the 16 pixels: half of a 32-pixel mask word
          const unsigned bits = mask_sm[(group >> 1) * kCh + ch] >> ((group & 1) * 16);
          const uint4* tab = reinterpret_cast<const uint4*>(table + group * 16);
#pragma unroll
          for (int e4 = 0; e4 < 4; ++e4) {
            const uint4 off = tab[e4];                // broadcast: 4 row offsets per load
            const unsigned o[4] = {off.x, off.y, off.z, off.w};
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const int e = 4 * e4 + j;
              const float x = grad_sm[o[j] + ch];
              const float g = (bits >> e) & 1u ? x : 0.f;
              v[k][e] = g;
              vmax = fmaxf(vmax, fabsf(g));
              vsum += g;
            }
          }
        } else {
#pragma unroll
          for (int e = 0; e < 16; ++e) v[k][e] = 0.f;
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&grad_empty[b]);  // the tile is in registers: refill the buffer
      bsum += vsum;
      float* r = red + (it & 1) * (kWorkers * kCh);
      r[warp * kCh + ch] = vmax;
      named_bar_sync(1, kWorkerThreads);
      float mx = r[ch];
#pragma unroll
      for (int k = 1; k < kWorkers; ++k) mx = fmaxf(mx, r[k * kCh + ch]);
      const float s = mx > 0.f ? mx / 127.f : 1.f, inv = 1.f / s;
      mbar_wait(&gq_empty[b], (unsigned)(((it >> 1) & 1) ^ 1));   // MMAs of frame it-2 have read it
      if (warp == 0) scale[b * kCh + ch] = s * (1.f / 254.f);   // folds (q1 * 254 + q2) back
      uint8_t* out = gq + b * kGqBytes;
#pragma unroll
      for (int k = 0; k < 2; ++k) {
        const int group = warp + kWorkers * k;
        if (group < kGroups - 1) {
          unsigned w1[4], w2[4];
#pragma unroll
          for (int qq = 0; qq < 4; ++qq) {
            unsigned b1[4], b2[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) quantise2(v[k][4 * qq + e] * inv, &b1[e], &b2[e]);
            w1[qq] = pack4b(b1[0], b1[1], b1[2], b1[3]);
            w2[qq] = pack4b(b2[0], b2[1], b2[2], b2[3]);
          }
          *reinterpret_cast<uint4*>(out + group * 1024 + ch * 16) =
              make_uint4(w1[0], w1[1], w1[2], w1[3]);
          *reinterpret_cast<uint4*>(out + group * 1024 + (32 + ch) * 16) =
              make_uint4(w2[0], w2[1], w2[2], w2[3]);
        }
      }
      fence_proxy_async_smem();                    // digits -> visible to the tensor core
      __syncwarp();
      if (lane == 0) mbar_arrive(&gq_full[b]);
    };

    auto fold_frame = [&](int it) {
      const int b = it & 1;
      mbar_wait(&tfull[b], (unsigned)((it >> 1) & 1));
      tcgen05_fence_after();
      // the M = 64 accumulator of quadrant `quad` occupies lanes 0-15 of every 32-lane quarter
      // (row = 16 quarter + lane): the 16x256b fragment spreads those 16 rows x 64 columns over
      // all 32 threads — thread t: rows t/4 and t/4 + 8, columns 8 rep + 2 (t % 4) + {0, 1}.
      // Columns c and 32 + c (the two digit planes of channel c) land in the same thread.
      const uint32_t taddr = tmem + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(b * 256 + quad * 64);
      uint32_t v[32];
      tmem_ld_16x256x8(taddr, v);
      tmem_ld_wait();
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&tempty[b]);
      const float* sc = scale + b * kCh + 2 * (lane & 3);
#pragma unroll
      for (int rep = 0; rep < 4; ++rep) {
        const float2 s2 = *reinterpret_cast<const float2*>(sc + 8 * rep);
#pragma unroll
        for (int rs = 0; rs < 2; ++rs) {
#pragma unroll
          for (int h = 0; h < 2; ++h) {
            // exact: |acc1 * 254 + acc2| <= 256 * 255 * 127 * 255 < 2^31
            const int both = (int)v[4 * rep + 2 * rs + h] * 254 + (int)v[4 * (rep + 4) + 2 * rs + h];
            wsum[(rs * 4 + rep) * 2 + h] += (float)both * (h ? s2.y : s2.x);
          }
        }
      }
    };

    quantise_frame(0);
    for (int it = 0; it < nframes; ++it) {
      if (it + 1 < nframes) quantise_frame(it + 1);
      fold_frame(it);
    }

    // ---- per-CTA partials: partial_w[cta][quadrant][tap = 16 i + 4 j + c][channel]
#pragma unroll
    for (int rs = 0; rs < 2; ++rs) {
      float* pw = partial_w + (size_t)blockIdx.x * kPartial +
                  (size_t)(quad * 64 + quarter * 16 + (lane >> 2) + 8 * rs) * kCh + 2 * (lane & 3);
#pragma unroll
      for (int rep = 0; rep < 4; ++rep) {
        *reinterpret_cast<float2*>(pw + 8 * rep) =
            make_float2(wsum[(rs * 4 + rep) * 2], wsum[(rs * 4 + rep) * 2 + 1]);
      }
    }
    named_bar_sync(1, kWorkerThreads);
    red[warp * kCh + ch] = bsum;
    named_bar_sync(1, kWorkerThreads);
    if (warp == 0) {
      float bt = 0.f;
#pragma unroll
      for (int k = 0; k < kWorkers; ++k) bt += red[k * kCh + ch];
      partial_b[(size_t)blockIdx.x * kCh + ch] = bt;
    }
  }
  tcgen05_fence_before();
  __syncthreads();
  if (warp == kWorkers + 1) {
    tcgen05_fence_after();
    tmem_dealloc(tmem, kTmemCols);
  }
}

// grad_w[n][c][4a+i][4b+j] = (1/255) * sum_cta partial_w[cta][a*2+b][(i*4+j)*4+c][n]
// Blocks 0 .. kPartial/32 - 1 take 32 consecutive elements of the partial layout (one 128-byte
// line per CTA partial); the block's 8 warps sum interleaved subsets of the CTAs and the subsets
// are then added in fixed order.  The last block sums the bias partials the same way.
__global__ void __launch_bounds__(256)
stem_bwd_reduce_kernel(const float* __restrict__ partial_w, const float* __restrict__ partial_b,
                       int ctas, float* __restrict__ grad_w, float* __restrict__ grad_b) {
  constexpr int kSlots = 8;
  __shared__ double slot[kSlots][32];
  const int lane = threadIdx.x & 31, k = threadIdx.x >> 5;
  const bool bias = blockIdx.x == kPartial / 32;
  const float* src = bias ? partial_b + lane : partial_w + (size_t)blockIdx.x * 32 + lane;
  const size_t pitch = bias ? kCh : kPartial;
  double s = 0.0;
#pragma unroll 4
  for (int b = k; b < ctas; b += kSlots) s += (double)__ldg(src + (size_t)b * pitch);
  slot[k][lane] = s;
  __syncthreads();
  if (threadIdx.x < 32) {
    double total = 0.0;
#pragma unroll
    for (int q = 0; q < kSlots; ++q) total += slot[q][lane];
    if (bias) {
      grad_b[lane] = (float)total;
    } else {
      const int e = blockIdx.x * 32 + lane;   // over [4 quadrants][64 taps][32 ch]
      const int n = e & 31, tap = (e >> 5) & 63, quadrant = e >> 11;
      const int c = tap & 3, j = (tap >> 2) & 3, i = tap >> 4;
      const int kh = 4 * (quadrant >> 1) + i, kw = 4 * (quadrant & 1) + j;
      grad_w[((n * 4 + c) * 8 + kh) * 8 + kw] = (float)(total * (1.0 / 255.0));
    }
  }
}

struct FramesMapCache {
  const void* base[8];
  long long n[8];
  CUtensorMap map[8];
  int used = 0, next = 0;
};

bool frames_map(CUtensorMap* out, const void* base, long long n) {
  static thread_local FramesMapCache cache;
  for (int i = 0; i < cache.used; ++i) {
    if (cache.base[i] == base && cache.n[i] == n) {
      *out = cache.map[i];
      return true;
    }
  }
  TmapEncodeFn enc = tmap_encode_fn();
  if (enc == nullptr) return false;
  cuuint64_t dims[4] = {84, 21, 4, (cuuint64_t)n};
  cuuint64_t strides[3] = {4 * 336, 336, (cuuint64_t)kImgBytes};
  cuuint32_t box[4] = {84, 21, 4, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  if (enc(out, CU_TENSOR_MAP_DATA_TYPE_UINT32, 4, const_cast<void*>(base), dims, strides, box, estr,
          CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
    return false;
  const int s = cache.used < 8 ? cache.used++ : cache.next;
  cache.next = (s + 1) % 8;
  cache.base[s] = base;
  cache.n[s] = n;
  cache.map[s] = *out;
  return true;
}

}  // namespace

bool stem_tc_available();
}  // namespace derl

using namespace derl;

// one CTA per SM: [grid][kPartial] weight partials, then [grid][kCh] bias partials
extern "C" size_t derl_b200_stem_backward_workspace_bytes(void) {
  return (size_t)sm_count() * (kPartial + kCh) * sizeof(float);
}

extern "C" int derl_b200_stem_backward_masked(const uint8_t* frames, const int64_t* rows_dev,
                                              int64_t batch, const float* grad_out,
                                              const uint32_t* relu_mask, int blocked,
                                              float* grad_weight, float* grad_bias,
                                              void* workspace, size_t workspace_bytes,
                                              void* stream) {
  DERL_REQUIRE(frames && grad_out && relu_mask && grad_weight && grad_bias && workspace &&
                   batch >= 1, "stem_backward_masked: bad arguments");
  DERL_REQUIRE(blocked == 0 || blocked == 1, "stem_backward_masked: blocked must be 0 or 1");
  DERL_REQUIRE((((uintptr_t)frames | (uintptr_t)grad_out | (uintptr_t)relu_mask) & 15) == 0,
               "stem_backward_masked: inputs must be 16-byte aligned");
  int rc = require_device();
  if (rc != DERL_OK) return rc;
  if (workspace_bytes < derl_b200_stem_backward_workspace_bytes()) {
    set_error("stem_backward_masked: workspace %zu B too small", workspace_bytes);
    return DERL_E_WORKSPACE;
  }
  DERL_REQUIRE(stem_tc_available(), "stem_backward_masked: cuTensorMapEncodeTiled is unavailable");
  const long long* rows = reinterpret_cast<const long long*>(rows_dev);
  CUtensorMap tm_frames;
  if (!frames_map(&tm_frames, frames, rows ? (1ll << 30) : batch)) {
    set_error("stem_backward: cuTensorMapEncodeTiled failed (batch %lld)", (long long)batch);
    return DERL_E_CUDA;
  }
  if (int rc_attr = ensure_dynamic_smem(reinterpret_cast<const void*>(stem_bwd_tc_kernel),
                                        BtSmem::alloc))
    return rc_attr;
  cudaStream_t st = as_stream(stream);
  long long grid = sm_count();
  if (grid > batch) grid = batch;
  float* partial_w = reinterpret_cast<float*>(workspace);
  float* partial_b = partial_w + (size_t)grid * kPartial;
  stem_bwd_tc_kernel<<<(unsigned)grid, kThreads, BtSmem::alloc, st>>>(
      tm_frames, rows, grad_out, relu_mask, partial_w, partial_b, batch, blocked);
  DERL_LAUNCH_CHECK("stem_bwd_tc_kernel");
  stem_bwd_reduce_kernel<<<kPartial / 32 + 1, 256, 0, st>>>(partial_w, partial_b, (int)grid,
                                                           grad_weight, grad_bias);
  DERL_LAUNCH_CHECK("stem_bwd_reduce_kernel");
  return DERL_OK;
}
