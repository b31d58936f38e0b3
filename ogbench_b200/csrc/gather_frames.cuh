// Image-observation gathers with frame stacking and the random-crop shift fused in.
//
//   out[g, y, x, f*C + c] = frame_f(g)[ clamp(y + dy_g, 0, H-1), clamp(x + dx_g, 0, W-1), c ]
//   frame_f(g) = observations[ max(row_g - (FS-1-f), first_row_g) ]          (oldest frame first)
//
// which is datasets.py:359-366 (get_stacked_observations) followed by datasets.py:17-33,329-339
// (edge-pad by `padding`, dynamic_slice at (cy, cx); dy = cy - padding, dx = cx - padding) in closed form.
// The reference materialises the stacked batch and then round-trips every key through an XLA device for the
// crop; here each output byte is produced once, straight from the un-stacked resident frames.
//
// gather_frames_tma_kernel: uint8 HWC images with C == 3 (the 64x64x3 OGBench pixels).
//   * load  : one cp.async.bulk.tensor (TMA, tile mode) per source frame and row band.  The box is issued at row
//             coordinate y0+dy, so the vertical crop shift is applied by the TMA unit; rows outside the image
//             arrive as zero fill and are never read (row index clamp = edge replication).  The innermost TMA
//             coordinate has to stay 16-byte aligned (an unaligned one faults on sm_100a), so the horizontal
//             shift of 3*dx bytes is applied when reading shared memory: 13 words + a funnel shift per frame,
//             and the first/last pixel group patches its out-of-image pixels with the edge pixel in registers.
//   * permute: each thread turns 16 pixels x FS frames into 16 x 3FS interleaved output bytes with byte permutes
//             and writes them as 16-byte shared stores into the output image.
//   * store : one cp.async.bulk (TMA) shared->global per band; the band is a contiguous, 16-byte-aligned span
//             of the dense output.
// gather_frames_generic_kernel: any dtype / shape / padding, element-granular; correctness fallback on device.
#pragma once
#include <cuda.h>
#include "device_common.cuh"

namespace ogb {

constexpr int kMaxFrameJobs = 16;
constexpr int kFramesThreads = 128;
constexpr int kGroupPx = 16;  // pixels per thread task: 16 px * 3 B = 48 B = 3 x 16-byte loads per frame

struct FrameJob {
  const uint8_t* src;     // generic kernel only
  uint8_t* dst;           // dense [total_rows, H, W, FS*C*itemsize]
  int64_t src_row_stride; // bytes between consecutive dataset rows of the source field
  int32_t slot;
  int32_t crop;           // this key is in the reference's augmentation list
  int32_t fs;             // frames to stack (1 = plain gather)
  int32_t pad_;
};

struct FramesParams {
  const int32_t* vec_rows;   // [slot][total_rows]
  const int32_t* vec_init;   // [slot][total_rows] first row of the trajectory segment (may be null when fs == 1)
  const int8_t* crop;        // [total_rows][2] (dy, dx), -128 = not augmented; may be null
  int64_t total_rows;
  int64_t row_begin, row_end; // rows this launch handles
  int32_t H, W;              // image rows / pixels per row
  int32_t inner_bytes;       // C * itemsize
  int32_t band_rows;         // TMA kernel: rows per CTA item
  int32_t n_bands;
  int32_t n_jobs;
  FrameJob jobs[kMaxFrameJobs];
};

// ------------------------------------------------ PTX wrappers ------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "WAIT_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra.uni WAIT_DONE;\n\t"
      "bra.uni WAIT_LOOP;\n\t"
      "WAIT_DONE:\n\t}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// TMA tile load of a [1, rows, row_bytes] box of the u8 tensor (row_bytes, H, N) into shared memory
__device__ __forceinline__ void tma_load_3d(void* smem_dst, const CUtensorMap* tmap, int c0, int c1, int c2, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
      ::"r"(smem_u32(smem_dst)), "l"(tmap), "r"(c0), "r"(c1), "r"(c2), "r"(smem_u32(bar)) : "memory");
}
// TMA bulk store shared -> global (contiguous, 16-byte aligned, size multiple of 16)
__device__ __forceinline__ void tma_store_bulk(void* gmem_dst, const void* smem_src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gmem_dst), "r"(smem_u32(smem_src)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_store_commit_and_wait_read() {
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
  asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}

// byte helpers on register arrays; all indices are compile-time constants after unrolling
__device__ __forceinline__ uint32_t get_byte(const uint32_t* w, int byte_index) {
  return (w[byte_index >> 2] >> (8 * (byte_index & 3))) & 0xffu;
}
__device__ __forceinline__ void set_byte(uint32_t* w, int byte_index, uint32_t v) {
  const int sh = 8 * (byte_index & 3);
  w[byte_index >> 2] = (w[byte_index >> 2] & ~(0xffu << sh)) | (v << sh);
}

// Shared-memory distance between the FS source bands: a tensor (TMA) copy needs a 128-byte-aligned shared destination,
// and band_rows * W * 3 is not a multiple of 128 for every band height (17 rows of 16 px: 816 B).
__host__ __device__ constexpr int frame_stride_bytes(int band_bytes) { return (band_bytes + 127) & ~127; }

// ------------------------------------------------ TMA kernel ------------------------------------------------
// grid: one CTA per (batch row g, job, band); dynamic smem = FS * (frame_stride_bytes(band_bytes) + band_bytes), with
// band_bytes = band_rows * W * 3.
template <int FS>
__global__ void __launch_bounds__(kFramesThreads) gather_frames_tma_kernel(const __grid_constant__ CUtensorMap tmap,
                                                                           const __grid_constant__ FramesParams p) {
  constexpr int C = 3;
  constexpr int kSrcWords = kGroupPx * C / 4;        // 12 words per frame per task
  constexpr int kOutWords = kSrcWords * FS;          // 36 for FS = 3
  constexpr int kMaxPad = 4;                         // edge patch handles |dx| <= 4
  extern __shared__ __align__(128) uint8_t smem[];
  __shared__ __align__(8) uint64_t bar;

  const int row_bytes = p.W * C;                     // one image row of one frame
  const int RB = p.band_rows;
  const int band_bytes = RB * row_bytes;             // per frame
  const int frame_stride = frame_stride_bytes(band_bytes);
  uint8_t* s_in = smem;
  uint8_t* s_out = smem + (size_t)FS * frame_stride;

  const int64_t item = blockIdx.x;
  const int band = (int)(item % p.n_bands);
  const int j = (int)((item / p.n_bands) % p.n_jobs);
  const int64_t g = p.row_begin + item / ((int64_t)p.n_bands * p.n_jobs);
  const FrameJob& job = p.jobs[j];

  int dy = 0, dx = 0;
  if (job.crop && p.crop != nullptr) {
    const int cy = p.crop[2 * g], cx = p.crop[2 * g + 1];
    if (cy != -128) { dy = cy; dx = cx; }
  }
  const int y0 = band * RB;

  if (threadIdx.x == 0) {
    mbar_init(&bar, 1);
    fence_barrier_init();
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    const int32_t row = p.vec_rows[(int64_t)job.slot * p.total_rows + g];
    const int32_t first = (FS > 1) ? p.vec_init[(int64_t)job.slot * p.total_rows + g] : row;
    mbar_expect_tx(&bar, (uint32_t)(FS * band_bytes));
#pragma unroll
    for (int f = 0; f < FS; ++f) {
      int32_t fr = row - (FS - 1 - f);
      fr = fr > first ? fr : first;                  // np.maximum(idxs - i, initial_state_idxs)  datasets.py:364
      tma_load_3d(s_in + (size_t)f * frame_stride, &tmap, 0, y0 + dy, fr, &bar);
    }
  }
  mbar_wait(&bar, 0);

  // valid (in-image) part of what the TMA delivered; everything else is zero fill to be replaced by the edge
  const int r_lo = max(0, -(y0 + dy)), r_hi = min(RB - 1, p.H - 1 - y0 - dy);
  const int groups = p.W / kGroupPx;
  const int out_row_bytes = row_bytes * FS;

  for (int task = threadIdx.x; task < RB * groups; task += blockDim.x) {
    const int rr = task / groups, gq = task - rr * groups;
    const int rc = min(max(rr, r_lo), r_hi);         // row clamp = edge replication in y
    uint32_t src[FS][kSrcWords];
    if (dx == 0) {                                   // aligned fast path: 3 x 16-byte shared loads per frame
#pragma unroll
      for (int f = 0; f < FS; ++f) {
        const uint4* sp = reinterpret_cast<const uint4*>(s_in + (size_t)f * frame_stride + (size_t)rc * row_bytes + gq * (kGroupPx * C));
#pragma unroll
        for (int q = 0; q < kSrcWords / 4; ++q) {
          const uint4 v = sp[q];
          src[f][4 * q + 0] = v.x; src[f][4 * q + 1] = v.y; src[f][4 * q + 2] = v.z; src[f][4 * q + 3] = v.w;
        }
      }
    } else {
      // x shift: the 48-byte window starts 3*dx bytes off the group boundary -> 13 words + a funnel shift.
      // Word indices are clamped into the row; bytes fetched through a clamped index only ever belong to
      // out-of-image pixels, which the edge patch below overwrites.
      const int o = gq * (kGroupPx * C) + C * dx;
      const int w0 = o >> 2;                         // floor(o / 4), also for negative o
      const uint32_t sh8 = (uint32_t)(o & 3) * 8u;
      const int last_word = (row_bytes >> 2) - 1;
#pragma unroll
      for (int f = 0; f < FS; ++f) {
        const uint32_t* rowp = reinterpret_cast<const uint32_t*>(s_in + (size_t)f * frame_stride + (size_t)rc * row_bytes);
        uint32_t w[kSrcWords + 1];
#pragma unroll
        for (int k = 0; k <= kSrcWords; ++k) w[k] = rowp[min(max(w0 + k, 0), last_word)];
#pragma unroll
        for (int k = 0; k < kSrcWords; ++k) src[f][k] = __funnelshift_r(w[k], w[k + 1], sh8);
      }
      // edge replication in x: only the first group (dx < 0) or the last group (dx > 0) has out-of-image pixels
      if (dx < 0 && gq == 0) {
#pragma unroll
        for (int f = 0; f < FS; ++f) {
          const uint8_t* px = s_in + (size_t)f * frame_stride + (size_t)rc * row_bytes;   // source pixel 0
          const uint32_t e0 = px[0], e1 = px[1], e2 = px[2];
#pragma unroll
          for (int k = 0; k < kMaxPad; ++k) {
            if (k < -dx) { set_byte(src[f], 3 * k, e0); set_byte(src[f], 3 * k + 1, e1); set_byte(src[f], 3 * k + 2, e2); }
          }
        }
      } else if (dx > 0 && gq == groups - 1) {
#pragma unroll
        for (int f = 0; f < FS; ++f) {
          const uint8_t* px = s_in + (size_t)f * frame_stride + (size_t)rc * row_bytes + (p.W - 1) * C;  // source pixel W-1
          const uint32_t e0 = px[0], e1 = px[1], e2 = px[2];
#pragma unroll
          for (int k = 0; k < kMaxPad; ++k) {
            const int q = kGroupPx - 1 - k;
            if (k < dx) { set_byte(src[f], 3 * q, e0); set_byte(src[f], 3 * q + 1, e1); set_byte(src[f], 3 * q + 2, e2); }
          }
        }
      }
    }
    // interleave: output byte o of the group = pixel o / (3 FS), channel o % (3 FS) -> frame ch / 3, colour ch % 3
    uint32_t out[kOutWords];
#pragma unroll
    for (int k = 0; k < kOutWords; ++k) {
      uint32_t w = 0;
#pragma unroll
      for (int b = 0; b < 4; ++b) {
        const int o = 4 * k + b;
        const int px = o / (C * FS), ch = o % (C * FS);
        const int f = ch / C, c = ch % C;
        w |= get_byte(src[f], px * C + c) << (8 * b);
      }
      out[k] = w;
    }
    uint4* dp = reinterpret_cast<uint4*>(s_out + (size_t)rr * out_row_bytes + (size_t)gq * (kGroupPx * C * FS));
#pragma unroll
    for (int q = 0; q < kOutWords / 4; ++q) dp[q] = make_uint4(out[4 * q], out[4 * q + 1], out[4 * q + 2], out[4 * q + 3]);
  }
  fence_async_smem();  // make the generic-proxy shared stores visible to the TMA (async proxy) store
  __syncthreads();
  if (threadIdx.x == 0) {
    uint8_t* gdst = job.dst + ((size_t)g * p.H + y0) * out_row_bytes;
    tma_store_bulk(gdst, s_out, (uint32_t)(RB * out_row_bytes));
    tma_store_commit_and_wait_read();
  }
}

// ------------------------------------------------ generic fallback ------------------------------------------------
// One thread per output chunk of `1 << vec_log2` bytes; chunk index space [g][y][x][f][inner / vec].
__global__ void __launch_bounds__(256) gather_frames_generic_kernel(const __grid_constant__ FramesParams p, const int job_index,
                                                                    const int vec_log2) {
  const FrameJob& job = p.jobs[job_index];
  const int fs = job.fs;
  const int chunks_inner = p.inner_bytes >> vec_log2;
  const int64_t per_row = (int64_t)p.H * p.W * fs * chunks_inner;
  const int64_t total = p.row_end * per_row;
  for (int64_t e = p.row_begin * per_row + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int64_t g = e / per_row;
    int64_t rem = e - g * per_row;
    const int ci = (int)(rem % chunks_inner); rem /= chunks_inner;
    const int f = (int)(rem % fs); rem /= fs;
    const int x = (int)(rem % p.W);
    const int y = (int)(rem / p.W);
    int dy = 0, dx = 0;
    if (job.crop && p.crop != nullptr) {
      const int cy = p.crop[2 * g], cx = p.crop[2 * g + 1];
      if (cy != -128) { dy = cy; dx = cx; }
    }
    const int sy = min(max(y + dy, 0), p.H - 1), sx = min(max(x + dx, 0), p.W - 1);
    const int32_t row = p.vec_rows[(int64_t)job.slot * p.total_rows + g];
    int32_t fr = row;
    if (fs > 1) {
      const int32_t first = p.vec_init[(int64_t)job.slot * p.total_rows + g];
      fr = row - (fs - 1 - f);
      fr = fr > first ? fr : first;
    }
    const uint8_t* sp = job.src + (size_t)fr * job.src_row_stride + ((size_t)sy * p.W + sx) * p.inner_bytes + ((size_t)ci << vec_log2);
    uint8_t* dp = job.dst + (size_t)e * ((size_t)1 << vec_log2);
    switch (vec_log2) {
      case 4: *reinterpret_cast<uint4*>(dp) = __ldg(reinterpret_cast<const uint4*>(sp)); break;
      case 3: *reinterpret_cast<uint2*>(dp) = __ldg(reinterpret_cast<const uint2*>(sp)); break;
      case 2: *reinterpret_cast<uint32_t*>(dp) = __ldg(reinterpret_cast<const uint32_t*>(sp)); break;
      case 1: *reinterpret_cast<uint16_t*>(dp) = __ldg(reinterpret_cast<const uint16_t*>(sp)); break;
      default: *dp = __ldg(sp); break;
    }
  }
}

}  // namespace ogb
