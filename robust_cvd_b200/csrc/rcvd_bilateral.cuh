// rcvd_bilateral.cuh -- spatio-temporal bilateral depth filter (DepthVideoProcessor::bilateralFilter, reference
// lib/Processor.cpp:183-313).
//
// One thread per output pixel, one CTA per 32 x 8 output tile of one frame.  The window frames are visited in the
// reference's order (window frame, then row, then column): one TMA load (cp.async.bulk.tensor.3d, one elected thread)
// stages the depth halo tile of a window frame -- and the colour halo tile when the colour term is on -- into a two-slot
// shared-memory ring, completion signalled on an mbarrier, so the next frame's tile is in flight while the current one is
// consumed.  Only one frame is resident per slot, so the shared-memory footprint depends on the spatial radius alone.
// The window itself is clamped to the image (not padded); halo elements outside the image are loaded but never read.
//
// Weight of a sample (:265-280): exponent = 0 (+ -(d - d_ref)^2 / depthSigma^2 if depthSigma > 0) (+ -(sum over channels 0, 1, 2
// of (c - c_ref)^2) / colorSigma^2 if colorSigma > 0); weight = exponent != 0 ? expf(exponent) : 1.  Float32 with explicit
// round-to-nearest intrinsics (no FMA contraction) and the accurate expf.  Output: weighted mean (sumWeight > 0, else 0), or the
// first depth of the (depth, weight)-sorted samples whose cumulative weight reaches sumWeight / 2 (0 if none does: NaN weights,
// where the reference leaves the pixel uninitialised).
//
// Layout: padded depth planes [P][Hp][Wp] f32 and colour planes [F][Hp][3 Wp] f32 (interleaved channels).  Image pixel (y, x)
// sits at padded (y + r, x + pad_l) with pad_l = r rounded up to a multiple of 4, the rest is zero.  Every halo box then starts
// at the padded coordinate (tile_y, tile_x): never negative and always 16-byte aligned, and Wp / Hp are at least one box, so
// the TMA reads past the tensor only at its far ends.  Wp is a multiple of 4, so every stride is a multiple of 16 bytes.
// Planes 0..F-1 are the transformed
// depth of the frames; with in_place, plane F + k receives output k after the depth transform of its frame has been applied
// again (what DepthFrame::depth() returns after setDepth, lib/DepthStream.cpp:275-291), and later launches read that plane for
// the frame instead of plane f.
#pragma once
#include <cuda.h>
#include <stdint.h>
#include "rcvd_update.cuh"
#include "rcvd_dense.cuh"

namespace rcvd {

constexpr int kBilTW = 32, kBilTH = 8, kBilThreads = kBilTW * kBilTH;

struct BilateralArgs {
  float* out;                    // [num_out][h][w]
  float* depth;                  // depth planes (see above); written only at planes F + k (in place)
  const float* color;            // nullptr when the colour term is off
  const int* out_frames;         // [num_out] local frame index of output k, ascending
  const int* retrans;            // [F] output index of the frame, -1 if it is not an output (in place)
  const double* xparams;         // [num_out][L.nf] frame parameter vector, depth-transform params at L.offD (in place)
  float2* scratch;               // median: [pixels of the launch][max_samples] (depth, weight)
  rcvd_config cfg; Layout L;     // depth transform (in place)
  int F, w, h, Wp, Hp, pad_l;
  int out_begin;                 // output index of blockIdx.z == 0
  int y_begin, y_end;            // rows of this launch (row bands of the median scratch)
  int spatial_radius, frame_radius, max_samples;
  int box_w, box_h;              // TMA boxes: depth [box_h][box_w], colour [box_h][3 box_w] floats
  uint32_t stage_bytes, depth_bytes;   // one ring slot / its depth part (both multiples of 1024 bytes)
  float depth_sigma2, color_sigma2;    // <= 0: term off
};

__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
               ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2) : "memory");
}

// (depth, weight) lexicographic order of std::sort on std::pair<float, float>
__device__ __forceinline__ bool pair_less(float2 a, float2 b) { return a.x < b.x || (a.x == b.x && a.y < b.y); }

template <bool MEDIAN, bool IN_PLACE>
__global__ void __launch_bounds__(kBilThreads) k_bilateral(const __grid_constant__ CUtensorMap tm_depth, const __grid_constant__ CUtensorMap tm_color,
                                                           BilateralArgs a) {
  extern __shared__ __align__(128) unsigned char bil_smem[];
  uint64_t* bars = reinterpret_cast<uint64_t*>(bil_smem + 2 * a.stage_bytes);
  const int tx = threadIdx.x % kBilTW, ty = threadIdx.x / kBilTW;
  const int tile_x = blockIdx.x * kBilTW, tile_y = a.y_begin + blockIdx.y * kBilTH;
  const int x = tile_x + tx, y = tile_y + ty;
  const bool live = x < a.w && y < a.y_end;
  const int k = a.out_begin + blockIdx.z;
  const int frame = a.out_frames[k];
  const int r = a.spatial_radius;
  const int f0 = max(0, frame - a.frame_radius), f1 = min(a.F - 1, frame + a.frame_radius), nf = f1 - f0 + 1;
  const bool use_d = a.depth_sigma2 > 0.f, use_c = a.color_sigma2 > 0.f;
  const int ox = tile_x - a.pad_l, oy = tile_y - r;   // image coordinates of halo element (0, 0)
  const int cw = 3 * a.Wp, cbox_w = 3 * a.box_w;

  auto issue = [&](int i) {   // window frame f0 + i into ring slot i & 1
    const int g = f0 + i;
    const int plane = (IN_PLACE && g < frame && a.retrans[g] >= 0) ? a.F + a.retrans[g] : g;   // filtered earlier in this call
    unsigned char* slot = bil_smem + (size_t)(i & 1) * a.stage_bytes;
    uint64_t* bar = bars + (i & 1);
    mbar_expect_tx(bar, (uint32_t)(a.box_w * a.box_h * 4 + (use_c ? cbox_w * a.box_h * 4 : 0)));
    tma_load_3d(slot, &tm_depth, bar, tile_x, tile_y, plane);   // padded coordinates of halo element (0, 0)
    if (use_c) tma_load_3d(slot + a.depth_bytes, &tm_color, bar, 3 * tile_x, tile_y, g);
  };
  if (threadIdx.x == 0) {
    mbar_init(bars, 1); mbar_init(bars + 1, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    issue(0);
    if (nf > 1) issue(1);
  }
  __syncthreads();

  float dref = 0.f, cr0 = 0.f, cr1 = 0.f, cr2 = 0.f;
  if (live) {
    dref = a.depth[((size_t)frame * a.Hp + y + r) * a.Wp + x + a.pad_l];
    if (use_c) { const float* c = a.color + ((size_t)frame * a.Hp + y + r) * cw + 3 * (x + a.pad_l); cr0 = c[0]; cr1 = c[1]; cr2 = c[2]; }
  }
  const int x0 = max(0, x - r), x1 = min(a.w - 1, x + r), y0 = max(0, y - r), y1 = min(a.h - 1, y + r);
  const size_t pix = ((size_t)blockIdx.z * (a.y_end - a.y_begin) + (y - a.y_begin)) * a.w + x;
  float2* mine = MEDIAN && live ? a.scratch + pix * a.max_samples : nullptr;
  int n = 0; float dsum = 0.f, wsum = 0.f;
  for (int i = 0; i < nf; ++i) {
    mbar_wait(bars + (i & 1), (uint32_t)((i >> 1) & 1));
    if (live) {
      const float* D = reinterpret_cast<const float*>(bil_smem + (size_t)(i & 1) * a.stage_bytes);
      const float* Cs = reinterpret_cast<const float*>(bil_smem + (size_t)(i & 1) * a.stage_bytes + a.depth_bytes);
      for (int wy = y0; wy <= y1; ++wy) {
        const float* drow = D + (wy - oy) * a.box_w - ox;
        const float* crow = Cs + (wy - oy) * cbox_w - 3 * ox;
        for (int wx = x0; wx <= x1; ++wx) {
          const float d = drow[wx];
          float e = 0.f;
          if (use_d) {
            const float diff = __fsub_rn(d, dref);
            e = __fadd_rn(e, __fdiv_rn(-__fmul_rn(diff, diff), a.depth_sigma2));
          }
          if (use_c) {
            const float* c = crow + 3 * wx;
            const float c0 = __fsub_rn(c[0], cr0), c1 = __fsub_rn(c[1], cr1), c2 = __fsub_rn(c[2], cr2);
            const float s = __fadd_rn(__fadd_rn(__fmul_rn(c0, c0), __fmul_rn(c1, c1)), __fmul_rn(c2, c2));
            e = __fadd_rn(e, __fdiv_rn(-s, a.color_sigma2));
          }
          const float wgt = e != 0.f ? expf(e) : 1.f;
          if (MEDIAN) mine[n++] = make_float2(d, wgt);
          else dsum = __fadd_rn(dsum, __fmul_rn(d, wgt));
          wsum = __fadd_rn(wsum, wgt);
        }
      }
    }
    __syncthreads();   // every thread is done with slot i & 1
    if (threadIdx.x == 0 && i + 2 < nf) issue(i + 2);
  }
  if (!live) return;
  float result;
  if (MEDIAN) {
    for (int i = 1; i < n; ++i) {   // insertion sort: equal pairs are indistinguishable, so any stable order is std::sort's
      const float2 v = mine[i]; int j = i - 1;
      while (j >= 0 && pair_less(v, mine[j])) { mine[j + 1] = mine[j]; --j; }
      mine[j + 1] = v;
    }
    const float half = __fdiv_rn(wsum, 2.f);
    float cum = 0.f; result = 0.f;
    for (int i = 0; i < n; ++i) { cum = __fadd_rn(cum, mine[i].y); if (cum >= half) { result = mine[i].x; break; } }
  } else {
    result = wsum > 0.f ? __fdiv_rn(dsum, wsum) : 0.f;
  }
  a.out[((size_t)k * a.h + y) * a.w + x] = result;
  if (IN_PLACE) {   // what DepthFrame::depth() of this frame returns after setDepth: rcvd_depth_apply's arithmetic (k_dense<0>)
    float lx, ly; dense_loc(x, y, a.w, a.h, lx, ly);
    Gather g; gather_depth(a.cfg, lx, ly, g);
    a.depth[((size_t)(a.F + k) * a.Hp + y + r) * a.Wp + x + a.pad_l] = (float)depth_value(a.cfg, a.L, g, result, a.xparams + (size_t)k * a.L.nf);
  }
}

}  // namespace rcvd
