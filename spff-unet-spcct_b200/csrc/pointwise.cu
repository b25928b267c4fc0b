// CUDA-core kernels of the hot path that are not GEMM-shaped enough for the tensor pipe:
//   * the Cin = 1 stem convolution (enc1.pre.0 / enc1.b1.0, reference innovative3D/models.py:616-618
//     with in_channels = 1, models.py:1551) — 27 taps x 32 outputs per voxel: forward on the CUDA cores,
//     weight gradient as a warp-level mma.sync GEMM (the network input needs no gradient);
//   * the 1x1x1 classification head nn.Conv3d(32, num_classes, 1) (models.py:674) forward, arg-max
//     and backward, fused with the loss for training and, forward only, for evaluation;
//   * cross-entropy with ignore_index + the hard confusion tally that macro_dice_loss and
//     per_class_metrics_3d derive all their counts from (innovative3D/helpers.py:668-725, 782-803);
//   * the averaged softmax of ensembles and mirror test-time augmentation: the head's softmax added into
//     an fp32 probability accumulator, and one finishing pass to arg-max / probabilities / tallies, optionally
//     temperature-scaled; the statistics of the temperature fit on that accumulator;
//   * Adam (BaseLitModel.configure_optimizers, models.py:591-594).
// All are bandwidth-bound: one thread per voxel (or per 16-byte channel vector), coalesced
// accesses, weights broadcast from constant / shared memory. The exception is the temperature fit, which evaluates
// G x K exponentials per voxel and is compute-bound.
#include "common.h"
#include "ptx.cuh"

#include <cfloat>
#include <cmath>
#include <cuda_bf16.h>
#include <cuda_fp16.h>

namespace spff {
namespace {

constexpr int kMaxK = 16;     // classes
constexpr int kHeadC = 32;    // head input channels
constexpr int kStemCo = 32;   // stem output channels

__constant__ float c_head_w[kMaxK * kHeadC];
__constant__ float c_head_b[kMaxK];

__device__ __forceinline__ uint32_t smem_u32_local(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ uint32_t pack_bf16x2_local(float lo, float hi) {
  const __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<const uint32_t*>(&v);
}
__device__ __forceinline__ void unpack8(const uint4& v, float (&f)[8]) {
  const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&v);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    float2 t = __bfloat1622float2(h[i]);
    f[2 * i] = t.x;
    f[2 * i + 1] = t.y;
  }
}
__device__ __forceinline__ uint4 pack8(const float (&f)[8]) {
  uint4 v;
  __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&v);
#pragma unroll
  for (int i = 0; i < 4; ++i) h[i] = __floats2bfloat162_rn(f[2 * i], f[2 * i + 1]);
  return v;
}

// ---------------------------------------------------------------------------------------------
// stem: y[pos][co] = sum_tap x[pos+tap] * w[co][tap]     x fp32 [N,1,D,H,W], y bf16 position-major
// one thread = one voxel x 8 output channels
// ---------------------------------------------------------------------------------------------
// A thread owns a strip of kStrip consecutive w positions of one (n,d,h) row and 8 (forward) or 4
// (weight gradient) output channels: the 3 x (kStrip+2) input window of each (kd,kh) row is loaded
// once and reused by the 3 kw taps of every position of the strip, the tap weights once per strip.
constexpr int kStrip = 4;

__device__ __forceinline__ void stem_decode(long long i, int cg, int strips, const spff_shape& s, int& v, int& w0,
                                            int& hq, int& dq, long long& rowbase) {
  v = static_cast<int>(i % cg);
  const long long t = i / cg;
  const int st = static_cast<int>(t % strips);
  const long long row = t / strips;            // (n*d + dq)*h + hq
  hq = static_cast<int>(row % s.h);
  dq = static_cast<int>((row / s.h) % s.d);
  w0 = st * kStrip;
  rowbase = row * s.w;
}

// loads x[(dq+kd-1), (hq+kh-1), w0-1 .. w0+kStrip] (zero outside the volume)
__device__ __forceinline__ void stem_window(const float* __restrict__ x, long long rowbase, int w0, int hq, int dq, int kd,
                                            int kh, const spff_shape& s, float (&xw)[kStrip + 2]) {
  const int d2 = dq + kd - 1, h2 = hq + kh - 1;
  const bool rok = d2 >= 0 && d2 < s.d && h2 >= 0 && h2 < s.h;
  const float* xr = x + rowbase + (static_cast<long long>(kd - 1) * s.h + (kh - 1)) * s.w + w0 - 1;
#pragma unroll
  for (int j = 0; j < kStrip + 2; ++j) {
    const int w2 = w0 - 1 + j;
    xw[j] = (rok && w2 >= 0 && w2 < s.w) ? __ldg(xr + j) : 0.f;
  }
}

__global__ void __launch_bounds__(256)
stem_fwd_kernel(const float* __restrict__ x, const float* __restrict__ w, __nv_bfloat16* __restrict__ y, long long ldy,
                int cout, spff_shape s) {
  extern __shared__ float sw[];  // [27][cout]
  for (int i = threadIdx.x; i < 27 * cout; i += blockDim.x) sw[(i % 27) * cout + i / 27] = w[i];
  __syncthreads();
  const int c8 = cout / 8;
  const int strips = (s.w + kStrip - 1) / kStrip;
  const long long total = static_cast<long long>(s.n) * s.d * s.h * strips * c8;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    int v, w0, hq, dq;
    long long rowbase;
    stem_decode(i, c8, strips, s, v, w0, hq, dq, rowbase);
    float acc[kStrip][8];
#pragma unroll
    for (int j = 0; j < kStrip; ++j)
#pragma unroll
      for (int k = 0; k < 8; ++k) acc[j][k] = 0.f;
#pragma unroll
    for (int kd = 0; kd < 3; ++kd) {
#pragma unroll
      for (int kh = 0; kh < 3; ++kh) {
        float xw[kStrip + 2];
        stem_window(x, rowbase, w0, hq, dq, kd, kh, s, xw);
#pragma unroll
        for (int kw = 0; kw < 3; ++kw) {
          const float4* wr = reinterpret_cast<const float4*>(sw + ((kd * 3 + kh) * 3 + kw) * cout + v * 8);
          const float4 wa = wr[0], wb = wr[1];
          const float wv[8] = {wa.x, wa.y, wa.z, wa.w, wb.x, wb.y, wb.z, wb.w};
#pragma unroll
          for (int j = 0; j < kStrip; ++j)
#pragma unroll
            for (int k = 0; k < 8; ++k) acc[j][k] = fmaf(xw[j + kw], wv[k], acc[j][k]);
        }
      }
    }
#pragma unroll
    for (int j = 0; j < kStrip; ++j)
      if (w0 + j < s.w) *reinterpret_cast<uint4*>(y + (rowbase + w0 + j) * ldy + v * 8) = pack8(acc[j]);
  }
}

// The same convolution with the InstanceNorm / BatchNorm statistics of its output taken in the epilogue (fp32
// accumulators, before the bf16 rounding): grid = (slots, n), a block strides over the items of ONE sample and
// writes one partial row partial[n][slot][2][cout] = {sum, sum of squares} — the layout of the tensor-core conv's
// epilogue partials, reduced in a fixed order by spff_in_coeffs_from_partials / spff_bn_coeffs. Replaces the
// separate spff_in_stats pass over the stem output.
__global__ void __launch_bounds__(256, 2)   // <= 128 registers: two resident blocks (152 and one block without the cap)
stem_fwd_stats_kernel(const float* __restrict__ x, const float* __restrict__ w, __nv_bfloat16* __restrict__ y, long long ldy,
                      int cout, spff_shape s, float* __restrict__ partial) {
  extern __shared__ float sw[];  // [27][cout], then [8 warps][2][cout] for the block reduction
  for (int i = threadIdx.x; i < 27 * cout; i += blockDim.x) sw[(i % 27) * cout + i / 27] = w[i];
  __syncthreads();
  float* red = sw + 27 * cout;
  const int c8 = cout / 8;                       // a power of two <= 32 (checked by the host)
  const int strips = (s.w + kStrip - 1) / kStrip;
  const long long per_sample = static_cast<long long>(s.d) * s.h * strips * c8;
  const long long n0 = static_cast<long long>(blockIdx.y) * per_sample;
  float ssum[8], ssq[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) ssum[k] = ssq[k] = 0.f;
  // the stride is a multiple of c8: a thread keeps its channel vector v for all its items
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < per_sample;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    int v, w0, hq, dq;
    long long rowbase;
    stem_decode(n0 + i, c8, strips, s, v, w0, hq, dq, rowbase);
    float acc[kStrip][8];
#pragma unroll
    for (int j = 0; j < kStrip; ++j)
#pragma unroll
      for (int k = 0; k < 8; ++k) acc[j][k] = 0.f;
#pragma unroll
    for (int kd = 0; kd < 3; ++kd) {
#pragma unroll
      for (int kh = 0; kh < 3; ++kh) {
        float xw[kStrip + 2];
        stem_window(x, rowbase, w0, hq, dq, kd, kh, s, xw);
#pragma unroll
        for (int kw = 0; kw < 3; ++kw) {
          const float4* wr = reinterpret_cast<const float4*>(sw + ((kd * 3 + kh) * 3 + kw) * cout + v * 8);
          const float4 wa = wr[0], wb = wr[1];
          const float wv[8] = {wa.x, wa.y, wa.z, wa.w, wb.x, wb.y, wb.z, wb.w};
#pragma unroll
          for (int j = 0; j < kStrip; ++j)
#pragma unroll
            for (int k = 0; k < 8; ++k) acc[j][k] = fmaf(xw[j + kw], wv[k], acc[j][k]);
        }
      }
    }
#pragma unroll
    for (int j = 0; j < kStrip; ++j) {
      if (w0 + j < s.w) {
        *reinterpret_cast<uint4*>(y + (rowbase + w0 + j) * ldy + v * 8) = pack8(acc[j]);
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          ssum[k] += acc[j][k];
          ssq[k] = fmaf(acc[j][k], acc[j][k], ssq[k]);
        }
      }
    }
  }
  // lanes with the same v (lane % c8) fold by shuffles, the 8 warps meet in shared memory, fixed order
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int off = 16; off >= c8; off >>= 1) {
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      ssum[k] += __shfl_xor_sync(0xffffffffu, ssum[k], off);
      ssq[k] += __shfl_xor_sync(0xffffffffu, ssq[k], off);
    }
  }
  if (lane < c8) {
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      red[(warp * 2 + 0) * cout + lane * 8 + k] = ssum[k];
      red[(warp * 2 + 1) * cout + lane * 8 + k] = ssq[k];
    }
  }
  __syncthreads();
  for (int idx = threadIdx.x; idx < 2 * cout; idx += blockDim.x) {
    float t = 0.f;
    for (int wp = 0; wp < 8; ++wp) t += red[wp * 2 * cout + idx];
    partial[(static_cast<size_t>(blockIdx.y) * gridDim.x + blockIdx.x) * 2 * cout + idx] = t;
  }
}

// ---------------------------------------------------------------------------------------------
// Stem forward on the tensor cores (the default of spff_conv3d_stem_fwd_stats): the implicit GEMM
// M = positions, K = 27 taps (padded to 32), N = 32 channels with warp-level mma.sync m16n8k16. Both
// operands are split into a bf16 head and a bf16 remainder and the three significant products
// hi*hi + lo*hi + hi*lo are accumulated in fp32, so the sums carry ~2^-16 relative error (the fp32
// FMA kernel above: 2^-24; the bf16 rounding of the stored output: 2^-9). A warp owns one segment of
// <= 128 positions of an image row at a time: it stages the 9 x (128 + 2) input window once (hi and lo
// planes), gathers the im2col A fragments from it, and transposes each 16 x 32 output tile through
// shared memory so every lane stores 32 contiguous bytes. Statistics as in the kernel above.
// ---------------------------------------------------------------------------------------------
constexpr int kSfWarps = 8;
constexpr int kSfSeg = 128;                  // positions per segment
constexpr int kSfPitch = kSfSeg + 8;         // window elements per row; column c of the window sits at index c + 3, so that the
                                             // 128 core columns start 16-byte aligned
constexpr int kSfOutPitch = 40;              // bf16 per staged output row (32 + 8 pad: conflict-free)
constexpr int kSfSmemBytes = kSfWarps * 9 * kSfPitch * 4 + kSfWarps * 16 * kSfOutPitch * 2;

__device__ __forceinline__ void split_bf16(float v, __nv_bfloat16& hi, __nv_bfloat16& lo) {
  hi = __float2bfloat16(v);
  lo = __float2bfloat16(v - __bfloat162float(hi));
}
__device__ __forceinline__ uint32_t pack_u16(const __nv_bfloat16 a, const __nv_bfloat16 b) {
  return static_cast<uint32_t>(__bfloat16_as_ushort(a)) | (static_cast<uint32_t>(__bfloat16_as_ushort(b)) << 16);
}
// one window element: bf16 head in the low half, bf16 remainder in the high half
__device__ __forceinline__ uint32_t split_packed(float v) {
  __nv_bfloat16 hi, lo;
  split_bf16(v, hi, lo);
  return pack_u16(hi, lo);
}
__device__ __forceinline__ void mma_bf16_16816(float (&c)[4], const uint32_t (&a)[4], const uint32_t (&b)[2]) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}

__global__ void __launch_bounds__(kSfWarps * 32, 2)
stem_fwd_stats_mma_kernel(const float* __restrict__ x, const float* __restrict__ w, __nv_bfloat16* __restrict__ y,
                          long long ldy, spff_shape s, float* __restrict__ partial) {
  extern __shared__ __align__(16) unsigned char sf_smem[];
  uint32_t* xs_all = reinterpret_cast<uint32_t*>(sf_smem);                     // [warp][9][kSfPitch] (hi | lo << 16)
  __nv_bfloat16* os_all = reinterpret_cast<__nv_bfloat16*>(xs_all + kSfWarps * 9 * kSfPitch);   // [warp][16][kSfOutPitch]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int g = lane >> 2, t = lane & 3;
  uint32_t* xw = xs_all + warp * 9 * kSfPitch;
  __nv_bfloat16* os = os_all + warp * 16 * kSfOutPitch;
  // B fragments (K = tap, N = channel), constant for the whole launch; taps >= 27 carry zero weights, so the A
  // values gathered for them do not matter
  uint32_t bh[2][4][2], bl[2][4][2];
  int toff[2][2][2];
#pragma unroll
  for (int ks = 0; ks < 2; ++ks)
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const int k0 = 16 * ks + 2 * t + 8 * j;
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int k = k0 + e;
        toff[ks][j][e] = k < 27 ? (k / 3) * kSfPitch + k % 3 + 3 : 3;
      }
#pragma unroll
      for (int nt = 0; nt < 4; ++nt) {
        const int n = 8 * nt + g;
        const float w0 = k0 < 27 ? __ldg(w + n * 27 + k0) : 0.f;
        const float w1 = k0 + 1 < 27 ? __ldg(w + n * 27 + k0 + 1) : 0.f;
        __nv_bfloat16 h0, l0, h1, l1;
        split_bf16(w0, h0, l0);
        split_bf16(w1, h1, l1);
        bh[ks][nt][j] = pack_u16(h0, h1);
        bl[ks][nt][j] = pack_u16(l0, l1);
      }
    }
  float ssum[4][2], ssq[4][2];
#pragma unroll
  for (int nt = 0; nt < 4; ++nt) ssum[nt][0] = ssum[nt][1] = ssq[nt][0] = ssq[nt][1] = 0.f;
  const bool wide = ((ldy & 15) == 0) && ((reinterpret_cast<uintptr_t>(y) & 31) == 0);
  const bool xvec = (s.w % 4 == 0) && ((reinterpret_cast<uintptr_t>(x) & 15) == 0);   // 16-byte loads of the window rows
  const int segs = (s.w + kSfSeg - 1) / kSfSeg;
  const int nwork = s.d * s.h * segs;                         // of this sample
  const long long row0 = static_cast<long long>(blockIdx.y) * s.d * s.h;
  for (int work = blockIdx.x * kSfWarps + warp; work < nwork; work += gridDim.x * kSfWarps) {
    const int sg = work % segs;
    const int rw = work / segs;                               // dd*h + hh
    const int hh = rw % s.h, dd = rw / s.h;
    const long long row = row0 + rw;
    const int w0 = sg * kSfSeg;
    const int wn = min(kSfSeg, s.w - w0);
    const int wpad = (wn + 15) & ~15;
    // input window, split: xw[kd*3+kh][c + 3] = x[dd+kd-1][hh+kh-1][w0 + c - 1]
#pragma unroll
    for (int r = 0; r < 9; ++r) {
      const int d2 = dd + r / 3 - 1, h2 = hh + r % 3 - 1;
      const bool rok = d2 >= 0 && d2 < s.d && h2 >= 0 && h2 < s.h;
      const float* xr = x + (row + static_cast<long long>(r / 3 - 1) * s.h + (r % 3 - 1)) * s.w + w0;   // column 1 of the window
      uint32_t* dst = xw + r * kSfPitch;
      if (xvec) {
        // every lane: 4 core columns (one 16-byte load, one 16-byte store); lanes 0 / 1: the left / right halo column
        const int c4 = 4 * lane;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (rok && w0 + c4 < s.w) v = __ldg(reinterpret_cast<const float4*>(xr + c4));
        *reinterpret_cast<uint4*>(dst + 4 + c4) = make_uint4(split_packed(v.x), split_packed(v.y), split_packed(v.z), split_packed(v.w));
        if (lane < 2) {
          const int w2 = lane == 0 ? w0 - 1 : w0 + kSfSeg;
          const float hv = (rok && w2 >= 0 && w2 < s.w) ? __ldg(xr + (w2 - w0)) : 0.f;
          dst[lane == 0 ? 3 : 4 + kSfSeg] = split_packed(hv);
        }
      } else {
        for (int c = lane; c < wpad + 2; c += 32) {
          const int w2 = w0 + c - 1;
          const float v = (rok && w2 >= 0 && w2 < s.w) ? __ldg(xr + c - 1) : 0.f;
          dst[c + 3] = split_packed(v);
        }
      }
    }
    __syncwarp();
    __nv_bfloat16* yrow = y + (row * s.w + w0) * ldy;
    for (int mt = 0; mt < wpad / 16; ++mt) {
      const int p = mt * 16 + g;
      uint32_t ah[2][4], al[2][4];
#pragma unroll
      for (int ks = 0; ks < 2; ++ks)
#pragma unroll
        for (int j = 0; j < 2; ++j)
#pragma unroll
          for (int rh = 0; rh < 2; ++rh) {
            const uint32_t u0 = xw[toff[ks][j][0] + p + 8 * rh], u1 = xw[toff[ks][j][1] + p + 8 * rh];
            ah[ks][2 * j + rh] = __byte_perm(u0, u1, 0x5410);     // the two heads
            al[ks][2 * j + rh] = __byte_perm(u0, u1, 0x7632);     // the two remainders
          }
      float acc[4][4];
#pragma unroll
      for (int nt = 0; nt < 4; ++nt) {
        acc[nt][0] = acc[nt][1] = acc[nt][2] = acc[nt][3] = 0.f;
#pragma unroll
        for (int ks = 0; ks < 2; ++ks) {   // smallest products first
          mma_bf16_16816(acc[nt], al[ks], bh[ks][nt]);
          mma_bf16_16816(acc[nt], ah[ks], bl[ks][nt]);
        }
#pragma unroll
        for (int ks = 0; ks < 2; ++ks) mma_bf16_16816(acc[nt], ah[ks], bh[ks][nt]);
      }
      const bool ok0 = p < wn, ok1 = p + 8 < wn;
#pragma unroll
      for (int nt = 0; nt < 4; ++nt) {
        if (ok0) {
          ssum[nt][0] += acc[nt][0];
          ssum[nt][1] += acc[nt][1];
          ssq[nt][0] = fmaf(acc[nt][0], acc[nt][0], ssq[nt][0]);
          ssq[nt][1] = fmaf(acc[nt][1], acc[nt][1], ssq[nt][1]);
        }
        if (ok1) {
          ssum[nt][0] += acc[nt][2];
          ssum[nt][1] += acc[nt][3];
          ssq[nt][0] = fmaf(acc[nt][2], acc[nt][2], ssq[nt][0]);
          ssq[nt][1] = fmaf(acc[nt][3], acc[nt][3], ssq[nt][1]);
        }
        *reinterpret_cast<uint32_t*>(&os[g * kSfOutPitch + 8 * nt + 2 * t]) = pack_bf16x2_local(acc[nt][0], acc[nt][1]);
        *reinterpret_cast<uint32_t*>(&os[(g + 8) * kSfOutPitch + 8 * nt + 2 * t]) = pack_bf16x2_local(acc[nt][2], acc[nt][3]);
      }
      __syncwarp();
      {
        const int pr = lane >> 1, half = lane & 1;
        if (mt * 16 + pr < wn) {
          const uint4* src = reinterpret_cast<const uint4*>(&os[pr * kSfOutPitch + half * 16]);
          const uint4 v0 = src[0], v1 = src[1];
          __nv_bfloat16* dst = yrow + static_cast<long long>(mt * 16 + pr) * ldy + half * 16;
          if (wide) {
            st_global_v8(dst, v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w);
          } else {
            *reinterpret_cast<uint4*>(dst) = v0;
            *reinterpret_cast<uint4*>(dst + 8) = v1;
          }
        }
      }
      __syncwarp();
    }
  }
  // lanes with the same t hold the same channels: fold over g by shuffles, then the 8 warps in shared memory
#pragma unroll
  for (int off = 4; off <= 16; off <<= 1)
#pragma unroll
    for (int nt = 0; nt < 4; ++nt)
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        ssum[nt][e] += __shfl_xor_sync(0xffffffffu, ssum[nt][e], off);
        ssq[nt][e] += __shfl_xor_sync(0xffffffffu, ssq[nt][e], off);
      }
  __syncthreads();                                            // every warp is done with its staging tiles
  float* red = reinterpret_cast<float*>(os_all);              // [warp][2][32]
  if (g == 0) {
#pragma unroll
    for (int nt = 0; nt < 4; ++nt)
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        red[(warp * 2 + 0) * kStemCo + 8 * nt + 2 * t + e] = ssum[nt][e];
        red[(warp * 2 + 1) * kStemCo + 8 * nt + 2 * t + e] = ssq[nt][e];
      }
  }
  __syncthreads();
  for (int idx = threadIdx.x; idx < 2 * kStemCo; idx += blockDim.x) {
    float tot = 0.f;
    for (int wp = 0; wp < kSfWarps; ++wp) tot += red[wp * 2 * kStemCo + idx];
    partial[(static_cast<size_t>(blockIdx.y) * gridDim.x + blockIdx.x) * 2 * kStemCo + idx] = tot;
  }
}

// ---------------------------------------------------------------------------------------------
// Stem weight gradient on the tensor cores. dw[tap][co] = sum_pos x[pos + off(tap)] * dy[pos][co] is a
// GEMM with M = 27 taps (padded to 32), N = 32 output channels, K = positions. The operands are far
// too small for a tcgen05 tile pipeline (one 32 x 32 accumulator), so this uses warp-level
// mma.sync m16n8k16 (bf16 in, fp32 accumulate): a warp owns one segment of <= 128 positions of an
// image row at a time, stages the 9 x (128 + 2) input window (fp32 -> bf16) and 16-position dy tiles
// in shared memory, builds the im2col A fragments straight from the window (tap = row/column offset)
// and keeps the 32 x 32 accumulator in registers across all its segments.
// x enters the product rounded to bf16 (the forward stem reads it in fp32): a 2^-9 relative,
// zero-mean perturbation per element of a sum over ~10^8 positions.
// ---------------------------------------------------------------------------------------------
constexpr int kSwgWarps = 8;
constexpr int kSwgSeg = 128;                 // positions per segment
constexpr int kSwgWin = kSwgSeg + 8;         // window row: column c at index c + 3 (the 128 core columns start 8-byte aligned), +2 halo,
                                             // + slack so that the 32-bit pair loads stay inside
constexpr int kSwgDyPitch = 40;              // bf16 per staged dy row (32 + 8 pad: conflict-free ldmatrix)
constexpr int kSwgBlocksPerSm = 2;

__global__ void __launch_bounds__(kSwgWarps * 32, kSwgBlocksPerSm)
stem_wgrad_mma_kernel(const float* __restrict__ x, const __nv_bfloat16* __restrict__ dy, long long lddy, spff_shape s,
                      float* __restrict__ partial /* [block][27][32] */) {
  __shared__ __align__(16) __nv_bfloat16 xs[kSwgWarps][9][kSwgWin];
  __shared__ __align__(16) __nv_bfloat16 dys[kSwgWarps][16][kSwgDyPitch];
  __shared__ float red[32 * 33];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int g = lane >> 2, t = lane & 3;
  float acc[2][4][4];
#pragma unroll
  for (int a = 0; a < 2; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b)
#pragma unroll
      for (int c = 0; c < 4; ++c) acc[a][b][c] = 0.f;
  // the four im2col rows (taps) this thread feeds: g, g+8, g+16, g+24 -> element offset inside the window
  int toff[4];
  bool tok[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int tap = g + 8 * i;
    tok[i] = tap < 27;
    const int kd = tap / 9, kh = (tap / 3) % 3, kw = tap % 3;
    toff[i] = tok[i] ? (kd * 3 + kh) * kSwgWin + kw + 3 : 0;
  }
  const int segs = (s.w + kSwgSeg - 1) / kSwgSeg;
  const long long nwork = static_cast<long long>(s.n) * s.d * s.h * segs;
  const bool xvec = (s.w % 4 == 0) && ((reinterpret_cast<uintptr_t>(x) & 15) == 0);   // 16-byte loads of the window rows
  const __nv_bfloat16* xw = &xs[warp][0][0];
  const uint32_t* xw32 = reinterpret_cast<const uint32_t*>(xw);
  for (long long work = static_cast<long long>(blockIdx.x) * kSwgWarps + warp; work < nwork;
       work += static_cast<long long>(gridDim.x) * kSwgWarps) {
    const int sg = static_cast<int>(work % segs);
    const long long row = work / segs;                       // (n*d + dd)*h + hh
    const int hh = static_cast<int>(row % s.h);
    const int dd = static_cast<int>((row / s.h) % s.d);
    const int w0 = sg * kSwgSeg;
    const int wn = min(kSwgSeg, s.w - w0);                    // valid positions of this segment
    const int wpad = (wn + 15) & ~15;
    // input window: xs[kd*3+kh][c + 3] = x[dd+kd-1][hh+kh-1][w0 + c - 1]
#pragma unroll
    for (int r = 0; r < 9; ++r) {
      const int d2 = dd + r / 3 - 1, h2 = hh + r % 3 - 1;
      const bool rok = d2 >= 0 && d2 < s.d && h2 >= 0 && h2 < s.h;
      const float* xr = x + (row + static_cast<long long>(r / 3 - 1) * s.h + (r % 3 - 1)) * s.w + w0;   // window column 1
      __nv_bfloat16* dst = &xs[warp][r][0];
      if (xvec) {
        // every lane: 4 core columns (one 16-byte load, one 8-byte store); lanes 0 / 1: the left / right halo column
        const int c4 = 4 * lane;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (rok && w0 + c4 < s.w) v = __ldg(reinterpret_cast<const float4*>(xr + c4));
        *reinterpret_cast<uint2*>(dst + 4 + c4) = make_uint2(pack_bf16x2_local(v.x, v.y), pack_bf16x2_local(v.z, v.w));
        if (lane < 2) {
          const int w2 = lane == 0 ? w0 - 1 : w0 + kSwgSeg;
          const float hv = (rok && w2 >= 0 && w2 < s.w) ? __ldg(xr + (w2 - w0)) : 0.f;
          dst[lane == 0 ? 3 : 4 + kSwgSeg] = __float2bfloat16(hv);
        }
      } else {
        for (int c = lane; c < wpad + 2; c += 32) {
          const int w2 = w0 + c - 1;
          const float v = (rok && w2 >= 0 && w2 < s.w) ? __ldg(xr + c - 1) : 0.f;
          dst[c + 3] = __float2bfloat16(v);
        }
      }
    }
    __syncwarp();
    const __nv_bfloat16* dyrow = dy + (row * s.w + w0) * lddy;
    for (int ks = 0; ks < wpad / 16; ++ks) {
      {  // stage 16 positions x 32 channels of dy (zeros past the row end)
        const int pos = lane >> 1, half = lane & 1;
        uint4 v0 = make_uint4(0, 0, 0, 0), v1 = v0;
        if (ks * 16 + pos < wn) {
          const uint4* src = reinterpret_cast<const uint4*>(dyrow + static_cast<long long>(ks * 16 + pos) * lddy + half * 16);
          v0 = __ldg(src);
          v1 = __ldg(src + 1);
        }
        uint4* dst = reinterpret_cast<uint4*>(&dys[warp][pos][half * 16]);
        dst[0] = v0;
        dst[1] = v1;
      }
      __syncwarp();
      uint32_t bfr[4][2];
#pragma unroll
      for (int h2 = 0; h2 < 2; ++h2) {  // one ldmatrix.x4.trans = B fragments of two 8-channel tiles
        const int mi = lane >> 3, r = lane & 7;
        const uint32_t addr = smem_u32_local(&dys[warp][r + 8 * (mi & 1)][8 * (2 * h2 + (mi >> 1))]);
        asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
                     : "=r"(bfr[2 * h2][0]), "=r"(bfr[2 * h2][1]), "=r"(bfr[2 * h2 + 1][0]), "=r"(bfr[2 * h2 + 1][1])
                     : "r"(addr));
      }
      uint32_t afr[2][4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {       // row g + 8*i: m-tile i/2, fragment registers (i%2) and (i%2)+2
#pragma unroll
        for (int kh2 = 0; kh2 < 2; ++kh2) {
          const int e = toff[i] + ks * 16 + 2 * t + 8 * kh2;   // element index of the pair (e, e+1)
          const uint32_t lo = xw32[e >> 1], hi = xw32[(e >> 1) + 1];
          const uint32_t v = __funnelshift_r(lo, hi, (e & 1) * 16);
          afr[i >> 1][(i & 1) + 2 * kh2] = tok[i] ? v : 0u;
        }
      }
#pragma unroll
      for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int nt = 0; nt < 4; ++nt)
          asm volatile(
              "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
              : "+f"(acc[mt][nt][0]), "+f"(acc[mt][nt][1]), "+f"(acc[mt][nt][2]), "+f"(acc[mt][nt][3])
              : "r"(afr[mt][0]), "r"(afr[mt][1]), "r"(afr[mt][2]), "r"(afr[mt][3]), "r"(bfr[nt][0]), "r"(bfr[nt][1]));
      __syncwarp();
    }
  }
  // block reduction of the eight 32 x 32 accumulators (row = tap, column = channel): the warps add
  // their fragments one after the other, so the summation order is fixed (bit-reproducible)
  for (int i = threadIdx.x; i < 32 * 33; i += blockDim.x) red[i] = 0.f;
  __syncthreads();
  for (int wv = 0; wv < kSwgWarps; ++wv) {
    if (warp == wv) {
#pragma unroll
      for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int nt = 0; nt < 4; ++nt) {
          const int r0 = 16 * mt + g, c0 = 8 * nt + 2 * t;
          red[r0 * 33 + c0] += acc[mt][nt][0];
          red[r0 * 33 + c0 + 1] += acc[mt][nt][1];
          red[(r0 + 8) * 33 + c0] += acc[mt][nt][2];
          red[(r0 + 8) * 33 + c0 + 1] += acc[mt][nt][3];
        }
    }
    __syncthreads();
  }
  for (int i = threadIdx.x; i < 27 * 32; i += blockDim.x)
    partial[static_cast<size_t>(blockIdx.x) * 27 * 32 + i] = red[(i / 32) * 33 + (i % 32)];
}

// dw[co][tap] = beta*dw + sum_blocks partial[block][tap][co]
__global__ void stem_wgrad_reduce_kernel(const float* __restrict__ partial, int blocks, int cout, float beta,
                                         float* __restrict__ dw) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;  // index into [tap][co]
  if (i >= 27 * cout) return;
  float v = 0.f;
  for (int b = 0; b < blocks; ++b) v += partial[static_cast<size_t>(b) * 27 * cout + i];
  const int t = i / cout, co = i % cout;
  float* dst = dw + co * 27 + t;
  *dst = (beta == 0.f) ? v : fmaf(beta, *dst, v);
}

// ---------------------------------------------------------------------------------------------
// head: logits[n][k][d][hw] = b[k] + sum_c x[pos][c] * w[k][c]   (weights in constant memory)
// ---------------------------------------------------------------------------------------------
template <bool ARGMAX>
__global__ void __launch_bounds__(256)
head_fwd_kernel(const __nv_bfloat16* __restrict__ x, long long ldx, float* __restrict__ logits,
                uint8_t* __restrict__ labels, int K, long long dhw, long long total) {
  for (long long pos = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; pos < total;
       pos += static_cast<long long>(gridDim.x) * blockDim.x) {
    float xv[kHeadC];
#pragma unroll
    for (int v = 0; v < kHeadC / 8; ++v) {
      float f[8];
      unpack8(__ldg(reinterpret_cast<const uint4*>(x + pos * ldx) + v), f);
#pragma unroll
      for (int i = 0; i < 8; ++i) xv[v * 8 + i] = f[i];
    }
    const long long n = pos / dhw, r = pos % dhw;
    float best = -INFINITY;
    int arg = 0;
#pragma unroll
    for (int k = 0; k < kMaxK; ++k) {
      if (k < K) {
        float a = c_head_b[k];
#pragma unroll
        for (int c = 0; c < kHeadC; ++c) a = fmaf(xv[c], c_head_w[k * kHeadC + c], a);
        if (ARGMAX) {
          if (a > best) {
            best = a;
            arg = k;
          }
        } else {
          logits[(n * K + k) * dhw + r] = a;
        }
      }
    }
    if (ARGMAX) labels[pos] = static_cast<uint8_t>(arg);
  }
}

// head backward: one thread = one voxel x 8 channels.
//   dx[pos][c] = sum_k dl[k][pos] * w[k][c];  partial dW[k][c], db[k] per block -> workspace
__global__ void __launch_bounds__(256)
head_bwd_kernel(const float* __restrict__ dlogits, const __nv_bfloat16* __restrict__ x, long long ldx,
                __nv_bfloat16* __restrict__ dx, long long lddx, int K, long long dhw, long long total,
                float* __restrict__ partial /* [block][K*32 + K] */) {
  extern __shared__ float red[];  // [warps][kMaxK*8*4 + kMaxK]
  constexpr int V = kHeadC / 8;   // 4 threads per voxel
  float accw[kMaxK][8];
  float accb[kMaxK];
#pragma unroll
  for (int k = 0; k < kMaxK; ++k) {
    accb[k] = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) accw[k][i] = 0.f;
  }
  const int v = threadIdx.x % V;
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < total * V;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long pos = i / V;
    const long long n = pos / dhw, r = pos % dhw;
    float f[8], o[8];
    unpack8(__ldg(reinterpret_cast<const uint4*>(x + pos * ldx) + v), f);
#pragma unroll
    for (int c = 0; c < 8; ++c) o[c] = 0.f;
#pragma unroll
    for (int k = 0; k < kMaxK; ++k) {
      if (k < K) {
        const float g = __ldg(dlogits + (n * K + k) * dhw + r);
        accb[k] += g;
#pragma unroll
        for (int c = 0; c < 8; ++c) {
          accw[k][c] = fmaf(g, f[c], accw[k][c]);
          o[c] = fmaf(g, c_head_w[k * kHeadC + v * 8 + c], o[c]);
        }
      }
    }
    if (dx) *reinterpret_cast<uint4*>(dx + pos * lddx + v * 8) = pack8(o);
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
  const int stride = kMaxK * kHeadC + kMaxK;
#pragma unroll
  for (int k = 0; k < kMaxK; ++k) {
    if (k < K) {
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        float t = accw[k][c];
        for (int off = 16; off >= V; off >>= 1) t += __shfl_xor_sync(0xffffffffu, t, off);
        if (lane < V) red[warp * stride + k * kHeadC + lane * 8 + c] = t;
      }
      float t = (v == 0) ? accb[k] : 0.f;
      for (int off = 16; off > 0; off >>= 1) t += __shfl_xor_sync(0xffffffffu, t, off);
      if (lane == 0) red[warp * stride + kMaxK * kHeadC + k] = t;
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < K * kHeadC + K; i += blockDim.x) {
    const int src = i < K * kHeadC ? i : kMaxK * kHeadC + (i - K * kHeadC);
    float t = 0.f;
    for (int wv = 0; wv < nwarps; ++wv) t += red[wv * stride + src];
    partial[static_cast<size_t>(blockIdx.x) * (K * kHeadC + K) + i] = t;
  }
}

__global__ void head_bwd_reduce_kernel(const float* __restrict__ partial, int blocks, int K, float beta,
                                       float* __restrict__ dw, float* __restrict__ db) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int tot = K * kHeadC + K;
  if (i >= tot) return;
  float t = 0.f;
  for (int b = 0; b < blocks; ++b) t += partial[static_cast<size_t>(b) * tot + i];
  float* dst = i < K * kHeadC ? dw + i : db + (i - K * kHeadC);
  *dst = (beta == 0.f) ? t : fmaf(beta, *dst, t);
}

// ---------------------------------------------------------------------------------------------
// cross entropy + confusion tally over fp32 logits [N,K,D,H,W]
// ---------------------------------------------------------------------------------------------
template <typename LabelT>
__device__ __forceinline__ int load_label(const void* labels, long long i) {
  return static_cast<int>(static_cast<const LabelT*>(labels)[i]);
}

template <typename LabelT, bool GRAD>
__global__ void __launch_bounds__(256)
ce_kernel(const float* __restrict__ logits, const void* __restrict__ labels, int ignore_index, int K, long long dhw,
          long long total, double* __restrict__ acc, unsigned long long* __restrict__ counts,
          unsigned long long* __restrict__ confusion, const unsigned long long* __restrict__ n_valid,
          const float* __restrict__ gscale, float* __restrict__ dlogits) {
  __shared__ unsigned int s_conf[kMaxK * kMaxK];
  __shared__ float s_nll[8];
  __shared__ unsigned int s_cnt[8];
  if (!GRAD) {
    for (int i = threadIdx.x; i < K * K; i += blockDim.x) s_conf[i] = 0;
    __syncthreads();
  }
  float scale = 0.f;
  if (GRAD) {
    const unsigned long long nv = n_valid[0];
    scale = (nv > 0 ? 1.f / static_cast<float>(nv) : 0.f) * (gscale ? gscale[0] : 1.f);
  }
  float nll_sum = 0.f;
  unsigned int cnt = 0;
  for (long long pos = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; pos < total;
       pos += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long n = pos / dhw, r = pos % dhw;
    const int lab = load_label<LabelT>(labels, pos);
    const bool valid = lab != ignore_index;
    float l[kMaxK];
    float mx = -INFINITY;
    int arg = 0;
#pragma unroll
    for (int k = 0; k < kMaxK; ++k) {
      if (k < K) {
        l[k] = __ldg(logits + (n * K + k) * dhw + r);
        if (l[k] > mx) {
          mx = l[k];
          arg = k;
        }
      }
    }
    float se = 0.f;
#pragma unroll
    for (int k = 0; k < kMaxK; ++k)
      if (k < K) se += __expf(l[k] - mx);
    if (GRAD) {
      const float inv = 1.f / se;
#pragma unroll
      for (int k = 0; k < kMaxK; ++k)
        if (k < K) {
          float g = 0.f;
          if (valid) g = (__expf(l[k] - mx) * inv - (k == lab ? 1.f : 0.f)) * scale;
          dlogits[(n * K + k) * dhw + r] = g;
        }
    } else if (valid) {
      float ll = 0.f;
#pragma unroll
      for (int k = 0; k < kMaxK; ++k)
        if (k < K && k == lab) ll = l[k];
      nll_sum += (mx + __logf(se)) - ll;
      ++cnt;
      if (lab >= 0 && lab < K) atomicAdd(&s_conf[lab * K + arg], 1u);
    }
  }
  if (!GRAD) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int o = 16; o > 0; o >>= 1) {
      nll_sum += __shfl_xor_sync(0xffffffffu, nll_sum, o);
      cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    }
    if (lane == 0) {
      s_nll[warp] = nll_sum;
      s_cnt[warp] = cnt;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
      double t = 0;
      unsigned long long c = 0;
      for (int wv = 0; wv < (blockDim.x >> 5); ++wv) {
        t += s_nll[wv];
        c += s_cnt[wv];
      }
      atomicAdd(acc, t);
      atomicAdd(counts, c);
    }
    for (int i = threadIdx.x; i < K * K; i += blockDim.x)
      if (s_conf[i]) atomicAdd(confusion + i, static_cast<unsigned long long>(s_conf[i]));
  }
}

// ---------------------------------------------------------------------------------------------
// Fused training head: 1x1x1 conv (models.py:674) + cross entropy / confusion tally
// (helpers.py:782-803, 668-725) + their backward, in ONE pass over the last activation.
//   logits[k] = b[k] + x . w[k]            (registers only - the [N,K,D,H,W] logits are never stored)
//   acc += nll, counts += valid, confusion[label][argmax] += 1
//   dl[k] = (softmax[k] - [k == label]) * gscale / n_valid   (0 on ignored voxels)
//   dx = dl . w  (bf16),   partial dW[k][c] = sum dl[k] x[c],   partial db[k] = sum dl[k]
// One thread = one voxel for the per-voxel math (weights broadcast from constant memory); the
// outer product for dW is transposed through shared memory so that lane c owns column c of dW
// (13 accumulators) and sweeps the 32 voxels of its warp: 1 bf16 + 4 broadcast float4 loads per
// 13 FMAs. Traffic: 64 B read + 64 B written per voxel (+ label), against 52 B/voxel of fp32 logits
// written and read three times by the unfused sequence.
// ---------------------------------------------------------------------------------------------
constexpr int kHeadLossWarps = 8;
constexpr int kHeadLossBlocksPerSm = 2;

template <typename LabelT>
__global__ void __launch_bounds__(kHeadLossWarps * 32, kHeadLossBlocksPerSm)
head_loss_kernel(const __nv_bfloat16* __restrict__ x, long long ldx, const void* __restrict__ labels, int ignore_index,
                 int K, long long total, const unsigned long long* __restrict__ n_valid,
                 const float* __restrict__ gscale, double* __restrict__ acc, unsigned long long* __restrict__ counts,
                 unsigned long long* __restrict__ confusion, __nv_bfloat16* __restrict__ dx, long long lddx,
                 float* __restrict__ partial /* [block][K*32 + K] */) {
  // 32 KB: per-warp transpose tiles; re-used as the block-reduction scratch once the loop is done
  __shared__ __align__(16) unsigned char sraw[kHeadLossWarps * 32 * (kHeadC * 2 + kMaxK * 4)];
  auto sx = reinterpret_cast<__nv_bfloat16(*)[32][kHeadC]>(sraw);                                   // 16 KB
  auto sdl = reinterpret_cast<float(*)[32][kMaxK]>(sraw + kHeadLossWarps * 32 * kHeadC * 2);       // 16 KB
  auto sred = reinterpret_cast<float(*)[kMaxK * kHeadC + kMaxK]>(sraw);                             // 16.5 KB
  static_assert(sizeof(float) * kHeadLossWarps * (kMaxK * kHeadC + kMaxK) <= sizeof(sraw), "reduction scratch");
  __shared__ unsigned int s_conf[kMaxK * kMaxK];
  __shared__ float s_nll[kHeadLossWarps];
  __shared__ unsigned int s_cnt[kHeadLossWarps];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int i = threadIdx.x; i < K * K; i += blockDim.x) s_conf[i] = 0;
  __syncthreads();
  const unsigned long long nv = n_valid[0];
  const float scale = (nv > 0 ? 1.f / static_cast<float>(nv) : 0.f) * (gscale ? gscale[0] : 1.f);
  float dw[kMaxK], db[kMaxK];
#pragma unroll
  for (int k = 0; k < kMaxK; ++k) dw[k] = db[k] = 0.f;
  float nll_sum = 0.f;
  unsigned int cnt = 0;
  const long long ntiles = (total + 31) / 32;
  for (long long tile = static_cast<long long>(blockIdx.x) * kHeadLossWarps + warp; tile < ntiles;
       tile += static_cast<long long>(gridDim.x) * kHeadLossWarps) {
    const long long pos = tile * 32 + lane;
    const bool inb = pos < total;
    uint4 raw[kHeadC / 8];
    float xv[kHeadC];
#pragma unroll
    for (int v = 0; v < kHeadC / 8; ++v) {
      raw[v] = inb ? __ldg(reinterpret_cast<const uint4*>(x + pos * ldx) + v) : make_uint4(0, 0, 0, 0);
      float f[8];
      unpack8(raw[v], f);
#pragma unroll
      for (int i = 0; i < 8; ++i) xv[v * 8 + i] = f[i];
    }
    const int lab = inb ? static_cast<int>(static_cast<const LabelT*>(labels)[pos]) : ignore_index;
    const bool valid = inb && lab != ignore_index;
    float l[kMaxK];
    float mx = -INFINITY;
    int arg = 0;
#pragma unroll
    for (int k = 0; k < kMaxK; ++k) {
      if (k < K) {
        float a = c_head_b[k];
#pragma unroll
        for (int c = 0; c < kHeadC; ++c) a = fmaf(xv[c], c_head_w[k * kHeadC + c], a);
        l[k] = a;
        if (a > mx) {
          mx = a;
          arg = k;
        }
      }
    }
    float se = 0.f;
#pragma unroll
    for (int k = 0; k < kMaxK; ++k)
      if (k < K) {
        l[k] = __expf(l[k] - mx);   // l[] now holds exp(logit - max); the label's logit is recovered below
        se += l[k];
      }
    const float inv = 1.f / se;
    if (valid) {
      float el = 1.f;
#pragma unroll
      for (int k = 0; k < kMaxK; ++k)
        if (k < K && k == lab) el = l[k];
      nll_sum += __logf(se) - __logf(el);
      ++cnt;
      if (lab >= 0 && lab < K) atomicAdd(&s_conf[lab * K + arg], 1u);
    }
    float o[kHeadC];
#pragma unroll
    for (int c = 0; c < kHeadC; ++c) o[c] = 0.f;
#pragma unroll
    for (int k = 0; k < kMaxK; ++k) {
      float g = 0.f;
      if (k < K && valid) g = (l[k] * inv - (k == lab ? 1.f : 0.f)) * scale;
      l[k] = g;   // l[] now holds d(logits)
      if (k < K) {
        db[k] += g;
#pragma unroll
        for (int c = 0; c < kHeadC; ++c) o[c] = fmaf(g, c_head_w[k * kHeadC + c], o[c]);
      }
    }
    if (inb && dx) {
#pragma unroll
      for (int v = 0; v < kHeadC / 8; ++v) {
        float f[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) f[i] = o[v * 8 + i];
        *reinterpret_cast<uint4*>(dx + pos * lddx + v * 8) = pack8(f);
      }
    }
    // transpose through shared memory: lane c accumulates dW[:, c] over the warp's 32 voxels
#pragma unroll
    for (int v = 0; v < kHeadC / 8; ++v) *reinterpret_cast<uint4*>(&sx[warp][lane][v * 8]) = raw[v];
#pragma unroll
    for (int v = 0; v < kMaxK / 4; ++v)
      *reinterpret_cast<float4*>(&sdl[warp][lane][v * 4]) = make_float4(l[v * 4], l[v * 4 + 1], l[v * 4 + 2], l[v * 4 + 3]);
    __syncwarp();
#pragma unroll 4
    for (int j = 0; j < 32; ++j) {
      const float xs = __bfloat162float(sx[warp][j][lane]);
      float d[kMaxK];
#pragma unroll
      for (int v = 0; v < kMaxK / 4; ++v) {
        const float4 t = *reinterpret_cast<const float4*>(&sdl[warp][j][v * 4]);
        d[v * 4] = t.x;
        d[v * 4 + 1] = t.y;
        d[v * 4 + 2] = t.z;
        d[v * 4 + 3] = t.w;
      }
#pragma unroll
      for (int k = 0; k < kMaxK; ++k)
        if (k < K) dw[k] = fmaf(d[k], xs, dw[k]);
    }
    __syncwarp();
  }
  // block reduction: dW columns are already per lane; db and the loss statistics need a warp sum
  __syncthreads();   // every warp is done with its transpose tiles
#pragma unroll
  for (int k = 0; k < kMaxK; ++k) {
    if (k < K) {
      sred[warp][k * kHeadC + lane] = dw[k];
      float t = db[k];
      for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
      if (lane == 0) sred[warp][kMaxK * kHeadC + k] = t;
    }
  }
  for (int o = 16; o > 0; o >>= 1) {
    nll_sum += __shfl_xor_sync(0xffffffffu, nll_sum, o);
    cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
  }
  if (lane == 0) {
    s_nll[warp] = nll_sum;
    s_cnt[warp] = cnt;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < K * kHeadC + K; i += blockDim.x) {
    const int src = i < K * kHeadC ? i : kMaxK * kHeadC + (i - K * kHeadC);
    float t = 0.f;
    for (int wv = 0; wv < kHeadLossWarps; ++wv) t += sred[wv][src];
    partial[static_cast<size_t>(blockIdx.x) * (K * kHeadC + K) + i] = t;
  }
  if (threadIdx.x == 0) {
    double t = 0;
    unsigned long long c = 0;
    for (int wv = 0; wv < kHeadLossWarps; ++wv) {
      t += s_nll[wv];
      c += s_cnt[wv];
    }
    atomicAdd(acc, t);
    atomicAdd(counts, c);
  }
  for (int i = threadIdx.x; i < K * K; i += blockDim.x)
    if (s_conf[i]) atomicAdd(confusion + i, static_cast<unsigned long long>(s_conf[i]));
}

// ---------------------------------------------------------------------------------------------
// Tensor-core version of the fused training head (same contract as head_loss_kernel above, which stays
// as the reference implementation behind spff_debug_set(2, 1)). The three tiny contractions of the head
//   logits[16 pos x 16 cls] = x[16 x 32] . W^T,   dx[16 x 32] = dl[16 x 16] . W,   dW[16 x 32] += dl^T . x
// run as warp-level mma.sync m16n8k16 tiles of 16 positions; softmax / CE / arg-max / confusion work on
// the accumulator fragments (a position's 16 logits live in the 4 lanes of a quad). fp32 accuracy is
// kept by splitting the fp32 operands into bf16 hi + lo parts (W for the logits and dx, dl for dx and dW):
// x is bf16 already, so logits carry ~2^-17 relative error and the loss, the tallies and the gradients
// match the CUDA-core kernel to fp32 rounding.
// ---------------------------------------------------------------------------------------------
constexpr int kHmWarps = 8;
constexpr int kHmBlocksPerSm = 2;
constexpr int kHmXPitch = 40;   // bf16 per staged x / dx row (32 + 8 pad)
constexpr int kHmDPitch = 24;   // bf16 per staged dl row (16 + 8 pad)

__device__ __forceinline__ void split_bf16x2(float v0, float v1, uint32_t& hi, uint32_t& lo) {
  const __nv_bfloat16 h0 = __float2bfloat16(v0), h1 = __float2bfloat16(v1);
  const __nv_bfloat162 h = __halves2bfloat162(h0, h1);
  const __nv_bfloat162 l = __floats2bfloat162_rn(v0 - __bfloat162float(h0), v1 - __bfloat162float(h1));
  hi = *reinterpret_cast<const uint32_t*>(&h);
  lo = *reinterpret_cast<const uint32_t*>(&l);
}

// ---- pieces shared by the fused training head (head_loss_mma_kernel) and the fused evaluation head
// (head_eval_mma_kernel): one warp works on tiles of 16 positions x 32 channels; g = lane / 4, t = lane % 4.

// B fragments of the logits contraction: B[k=ch][n=class] as bf16 hi + lo of W, plus the bias (classes >= K are zero)
struct HmLogitW {
  uint32_t hi[2][2][2], lo[2][2][2];   // [class tile][k step][b0,b1]
  float bias[2][2];
};

__device__ __forceinline__ void hm_logit_weights(int K, int g, int t, HmLogitW& w) {
  auto wv = [&](int k, int c) -> float { return k < K ? c_head_w[k * kHeadC + c] : 0.f; };
#pragma unroll
  for (int nt = 0; nt < 2; ++nt)
#pragma unroll
    for (int ks = 0; ks < 2; ++ks)
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int cls = 8 * nt + g, ch = 16 * ks + 8 * h + 2 * t;
        split_bf16x2(wv(cls, ch), wv(cls, ch + 1), w.hi[nt][ks][h], w.lo[nt][ks][h]);
      }
#pragma unroll
  for (int nt = 0; nt < 2; ++nt)
#pragma unroll
    for (int e = 0; e < 2; ++e) w.bias[nt][e] = (8 * nt + 2 * t + e) < K ? c_head_b[8 * nt + 2 * t + e] : 0.f;
}

// x rows (two 16-byte halves per lane) and the labels of rows g, g + 8 of `tile`; zeros / ignore_index past `total`
template <typename LabelT>
__device__ __forceinline__ void hm_fetch(const __nv_bfloat16* __restrict__ x, long long ldx, const void* __restrict__ labels,
                                         int ignore_index, long long total, long long ntiles, long long tile, int lane,
                                         uint4& nx0, uint4& nx1, int (&nlab)[2]) {
  const int g = lane >> 2;
  nx0 = nx1 = make_uint4(0, 0, 0, 0);
  nlab[0] = nlab[1] = ignore_index;
  if (tile >= ntiles) return;
  const long long q0 = tile * 16;
  const int pos = lane >> 1, half = lane & 1;
  if (q0 + pos < total) {
    const uint4* src = reinterpret_cast<const uint4*>(x + (q0 + pos) * ldx + half * 16);
    nx0 = __ldg(src);
    nx1 = __ldg(src + 1);
  }
#pragma unroll
  for (int rr = 0; rr < 2; ++rr)
    if (q0 + g + 8 * rr < total) nlab[rr] = static_cast<int>(static_cast<const LabelT*>(labels)[q0 + g + 8 * rr]);
}

// stage the fetched 16 positions x 32 channels into the warp's tile
__device__ __forceinline__ void hm_stage(__nv_bfloat16 (*xs)[kHmXPitch], int lane, const uint4& nx0, const uint4& nx1) {
  const int pos = lane >> 1, half = lane & 1;
  uint4* dst = reinterpret_cast<uint4*>(&xs[pos][half * 16]);
  dst[0] = nx0;
  dst[1] = nx1;
}

// logits of the staged tile: l[class tile][row g: 0..1 | row g + 8: 2..3] for classes 8 * tile + 2t + {0, 1}
__device__ __forceinline__ void hm_logits(__nv_bfloat16 (*xs)[kHmXPitch], int lane, const HmLogitW& w, float (&l)[2][4]) {
#pragma unroll
  for (int nt = 0; nt < 2; ++nt) {
    l[nt][0] = l[nt][2] = w.bias[nt][0];
    l[nt][1] = l[nt][3] = w.bias[nt][1];
  }
#pragma unroll
  for (int ks = 0; ks < 2; ++ks) {
    uint32_t a[4];
    const int mi = lane >> 3, r = lane & 7;
    const uint32_t addr = smem_u32_local(&xs[r + 8 * (mi & 1)][16 * ks + 8 * (mi >> 1)]);
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
                 : "=r"(a[0]), "=r"(a[1]), "=r"(a[2]), "=r"(a[3]) : "r"(addr));
#pragma unroll
    for (int nt = 0; nt < 2; ++nt) {
      mma_bf16_16816(l[nt], a, w.hi[nt][ks]);
      mma_bf16_16816(l[nt], a, w.lo[nt][ks]);
    }
  }
}

// softmax statistics of row g + 8 * rr (the 4 lanes of a quad hold 4 classes each): the row's maximum and its first
// arg-max (torch.argmax), e[q] = exp(v[q] - max) of this lane's classes cls[q], their quad sum se, and the logit of
// class `lab` (0 when `lab` is not a class)
__device__ __forceinline__ void hm_row_softmax(const float (&l)[2][4], int rr, int t, int K, int lab, float (&v)[4],
                                               int (&cls)[4], float& mx, int& arg, float (&e)[4], float& se, float& ll) {
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    cls[q] = 8 * (q >> 1) + 2 * t + (q & 1);
    v[q] = cls[q] < K ? l[q >> 1][2 * rr + (q & 1)] : -INFINITY;
  }
  mx = v[0];
  arg = cls[0];
#pragma unroll
  for (int q = 1; q < 4; ++q)
    if (v[q] > mx) {   // ascending class order inside the thread: strict > keeps the first maximum
      mx = v[q];
      arg = cls[q];
    }
#pragma unroll
  for (int o = 1; o <= 2; o <<= 1) {
    const float om = __shfl_xor_sync(0xffffffffu, mx, o);
    const int oa = __shfl_xor_sync(0xffffffffu, arg, o);
    if (om > mx || (om == mx && oa < arg)) {
      mx = om;
      arg = oa;
    }
  }
  se = 0.f;
  ll = 0.f;
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    e[q] = cls[q] < K ? __expf(v[q] - mx) : 0.f;
    se += e[q];
    if (cls[q] == lab) ll = v[q];
  }
#pragma unroll
  for (int o = 1; o <= 2; o <<= 1) {
    se += __shfl_xor_sync(0xffffffffu, se, o);
    ll += __shfl_xor_sync(0xffffffffu, ll, o);
  }
}

template <typename LabelT>
__global__ void __launch_bounds__(kHmWarps * 32, kHmBlocksPerSm)
head_loss_mma_kernel(const __nv_bfloat16* __restrict__ x, long long ldx, const void* __restrict__ labels, int ignore_index,
                     int K, long long total, const unsigned long long* __restrict__ n_valid,
                     const float* __restrict__ gscale, double* __restrict__ acc, unsigned long long* __restrict__ counts,
                     unsigned long long* __restrict__ confusion, __nv_bfloat16* __restrict__ dx, long long lddx,
                     float* __restrict__ partial /* [block][K*32 + K] */) {
  __shared__ __align__(16) __nv_bfloat16 xs[kHmWarps][16][kHmXPitch];
  __shared__ __align__(16) __nv_bfloat16 os[kHmWarps][16][kHmXPitch];
  __shared__ __align__(16) __nv_bfloat16 dls[kHmWarps][2][16][kHmDPitch];
  __shared__ float red[kMaxK * kHeadC + kMaxK];
  __shared__ unsigned int s_conf[kMaxK * kMaxK];
  __shared__ float s_nll[kHmWarps];
  __shared__ unsigned int s_cnt[kHmWarps];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int g = lane >> 2, t = lane & 3;
  for (int i = threadIdx.x; i < K * K; i += blockDim.x) s_conf[i] = 0;
  for (int i = threadIdx.x; i < kMaxK * kHeadC + kMaxK; i += blockDim.x) red[i] = 0.f;
  __syncthreads();
  const unsigned long long nv = n_valid[0];
  const float scale = (nv > 0 ? 1.f / static_cast<float>(nv) : 0.f) * (gscale ? gscale[0] : 1.f);

  // weight fragments (constant memory -> registers), classes >= K are zero
  auto wv = [&](int k, int c) -> float { return k < K ? c_head_w[k * kHeadC + c] : 0.f; };
  HmLogitW wl;
  hm_logit_weights(K, g, t, wl);
  uint32_t wd_hi[4][2], wd_lo[4][2];          // dx: [channel tile][b0,b1]: B[k=class][n=ch]
#pragma unroll
  for (int j = 0; j < 4; ++j)
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int cls = 8 * h + 2 * t, ch = 8 * j + g;
      split_bf16x2(wv(cls, ch), wv(cls + 1, ch), wd_hi[j][h], wd_lo[j][h]);
    }

  float dwacc[4][4], dbp[2][2];
#pragma unroll
  for (int j = 0; j < 4; ++j)
#pragma unroll
    for (int e = 0; e < 4; ++e) dwacc[j][e] = 0.f;
  dbp[0][0] = dbp[0][1] = dbp[1][0] = dbp[1][1] = 0.f;
  float nll_sum = 0.f;
  unsigned int cnt = 0;

  const long long ntiles = (total + 15) / 16;
  const long long tstep = static_cast<long long>(gridDim.x) * kHmWarps;
  // software prefetch: the x rows and the labels of the NEXT tile are requested before the current one is
  // computed, so the two global round trips per tile overlap the tensor-core work instead of preceding it
  uint4 nx0 = make_uint4(0, 0, 0, 0), nx1 = nx0;
  int nlab[2] = {ignore_index, ignore_index};
  hm_fetch<LabelT>(x, ldx, labels, ignore_index, total, ntiles, static_cast<long long>(blockIdx.x) * kHmWarps + warp, lane,
                   nx0, nx1, nlab);
  for (long long tile = static_cast<long long>(blockIdx.x) * kHmWarps + warp; tile < ntiles; tile += tstep) {
    const long long p0 = tile * 16;
    const int clab[2] = {nlab[0], nlab[1]};
    hm_stage(xs[warp], lane, nx0, nx1);   // 16 positions x 32 channels (zeros past the end)
    hm_fetch<LabelT>(x, ldx, labels, ignore_index, total, ntiles, tile + tstep, lane, nx0, nx1, nlab);
    __syncwarp();
    // ---- logits
    float l[2][4];
    hm_logits(xs[warp], lane, wl, l);
    // ---- per-row softmax / CE / arg-max: row g (values [nt][0..1]) and row g + 8 (values [nt][2..3])
    float dl[2][4];
#pragma unroll
    for (int rr = 0; rr < 2; ++rr) {
      const long long pos = p0 + g + 8 * rr;
      const bool inb = pos < total;
      const int lab = clab[rr];
      const bool valid = inb && lab != ignore_index;
      float v[4], mx, e[4], se, ll;
      int cls[4], arg;
      hm_row_softmax(l, rr, t, K, lab, v, cls, mx, arg, e, se, ll);
      if (valid && t == 0) {
        nll_sum += (mx + __logf(se)) - ll;
        ++cnt;
        if (lab >= 0 && lab < K) atomicAdd(&s_conf[lab * K + arg], 1u);
      }
      const float inv = 1.f / se;
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        float gq = 0.f;
        if (valid && cls[q] < K) gq = (e[q] * inv - (cls[q] == lab ? 1.f : 0.f)) * scale;
        dl[q >> 1][2 * rr + (q & 1)] = gq;
        dbp[q >> 1][q & 1] += gq;
      }
    }
    // ---- dl as bf16 hi + lo A fragments (row g | row g+8, classes 2t.. | 8+2t..)
    uint32_t ah[4], al[4];
    split_bf16x2(dl[0][0], dl[0][1], ah[0], al[0]);
    split_bf16x2(dl[0][2], dl[0][3], ah[1], al[1]);
    split_bf16x2(dl[1][0], dl[1][1], ah[2], al[2]);
    split_bf16x2(dl[1][2], dl[1][3], ah[3], al[3]);
    // ---- dx = dl . W  -> staged, then 16-byte coalesced stores
    if (dx) {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        float o[4] = {0.f, 0.f, 0.f, 0.f};
        mma_bf16_16816(o, ah, wd_hi[j]);
        mma_bf16_16816(o, al, wd_hi[j]);
        mma_bf16_16816(o, ah, wd_lo[j]);
        *reinterpret_cast<uint32_t*>(&os[warp][g][8 * j + 2 * t]) = pack_bf16x2_local(o[0], o[1]);
        *reinterpret_cast<uint32_t*>(&os[warp][g + 8][8 * j + 2 * t]) = pack_bf16x2_local(o[2], o[3]);
      }
    }
    // ---- stage dl (hi, lo) for the transposed operand of dW
    *reinterpret_cast<uint32_t*>(&dls[warp][0][g][2 * t]) = ah[0];
    *reinterpret_cast<uint32_t*>(&dls[warp][0][g + 8][2 * t]) = ah[1];
    *reinterpret_cast<uint32_t*>(&dls[warp][0][g][8 + 2 * t]) = ah[2];
    *reinterpret_cast<uint32_t*>(&dls[warp][0][g + 8][8 + 2 * t]) = ah[3];
    *reinterpret_cast<uint32_t*>(&dls[warp][1][g][2 * t]) = al[0];
    *reinterpret_cast<uint32_t*>(&dls[warp][1][g + 8][2 * t]) = al[1];
    *reinterpret_cast<uint32_t*>(&dls[warp][1][g][8 + 2 * t]) = al[2];
    *reinterpret_cast<uint32_t*>(&dls[warp][1][g + 8][8 + 2 * t]) = al[3];
    __syncwarp();
    if (dx) {
      const int pos = lane >> 1, half = lane & 1;
      if (p0 + pos < total) {
        const uint4* src = reinterpret_cast<const uint4*>(&os[warp][pos][half * 16]);
        uint4* dst = reinterpret_cast<uint4*>(dx + (p0 + pos) * lddx + half * 16);
        dst[0] = src[0];
        dst[1] = src[1];
      }
    }
    // ---- dW[class][ch] += dl^T . x   (A = dl^T through ldmatrix.trans, B = x through ldmatrix.trans)
    {
      const int mi = lane >> 3, r = lane & 7;
      uint32_t th[4], tl[4];
      const uint32_t ad_hi = smem_u32_local(&dls[warp][0][r + 8 * (mi >> 1)][8 * (mi & 1)]);
      const uint32_t ad_lo = smem_u32_local(&dls[warp][1][r + 8 * (mi >> 1)][8 * (mi & 1)]);
      asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
                   : "=r"(th[0]), "=r"(th[1]), "=r"(th[2]), "=r"(th[3]) : "r"(ad_hi));
      asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
                   : "=r"(tl[0]), "=r"(tl[1]), "=r"(tl[2]), "=r"(tl[3]) : "r"(ad_lo));
#pragma unroll
      for (int h2 = 0; h2 < 2; ++h2) {
        uint32_t bx[4];
        const uint32_t ax = smem_u32_local(&xs[warp][r + 8 * (mi & 1)][8 * (2 * h2 + (mi >> 1))]);
        asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
                     : "=r"(bx[0]), "=r"(bx[1]), "=r"(bx[2]), "=r"(bx[3]) : "r"(ax));
        const uint32_t b0[2] = {bx[0], bx[1]}, b1[2] = {bx[2], bx[3]};
        mma_bf16_16816(dwacc[2 * h2], th, b0);
        mma_bf16_16816(dwacc[2 * h2], tl, b0);
        mma_bf16_16816(dwacc[2 * h2 + 1], th, b1);
        mma_bf16_16816(dwacc[2 * h2 + 1], tl, b1);
      }
    }
    __syncwarp();
  }
  // ---- block reduction in a fixed order (warp after warp): dW fragments (row = class g | g+8, col = 8j + 2t..), db
#pragma unroll
  for (int nt = 0; nt < 2; ++nt)
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      float v = dbp[nt][e];
      for (int o = 4; o <= 16; o <<= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      dbp[nt][e] = v;
    }
  for (int o = 16; o > 0; o >>= 1) {
    nll_sum += __shfl_xor_sync(0xffffffffu, nll_sum, o);
    cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
  }
  if (lane == 0) {
    s_nll[warp] = nll_sum;
    s_cnt[warp] = cnt;
  }
  for (int wvv = 0; wvv < kHmWarps; ++wvv) {
    if (warp == wvv) {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        red[g * kHeadC + 8 * j + 2 * t] += dwacc[j][0];
        red[g * kHeadC + 8 * j + 2 * t + 1] += dwacc[j][1];
        red[(g + 8) * kHeadC + 8 * j + 2 * t] += dwacc[j][2];
        red[(g + 8) * kHeadC + 8 * j + 2 * t + 1] += dwacc[j][3];
      }
      if (g == 0) {
#pragma unroll
        for (int nt = 0; nt < 2; ++nt)
#pragma unroll
          for (int e = 0; e < 2; ++e) red[kMaxK * kHeadC + 8 * nt + 2 * t + e] += dbp[nt][e];
      }
    }
    __syncthreads();
  }
  for (int i = threadIdx.x; i < K * kHeadC + K; i += blockDim.x) {
    const int src = i < K * kHeadC ? i : kMaxK * kHeadC + (i - K * kHeadC);
    partial[static_cast<size_t>(blockIdx.x) * (K * kHeadC + K) + i] = red[src];
  }
  if (threadIdx.x == 0) {
    double tt = 0;
    unsigned long long c = 0;
    for (int wvv = 0; wvv < kHmWarps; ++wvv) {
      tt += s_nll[wvv];
      c += s_cnt[wvv];
    }
    atomicAdd(acc, tt);
    atomicAdd(counts, c);
  }
  for (int i = threadIdx.x; i < K * K; i += blockDim.x)
    if (s_conf[i]) atomicAdd(confusion + i, static_cast<unsigned long long>(s_conf[i]));
}

// ---------------------------------------------------------------------------------------------
// Fused EVALUATION head: the logits / softmax / arg-max of head_loss_mma_kernel (same functions, so the same
// numbers) followed by the CE / confusion tally of ce_kernel, with no gradient. Block (x, y) works on sample y
// only, so a block's tally belongs to one sample: it is kept in shared memory and flushed once per block to
// the batch arrays and, when given, to the sample's row of the per-sample arrays. Optionally the arg-max map
// (the one the tally counts) is written. Traffic: the 64 B of x + the label per voxel (+ 1 B of arg-max).
//
// HIST adds the ranking statistics: for every counted voxel (label in [0, K), not ignore_index) and every class c,
// p_c = e_c / se (IEEE division) falls in bin min(floor(p_c * T), T - 1) of hist[c][label == c ? 0 : 1][T], a
// sufficient statistic of the ROC and PR curves at the thresholds i / T. The block-private histogram is uint32
// [K][2][T] in dynamic shared memory. The two bins almost every voxel lands in once the model is trained (a negative
// in bin 0, a positive in bin T - 1) are counted in registers per lane and added at the flush, so that they do not
// serialise the block on two shared addresses.
// ---------------------------------------------------------------------------------------------
constexpr int kHeBlocksPerSm = 3;
constexpr int kHeMinBins = 16, kHeMaxBins = 1024;

template <typename LabelT, bool HIST>
__global__ void __launch_bounds__(kHmWarps * 32, kHeBlocksPerSm)
head_eval_mma_kernel(const __nv_bfloat16* __restrict__ x, long long ldx, const void* __restrict__ labels, int ignore_index,
                     int K, long long dhw, double* __restrict__ acc, unsigned long long* __restrict__ counts,
                     unsigned long long* __restrict__ confusion, double* __restrict__ sample_acc,
                     unsigned long long* __restrict__ sample_counts, unsigned long long* __restrict__ sample_confusion,
                     uint8_t* __restrict__ labels_out, int T, unsigned long long* __restrict__ hist,
                     unsigned long long* __restrict__ sample_hist) {
  __shared__ __align__(16) __nv_bfloat16 xs[kHmWarps][16][kHmXPitch];
  __shared__ unsigned int s_conf[kMaxK * kMaxK];
  __shared__ float s_nll[kHmWarps];
  __shared__ unsigned int s_cnt[kHmWarps];
  extern __shared__ unsigned int s_hist[];   // HIST: [K][2][T]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int g = lane >> 2, t = lane & 3;
  for (int i = threadIdx.x; i < K * K; i += blockDim.x) s_conf[i] = 0;
  if constexpr (HIST)
    for (int i = threadIdx.x; i < K * 2 * T; i += blockDim.x) s_hist[i] = 0;
  unsigned int hot_neg[4] = {0, 0, 0, 0}, hot_pos[4] = {0, 0, 0, 0};   // HIST: bin 0 of negatives, bin T - 1 of positives
  __syncthreads();
  HmLogitW wl;
  hm_logit_weights(K, g, t, wl);
  const long long n = blockIdx.y;
  const long long base = n * dhw;   // this block's sample: positions [base, base + dhw)
  x += base * ldx;
  labels = static_cast<const LabelT*>(labels) + base;
  if (labels_out) labels_out += base;
  float nll_sum = 0.f;
  unsigned int cnt = 0;
  const long long ntiles = (dhw + 15) / 16;
  const long long tstep = static_cast<long long>(gridDim.x) * kHmWarps;
  uint4 nx0 = make_uint4(0, 0, 0, 0), nx1 = nx0;
  int nlab[2] = {ignore_index, ignore_index};
  hm_fetch<LabelT>(x, ldx, labels, ignore_index, dhw, ntiles, static_cast<long long>(blockIdx.x) * kHmWarps + warp, lane,
                   nx0, nx1, nlab);
  for (long long tile = static_cast<long long>(blockIdx.x) * kHmWarps + warp; tile < ntiles; tile += tstep) {
    const long long p0 = tile * 16;
    const int clab[2] = {nlab[0], nlab[1]};
    hm_stage(xs[warp], lane, nx0, nx1);
    hm_fetch<LabelT>(x, ldx, labels, ignore_index, dhw, ntiles, tile + tstep, lane, nx0, nx1, nlab);
    __syncwarp();
    float l[2][4];
    hm_logits(xs[warp], lane, wl, l);
#pragma unroll
    for (int rr = 0; rr < 2; ++rr) {
      const long long pos = p0 + g + 8 * rr;
      const bool inb = pos < dhw;
      const int lab = clab[rr];
      float v[4], mx, e[4], se, ll;
      int cls[4], arg;
      hm_row_softmax(l, rr, t, K, lab, v, cls, mx, arg, e, se, ll);
      if (inb && t == 0) {
        if (labels_out) labels_out[pos] = static_cast<uint8_t>(arg);
        if (lab != ignore_index) {
          nll_sum += (mx + __logf(se)) - ll;
          ++cnt;
          if (lab >= 0 && lab < K) atomicAdd(&s_conf[lab * K + arg], 1u);
        }
      }
      if constexpr (HIST) {   // all four lanes of the quad: classes cls[0..3] of this row
        if (inb && lab != ignore_index && lab >= 0 && lab < K) {
#pragma unroll
          for (int q = 0; q < 4; ++q)
            if (cls[q] < K) {
              const float p = __fdiv_rn(e[q], se);
              const int bin = min(static_cast<int>(__fmul_rn(p, static_cast<float>(T))), T - 1);
              const bool positive = cls[q] == lab;
              if (positive && bin == T - 1)
                ++hot_pos[q];
              else if (!positive && bin == 0)
                ++hot_neg[q];
              else
                atomicAdd(&s_hist[(cls[q] * 2 + (positive ? 0 : 1)) * T + bin], 1u);
            }
        }
      }
    }
    __syncwarp();   // the tile is read before the next iteration overwrites it
  }
  for (int o = 16; o > 0; o >>= 1) {
    nll_sum += __shfl_xor_sync(0xffffffffu, nll_sum, o);
    cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
  }
  if (lane == 0) {
    s_nll[warp] = nll_sum;
    s_cnt[warp] = cnt;
  }
  if constexpr (HIST) {   // the register bins: sum over the 8 lanes holding the same classes, then one add per warp
#pragma unroll
    for (int q = 0; q < 4; ++q) {
#pragma unroll
      for (int o = 4; o < 32; o <<= 1) {
        hot_pos[q] += __shfl_xor_sync(0xffffffffu, hot_pos[q], o);
        hot_neg[q] += __shfl_xor_sync(0xffffffffu, hot_neg[q], o);
      }
      const int c = 8 * (q >> 1) + 2 * t + (q & 1);
      if (g == 0 && c < K) {
        if (hot_pos[q]) atomicAdd(&s_hist[(c * 2 + 0) * T + T - 1], hot_pos[q]);
        if (hot_neg[q]) atomicAdd(&s_hist[(c * 2 + 1) * T + 0], hot_neg[q]);
      }
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double tt = 0;
    unsigned long long c = 0;
    for (int wvv = 0; wvv < kHmWarps; ++wvv) {
      tt += s_nll[wvv];
      c += s_cnt[wvv];
    }
    atomicAdd(acc, tt);
    atomicAdd(counts, c);
    if (sample_acc) {
      atomicAdd(sample_acc + n, tt);
      atomicAdd(sample_counts + n, c);
    }
  }
  for (int i = threadIdx.x; i < K * K; i += blockDim.x)
    if (s_conf[i]) {
      atomicAdd(confusion + i, static_cast<unsigned long long>(s_conf[i]));
      if (sample_confusion) atomicAdd(sample_confusion + n * K * K + i, static_cast<unsigned long long>(s_conf[i]));
    }
  if constexpr (HIST)
    for (int i = threadIdx.x; i < K * 2 * T; i += blockDim.x)
      if (s_hist[i]) {
        atomicAdd(hist + i, static_cast<unsigned long long>(s_hist[i]));
        if (sample_hist) atomicAdd(sample_hist + n * K * 2 * T + i, static_cast<unsigned long long>(s_hist[i]));
      }
}

// ---------------------------------------------------------------------------------------------
// Averaged softmax (ensembles, mirror TTA). head_prob_accum_kernel: the logits / softmax of head_eval_mma_kernel
// (same functions, so the same numbers), p_c = e_c / se with the IEEE division the histogram uses, added into the
// fp32 accumulator acc [n][d][h][w][16] at the position mirrored back by `flip` (1 = H, 2 = W). Within one (n, d)
// plane the flip is a bijection, so every accumulator element has exactly one writer per launch: plain
// load-add-store, deterministic. beta = 0 stores p (and 0 for classes >= K) without reading acc.
// ENT: also ent [n][d][h'][w'] = beta * ent + H(p), the entropy of this pass's softmax, at the same mirrored position
// (the expected-entropy plane of the mutual information). From the row's softmax statistics:
// H = log(se) - sum_{c<K} e_c (v_c - mx) / se, the quad's partial sums reduced with two shuffles; lane t = 0 of the
// row writes it (one writer per element per launch, as for acc).
// ---------------------------------------------------------------------------------------------
constexpr int kPaBlocksPerSm = 3;

// x rows (two 16-byte halves per lane) of `tile`; zeros past `total` (hm_fetch without labels)
__device__ __forceinline__ void hm_fetch_x(const __nv_bfloat16* __restrict__ x, long long ldx, long long total,
                                           long long ntiles, long long tile, int lane, uint4& nx0, uint4& nx1) {
  nx0 = nx1 = make_uint4(0, 0, 0, 0);
  if (tile >= ntiles) return;
  const long long q0 = tile * 16;
  const int pos = lane >> 1, half = lane & 1;
  if (q0 + pos < total) {
    const uint4* src = reinterpret_cast<const uint4*>(x + (q0 + pos) * ldx + half * 16);
    nx0 = __ldg(src);
    nx1 = __ldg(src + 1);
  }
}

template <bool ENT>
__global__ void __launch_bounds__(kHmWarps * 32, kPaBlocksPerSm)
head_prob_accum_kernel(const __nv_bfloat16* __restrict__ x, long long ldx, int K, int H, int W, long long dhw, int flip,
                       int beta, float* __restrict__ acc, float* __restrict__ ent) {
  __shared__ __align__(16) __nv_bfloat16 xs[kHmWarps][16][kHmXPitch];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int g = lane >> 2, t = lane & 3;
  HmLogitW wl;
  hm_logit_weights(K, g, t, wl);
  const long long n = blockIdx.y;
  x += n * dhw * ldx;
  acc += n * dhw * kMaxK;
  if constexpr (ENT) ent += n * dhw;
  const long long hw = static_cast<long long>(H) * W;
  const long long ntiles = (dhw + 15) / 16;
  const long long tstep = static_cast<long long>(gridDim.x) * kHmWarps;
  uint4 nx0, nx1;
  hm_fetch_x(x, ldx, dhw, ntiles, static_cast<long long>(blockIdx.x) * kHmWarps + warp, lane, nx0, nx1);
  for (long long tile = static_cast<long long>(blockIdx.x) * kHmWarps + warp; tile < ntiles; tile += tstep) {
    const long long p0 = tile * 16;
    hm_stage(xs[warp], lane, nx0, nx1);
    hm_fetch_x(x, ldx, dhw, ntiles, tile + tstep, lane, nx0, nx1);
    __syncwarp();
    float l[2][4];
    hm_logits(xs[warp], lane, wl, l);
#pragma unroll
    for (int rr = 0; rr < 2; ++rr) {
      const long long pos = p0 + g + 8 * rr;
      float v[4], mx, e[4], se, ll;
      int cls[4], arg;
      hm_row_softmax(l, rr, t, K, -1, v, cls, mx, arg, e, se, ll);
      float h_p = 0.f;
      if constexpr (ENT) {
        float ev = 0.f;
#pragma unroll
        for (int q = 0; q < 4; ++q)
          if (cls[q] < K) ev = fmaf(e[q], v[q] - mx, ev);   // classes >= K: v = -inf, e = 0, and 0 * -inf is NaN
#pragma unroll
        for (int o = 1; o <= 2; o <<= 1) ev += __shfl_xor_sync(0xffffffffu, ev, o);
        h_p = __logf(se) - __fdividef(ev, se);
      }
      if (pos < dhw) {
        const long long plane = pos / hw, rem = pos - plane * hw;
        int hh = static_cast<int>(rem / W), ww = static_cast<int>(rem - static_cast<long long>(hh) * W);
        if (flip & 1) hh = H - 1 - hh;
        if (flip & 2) ww = W - 1 - ww;
        float* dst = acc + (plane * hw + static_cast<long long>(hh) * W + ww) * kMaxK;
#pragma unroll
        for (int j = 0; j < 2; ++j) {   // this lane's classes 8j + 2t, 8j + 2t + 1 (e[2j], e[2j + 1])
          const int c0 = 8 * j + 2 * t;
          const float2 p = make_float2(c0 < K ? __fdiv_rn(e[2 * j], se) : 0.f, c0 + 1 < K ? __fdiv_rn(e[2 * j + 1], se) : 0.f);
          float2* d2 = reinterpret_cast<float2*>(dst + c0);
          if (!beta) {
            *d2 = p;
          } else if (c0 + 1 < K) {
            float2 o = *d2;
            o.x = __fadd_rn(o.x, p.x);
            o.y = __fadd_rn(o.y, p.y);
            *d2 = o;
          } else if (c0 < K) {
            dst[c0] = __fadd_rn(dst[c0], p.x);
          }
        }
        if constexpr (ENT) {
          if (t == 0) {
            float* de = ent + plane * hw + static_cast<long long>(hh) * W + ww;
            *de = beta ? __fadd_rn(*de, h_p) : h_p;
          }
        }
      }
    }
    __syncwarp();   // the tile is read before the next iteration overwrites it
  }
}

// prob_finalize_kernel: one thread per position of sample blockIdx.y. p̄_c = scale * acc_c; the arg-max is the first
// maximum of acc_c over c < K (on acc, so that the scaling cannot create ties). With labels: a label equal to
// ignore_index is not counted; a label in [0, K) counts, adds -log(max(p̄_y, FLT_MIN)) to the nll and one to
// confusion[y][arg] (and, with HIST, every class's p̄_c to bin min(floor(p̄_c * T), T - 1) of hist[c][y == c ? 0 : 1]);
// any other label counts only. Tallies are block-private in shared memory and flushed once per block, as in
// head_eval_mma_kernel (the register bins too).
// UNC (spff_prob_finalize_unc, outputs in `u`): per position H[p̄] = -sum_{c<K} p̄_c log p̄_c (0 log 0 = 0) and, with the
// expected-entropy plane u.ent, MI = max(H[p̄] - scale * ent, 0); optional fp16 maps, and both rounded per position to
// the 2^-24 fixed point and summed in integers (bit-reproducible whatever the launch order). With u.calib (needs labels),
// every counted voxel (label in [0, K)) adds to confidence bin min(floor(conf * Tc), Tc - 1), conf = p̄_arg: one count,
// one if arg == label, and conf in units of 2^-24; its Brier term sum_c (p̄_c - [c == y])^2 is reduced like the nll.
// The top bin is counted in registers (a trained model puts most voxels there); the UNC tallies live in dynamic shared
// memory behind the HIST histogram: ull [2] uncertainty sums, ull [Tc] confidence sums, u32 [2][Tc] counts, float [8].
// TEMP (spff_prob_finalize_tempered, inv_t = β = 1/T): p̃_c = p̄_c^β / sum_{c'<K} p̄_c'^β, computed as
// e_c = exp(β (log p̄_c - log p̄_arg)) / sum e (accurate logf / expf; p̄_c = 0 stays 0), replaces p̄ everywhere below:
// proba_out, nll, HIST, H[p̃] (entropy_out and the H sum), the confidence p̃_arg and Brier. The arg-max is still taken
// on acc (p̃ is a monotone map of p̄) and the mutual information keeps H[p̄], the untempered passes' disagreement.
constexpr int kPfThreads = 256;
constexpr float kFix24 = 16777216.f;   // 2^24

// the block's uncertainty sums into unc[2] and its sample's row of sample_unc [N][2]
__device__ __forceinline__ void prob_finalize_flush_unc(const spff_unc_out& u, long long n, const unsigned long long* s_u) {
  auto unc = reinterpret_cast<unsigned long long*>(u.unc);
  auto sunc = reinterpret_cast<unsigned long long*>(u.sample_unc);
  atomicAdd(unc, s_u[0]);
  atomicAdd(unc + 1, s_u[1]);
  if (sunc) {
    atomicAdd(sunc + 2 * n, s_u[0]);
    atomicAdd(sunc + 2 * n + 1, s_u[1]);
  }
}

template <typename LabelT, bool HIST, bool UNC = false, bool TEMP = false>
__global__ void __launch_bounds__(kPfThreads)
prob_finalize_kernel(const float* __restrict__ acc, int K, long long dhw, float scale, const void* __restrict__ labels,
                     int ignore_index, double* __restrict__ nll, unsigned long long* __restrict__ counts,
                     unsigned long long* __restrict__ confusion, double* __restrict__ sample_acc,
                     unsigned long long* __restrict__ sample_counts, unsigned long long* __restrict__ sample_confusion,
                     uint8_t* __restrict__ labels_out, __half* __restrict__ proba_out, int T,
                     unsigned long long* __restrict__ hist, unsigned long long* __restrict__ sample_hist,
                     spff_unc_out u, float inv_t) {
  __shared__ unsigned int s_conf[kMaxK * kMaxK];
  __shared__ float s_nll[kPfThreads / 32];
  __shared__ unsigned int s_cnt[kPfThreads / 32];
  extern __shared__ unsigned int s_hist[];   // HIST: [K][2][T]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (int i = threadIdx.x; i < K * K; i += blockDim.x) s_conf[i] = 0;
  if constexpr (HIST)
    for (int i = threadIdx.x; i < K * 2 * T; i += blockDim.x) s_hist[i] = 0;
  unsigned int hot_neg[kMaxK], hot_pos[kMaxK];   // HIST: bin 0 of negatives, bin T - 1 of positives
#pragma unroll
  for (int c = 0; c < kMaxK; ++c) hot_neg[c] = hot_pos[c] = 0;
  [[maybe_unused]] unsigned long long* s_u = nullptr;   // UNC: [0] sum H, [1] sum MI, [2, 2 + Tc) confidence sums
  [[maybe_unused]] unsigned int* s_cal = nullptr;       // UNC: [0][Tc] counted, [1][Tc] correct
  [[maybe_unused]] float* s_brier = nullptr;            // UNC: per warp
  [[maybe_unused]] const int Tc = UNC && u.calib ? u.cal_bins : 0;
  [[maybe_unused]] long long h_sum = 0, mi_sum = 0, top_conf = 0;
  [[maybe_unused]] unsigned int top_cnt = 0, top_cor = 0;
  [[maybe_unused]] float brier_sum = 0.f;
  if constexpr (UNC) {
    extern __shared__ unsigned long long s_dyn64[];
    s_u = s_dyn64 + (HIST ? K * T : 0);
    s_cal = reinterpret_cast<unsigned int*>(s_u + 2 + Tc);
    s_brier = reinterpret_cast<float*>(s_cal + 2 * Tc);
    for (int i = threadIdx.x; i < 2 + Tc; i += blockDim.x) s_u[i] = 0;
    for (int i = threadIdx.x; i < 2 * Tc; i += blockDim.x) s_cal[i] = 0;
  }
  __syncthreads();
  const long long n = blockIdx.y;
  acc += n * dhw * kMaxK;
  const LabelT* lab_in = labels ? static_cast<const LabelT*>(labels) + n * dhw : nullptr;
  if (labels_out) labels_out += n * dhw;
  if (proba_out) proba_out += n * K * dhw;
  float nll_sum = 0.f;
  unsigned int cnt = 0;
  for (long long pos = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; pos < dhw;
       pos += static_cast<long long>(gridDim.x) * blockDim.x) {
    float a[kMaxK];
    const float4* src = reinterpret_cast<const float4*>(acc + pos * kMaxK);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float4 q = __ldg(src + j);
      a[4 * j] = q.x;
      a[4 * j + 1] = q.y;
      a[4 * j + 2] = q.z;
      a[4 * j + 3] = q.w;
    }
    int arg = 0;
    float mx = a[0];
#pragma unroll
    for (int c = 1; c < kMaxK; ++c)
      if (c < K && a[c] > mx) {   // ascending class order: strict > keeps the first maximum
        mx = a[c];
        arg = c;
      }
    float p[kMaxK];
#pragma unroll
    for (int c = 0; c < kMaxK; ++c) p[c] = __fmul_rn(scale, a[c]);
    [[maybe_unused]] float hb_bar = 0.f;   // TEMP: H[p̄] for the mutual information, as the untempered pass sums it
    [[maybe_unused]] float p_arg = 0.f;    // TEMP: p̃_arg
    if constexpr (TEMP) {
      const float l_arg = logf(__fmul_rn(scale, mx));
      float se = 0.f;
#pragma unroll
      for (int c = 0; c < kMaxK; ++c) {
        float e = 0.f;
        if (c < K && p[c] > 0.f) {
          const float l = logf(p[c]);
          if constexpr (UNC) hb_bar = fmaf(-p[c], l, hb_bar);
          e = expf(inv_t * (l - l_arg));
        }
        p[c] = e;
        se += e;
      }
#pragma unroll
      for (int c = 0; c < kMaxK; ++c) {
        if (se > 0.f) p[c] = __fdiv_rn(p[c], se);   // se = 0 only for an all-zero accumulator row: p̃ = 0
        if (c == arg) p_arg = p[c];
      }
    }
    if (labels_out) labels_out[pos] = static_cast<uint8_t>(arg);
    if (proba_out) {
#pragma unroll
      for (int c = 0; c < kMaxK; ++c)
        if (c < K) proba_out[c * dhw + pos] = __float2half_rn(p[c]);
    }
    if constexpr (UNC) {
      float hb = 0.f;
#pragma unroll
      for (int c = 0; c < kMaxK; ++c)
        if (c < K && p[c] > 0.f) hb = fmaf(-p[c], logf(p[c]), hb);
      hb = fmaxf(hb, 0.f);   // p̄_c may exceed 1 by an ulp
      float mi = 0.f;
      if constexpr (TEMP) {
        if (u.ent) mi = fmaxf(fmaxf(hb_bar, 0.f) - __fmul_rn(scale, __ldg(u.ent + n * dhw + pos)), 0.f);
      } else {
        if (u.ent) mi = fmaxf(hb - __fmul_rn(scale, __ldg(u.ent + n * dhw + pos)), 0.f);
      }
      if (u.entropy_out) static_cast<__half*>(u.entropy_out)[n * dhw + pos] = __float2half_rn(hb);
      if (u.mi_out) static_cast<__half*>(u.mi_out)[n * dhw + pos] = __float2half_rn(mi);
      h_sum += __float2ll_rn(hb * kFix24);
      mi_sum += __float2ll_rn(mi * kFix24);
    }
    if (lab_in) {
      const int lab = static_cast<int>(lab_in[pos]);
      if (lab != ignore_index) {
        ++cnt;
        if (lab >= 0 && lab < K) {
          float py = p[0];
#pragma unroll
          for (int c = 1; c < kMaxK; ++c)
            if (c == lab) py = p[c];
          nll_sum += -logf(fmaxf(py, FLT_MIN));
          atomicAdd(&s_conf[lab * K + arg], 1u);
          if constexpr (HIST) {
#pragma unroll
            for (int c = 0; c < kMaxK; ++c)
              if (c < K) {
                const int bin = min(static_cast<int>(__fmul_rn(p[c], static_cast<float>(T))), T - 1);
                const bool positive = c == lab;
                if (positive && bin == T - 1)
                  ++hot_pos[c];
                else if (!positive && bin == 0)
                  ++hot_neg[c];
                else
                  atomicAdd(&s_hist[(c * 2 + (positive ? 0 : 1)) * T + bin], 1u);
              }
          }
          if constexpr (UNC) {
            if (Tc) {
              const float conf = TEMP ? p_arg : __fmul_rn(scale, mx);   // p̄_arg (p̃_arg)
              const int bin = min(static_cast<int>(__fmul_rn(conf, static_cast<float>(Tc))), Tc - 1);
              const long long cfix = __float2ll_rn(conf * kFix24);
              const unsigned int correct = arg == lab ? 1u : 0u;
              if (bin == Tc - 1) {
                ++top_cnt;
                top_cor += correct;
                top_conf += cfix;
              } else {
                atomicAdd(&s_cal[bin], 1u);
                if (correct) atomicAdd(&s_cal[Tc + bin], 1u);
                atomicAdd(&s_u[2 + bin], static_cast<unsigned long long>(cfix));
              }
              float b = 0.f;
#pragma unroll
              for (int c = 0; c < kMaxK; ++c)
                if (c < K) {
                  const float dlt = c == lab ? p[c] - 1.f : p[c];
                  b = fmaf(dlt, dlt, b);
                }
              brier_sum += b;
            }
          }
        }
      }
    }
  }
  if constexpr (UNC) {
    for (int o = 16; o > 0; o >>= 1) {
      h_sum += __shfl_xor_sync(0xffffffffu, h_sum, o);
      mi_sum += __shfl_xor_sync(0xffffffffu, mi_sum, o);
    }
    if (lane == 0) {
      atomicAdd(&s_u[0], static_cast<unsigned long long>(h_sum));
      atomicAdd(&s_u[1], static_cast<unsigned long long>(mi_sum));
    }
    if (!lab_in) {
      __syncthreads();
      if (threadIdx.x == 0 && u.unc) prob_finalize_flush_unc(u, n, s_u);
      return;
    }
    if (Tc) {
      for (int o = 16; o > 0; o >>= 1) {
        top_cnt += __shfl_xor_sync(0xffffffffu, top_cnt, o);
        top_cor += __shfl_xor_sync(0xffffffffu, top_cor, o);
        top_conf += __shfl_xor_sync(0xffffffffu, top_conf, o);
        brier_sum += __shfl_xor_sync(0xffffffffu, brier_sum, o);
      }
      if (lane == 0) {
        s_brier[warp] = brier_sum;
        if (top_cnt) {
          atomicAdd(&s_cal[Tc - 1], top_cnt);
          if (top_cor) atomicAdd(&s_cal[2 * Tc - 1], top_cor);
          atomicAdd(&s_u[2 + Tc - 1], static_cast<unsigned long long>(top_conf));
        }
      }
    }
  }
  if (!lab_in) return;
  for (int o = 16; o > 0; o >>= 1) {
    nll_sum += __shfl_xor_sync(0xffffffffu, nll_sum, o);
    cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
  }
  if (lane == 0) {
    s_nll[warp] = nll_sum;
    s_cnt[warp] = cnt;
  }
  if constexpr (HIST) {   // the register bins: a warp sum, then one shared add per warp and class
#pragma unroll
    for (int c = 0; c < kMaxK; ++c) {
      if (c >= K) break;
      unsigned int hp = hot_pos[c], hn = hot_neg[c];
      for (int o = 16; o > 0; o >>= 1) {
        hp += __shfl_xor_sync(0xffffffffu, hp, o);
        hn += __shfl_xor_sync(0xffffffffu, hn, o);
      }
      if (lane == 0) {
        if (hp) atomicAdd(&s_hist[(c * 2 + 0) * T + T - 1], hp);
        if (hn) atomicAdd(&s_hist[(c * 2 + 1) * T + 0], hn);
      }
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double tt = 0;
    unsigned long long c = 0;
    for (int wv = 0; wv < kPfThreads / 32; ++wv) {
      tt += s_nll[wv];
      c += s_cnt[wv];
    }
    atomicAdd(nll, tt);
    atomicAdd(counts, c);
    if (sample_acc) {
      atomicAdd(sample_acc + n, tt);
      atomicAdd(sample_counts + n, c);
    }
  }
  for (int i = threadIdx.x; i < K * K; i += blockDim.x)
    if (s_conf[i]) {
      atomicAdd(confusion + i, static_cast<unsigned long long>(s_conf[i]));
      if (sample_confusion) atomicAdd(sample_confusion + n * K * K + i, static_cast<unsigned long long>(s_conf[i]));
    }
  if constexpr (HIST)
    for (int i = threadIdx.x; i < K * 2 * T; i += blockDim.x)
      if (s_hist[i]) {
        atomicAdd(hist + i, static_cast<unsigned long long>(s_hist[i]));
        if (sample_hist) atomicAdd(sample_hist + n * K * 2 * T + i, static_cast<unsigned long long>(s_hist[i]));
      }
  if constexpr (UNC) {
    if (threadIdx.x == 0) {
      if (u.unc) prob_finalize_flush_unc(u, n, s_u);
      if (Tc) {
        double bt = 0;
        for (int wv = 0; wv < kPfThreads / 32; ++wv) bt += s_brier[wv];
        atomicAdd(u.brier, bt);
        if (u.sample_brier) atomicAdd(u.sample_brier + n, bt);
      }
    }
    auto cal = reinterpret_cast<unsigned long long*>(u.calib);
    auto scal = reinterpret_cast<unsigned long long*>(u.sample_calib);
    for (int i = threadIdx.x; i < Tc; i += blockDim.x) {
      const unsigned long long v[3] = {s_cal[i], s_cal[Tc + i], s_u[2 + i]};
#pragma unroll
      for (int r = 0; r < 3; ++r)
        if (v[r]) {
          atomicAdd(cal + r * Tc + i, v[r]);
          if (scal) atomicAdd(scal + (n * 3 + r) * Tc + i, v[r]);
        }
    }
  }
}

// prob_temp_fit_kernel: the statistics of the temperature fit on the pooled p̄ = scale * acc. A voxel counts when its
// label y is in [0, K) and not ignore_index. With l_c = log p̄_c, m = l_arg (the first maximum of acc, as in
// prob_finalize_kernel) and d_c = l_c - m over the classes c != arg with p̄_c > 0, for each grid value β_g:
//   f(β)  = log sum_c exp(β l_c) - β l_y = β (m - l_y) + log1p(s1),            s1 = sum_c exp(β d_c),
//   f'(β) = sum_c p̃_c l_c - l_y         = (m - l_y) + sum_c exp(β d_c) d_c / (1 + s1),
// the forms without cancellation when y = arg; a voxel with p̄_y = 0 adds -log FLT_MIN to f and 0 to f' (the nll rule
// of prob_finalize_kernel). Accurate logf / expf / log1pf. Each warp takes tiles of 32 voxels of the flattened
// [N*D*H*W] grid: lane i stages voxel i's d_c and m - l_y in shared memory, then lane j evaluates grid points j and
// j + 32 over the tile's voxels (broadcast reads) and adds f, f' into fp64 registers. The block's sums (warps added in
// order) and its count go to partial[block][2G + 1] (count as u64 bits); prob_temp_fit_reduce_kernel adds the blocks in
// order. No floating-point atomics, so the result is bit-reproducible for a given grid; fp64 cannot overflow.
constexpr int kTfThreads = 256, kTfBlocksPerSm = 4, kTfMaxG = 64;
constexpr float kTfSkip = -1.f, kTfZeroY = -2.f;   // staged m - l_y (>= 0 otherwise): not counted, p̄_y = 0

template <typename LabelT>
__global__ void __launch_bounds__(kTfThreads, kTfBlocksPerSm)
prob_temp_fit_kernel(const float* __restrict__ acc, int K, long long total, float scale,
                     const LabelT* __restrict__ labels, int ignore_index, const float* __restrict__ betas, int G,
                     double* __restrict__ partial) {
  constexpr int kWarps = kTfThreads / 32;
  __shared__ float s_d[kWarps][32][kMaxK + 1];   // per voxel of the warp's tile: d_c (-inf: left out), m - l_y
  __shared__ double s_part[kWarps][2 * kTfMaxG];
  __shared__ unsigned int s_cnt[kWarps];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float beta[2];
#pragma unroll
  for (int j = 0; j < 2; ++j) beta[j] = lane + 32 * j < G ? __ldg(betas + lane + 32 * j) : 1.f;
  double sf[2] = {0.0, 0.0}, sd[2] = {0.0, 0.0};
  unsigned int cnt = 0;
  const long long ntiles = (total + 31) / 32;
  for (long long tile = static_cast<long long>(blockIdx.x) * kWarps + warp; tile < ntiles;
       tile += static_cast<long long>(gridDim.x) * kWarps) {
    const long long pos = tile * 32 + lane;
    float dy = kTfSkip;
    if (pos < total) {
      const int lab = static_cast<int>(labels[pos]);
      if (lab != ignore_index && lab >= 0 && lab < K) {
        ++cnt;
        float a[kMaxK];
        const float4* src = reinterpret_cast<const float4*>(acc + pos * kMaxK);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float4 q = __ldg(src + j);
          a[4 * j] = q.x;
          a[4 * j + 1] = q.y;
          a[4 * j + 2] = q.z;
          a[4 * j + 3] = q.w;
        }
        int arg = 0;
        float mx = a[0];
#pragma unroll
        for (int c = 1; c < kMaxK; ++c)
          if (c < K && a[c] > mx) {
            mx = a[c];
            arg = c;
          }
        const float m = logf(__fmul_rn(scale, mx));
#pragma unroll
        for (int c = 0; c < kMaxK; ++c) {
          const float p = __fmul_rn(scale, a[c]);
          const float l = c < K && p > 0.f ? logf(p) : 0.f;
          if (c < K) s_d[warp][lane][c] = c != arg && p > 0.f ? l - m : -INFINITY;
          if (c == lab) dy = p > 0.f ? m - l : kTfZeroY;
        }
      }
    }
    s_d[warp][lane][kMaxK] = dy;
    __syncwarp();
    for (int v = 0; v < 32; ++v) {
      const float dyv = s_d[warp][v][kMaxK];   // the same for all lanes: no divergence
      if (dyv == kTfSkip) continue;
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        if (lane + 32 * j >= G) continue;
        if (dyv == kTfZeroY) {
          sf[j] += static_cast<double>(-logf(FLT_MIN));
          continue;
        }
        float s1 = 0.f, t = 0.f;
#pragma unroll
        for (int c = 0; c < kMaxK; ++c)
          if (c < K) {
            const float dc = s_d[warp][v][c];
            const float e = expf(beta[j] * dc);   // dc = -inf: e = 0
            s1 += e;
            if (e > 0.f) t = fmaf(e, dc, t);
          }
        sf[j] += fma(static_cast<double>(beta[j]), static_cast<double>(dyv), static_cast<double>(log1pf(s1)));
        sd[j] += static_cast<double>(dyv) + static_cast<double>(t / (1.f + s1));
      }
    }
    __syncwarp();   // the tile is read before the next one is staged
  }
#pragma unroll
  for (int j = 0; j < 2; ++j)
    if (lane + 32 * j < G) {
      s_part[warp][lane + 32 * j] = sf[j];
      s_part[warp][G + lane + 32 * j] = sd[j];
    }
  for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
  if (lane == 0) s_cnt[warp] = cnt;
  __syncthreads();
  double* out = partial + static_cast<long long>(blockIdx.x) * (2 * G + 1);
  for (int i = threadIdx.x; i < 2 * G; i += blockDim.x) {
    double s = 0.0;
    for (int wv = 0; wv < kWarps; ++wv) s += s_part[wv][i];
    out[i] = s;
  }
  if (threadIdx.x == 0) {
    unsigned long long c = 0;
    for (int wv = 0; wv < kWarps; ++wv) c += s_cnt[wv];
    reinterpret_cast<unsigned long long*>(out)[2 * G] = c;
  }
}

// sums[i] += the blocks' partial[b][i] added in block order (i < 2G); counted += the blocks' counts
__global__ void prob_temp_fit_reduce_kernel(const double* __restrict__ partial, int blocks, int G,
                                            double* __restrict__ sums, unsigned long long* __restrict__ counted) {
  const int i = threadIdx.x, stride = 2 * G + 1;
  if (i < 2 * G) {
    double s = 0.0;
    for (int b = 0; b < blocks; ++b) s += partial[static_cast<long long>(b) * stride + i];
    sums[i] += s;
  } else if (i == 2 * G) {
    unsigned long long c = 0;
    for (int b = 0; b < blocks; ++b) c += reinterpret_cast<const unsigned long long*>(partial)[static_cast<long long>(b) * stride + i];
    *counted += c;
  }
}

// ---------------------------------------------------------------------------------------------
// Adam (torch.optim.Adam semantics, no weight decay / amsgrad)
// ---------------------------------------------------------------------------------------------
__global__ void adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                            float* __restrict__ v, long long n, float lr, float b1, float b2, float eps, float bc1,
                            float bc2_sqrt, float gscale) {
  for (long long i = blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const float gi = g[i] * gscale;
    const float mi = b1 * m[i] + (1.f - b1) * gi;
    const float vi = b2 * v[i] + (1.f - b2) * gi * gi;
    m[i] = mi;
    v[i] = vi;
    const float denom = sqrtf(vi) / bc2_sqrt + eps;
    p[i] -= (lr / bc1) * (mi / denom);
  }
}

int grid_for(long long work_items, int block, int per_sm) {
  long long b = (work_items + block - 1) / block;
  const long long cap = static_cast<long long>(num_sms()) * per_sm;
  if (b > cap) b = cap;
  if (b < 1) b = 1;
  return static_cast<int>(b);
}

int upload_head(const float* w, const float* b, int K, int cin, cudaStream_t st) {
  if (cin != kHeadC || K <= 0 || K > kMaxK) {
    set_error("head: needs cin == %d and 0 < classes <= %d (got %d, %d)", kHeadC, kMaxK, cin, K);
    return SPFF_ERR_BAD_ARGUMENT;
  }
  SPFF_CUDA(cudaMemcpyToSymbolAsync(c_head_w, w, sizeof(float) * K * kHeadC, 0, cudaMemcpyDeviceToDevice, st));
  if (b)
    SPFF_CUDA(cudaMemcpyToSymbolAsync(c_head_b, b, sizeof(float) * K, 0, cudaMemcpyDeviceToDevice, st));
  return 0;
}

constexpr int kHeadBwdBlocksPerSm = 2;

}  // namespace
}  // namespace spff

#define SPFF_ENTRY_CHECK()        \
  do {                            \
    int _e = spff_device_check(); \
    if (_e) return _e;            \
  } while (0)

typedef __nv_bfloat16 bf16;

namespace {

template <typename LabelT>
int head_eval_hist_attr() {   // once per device: the [K][2][T] histogram may exceed the 48 KB default (128 KB at most)
  static bool attr_set[spff::kMaxDevices] = {};
  const int dev = spff::current_device();
  if (!attr_set[dev]) {
    SPFF_CUDA(cudaFuncSetAttribute(spff::head_eval_mma_kernel<LabelT, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   static_cast<int>(sizeof(unsigned int) * spff::kMaxK * 2 * spff::kHeMaxBins)));
    attr_set[dev] = true;
  }
  return 0;
}

// spff_head_eval and spff_head_eval_hist: bins = 0 and hist = NULL select the kernel without the histogram
int head_eval_launch(const char* name, const void* x, long long ldx, int cin, const float* w, const float* b,
                     const void* labels, int label_bytes, int ignore_index, int k, spff_shape s, double* acc,
                     long long* counts, long long* confusion, double* sample_acc, long long* sample_counts,
                     long long* sample_confusion, uint8_t* labels_out, int bins, long long* hist, long long* sample_hist,
                     void* stream) {
  SPFF_REQUIRE(x && w && b && labels && acc && counts && confusion, "%s: null pointer", name);
  SPFF_REQUIRE((sample_acc != nullptr) == (sample_counts != nullptr) && (sample_acc != nullptr) == (sample_confusion != nullptr),
               "%s: the per-sample arrays are given together or not at all", name);
  SPFF_REQUIRE(label_bytes == 1 || label_bytes == 8, "%s: labels must be uint8 or int64", name);
  SPFF_REQUIRE(ldx >= cin && ldx % 8 == 0, "%s: bad channel pitch", name);
  SPFF_REQUIRE(s.n > 0 && s.n <= 65535 && s.d > 0 && s.h > 0 && s.w > 0, "%s: bad shape", name);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int e = spff::upload_head(w, b, k, cin, st);
  if (e) return e;
  const long long dhw = static_cast<long long>(s.d) * s.h * s.w;
  // blocks never straddle samples (grid.y = sample); grid.x spreads a sample over enough blocks for ~4 waves of
  // kHeBlocksPerSm resident blocks per SM, and no more blocks than the sample has warp tiles for
  const long long warp_tiles = ((dhw + 15) / 16 + spff::kHmWarps - 1) / spff::kHmWarps;
  long long per = (4LL * spff::kHeBlocksPerSm * spff::num_sms() + s.n - 1) / s.n;
  if (per > warp_tiles) per = warp_tiles;
  if (per < 1) per = 1;
  const dim3 grid(static_cast<unsigned>(per), s.n);
  auto cnt = reinterpret_cast<unsigned long long*>(counts);
  auto conf = reinterpret_cast<unsigned long long*>(confusion);
  auto scnt = reinterpret_cast<unsigned long long*>(sample_counts);
  auto sconf = reinterpret_cast<unsigned long long*>(sample_confusion);
  auto hst = reinterpret_cast<unsigned long long*>(hist);
  auto shst = reinterpret_cast<unsigned long long*>(sample_hist);
  const size_t hist_smem = sizeof(unsigned int) * k * 2 * bins;
  if (hist) {
    e = label_bytes == 1 ? head_eval_hist_attr<uint8_t>() : head_eval_hist_attr<long long>();
    if (e) return e;
  }
  if (label_bytes == 1 && !hist)
    spff::head_eval_mma_kernel<uint8_t, false><<<grid, spff::kHmWarps * 32, 0, st>>>(
        static_cast<const bf16*>(x), ldx, labels, ignore_index, k, dhw, acc, cnt, conf, sample_acc, scnt, sconf, labels_out,
        0, nullptr, nullptr);
  else if (!hist)
    spff::head_eval_mma_kernel<long long, false><<<grid, spff::kHmWarps * 32, 0, st>>>(
        static_cast<const bf16*>(x), ldx, labels, ignore_index, k, dhw, acc, cnt, conf, sample_acc, scnt, sconf, labels_out,
        0, nullptr, nullptr);
  else if (label_bytes == 1)
    spff::head_eval_mma_kernel<uint8_t, true><<<grid, spff::kHmWarps * 32, hist_smem, st>>>(
        static_cast<const bf16*>(x), ldx, labels, ignore_index, k, dhw, acc, cnt, conf, sample_acc, scnt, sconf, labels_out,
        bins, hst, shst);
  else
    spff::head_eval_mma_kernel<long long, true><<<grid, spff::kHmWarps * 32, hist_smem, st>>>(
        static_cast<const bf16*>(x), ldx, labels, ignore_index, k, dhw, acc, cnt, conf, sample_acc, scnt, sconf, labels_out,
        bins, hst, shst);
  SPFF_CUDA(cudaGetLastError());
  return 0;
}

template <typename LabelT, bool TEMP>
int prob_finalize_hist_attr() {   // once per device, as head_eval_hist_attr
  static bool attr_set[spff::kMaxDevices] = {};
  const int dev = spff::current_device();
  if (!attr_set[dev]) {
    SPFF_CUDA(cudaFuncSetAttribute(spff::prob_finalize_kernel<LabelT, true, false, TEMP>,
                                   cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   static_cast<int>(sizeof(unsigned int) * spff::kMaxK * 2 * spff::kHeMaxBins)));
    attr_set[dev] = true;
  }
  return 0;
}

// spff_head_prob_accum (with_ent = false) and spff_head_prob_accum_ent (with_ent = true, ent required)
int head_prob_accum_launch(const char* name, bool with_ent, const void* x, long long ldx, int cin, const float* w,
                           const float* b, int k, spff_shape s, int flip, int beta, float* acc, float* ent, void* stream) {
  SPFF_REQUIRE(x && w && b && acc && (ent || !with_ent), "%s: null pointer", name);
  SPFF_REQUIRE(k >= 2 && k <= spff::kMaxK, "%s: classes must be in [2, %d] (got %d)", name, spff::kMaxK, k);
  SPFF_REQUIRE(flip >= 0 && flip <= 3, "%s: flip is a bit set of 1 (H) and 2 (W) (got %d)", name, flip);
  SPFF_REQUIRE(beta == 0 || beta == 1, "%s: beta must be 0 or 1 (got %d)", name, beta);
  SPFF_REQUIRE((reinterpret_cast<uintptr_t>(acc) & 15) == 0, "%s: acc must be 16-byte aligned", name);
  SPFF_REQUIRE(!with_ent || (reinterpret_cast<uintptr_t>(ent) & 3) == 0, "%s: ent must be 4-byte aligned", name);
  SPFF_REQUIRE(ldx >= cin && ldx % 8 == 0, "%s: bad channel pitch", name);
  SPFF_REQUIRE(s.n > 0 && s.n <= 65535 && s.d > 0 && s.h > 0 && s.w > 0, "%s: bad shape (N must be <= 65535)", name);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int e = spff::upload_head(w, b, k, cin, st);
  if (e) return e;
  const long long dhw = static_cast<long long>(s.d) * s.h * s.w;
  // the grid of head_eval: one block row per sample, ~4 waves of resident blocks, no more blocks than warp tiles
  const long long warp_tiles = ((dhw + 15) / 16 + spff::kHmWarps - 1) / spff::kHmWarps;
  long long per = (4LL * spff::kPaBlocksPerSm * spff::num_sms() + s.n - 1) / s.n;
  if (per > warp_tiles) per = warp_tiles;
  if (per < 1) per = 1;
  const dim3 grid(static_cast<unsigned>(per), s.n);
  if (with_ent)
    spff::head_prob_accum_kernel<true><<<grid, spff::kHmWarps * 32, 0, st>>>(static_cast<const bf16*>(x), ldx, k, s.h, s.w,
                                                                            dhw, flip, beta, acc, ent);
  else
    spff::head_prob_accum_kernel<false><<<grid, spff::kHmWarps * 32, 0, st>>>(static_cast<const bf16*>(x), ldx, k, s.h, s.w,
                                                                             dhw, flip, beta, acc, nullptr);
  SPFF_CUDA(cudaGetLastError());
  return 0;
}

constexpr int kUncMinBins = 2, kUncMaxBins = 1024;

// dynamic shared memory of prob_finalize_kernel: the HIST histogram, then the UNC tallies (see the kernel)
size_t prob_finalize_smem(bool unc, int k, int bins, int cal_bins) {
  return sizeof(unsigned int) * k * 2 * bins +
         (unc ? sizeof(unsigned long long) * (2 + cal_bins) + sizeof(unsigned int) * 2 * cal_bins +
                    sizeof(float) * (spff::kPfThreads / 32)
              : 0);
}

template <typename LabelT, bool HIST, bool TEMP>
int prob_finalize_unc_attr() {   // once per device, as head_eval_hist_attr
  static bool attr_set[spff::kMaxDevices] = {};
  const int dev = spff::current_device();
  if (!attr_set[dev]) {
    SPFF_CUDA(cudaFuncSetAttribute(spff::prob_finalize_kernel<LabelT, HIST, true, TEMP>,
                                   cudaFuncAttributeMaxDynamicSharedMemorySize,
                                   static_cast<int>(prob_finalize_smem(true, spff::kMaxK, HIST ? spff::kHeMaxBins : 0,
                                                                       kUncMaxBins))));
    attr_set[dev] = true;
  }
  return 0;
}

template <typename LabelT, bool HIST, bool UNC, bool TEMP>
int prob_finalize_run(dim3 grid, size_t smem, cudaStream_t st, const float* acc, int k, long long dhw, float scale,
                      const void* labels, int ignore_index, double* nll, long long* counts, long long* confusion,
                      double* sample_acc, long long* sample_counts, long long* sample_confusion, uint8_t* labels_out,
                      int T, long long* hist, long long* sample_hist, void* proba_out, const spff_unc_out& u,
                      float inv_t) {
  if constexpr (HIST && !UNC) {
    const int e = prob_finalize_hist_attr<LabelT, TEMP>();
    if (e) return e;
  }
  if constexpr (UNC) {
    const int e = prob_finalize_unc_attr<LabelT, HIST, TEMP>();
    if (e) return e;
  }
  spff::prob_finalize_kernel<LabelT, HIST, UNC, TEMP><<<grid, spff::kPfThreads, smem, st>>>(
      acc, k, dhw, scale, labels, ignore_index, nll, reinterpret_cast<unsigned long long*>(counts),
      reinterpret_cast<unsigned long long*>(confusion), sample_acc, reinterpret_cast<unsigned long long*>(sample_counts),
      reinterpret_cast<unsigned long long*>(sample_confusion), labels_out, static_cast<__half*>(proba_out), T,
      reinterpret_cast<unsigned long long*>(hist), reinterpret_cast<unsigned long long*>(sample_hist), u, inv_t);
  SPFF_CUDA(cudaGetLastError());
  return 0;
}

// spff_prob_finalize (with_unc = false), spff_prob_finalize_unc (with_unc = true, unc required) and
// spff_prob_finalize_tempered (temp = true; with_unc = unc != NULL)
int prob_finalize_launch(const char* name, bool with_unc, const float* acc, int k, spff_shape s, float scale,
                         const void* labels, int label_bytes, int ignore_index, double* nll, long long* counts,
                         long long* confusion, double* sample_acc, long long* sample_counts, long long* sample_confusion,
                         uint8_t* labels_out, int bins, long long* hist, long long* sample_hist, void* proba_out,
                         const spff_unc_out* unc, void* stream, bool temp = false, float inv_t = 1.f) {
  SPFF_REQUIRE(acc, "%s: null accumulator", name);
  SPFF_REQUIRE(k >= 2 && k <= spff::kMaxK, "%s: classes must be in [2, %d] (got %d)", name, spff::kMaxK, k);
  SPFF_REQUIRE((reinterpret_cast<uintptr_t>(acc) & 15) == 0, "%s: acc must be 16-byte aligned", name);
  SPFF_REQUIRE(s.n > 0 && s.n <= 65535 && s.d > 0 && s.h > 0 && s.w > 0, "%s: bad shape (N must be <= 65535)", name);
  SPFF_REQUIRE(scale > 0.f, "%s: scale must be positive", name);
  SPFF_REQUIRE(!temp || (inv_t > 0.f && std::isfinite(inv_t)), "%s: inv_temperature must be positive and finite (got %g)",
               name, static_cast<double>(inv_t));
  SPFF_REQUIRE(!labels || label_bytes == 1 || label_bytes == 8, "%s: labels must be uint8 or int64", name);
  SPFF_REQUIRE(labels ? (nll && counts && confusion) : !(nll || counts || confusion || sample_acc || hist),
               "%s: the tally (nll, counts, confusion) is given exactly when the labels are", name);
  SPFF_REQUIRE((sample_acc != nullptr) == (sample_counts != nullptr) && (sample_acc != nullptr) == (sample_confusion != nullptr),
               "%s: the per-sample arrays are given together or not at all", name);
  SPFF_REQUIRE(!hist || (bins >= spff::kHeMinBins && bins <= spff::kHeMaxBins),
               "%s: bins must be in [%d, %d] (got %d)", name, spff::kHeMinBins, spff::kHeMaxBins, bins);
  SPFF_REQUIRE(hist || !sample_hist, "%s: sample_hist needs hist", name);
  SPFF_REQUIRE(!hist || (sample_hist != nullptr) == (sample_acc != nullptr),
               "%s: the per-sample histogram is given exactly when the per-sample tallies are", name);
  spff_unc_out u = {};
  if (with_unc) {
    SPFF_REQUIRE(unc, "%s: null output struct", name);
    u = *unc;
    SPFF_REQUIRE(!u.calib || (u.cal_bins >= kUncMinBins && u.cal_bins <= kUncMaxBins),
                 "%s: cal_bins must be in [%d, %d] (got %d)", name, kUncMinBins, kUncMaxBins, u.cal_bins);
    SPFF_REQUIRE(!u.calib || labels, "%s: calib needs labels", name);
    SPFF_REQUIRE(!u.sample_calib || (u.calib && sample_acc), "%s: sample_calib needs calib and the per-sample tallies",
                 name);
    SPFF_REQUIRE(!(u.calib && sample_acc) || u.sample_calib,
                 "%s: with calib, sample_calib is given exactly when the per-sample tallies are", name);
    SPFF_REQUIRE((u.brier != nullptr) == (u.calib != nullptr), "%s: brier is given exactly when calib is", name);
    SPFF_REQUIRE((u.sample_brier != nullptr) == (u.sample_calib != nullptr),
                 "%s: sample_brier is given exactly when sample_calib is", name);
    SPFF_REQUIRE(!u.mi_out || u.ent, "%s: mi_out needs ent", name);
    SPFF_REQUIRE(!u.sample_unc || u.unc, "%s: sample_unc needs unc", name);
    SPFF_REQUIRE((reinterpret_cast<uintptr_t>(u.ent) & 3) == 0, "%s: ent must be 4-byte aligned", name);
    if (!u.calib) u.cal_bins = 0;
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const long long dhw = static_cast<long long>(s.d) * s.h * s.w;
  const long long blocks_needed = (dhw + spff::kPfThreads - 1) / spff::kPfThreads;
  long long per = (16LL * spff::num_sms() + s.n - 1) / s.n;   // ~2 waves of 8 resident blocks per SM
  if (per > blocks_needed) per = blocks_needed;
  if (per < 1) per = 1;
  const dim3 grid(static_cast<unsigned>(per), s.n);
  const int T = hist ? bins : 0;
  const size_t smem = prob_finalize_smem(with_unc, k, T, u.cal_bins);
  const bool wide = label_bytes == 8;
#define SPFF_PF_RUN(L, H, U)                                                                                              \
  prob_finalize_run<L, H, U, false>(grid, smem, st, acc, k, dhw, scale, labels, ignore_index, nll, counts, confusion,     \
                                    sample_acc, sample_counts, sample_confusion, labels_out, T, hist, sample_hist,         \
                                    proba_out, u, 1.f)
#define SPFF_PF_RUN_T(L, H, U)                                                                                            \
  prob_finalize_run<L, H, U, true>(grid, smem, st, acc, k, dhw, scale, labels, ignore_index, nll, counts, confusion,      \
                                   sample_acc, sample_counts, sample_confusion, labels_out, T, hist, sample_hist,          \
                                   proba_out, u, inv_t)
  if (temp) {
    if (!with_unc) {
      if (!hist) return wide ? SPFF_PF_RUN_T(long long, false, false) : SPFF_PF_RUN_T(uint8_t, false, false);
      return wide ? SPFF_PF_RUN_T(long long, true, false) : SPFF_PF_RUN_T(uint8_t, true, false);
    }
    if (!hist) return wide ? SPFF_PF_RUN_T(long long, false, true) : SPFF_PF_RUN_T(uint8_t, false, true);
    return wide ? SPFF_PF_RUN_T(long long, true, true) : SPFF_PF_RUN_T(uint8_t, true, true);
  }
  if (!with_unc) {
    if (!hist) return wide ? SPFF_PF_RUN(long long, false, false) : SPFF_PF_RUN(uint8_t, false, false);
    return wide ? SPFF_PF_RUN(long long, true, false) : SPFF_PF_RUN(uint8_t, true, false);
  }
  if (!hist) return wide ? SPFF_PF_RUN(long long, false, true) : SPFF_PF_RUN(uint8_t, false, true);
  return wide ? SPFF_PF_RUN(long long, true, true) : SPFF_PF_RUN(uint8_t, true, true);
#undef SPFF_PF_RUN
#undef SPFF_PF_RUN_T
}

// blocks of prob_temp_fit_kernel (and rows of its workspace): ~one wave of kTfBlocksPerSm resident blocks per SM, no
// more than the warp tiles need
long long prob_temp_fit_blocks(spff_shape s) {
  const long long total = static_cast<long long>(s.n) * s.d * s.h * s.w;
  const long long tiles = (total + 31) / 32;
  long long blocks = (tiles + spff::kTfThreads / 32 - 1) / (spff::kTfThreads / 32);
  const long long cap = static_cast<long long>(spff::num_sms()) * spff::kTfBlocksPerSm;
  if (blocks > cap) blocks = cap;
  return blocks < 1 ? 1 : blocks;
}

bool prob_temp_fit_shape_ok(int k, spff_shape s, int g) {
  return k >= 2 && k <= spff::kMaxK && g >= 1 && g <= spff::kTfMaxG && s.n > 0 && s.n <= 65535 && s.d > 0 && s.h > 0 &&
         s.w > 0;
}

}  // namespace

extern "C" {

int spff_conv3d_stem_fwd(const float* x, const float* w, void* y, long long ldy, int cout, spff_shape s,
                         void* stream) {
  SPFF_ENTRY_CHECK();
  SPFF_REQUIRE(x && w && y && cout % 8 == 0 && cout > 0 && cout <= 256, "conv3d_stem_fwd: bad arguments (cout %d)", cout);
  const long long total = static_cast<long long>(s.n) * s.d * s.h * s.w * (cout / 8);
  const int grid = spff::grid_for(total, 256, 16);
  spff::stem_fwd_kernel<<<grid, 256, 27 * cout * sizeof(float), static_cast<cudaStream_t>(stream)>>>(
      x, w, static_cast<bf16*>(y), ldy, cout, s);
  SPFF_CUDA(cudaGetLastError());
  return 0;
}

int spff_conv3d_stem_stat_slots(spff_shape s) {
  if (s.n <= 0 || s.d <= 0 || s.h <= 0 || s.w <= 0) return 0;
  // ~16 blocks per SM over the whole launch, at least 4 items per thread
  const long long per_sample = static_cast<long long>(s.d) * s.h * ((s.w + spff::kStrip - 1) / spff::kStrip) * 4;
  long long slots = (16LL * spff::num_sms() + s.n - 1) / s.n;
  const long long cap = (per_sample + 4 * 256 - 1) / (4 * 256);
  if (slots > cap) slots = cap;
  if (slots < 1) slots = 1;
  return static_cast<int>(slots);
}

int spff_conv3d_stem_fwd_stats(const float* x, const float* w, void* y, long long ldy, int cout, spff_shape s,
                               float* stat_partial, void* stream) {
  SPFF_ENTRY_CHECK();
  SPFF_REQUIRE(x && w && y && stat_partial, "conv3d_stem_fwd_stats: null pointer");
  SPFF_REQUIRE(cout == 32, "conv3d_stem_fwd_stats: cout must be 32 (got %d)", cout);
  SPFF_REQUIRE(s.n > 0 && s.n <= 65535 && s.d > 0 && s.h > 0 && s.w > 0, "conv3d_stem_fwd_stats: bad shape");
  dim3 grid(spff_conv3d_stem_stat_slots(s), s.n);
  if (spff::debug_flag(8) == 0) {   // tensor-core kernel (default); spff_debug_set(8, 1) selects the fp32 FMA kernel
    static bool attr_set[spff::kMaxDevices] = {};
    const int dev = spff::current_device();
    if (!attr_set[dev]) {
      SPFF_CUDA(cudaFuncSetAttribute(spff::stem_fwd_stats_mma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     spff::kSfSmemBytes));
      attr_set[dev] = true;
    }
    spff::stem_fwd_stats_mma_kernel<<<grid, spff::kSfWarps * 32, spff::kSfSmemBytes, static_cast<cudaStream_t>(stream)>>>(
        x, w, static_cast<bf16*>(y), ldy, s, stat_partial);
    SPFF_CUDA(cudaGetLastError());
    return 0;
  }
  const size_t smem = (27 + 16) * cout * sizeof(float);
  spff::stem_fwd_stats_kernel<<<grid, 256, smem, static_cast<cudaStream_t>(stream)>>>(x, w, static_cast<bf16*>(y), ldy, cout, s,
                                                                                     stat_partial);
  SPFF_CUDA(cudaGetLastError());
  return 0;
}

size_t spff_conv3d_stem_wgrad_workspace(int cout) {
  return static_cast<size_t>(spff::num_sms()) * spff::kSwgBlocksPerSm * 27 * cout * sizeof(float);
}

int spff_conv3d_stem_wgrad(const float* x, const void* dy, long long lddy, int cout, spff_shape s, float* dw,
                           float beta, void* workspace, size_t workspace_bytes, void* stream) {
  SPFF_ENTRY_CHECK();
  SPFF_REQUIRE(x && dy && dw && workspace, "conv3d_stem_wgrad: null pointer");
  SPFF_REQUIRE(cout == spff::kStemCo, "conv3d_stem_wgrad: cout must be %d (got %d)", spff::kStemCo, cout);
  if (workspace_bytes < spff_conv3d_stem_wgrad_workspace(cout)) {
    spff::set_error("conv3d_stem_wgrad: workspace too small");
    return SPFF_ERR_WORKSPACE;
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int blocks = spff::num_sms() * spff::kSwgBlocksPerSm;
  SPFF_REQUIRE(lddy % 8 == 0 && (reinterpret_cast<uintptr_t>(dy) & 15) == 0, "conv3d_stem_wgrad: dy must be 16-byte aligned");
  spff::stem_wgrad_mma_kernel<<<blocks, spff::kSwgWarps * 32, 0, st>>>(x, static_cast<const bf16*>(dy), lddy, s,
                                                                      static_cast<float*>(workspace));
  spff::stem_wgrad_reduce_kernel<<<(27 * cout + 127) / 128, 128, 0, st>>>(static_cast<const float*>(workspace), blocks,
                                                                         cout, beta, dw);
  SPFF_CUDA(cudaGetLastError());
  return 0;
}

int spff_head_fwd(const void* x, long long ldx, int cin, const float* w, const float* b, float* logits, int k,
                  spff_shape s, void* stream) {
  SPFF_ENTRY_CHECK();
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int e = spff::upload_head(w, b, k, cin, st);
  if (e) return e;
  const long long total = static_cast<long long>(s.n) * s.d * s.h * s.w;
  spff::head_fwd_kernel<false><<<spff::grid_for(total, 256, 8), 256, 0, st>>>(
      static_cast<const bf16*>(x), ldx, logits, nullptr, k, static_cast<long long>(s.d) * s.h * s.w, total);
  SPFF_CUDA(cudaGetLastError());
  return 0;
}

int spff_head_argmax(const void* x, long long ldx, int cin, const float* w, const float* b, uint8_t* labels, int k,
                     spff_shape s, void* stream) {
  SPFF_ENTRY_CHECK();
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int e = spff::upload_head(w, b, k, cin, st);
  if (e) return e;
  const long long total = static_cast<long long>(s.n) * s.d * s.h * s.w;
  spff::head_fwd_kernel<true><<<spff::grid_for(total, 256, 8), 256, 0, st>>>(
      static_cast<const bf16*>(x), ldx, nullptr, labels, k, static_cast<long long>(s.d) * s.h * s.w, total);
  SPFF_CUDA(cudaGetLastError());
  return 0;
}

size_t spff_head_bwd_workspace(int k) {
  return static_cast<size_t>(spff::num_sms()) * spff::kHeadBwdBlocksPerSm * (k * spff::kHeadC + k) * sizeof(float);
}

int spff_head_bwd(const float* dlogits, const void* x, long long ldx, int cin, const float* w, void* dx,
                  long long lddx, float* dw, float* db, float beta, int k, spff_shape s, void* workspace,
                  size_t workspace_bytes, void* stream) {
  SPFF_ENTRY_CHECK();
  SPFF_REQUIRE(dlogits && x && w && dw && db && workspace, "head_bwd: null pointer");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int e = spff::upload_head(w, nullptr, k, cin, st);
  if (e) return e;
  if (workspace_bytes < spff_head_bwd_workspace(k)) {
    spff::set_error("head_bwd: workspace too small");
    return SPFF_ERR_WORKSPACE;
  }
  const long long total = static_cast<long long>(s.n) * s.d * s.h * s.w;
  const int blocks = spff::num_sms() * spff::kHeadBwdBlocksPerSm;
  const size_t smem = 8 * (spff::kMaxK * spff::kHeadC + spff::kMaxK) * sizeof(float);
  spff::head_bwd_kernel<<<blocks, 256, smem, st>>>(dlogits, static_cast<const bf16*>(x), ldx, static_cast<bf16*>(dx),
                                                  lddx, k, static_cast<long long>(s.d) * s.h * s.w, total,
                                                  static_cast<float*>(workspace));
  const int tot = k * spff::kHeadC + k;
  spff::head_bwd_reduce_kernel<<<(tot + 127) / 128, 128, 0, st>>>(static_cast<const float*>(workspace), blocks, k, beta,
                                                                 dw, db);
  SPFF_CUDA(cudaGetLastError());
  return 0;
}

int spff_ce_confusion(const float* logits, const void* labels, int label_bytes, int ignore_index, int k,
                      spff_shape s, double* acc, long long* counts, long long* confusion, void* stream) {
  SPFF_ENTRY_CHECK();
  SPFF_REQUIRE(logits && labels && acc && counts && confusion, "ce_confusion: null pointer");
  SPFF_REQUIRE(k > 0 && k <= spff::kMaxK, "ce_confusion: classes must be in 1..%d", spff::kMaxK);
  SPFF_REQUIRE(label_bytes == 1 || label_bytes == 8, "ce_confusion: labels must be uint8 or int64");
  const long long total = static_cast<long long>(s.n) * s.d * s.h * s.w;
  const long long dhw = static_cast<long long>(s.d) * s.h * s.w;
  const int grid = spff::grid_for(total, 256, 8);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  auto cnt = reinterpret_cast<unsigned long long*>(counts);
  auto conf = reinterpret_cast<unsigned long long*>(confusion);
  if (label_bytes == 1)
    spff::ce_kernel<uint8_t, false><<<grid, 256, 0, st>>>(logits, labels, ignore_index, k, dhw, total, acc, cnt, conf,
                                                          nullptr, nullptr, nullptr);
  else
    spff::ce_kernel<long long, false><<<grid, 256, 0, st>>>(logits, labels, ignore_index, k, dhw, total, acc, cnt, conf,
                                                            nullptr, nullptr, nullptr);
  SPFF_CUDA(cudaGetLastError());
  return 0;
}

int spff_ce_grad(const float* logits, const void* labels, int label_bytes, int ignore_index, int k, spff_shape s,
                 const long long* n_valid, const float* gscale, float* dlogits, void* stream) {
  SPFF_ENTRY_CHECK();
  SPFF_REQUIRE(logits && labels && n_valid && dlogits, "ce_grad: null pointer");
  SPFF_REQUIRE(k > 0 && k <= spff::kMaxK, "ce_grad: classes must be in 1..%d", spff::kMaxK);
  SPFF_REQUIRE(label_bytes == 1 || label_bytes == 8, "ce_grad: labels must be uint8 or int64");
  const long long total = static_cast<long long>(s.n) * s.d * s.h * s.w;
  const long long dhw = static_cast<long long>(s.d) * s.h * s.w;
  const int grid = spff::grid_for(total, 256, 8);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  auto nv = reinterpret_cast<const unsigned long long*>(n_valid);
  if (label_bytes == 1)
    spff::ce_kernel<uint8_t, true><<<grid, 256, 0, st>>>(logits, labels, ignore_index, k, dhw, total, nullptr, nullptr,
                                                         nullptr, nv, gscale, dlogits);
  else
    spff::ce_kernel<long long, true><<<grid, 256, 0, st>>>(logits, labels, ignore_index, k, dhw, total, nullptr,
                                                           nullptr, nullptr, nv, gscale, dlogits);
  SPFF_CUDA(cudaGetLastError());
  return 0;
}

size_t spff_head_loss_workspace(int k) {
  return static_cast<size_t>(spff::num_sms()) * spff::kHeadLossBlocksPerSm * (k * spff::kHeadC + k) * sizeof(float);
}

int spff_head_loss_fused(const void* x, long long ldx, int cin, const float* w, const float* b, const void* labels,
                         int label_bytes, int ignore_index, int k, spff_shape s, const long long* n_valid,
                         const float* gscale, double* acc, long long* counts, long long* confusion, void* dx,
                         long long lddx, float* dw, float* db, float beta, void* workspace, size_t workspace_bytes,
                         void* stream) {
  SPFF_ENTRY_CHECK();
  SPFF_REQUIRE(x && w && b && labels && n_valid && acc && counts && confusion && dw && db && workspace,
               "head_loss_fused: null pointer");
  SPFF_REQUIRE(label_bytes == 1 || label_bytes == 8, "head_loss_fused: labels must be uint8 or int64");
  SPFF_REQUIRE(ldx >= cin && ldx % 8 == 0 && (!dx || (lddx >= cin && lddx % 8 == 0)), "head_loss_fused: bad channel pitch");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int e = spff::upload_head(w, b, k, cin, st);
  if (e) return e;
  if (workspace_bytes < spff_head_loss_workspace(k)) {
    spff::set_error("head_loss_fused: workspace too small");
    return SPFF_ERR_WORKSPACE;
  }
  const long long total = static_cast<long long>(s.n) * s.d * s.h * s.w;
  const int blocks = spff::num_sms() * spff::kHeadLossBlocksPerSm;
  auto nv = reinterpret_cast<const unsigned long long*>(n_valid);
  auto cnt = reinterpret_cast<unsigned long long*>(counts);
  auto conf = reinterpret_cast<unsigned long long*>(confusion);
  if (spff::debug_flag(2) == 0) {   // tensor-core path (default); spff_debug_set(2, 1) selects the CUDA-core kernel
    static_assert(spff::kHmBlocksPerSm == spff::kHeadLossBlocksPerSm, "the two kernels share the partial workspace");
    if (label_bytes == 1)
      spff::head_loss_mma_kernel<uint8_t><<<blocks, spff::kHmWarps * 32, 0, st>>>(
          static_cast<const bf16*>(x), ldx, labels, ignore_index, k, total, nv, gscale, acc, cnt, conf,
          static_cast<bf16*>(dx), lddx, static_cast<float*>(workspace));
    else
      spff::head_loss_mma_kernel<long long><<<blocks, spff::kHmWarps * 32, 0, st>>>(
          static_cast<const bf16*>(x), ldx, labels, ignore_index, k, total, nv, gscale, acc, cnt, conf,
          static_cast<bf16*>(dx), lddx, static_cast<float*>(workspace));
  } else if (label_bytes == 1)
    spff::head_loss_kernel<uint8_t><<<blocks, spff::kHeadLossWarps * 32, 0, st>>>(
        static_cast<const bf16*>(x), ldx, labels, ignore_index, k, total, nv, gscale, acc, cnt, conf,
        static_cast<bf16*>(dx), lddx, static_cast<float*>(workspace));
  else
    spff::head_loss_kernel<long long><<<blocks, spff::kHeadLossWarps * 32, 0, st>>>(
        static_cast<const bf16*>(x), ldx, labels, ignore_index, k, total, nv, gscale, acc, cnt, conf,
        static_cast<bf16*>(dx), lddx, static_cast<float*>(workspace));
  const int tot = k * spff::kHeadC + k;
  spff::head_bwd_reduce_kernel<<<(tot + 127) / 128, 128, 0, st>>>(static_cast<const float*>(workspace), blocks, k, beta,
                                                                 dw, db);
  SPFF_CUDA(cudaGetLastError());
  return 0;
}

int spff_head_eval(const void* x, long long ldx, int cin, const float* w, const float* b, const void* labels,
                   int label_bytes, int ignore_index, int k, spff_shape s, double* acc, long long* counts,
                   long long* confusion, double* sample_acc, long long* sample_counts, long long* sample_confusion,
                   uint8_t* labels_out, void* stream) {
  SPFF_ENTRY_CHECK();
  return head_eval_launch("head_eval", x, ldx, cin, w, b, labels, label_bytes, ignore_index, k, s, acc, counts, confusion,
                          sample_acc, sample_counts, sample_confusion, labels_out, 0, nullptr, nullptr, stream);
}

int spff_head_eval_hist(const void* x, long long ldx, int cin, const float* w, const float* b, const void* labels,
                        int label_bytes, int ignore_index, int k, spff_shape s, double* acc, long long* counts,
                        long long* confusion, double* sample_acc, long long* sample_counts, long long* sample_confusion,
                        uint8_t* labels_out, int bins, long long* hist, long long* sample_hist, void* stream) {
  SPFF_ENTRY_CHECK();
  SPFF_REQUIRE(bins >= spff::kHeMinBins && bins <= spff::kHeMaxBins, "head_eval_hist: bins must be in [%d, %d] (got %d)",
               spff::kHeMinBins, spff::kHeMaxBins, bins);
  SPFF_REQUIRE(hist, "head_eval_hist: null histogram");
  SPFF_REQUIRE((sample_hist != nullptr) == (sample_acc != nullptr),
               "head_eval_hist: the per-sample histogram is given exactly when the per-sample tallies are");
  return head_eval_launch("head_eval_hist", x, ldx, cin, w, b, labels, label_bytes, ignore_index, k, s, acc, counts,
                          confusion, sample_acc, sample_counts, sample_confusion, labels_out, bins, hist, sample_hist,
                          stream);
}

int spff_head_prob_accum(const void* x, long long ldx, int cin, const float* w, const float* b, int k, spff_shape s,
                         int flip, int beta, float* acc, void* stream) {
  SPFF_ENTRY_CHECK();
  return head_prob_accum_launch("head_prob_accum", false, x, ldx, cin, w, b, k, s, flip, beta, acc, nullptr, stream);
}

int spff_head_prob_accum_ent(const void* x, long long ldx, int cin, const float* w, const float* b, int k, spff_shape s,
                             int flip, int beta, float* acc, float* ent, void* stream) {
  SPFF_ENTRY_CHECK();
  return head_prob_accum_launch("head_prob_accum_ent", true, x, ldx, cin, w, b, k, s, flip, beta, acc, ent, stream);
}

int spff_prob_finalize(const float* acc, int k, spff_shape s, float scale, const void* labels, int label_bytes,
                       int ignore_index, double* nll, long long* counts, long long* confusion, double* sample_acc,
                       long long* sample_counts, long long* sample_confusion, uint8_t* labels_out, int bins,
                       long long* hist, long long* sample_hist, void* proba_out, void* stream) {
  SPFF_ENTRY_CHECK();
  return prob_finalize_launch("prob_finalize", false, acc, k, s, scale, labels, label_bytes, ignore_index, nll, counts,
                              confusion, sample_acc, sample_counts, sample_confusion, labels_out, bins, hist, sample_hist,
                              proba_out, nullptr, stream);
}

int spff_prob_finalize_unc(const float* acc, int k, spff_shape s, float scale, const void* labels, int label_bytes,
                           int ignore_index, double* nll, long long* counts, long long* confusion, double* sample_acc,
                           long long* sample_counts, long long* sample_confusion, uint8_t* labels_out, int bins,
                           long long* hist, long long* sample_hist, void* proba_out, const spff_unc_out* unc,
                           void* stream) {
  SPFF_ENTRY_CHECK();
  return prob_finalize_launch("prob_finalize_unc", true, acc, k, s, scale, labels, label_bytes, ignore_index, nll, counts,
                              confusion, sample_acc, sample_counts, sample_confusion, labels_out, bins, hist, sample_hist,
                              proba_out, unc, stream);
}

int spff_prob_finalize_tempered(const float* acc, int k, spff_shape s, float scale, const void* labels, int label_bytes,
                                int ignore_index, double* nll, long long* counts, long long* confusion,
                                double* sample_acc, long long* sample_counts, long long* sample_confusion,
                                uint8_t* labels_out, int bins, long long* hist, long long* sample_hist, void* proba_out,
                                const spff_unc_out* unc, float inv_temperature, void* stream) {
  SPFF_ENTRY_CHECK();
  return prob_finalize_launch("prob_finalize_tempered", unc != nullptr, acc, k, s, scale, labels, label_bytes,
                              ignore_index, nll, counts, confusion, sample_acc, sample_counts, sample_confusion,
                              labels_out, bins, hist, sample_hist, proba_out, unc, stream, true, inv_temperature);
}

size_t spff_prob_temp_fit_workspace(int k, spff_shape s, int g) {
  if (!prob_temp_fit_shape_ok(k, s, g)) return 0;
  return static_cast<size_t>(prob_temp_fit_blocks(s)) * (2 * g + 1) * sizeof(double);
}

int spff_prob_temp_fit(const float* acc, int k, spff_shape s, float scale, const void* labels, int label_bytes,
                       int ignore_index, const float* betas, int g, double* sums, long long* counted, void* workspace,
                       size_t workspace_bytes, void* stream) {
  SPFF_ENTRY_CHECK();
  SPFF_REQUIRE(acc && labels && betas && sums && counted && workspace, "prob_temp_fit: null pointer");
  SPFF_REQUIRE(k >= 2 && k <= spff::kMaxK, "prob_temp_fit: classes must be in [2, %d] (got %d)", spff::kMaxK, k);
  SPFF_REQUIRE(g >= 1 && g <= spff::kTfMaxG, "prob_temp_fit: grid points must be in [1, %d] (got %d)", spff::kTfMaxG, g);
  SPFF_REQUIRE((reinterpret_cast<uintptr_t>(acc) & 15) == 0, "prob_temp_fit: acc must be 16-byte aligned");
  SPFF_REQUIRE(s.n > 0 && s.n <= 65535 && s.d > 0 && s.h > 0 && s.w > 0, "prob_temp_fit: bad shape (N must be <= 65535)");
  SPFF_REQUIRE(scale > 0.f, "prob_temp_fit: scale must be positive");
  SPFF_REQUIRE(label_bytes == 1 || label_bytes == 8, "prob_temp_fit: labels must be uint8 or int64");
  if (workspace_bytes < spff_prob_temp_fit_workspace(k, s, g)) {
    spff::set_error("prob_temp_fit: workspace too small");
    return SPFF_ERR_WORKSPACE;
  }
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const long long total = static_cast<long long>(s.n) * s.d * s.h * s.w;
  const int blocks = static_cast<int>(prob_temp_fit_blocks(s));
  auto part = static_cast<double*>(workspace);
  if (label_bytes == 1)
    spff::prob_temp_fit_kernel<uint8_t><<<blocks, spff::kTfThreads, 0, st>>>(
        acc, k, total, scale, static_cast<const uint8_t*>(labels), ignore_index, betas, g, part);
  else
    spff::prob_temp_fit_kernel<long long><<<blocks, spff::kTfThreads, 0, st>>>(
        acc, k, total, scale, static_cast<const long long*>(labels), ignore_index, betas, g, part);
  spff::prob_temp_fit_reduce_kernel<<<1, 160, 0, st>>>(part, blocks, g, sums,
                                                       reinterpret_cast<unsigned long long*>(counted));
  SPFF_CUDA(cudaGetLastError());
  return 0;
}

int spff_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, long long n, float lr,
                   float beta1, float beta2, float eps, int step, float grad_scale, void* stream) {
  SPFF_ENTRY_CHECK();
  SPFF_REQUIRE(param && grad && exp_avg && exp_avg_sq && n >= 0 && step >= 1, "adam_step: bad arguments");
  if (n == 0) return 0;
  const float bc1 = 1.f - powf(beta1, static_cast<float>(step));
  const float bc2 = 1.f - powf(beta2, static_cast<float>(step));
  spff::adam_kernel<<<spff::grid_for(n, 256, 8), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      param, grad, exp_avg, exp_avg_sq, n, lr, beta1, beta2, eps, bc1, sqrtf(bc2), grad_scale);
  SPFF_CUDA(cudaGetLastError());
  return 0;
}

}  // extern "C"
