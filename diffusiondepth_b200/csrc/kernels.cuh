// Everything on the hot path that is not the tensor-core convolution: layout changes at the ABI
// boundary, the fp16 hi/lo split, GroupNorm finalize/apply (+ReLU, + condition injection), the collapsed
// DDIM update, the fused depth-latent decoder and an fp32 CUDA-core convolution used for validation.
// All activations are NHWC inside the engine.
#pragma once
#include <type_traits>

#include "conv_umma.cuh"

#include "ptx.cuh"

namespace dd {

__device__ __forceinline__ void split_f16(float v, float scale, __half& hi, __half& lo, bool& overflow) {
  const float s = v * scale;
  overflow |= (fabsf(s) > 60000.f);
  hi = __float2half_rn(s);
  lo = __float2half_rn(s - __half2float(hi));
}

// ------------------------------------------------------------------ NCHW <-> NHWC
// in [B][C][P] -> out [B][P][C]  (32x32 smem transpose; P = H*W)
__global__ void nchw_to_nhwc_kernel(const float* __restrict__ in, float* __restrict__ out, int C, int P) {
  __shared__ float t[32][33];
  const int b = blockIdx.z;
  const int p0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  const float* src = in + static_cast<size_t>(b) * C * P;
  float* dst = out + static_cast<size_t>(b) * C * P;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int c = c0 + i, pp = p0 + threadIdx.x;
    t[i][threadIdx.x] = (c < C && pp < P) ? src[static_cast<size_t>(c) * P + pp] : 0.f;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int pp = p0 + i, c = c0 + threadIdx.x;
    if (pp < P && c < C) dst[static_cast<size_t>(pp) * C + c] = t[threadIdx.x][i];
  }
}
__global__ void nhwc_to_nchw_kernel(const float* __restrict__ in, float* __restrict__ out, int C, int P) {
  __shared__ float t[32][33];
  const int b = blockIdx.z;
  const int p0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  const float* src = in + static_cast<size_t>(b) * C * P;
  float* dst = out + static_cast<size_t>(b) * C * P;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int pp = p0 + i, c = c0 + threadIdx.x;
    t[i][threadIdx.x] = (pp < P && c < C) ? src[static_cast<size_t>(pp) * C + c] : 0.f;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int c = c0 + i, pp = p0 + threadIdx.x;
    if (c < C && pp < P) dst[static_cast<size_t>(c) * P + pp] = t[threadIdx.x][i];
  }
}

// fp32 NHWC -> scaled fp16 hi/lo planes (n elements, vectorised by 4)
__global__ void split_planes_kernel(const float* __restrict__ x, __half* __restrict__ hi, __half* __restrict__ lo,
                                    size_t n4, float scale, int* status) {
  bool ov = false;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n4;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const float4 v = reinterpret_cast<const float4*>(x)[i];
    __align__(8) __half h[4];
    __align__(8) __half l[4];
    split_f16(v.x, scale, h[0], l[0], ov);
    split_f16(v.y, scale, h[1], l[1], ov);
    split_f16(v.z, scale, h[2], l[2], ov);
    split_f16(v.w, scale, h[3], l[3], ov);
    reinterpret_cast<uint2*>(hi)[i] = *reinterpret_cast<const uint2*>(h);
    reinterpret_cast<uint2*>(lo)[i] = *reinterpret_cast<const uint2*>(l);
  }
  if (ov) atomicOr(status, 1);
}

// fp32 NHWC -> fp16 hi plane + e4m3 a8 / l8 planes (standalone-layer path of the fp8-correction kernel)
__global__ void split_planes8_kernel(const float* __restrict__ x, __half* __restrict__ hi, uint8_t* __restrict__ a8,
                                     uint8_t* __restrict__ l8, size_t n8, float scale, int* status) {
  bool ov = false;
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n8;
       i += static_cast<size_t>(gridDim.x) * blockDim.x) {
    const float4 u0 = reinterpret_cast<const float4*>(x)[2 * i], u1 = reinterpret_cast<const float4*>(x)[2 * i + 1];
    const float v[8] = {u0.x, u0.y, u0.z, u0.w, u1.x, u1.y, u1.z, u1.w};
    __align__(16) __half h[8];
    __align__(8) uint16_t pa[4];
    __align__(8) uint16_t pl[4];
#pragma unroll
    for (int j = 0; j < 8; j += 2) {
      const float s0 = v[j] * scale, s1 = v[j + 1] * scale;
      ov |= (fabsf(s0) > kF8ActMax) | (fabsf(s1) > kF8ActMax);
      h[j] = __float2half_rn(s0);
      h[j + 1] = __float2half_rn(s1);
      pa[j >> 1] = e4m3x2(s0 * kF8ActDiv, s1 * kF8ActDiv);
      pl[j >> 1] = e4m3x2((s0 - __half2float(h[j])) * kF8LoMul, (s1 - __half2float(h[j + 1])) * kF8LoMul);
    }
    reinterpret_cast<uint4*>(hi)[i] = *reinterpret_cast<const uint4*>(h);
    reinterpret_cast<uint2*>(a8)[i] = *reinterpret_cast<const uint2*>(pa);
    reinterpret_cast<uint2*>(l8)[i] = *reinterpret_cast<const uint2*>(pl);
  }
  if (ov) atomicOr(status, 1);
}

// ------------------------------------------------------------------ weight pre-pack
// fp8-correction weight planes [tap][COUT][CIN] bytes: w8 = e4m3(t w / 512) (partner of the activation l8, scaled by
// 512), lw8 = e4m3((t w - fp16(t w)) * 4) (partner of a8, scaled by 1/4); t = the layer's fp16 weight scale
__global__ void pack_conv_weight8_kernel(const float* __restrict__ w, uint8_t* __restrict__ w8, uint8_t* __restrict__ lw8,
                                         int cout, int cin, float scale) {
  const int n = cout * cin * 9;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const int tap = i % 9, ci = (i / 9) % cin, co = i / (9 * cin);
    const float s = w[i] * scale;
    const float h = __half2float(__float2half_rn(s));
    const size_t o = (static_cast<size_t>(tap) * cout + co) * cin + ci;
    w8[o] = static_cast<uint8_t>(e4m3x2(s * (1.f / kF8LoMul), 0.f) & 0xff);
    lw8[o] = static_cast<uint8_t>(e4m3x2((s - h) * (1.f / kF8ActDiv), 0.f) & 0xff);
  }
}

// w [COUT][CIN][3][3] fp32 -> hi/lo fp16 [tap][COUT][CIN] (scaled) and fp32 [tap][CIN][COUT] (SIMT path)
__global__ void pack_conv_weight_kernel(const float* __restrict__ w, __half* __restrict__ hi, __half* __restrict__ lo,
                                        float* __restrict__ w_simt, int cout, int cin, float scale) {
  const int n = cout * cin * 9;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const int tap = i % 9, ci = (i / 9) % cin, co = i / (9 * cin);
    const float v = w[i];
    const float s = v * scale;
    const __half h = __float2half_rn(s);
    const size_t o = (static_cast<size_t>(tap) * cout + co) * cin + ci;
    hi[o] = h;
    lo[o] = __float2half_rn(s - __half2float(h));
    w_simt[(static_cast<size_t>(tap) * cin + ci) * cout + co] = v;
  }
}
// max |w| over n elements.  *out must be zeroed before the launch; any grid size: blocks combine through an integer
// atomicMax on the bit pattern (non-negative floats order like unsigned ints; NaN sorts above inf, so it still surfaces).
__global__ void absmax_kernel(const float* __restrict__ w, int n, float* __restrict__ out) {
  __shared__ float sm[256];
  float m = 0.f;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const float v = fabsf(w[i]);
    m = (v > m || v != v) ? v : m;
  }
  sm[threadIdx.x] = m;
  __syncthreads();
  for (int s = 128; s > 0; s >>= 1) {
    if (threadIdx.x < s) {
      const float o = sm[threadIdx.x + s];
      if (o > sm[threadIdx.x] || o != o) sm[threadIdx.x] = o;
    }
    __syncthreads();
  }
  if (threadIdx.x == 0) atomicMax(reinterpret_cast<unsigned int*>(out), __float_as_uint(sm[0]));
}

// ------------------------------------------------------------------ GroupNorm(4, C) finalize
// partial [tiles_total][4][2] (fp32 sums over one 128-pixel tile) -> mean/rstd per (image, group).
// Combined in fp64 in a fixed order (deterministic; SURVEY.md §7.2-4).
__global__ void gn_finalize_kernel(const float* __restrict__ partial, int tiles_per_img, double inv_count, float eps,
                                   float* __restrict__ mean_rstd /* [B][4][2] */) {
  const int b = blockIdx.x >> 2, g = blockIdx.x & 3;
  double s = 0.0, s2 = 0.0;
  for (int t = threadIdx.x; t < tiles_per_img; t += blockDim.x) {
    const float* q = partial + (static_cast<size_t>(b) * tiles_per_img + t) * 8 + g * 2;
    s += static_cast<double>(q[0]);
    s2 += static_cast<double>(q[1]);
  }
  __shared__ double sh[2][32];
  for (int o = 16; o > 0; o >>= 1) {
    s += __shfl_xor_sync(0xffffffffu, s, o);
    s2 += __shfl_xor_sync(0xffffffffu, s2, o);
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) {
    sh[0][warp] = s;
    sh[1][warp] = s2;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double a = 0.0, a2 = 0.0;
    for (int w = 0; w < static_cast<int>(blockDim.x >> 5); ++w) {
      a += sh[0][w];
      a2 += sh[1][w];
    }
    const double mean = a * inv_count;
    double var = a2 * inv_count - mean * mean;
    if (var < 0.0) var = 0.0;
    mean_rstd[(b * 4 + g) * 2 + 0] = static_cast<float>(mean);
    mean_rstd[(b * 4 + g) * 2 + 1] = static_cast<float>(1.0 / sqrt(var + static_cast<double>(eps)));
  }
}

// ------------------------------------------------------------------ GroupNorm apply + ReLU (+ condition) -> fp16 planes
// COND: 0 none, 1 add cond at the same resolution (Res head, reference ddim_depth_estimate_res.py:340),
//       2 add bilinear-upsampled cond, align_corners=True (Swin head UpSample_add, ..._swin_addHAHI.py:331-333);
// in both cases the per-image time-embedding row is added too (feat = cond + temb, head :367-372).
struct ApplyArgs {
  const float* y;          // [B][P][C]
  const float* mean_rstd;  // [B][4][2]
  const float* gamma;      // [C]
  const float* beta;       // [C]
  const float* cond;       // NHWC [B][ch][cw][C]
  const float* temb;       // [.. ][C], image b uses temb + b*temb_bstride
  int temb_bstride;
  int H, W, ch, cw;
  float ry, rx;            // (ch-1)/(H-1), (cw-1)/(W-1) in fp32 as ATen computes them
  __half* out_hi;
  __half* out_lo;
  uint8_t* out_a8;         // non-null: the consumer uses fp8 corrections -> write e4m3 planes a8 / l8 instead of fp16 lo
  uint8_t* out_l8;
  float scale;
  int* status;
};

// 8 consecutive channels of one pixel -> operand planes (fp16 hi + fp16 lo, or fp16 hi + e4m3 a8 + e4m3 l8)
__device__ __forceinline__ void store_planes8(const float (&v)[8], float scale, __half* out_hi, __half* out_lo,
                                              uint8_t* out_a8, uint8_t* out_l8, size_t off, bool& ov) {
  __align__(16) __half h[8];
  if (out_a8 != nullptr) {
    __align__(8) uint16_t a8[4];
    __align__(8) uint16_t l8[4];
#pragma unroll
    for (int j = 0; j < 8; j += 2) {
      const float s0 = v[j] * scale, s1 = v[j + 1] * scale;
      ov |= (fabsf(s0) > kF8ActMax) | (fabsf(s1) > kF8ActMax);
      h[j] = __float2half_rn(s0);
      h[j + 1] = __float2half_rn(s1);
      a8[j >> 1] = e4m3x2(s0 * kF8ActDiv, s1 * kF8ActDiv);
      l8[j >> 1] = e4m3x2((s0 - __half2float(h[j])) * kF8LoMul, (s1 - __half2float(h[j + 1])) * kF8LoMul);
    }
    *reinterpret_cast<uint4*>(out_hi + off) = *reinterpret_cast<const uint4*>(h);
    *reinterpret_cast<uint2*>(out_a8 + off) = *reinterpret_cast<const uint2*>(a8);
    *reinterpret_cast<uint2*>(out_l8 + off) = *reinterpret_cast<const uint2*>(l8);
  } else {
    __align__(16) __half l[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) split_f16(v[j], scale, h[j], l[j], ov);
    *reinterpret_cast<uint4*>(out_hi + off) = *reinterpret_cast<const uint4*>(h);
    *reinterpret_cast<uint4*>(out_lo + off) = *reinterpret_cast<const uint4*>(l);
  }
}

template <int C, int COND>
__global__ void __launch_bounds__(256) gn_apply_split_kernel(const ApplyArgs a) {
  constexpr int VEC = 8;             // channels per thread
  constexpr int TPP = C / VEC;       // threads per pixel
  constexpr int PPB = 256 / TPP;     // pixels per block
  __shared__ float sa[C], sb[C];
  const int b = blockIdx.y;
  const int P = a.H * a.W;
  for (int c = threadIdx.x; c < C; c += 256) {
    const int g = c / (C / 4);
    const float mean = a.mean_rstd[(b * 4 + g) * 2], rstd = a.mean_rstd[(b * 4 + g) * 2 + 1];
    const float sc = rstd * a.gamma[c];
    sa[c] = sc;
    sb[c] = a.beta[c] - sc * mean;
  }
  __syncthreads();
  const int pl = threadIdx.x / TPP, c0 = (threadIdx.x % TPP) * VEC;
  const int pix = blockIdx.x * PPB + pl;
  if (pix >= P) return;
  const size_t off = (static_cast<size_t>(b) * P + pix) * C + c0;
  float v[VEC];
  {
    const float4 u0 = *reinterpret_cast<const float4*>(a.y + off);
    const float4 u1 = *reinterpret_cast<const float4*>(a.y + off + 4);
    v[0] = u0.x; v[1] = u0.y; v[2] = u0.z; v[3] = u0.w;
    v[4] = u1.x; v[5] = u1.y; v[6] = u1.z; v[7] = u1.w;
  }
#pragma unroll
  for (int j = 0; j < VEC; ++j) v[j] = fmaxf(fmaf(v[j], sa[c0 + j], sb[c0 + j]), 0.f);

  if constexpr (COND != 0) {
    const float* te = a.temb + static_cast<size_t>(b) * a.temb_bstride + c0;
    float cv[VEC];
    if constexpr (COND == 1) {
      const float* cp = a.cond + (static_cast<size_t>(b) * P + pix) * C + c0;
      const float4 u0 = *reinterpret_cast<const float4*>(cp);
      const float4 u1 = *reinterpret_cast<const float4*>(cp + 4);
      cv[0] = u0.x; cv[1] = u0.y; cv[2] = u0.z; cv[3] = u0.w;
      cv[4] = u1.x; cv[5] = u1.y; cv[6] = u1.z; cv[7] = u1.w;
#pragma unroll
      for (int j = 0; j < VEC; ++j) cv[j] += te[j];
    } else {
      // ATen upsample_bilinear2d, align_corners=True: src = scale * dst, lambda1 = frac, lambda0 = 1 - lambda1;
      // the time embedding is constant over space so interp(cond + temb) == interp(cond) + temb up to rounding;
      // we follow the reference order: (cond + temb) first, then interpolate.
      const int oy = pix / a.W, ox = pix % a.W;
      const float fy = a.ry * oy, fx = a.rx * ox;
      const int y0 = static_cast<int>(fy), x0 = static_cast<int>(fx);
      const int y1 = y0 + (y0 < a.ch - 1 ? 1 : 0), x1 = x0 + (x0 < a.cw - 1 ? 1 : 0);
      const float ly1 = fy - y0, lx1 = fx - x0, ly0 = 1.f - ly1, lx0 = 1.f - lx1;
      const float* base = a.cond + static_cast<size_t>(b) * a.ch * a.cw * C + c0;
      const float* p00 = base + (static_cast<size_t>(y0) * a.cw + x0) * C;
      const float* p01 = base + (static_cast<size_t>(y0) * a.cw + x1) * C;
      const float* p10 = base + (static_cast<size_t>(y1) * a.cw + x0) * C;
      const float* p11 = base + (static_cast<size_t>(y1) * a.cw + x1) * C;
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const float4 q00 = *reinterpret_cast<const float4*>(p00 + 4 * h);
        const float4 q01 = *reinterpret_cast<const float4*>(p01 + 4 * h);
        const float4 q10 = *reinterpret_cast<const float4*>(p10 + 4 * h);
        const float4 q11 = *reinterpret_cast<const float4*>(p11 + 4 * h);
        const float t0 = te[4 * h], t1 = te[4 * h + 1], t2 = te[4 * h + 2], t3 = te[4 * h + 3];
        cv[4 * h + 0] = ly0 * (lx0 * (q00.x + t0) + lx1 * (q01.x + t0)) + ly1 * (lx0 * (q10.x + t0) + lx1 * (q11.x + t0));
        cv[4 * h + 1] = ly0 * (lx0 * (q00.y + t1) + lx1 * (q01.y + t1)) + ly1 * (lx0 * (q10.y + t1) + lx1 * (q11.y + t1));
        cv[4 * h + 2] = ly0 * (lx0 * (q00.z + t2) + lx1 * (q01.z + t2)) + ly1 * (lx0 * (q10.z + t2) + lx1 * (q11.z + t2));
        cv[4 * h + 3] = ly0 * (lx0 * (q00.w + t3) + lx1 * (q01.w + t3)) + ly1 * (lx0 * (q10.w + t3) + lx1 * (q11.w + t3));
      }
    }
#pragma unroll
    for (int j = 0; j < VEC; ++j) v[j] = cv[j] + v[j];
  }

  bool ov = false;
  store_planes8(v, a.scale, a.out_hi, a.out_lo, a.out_a8, a.out_l8, off, ov);
  if (ov) atomicOr(a.status, 1);
}

// Swin-head variant of the above for C = 256 with the bilinear (align_corners=True) condition injection, organised around
// SOURCE REUSE IN REGISTERS.  ncu on the tiled versions (profiles/r02_loop_convs_ncu_full_summary_session1.csv): DRAM traffic
// was exactly algorithmic (548 MB read, 381 MB written) at 51 % of the DRAM peak while `l1tex__throughput` sat at 92 %: every
// output pixel pulled its four 1 KB taps out of shared memory, 4 KB of shared-memory reads per KB of output, and neither
// staging the conv outputs by cp.async.bulk nor a persistent three-stage ring moved it (267 -> 244 -> 246 us inside the
// replayed graph, profiles/README.md "Round 2, session 2").  With the condition at half the latent resolution the 2 x 2 output
// "quad" (rows 2i-1, 2i; columns 2j-1, 2j) interpolates from the SAME 2 x 2 source pixels (i-1, i) x (j-1, j).  64 threads x
// 4 channels = one quad x 256 channels: they load the four source pixels and the quad's (up to) four conv outputs straight
// from global memory into registers (8 x LDG.128 per thread in flight, coalesced 1 KB rows, no shared memory), fold the
// bilinear weights of each output onto the quad's sources (w_rc = wy_r * wx_c; an index that is not one of the two loaded
// rows / columns — any geometry other than exact 2x — takes the per-tap path below) and write the operand planes.  L1
// traffic per output pixel: 1 KB of taps instead of 4.  The power-of-two operand scale is folded into the GroupNorm affine,
// the time embedding and the weights (exact), and the time embedding enters once (interp(cond + te) == interp(cond) + te *
// (sum of the weights), which is 1 within 2 ulp).

// V (4 or 8) consecutive channels of one pixel, ALREADY multiplied by the operand scale -> planes; `mx` collects max |s|
template <int V>
__device__ __forceinline__ void store_planes_scaled(const float (&s)[V], __half* out_hi, __half* out_lo, uint8_t* out_a8,
                                                    uint8_t* out_l8, size_t off, float& mx) {
  static_assert(V == 4 || V == 8, "4 or 8 channels per thread");
  using VH = typename std::conditional<V == 8, uint4, uint2>::type;  // V fp16 values
  using VB = typename std::conditional<V == 8, uint2, uint32_t>::type;  // V e4m3 values
  __align__(16) __half2 h[V / 2];
#pragma unroll
  for (int j = 0; j < V / 2; ++j) {
    h[j] = __floats2half2_rn(s[2 * j], s[2 * j + 1]);
    mx = fmaxf(mx, fmaxf(fabsf(s[2 * j]), fabsf(s[2 * j + 1])));
  }
  *reinterpret_cast<VH*>(out_hi + off) = *reinterpret_cast<const VH*>(h);
  if (out_a8 != nullptr) {
    __align__(8) uint16_t a8[V / 2];
    __align__(8) uint16_t l8[V / 2];
#pragma unroll
    for (int j = 0; j < V / 2; ++j) {
      const float2 hf = __half22float2(h[j]);
      a8[j] = e4m3x2(s[2 * j] * kF8ActDiv, s[2 * j + 1] * kF8ActDiv);
      l8[j] = e4m3x2((s[2 * j] - hf.x) * kF8LoMul, (s[2 * j + 1] - hf.y) * kF8LoMul);
    }
    *reinterpret_cast<VB*>(out_a8 + off) = *reinterpret_cast<const VB*>(a8);
    *reinterpret_cast<VB*>(out_l8 + off) = *reinterpret_cast<const VB*>(l8);
  } else {
    __align__(16) __half2 l[V / 2];
#pragma unroll
    for (int j = 0; j < V / 2; ++j) {
      const float2 hf = __half22float2(h[j]);
      l[j] = __floats2half2_rn(s[2 * j] - hf.x, s[2 * j + 1] - hf.y);
    }
    *reinterpret_cast<VH*>(out_lo + off) = *reinterpret_cast<const VH*>(l);
  }
}

__device__ __forceinline__ void ld4(const float* p, float (&v)[4]) {
  const float4 u = __ldg(reinterpret_cast<const float4*>(p));
  v[0] = u.x; v[1] = u.y; v[2] = u.z; v[3] = u.w;
}
__device__ __forceinline__ void ld4_stream(const float* p, float (&v)[4]) {
  const float4 u = __ldcs(reinterpret_cast<const float4*>(p));
  v[0] = u.x; v[1] = u.y; v[2] = u.z; v[3] = u.w;
}

// ATen upsample_bilinear2d (align_corners=True) source index / weights of one output coordinate
struct Lerp1 {
  int i0, i1;
  float l0, l1;
};
__device__ __forceinline__ Lerp1 lerp_coord(float ratio, int o, int n_src) {
  Lerp1 r;
  const float f = ratio * o;
  r.i0 = static_cast<int>(f);
  r.i1 = r.i0 + (r.i0 < n_src - 1 ? 1 : 0);
  r.l1 = f - r.i0;
  r.l0 = 1.f - r.l1;
  return r;
}

// V = channels per thread (4: 64 threads per quad, 80 registers, 3 blocks of 256 threads per SM).  Measured variants that
// changed nothing inside the graph (profiles/README.md, session 2): 8 channels per thread / one warp per quad (128
// registers, 2 blocks: 214.5 vs 214.5 us, and convA behind it 30 us slower), one quad per 64-thread block so that the
// quad's scalars are warp-uniform (189-216 vs 201-220 us).  ncu at 1.89 GHz: 185 us, DRAM 61 % of its peak, issue-active
// 72 %, ALU pipe 57 %: at the power-capped clock of the replayed graph the kernel is issue-bound on its per-quad scalar work.
template <int V>
__device__ __forceinline__ void ldv(const float* p, float (&v)[V]) {
#pragma unroll
  for (int i = 0; i < V / 4; ++i) ld4(p + 4 * i, *reinterpret_cast<float(*)[4]>(&v[4 * i]));
}
template <int V>
__device__ __forceinline__ void ldv_stream(const float* p, float (&v)[V]) {
#pragma unroll
  for (int i = 0; i < V / 4; ++i) ld4_stream(p + 4 * i, *reinterpret_cast<float(*)[4]>(&v[4 * i]));
}
template <int V, int QPB>  // QPB quads (consecutive quad columns) per block of QPB * 256 / V threads
__global__ void __launch_bounds__(QPB * 256 / V, 12 / QPB) gn_apply_up_split_kernel(const ApplyArgs a) {
  constexpr int C = 256, TPQ = C / V;
  // Blocks are dispatched in increasing (z, y, x); this kernel walks the images and quad rows BACKWARDS (DD_UP_FORWARD: A/B
  // build): its producer (the persistent 64 -> 256 conv, tiles in increasing order) has just written the END of the conv
  // output, which is what still sits in the 126 MB L2, and its consumer (convA, tiles in increasing order) starts with what
  // this kernel wrote LAST.
#ifdef DD_UP_FORWARD
  const int b = blockIdx.z, qy = blockIdx.y;
#else
  const int b = gridDim.z - 1 - blockIdx.z, qy = gridDim.y - 1 - blockIdx.y;
#endif
  const int qx = QPB == 1 ? blockIdx.x : blockIdx.x * QPB + threadIdx.x / TPQ;  // quad q: output columns {2q - 1, 2q} in [0, W)
  if (QPB > 1 && qx > a.W / 2) return;
  const int c0 = (threadIdx.x % TPQ) * V;
  const int P = a.H * a.W;
  const int ox[2] = {max(2 * qx - 1, 0), min(2 * qx, a.W - 1)};
  const int oy[2] = {max(2 * qy - 1, 0), min(2 * qy, a.H - 1)};
  const int nx = ox[1] > ox[0] ? 2 : 1, ny = oy[1] > oy[0] ? 2 : 1;
  // the two source rows / columns this quad keeps in registers
  const int xa = static_cast<int>(a.rx * ox[0]), xb = min(xa + 1, a.cw - 1);
  const int ya = static_cast<int>(a.ry * oy[0]), yb = min(ya + 1, a.ch - 1);
  const float* cbase = a.cond + static_cast<size_t>(b) * a.ch * a.cw * C + c0;
  float S[2][2][V];
  ldv<V>(cbase + (static_cast<size_t>(ya) * a.cw + xa) * C, S[0][0]);
  ldv<V>(cbase + (static_cast<size_t>(ya) * a.cw + xb) * C, S[0][1]);
  ldv<V>(cbase + (static_cast<size_t>(yb) * a.cw + xa) * C, S[1][0]);
  ldv<V>(cbase + (static_cast<size_t>(yb) * a.cw + xb) * C, S[1][1]);
  float Y[2][2][V];
#pragma unroll
  for (int r = 0; r < 2; ++r)
#pragma unroll
    for (int c = 0; c < 2; ++c)
      if (r < ny && c < nx)
        ldv_stream<V>(a.y + (static_cast<size_t>(b) * P + static_cast<size_t>(oy[r]) * a.W + ox[c]) * C + c0, Y[r][c]);
  // per-image constants of this thread's channels, pre-multiplied by the (power-of-two) operand scale
  float sa[V], sb[V], te[V];
  {
    const int g = c0 / (C / 4);
    const float mean = a.mean_rstd[(b * 4 + g) * 2], rstd = a.mean_rstd[(b * 4 + g) * 2 + 1];
    float gm[V], bt[V], tt[V];
    ldv<V>(a.gamma + c0, gm);
    ldv<V>(a.beta + c0, bt);
    ldv<V>(a.temb + static_cast<size_t>(b) * a.temb_bstride + c0, tt);
#pragma unroll
    for (int j = 0; j < V; ++j) {
      const float scl = rstd * gm[j];  // same rounding as the generic kernel: (rstd * gamma), beta - that * mean
      sa[j] = scl * a.scale;
      sb[j] = (bt[j] - scl * mean) * a.scale;
      te[j] = tt[j] * a.scale;
    }
  }
  float mx = 0.f;
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    if (r >= ny) break;
    const Lerp1 ly = lerp_coord(a.ry, oy[r], a.ch);
    const bool oky = (ly.i0 == ya || ly.i0 == yb) && (ly.i1 == ya || ly.i1 == yb);
    // weights of the two loaded source rows (a clamped pair ya == yb puts everything on row a)
    const float wya = (ly.i0 == ya ? ly.l0 : 0.f) + (ly.i1 == ya ? ly.l1 : 0.f);
    const float wyb = yb != ya ? (ly.i0 == yb ? ly.l0 : 0.f) + (ly.i1 == yb ? ly.l1 : 0.f) : 0.f;
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      if (c >= nx) break;
      const Lerp1 lx = lerp_coord(a.rx, ox[c], a.cw);
      const bool ok = oky && (lx.i0 == xa || lx.i0 == xb) && (lx.i1 == xa || lx.i1 == xb);
      float sv[V];
      if (ok) {
        const float wxa = (lx.i0 == xa ? lx.l0 : 0.f) + (lx.i1 == xa ? lx.l1 : 0.f);
        const float wxb = xb != xa ? (lx.i0 == xb ? lx.l0 : 0.f) + (lx.i1 == xb ? lx.l1 : 0.f) : 0.f;
        const float w00 = wya * wxa * a.scale, w01 = wya * wxb * a.scale, w10 = wyb * wxa * a.scale, w11 = wyb * wxb * a.scale;
#pragma unroll
        for (int j = 0; j < V; ++j) {
          const float gn = fmaxf(fmaf(Y[r][c][j], sa[j], sb[j]), 0.f);
          float up = fmaf(w00, S[0][0][j], te[j]);
          up = fmaf(w01, S[0][1][j], up);
          up = fmaf(w10, S[1][0][j], up);
          up = fmaf(w11, S[1][1][j], up);
          sv[j] = up + gn;
        }
      } else {  // geometry other than 2x: this output's taps are not the quad's sources — fetch them
        float q00[V], q01[V], q10[V], q11[V];
        ldv<V>(cbase + (static_cast<size_t>(ly.i0) * a.cw + lx.i0) * C, q00);
        ldv<V>(cbase + (static_cast<size_t>(ly.i0) * a.cw + lx.i1) * C, q01);
        ldv<V>(cbase + (static_cast<size_t>(ly.i1) * a.cw + lx.i0) * C, q10);
        ldv<V>(cbase + (static_cast<size_t>(ly.i1) * a.cw + lx.i1) * C, q11);
        const float w00 = ly.l0 * lx.l0 * a.scale, w01 = ly.l0 * lx.l1 * a.scale, w10 = ly.l1 * lx.l0 * a.scale,
                    w11 = ly.l1 * lx.l1 * a.scale;
#pragma unroll
        for (int j = 0; j < V; ++j) {
          const float gn = fmaxf(fmaf(Y[r][c][j], sa[j], sb[j]), 0.f);
          float up = fmaf(w00, q00[j], te[j]);
          up = fmaf(w01, q01[j], up);
          up = fmaf(w10, q10[j], up);
          up = fmaf(w11, q11[j], up);
          sv[j] = up + gn;
        }
      }
      const size_t off = (static_cast<size_t>(b) * P + static_cast<size_t>(oy[r]) * a.W + ox[c]) * C + c0;
      store_planes_scaled<V>(sv, a.out_hi, a.out_lo, a.out_a8, a.out_l8, off, mx);
    }
  }
  if (mx > (a.out_a8 != nullptr ? kF8ActMax : 60000.f)) atomicOr(a.status, 1);
}

// ------------------------------------------------------------------ last GN + ReLU (C = 16) fused with the DDIM update
// eps = relu(gn(y6));  x <- c_x * x + c_eps * eps   (reference scheduling_ddim.py:285-326 with eta = 0,
// collapsed; SURVEY.md §3.3).  Also refreshes the fp16 planes of x for the next step's first conv.
// If eps_out != nullptr, only eps is written (bare denoiser call) and x is left untouched.
// Stochastic DDIM (eta > 0, gn_relu_ddim_stoch_kernel): x <- fmaf(sigma, z, c_x * x + c_eps * eps), z = this step's
// noise (reference scheduling_ddim.py:313-350); c_x / c_eps then carry sigma in c_eps = sqrt(1 - a_p - sigma^2) - ...
// With sigma = 0 the update is bit-identical to gn_relu_ddim_kernel's.
struct FinalArgs {
  const float* y;          // [B][P][16]
  const float* mean_rstd;  // [B][4][2]
  const float* gamma;
  const float* beta;
  float* x;                // [B][P][16] fp32 latent (in/out)
  __half* x_hi;
  __half* x_lo;
  float* eps_out;          // optional [B][P][16]
  float cx, ce, scale;
  int P;
  int* status;
  const float* z;          // stochastic kernel only: this step's noise [B][P][16]
  float sigma;             // stochastic kernel only
};
template <bool STOCH>
__device__ __forceinline__ void gn_relu_ddim_body(const FinalArgs& a) {
  const int b = blockIdx.y;
  const size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x;  // float4 index within image
  if (i >= static_cast<size_t>(a.P) * 4) return;
  const int g = static_cast<int>(i & 3);  // 16 channels / 4 per float4 = group index
  const float mean = a.mean_rstd[(b * 4 + g) * 2], rstd = a.mean_rstd[(b * 4 + g) * 2 + 1];
  const size_t o4 = static_cast<size_t>(b) * a.P * 4 + i;
  const float4 yv = reinterpret_cast<const float4*>(a.y)[o4];
  const float4 ga = reinterpret_cast<const float4*>(a.gamma)[g];
  const float4 be = reinterpret_cast<const float4*>(a.beta)[g];
  float e[4] = {yv.x, yv.y, yv.z, yv.w};
  const float gg[4] = {ga.x, ga.y, ga.z, ga.w}, bb[4] = {be.x, be.y, be.z, be.w};
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float sc = rstd * gg[j];
    e[j] = fmaxf(fmaf(e[j], sc, bb[j] - sc * mean), 0.f);
  }
  if (a.eps_out) {
    reinterpret_cast<float4*>(a.eps_out)[o4] = make_float4(e[0], e[1], e[2], e[3]);
    return;
  }
  const float4 xv = reinterpret_cast<const float4*>(a.x)[o4];
  float xn[4] = {xv.x, xv.y, xv.z, xv.w};
  float zn[4] = {0.f, 0.f, 0.f, 0.f};
  if (STOCH) {
    const float4 zv = reinterpret_cast<const float4*>(a.z)[o4];
    zn[0] = zv.x; zn[1] = zv.y; zn[2] = zv.z; zn[3] = zv.w;
  }
  bool ov = false;
  __align__(8) __half h[4];
  __align__(8) __half l[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    if (STOCH)
      xn[j] = fmaf(a.sigma, zn[j], a.cx * xn[j] + a.ce * e[j]);
    else
      xn[j] = a.cx * xn[j] + a.ce * e[j];
    split_f16(xn[j], a.scale, h[j], l[j], ov);
  }
  reinterpret_cast<float4*>(a.x)[o4] = make_float4(xn[0], xn[1], xn[2], xn[3]);
  reinterpret_cast<uint2*>(a.x_hi)[o4] = *reinterpret_cast<const uint2*>(h);
  reinterpret_cast<uint2*>(a.x_lo)[o4] = *reinterpret_cast<const uint2*>(l);
  if (ov) atomicOr(a.status, 1);
}
__global__ void __launch_bounds__(256) gn_relu_ddim_kernel(const FinalArgs a) { gn_relu_ddim_body<false>(a); }
__global__ void __launch_bounds__(256) gn_relu_ddim_stoch_kernel(const FinalArgs a) { gn_relu_ddim_body<true>(a); }

// ------------------------------------------------------------------ fp32 CUDA-core 3x3 conv (validation / DD_FLAG_SIMT_CONV)
// Same operands and epilogues as the tcgen05 kernel: input fp16 hi/lo planes (x = (hi+lo)/scale), weights fp32
// [tap][CIN][COUT].  One block = one 8x16 pixel tile x CO_T output channels.
struct SimtArgs {
  const __half* in_hi;
  const __half* in_lo;
  float in_inv_scale;
  const float* w;          // [9][CIN][COUT]
  ConvArgs c;
};

template <int CIN, int COUT, int EPI>
__global__ void __launch_bounds__(256) conv3x3_simt_kernel(const SimtArgs a) {
  constexpr int CO_T = COUT < 64 ? COUT : 64;
  constexpr int CK = 16;                 // input channels per smem chunk
  constexpr int CGS = CO_T / 4;          // channel groups of 4
  constexpr int PGS = 256 / CGS;         // pixel groups
  constexpr int PXT = TILE_M / PGS;      // pixels per thread (8 or 2)
  __shared__ float s_in[(TILE_H + 2) * (TILE_W + 2)][CK];
  __shared__ float s_w[9][CK][CO_T];
  __shared__ float s_red[4][2];
  const ConvArgs& p = a.c;
  const int tile = blockIdx.x;
  const int co0 = blockIdx.y * CO_T;
  const int tx = tile % p.tiles_x, ty = (tile / p.tiles_x) % p.tiles_y, img = tile / (p.tiles_x * p.tiles_y);
  const int x0 = tx * TILE_W, y0 = ty * TILE_H;
  const int cg = threadIdx.x % CGS, pg = threadIdx.x / CGS;
  float acc[PXT][4];
#pragma unroll
  for (int i = 0; i < PXT; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  if (threadIdx.x < 8) (&s_red[0][0])[threadIdx.x] = 0.f;

  for (int k0 = 0; k0 < CIN; k0 += CK) {
    __syncthreads();
    for (int i = threadIdx.x; i < (TILE_H + 2) * (TILE_W + 2) * CK; i += 256) {
      const int ci = i % CK, hp = i / CK;
      const int yy = y0 + hp / (TILE_W + 2) - 1, xx = x0 + hp % (TILE_W + 2) - 1;
      float v = 0.f;
      if (yy >= 0 && yy < p.H && xx >= 0 && xx < p.W) {
        const size_t o = ((static_cast<size_t>(img) * p.H + yy) * p.W + xx) * CIN + k0 + ci;
        v = (__half2float(a.in_hi[o]) + __half2float(a.in_lo[o])) * a.in_inv_scale;
      }
      s_in[hp][ci] = v;
    }
    for (int i = threadIdx.x; i < 9 * CK * CO_T; i += 256) {
      const int co = i % CO_T, ci = (i / CO_T) % CK, tap = i / (CO_T * CK);
      s_w[tap][ci][co] = a.w[(static_cast<size_t>(tap) * CIN + k0 + ci) * COUT + co0 + co];
    }
    __syncthreads();
#pragma unroll
    for (int tap = 0; tap < 9; ++tap) {
      const int dy = tap / 3, dx = tap % 3;
#pragma unroll 4
      for (int ci = 0; ci < CK; ++ci) {
        const float4 w4 = *reinterpret_cast<const float4*>(&s_w[tap][ci][cg * 4]);
#pragma unroll
        for (int i = 0; i < PXT; ++i) {
          const int m = pg * PXT + i;
          const float v = s_in[((m >> 4) + dy) * (TILE_W + 2) + (m & 15) + dx][ci];
          acc[i][0] = fmaf(v, w4.x, acc[i][0]);
          acc[i][1] = fmaf(v, w4.y, acc[i][1]);
          acc[i][2] = fmaf(v, w4.z, acc[i][2]);
          acc[i][3] = fmaf(v, w4.w, acc[i][3]);
        }
      }
    }
  }
  // epilogue
  float ls[4] = {0.f, 0.f, 0.f, 0.f}, ls2[4] = {0.f, 0.f, 0.f, 0.f};
  bool ov = false;
#pragma unroll
  for (int i = 0; i < PXT; ++i) {
    const int m = pg * PXT + i;
    const int y = y0 + (m >> 4), x = x0 + (m & 15);
    if (y >= p.H || x >= p.W) continue;
    const size_t pix = (static_cast<size_t>(img) * p.H + y) * p.W + x;
    float v[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) v[j] = acc[i][j] + p.bias[co0 + cg * 4 + j];
    if constexpr (EPI == EPI_SPLIT) {
      __align__(8) __half h[4];
      __align__(8) __half l[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) split_f16(v[j], p.split_scale, h[j], l[j], ov);
      *reinterpret_cast<uint2*>(p.out_hi + pix * COUT + co0 + cg * 4) = *reinterpret_cast<const uint2*>(h);
      *reinterpret_cast<uint2*>(p.out_lo + pix * COUT + co0 + cg * 4) = *reinterpret_cast<const uint2*>(l);
    } else {
      *reinterpret_cast<float4*>(p.y32 + pix * COUT + co0 + cg * 4) = make_float4(v[0], v[1], v[2], v[3]);
      if constexpr (EPI == EPI_F32_STATS) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int g = (co0 + cg * 4 + j) / (COUT / 4);
          const int gl = (COUT / 4 >= CO_T) ? 0 : (g - co0 / (COUT / 4));
          ls[gl] += v[j];
          ls2[gl] = fmaf(v[j], v[j], ls2[gl]);
        }
      }
    }
  }
  if constexpr (EPI == EPI_F32_STATS) {
    constexpr int NG = (COUT / 4 >= CO_T) ? 1 : CO_T / (COUT / 4);  // groups covered by this block
#pragma unroll
    for (int g = 0; g < NG; ++g) {
      atomicAdd(&s_red[g][0], ls[g]);
      atomicAdd(&s_red[g][1], ls2[g]);
    }
    __syncthreads();
    if (threadIdx.x < NG * 2) {
      const int g = threadIdx.x >> 1, which = threadIdx.x & 1;
      const int gg = co0 / (COUT / 4) + g;
      p.stats_partial[(static_cast<size_t>(tile) * 4 + gg) * 2 + which] = s_red[g][which];
    }
  }
  if constexpr (EPI == EPI_SPLIT) {
    if (ov) atomicOr(p.status, 1);
  }
}

// ------------------------------------------------------------------ depth-latent decoder (inv_t), fully fused
// ConvTranspose2d(16,16,k4,s2,p1)+b -> BN(eval, folded) -> ReLU -> Conv2d(16,1,3,1,1)+b -> z
// depth = 1 / clamp(sigmoid(z), 1e-6) - 1          (reference src/model/ops/depth_transform.py:20-26,33-35)
// One block = 8 x 32 output pixels; latent patch and the 10 x 34 x 16 intermediate stay in shared memory.
struct DecoderArgs {
  const float* x;      // latent NHWC [B][h][w][16]
  const float* wt;     // folded ConvT weights [ky][kx][ci][co]
  const float* bt;     // folded bias [16]
  const float* wc;     // final conv [tap][ci]
  float bc;            // final conv bias
  float* logit;        // optional [B][2h][2w]
  float* depth;        // [B][2h][2w]
  int h, w;
  float eps;
};
constexpr int DEC_TH = 8, DEC_TW = 32;
constexpr int DEC_SMEM = ((DEC_TH / 2 + 2) * (DEC_TW / 2 + 2) * 16 + (DEC_TH + 2) * (DEC_TW + 2) * 20 + 4096 + 144 + 16) * 4;
// Round 2 (ncu: the first version spent 618 us per call with the shared-memory pipe 96 % busy — scalar weight reads in
// the transposed conv, two scalar reads per FMA in the final conv): the transposed conv walks the intermediate pixels
// PARITY CLASS by parity class, so a warp's (ky, kx) taps and output-channel half are uniform and the folded weights come
// in as broadcast float4s (2 x LDS.128 + 1 latent read per 8 FMAs); the final conv reads both the intermediate (row stride
// 20 floats: conflict-free 16-byte reads) and its weights as float4s (8 x LDS.128 per 16 FMAs).
__global__ void __launch_bounds__(256) decoder_kernel(const DecoderArgs a) {
  constexpr int LH = DEC_TH / 2 + 2, LW = DEC_TW / 2 + 2;  // latent patch 6 x 18
  constexpr int MH = DEC_TH + 2, MW = DEC_TW + 2;          // intermediate 10 x 34
  constexpr int CH = MH / 2, CW = MW / 2, CPX = CH * CW;   // pixels per parity class: 5 x 17 = 85
  constexpr int CPAD = 96;                                 // padded to whole warps
  extern __shared__ __align__(16) float dec_smem[];  // DEC_SMEM bytes (above the 48 KB static limit)
  float (*s_lat)[16] = reinterpret_cast<float (*)[16]>(dec_smem);
  float (*s_mid)[20] = reinterpret_cast<float (*)[20]>(dec_smem + LH * LW * 16);
  float* s_wt = dec_smem + LH * LW * 16 + MH * MW * 20;
  float* s_wc = s_wt + 16 * 16 * 16;
  float* s_bt = s_wc + 9 * 16;
  const int b = blockIdx.z;
  const int Y0 = blockIdx.y * DEC_TH, X0 = blockIdx.x * DEC_TW;
  const int H = 2 * a.h, W = 2 * a.w;
  for (int i = threadIdx.x; i < 1024; i += 256) reinterpret_cast<float4*>(s_wt)[i] = reinterpret_cast<const float4*>(a.wt)[i];
  if (threadIdx.x < 144) s_wc[threadIdx.x] = a.wc[threadIdx.x];
  if (threadIdx.x < 16) s_bt[threadIdx.x] = a.bt[threadIdx.x];
  const int ly0 = Y0 / 2 - 1, lx0 = X0 / 2 - 1;
  for (int i = threadIdx.x; i < LH * LW * 4; i += 256) {
    const int q = i & 3, lp = i >> 2;
    const int yy = ly0 + lp / LW, xx = lx0 + lp % LW;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (yy >= 0 && yy < a.h && xx >= 0 && xx < a.w)
      v = reinterpret_cast<const float4*>(a.x + ((static_cast<size_t>(b) * a.h + yy) * a.w + xx) * 16)[q];
    *reinterpret_cast<float4*>(&s_lat[lp][q * 4]) = v;
  }
  __syncthreads();
  // transposed conv: out(Y, X) gathers the 2x2 latent pixels iy = (Y + 1 - ky) / 2 with matching parity.  Work item =
  // (parity class, output-channel half, pixel of the class): 4 x 2 x 96 slots = 3 rounds of 256 threads, warp-uniform
  // class and half.
  for (int it = threadIdx.x; it < 8 * CPAD; it += 256) {
    const int cls = it / (2 * CPAD), half = (it / CPAD) & 1, pi = it % CPAD;
    if (pi >= CPX) continue;
    // mid row my (0..9) <-> Y = Y0 - 1 + my; class parity py = (Y + 1) & 1 = (Y0 + my) & 1 -> Y0 is even: py = my & 1
    const int py = cls >> 1, px = cls & 1;
    const int my = 2 * (pi / CW) + py, mx = 2 * (pi % CW) + px;
    const int Y = Y0 - 1 + my, X = X0 - 1 + mx;
    float o[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) o[j] = 0.f;
    if (Y >= 0 && Y < H && X >= 0 && X < W) {
#pragma unroll
      for (int j = 0; j < 8; ++j) o[j] = s_bt[half * 8 + j];
      const int ky0 = (Y + 1) & 1, kx0 = (X + 1) & 1;  // == py, px (warp-uniform)
#pragma unroll
      for (int a2 = 0; a2 < 2; ++a2) {
        const int ky = ky0 + 2 * a2;
        const int iy = (Y + 1 - ky) / 2;  // exact: numerator even
        if (Y + 1 - ky < 0 || iy >= a.h) continue;
#pragma unroll
        for (int b2 = 0; b2 < 2; ++b2) {
          const int kx = kx0 + 2 * b2;
          const int ix = (X + 1 - kx) / 2;
          if (X + 1 - kx < 0 || ix >= a.w) continue;
          const float* lp = s_lat[(iy - ly0) * LW + (ix - lx0)];
          const float* wp = s_wt + ((ky * 4 + kx) * 16) * 16 + half * 8;
#pragma unroll
          for (int c4 = 0; c4 < 4; ++c4) {
            const float4 lv = *reinterpret_cast<const float4*>(lp + 4 * c4);
            const float l4[4] = {lv.x, lv.y, lv.z, lv.w};
#pragma unroll
            for (int cc = 0; cc < 4; ++cc) {
              const float4 w0 = *reinterpret_cast<const float4*>(wp + (4 * c4 + cc) * 16);
              const float4 w1 = *reinterpret_cast<const float4*>(wp + (4 * c4 + cc) * 16 + 4);
              const float v = l4[cc];
              o[0] = fmaf(v, w0.x, o[0]); o[1] = fmaf(v, w0.y, o[1]); o[2] = fmaf(v, w0.z, o[2]); o[3] = fmaf(v, w0.w, o[3]);
              o[4] = fmaf(v, w1.x, o[4]); o[5] = fmaf(v, w1.y, o[5]); o[6] = fmaf(v, w1.z, o[6]); o[7] = fmaf(v, w1.w, o[7]);
            }
          }
        }
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) o[j] = fmaxf(o[j], 0.f);
    }
    float* mp = s_mid[my * MW + mx] + half * 8;
    *reinterpret_cast<float4*>(mp) = make_float4(o[0], o[1], o[2], o[3]);
    *reinterpret_cast<float4*>(mp + 4) = make_float4(o[4], o[5], o[6], o[7]);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < DEC_TH * DEC_TW; i += 256) {
    const int yy = i / DEC_TW, xx = i % DEC_TW;
    const int Y = Y0 + yy, X = X0 + xx;
    if (Y >= H || X >= W) continue;
    float z = a.bc;
#pragma unroll
    for (int tap = 0; tap < 9; ++tap) {
      const float* mp = s_mid[(yy + tap / 3) * MW + xx + tap % 3];
#pragma unroll
      for (int c4 = 0; c4 < 4; ++c4) {
        const float4 mv = *reinterpret_cast<const float4*>(mp + 4 * c4);
        const float4 wv = *reinterpret_cast<const float4*>(s_wc + tap * 16 + 4 * c4);
        z = fmaf(mv.x, wv.x, z); z = fmaf(mv.y, wv.y, z); z = fmaf(mv.z, wv.z, z); z = fmaf(mv.w, wv.w, z);
      }
    }
    const size_t o = (static_cast<size_t>(b) * H + Y) * W + X;
    if (a.logit) a.logit[o] = z;
    const float s = 1.0f / (1.0f + expf(-z));
    a.depth[o] = 1.0f / fmaxf(s, a.eps) - 1.0f;
  }
}

// ------------------------------------------------------------------ depth-latent encoder (t), fully fused
// Conv2d(1,16,3,s2,p1, no bias) + BN(eval, folded) + LeakyReLU(0.2) -> Conv2d(16,16,3,1,1, no bias) + BN(folded) -> tanh
// (reference src/model/ops/depth_transform.py:15-19,29-31; conv_bn_relu = src/model/common.py:45-60).
// One block = 16 x 16 latent pixels; the 18 x 18 x 16 intermediate stays in shared memory.  Output NCHW [B,16,h,w]
// (the head only returns it as `pred_init` / `gt_map_t`).
struct EncoderArgs {
  const float* depth;  // [B,1,H,W]
  const float* w1;     // [9][16]      folded (tap, co)
  const float* b1;     // [16]
  const float* w2;     // [9][16][16]  folded (tap, ci, co)
  const float* b2;     // [16]
  float* out;          // [B,16,h,w]
  int H, W, h, w;
};
__global__ void __launch_bounds__(256) encoder_kernel(const EncoderArgs a) {
  constexpr int T = 16, M = T + 2, D = 2 * M + 1;  // mid tile 18x18, depth tile 37x37
  __shared__ float s_d[D * D];
  __shared__ float s_mid[M * M][17];
  __shared__ float s_w1[9 * 16], s_b1[16], s_w2[9 * 16 * 16], s_b2[16];
  const int b = blockIdx.z, y0 = blockIdx.y * T, x0 = blockIdx.x * T;
  for (int i = threadIdx.x; i < 9 * 16 * 16; i += 256) s_w2[i] = a.w2[i];
  if (threadIdx.x < 144) s_w1[threadIdx.x] = a.w1[threadIdx.x];
  if (threadIdx.x < 16) {
    s_b1[threadIdx.x] = a.b1[threadIdx.x];
    s_b2[threadIdx.x] = a.b2[threadIdx.x];
  }
  // mid pixel (my, mx) (latent coords y0-1+my) reads depth rows 2*(y0-1+my)-1 .. +1  -> depth origin 2*(y0-1)-1
  const int dy0 = 2 * (y0 - 1) - 1, dx0 = 2 * (x0 - 1) - 1;
  for (int i = threadIdx.x; i < D * D; i += 256) {
    const int yy = dy0 + i / D, xx = dx0 + i % D;
    s_d[i] = (yy >= 0 && yy < a.H && xx >= 0 && xx < a.W) ? a.depth[(static_cast<size_t>(b) * a.H + yy) * a.W + xx] : 0.f;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < M * M * 4; i += 256) {
    const int cq = i & 3, mp = i >> 2;
    const int my = mp / M, mx = mp % M;
    const int ly = y0 - 1 + my, lx = x0 - 1 + mx;
    float o[4] = {0.f, 0.f, 0.f, 0.f};
    if (ly >= 0 && ly < a.h && lx >= 0 && lx < a.w) {  // zero padding of the second conv outside the latent grid
#pragma unroll
      for (int j = 0; j < 4; ++j) o[j] = s_b1[cq * 4 + j];
#pragma unroll
      for (int tap = 0; tap < 9; ++tap) {
        const float v = s_d[(2 * my + tap / 3) * D + 2 * mx + tap % 3];
#pragma unroll
        for (int j = 0; j < 4; ++j) o[j] = fmaf(v, s_w1[tap * 16 + cq * 4 + j], o[j]);
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) o[j] = o[j] > 0.f ? o[j] : 0.2f * o[j];
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) s_mid[mp][cq * 4 + j] = o[j];
  }
  __syncthreads();
  const int py = threadIdx.x / T, px = threadIdx.x % T;
  const int ly = y0 + py, lx = x0 + px;
  if (ly >= a.h || lx >= a.w) return;
  float acc[16];
#pragma unroll
  for (int co = 0; co < 16; ++co) acc[co] = s_b2[co];
#pragma unroll
  for (int tap = 0; tap < 9; ++tap) {
    const float* mp = s_mid[(py + tap / 3) * M + px + tap % 3];
#pragma unroll
    for (int ci = 0; ci < 16; ++ci) {
      const float v = mp[ci];
#pragma unroll
      for (int co = 0; co < 16; ++co) acc[co] = fmaf(v, s_w2[(tap * 16 + ci) * 16 + co], acc[co]);
    }
  }
#pragma unroll
  for (int co = 0; co < 16; ++co)
    a.out[((static_cast<size_t>(b) * 16 + co) * a.h + ly) * a.w + lx] = tanhf(acc[co]);
}

}  // namespace dd
