// Bandwidth-bound pieces of the DLA-34 path: the three 7x7 stems (reference NCHW fp32 inputs in,
// NHWC activations out), Tree.downsample (2x2 max-pool), IDAUp's depthwise transposed-conv
// upsample fused with the skip add, and the pre_hm gaussian splat.
#include "common.cuh"

namespace ctb {

// ------------------------------------------------------------------------------------------
// stem: out = relu(bn(conv7(img))) + relu(bn(conv7(pre_img))) + relu(bn(conv7(pre_hm)))
// (dla.py:238-242,256-267,305-311 -- note ReLU is applied per stem BEFORE the sum)
// ------------------------------------------------------------------------------------------
constexpr int ST = 16;            // 16x16 output pixels per CTA
constexpr int SH = ST + 6;        // halo side

template <typename T>
__global__ void __launch_bounds__(ST * ST)
stem_kernel(const float* __restrict__ img, const float* __restrict__ pre, const float* __restrict__ hm,
            const float* __restrict__ w, const float* __restrict__ shift, T* __restrict__ out,
            int B, int H, int W, int ld_out) {
  __shared__ float halo[7][SH][SH + 1];
  __shared__ __align__(16) float ws[49 * 7 * 16];
  const int tx = threadIdx.x % ST, ty = threadIdx.x / ST;
  const int x0 = blockIdx.x * ST, y0 = blockIdx.y * ST, b = blockIdx.z;
  const size_t plane = (size_t)H * W;
  for (int i = threadIdx.x; i < 49 * 7 * 16; i += ST * ST) ws[i] = w[i];
  for (int i = threadIdx.x; i < 7 * SH * SH; i += ST * ST) {
    const int ch = i / (SH * SH), r = i % (SH * SH), hy = r / SH, hx = r % SH;
    const int gy = y0 + hy - 3, gx = x0 + hx - 3;
    float v = 0.f;
    if (gy >= 0 && gy < H && gx >= 0 && gx < W) {
      if (ch < 3) v = __ldg(img + ((size_t)b * 3 + ch) * plane + (size_t)gy * W + gx);
      else if (ch < 6) { if (pre) v = __ldg(pre + ((size_t)b * 3 + ch - 3) * plane + (size_t)gy * W + gx); }
      else { if (hm) v = __ldg(hm + (size_t)b * plane + (size_t)gy * W + gx); }
    }
    halo[ch][hy][hx] = v;
  }
  __syncthreads();
  float a0[16], a1[16], a2[16];
#pragma unroll
  for (int o = 0; o < 16; ++o) { a0[o] = 0.f; a1[o] = 0.f; a2[o] = 0.f; }
  for (int ky = 0; ky < 7; ++ky) {
#pragma unroll
    for (int kx = 0; kx < 7; ++kx) {
      const float* wt = ws + (ky * 7 + kx) * 7 * 16;
#pragma unroll
      for (int ch = 0; ch < 7; ++ch) {
        const float v = halo[ch][ty + ky][tx + kx];
        const float4* w4 = reinterpret_cast<const float4*>(wt + ch * 16);
        float* acc = ch < 3 ? a0 : (ch < 6 ? a1 : a2);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const float4 ww = w4[q];
          acc[q * 4 + 0] = fmaf(v, ww.x, acc[q * 4 + 0]);
          acc[q * 4 + 1] = fmaf(v, ww.y, acc[q * 4 + 1]);
          acc[q * 4 + 2] = fmaf(v, ww.z, acc[q * 4 + 2]);
          acc[q * 4 + 3] = fmaf(v, ww.w, acc[q * 4 + 3]);
        }
      }
    }
  }
  const int gy = y0 + ty, gx = x0 + tx;
  if (gy < H && gx < W) {
    T* o = out + ((size_t)b * plane + (size_t)gy * W + gx) * ld_out;
#pragma unroll
    for (int c = 0; c < 16; ++c) {
      float v = fmaxf(a0[c] + shift[c], 0.f);
      if (pre) v += fmaxf(a1[c] + shift[16 + c], 0.f);
      if (hm) v += fmaxf(a2[c] + shift[32 + c], 0.f);
      Elem<T>::st(o + c, v);
    }
  }
}

// ------------------------------------------------------------------------------------------
// stem input packing for the tensor-core stem: fp32 NCHW x3 -> bf16 NHWC [.,8]
__global__ void pack_stem_kernel(const float* __restrict__ img, const float* __restrict__ pre,
                                 const float* __restrict__ hm, uint4* __restrict__ out, int B, int H, int W) {
  const size_t plane = (size_t)H * W, total = (size_t)B * plane;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const size_t b = i / plane, r = i - b * plane;
    float v[8];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      v[c] = __ldg(img + (b * 3 + c) * plane + r);
      v[3 + c] = pre ? __ldg(pre + (b * 3 + c) * plane + r) : 0.f;
    }
    v[6] = hm ? __ldg(hm + b * plane + r) : 0.f;
    v[7] = 0.f;
    uint4 o;
    __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&o);
#pragma unroll
    for (int q = 0; q < 4; ++q) h[q] = __floats2bfloat162_rn(v[2 * q], v[2 * q + 1]);
    out[i] = o;
  }
}

// fp32 variant for the bf16x3 engine: fp32 NCHW x3 -> fp32 NHWC [.,8]
__global__ void pack_stem_f32_kernel(const float* __restrict__ img, const float* __restrict__ pre,
                                     const float* __restrict__ hm, float4* __restrict__ out, int B, int H, int W) {
  const size_t plane = (size_t)H * W, total = (size_t)B * plane;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const size_t b = i / plane, r = i - b * plane;
    float v[8];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      v[c] = __ldg(img + (b * 3 + c) * plane + r);
      v[3 + c] = pre ? __ldg(pre + (b * 3 + c) * plane + r) : 0.f;
    }
    v[6] = hm ? __ldg(hm + b * plane + r) : 0.f;
    v[7] = 0.f;
    out[2 * i] = make_float4(v[0], v[1], v[2], v[3]);
    out[2 * i + 1] = make_float4(v[4], v[5], v[6], v[7]);
  }
}

// ------------------------------------------------------------------------------------------
// Tree.downsample: 2x2 max-pool, 16-byte vectors (8 bf16 / 4 fp32 channels per thread), output may be a channel
// slice of a concat buffer (ld_out)
// ------------------------------------------------------------------------------------------
template <typename T> struct VecIO;
template <> struct VecIO<float> {
  static constexpr int N = 4;
  static __device__ __forceinline__ void ld(const float* p, float (&v)[4]) {
    const float4 t = __ldg(reinterpret_cast<const float4*>(p));
    v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
  }
  static __device__ __forceinline__ void st(float* p, const float (&v)[4]) {
    *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
  }
};
template <> struct VecIO<__nv_bfloat16> {
  static constexpr int N = 8;
  static __device__ __forceinline__ void ld(const __nv_bfloat16* p, float (&v)[8]) {
    const uint4 t = __ldg(reinterpret_cast<const uint4*>(p));
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&t);
#pragma unroll
    for (int q = 0; q < 4; ++q) { const float2 f = __bfloat1622float2(h[q]); v[2 * q] = f.x; v[2 * q + 1] = f.y; }
  }
  static __device__ __forceinline__ void st(__nv_bfloat16* p, const float (&v)[8]) {
    uint4 t;
    __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&t);
#pragma unroll
    for (int q = 0; q < 4; ++q) h[q] = __floats2bfloat162_rn(v[2 * q], v[2 * q + 1]);
    *reinterpret_cast<uint4*>(p) = t;
  }
};

// 16 raw bytes now, conversion at the point of use (keeps several loads in flight without holding their fp32 copies)
// (asm volatile: the loads keep their program order -- the compiler otherwise sinks the long-latency skip load below the FMAs)
__device__ __forceinline__ uint4 ld_raw16(const void* p) {
  uint4 r;
  asm volatile("ld.global.nc.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
  return r;
}
__device__ __forceinline__ void cvt_raw16(const uint4& t, float (&v)[4]) {
  v[0] = __uint_as_float(t.x); v[1] = __uint_as_float(t.y); v[2] = __uint_as_float(t.z); v[3] = __uint_as_float(t.w);
}
__device__ __forceinline__ void cvt_raw16(const uint4& t, float (&v)[8]) {
  const uint32_t u[4] = {t.x, t.y, t.z, t.w};                     // bf16 -> fp32 is a shift / a mask (exact)
#pragma unroll
  for (int q = 0; q < 4; ++q) { v[2 * q] = __uint_as_float(u[q] << 16); v[2 * q + 1] = __uint_as_float(u[q] & 0xffff0000u); }
}

template <typename T>
__global__ void maxpool2_kernel(const T* __restrict__ x, T* __restrict__ out, int B, int H, int W, int C,
                                int ld_in, int ld_out) {
  constexpr int V = VecIO<T>::N;
  const int OH = H / 2, OW = W / 2, CV = C / V;
  const size_t total = (size_t)B * OH * OW * CV;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total;
       i += (size_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % CV) * V;
    size_t p = i / CV;
    const int ox = p % OW; p /= OW;
    const int oy = p % OH;
    const int b = p / OH;
    const T* s = x + (((size_t)b * H + 2 * oy) * W + 2 * ox) * ld_in + c;
    float v0[V], v1[V], v2[V], v3[V];
    VecIO<T>::ld(s, v0); VecIO<T>::ld(s + ld_in, v1);
    VecIO<T>::ld(s + (size_t)W * ld_in, v2); VecIO<T>::ld(s + (size_t)(W + 1) * ld_in, v3);
#pragma unroll
    for (int q = 0; q < V; ++q) v0[q] = fmaxf(fmaxf(v0[q], v1[q]), fmaxf(v2[q], v3[q]));
    VecIO<T>::st(out + (((size_t)b * OH + oy) * OW + ox) * ld_out + c, v0);
  }
}

// ------------------------------------------------------------------------------------------
// depthwise ConvTranspose2d(k=2f, stride f, pad f/2, no bias) + skip  (dla.py:529-531,543-545)
// One thread = one output pixel x 16 bytes of channels (8 bf16 / 4 fp32): every access is a full
// 16-byte vector, consecutive threads walk consecutive channel groups then pixels (coalesced).
// w is channel-last: fp32 [2f][2f][C].
// ------------------------------------------------------------------------------------------
template <typename T>
__global__ void upsample_add_kernel(const T* __restrict__ x, const T* __restrict__ skip,
                                    const float* __restrict__ w, T* __restrict__ out, int B, int H, int W,
                                    int C, int f, int ld_in, int ld_skip, int ld_out) {
  constexpr int V = VecIO<T>::N;
  const int OH = H * f, OW = W * f, pad = f / 2, k = 2 * f, CV = C / V;
  const size_t total = (size_t)B * OH * OW * CV;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total;
       i += (size_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % CV) * V;
    size_t p = i / CV;
    const int ox = p % OW; p /= OW;
    const int oy = p % OH;
    const int b = p / OH;
    float acc[V];
#pragma unroll
    for (int q = 0; q < V; ++q) acc[q] = 0.f;
    const int iy_hi = (oy + pad) / f, ix_hi = (ox + pad) / f;
#pragma unroll
    for (int dy = 0; dy < 2; ++dy) {
      const int iy = iy_hi - dy;
      const int ky = oy + pad - iy * f;
      if (iy < 0 || iy >= H || ky >= k) continue;
#pragma unroll
      for (int dx = 0; dx < 2; ++dx) {
        const int ix = ix_hi - dx;
        const int kx = ox + pad - ix * f;
        if (ix < 0 || ix >= W || kx >= k) continue;
        float xv[V], wv[V];
        VecIO<T>::ld(x + (((size_t)b * H + iy) * W + ix) * ld_in + c, xv);
        const float* wp = w + ((size_t)ky * k + kx) * C + c;
#pragma unroll
        for (int q = 0; q < V; q += 4) {
          const float4 t = __ldg(reinterpret_cast<const float4*>(wp + q));
          wv[q] = t.x; wv[q + 1] = t.y; wv[q + 2] = t.z; wv[q + 3] = t.w;
        }
#pragma unroll
        for (int q = 0; q < V; ++q) acc[q] = fmaf(xv[q], wv[q], acc[q]);
      }
    }
    const size_t op = ((size_t)b * OH + oy) * OW + ox;
    if (skip) {
      float sv[V];
      VecIO<T>::ld(skip + op * ld_skip + c, sv);
#pragma unroll
      for (int q = 0; q < V; ++q) acc[q] += sv[q];
    }
    VecIO<T>::st(out + op * ld_out + c, acc);
  }
}

// Same operator, weights held in registers: an output pixel's 2x2 taps depend only on its phase (oy mod f, ox mod f),
// so blockIdx.y = phase, a thread keeps one channel vector's 4 x V tap weights for its whole lifetime and walks the
// pixels of that phase (8 lanes x 16 B = one 128-byte line per pixel at C = 64): 4 input loads + 1 skip load per
// output vector instead of 4 + 8 weight loads + 1.  Accumulation order = upsample_add_kernel's (bit-identical).
template <typename T>
__global__ void __launch_bounds__(256)
upsample_add_phase_kernel(const T* __restrict__ x, const T* __restrict__ skip, const float* __restrict__ w,
                          T* __restrict__ out, int B, int H, int W, int C, int f, int ld_in, int ld_skip, int ld_out) {
  constexpr int V = VecIO<T>::N;
  const int OW = W * f, OH = H * f, pad = f / 2, k = 2 * f, CV = C / V;
  const int py = blockIdx.y / f, px = blockIdx.y - py * f;
  const int cg = threadIdx.x % CV, c = cg * V;
  const int dyh = (py + pad) / f, ky0 = (py + pad) - dyh * f;     // taps: (iy = m + dyh, ky0), (iy - 1, ky0 + f)
  const int dxh = (px + pad) / f, kx0 = (px + pad) - dxh * f;
  float wr[2][2][V];
#pragma unroll
  for (int dy = 0; dy < 2; ++dy)
#pragma unroll
    for (int dx = 0; dx < 2; ++dx) {
      const int ky = ky0 + dy * f, kx = kx0 + dx * f;
      const float* wp = w + ((size_t)ky * k + kx) * C + c;
#pragma unroll
      for (int q = 0; q < V; q += 4) {
        const float4 t = __ldg(reinterpret_cast<const float4*>(wp + q));
        wr[dy][dx][q] = t.x; wr[dy][dx][q + 1] = t.y; wr[dy][dx][q + 2] = t.z; wr[dy][dx][q + 3] = t.w;
      }
    }
  const int slots = blockDim.x / CV;
  const int total = B * H * W;
  for (int j = blockIdx.x * slots + threadIdx.x / CV; j < total; j += gridDim.x * slots) {
    const int n = j % W;
    const int t = j / W;
    const int m = t % H, b = t / H;
    const int oy = m * f + py, ox = n * f + px;
    float acc[V];
#pragma unroll
    for (int q = 0; q < V; ++q) acc[q] = 0.f;
#pragma unroll
    for (int dy = 0; dy < 2; ++dy) {
      const int iy = m + dyh - dy;
      if (iy < 0 || iy >= H) continue;
#pragma unroll
      for (int dx = 0; dx < 2; ++dx) {
        const int ix = n + dxh - dx;
        if (ix < 0 || ix >= W) continue;
        float xv[V];
        VecIO<T>::ld(x + (((size_t)b * H + iy) * W + ix) * ld_in + c, xv);
#pragma unroll
        for (int q = 0; q < V; ++q) acc[q] = fmaf(xv[q], wr[dy][dx][q], acc[q]);
      }
    }
    const size_t op = ((size_t)b * OH + oy) * OW + ox;
    if (skip) {
      float sv[V];
      VecIO<T>::ld(skip + op * ld_skip + c, sv);
#pragma unroll
      for (int q = 0; q < V; ++q) acc[q] += sv[q];
    }
    VecIO<T>::st(out + op * ld_out + c, acc);
  }
}

// Same operator again, all f*f phases of an input pixel inside ONE warp / CTA: slot (= thread / channel vectors) % f*f is
// the thread's phase (weights in registers as above), slot / f*f walks the INPUT pixels.  The 2x2 taps of the f*f
// phases of neighbouring input pixels touch the same 3x3 input lines, which now hit in L1 instead of being fetched
// from L2 by f*f different CTAs (the phase kernel moved ~6x the output bytes over the L2 -> SM fabric: 64 us for a
// 151 MB layer), and the f output pixels of a row are adjacent 16-byte-vector groups: one contiguous f*C*2-byte store.
// Accumulation order = upsample_add_kernel's (bit-identical).
template <typename T>
__global__ void __launch_bounds__(256)
upsample_add_warp_kernel(const T* __restrict__ x, const T* __restrict__ skip, const float* __restrict__ w,
                         T* __restrict__ out, int B, int H, int W, int C, int f, int ld_in, int ld_skip, int ld_out) {
  constexpr int V = VecIO<T>::N;
  const int OW = W * f, OH = H * f, pad = f / 2, k = 2 * f, CV = C / V, ff = f * f;
  const int slot = threadIdx.x / CV, cg = threadIdx.x - slot * CV, c = cg * V;
  const int phase = slot % ff, sub = slot / ff;
  const int py = phase / f, px = phase - py * f;
  const int dyh = (py + pad) / f, ky0 = (py + pad) - dyh * f;     // taps: (iy = m + dyh, ky0), (iy - 1, ky0 + f)
  const int dxh = (px + pad) / f, kx0 = (px + pad) - dxh * f;
  float wr[2][2][V];
#pragma unroll
  for (int dy = 0; dy < 2; ++dy)
#pragma unroll
    for (int dx = 0; dx < 2; ++dx) {
      const int ky = ky0 + dy * f, kx = kx0 + dx * f;
      const float* wp = w + ((size_t)ky * k + kx) * C + c;
#pragma unroll
      for (int q = 0; q < V; q += 4) {
        const float4 t = __ldg(reinterpret_cast<const float4*>(wp + q));
        wr[dy][dx][q] = t.x; wr[dy][dx][q + 1] = t.y; wr[dy][dx][q + 2] = t.z; wr[dy][dx][q + 3] = t.w;
      }
    }
  // Index arithmetic is 32-bit and incremental (the host checks that every tensor has < 2^31 elements): (b, m, n) advance
  // by the constant grid stride with carries instead of two divisions per pixel, and the four taps are constant element
  // offsets from one base -- the integer work was 4x the 32 FMAs of an output vector (ncu: issue slots 55-60 % busy at
  // 21 % of the DRAM bandwidth).
  const int per_cta = (blockDim.x / CV) / ff;                      // input pixels per CTA per iteration
  const int total = B * H * W;
  const int stride = gridDim.x * per_cta;
  const int s_n = stride % W, s_t = stride / W;                    // stride = s_t * W + s_n, s_t rows (over b, m)
  int j = blockIdx.x * per_cta + sub;
  int n = j % W, t = j / W;                                        // t = b * H + m
  int m = t % H;
  const int s_m = s_t % H;
  const int tap_off[2][2] = {{(dyh * W + dxh) * ld_in, (dyh * W + dxh - 1) * ld_in},
                             {((dyh - 1) * W + dxh) * ld_in, ((dyh - 1) * W + dxh - 1) * ld_in}};
  const T* xc = x + c;
  const T* sc = skip ? skip + c : nullptr;
  T* oc = out + c;
  for (; j < total; j += stride) {
    // the four tap loads and the skip load are issued together (no branch between them: a tap outside the image reads
    // the centre pixel instead and contributes through a zero -- fma(0, w, acc) == acc, so the result is unchanged)
    const int in_base = (t * W + n) * ld_in;
    const int op = (t * f + py) * OW + n * f + px;                 // ((b * OH + oy) * OW + ox), oy = m f + py
    uint4 raw[2][2], raw_s = make_uint4(0, 0, 0, 0);
    if (sc) raw_s = ld_raw16(sc + op * ld_skip);                   // the DRAM stream first
#pragma unroll
    for (int dy = 0; dy < 2; ++dy)
#pragma unroll
      for (int dx = 0; dx < 2; ++dx) {
        const bool ok = (unsigned)(m + dyh - dy) < (unsigned)H && (unsigned)(n + dxh - dx) < (unsigned)W;
        raw[dy][dx] = ld_raw16(xc + (in_base + (ok ? tap_off[dy][dx] : 0)));
        if (!ok) raw[dy][dx] = make_uint4(0, 0, 0, 0);             // +0.0 in both dtypes
      }
    float acc[V];
#pragma unroll
    for (int q = 0; q < V; ++q) acc[q] = 0.f;
#pragma unroll
    for (int dy = 0; dy < 2; ++dy)
#pragma unroll
      for (int dx = 0; dx < 2; ++dx) {
        float xv[V];
        cvt_raw16(raw[dy][dx], xv);
#pragma unroll
        for (int q = 0; q < V; ++q) acc[q] = fmaf(xv[q], wr[dy][dx][q], acc[q]);
      }
    if (sc) {
      float sv[V];
      cvt_raw16(raw_s, sv);
#pragma unroll
      for (int q = 0; q < V; ++q) acc[q] += sv[q];
    }
    VecIO<T>::st(oc + op * ld_out, acc);
    n += s_n; t += s_t; m += s_m;
    if (n >= W) { n -= W; ++t; ++m; }
    while (m >= H) m -= H;
  }
}

// ------------------------------------------------------------------------------------------
// pre_hm splat: draw_umich_gaussian image.py:128-154 (gaussian2D in float64, np.maximum)
// ------------------------------------------------------------------------------------------
__global__ void render_pre_hm_kernel(const float* __restrict__ boxes, int n, float* __restrict__ hm,
                                     int B, int H, int W) {
  const int i = blockIdx.x;
  if (i >= n) return;
  const int b = (int)boxes[i * 5 + 0], cx = (int)boxes[i * 5 + 1], cy = (int)boxes[i * 5 + 2];
  const int r = (int)boxes[i * 5 + 3];
  if (b < 0 || b >= B) return;
  const double sigma = (double)(2 * r + 1) / 6.0;
  const int left = min(cx, r), right = min(W - cx, r + 1), top = min(cy, r), bottom = min(H - cy, r + 1);
  const int w = left + right, h = top + bottom;
  if (w <= 0 || h <= 0) return;
  for (int j = threadIdx.x; j < w * h; j += blockDim.x) {
    const int yy = j / w - top, xx = j % w - left;
    double v = exp(-(double)(xx * xx + yy * yy) / (2.0 * sigma * sigma));
    if (v < 2.220446049250313e-16) v = 0.0;
    const float fv = (float)v;
    atomicMax(reinterpret_cast<int*>(hm + ((size_t)b * H + cy + yy) * W + cx + xx), __float_as_int(fv));
  }
}

}  // namespace ctb

using namespace ctb;

extern "C" int ct_stem_forward(const float* img, const float* pre_img, const float* pre_hm, const float* w,
                               const float* shift, void* out, int32_t dtype, int32_t B, int32_t H,
                               int32_t W, int32_t ld_out, void* stream) {
  CT_REQUIRE(img && w && shift && out, "null pointer");
  CT_REQUIRE(B > 0 && H > 0 && W > 0 && ld_out >= 16, "bad shape");
  dim3 grid((W + ST - 1) / ST, (H + ST - 1) / ST, B);
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == CT_F32)
    stem_kernel<float><<<grid, ST * ST, 0, st>>>(img, pre_img, pre_hm, w, shift, (float*)out, B, H, W, ld_out);
  else
    stem_kernel<__nv_bfloat16><<<grid, ST * ST, 0, st>>>(img, pre_img, pre_hm, w, shift,
                                                         (__nv_bfloat16*)out, B, H, W, ld_out);
  return after_launch();
}

static inline int ew_blocks(size_t total);

extern "C" int ct_pack_stem_input(const float* img, const float* pre_img, const float* pre_hm, void* out,
                                  int32_t B, int32_t H, int32_t W, void* stream) {
  CT_REQUIRE(img && out, "null pointer");
  CT_REQUIRE(B > 0 && H > 0 && W > 0, "bad shape");
  const size_t total = (size_t)B * H * W;
  pack_stem_kernel<<<ew_blocks(total), 256, 0, (cudaStream_t)stream>>>(img, pre_img, pre_hm, (uint4*)out, B, H, W);
  return after_launch();
}

extern "C" int ct_pack_stem_input_f32(const float* img, const float* pre_img, const float* pre_hm, float* out,
                                      int32_t B, int32_t H, int32_t W, void* stream) {
  CT_REQUIRE(img && out, "null pointer");
  CT_REQUIRE(B > 0 && H > 0 && W > 0, "bad shape");
  const size_t total = (size_t)B * H * W;
  pack_stem_f32_kernel<<<ew_blocks(total), 256, 0, (cudaStream_t)stream>>>(img, pre_img, pre_hm, (float4*)out, B, H, W);
  return after_launch();
}

static inline int ew_blocks(size_t total) {
  size_t b = (total + 255) / 256;
  return (int)(b < 148 * 16 ? (b ? b : 1) : 148 * 16);
}

extern "C" int ct_maxpool2(const void* x, void* out, int32_t dtype, int32_t B, int32_t H, int32_t W,
                           int32_t C, int32_t ld_in, int32_t ld_out, void* stream) {
  CT_REQUIRE(x && out, "null pointer");
  CT_REQUIRE(H % 2 == 0 && W % 2 == 0, "odd spatial size");
  const int vecw = dtype == CT_F32 ? 4 : 8;
  CT_REQUIRE(C % vecw == 0 && ld_in % vecw == 0 && ld_out % vecw == 0, "channels / strides must be multiples of 16 bytes");
  const size_t total = (size_t)B * (H / 2) * (W / 2) * (C / vecw);
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == CT_F32)
    maxpool2_kernel<float><<<ew_blocks(total), 256, 0, st>>>((const float*)x, (float*)out, B, H, W, C, ld_in, ld_out);
  else
    maxpool2_kernel<__nv_bfloat16><<<ew_blocks(total), 256, 0, st>>>(
        (const __nv_bfloat16*)x, (__nv_bfloat16*)out, B, H, W, C, ld_in, ld_out);
  return after_launch();
}

// MaxPool2d(2,2) of a tensor stored space-to-depth ([B, H2, W2, (sy, sx, C)], CT_OUT_NHWC_S2D): the window of output pixel
// p is the four C-channel groups of input pixel p -- a per-pixel max over channel groups, one 16-byte vector per thread.
template <typename T>
__global__ void maxpool2_s2d_kernel(const T* __restrict__ x, T* __restrict__ out, size_t P, int C, int ld_in, int ld_out) {
  constexpr int V = VecIO<T>::N;
  const int CV = C / V;
  const size_t total = P * CV;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % CV) * V;
    const size_t p = i / CV;
    const T* s = x + p * ld_in + c;
    float v0[V], v1[V], v2[V], v3[V];
    VecIO<T>::ld(s, v0); VecIO<T>::ld(s + C, v1); VecIO<T>::ld(s + 2 * C, v2); VecIO<T>::ld(s + 3 * C, v3);
#pragma unroll
    for (int q = 0; q < V; ++q) v0[q] = fmaxf(fmaxf(v0[q], v1[q]), fmaxf(v2[q], v3[q]));
    VecIO<T>::st(out + p * ld_out + c, v0);
  }
}

extern "C" int ct_maxpool2_s2d(const void* x, void* out, int32_t dtype, int32_t B, int32_t H2, int32_t W2, int32_t C,
                               int32_t ld_in, int32_t ld_out, void* stream) {
  CT_REQUIRE(x && out, "null pointer");
  const int vecw = dtype == CT_F32 ? 4 : 8;
  CT_REQUIRE(C % vecw == 0 && ld_in % vecw == 0 && ld_out % vecw == 0 && ld_in >= 4 * C,
             "channels / strides must be multiples of 16 bytes, ld_in >= 4 C");
  const size_t P = (size_t)B * H2 * W2, total = P * (C / vecw);
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == CT_F32)
    maxpool2_s2d_kernel<float><<<ew_blocks(total), 256, 0, st>>>((const float*)x, (float*)out, P, C, ld_in, ld_out);
  else
    maxpool2_s2d_kernel<__nv_bfloat16><<<ew_blocks(total), 256, 0, st>>>((const __nv_bfloat16*)x, (__nv_bfloat16*)out, P, C,
                                                                        ld_in, ld_out);
  return after_launch();
}

extern "C" int ct_upsample_add(const void* x, const void* skip, const float* w, void* out, int32_t dtype,
                               int32_t B, int32_t H, int32_t W, int32_t C, int32_t f, int32_t ld_in,
                               int32_t ld_skip, int32_t ld_out, void* stream) {
  CT_REQUIRE(x && w && out, "null pointer");
  CT_REQUIRE(f == 2 || f == 4 || f == 8, "unsupported upsample factor");
  const int vec = dtype == CT_F32 ? 4 : 8;
  CT_REQUIRE(C % vec == 0 && ld_in % vec == 0 && ld_out % vec == 0 && (skip == nullptr || ld_skip % vec == 0),
             "channels / strides must be multiples of the 16-byte vector width");
  const size_t total = (size_t)B * H * f * W * f * (C / vec);
  cudaStream_t st = (cudaStream_t)stream;
  const int cv = C / vec;
  if (cv <= 256 && 256 % cv == 0 && (256 / cv) % (f * f) == 0 &&
      (size_t)B * H * f * W * f * (size_t)(ld_out > ld_skip ? ld_out : ld_skip) < (1ull << 31) && (size_t)B * H * W * ld_in < (1ull << 31)) {
    // all phases of an input pixel in one CTA (L1 reuse of the taps); grid: a few CTAs per SM, grid-stride over pixels
    const int per_cta = (256 / cv) / (f * f);
    long gx = ((long)B * H * W + per_cta - 1) / per_cta;
    if (gx > 148 * 8) gx = 148 * 8;
    if (dtype == CT_F32)
      upsample_add_warp_kernel<float><<<(int)gx, 256, 0, st>>>(
          (const float*)x, (const float*)skip, w, (float*)out, B, H, W, C, f, ld_in, ld_skip, ld_out);
    else
      upsample_add_warp_kernel<__nv_bfloat16><<<(int)gx, 256, 0, st>>>(
          (const __nv_bfloat16*)x, (const __nv_bfloat16*)skip, w, (__nv_bfloat16*)out, B, H, W, C, f,
          ld_in, ld_skip, ld_out);
    return after_launch();
  }
  if (cv <= 256 && 256 % cv == 0 && (size_t)B * H * W < (1u << 30)) {
    // phase kernel: grid.y = f*f phases, grid.x sized so that all phases together fill the GPU a few times over
    const int slots = 256 / cv;
    int gx = (int)(((size_t)B * H * W + slots - 1) / slots);
    const int cap = (148 * 8 + f * f - 1) / (f * f);
    if (gx > cap) gx = cap;
    if (gx < 1) gx = 1;
    dim3 grid(gx, f * f);
    if (dtype == CT_F32)
      upsample_add_phase_kernel<float><<<grid, 256, 0, st>>>(
          (const float*)x, (const float*)skip, w, (float*)out, B, H, W, C, f, ld_in, ld_skip, ld_out);
    else
      upsample_add_phase_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>(
          (const __nv_bfloat16*)x, (const __nv_bfloat16*)skip, w, (__nv_bfloat16*)out, B, H, W, C, f,
          ld_in, ld_skip, ld_out);
    return after_launch();
  }
  if (dtype == CT_F32)
    upsample_add_kernel<float><<<ew_blocks(total), 256, 0, st>>>(
        (const float*)x, (const float*)skip, w, (float*)out, B, H, W, C, f, ld_in, ld_skip, ld_out);
  else
    upsample_add_kernel<__nv_bfloat16><<<ew_blocks(total), 256, 0, st>>>(
        (const __nv_bfloat16*)x, (const __nv_bfloat16*)skip, w, (__nv_bfloat16*)out, B, H, W, C, f,
        ld_in, ld_skip, ld_out);
  return after_launch();
}

extern "C" int ct_render_pre_hm(const float* boxes, int32_t n, float* pre_hm, int32_t B, int32_t H,
                                int32_t W, void* stream) {
  CT_REQUIRE(pre_hm, "null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  CT_CUDA_OK(cudaMemsetAsync(pre_hm, 0, (size_t)B * H * W * sizeof(float), st));
  if (n <= 0) return CT_OK;
  CT_REQUIRE(boxes, "null boxes");
  render_pre_hm_kernel<<<n, 256, 0, st>>>(boxes, n, pre_hm, B, H, W);
  return after_launch();
}
