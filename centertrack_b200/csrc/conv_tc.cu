// tcgen05 implicit-GEMM convolution / DCNv2 for sm_100a (bf16 operands, fp32 accumulate in TMEM).
//
//   D[128 pixels x n_tile channels] (TMEM)  +=  A[128 x 64] (smem, gathered)  x  B[n_tile x 64]^T (smem)
//
// * No im2row buffer in HBM: producer warps gather each 64-wide K slice (tap-major, k = tap*C_in + c)
//   of the A operand straight into the 128B-swizzled K-major shared-memory layout the UMMA smem
//   descriptor expects.  For CT_A_DCN the gather is the DCNv2 bilinear sample x mask (the reference's
//   `columns` tensor never exists).
// * Weights are pre-packed on the host as ready-made swizzled tile images, so one TMA bulk copy
//   (cp.async.bulk, mbarrier complete_tx) per K slice brings the B tile.
// * One elected thread issues tcgen05.mma (M=128, N=n_tile, K=16) x4 per slice; tcgen05.commit
//   releases the smem stage back to the producers and finally signals the epilogue.
// * Epilogue: tcgen05.ld (32 lanes x 16 columns per warp), + folded-BN shift, + residual, ReLU,
//   then bf16 NHWC / fp32 NHWC (DCN offsets, sigmoid on the mask channels) / fp32 NCHW (heads,
//   sigmoid / depth transform) stores.
//
// CTA = 288 threads: warps 0-7 producers then epilogue (warp w reads TMEM lanes 32(w%4).., warps 0-3 the even
// 16-column chunks, warps 4-7 the odd ones), warp 8 = TMEM allocator + MMA issuer.  Eight producer warps
// (two per SM sub-partition) because the gather is latency-bound: more warps = more loads in flight.
// Two CTAs are co-resident per SM so one CTA's epilogue overlaps another's main loop.
#include "conv_common.cuh"
#include "sm100.cuh"

namespace ctb {

constexpr int TC_BM = 128;           // output pixels per CTA (UMMA M)
constexpr int TC_BK = 64;            // K elements per pipeline stage (one 128B swizzle atom of bf16)
constexpr int TC_THREADS = 288;        // 8 producer/epilogue warps + 1 MMA warp
constexpr int TC_PRODUCERS = 256;
constexpr int TC_NROW = TC_BM * 8 / TC_PRODUCERS;   // A-tile rows per producer thread per K slice (4)
constexpr int A_STAGE_BYTES = TC_BM * 128;
// CT_A_DCN_WIN: pixels of offset margin staged around a patch's 3x3 footprint (samples that leave it read global memory).
// Margins 1 / 2 / 3 measured on B200: 2 is fastest (DESIGN.md).
constexpr int DCN_WIN_MARGIN = 2;

struct TcArgs {
  ConvGeom g;
  const __nv_bfloat16* x;       // X3 engine: fp32 activations behind the same pointers (xf() / residual_f())
  const __nv_bfloat16* w;       // packed tiles (X3: [hi tile][lo tile] per K slice)
  const float* shift;
  const __nv_bfloat16* residual;
  const float* om;
  void* out;
  int n_tile, k_slices, stages, tmem_cols, a_mode;
  int tiles_x, tiles_y;         // CT_A_DCN_WIN: an M tile is an 8 (y) x 16 (x) pixel patch of one image;
                                // 0: 128 consecutive pixels in b,y,x order
  int win_m, win_pw, win_ph;    // CT_A_DCN_WIN: offset margin (px) and the staged window (pixels) of one 8x16 patch
  uint32_t win_bytes;           // bytes of one 64-channel window (= TMA box)
};

// CT_A_DCN_WIN sampling record (16 bytes): global fall-back offset of the clamped top-left corner (channel 0 of the
// chunk is added by the reader), window-relative location + flags, and the four mask-scaled bilinear weights in bf16.
// The blend runs in packed bf16 (fma.rn.bf16x2: four roundings per sample instead of one): measured with the oracle
// on the full network this moves the end-to-end error of the bf16 engine by 1 % of itself (0.0340 -> 0.0344 relative
// rms at the 64-channel feature) and removes 60 % of the producer's instructions (no unpack, no fp32->bf16 pack).
struct __align__(16) DcnWinEntry { int goff; uint32_t meta; uint32_t w01, w23; };
constexpr uint32_t WIN_DX = 1u << 16, WIN_DY = 1u << 17, WIN_IN = 1u << 18;

__device__ __forceinline__ uint4 lds16(uint32_t addr) {
  uint4 r;
  asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "r"(addr));
  return r;
}

// output pixel (linear b,y,x index) of GEMM row r of M tile mt; g.P_out when the row is padding
__device__ __forceinline__ int tc_pixel(const TcArgs& a, int mt, int r) {
  const ConvGeom& g = a.g;
  if (a.tiles_x == 0) { const int p = mt * TC_BM + r; return p < g.P_out ? p : g.P_out; }
  const int tpi = a.tiles_x * a.tiles_y;
  const int b = mt / tpi, t = mt - b * tpi;
  const int ty = t / a.tiles_x, tx = t - ty * a.tiles_x;
  const int oy = ty * 8 + (r >> 4), ox = tx * 16 + (r & 15);
  return (oy < g.OH && ox < g.OW) ? (b * g.OH + oy) * g.OW + ox : g.P_out;
}

// Optional timeline of the middle CTA (ct_debug_trace): clock64() stamps -- 0 start, 1 rows set up, 2 DCN table built,
// 8+s producer warp 0 finished slice s, 4 MMA warp committed, 5 epilogue saw the accumulator, 6 epilogue done.
__device__ unsigned long long* g_tc_trace = nullptr;
// The pointer is read ONCE per thread at kernel entry (tc_trace_ptr): a stamp that re-read the global cost the stamping
// thread a dependent load per slice even with tracing off.
__device__ __forceinline__ unsigned long long* tc_trace_ptr() {
  unsigned long long* t = g_tc_trace;
  return (t != nullptr && blockIdx.x == gridDim.x / 2 && blockIdx.y == 0) ? t : nullptr;
}
__device__ __forceinline__ void tc_stamp(unsigned long long* t, int k) {
  if (t != nullptr && k < 256) t[k] = (unsigned long long)clock64();
}

__device__ __forceinline__ uint4 ldg_nc16(const void* p) {
  uint4 r;
  asm volatile("ld.global.nc.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
  return r;
}
__device__ __forceinline__ void sts16(uint32_t addr, uint4 v) {
  asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

// Per (tap, output pixel) DCNv2 sampling record, built once per CTA: clamped top-left corner as a 32-bit element
// offset (image base included, channel 0), element strides to the x+1 / y+1 corners (0 when that neighbour is
// outside the image, so every load address is valid and the loads need no predicate), and the four bilinear
// weights already multiplied by the modulation mask and zeroed for corners / samples outside the image.
struct __align__(16) DcnEntry { int off, dxo, dyo, pad; float w00, w01, w10, w11; };   // 32 bytes

// bf16x2 word -> two fp32 lanes of one 64-bit register (lo = x << 16, hi = x & 0xffff0000: one ALU op each), then
// packed fp32 math (FMUL2 / FFMA2): 8 channels x 1 corner = 8 unpack + 4 packed FMAs.
__device__ __forceinline__ unsigned long long bf2_to_f2(uint32_t x) {
  unsigned long long r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "r"(x << 16), "r"(x & 0xffff0000u));
  return r;
}
__device__ __forceinline__ unsigned long long dup_f2(float w) {
  unsigned long long r;
  asm("mov.b64 %0, {%1, %1};" : "=l"(r) : "r"(__float_as_uint(w)));
  return r;
}
__device__ __forceinline__ void scale8(unsigned long long (&acc)[4], uint4 v, float w) {
  const unsigned long long ww = dup_f2(w);
  const uint32_t x[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
  for (int q = 0; q < 4; ++q) asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(acc[q]) : "l"(bf2_to_f2(x[q])), "l"(ww));
}
__device__ __forceinline__ void blend8(unsigned long long (&acc)[4], uint4 v, float w) {
  const unsigned long long ww = dup_f2(w);
  const uint32_t x[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
  for (int q = 0; q < 4; ++q) asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(acc[q]) : "l"(bf2_to_f2(x[q])), "l"(ww));
}
__device__ __forceinline__ uint32_t bmul2(uint32_t a, uint32_t b) {
  uint32_t d;
  asm("mul.rn.bf16x2 %0, %1, %2;" : "=r"(d) : "r"(a), "r"(b));
  return d;
}
__device__ __forceinline__ uint32_t bfma2(uint32_t a, uint32_t b, uint32_t c) {
  uint32_t d;
  asm("fma.rn.bf16x2 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
  return d;
}
__device__ __forceinline__ uint32_t dup_bf2(float w) {      // {bf16(w), bf16(w)}
  uint32_t d;
  asm("cvt.rn.bf16x2.f32 %0, %1, %1;" : "=r"(d) : "f"(w));
  return d;
}
__device__ __forceinline__ uint4 pack8(const unsigned long long (&acc)[4]) {
  uint32_t o[4];
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    uint32_t lo, hi;
    asm("mov.b64 {%0, %1}, %2;" : "=r"(lo), "=r"(hi) : "l"(acc[q]));
    const __nv_bfloat162 h = __floats2bfloat162_rn(__uint_as_float(lo), __uint_as_float(hi));
    o[q] = *reinterpret_cast<const uint32_t*>(&h);
  }
  return make_uint4(o[0], o[1], o[2], o[3]);
}

// ---- bf16x3 ("X3") engine: fp32 activations, every operand split into bf16 hi + bf16 lo = x - hi (both exact in
// fp32), and D += A_hi B_hi + A_hi B_lo + A_lo B_hi on the tensor cores with fp32 accumulation: the dropped
// A_lo B_lo term and the rounding of lo are ~2^-16 / 2^-17 relative, i.e. ~1e-5 per layer instead of bf16's 4e-3.
__device__ __forceinline__ void split8(const float4 lo4, const float4 hi4, uint4& h, uint4& l) {
  const float f[8] = {lo4.x, lo4.y, lo4.z, lo4.w, hi4.x, hi4.y, hi4.z, hi4.w};
  uint32_t hh[4], ll[4];
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    const __nv_bfloat162 hp = __floats2bfloat162_rn(f[2 * q], f[2 * q + 1]);
    const float2 hf = __bfloat1622float2(hp);
    const __nv_bfloat162 lp = __floats2bfloat162_rn(f[2 * q] - hf.x, f[2 * q + 1] - hf.y);
    hh[q] = *reinterpret_cast<const uint32_t*>(&hp);
    ll[q] = *reinterpret_cast<const uint32_t*>(&lp);
  }
  h = make_uint4(hh[0], hh[1], hh[2], hh[3]);
  l = make_uint4(ll[0], ll[1], ll[2], ll[3]);
}
__device__ __forceinline__ float4 ldg_nc_f4(const float* p) {
  float4 r;
  asm volatile("ld.global.nc.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p));
  return r;
}

template <bool X3>
__global__ void __launch_bounds__(TC_THREADS, X3 ? 1 : 2)
conv_tc_kernel(const TcArgs a, const __grid_constant__ CUtensorMap tmap) {
  extern __shared__ __align__(1024) unsigned char smem_dyn[];
  // SWIZZLE_128B operands need 1024B-aligned stage bases: align by hand (launch adds 1 KB of slack)
  unsigned char* smem = smem_dyn + ((1024u - (smem_u32(smem_dyn) & 1023u)) & 1023u);
  const ConvGeom& g = a.g;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  unsigned long long* const trace = tc_trace_ptr();
  const int S = a.stages;
  const uint32_t b_tile_bytes = (uint32_t)a.n_tile * 128u;                    // one bf16 weight tile of a K slice
  const uint32_t b_stage_bytes = X3 ? 2u * b_tile_bytes : b_tile_bytes;       // X3: [hi][lo]
  constexpr uint32_t a_stage_bytes = X3 ? 2u * A_STAGE_BYTES : A_STAGE_BYTES; // X3: [hi 16 KB][lo 16 KB]
  const float* xf = reinterpret_cast<const float*>(a.x);

  // carve shared memory
  const uint32_t smem_base = smem_u32(smem);
  const uint32_t sA = smem_base;
  const uint32_t sB = sA + S * a_stage_bytes;
  const uint32_t off_bar = S * a_stage_bytes + S * b_stage_bytes;
  const uint32_t bars = smem_base + off_bar;           // full[S], empty[S], tmem_full, win_full
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + off_bar + (2 * S + 2) * 8);
  DcnEntry* dcn_tab = reinterpret_cast<DcnEntry*>(smem + off_bar + (2 * S + 2) * 8 + 16);  // 16B aligned
  auto full_bar = [&](int s) { return bars + 8u * s; };
  auto empty_bar = [&](int s) { return bars + 8u * (S + s); };
  const uint32_t tmem_full_bar = bars + 8u * (2 * S);
  const uint32_t win_bar = bars + 8u * (2 * S + 1);
  const bool win = !X3 && a.a_mode == CT_A_DCN_WIN;
  // CT_A_DCN_WIN: [table 9 x 128 x 16 B][window, 128B aligned]
  DcnWinEntry* win_tab = reinterpret_cast<DcnWinEntry*>(dcn_tab);
  const uint32_t s_win = (smem_u32(dcn_tab) + 9u * TC_BM * 16u + 127u) & ~127u;

  const int mt = blockIdx.x;
  const int nt = blockIdx.y;
  const int n0 = nt * a.n_tile;
  if (tid == 0) tc_stamp(trace, 0);
  pdl_trigger();                       // the next kernel of the stream may start its own prologue now

  if (tid == 0) {
    for (int s = 0; s < S; ++s) { mbarrier_init(full_bar(s), TC_PRODUCERS / 32); mbarrier_init(empty_bar(s), 1); }
    mbarrier_init(tmem_full_bar, 1);
    mbarrier_init(win_bar, 1);
    fence_mbarrier_init();
  }
  if (warp == 8) {
    tcgen05_alloc(smem_u32((const void*)tmem_slot), (uint32_t)a.tmem_cols);
    tcgen05_relinquish_alloc_permit();
  }
  tcgen05_fence_before_thread_sync();
  __syncthreads();
  tcgen05_fence_after_thread_sync();
  const uint32_t tmem_base = *tmem_slot;
  if (tid == 0) tc_stamp(trace, 7);
  pdl_wait();                          // everything below reads what the previous kernel wrote

  if (warp < 8) {
    // =========================== A producers ===========================
    const int q = tid & 7;                 // 16-byte chunk (8 channels) inside the 64-wide K slice
    const int r0 = tid >> 3;               // rows r0 + 32*i, i < TC_NROW
    const uint32_t swz = (uint32_t)((q ^ (r0 & 7)) << 4);
    const int HWo = g.OH * g.OW;
    int row_off[TC_NROW], row_iy[TC_NROW], row_ix[TC_NROW];   // element offset / coords of the window's top-left input pixel
    if (a.a_mode != CT_A_CONV) {
      // DCN rows come from the sampling table
#pragma unroll
      for (int i = 0; i < TC_NROW; ++i) { row_off[i] = 0; row_iy[i] = -100000; row_ix[i] = -100000; }
    } else {
      // linear tiles: one division pair for the first row, the other rows (+32 pixels each) by carry propagation
      int p = mt * TC_BM + r0;
      int b = p / HWo, r = p - b * HWo;
      int oy = r / g.OW, ox = r - oy * g.OW;
#pragma unroll
      for (int i = 0; i < TC_NROW; ++i) {
        if (p < g.P_out) {
          row_iy[i] = oy * g.stride - g.pad;
          row_ix[i] = ox * g.stride - g.pad_w;
          row_off[i] = (b * g.H * g.W + row_iy[i] * g.W + row_ix[i]) * g.ld_in;
        } else {
          row_off[i] = 0; row_iy[i] = -100000; row_ix[i] = -100000;
        }
        p += 32; ox += 32;
        while (ox >= g.OW) { ox -= g.OW; ++oy; }
        while (oy >= g.OH) { oy -= g.OH; ++b; }
      }
    }
    if (tid == 0) tc_stamp(trace, 1);
    int win_x0 = 0, win_y0 = 0, win_b = 0;
    if (win) {
      // window origin of this 8x16 patch: one kernel-halo pixel + the offset margin to the top/left
      const int tpi = a.tiles_x * a.tiles_y;
      win_b = mt / tpi;
      const int t = mt - win_b * tpi;
      const int ty = t / a.tiles_x, tx = t - ty * a.tiles_x;
      win_y0 = ty * 8 - 1 - a.win_m;
      win_x0 = tx * 16 - 1 - a.win_m;
      if (tid == 0) {                                   // first 64-channel chunk of the window: TMA, zero fill outside
        mbarrier_arrive_expect_tx(win_bar, a.win_bytes);      // count 1: this arrival + the TMA's bytes complete the phase
        cp_async_bulk_tensor_4d(s_win, &tmap, 0, win_x0, win_y0, win_b, win_bar);
      }
      // Two threads per row (taps 0-4 and 5-8) so that all eight producer warps build the table.  The 27 offset / mask
      // floats of a row sit in one 128-byte line of `om`; each thread loads only the 16-byte chunks its taps need.
      const int trow = tid & (TC_BM - 1), thalf = tid >> 7;            // thalf 0: taps 0..4, thalf 1: taps 5..8
      const int tap0 = thalf ? 5 : 0, tap1 = thalf ? 9 : 5;
      const int tp = tc_pixel(a, mt, trow);
      const bool ok = tp < g.P_out;
      {
        int oy = 0, ox = 0, img = 0;
        float om[28];
#pragma unroll
        for (int j = 0; j < 28; ++j) om[j] = 0.f;
        if (ok) {
          const int bb = tp / HWo, r = tp - bb * HWo;
          oy = r / g.OW; ox = r - oy * g.OW; img = bb * g.H * g.W;
          const float4* omp = reinterpret_cast<const float4*>(a.om + (size_t)tp * g.ld_om);
          // floats [2 tap0, 2 tap1) and [18 + tap0, 18 + tap1): chunks 0-2, 4-5 (thalf 0) / 2-6 (thalf 1)
#pragma unroll
          for (int j = 0; j < 7; ++j) {
            const bool need = thalf ? (j >= 2) : (j <= 2 || j == 4 || j == 5);
            if (need) {
              const float4 t4 = __ldg(omp + j);
              om[4 * j] = t4.x; om[4 * j + 1] = t4.y; om[4 * j + 2] = t4.z; om[4 * j + 3] = t4.w;
            }
          }
        }
#pragma unroll
        for (int tap = 0; tap < 9; ++tap) {
          if (tap < tap0 || tap >= tap1) continue;
          DcnWinEntry e; e.goff = 0; e.meta = WIN_IN; e.w01 = 0u; e.w23 = 0u;
          if (ok) {
            const float py = (float)(oy - 1 + tap / 3) + om[2 * tap];
            const float px = (float)(ox - 1 + tap % 3) + om[2 * tap + 1];
            if (py > -1.f && py < (float)g.H && px > -1.f && px < (float)g.W) {
              const float y0f = floorf(py), x0f = floorf(px);
              const int y0 = (int)y0f, x0 = (int)x0f;
              const float ly = py - y0f, lx = px - x0f, hy = 1.f - ly, hx = 1.f - lx, m = om[18 + tap];
              const bool y0ok = y0 >= 0, y1ok = y0 + 1 <= g.H - 1, x0ok = x0 >= 0, x1ok = x0 + 1 <= g.W - 1;
              const int yc = max(y0, 0), xc = max(x0, 0);
              e.goff = (img + yc * g.W + xc) * g.ld_in;
              const bool dx = x0ok && x1ok, dy = y0ok && y1ok;
              const bool inside = y0 >= win_y0 && y0 + 1 <= win_y0 + a.win_ph - 1 && x0 >= win_x0 && x0 + 1 <= win_x0 + a.win_pw - 1;
              const uint32_t woff16 = (uint32_t)((yc - win_y0) * a.win_pw + (xc - win_x0)) * 8u;   // 128 B per pixel
              e.meta = (inside ? (woff16 | WIN_IN) : 0u) | (dx ? WIN_DX : 0u) | (dy ? WIN_DY : 0u);
              const float w00 = (y0ok && x0ok) ? hy * hx * m : 0.f, w01 = (y0ok && x1ok) ? hy * lx * m : 0.f;
              const float w10 = (y1ok && x0ok) ? ly * hx * m : 0.f, w11 = (y1ok && x1ok) ? ly * lx * m : 0.f;
              const __nv_bfloat162 wa = __floats2bfloat162_rn(w00, w01), wb = __floats2bfloat162_rn(w10, w11);
              e.w01 = *reinterpret_cast<const uint32_t*>(&wa);
              e.w23 = *reinterpret_cast<const uint32_t*>(&wb);
            }
          }
          win_tab[tap * TC_BM + trow] = e;
        }
      }
      asm volatile("bar.sync 1, 256;" ::: "memory");
      if (tid == 0) tc_stamp(trace, 2);
    }
    if (a.a_mode == CT_A_DCN) {
      // per (tap,row) sampling records, computed once per CTA (row = tid, threads 0..127)
      const int p = tid < TC_BM ? tc_pixel(a, mt, tid) : g.P_out;
      const bool ok = p < g.P_out;
      if (tid < TC_BM) {
        int oy = 0, ox = 0, img = 0;
        float om[28];
        if (ok) {
          const int bb = p / HWo, r = p - bb * HWo;
          oy = r / g.OW; ox = r - oy * g.OW; img = bb * g.H * g.W;
          const float4* omp = reinterpret_cast<const float4*>(a.om + (size_t)p * g.ld_om);
#pragma unroll
          for (int j = 0; j < 7; ++j) {
            const float4 t = __ldg(omp + j);
            om[4 * j] = t.x; om[4 * j + 1] = t.y; om[4 * j + 2] = t.z; om[4 * j + 3] = t.w;
          }
        }
#pragma unroll
        for (int tap = 0; tap < 9; ++tap) {
          DcnEntry e; e.off = 0; e.dxo = 0; e.dyo = 0; e.pad = 0; e.w00 = e.w01 = e.w10 = e.w11 = 0.f;
          if (ok) {
            const float py = (float)(oy - 1 + tap / 3) + om[2 * tap];
            const float px = (float)(ox - 1 + tap % 3) + om[2 * tap + 1];
            if (py > -1.f && py < (float)g.H && px > -1.f && px < (float)g.W) {
              const float y0f = floorf(py), x0f = floorf(px);
              const int y0 = (int)y0f, x0 = (int)x0f;
              const float ly = py - y0f, lx = px - x0f, hy = 1.f - ly, hx = 1.f - lx, m = om[18 + tap];
              const bool y0ok = y0 >= 0, y1ok = y0 + 1 <= g.H - 1, x0ok = x0 >= 0, x1ok = x0 + 1 <= g.W - 1;
              e.off = (img + max(y0, 0) * g.W + max(x0, 0)) * g.ld_in;
              e.dxo = (x0ok && x1ok) ? g.ld_in : 0;
              e.dyo = (y0ok && y1ok) ? g.W * g.ld_in : 0;
              e.w00 = (y0ok && x0ok) ? hy * hx * m : 0.f;
              e.w01 = (y0ok && x1ok) ? hy * lx * m : 0.f;
              e.w10 = (y1ok && x0ok) ? ly * hx * m : 0.f;
              e.w11 = (y1ok && x1ok) ? ly * lx * m : 0.f;
            }
          }
          dcn_tab[tap * TC_BM + tid] = e;
        }
      }
      asm volatile("bar.sync 1, 256;" ::: "memory");
      if (tid == 0) tc_stamp(trace, 2);
    }
    const int cin8 = g.C_in >> 3;
    const int ntaps = g.KH * g.KW;
    const size_t w_slice_elems = (size_t)(X3 ? 2 : 1) * a.n_tile * TC_BK;
    const __nv_bfloat16* wt = a.w + (size_t)nt * a.k_slices * w_slice_elems;

    if (win) {
      // ---- DCN sampled from a shared-memory window (CT_A_DCN_WIN).  K order = (64-channel chunk, tap, channel): one K
      // slice is one tap of one chunk, so the window of a chunk serves nine slices.  Per slice a thread blends its
      // four rows' 8-channel column: 16 LDS.128 (four corners x four rows) instead of 16 L1/L2 round trips; records
      // whose 2x2 footprint leaves the window (offset beyond the margin) take the global path.
      const int nchunks = g.C_in >> 6;
      const uint32_t pitch = (uint32_t)a.win_pw * 128u;
      const int gdx = g.ld_in, gdy = g.W * g.ld_in;
      int s = 0;
      for (int ch = 0; ch < nchunks; ++ch) {
        mbarrier_wait_parity(win_bar, (uint32_t)ch & 1u);
        for (int tap = 0; tap < 9; ++tap, ++s) {
          const int stage = s % S;
          const uint32_t ph = (uint32_t)(s / S) & 1u;
          mbarrier_wait_parity(empty_bar(stage), ph ^ 1u);
          if (tid == 0) {
            mbarrier_expect_tx(full_bar(stage), b_stage_bytes);
            cp_async_bulk(sB + stage * b_stage_bytes, wt + (size_t)s * w_slice_elems, b_stage_bytes, full_bar(stage));
          }
          const DcnWinEntry* tab = win_tab + tap * TC_BM + r0;
          uint4 e4[TC_NROW], v[TC_NROW][4];
#pragma unroll
          for (int i = 0; i < TC_NROW; ++i) e4[i] = *reinterpret_cast<const uint4*>(&tab[32 * i]);
#pragma unroll
          for (int i = 0; i < TC_NROW; ++i) {
            const uint32_t meta = e4[i].y;
            if (meta & WIN_IN) {
              const uint32_t base = s_win + ((meta & 0xffffu) << 4) + (uint32_t)(q << 4);
              const uint32_t dx = (meta & WIN_DX) ? 128u : 0u, dy = (meta & WIN_DY) ? pitch : 0u;
              v[i][0] = lds16(base); v[i][1] = lds16(base + dx);
              v[i][2] = lds16(base + dy); v[i][3] = lds16(base + dy + dx);
            } else {
              const __nv_bfloat16* p00 = a.x + ((int)e4[i].x + (ch << 6) + (q << 3));
              const int dx = (meta & WIN_DX) ? gdx : 0, dy = (meta & WIN_DY) ? gdy : 0;
              v[i][0] = ldg_nc16(p00); v[i][1] = ldg_nc16(p00 + dx);
              v[i][2] = ldg_nc16(p00 + dy); v[i][3] = ldg_nc16(p00 + dy + dx);
            }
          }
          const uint32_t dst = sA + stage * A_STAGE_BYTES + (uint32_t)r0 * 128u + swz;
#pragma unroll
          for (int i = 0; i < TC_NROW; ++i) {
            const uint32_t w0 = __byte_perm(e4[i].z, 0, 0x1010), w1 = __byte_perm(e4[i].z, 0, 0x3232);   // {w,w} pairs
            const uint32_t w2 = __byte_perm(e4[i].w, 0, 0x1010), w3 = __byte_perm(e4[i].w, 0, 0x3232);
            uint4 o;
            o.x = bmul2(v[i][0].x, w0); o.y = bmul2(v[i][0].y, w0); o.z = bmul2(v[i][0].z, w0); o.w = bmul2(v[i][0].w, w0);
            o.x = bfma2(v[i][1].x, w1, o.x); o.y = bfma2(v[i][1].y, w1, o.y); o.z = bfma2(v[i][1].z, w1, o.z); o.w = bfma2(v[i][1].w, w1, o.w);
            o.x = bfma2(v[i][2].x, w2, o.x); o.y = bfma2(v[i][2].y, w2, o.y); o.z = bfma2(v[i][2].z, w2, o.z); o.w = bfma2(v[i][2].w, w2, o.w);
            o.x = bfma2(v[i][3].x, w3, o.x); o.y = bfma2(v[i][3].y, w3, o.y); o.z = bfma2(v[i][3].z, w3, o.z); o.w = bfma2(v[i][3].w, w3, o.w);
            sts16(dst + i * 4096u, o);
          }
          __syncwarp();
          if (lane == 0) mbarrier_arrive(full_bar(stage));
          if (tid == 0) tc_stamp(trace, 8 + s);
        }
        if (ch + 1 < nchunks) {                       // every producer is done with this chunk's window: refill it
          asm volatile("bar.sync 1, 256;" ::: "memory");
          if (tid == 0) {
            mbarrier_arrive_expect_tx(win_bar, a.win_bytes);      // count 1: this arrival + the TMA's bytes complete the phase
            cp_async_bulk_tensor_4d(s_win, &tmap, (ch + 1) << 6, win_x0, win_y0, win_b, win_bar);
          }
        }
      }
    } else if constexpr (X3) {
      // ---- bf16x3 producers: fp32 activations, each 8-channel chunk = two 16-byte loads, split into hi / lo tiles
      auto begin_stage = [&](int s) {
        const int stage = s % S;
        const uint32_t ph = (uint32_t)(s / S) & 1u;
        mbarrier_wait_parity(empty_bar(stage), ph ^ 1u);
        if (tid == 0) {
          mbarrier_expect_tx(full_bar(stage), b_stage_bytes);
          cp_async_bulk(sB + stage * b_stage_bytes, wt + (size_t)s * w_slice_elems, b_stage_bytes, full_bar(stage));
        }
        return stage;
      };
      auto end_stage = [&](int s, int stage) {
        __syncwarp();
        if (lane == 0) mbarrier_arrive(full_bar(stage));
        if (tid == 0) tc_stamp(trace, 8 + s);
      };
      if (a.a_mode == CT_A_DCN) {
        float4 va[2][4][2], vb[2][4][2];
        auto load_half = [&](int tap, int c, int half, float4 (&v)[2][4][2]) {
          const DcnEntry* tab = dcn_tab + (tap < ntaps ? tap : 0) * TC_BM + r0 + 64 * half;
#pragma unroll
          for (int j = 0; j < 2; ++j) {
            const int4 o = *reinterpret_cast<const int4*>(&tab[32 * j]);     // off, dxo, dyo
            const float* p00 = xf + (o.x + c);
            v[j][0][0] = ldg_nc_f4(p00);             v[j][0][1] = ldg_nc_f4(p00 + 4);
            v[j][1][0] = ldg_nc_f4(p00 + o.y);       v[j][1][1] = ldg_nc_f4(p00 + o.y + 4);
            v[j][2][0] = ldg_nc_f4(p00 + o.z);       v[j][2][1] = ldg_nc_f4(p00 + o.z + 4);
            v[j][3][0] = ldg_nc_f4(p00 + o.z + o.y); v[j][3][1] = ldg_nc_f4(p00 + o.z + o.y + 4);
          }
        };
        auto blend_half = [&](int tap, int stage, int half, const float4 (&v)[2][4][2]) {
          const bool live = tap < ntaps;
          const DcnEntry* tab = dcn_tab + (live ? tap : 0) * TC_BM + r0 + 64 * half;
          const uint32_t dst = sA + stage * a_stage_bytes + (uint32_t)(r0 + 64 * half) * 128u + swz;
#pragma unroll
          for (int j = 0; j < 2; ++j) {
            const float4 w = *reinterpret_cast<const float4*>(&tab[32 * j].w00);
            const float ww[4] = {w.x, w.y, w.z, w.w};
            float4 acc[2];
#pragma unroll
            for (int h2 = 0; h2 < 2; ++h2) {
              acc[h2] = make_float4(ww[0] * v[j][0][h2].x, ww[0] * v[j][0][h2].y, ww[0] * v[j][0][h2].z, ww[0] * v[j][0][h2].w);
#pragma unroll
              for (int cn = 1; cn < 4; ++cn) {
                acc[h2].x = fmaf(ww[cn], v[j][cn][h2].x, acc[h2].x); acc[h2].y = fmaf(ww[cn], v[j][cn][h2].y, acc[h2].y);
                acc[h2].z = fmaf(ww[cn], v[j][cn][h2].z, acc[h2].z); acc[h2].w = fmaf(ww[cn], v[j][cn][h2].w, acc[h2].w);
              }
            }
            uint4 hi, lo;
            split8(acc[0], acc[1], hi, lo);
            if (!live) { hi = make_uint4(0, 0, 0, 0); lo = hi; }
            sts16(dst + j * 4096u, hi);
            sts16(dst + A_STAGE_BYTES + j * 4096u, lo);
          }
        };
        int tap = q / cin8, cq = q - tap * cin8;
        load_half(tap, cq << 3, 0, va);
        for (int s = 0; s < a.k_slices; ++s) {
          load_half(tap, cq << 3, 1, vb);
          const int stage = begin_stage(s);
          blend_half(tap, stage, 0, va);
          int ntap = tap, ncq = cq + 8;
          while (ncq >= cin8) { ncq -= cin8; ++ntap; }
          if (s + 1 < a.k_slices) load_half(ntap, ncq << 3, 0, va);
          blend_half(tap, stage, 1, vb);
          tap = ntap; cq = ncq;
          end_stage(s, stage);
        }
      } else {
        int ltap = q / cin8, lcq = q - ltap * cin8;
        auto load_slice = [&](bool in_range, float4 (&v)[TC_NROW][2]) {
#pragma unroll
          for (int i = 0; i < TC_NROW; ++i) { v[i][0] = make_float4(0.f, 0.f, 0.f, 0.f); v[i][1] = v[i][0]; }
          if (in_range && ltap < ntaps) {
            const int ky = ltap / g.KW, kx = ltap - ky * g.KW;
            const int tap_off = (ky * g.W + kx) * g.ld_in + (lcq << 3);
#pragma unroll
            for (int i = 0; i < TC_NROW; ++i)
              if ((unsigned)(row_iy[i] + ky) < (unsigned)g.H && (unsigned)(row_ix[i] + kx) < (unsigned)g.W) {
                const float* pp = xf + (row_off[i] + tap_off);
                v[i][0] = ldg_nc_f4(pp); v[i][1] = ldg_nc_f4(pp + 4);
              }
          }
          lcq += 8;
          while (lcq >= cin8) { lcq -= cin8; ++ltap; }
        };
        auto store_slice = [&](int s, const float4 (&v)[TC_NROW][2]) {
          const int stage = begin_stage(s);
          const uint32_t dst = sA + stage * a_stage_bytes + (uint32_t)r0 * 128u + swz;
#pragma unroll
          for (int i = 0; i < TC_NROW; ++i) {
            uint4 hi, lo;
            split8(v[i][0], v[i][1], hi, lo);
            sts16(dst + i * 4096u, hi);
            sts16(dst + A_STAGE_BYTES + i * 4096u, lo);
          }
          end_stage(s, stage);
        };
        const int KS = a.k_slices;
        float4 v0[TC_NROW][2], v1[TC_NROW][2], v2[TC_NROW][2];
        load_slice(0 < KS, v0);
        load_slice(1 < KS, v1);
        load_slice(2 < KS, v2);
        for (int s = 0; s < KS; s += 3) {
          store_slice(s, v0);
          load_slice(s + 3 < KS, v0);
          if (s + 1 < KS) { store_slice(s + 1, v1); load_slice(s + 4 < KS, v1); }
          if (s + 2 < KS) { store_slice(s + 2, v2); load_slice(s + 5 < KS, v2); }
        }
      }
    } else if (a.a_mode == CT_A_DCN) {
      // Software-pipelined by half slices (2 of the thread's 4 rows): the 8 corner loads of the next half are in
      // flight while the current half is blended (the gather is latency-bound -- memory-level parallelism first --
      // and the blend is issue-bound: packed FFMA2, one-op bf16 unpack).  A slice whose tap index runs past the
      // kernel (K padding) samples tap 0 with its result zeroed.
      uint4 va[2][4], vb[2][4];
      auto load_half = [&](int tap, int c, int half, uint4 (&v)[2][4]) {
        const DcnEntry* tab = dcn_tab + (tap < ntaps ? tap : 0) * TC_BM + r0 + 64 * half;
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          const int4 o = *reinterpret_cast<const int4*>(&tab[32 * j]);     // off, dxo, dyo
          const __nv_bfloat16* p00 = a.x + (o.x + c);
          v[j][0] = ldg_nc16(p00);
          v[j][1] = ldg_nc16(p00 + o.y);
          v[j][2] = ldg_nc16(p00 + o.z);
          v[j][3] = ldg_nc16(p00 + o.z + o.y);
        }
      };
      auto blend_half = [&](int tap, int stage, int half, const uint4 (&v)[2][4]) {
        const bool live = tap < ntaps;
        const DcnEntry* tab = dcn_tab + (live ? tap : 0) * TC_BM + r0 + 64 * half;
        const uint32_t dst = sA + stage * A_STAGE_BYTES + (uint32_t)(r0 + 64 * half) * 128u + swz;
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          // packed bf16 blend, same rounding points as the window sampler (weights to bf16, fma chain 00,01,10,11)
          const float4 w = *reinterpret_cast<const float4*>(&tab[32 * j].w00);
          const uint32_t w0 = dup_bf2(w.x), w1 = dup_bf2(w.y), w2 = dup_bf2(w.z), w3 = dup_bf2(w.w);
          uint4 o;
          o.x = bmul2(v[j][0].x, w0); o.y = bmul2(v[j][0].y, w0); o.z = bmul2(v[j][0].z, w0); o.w = bmul2(v[j][0].w, w0);
          o.x = bfma2(v[j][1].x, w1, o.x); o.y = bfma2(v[j][1].y, w1, o.y); o.z = bfma2(v[j][1].z, w1, o.z); o.w = bfma2(v[j][1].w, w1, o.w);
          o.x = bfma2(v[j][2].x, w2, o.x); o.y = bfma2(v[j][2].y, w2, o.y); o.z = bfma2(v[j][2].z, w2, o.z); o.w = bfma2(v[j][2].w, w2, o.w);
          o.x = bfma2(v[j][3].x, w3, o.x); o.y = bfma2(v[j][3].y, w3, o.y); o.z = bfma2(v[j][3].z, w3, o.z); o.w = bfma2(v[j][3].w, w3, o.w);
          sts16(dst + j * 4096u, live ? o : make_uint4(0, 0, 0, 0));
        }
      };
      // (tap, channel group) of this thread's 8-channel column in slice s, advanced incrementally (no division)
      int tap = q / cin8, cq = q - tap * cin8;
      load_half(tap, cq << 3, 0, va);
      for (int s = 0; s < a.k_slices; ++s) {
        const int stage = s % S;
        const uint32_t ph = (uint32_t)(s / S) & 1u;
        load_half(tap, cq << 3, 1, vb);
        mbarrier_wait_parity(empty_bar(stage), ph ^ 1u);
        if (tid == 0) {
          mbarrier_expect_tx(full_bar(stage), b_stage_bytes);
          cp_async_bulk(sB + stage * b_stage_bytes, wt + (size_t)s * a.n_tile * TC_BK, b_stage_bytes, full_bar(stage));
        }
        blend_half(tap, stage, 0, va);
        int ntap = tap, ncq = cq + 8;
        while (ncq >= cin8) { ncq -= cin8; ++ntap; }
        if (s + 1 < a.k_slices) load_half(ntap, ncq << 3, 0, va);
        blend_half(tap, stage, 1, vb);
        tap = ntap; cq = ncq;
        __syncwarp();
        if (lane == 0) mbarrier_arrive(full_bar(stage));      // one arrival per producer warp
        if (tid == 0) tc_stamp(trace, 8 + s);
      }
    } else {
      // Plain convolution gather, register-prefetched three K slices ahead (12 independent 16-byte loads in flight
      // per thread): one slice's loads alone leave the loop bound by the L2 round trip (~1700 cycles per slice
      // measured with tools/tc_trace.py).  (tap, channel group) advance incrementally with the load order.
      int ltap = q / cin8, lcq = q - ltap * cin8;
      auto load_slice = [&](bool in_range, uint4 (&v)[TC_NROW]) {
#pragma unroll
        for (int i = 0; i < TC_NROW; ++i) v[i] = make_uint4(0, 0, 0, 0);
        if (in_range && ltap < ntaps) {
          const int ky = ltap / g.KW, kx = ltap - ky * g.KW;
          const int tap_off = (ky * g.W + kx) * g.ld_in + (lcq << 3);      // same for every row of the slice
#pragma unroll
          for (int i = 0; i < TC_NROW; ++i)
            if ((unsigned)(row_iy[i] + ky) < (unsigned)g.H && (unsigned)(row_ix[i] + kx) < (unsigned)g.W)
              v[i] = ldg_nc16(a.x + (row_off[i] + tap_off));
        }
        lcq += 8;
        while (lcq >= cin8) { lcq -= cin8; ++ltap; }
      };
      auto store_slice = [&](int s, const uint4 (&v)[TC_NROW]) {
        const int stage = s % S;
        const uint32_t ph = (uint32_t)(s / S) & 1u;
        mbarrier_wait_parity(empty_bar(stage), ph ^ 1u);
        if (tid == 0) {
          mbarrier_expect_tx(full_bar(stage), b_stage_bytes);
          cp_async_bulk(sB + stage * b_stage_bytes, wt + (size_t)s * a.n_tile * TC_BK, b_stage_bytes, full_bar(stage));
        }
        const uint32_t dst = sA + stage * A_STAGE_BYTES + (uint32_t)r0 * 128u + swz;
#pragma unroll
        for (int i = 0; i < TC_NROW; ++i) sts16(dst + i * 4096u, v[i]);
        __syncwarp();
        if (lane == 0) mbarrier_arrive(full_bar(stage));      // one arrival per producer warp (256 arrivals on one
                                                          // shared-memory word serialise)
        if (tid == 0) tc_stamp(trace, 8 + s);
      };
      const int KS = a.k_slices;
      uint4 v0[TC_NROW], v1[TC_NROW], v2[TC_NROW];
      load_slice(0 < KS, v0);
      load_slice(1 < KS, v1);
      load_slice(2 < KS, v2);
      for (int s = 0; s < KS; s += 3) {
        store_slice(s, v0);
        load_slice(s + 3 < KS, v0);
        if (s + 1 < KS) { store_slice(s + 1, v1); load_slice(s + 4 < KS, v1); }
        if (s + 2 < KS) { store_slice(s + 2, v2); load_slice(s + 5 < KS, v2); }
      }
    }

    // =========================== epilogue ===========================
    mbarrier_wait_parity(tmem_full_bar, 0);
    tcgen05_fence_after_thread_sync();
    if (tid == 0) tc_stamp(trace, 5);
    const int wq = warp & 3, chalf = warp >> 2;      // TMEM lane quarter, column-chunk parity
    const int row = wq * 32 + lane;
    const int p = tc_pixel(a, mt, row);
    const bool p_ok = p < g.P_out;
    const uint32_t t_lane = tmem_base + ((uint32_t)(wq * 32) << 16);
    for (int col = chalf * 16; col < a.n_tile; col += 32) {
      uint32_t r[16];
      tcgen05_ld_32x32b_x16(t_lane + (uint32_t)col, r);
      const int o0 = n0 + col;
      if (!p_ok || o0 >= g.C_out) continue;
      float v[16];
#pragma unroll
      for (int j = 0; j < 16; ++j) v[j] = __uint_as_float(r[j]);
      if (a.shift) {
        if (o0 + 16 <= g.C_out && (reinterpret_cast<size_t>(a.shift + o0) & 15) == 0) {   // four 16-byte loads
          const float4* sh4 = reinterpret_cast<const float4*>(a.shift + o0);
#pragma unroll
          for (int j4 = 0; j4 < 4; ++j4) {
            const float4 sh = __ldg(sh4 + j4);
            v[4 * j4] += sh.x; v[4 * j4 + 1] += sh.y; v[4 * j4 + 2] += sh.z; v[4 * j4 + 3] += sh.w;
          }
        } else {
#pragma unroll
          for (int j = 0; j < 16; ++j) if (o0 + j < g.C_out) v[j] += __ldg(a.shift + o0 + j);
        }
      }
      if (X3 && g.out_mode == CT_OUT_NHWC) {            // fp32 activations in, fp32 activations out
        if (a.residual) {
          const float4* rp = reinterpret_cast<const float4*>(reinterpret_cast<const float*>(a.residual) + (size_t)p * g.ld_res + o0);
#pragma unroll
          for (int j4 = 0; j4 < 4; ++j4) {
            const float4 rr = ldg_nc_f4(reinterpret_cast<const float*>(rp + j4));
            v[4 * j4] += rr.x; v[4 * j4 + 1] += rr.y; v[4 * j4 + 2] += rr.z; v[4 * j4 + 3] += rr.w;
          }
        }
        if (g.relu) {
#pragma unroll
          for (int j = 0; j < 16; ++j) v[j] = fmaxf(v[j], 0.f);
        }
        float4* op = reinterpret_cast<float4*>(reinterpret_cast<float*>(a.out) + (size_t)p * g.ld_out + o0);
#pragma unroll
        for (int j4 = 0; j4 < 4; ++j4) op[j4] = make_float4(v[4 * j4], v[4 * j4 + 1], v[4 * j4 + 2], v[4 * j4 + 3]);
      } else if (g.out_mode == CT_OUT_NHWC) {
        if (a.residual) {
          const uint4* rp = reinterpret_cast<const uint4*>(a.residual + (size_t)p * g.ld_res + o0);
          const uint4 ra = ldg_nc16(rp), rb = ldg_nc16(rp + 1);
          const __nv_bfloat162* ha = reinterpret_cast<const __nv_bfloat162*>(&ra);
          const __nv_bfloat162* hb = reinterpret_cast<const __nv_bfloat162*>(&rb);
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const float2 fa = __bfloat1622float2(ha[j]), fb = __bfloat1622float2(hb[j]);
            v[2 * j] += fa.x; v[2 * j + 1] += fa.y; v[8 + 2 * j] += fb.x; v[8 + 2 * j + 1] += fb.y;
          }
        }
        if (g.relu) {
#pragma unroll
          for (int j = 0; j < 16; ++j) v[j] = fmaxf(v[j], 0.f);
        }
        uint4 oa, ob;
        __nv_bfloat162* pa = reinterpret_cast<__nv_bfloat162*>(&oa);
        __nv_bfloat162* pb = reinterpret_cast<__nv_bfloat162*>(&ob);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          pa[j] = __floats2bfloat162_rn(v[2 * j], v[2 * j + 1]);
          pb[j] = __floats2bfloat162_rn(v[8 + 2 * j], v[8 + 2 * j + 1]);
        }
        uint4* op = reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(a.out) + (size_t)p * g.ld_out + o0);
        op[0] = oa; op[1] = ob;
      } else if (g.out_mode == CT_OUT_NHWC_F32) {
        float* op = reinterpret_cast<float*>(a.out) + (size_t)p * g.ld_out + o0;
#pragma unroll
        for (int j = 0; j < 16; ++j) {
          if (g.relu) v[j] = fmaxf(v[j], 0.f);
          const float sg = sigmoidf_fast(v[j]);              // unconditional: keeps the 16 chains interleaved
          v[j] = (o0 + j >= g.sig_from) ? sg : v[j];
        }
        if (o0 + 16 <= g.ld_out && (g.ld_out & 3) == 0) {      // padded row: four 16-byte stores
#pragma unroll
          for (int j4 = 0; j4 < 4; ++j4)
            reinterpret_cast<float4*>(op)[j4] = make_float4(v[4 * j4], v[4 * j4 + 1], v[4 * j4 + 2], v[4 * j4 + 3]);
        } else {
#pragma unroll
          for (int j = 0; j < 16; ++j) if (o0 + j < g.C_out) op[j] = v[j];
        }
      } else {
        const int b = p / HWo, rr = p - b * HWo;
        float* op = reinterpret_cast<float*>(a.out) + ((size_t)b * g.C_out + o0) * HWo + rr;
        if (g.relu) {
#pragma unroll
          for (int j = 0; j < 16; ++j) v[j] = fmaxf(v[j], 0.f);
        }
        if (g.head_act == CT_HEAD_SIGMOID) {
#pragma unroll
          for (int j = 0; j < 16; ++j) v[j] = sigmoidf_fast(v[j]);
        } else if (g.head_act == CT_HEAD_DEPTH) {
#pragma unroll
          for (int j = 0; j < 16; ++j) v[j] = (__fdividef(1.f, sigmoidf_fast(v[j]) + 1e-6f) - 1.f) * g.depth_scale;
        }
#pragma unroll
        for (int j = 0; j < 16; ++j)
          if (o0 + j < g.C_out) op[(size_t)j * HWo] = v[j];
      }
    }
  } else if (lane == 0) {
    // =========================== MMA issuer (one thread) ===========================
    const uint32_t idesc = umma_idesc_bf16_m128(a.n_tile);
    for (int s = 0; s < a.k_slices; ++s) {
      const int stage = s % S;
      const uint32_t ph = (uint32_t)(s / S) & 1u;
      mbarrier_wait_parity(full_bar(stage), ph);
      // the producers' st.shared (acquired through the barrier) -> async proxy.  Fenced here rather than by every producer:
      // fence.proxy.async compiles to MEMBAR.ALL.CTA + FENCE.VIEW.ASYNC, and the MEMBAR drains the producer's prefetched loads
      fence_proxy_async_shared_cta();
      tcgen05_fence_after_thread_sync();
      const uint64_t ad = umma_sdesc_sw128(sA + stage * a_stage_bytes);
      const uint64_t bd = umma_sdesc_sw128(sB + stage * b_stage_bytes);
      if constexpr (X3) {
        const uint64_t ad_lo = umma_sdesc_sw128(sA + stage * a_stage_bytes + A_STAGE_BYTES);
        const uint64_t bd_lo = umma_sdesc_sw128(sB + stage * b_stage_bytes + b_tile_bytes);
#pragma unroll
        for (int k = 0; k < TC_BK / 16; ++k) {      // small cross terms first, then the hi x hi term
          tcgen05_mma(tmem_base, ad_lo + 2ull * k, bd + 2ull * k, idesc, (s > 0 || k > 0) ? 1u : 0u);
          tcgen05_mma(tmem_base, ad + 2ull * k, bd_lo + 2ull * k, idesc, 1u);
          tcgen05_mma(tmem_base, ad + 2ull * k, bd + 2ull * k, idesc, 1u);
        }
      } else {
#pragma unroll
        for (int k = 0; k < TC_BK / 16; ++k)
          tcgen05_mma(tmem_base, ad + 2ull * k, bd + 2ull * k, idesc, (s > 0 || k > 0) ? 1u : 0u);
      }
      tcgen05_commit(empty_bar(stage));     // frees this smem stage when the MMAs above have read it
    }
    tcgen05_commit(tmem_full_bar);           // accumulator complete -> epilogue
    tc_stamp(trace, 4);
  }

  tcgen05_fence_before_thread_sync();
  __syncthreads();
  if (tid == 0) tc_stamp(trace, 6);
  if (warp == 8) {
    tcgen05_fence_after_thread_sync();
    tcgen05_dealloc(tmem_base, (uint32_t)a.tmem_cols);
  }
}

// =====================================================================================================================
// Persistent DCNv2 kernel (CT_A_DCN_WIN layers with a single N tile, bf16 NHWC output): one CTA per SM walks its share
// of the 8x16-pixel output patches.  What the per-tile kernel above spends outside its slice loop -- TMEM allocation,
// barrier init, the sampling-table build behind an L2 round trip for `om`, the window TMA, the epilogue: 12 k of 30 k
// cycles per tile (tools/tc_trace.py) -- is taken off the critical path:
//   * the window of unit u+2 (unit = tile x 64-channel chunk) is requested when unit u is finished: two windows in
//     flight, a whole unit (9 slices) of latency cover;
//   * the sampling table of tile t+1 is built by the producers one tap per slice while they sample tile t
//     (its `om` values fetched one slice ahead), into the other of two table buffers;
//   * two TMEM accumulators: four dedicated epilogue warps drain tile t while the producers / MMA work on tile t+1.
//   * the window is requested ROW BY ROW, two rows per slice of the previous unit: one 43 KB request occupied the TMA
//     unit for ~5000 cycles and the per-slice weight copies queued behind it (a 5000-cycle bubble at every tile
//     boundary in the first version of this kernel, profiles/r02_tc_trace_persist.txt).
//   * every TMA request (weight tile per slice, window rows) is issued by a DEDICATED warp: issuing a bulk copy costs the
//     issuing thread hundreds of cycles, and with the requests on producer thread 0 its warp was the slowest of every
//     slice (A written 1700 cycles after the stage was acquired, fine-grained trace in profiles/r02_tc_trace_persist.txt).
// Warps 0-15 producers (sampling + table), warp 16 MMA issuer, warps 17-20 epilogue, warp 21 TMA issuer.
// =====================================================================================================================
constexpr int DP_PWARPS = 16;            // producer warps: a slice is a latency chain per warp (table LDS -> 16 LDS -> blend ->
                                         // STS -> fence -> arrive, ~1100-1500 cycles with 4 rows per thread): 16 warps x 2 rows
constexpr int DP_PRODUCERS = DP_PWARPS * 32;
constexpr int DP_NROW = TC_BM * 8 / DP_PRODUCERS;     // A-tile rows per producer thread per K slice (2)
constexpr int DP_THREADS = DP_PRODUCERS + 32 + 128 + 32 + 128;   // + MMA warp + 4 epilogue warps + TMA warp + 4 table warps
constexpr int DP_SA = 3;                 // A/B stages

__device__ __forceinline__ void dp_tile_origin(const TcArgs& a, int tile, int& b, int& ty, int& tx) {
  const int tpi = a.tiles_x * a.tiles_y;
  b = tile / tpi;
  const int t = tile - b * tpi;
  ty = t / a.tiles_x;
  tx = t - ty * a.tiles_x;
}

__global__ void __launch_bounds__(DP_THREADS, 1)
dcn_persist_kernel(const TcArgs a, const int tiles_total, const __grid_constant__ CUtensorMap tmap) {
  extern __shared__ __align__(1024) unsigned char smem_dyn[];
  unsigned char* smem = smem_dyn + ((1024u - (smem_u32(smem_dyn) & 1023u)) & 1023u);
  const ConvGeom& g = a.g;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  unsigned long long* const trace = tc_trace_ptr();
  const uint32_t b_tile_bytes = (uint32_t)a.n_tile * 128u;
  const uint32_t win_stride = (a.win_bytes + 127u) & ~127u;
  const uint32_t smem_base = smem_u32(smem);
  const uint32_t sA = smem_base;
  const uint32_t sB = sA + DP_SA * A_STAGE_BYTES;
  const uint32_t sWin = sB + DP_SA * b_tile_bytes;                       // 1024-aligned (both terms are)
  const uint32_t off_tab = DP_SA * A_STAGE_BYTES + DP_SA * b_tile_bytes + 2u * win_stride;
  DcnWinEntry* tabs = reinterpret_cast<DcnWinEntry*>(smem + off_tab);    // [2][9][128]
  const uint32_t off_bar = off_tab + 2u * 9u * TC_BM * 16u;
  const uint32_t bars = smem_base + off_bar;
  auto full_bar = [&](int s) { return bars + 8u * s; };
  auto empty_bar = [&](int s) { return bars + 8u * (DP_SA + s); };
  auto win_full = [&](int i) { return bars + 8u * (2 * DP_SA + i); };
  auto acc_full = [&](int i) { return bars + 8u * (2 * DP_SA + 2 + i); };
  auto acc_empty = [&](int i) { return bars + 8u * (2 * DP_SA + 4 + i); };
  auto win_empty = [&](int i) { return bars + 8u * (2 * DP_SA + 6 + i); };
  auto tab_full = [&](int i) { return bars + 8u * (2 * DP_SA + 8 + i); };
  auto tab_empty = [&](int i) { return bars + 8u * (2 * DP_SA + 10 + i); };
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + off_bar + 8 * (2 * DP_SA + 12));

  pdl_trigger();
  if (tid == 0) {
    for (int s = 0; s < DP_SA; ++s) { mbarrier_init(full_bar(s), DP_PWARPS + 1); mbarrier_init(empty_bar(s), 1); }   // 16 producer warps + the TMA warp's expect_tx arrival
    for (int i = 0; i < 2; ++i) {
      mbarrier_init(win_full(i), 1); mbarrier_init(acc_full(i), 1); mbarrier_init(acc_empty(i), 4); mbarrier_init(win_empty(i), DP_PWARPS);
      mbarrier_init(tab_full(i), 4); mbarrier_init(tab_empty(i), DP_PWARPS);
    }
    fence_mbarrier_init();
  }
  if (warp == DP_PWARPS) {
    tcgen05_alloc(smem_u32((const void*)tmem_slot), (uint32_t)a.tmem_cols);
    tcgen05_relinquish_alloc_permit();
  }
  tcgen05_fence_before_thread_sync();
  __syncthreads();
  tcgen05_fence_after_thread_sync();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();

  const int G = gridDim.x;
  const int nchunks = g.C_in >> 6;
  const int HWo = g.OH * g.OW;
  int n_my = 0;                                                          // tiles of this CTA
  if ((int)blockIdx.x < tiles_total) n_my = (tiles_total - 1 - (int)blockIdx.x) / G + 1;
  const int n_units = n_my * nchunks;

  if (warp < DP_PWARPS) {
    // ======================================= producers =======================================
    const int q = tid & 7, r0 = tid >> 3;                                // rows r0 + 64 i, i < DP_NROW
    const uint32_t swz = (uint32_t)((q ^ (r0 & 7)) << 4);
    const uint32_t pitch = (uint32_t)a.win_pw * 128u;
    const int gdx = g.ld_in, gdy = g.W * g.ld_in;
    // Nothing but the slice loop lives here: `fence.proxy.async` compiles to MEMBAR.ALL.CTA + FENCE.VIEW.ASYNC, and the
    // MEMBAR waits for every outstanding load of the thread, so a prefetch of the next tile's `om` floats in flight across
    // it cost the warp a full L2 round trip per slice.  The records are built by the table warps below.
    int s = 0;
    for (int t = 0; t < n_my; ++t) {
      const DcnWinEntry* tab_cur = tabs + (t & 1) * 9 * TC_BM;
      mbarrier_wait_parity(tab_full(t & 1), (uint32_t)(t >> 1) & 1u);
      for (int ch = 0; ch < nchunks; ++ch) {
        const int u = t * nchunks + ch;
        const uint32_t s_win = sWin + (uint32_t)(u & 1) * win_stride;
        mbarrier_wait_parity(win_full(u & 1), (uint32_t)(u >> 1) & 1u);
        for (int tap = 0; tap < 9; ++tap, ++s) {
          const int stage = s % DP_SA;
          const uint32_t ph = (uint32_t)(s / DP_SA) & 1u;
          mbarrier_wait_parity(empty_bar(stage), ph ^ 1u);
          if (tid == 0 && s < 60) tc_stamp(trace, 16 + 4 * s);
          const DcnWinEntry* tab = tab_cur + tap * TC_BM + r0;
          uint4 e4[DP_NROW], v[DP_NROW][4];
#pragma unroll
          for (int i = 0; i < DP_NROW; ++i) e4[i] = *reinterpret_cast<const uint4*>(&tab[64 * i]);
#pragma unroll
          for (int i = 0; i < DP_NROW; ++i) {
            const uint32_t meta = e4[i].y;
            if (meta & WIN_IN) {
              const uint32_t base = s_win + ((meta & 0xffffu) << 4) + (uint32_t)(q << 4);
              const uint32_t dx = (meta & WIN_DX) ? 128u : 0u, dy = (meta & WIN_DY) ? pitch : 0u;
              v[i][0] = lds16(base); v[i][1] = lds16(base + dx);
              v[i][2] = lds16(base + dy); v[i][3] = lds16(base + dy + dx);
            } else {
              const __nv_bfloat16* p00 = a.x + ((int)e4[i].x + (ch << 6) + (q << 3));
              const int dx = (meta & WIN_DX) ? gdx : 0, dy = (meta & WIN_DY) ? gdy : 0;
              v[i][0] = ldg_nc16(p00); v[i][1] = ldg_nc16(p00 + dx);
              v[i][2] = ldg_nc16(p00 + dy); v[i][3] = ldg_nc16(p00 + dy + dx);
            }
          }
          const uint32_t dst = sA + stage * A_STAGE_BYTES + (uint32_t)r0 * 128u + swz;
#pragma unroll
          for (int i = 0; i < DP_NROW; ++i) {
            const uint32_t w0 = __byte_perm(e4[i].z, 0, 0x1010), w1 = __byte_perm(e4[i].z, 0, 0x3232);
            const uint32_t w2 = __byte_perm(e4[i].w, 0, 0x1010), w3 = __byte_perm(e4[i].w, 0, 0x3232);
            uint4 o;
            o.x = bmul2(v[i][0].x, w0); o.y = bmul2(v[i][0].y, w0); o.z = bmul2(v[i][0].z, w0); o.w = bmul2(v[i][0].w, w0);
            o.x = bfma2(v[i][1].x, w1, o.x); o.y = bfma2(v[i][1].y, w1, o.y); o.z = bfma2(v[i][1].z, w1, o.z); o.w = bfma2(v[i][1].w, w1, o.w);
            o.x = bfma2(v[i][2].x, w2, o.x); o.y = bfma2(v[i][2].y, w2, o.y); o.z = bfma2(v[i][2].z, w2, o.z); o.w = bfma2(v[i][2].w, w2, o.w);
            o.x = bfma2(v[i][3].x, w3, o.x); o.y = bfma2(v[i][3].y, w3, o.y); o.z = bfma2(v[i][3].z, w3, o.z); o.w = bfma2(v[i][3].w, w3, o.w);
            sts16(dst + i * 8192u, o);
          }
          __syncwarp();
          if (lane == 0) mbarrier_arrive(full_bar(stage));
          if (tid == 0 && s < 60) tc_stamp(trace, 16 + 4 * s + 1);
        }
        if (lane == 0) mbarrier_arrive(win_empty(u & 1));                    // this warp is done with the unit's window
      }
      if (lane == 0) mbarrier_arrive(tab_empty(t & 1));                      // ... and with the tile's table
    }
  } else if (warp >= DP_PWARPS + 6) {
    // ======================================= table warps: one thread per A-tile row =======================================
    // Records of tile t into table t & 1, up to two tiles ahead of the producers.  A record is (global offset of corner 00,
    // window offset | flags, 4 bf16 corner weights with the modulation mask folded in); see conv_tc_kernel's window path.
    const int trow = tid - (DP_PWARPS + 6) * 32;
    for (int t = 0; t < n_my; ++t) {
      const int tile = (int)blockIdx.x + t * G;
      int b, ty, tx;
      dp_tile_origin(a, tile, b, ty, tx);
      const int oy = ty * 8 + (trow >> 4), ox = tx * 16 + (trow & 15);
      const bool ok = oy < g.OH && ox < g.OW;
      const int img = b * g.H * g.W;
      const int wy0 = ty * 8 - 1 - a.win_m, wx0 = tx * 16 - 1 - a.win_m;
      float omv[28];
#pragma unroll
      for (int j = 0; j < 28; ++j) omv[j] = 0.f;
      if (ok) {
        const float4* om4 = reinterpret_cast<const float4*>(a.om + (size_t)((b * g.OH + oy) * g.OW + ox) * g.ld_om);
#pragma unroll
        for (int j = 0; j < 7; ++j) {
          const float4 f = __ldg(om4 + j);
          omv[4 * j] = f.x; omv[4 * j + 1] = f.y; omv[4 * j + 2] = f.z; omv[4 * j + 3] = f.w;
        }
      }
      if (t >= 2) mbarrier_wait_parity(tab_empty(t & 1), (uint32_t)((t - 2) >> 1) & 1u);
      DcnWinEntry* tab = tabs + (t & 1) * 9 * TC_BM + trow;
#pragma unroll
      for (int tap = 0; tap < 9; ++tap) {
        DcnWinEntry e; e.goff = 0; e.meta = WIN_IN; e.w01 = 0u; e.w23 = 0u;
        if (ok) {
          const float py = (float)(oy - 1 + tap / 3) + omv[2 * tap];
          const float px = (float)(ox - 1 + tap % 3) + omv[2 * tap + 1];
          const float m = omv[18 + tap];
          if (py > -1.f && py < (float)g.H && px > -1.f && px < (float)g.W) {
            const float y0f = floorf(py), x0f = floorf(px);
            const int y0 = (int)y0f, x0 = (int)x0f;
            const float ly = py - y0f, lx = px - x0f, hy = 1.f - ly, hx = 1.f - lx;
            const bool y0ok = y0 >= 0, y1ok = y0 + 1 <= g.H - 1, x0ok = x0 >= 0, x1ok = x0 + 1 <= g.W - 1;
            const int yc = max(y0, 0), xc = max(x0, 0);
            e.goff = (img + yc * g.W + xc) * g.ld_in;
            const bool ddx = x0ok && x1ok, ddy = y0ok && y1ok;
            const bool inside = y0 >= wy0 && y0 + 1 <= wy0 + a.win_ph - 1 && x0 >= wx0 && x0 + 1 <= wx0 + a.win_pw - 1;
            const uint32_t woff16 = (uint32_t)((yc - wy0) * a.win_pw + (xc - wx0)) * 8u;
            e.meta = (inside ? (woff16 | WIN_IN) : 0u) | (ddx ? WIN_DX : 0u) | (ddy ? WIN_DY : 0u);
            const float w00 = (y0ok && x0ok) ? hy * hx * m : 0.f, w01 = (y0ok && x1ok) ? hy * lx * m : 0.f;
            const float w10 = (y1ok && x0ok) ? ly * hx * m : 0.f, w11 = (y1ok && x1ok) ? ly * lx * m : 0.f;
            const __nv_bfloat162 wa = __floats2bfloat162_rn(w00, w01), wb = __floats2bfloat162_rn(w10, w11);
            e.w01 = *reinterpret_cast<const uint32_t*>(&wa);
            e.w23 = *reinterpret_cast<const uint32_t*>(&wb);
          }
        }
        tab[tap * TC_BM] = e;
      }
      __syncwarp();
      if (lane == 0) mbarrier_arrive(tab_full(t & 1));
    }
  } else if (warp == DP_PWARPS + 5) {
    // ======================================= TMA issuer =======================================
    if (lane == 0 && n_my > 0) {
    // window of unit u, rows [ry0, ry1): one TMA request per row (tid 0 only); the first request arms the barrier
    auto issue_window_rows = [&](int u, int ry0, int ry1) {
      const int t = u / nchunks, ch = u - t * nchunks;
      int b, ty, tx;
      dp_tile_origin(a, (int)blockIdx.x + t * G, b, ty, tx);
      if (ry0 == 0) mbarrier_arrive_expect_tx(win_full(u & 1), a.win_bytes);
      const uint32_t row_bytes = (uint32_t)a.win_pw * 128u;
      for (int ry = ry0; ry < ry1 && ry < a.win_ph; ++ry)
        cp_async_bulk_tensor_4d(sWin + (uint32_t)(u & 1) * win_stride + (uint32_t)ry * row_bytes, &tmap, ch << 6, tx * 16 - 1 - a.win_m,
               ty * 8 - 1 - a.win_m + ry, b, win_full(u & 1));
    };
      issue_window_rows(0, 0, a.win_ph);
      int s = 0;
      for (int u = 0; u < n_units; ++u) {
        const int ch = u % nchunks;
        for (int tap = 0; tap < 9; ++tap, ++s) {
          const int stage = s % DP_SA;
          const uint32_t ph = (uint32_t)(s / DP_SA) & 1u;
          mbarrier_wait_parity(empty_bar(stage), ph ^ 1u);
          mbarrier_arrive_expect_tx(full_bar(stage), b_tile_bytes);        // the weight tile first: the MMA of this slice waits for it
          cp_async_bulk(sB + stage * b_tile_bytes, a.w + (size_t)(ch * 9 + tap) * a.n_tile * TC_BK, b_tile_bytes, full_bar(stage));
          // next unit's window into the other buffer, three rows per slice from tap 3 on: issuing a request costs this
          // thread ~100+ cycles, and 15 of them ahead of the first weight tiles of a unit stalled every tile boundary by
          // ~4000 cycles.  This warp runs at most DP_SA slices ahead of the producers, so by tap 3 they have released
          // the buffer (unit u - 1) and the wait below does not block.
          if (u + 1 < n_units && tap >= 3) {
            if (tap == 3 && u >= 1) mbarrier_wait_parity(win_empty((u + 1) & 1), (uint32_t)((u - 1) >> 1) & 1u);
            issue_window_rows(u + 1, 3 * (tap - 3), 3 * (tap - 3) + 3);
          }
        }
      }
    }
  } else if (warp == DP_PWARPS) {
    // ======================================= MMA issuer =======================================
    if (lane == 0) {
      const uint32_t idesc = umma_idesc_bf16_m128(a.n_tile);
      int s = 0;
      for (int t = 0; t < n_my; ++t) {
        const int ai = t & 1;
        mbarrier_wait_parity(acc_empty(ai), ((uint32_t)(t >> 1) & 1u) ^ 1u);
        tcgen05_fence_after_thread_sync();
        const uint32_t d_tmem = tmem_base + (uint32_t)(ai * a.n_tile);
        for (int sl = 0; sl < 9 * nchunks; ++sl, ++s) {
          const int stage = s % DP_SA;
          const uint32_t ph = (uint32_t)(s / DP_SA) & 1u;
          mbarrier_wait_parity(full_bar(stage), ph);
          fence_proxy_async_shared_cta();
          tcgen05_fence_after_thread_sync();
          if (s < 60) tc_stamp(trace, 16 + 4 * s + 2);
          const uint64_t ad = umma_sdesc_sw128(sA + stage * A_STAGE_BYTES);
          const uint64_t bd = umma_sdesc_sw128(sB + stage * b_tile_bytes);
#pragma unroll
          for (int k = 0; k < TC_BK / 16; ++k)
            tcgen05_mma(d_tmem, ad + 2ull * k, bd + 2ull * k, idesc, (sl > 0 || k > 0) ? 1u : 0u);
          tcgen05_commit(empty_bar(stage));
          if (s < 60) tc_stamp(trace, 16 + 4 * s + 3);
        }
        tcgen05_commit(acc_full(ai));
      }
    }
  } else {
    // ======================================= epilogue warps 17..20 (warp id % 4 = TMEM lane quarter) =======================================
    const int wq = warp & 3;                          // TMEM lane quarter this warp may read (warp id % 4)
    const int row = wq * 32 + lane;
    for (int t = 0; t < n_my; ++t) {
      const int ai = t & 1;
      int b, ty, tx;
      dp_tile_origin(a, (int)blockIdx.x + t * G, b, ty, tx);
      const int oy = ty * 8 + (row >> 4), ox = tx * 16 + (row & 15);
      const bool p_ok = oy < g.OH && ox < g.OW;
      const size_t p = ((size_t)b * g.OH + oy) * g.OW + ox;
      mbarrier_wait_parity(acc_full(ai), (uint32_t)(t >> 1) & 1u);
      tcgen05_fence_after_thread_sync();
      const uint32_t t_lane = tmem_base + ((uint32_t)(wq * 32) << 16) + (uint32_t)(ai * a.n_tile);
      for (int col = 0; col < a.n_tile; col += 16) {
        uint32_t r[16];
        tcgen05_ld_32x32b_x16(t_lane + (uint32_t)col, r);
        if (!p_ok || col >= g.C_out) continue;
        float v[16];
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] = __uint_as_float(r[j]);
        if (a.shift) {
          const float4* sh4 = reinterpret_cast<const float4*>(a.shift + col);
#pragma unroll
          for (int j4 = 0; j4 < 4; ++j4) {
            const float4 sh = __ldg(sh4 + j4);
            v[4 * j4] += sh.x; v[4 * j4 + 1] += sh.y; v[4 * j4 + 2] += sh.z; v[4 * j4 + 3] += sh.w;
          }
        }
        if (g.relu) {
#pragma unroll
          for (int j = 0; j < 16; ++j) v[j] = fmaxf(v[j], 0.f);
        }
        uint4 oa, ob;
        __nv_bfloat162* pa = reinterpret_cast<__nv_bfloat162*>(&oa);
        __nv_bfloat162* pb = reinterpret_cast<__nv_bfloat162*>(&ob);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          pa[j] = __floats2bfloat162_rn(v[2 * j], v[2 * j + 1]);
          pb[j] = __floats2bfloat162_rn(v[8 + 2 * j], v[8 + 2 * j + 1]);
        }
        uint4* op = reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(a.out) + p * g.ld_out + col);
        op[0] = oa; op[1] = ob;
      }
      tcgen05_fence_before_thread_sync();
      __syncwarp();
      if (lane == 0) mbarrier_arrive(acc_empty(ai));
    }
  }

  tcgen05_fence_before_thread_sync();
  __syncthreads();
  if (warp == DP_PWARPS) {
    tcgen05_fence_after_thread_sync();
    tcgen05_dealloc(tmem_base, (uint32_t)a.tmem_cols);
  }
}

int tc_set_trace(void* buf) {
  unsigned long long* p = (unsigned long long*)buf;
  return cudaMemcpyToSymbol(g_tc_trace, &p, sizeof(p)) == cudaSuccess ? CT_OK : CT_ERR_CUDA;
}

int conv_forward_tc(const ct_conv_desc* d, cudaStream_t st) {
  const bool x3 = d->engine == CT_ENGINE_TCGEN05_X3;     // fp32 activations, bf16 hi/lo split operands
  TcArgs a;
  a.g = make_geom(d);
  const ConvGeom& g = a.g;
  if (g.C_in % 8 != 0 || g.ld_in % 8 != 0)
    return fail(CT_ERR_INVALID, "conv_tc: C_in and ld_in must be multiples of 8%s (%ld,%ld)", "", g.C_in, g.ld_in);
  if (((uintptr_t)d->x & 15) || ((uintptr_t)d->w & 15) || ((uintptr_t)d->out & 15))
    return fail(CT_ERR_INVALID, "conv_tc: x/w/out must be 16-byte aligned%s", "");
  int n_tile = d->n_tile;
  if (n_tile <= 0 || n_tile % 16 != 0 || n_tile > 256)
    return fail(CT_ERR_INVALID, "conv_tc: n_tile must be a multiple of 16 in [16,256]%s (%ld)", "", n_tile);
  if (g.out_mode == CT_OUT_NHWC) {
    if (g.C_out % 16 != 0 || g.ld_out % 8 != 0)
      return fail(CT_ERR_INVALID, "conv_tc: NHWC output needs C_out %% 16 == 0 and ld_out %% 8 == 0%s", "");
    if (d->residual && (g.ld_res % 8 != 0 || ((uintptr_t)d->residual & 15)))
      return fail(CT_ERR_INVALID, "conv_tc: residual must be 16B aligned with ld_res %% 8 == 0%s", "");
  } else if (g.out_mode == CT_OUT_NHWC_F32) {
    if (d->residual) return fail(CT_ERR_INVALID, "conv_tc: residual unsupported for fp32 outputs%s", "");
  } else if (d->residual) {
    return fail(CT_ERR_INVALID, "conv_tc: residual unsupported for fp32 outputs%s", "");
  }
  if ((long long)g.B * g.H * g.W * g.ld_in >= (1ll << 31))
    return fail(CT_ERR_INVALID, "conv_tc: input tensor exceeds 2^31 elements (32-bit offsets)%s", "");
  a.x = (const __nv_bfloat16*)d->x;
  a.w = (const __nv_bfloat16*)d->w;
  a.shift = d->shift;
  a.residual = (const __nv_bfloat16*)d->residual;
  a.om = d->om;
  a.out = d->out;
  a.n_tile = n_tile;
  a.k_slices = (g.K_total + TC_BK - 1) / TC_BK;
  a.a_mode = d->a_mode;
  // CT_A_DCN_WIN needs 64-channel chunks and the bf16 engine; anything else samples from global memory (same results:
  // for C_in == 64 the two K orders coincide, otherwise the caller packed the weights chunk-major and must get WIN)
  const bool win = d->a_mode == CT_A_DCN_WIN;
  if (win && (x3 || g.C_in % 64 != 0))
    return fail(CT_ERR_INVALID, "conv_tc: CT_A_DCN_WIN needs the bf16 engine and C_in %% 64 == 0%s (%ld)", "", g.C_in);
  a.win_m = DCN_WIN_MARGIN;
  a.win_pw = 16 + 2 * a.win_m + 3;
  a.win_ph = 8 + 2 * a.win_m + 3;
  a.win_bytes = (uint32_t)(a.win_pw * a.win_ph * 128);
  int cols = 32;
  while (cols < n_tile) cols <<= 1;
  a.tmem_cols = cols;
  const size_t stage_bytes = (size_t)(x3 ? 2 : 1) * (A_STAGE_BYTES + n_tile * 128);
  auto smem_for = [&](int stg) {
    return (size_t)stg * stage_bytes + (2 * stg + 2) * 8 + 32 +
           (d->a_mode == CT_A_DCN ? 9 * TC_BM * sizeof(DcnEntry) : 0) +
           (win ? 9 * TC_BM * sizeof(DcnWinEntry) + 128 + a.win_bytes : 0) + 1024;
  };
  int stages = 4;                                   // keep >= 2 CTAs per SM when the tile allows it
  if (smem_for(stages) > 112 * 1024) stages = 3;
  if (d->a_mode == CT_A_DCN) {
    // the DCN gather, not the MMA, paces the pipeline: fewer stages leave more of the SM's 228 KB to L1, which
    // the bilinear corner reads (each input pixel is touched ~36 times) depend on
    stages = 2;
  }
  if (win) {
    // two CTAs per SM: table 18 KB + window 43 KB + stages x (16 KB + n_tile x 128 B) must stay under ~113 KB
    stages = 2;
    if (smem_for(2) > 113 * 1024) {                  // one CTA per SM anyway (wide N tile): deepen the pipeline instead
      stages = 4;
      while (stages > 2 && smem_for(stages) > 200 * 1024) --stages;
    }
    if (smem_for(stages) > 200 * 1024)
      return fail(CT_ERR_UNSUPPORTED, "conv_tc: DCN window does not fit in shared memory%s (%ld)", "", (long)smem_for(stages));
  }
  if (x3) {                                         // one CTA per SM (register-heavy producers): as deep as fits
    stages = 4;
    while (stages > 2 && smem_for(stages) > 200 * 1024) --stages;
    if (d->a_mode == CT_A_DCN && stages > 3) stages = 3;
    if (smem_for(stages) > 224 * 1024)
      return fail(CT_ERR_UNSUPPORTED, "conv_tc x3: tile does not fit in shared memory%s (%ld)", "", (long)n_tile);
  }
  if (stages > a.k_slices) stages = a.k_slices;
  a.stages = stages;
  const size_t smem = smem_for(stages);
  const int n_tiles = (g.C_out + n_tile - 1) / n_tile;
  a.tiles_x = a.tiles_y = 0;
  int m_tiles = (g.P_out + TC_BM - 1) / TC_BM;
  CUtensorMap tmap;
  memset(&tmap, 0, sizeof(tmap));
  if (win) {                                         // 8x16 patches (ragged at the right / bottom edge) + their windows
    a.tiles_x = (g.OW + 15) / 16;
    a.tiles_y = (g.OH + 7) / 8;
    m_tiles = g.B * a.tiles_x * a.tiles_y;
    // persistent form (a single N tile, bf16 NHWC output): one CTA per SM, two windows + two tables + two accumulators,
    // windows requested one row at a time (see dcn_persist_kernel)
    const size_t win_stride = ((size_t)a.win_bytes + 127) & ~(size_t)127;
    const size_t psmem = (size_t)DP_SA * (A_STAGE_BYTES + n_tile * 128) + 2 * win_stride + 2 * 9 * TC_BM * sizeof(DcnWinEntry) +
                         8 * (2 * DP_SA + 12) + 16 + 1024;
    const bool persist = n_tiles == 1 && g.out_mode == CT_OUT_NHWC && d->residual == nullptr && g.C_out % 16 == 0 &&
                         g.C_out == n_tile && ((uintptr_t)d->shift & 15) == 0 && psmem <= 227 * 1024;
    const int rc = encode_tmap_nhwc_bf16(&tmap, d->x, g.B, g.H, g.W, g.C_in, g.ld_in, 64, a.win_pw,
                                         persist ? 1 : a.win_ph, CU_TENSOR_MAP_SWIZZLE_NONE, "conv_tc");
    if (rc != CT_OK) return rc;
    if (persist) {
      int cols2 = 32;
      while (cols2 < 2 * n_tile) cols2 <<= 1;
      a.tmem_cols = cols2;
      CT_CUDA_OK(set_max_dynamic_smem_once((const void*)dcn_persist_kernel, 227 * 1024));
      const int sms = sm_count();
      const int pgrid = m_tiles < sms ? m_tiles : sms;
      CT_CUDA_OK(launch_kernel(dcn_persist_kernel, dim3(pgrid), dim3(DP_THREADS), psmem, st, true, a, m_tiles, tmap));
      return after_launch();
    }
  }
  dim3 grid(m_tiles, n_tiles);
  if (x3) {
    CT_CUDA_OK(set_max_dynamic_smem_once((const void*)conv_tc_kernel<true>, 227 * 1024));
    CT_CUDA_OK(launch_kernel(conv_tc_kernel<true>, grid, dim3(TC_THREADS), smem, st, true, a, tmap));
  } else {
    CT_CUDA_OK(set_max_dynamic_smem_once((const void*)conv_tc_kernel<false>, 200 * 1024));
    CT_CUDA_OK(launch_kernel(conv_tc_kernel<false>, grid, dim3(TC_THREADS), smem, st, true, a, tmap));
  }
  return after_launch();
}

}  // namespace ctb
