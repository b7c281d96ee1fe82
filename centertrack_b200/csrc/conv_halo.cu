// "Halo" tcgen05 convolution for stride-1 KxK layers whose weights fit in shared memory (C_in 8..256):
// the im2row-free design for the thin, high-resolution layers (stems, level0, the 64-channel 128x128
// layers, DCN offset convs, the fused head 3x3) where a per-tap gather is LSU-bound.
//
//   * Output tile = 8 (x) x 16 (y) pixels = 128 GEMM rows (32 x 4 for 1x1 convs writing NCHW planes).  Its input
//     neighbourhood (tile + halo) is fetched ONCE by TMA tensor copies (cp.async.bulk.tensor.4d, zero fill
//     outside the image = the conv's zero padding).  Staging modes: whole-pixel K-major rows of 32/64/128 bytes
//     with the matching hardware swizzle (C_in 16/32/64, and 64-channel chunks for C_in 128..256) -- one TMA
//     request per pixel row; C_in == 8 (the packed stem input): 16-byte rows, two taps paired in one K=16 MMA;
//     C_in == 48: un-swizzled 8-channel "planes" [halo_y][halo_x][8], one TMA request per plane.
//   * NO data is rearranged per tap: the A operand of tap (ky,kx) is the same shared-memory tile addressed
//     through a UMMA descriptor whose start address is shifted by (ky*pitch + kx) pixel rows (the UMMA swizzle is
//     a function of the shared-memory address, like the TMA's, so a shifted start needs no base-offset field);
//     SBO = halo row pitch: the next 8-row core-matrix group is the next tile row.
//   * Weights of one output-channel tile stay resident in shared memory for the CTA's lifetime
//     (persistent CTAs, static tile striding); 2 or 4 accumulator stages in TMEM so the epilogue of tile i
//     overlaps the MMAs of tile i+1 (and i+2); 2-4 halo stages.
//
// Warp roles (352 threads): warps 0-7 epilogue (warp w reads TMEM lanes 32(w%4)..; warps 0-3 take the even
// 16-column chunks, 4-7 the odd ones -- the epilogue is an instruction-latency chain, so two warps per SM
// sub-partition), warp 8 TMA producer, warps 9 and 10 MMA issuers (warp 9 also owns the TMEM allocation).
// TWO issuing warps because one thread sustains only one tcgen05.mma per ~100 cycles on B200 whatever N is
// (tools/mma_rate.cu: 91-115 cycles for N <= 128; two warps on separate accumulators reach 64.6 = the N=128 floor):
// warp 9 takes the even work items, warp 10 the odd ones; warp w owns accumulators w and w+2 and -- this matters --
// the halo stages of its own parity (stage = item % S with S even): a stage's full-barrier must only ever be
// waited on by ONE consumer warp, see the stage policy in conv_forward_halo().  Layers with few MMAs per item
// (the 1x1 heads) run a single MMA warp and three stages instead.
#include "conv_common.cuh"
#include "sm100.cuh"

namespace ctb {

constexpr int HT_W = 8, HT_H = 16;       // output tile (x, y)

// Optional timeline trace of CTA 0 (ct_debug_trace): 8 clock64() stamps per work item --
// 0 producer acquired the halo stage, 1 TMA issued, 2 MMA saw the halo, 3 MMA got a free accumulator,
// 4 MMAs issued + committed, 5 epilogue saw the accumulator, 6 epilogue released it.  Off (nullptr) by default.
__device__ unsigned long long* g_halo_trace = nullptr;
// The pointer is read once per thread at kernel entry: the MMA issuing thread is the critical resource of the thin layers
// and must not pay a dependent load per stamp when tracing is off.
__device__ __forceinline__ unsigned long long* h_trace_ptr() {
  unsigned long long* t = g_halo_trace;
  return (t != nullptr && blockIdx.x == 0) ? t : nullptr;
}
__device__ __forceinline__ void h_stamp(unsigned long long* t, int it, int k) {
  if (t != nullptr && it < 256) t[it * 8 + k] = (unsigned long long)clock64();
}
constexpr int H_THREADS = 352;           // 8 epilogue warps + TMA warp + 2 MMA warps
constexpr int H_EPI_WARPS = 8;

struct HaloArgs {
  ConvGeom g;
  const __nv_bfloat16* w;       // packed blocks (see ct_pack_weights, engine HALO)
  const float* shift;
  const __nv_bfloat16* residual;
  void* out;
  int n_tile, n_tiles_n, nblk, planes, pw, ph, plane_bytes, box_bytes, halo_stages, tmem_cols;
  int tw, th;                           // output tile: 8 x 16, or 32 x 4 for 1x1 convs writing NCHW planes
  int nacc;                             // TMEM accumulator stages (4 when 4*n_tile <= 512 columns, else 2)
  int mma_warps;                        // 2, or 1 when an item has few MMAs (nblk <= 16)
  int tiles_x, tiles_y, tiles_total;    // spatial tiles per image / total work items (incl. n tiles)
  int pair_taps;                        // 1: C_in == 8, one MMA = taps (kx, kx+1)
  int swz;                              // 0: un-swizzled 8-channel planes; else row bytes (32/64/128): whole
                                        //    pixel (all C_in channels) per K-major row, hardware swizzle
  int merged_xc;                        // 1: 3-D tensor map with (x, c) merged (C_in == ld_in == 8)
  int out_s2d;                          // CT_OUT_NHWC_S2D: pixel index remapped in the epilogue (g.out_mode = CT_OUT_NHWC)
  int sum3;                             // != 0: stem epilogue sum_g relu(group g + shift) -> 16 ch; bit g = group present
  uint32_t w_bytes;                     // bytes of one n-tile's weights
  // A-descriptor walk of one work item (all in 16-byte units, warp-uniform): for ky, kx|pair, chunk, kstep
  int m_nky, m_nkx, m_nc, m_nq;
  uint32_t m_sky, m_skx, m_sc, m_sq, m_alo, m_ahi;
};

// Watchdog report: when ct_debug_trace's buffer is host-mapped memory, a stuck wait leaves (site code, item,
// blockIdx, warp) in its last 4 words before trapping, so a protocol bug can be located post mortem.
__device__ volatile unsigned int* g_halo_dbg = nullptr;
__device__ __forceinline__ void halo_wait(uint32_t bar, uint32_t parity, int site, int item) {
  uint32_t spins = 0;
  while (!mbarrier_try_wait_parity(bar, parity)) {
    if (++spins > 4000000u) {
      volatile unsigned int* d = g_halo_dbg;
      if (d != nullptr && (threadIdx.x & 31) == 0) {
        d[0] = (unsigned)site; d[1] = (unsigned)item; d[2] = blockIdx.x; d[3] = threadIdx.x >> 5;
        __threadfence_system();
      }
      __trap();
    }
  }
}

__global__ void __launch_bounds__(H_THREADS, 2)
conv_halo_kernel(const HaloArgs a, const __grid_constant__ CUtensorMap tmap) {
  extern __shared__ __align__(1024) unsigned char hsm_dyn[];
  unsigned char* sm = hsm_dyn + ((1024u - (smem_u32(hsm_dyn) & 1023u)) & 1023u);
  const ConvGeom& g = a.g;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  unsigned long long* const trace = h_trace_ptr();
  const int S = a.halo_stages;
  const uint32_t halo_bytes = (uint32_t)a.planes * a.plane_bytes;

  // smem: [weights][halo stage 0..S-1][barriers][tmem slot]
  const uint32_t base = smem_u32(sm);
  const uint32_t sW = base;
  const uint32_t sH = base + ((a.w_bytes + 1023u) & ~1023u);
  const uint32_t off_bar = ((a.w_bytes + 1023u) & ~1023u) + S * halo_bytes;
  const uint32_t bars = base + off_bar;
  // barriers: w_full, halo_full[S], halo_empty[S], tmem_full[4], tmem_empty[4]
  const uint32_t w_full = bars;
  auto halo_full = [&](int s) { return bars + 8u * (1 + s); };
  auto halo_empty = [&](int s) { return bars + 8u * (1 + S + s); };
  auto tmem_full = [&](int s) { return bars + 8u * (1 + 2 * S + s); };
  auto tmem_empty = [&](int s) { return bars + 8u * (5 + 2 * S + s); };
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(sm + off_bar + 8 * (9 + 2 * S));
  const int NACC = a.nacc;

  pdl_trigger();                       // the next kernel of the stream may start its own prologue now
  if (tid == 0) {
    mbarrier_init(w_full, 1);
    for (int s = 0; s < S; ++s) { mbarrier_init(halo_full(s), 1); mbarrier_init(halo_empty(s), 1); }
    for (int s = 0; s < 4; ++s) { mbarrier_init(tmem_full(s), 1); mbarrier_init(tmem_empty(s), H_EPI_WARPS); }
    fence_mbarrier_init();
  }
  if (warp == 9) {
    tcgen05_alloc(smem_u32((const void*)tmem_slot), (uint32_t)a.tmem_cols);
    tcgen05_relinquish_alloc_permit();
  }
  // folded-BN shift / bias of this CTA's output-channel tile, staged once (read as float4 broadcasts)
  float* s_shift = reinterpret_cast<float*>(sm + off_bar + 256);      // barriers + TMEM slot use 204 bytes at S = 8 (< 256)
  {
    const int n0s = (blockIdx.x % a.n_tiles_n) * a.n_tile;
    for (int j = tid; j < 256; j += H_THREADS)
      s_shift[j] = (a.shift && j < a.n_tile && n0s + j < g.C_out) ? __ldg(a.shift + n0s + j) : 0.f;
  }
  tcgen05_fence_before_thread_sync();
  __syncthreads();
  tcgen05_fence_after_thread_sync();
  const uint32_t tmem_base = *tmem_slot;
  // the weights are constants: their bulk copy goes out BEFORE waiting for the previous kernel (PDL), so that it
  // overlaps that kernel's tail; everything after the wait reads activations the previous kernel produced
  if (warp == 8 && lane == 0) {
    mbarrier_arrive_expect_tx(w_full, a.w_bytes);
    cp_async_bulk(sW, reinterpret_cast<const unsigned char*>(a.w) + (size_t)(blockIdx.x % a.n_tiles_n) * a.w_bytes, a.w_bytes, w_full);
  }
  pdl_wait();

  // work items: n-tile major so that a CTA keeps ONE weight tile resident:  item = nt * spatial + sp
  // CTA c handles n-tile (c % n_tiles_n) and spatial tiles (c / n_tiles_n) + i * (gridDim.x / n_tiles_n)
  const int nt = blockIdx.x % a.n_tiles_n;
  const int sp0 = blockIdx.x / a.n_tiles_n;
  const int sp_stride = gridDim.x / a.n_tiles_n;
  const int sp_total = a.tiles_total;
  const int n0 = nt * a.n_tile;
  const int per_img = a.tiles_x * a.tiles_y;

  if (warp == 8) {
    if (lane == 0) {
      // ===================== TMA producer =====================
      int it = 0;
      for (int sp = sp0; sp < sp_total; sp += sp_stride, ++it) {
        const int s = it % S;
        const uint32_t ph = (uint32_t)(it / S) & 1u;
        halo_wait(halo_empty(s), ph ^ 1u, 1, it);
        h_stamp(trace, it, 0);
        const int b = sp / per_img, r = sp - b * per_img;
        const int ty = r / a.tiles_x, tx = r - ty * a.tiles_x;
        const int x0 = tx * a.tw - g.pad, y0 = ty * a.th - g.pad;
        mbarrier_arrive_expect_tx(halo_full(s), (uint32_t)(a.planes * a.box_bytes));   // TMA writes the full box (zero fill incl.)
        if (a.merged_xc) {
          cp_async_bulk_tensor_3d(sH + s * halo_bytes, &tmap, x0 * 8, y0, b, halo_full(s));
        } else {
          // un-swizzled: one 8-channel plane per copy; swizzled: one <=64-channel chunk (whole 128-byte rows)
          const int cstep = a.swz ? (a.swz >> 1) : 8;
          for (int p = 0; p < a.planes; ++p)
            cp_async_bulk_tensor_4d(sH + s * halo_bytes + p * a.plane_bytes, &tmap, p * cstep, x0, y0, b, halo_full(s));
        }
        h_stamp(trace, it, 1);
      }
    }
  } else if (warp == 9 || warp == 10) {
    // ===================== MMA issuers =====================
    // The whole warp runs this loop CONVERGENTLY and only the tcgen05.mma / commit statements are predicated on
    // the leader lane: the descriptors are then warp-uniform arithmetic on kernel parameters and loop counters,
    // which the compiler keeps in uniform registers.  (Issuing from a divergent `if (lane == 0)` region, or reading
    // descriptors from a shared-memory table, costs several R2UR moves per UTCHMMA: ~100 cycles per MMA.)
    const bool leader = lane == 0;
    const uint32_t idesc = umma_idesc_bf16_m128(a.n_tile);
    const uint32_t b_hi = (uint32_t)(umma_sdesc_none(0, (uint32_t)a.n_tile * 16u, 128u) >> 32);
    const uint32_t b_lo0 = (uint32_t)umma_sdesc_none(sW, (uint32_t)a.n_tile * 16u, 128u);
    const uint32_t b_step = ((uint32_t)a.n_tile * 32u) >> 4;          // descriptor start-address units (16 B)
    // per-warp table of A-descriptor low words for halo stage 0 (walk: ky, kx|pair, chunk, K-step)
    uint32_t* a_tab = reinterpret_cast<uint32_t*>(sm + off_bar + 256 + 1024) + (warp - 9) * 160;
    for (int blk = lane; blk < a.nblk; blk += 32) {
      int r = blk;
      const int q = r % a.m_nq; r /= a.m_nq;
      const int c = r % a.m_nc; r /= a.m_nc;
      const int kx = r % a.m_nkx, ky = r / a.m_nkx;
      a_tab[blk] = a.m_alo + (sH >> 4) + (uint32_t)ky * a.m_sky + (uint32_t)kx * a.m_skx + (uint32_t)c * a.m_sc +
                   (uint32_t)q * a.m_sq;
    }
    __syncwarp();
    halo_wait(w_full, 0, 2, 0);
    {
      const int parity = warp - 9;                         // this warp's items: it % mma_warps == parity
      const int nw = a.mma_warps;
      int it = parity;
      for (int sp = sp0 + parity * sp_stride; sp < sp_total && parity < nw; sp += nw * sp_stride, it += nw) {
        const int s = it % S;
        const uint32_t ph = (uint32_t)(it / S) & 1u;
        const int acc = it % NACC;                 // warp `parity` owns accumulators parity, parity + 2
        const uint32_t pa = (uint32_t)(it / NACC) & 1u;
        halo_wait(halo_full(s), ph, 3, it);
        if (leader) h_stamp(trace, it, 2);
        halo_wait(tmem_empty(acc), pa ^ 1u, 4, it);
        if (leader) h_stamp(trace, it, 3);
        tcgen05_fence_after_thread_sync();
        const uint32_t stage16 = ((uint32_t)s * halo_bytes) >> 4;      // start address field stays < 2^14
        const uint32_t d_tmem = tmem_base + (uint32_t)(acc * a.n_tile);
        uint32_t b_lo = b_lo0;
        uint32_t accum = 0;
        // A-descriptor low words of this item's MMAs: one shared-memory load per 32 MMAs (lane j holds block j),
        // then a register shuffle + add per MMA -- nothing else varies (B advances by a uniform step)
        for (int blk0 = 0; blk0 < a.nblk; blk0 += 32) {
          const uint32_t mine = a_tab[min(blk0 + lane, a.nblk - 1)];
          const int cnt = min(32, a.nblk - blk0);
          for (int j = 0; j < cnt; ++j) {
            const uint32_t a_lo = __shfl_sync(0xffffffffu, mine, j) + stage16;
            tcgen05_mma_elect(d_tmem, ((uint64_t)a.m_ahi << 32) | (uint64_t)a_lo, ((uint64_t)b_hi << 32) | (uint64_t)b_lo,
                        idesc, accum);
            accum = 1;
            b_lo += b_step;
          }
        }
        tcgen05_commit_elect(halo_empty(s));
        tcgen05_commit_elect(tmem_full(acc));
        if (leader) h_stamp(trace, it, 4);
      }
    }
  } else {
    // ===================== epilogue warps 0..7 =====================
    const int wq = warp & 3, chalf = warp >> 2;
    const int row = wq * 32 + lane;              // GEMM row = g*8 + r  ->  pixel (ty*16 + g, tx*8 + r)
    // 8 consecutive GEMM rows = 8 consecutive x; the 8-row groups then run along x (tw / 8 of them) before y
    const int gpr = a.tw >> 3;
    const int gy = (row >> 3) / gpr, rx = (((row >> 3) % gpr) << 3) | (row & 7);
    const int HWo = g.OH * g.OW;
    // Residual tiles are prefetched one work item ahead into registers (the load does not depend on the MMA):
    // issued right after the previous item consumed its copy, they land while this warp waits for the next
    // accumulator -- otherwise every item pays a full L2/HBM round trip inside the serial epilogue chain.
    constexpr int PF = 2;                      // 16-column chunks per warp that can be prefetched (n_tile <= 64)
    uint4 rq[PF][2];
    const bool use_res = a.residual != nullptr && g.out_mode == CT_OUT_NHWC && !a.sum3;
    auto prefetch_residual = [&](int sp_n) {
      const int bn = sp_n / per_img, rn = sp_n - bn * per_img;
      const int tyn = rn / a.tiles_x, txn = rn - tyn * a.tiles_x;
      const int oyn = tyn * a.th + gy, oxn = txn * a.tw + rx;
      const bool okn = oyn < g.OH && oxn < g.OW;
      const size_t pn = ((size_t)bn * g.OH + oyn) * g.OW + oxn;
#pragma unroll
      for (int i = 0; i < PF; ++i) {
        const int col = chalf * 16 + 32 * i;
        rq[i][0] = make_uint4(0, 0, 0, 0); rq[i][1] = make_uint4(0, 0, 0, 0);
        if (okn && col < a.n_tile && n0 + col < g.C_out) {
          const uint4* rp = reinterpret_cast<const uint4*>(a.residual + pn * g.ld_res + n0 + col);
          rq[i][0] = __ldg(rp); rq[i][1] = __ldg(rp + 1);
        }
      }
    };
    if (use_res && sp0 < sp_total) prefetch_residual(sp0);
    int it = 0;
    for (int sp = sp0; sp < sp_total; sp += sp_stride, ++it) {
      const int acc = it % NACC;
      const uint32_t pa = (uint32_t)(it / NACC) & 1u;
      const int b = sp / per_img, r = sp - b * per_img;
      const int ty = r / a.tiles_x, tx = r - ty * a.tiles_x;
      const int oy = ty * a.th + gy, ox = tx * a.tw + rx;
      const bool p_ok = oy < g.OH && ox < g.OW;
      const size_t p = a.out_s2d ? ((((size_t)b * (g.OH >> 1) + (oy >> 1)) * (g.OW >> 1) + (ox >> 1)) << 2) + (((oy & 1) << 1) | (ox & 1))
                                 : ((size_t)b * g.OH + oy) * g.OW + ox;
      halo_wait(tmem_full(acc), pa, 5, it);
      if (tid == 0) h_stamp(trace, it, 6 - 1);
      tcgen05_fence_after_thread_sync();
      const uint32_t t_lane = tmem_base + ((uint32_t)(wq * 32) << 16) + (uint32_t)(acc * a.n_tile);
      if (a.sum3) {
        // stem: three 16-channel groups, ReLU each (after its folded-BN shift), then sum (dla.py:307-311).
        // Warp half `chalf` produces output channels 8*chalf .. 8*chalf+7 (columns g*16 + 8*chalf + j).
        float s8[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) s8[j] = 0.f;
#pragma unroll
        for (int grp = 0; grp < 3; ++grp) {
          uint32_t rr[8];
          tcgen05_ld_32x32b_x8(t_lane + grp * 16 + chalf * 8, rr);
          if (!((a.sum3 >> grp) & 1)) continue;          // absent input (pre_img / pre_hm is None)
          const float4* sh4 = reinterpret_cast<const float4*>(s_shift + grp * 16 + chalf * 8);
          const float4 sa = sh4[0], sb = sh4[1];
          s8[0] += fmaxf(__uint_as_float(rr[0]) + sa.x, 0.f); s8[1] += fmaxf(__uint_as_float(rr[1]) + sa.y, 0.f);
          s8[2] += fmaxf(__uint_as_float(rr[2]) + sa.z, 0.f); s8[3] += fmaxf(__uint_as_float(rr[3]) + sa.w, 0.f);
          s8[4] += fmaxf(__uint_as_float(rr[4]) + sb.x, 0.f); s8[5] += fmaxf(__uint_as_float(rr[5]) + sb.y, 0.f);
          s8[6] += fmaxf(__uint_as_float(rr[6]) + sb.z, 0.f); s8[7] += fmaxf(__uint_as_float(rr[7]) + sb.w, 0.f);
        }
        if (p_ok) {
          uint4 o;
          __nv_bfloat162* po = reinterpret_cast<__nv_bfloat162*>(&o);
#pragma unroll
          for (int j = 0; j < 4; ++j) po[j] = __floats2bfloat162_rn(s8[2 * j], s8[2 * j + 1]);
          *reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(a.out) + p * g.ld_out + chalf * 8) = o;
        }
      } else {
        for (int col = chalf * 16; col < a.n_tile; col += 32) {
          uint32_t rr[16];
          tcgen05_ld_32x32b_x16(t_lane + (uint32_t)col, rr);
          if (tid == 0 && col == 0) h_stamp(trace, it, 7);
          const int o0 = n0 + col;
          if (!p_ok || o0 >= g.C_out) continue;
          float v[16];
          const float4* sh4 = reinterpret_cast<const float4*>(s_shift + col);
#pragma unroll
          for (int j4 = 0; j4 < 4; ++j4) {
            const float4 sh = sh4[j4];
            v[4 * j4 + 0] = __uint_as_float(rr[4 * j4 + 0]) + sh.x;
            v[4 * j4 + 1] = __uint_as_float(rr[4 * j4 + 1]) + sh.y;
            v[4 * j4 + 2] = __uint_as_float(rr[4 * j4 + 2]) + sh.z;
            v[4 * j4 + 3] = __uint_as_float(rr[4 * j4 + 3]) + sh.w;
          }
          if (g.out_mode == CT_OUT_NHWC) {
            if (a.residual) {
              uint4 ra, rb;
              const int ci = col >> 5;                     // this warp's chunk index
              if (ci < PF) {
                ra = rq[0][0]; rb = rq[0][1];
#pragma unroll
                for (int i = 1; i < PF; ++i) if (ci == i) { ra = rq[i][0]; rb = rq[i][1]; }
              } else {
                const uint4* rp = reinterpret_cast<const uint4*>(a.residual + p * g.ld_res + o0);
                ra = __ldg(rp); rb = __ldg(rp + 1);
              }
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
            __nv_bfloat162* pa2 = reinterpret_cast<__nv_bfloat162*>(&oa);
            __nv_bfloat162* pb2 = reinterpret_cast<__nv_bfloat162*>(&ob);
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              pa2[j] = __floats2bfloat162_rn(v[2 * j], v[2 * j + 1]);
              pb2[j] = __floats2bfloat162_rn(v[8 + 2 * j], v[8 + 2 * j + 1]);
            }
            uint4* op = reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(a.out) + p * g.ld_out + o0);
            op[0] = oa; op[1] = ob;
          } else if (g.out_mode == CT_OUT_NHWC_F32) {
            float* op = reinterpret_cast<float*>(a.out) + p * g.ld_out + o0;
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              if (g.relu) v[j] = fmaxf(v[j], 0.f);
              const float sg = sigmoidf_fast(v[j]);            // unconditional: keeps the 16 chains interleaved
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
            float* op = reinterpret_cast<float*>(a.out) + ((size_t)b * g.C_out + o0) * HWo + (size_t)oy * g.OW + ox;
            // transform all 16 values in straight-line code (the activation kind is uniform: hoisted out of the
            // loop), then the guarded stores -- per-element branches serialise the ex2/rcp chains (~190 cycles each)
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
      }
      if (use_res && sp + sp_stride < sp_total) prefetch_residual(sp + sp_stride);
      tcgen05_fence_before_thread_sync();
      __syncwarp();
      if (lane == 0) mbarrier_arrive(tmem_empty(acc));      // one arrival per epilogue warp frees the accumulator
      if (tid == 0) h_stamp(trace, it, 6);
    }
  }

  tcgen05_fence_before_thread_sync();
  __syncthreads();
  if (warp == 9) {
    tcgen05_fence_after_thread_sync();
    tcgen05_dealloc(tmem_base, (uint32_t)a.tmem_cols);
  }
}

// ---- host ----
int halo_set_trace(void* buf) {
  unsigned long long* p = (unsigned long long*)buf;
  return cudaMemcpyToSymbol(g_halo_trace, &p, sizeof(p)) == cudaSuccess ? CT_OK : CT_ERR_CUDA;
}
int halo_set_watch(void* mapped_host_buf) {
  unsigned int* p = (unsigned int*)mapped_host_buf;
  return cudaMemcpyToSymbol(g_halo_dbg, &p, sizeof(p)) == cudaSuccess ? CT_OK : CT_ERR_CUDA;
}

int halo_blocks(int C_in, int KH, int KW) {
  return C_in == 8 ? KH * ((KW + 1) / 2) : KH * KW * (C_in / 16);
}

int conv_forward_halo(const ct_conv_desc* d, cudaStream_t st) {
  HaloArgs a;
  a.g = make_geom(d);
  const ConvGeom& g = a.g;
  if (g.stride != 1 || g.pad != g.KH / 2 || g.KH != g.KW || g.OH != g.H || g.OW != g.W)
    return fail(CT_ERR_INVALID, "conv_halo: stride-1 'same' convolutions only%s", "");
  if (!(g.C_in == 8 || (g.C_in % 16 == 0 && g.C_in <= 64) || (g.C_in % 64 == 0 && g.C_in <= 256)) || g.ld_in % 8 != 0)
    return fail(CT_ERR_INVALID, "conv_halo: C_in must be 8, 16, 32, 48, 64, 128, 192 or 256 (ld_in %% 8 == 0)%s (%ld)", "", g.C_in);
  const int n_tile = d->n_tile;
  if (n_tile <= 0 || n_tile % 16 != 0 || n_tile > 256)
    return fail(CT_ERR_INVALID, "conv_halo: bad n_tile%s (%ld)", "", n_tile);
  if (((uintptr_t)d->x & 15) || ((uintptr_t)d->w & 15) || ((uintptr_t)d->out & 15))
    return fail(CT_ERR_INVALID, "conv_halo: x/w/out must be 16-byte aligned%s", "");
  a.sum3 = d->epilogue_sum3;
  a.out_s2d = 0;
  if (g.out_mode == CT_OUT_NHWC_S2D) {
    if ((g.OH | g.OW) & 1 || d->residual)
      return fail(CT_ERR_INVALID, "conv_halo: CT_OUT_NHWC_S2D needs even OH / OW, no residual%s", "");
    a.out_s2d = 1;
    a.g.out_mode = CT_OUT_NHWC;
  }
  if (a.sum3 && !(g.C_out == 48 && n_tile == 48 && g.out_mode == CT_OUT_NHWC && d->shift))
    return fail(CT_ERR_INVALID, "conv_halo: sum3 epilogue needs C_out == n_tile == 48, NHWC output, shift%s", "");
  if (g.out_mode == CT_OUT_NHWC && !a.sum3 && (g.C_out % 16 != 0 || g.ld_out % 8 != 0))
    return fail(CT_ERR_INVALID, "conv_halo: NHWC bf16 output needs C_out %% 16 == 0, ld_out %% 8 == 0%s", "");
  if (d->residual && (g.out_mode != CT_OUT_NHWC || g.ld_res % 8 != 0 || ((uintptr_t)d->residual & 15)))
    return fail(CT_ERR_INVALID, "conv_halo: residual only for NHWC bf16 outputs, 16B aligned%s", "");
  a.w = (const __nv_bfloat16*)d->w;
  a.shift = d->shift;
  a.residual = (const __nv_bfloat16*)d->residual;
  a.out = d->out;
  a.n_tile = n_tile;
  a.n_tiles_n = (g.C_out + n_tile - 1) / n_tile;
  a.pair_taps = g.C_in == 8;
  a.nblk = halo_blocks(g.C_in, g.KH, g.KW);
  if (a.nblk > 160) return fail(CT_ERR_UNSUPPORTED, "conv_halo: more than 160 K=16 blocks per tile%s (%ld)", "", (long)a.nblk);
  // operand staging mode: whole-pixel swizzled rows when C_in*2 is a swizzle width (one 32/64/128-byte TMA
  // request per halo pixel); C_in == 8 keeps the 16-byte un-swizzled rows but merges (x, c) in the tensor map
  // when the tensor is dense (ld_in == 8) so that one request covers a whole halo row; C_in == 48 stages un-swizzled
  // 8-channel planes.
  a.swz = (g.C_in > 64) ? 128 : ((g.C_in == 16 || g.C_in == 32 || g.C_in == 64) ? g.C_in * 2 : 0);
  a.merged_xc = (g.C_in == 8 && g.ld_in == 8) ? 1 : 0;
  a.planes = a.swz ? (g.C_in * 2 + a.swz - 1) / a.swz : g.C_in / 8;   // swizzled: 64-channel chunks
  // 1x1 convs writing fp32 NCHW planes (the 1x1 heads) use a 32 x 4 pixel tile: there is no halo, the TMA box
  // [4][32][c] is already the canonical K-major operand (8-pixel groups 8 rows apart), and every epilogue warp then
  // owns 32 consecutive x of one row: its per-channel store is one full 128-byte line instead of four 32-byte pieces.
  a.tw = HT_W; a.th = HT_H;
  if (g.KH == 1 && g.KW == 1 && g.out_mode == CT_OUT_NCHW_F32 && a.swz && g.OW % 32 == 0 && g.OH % 4 == 0) {
    a.tw = 32; a.th = 4;
  }
  a.pw = a.tw + g.KW - 1 + (a.pair_taps ? 1 : 0);
  a.ph = a.th + g.KH - 1;
  a.box_bytes = a.pw * a.ph * (a.swz ? a.swz : 16);
  a.plane_bytes = (a.box_bytes + 1023) / 1024 * 1024;
  a.w_bytes = (uint32_t)a.nblk * n_tile * 32u;
  if (a.pair_taps) {                 // one MMA = taps (ky, 2kp) and (ky, 2kp+1): K-core 1 is the next pixel
    a.m_nky = g.KH; a.m_nkx = (g.KW + 1) / 2; a.m_nc = 1; a.m_nq = 1;
    a.m_sky = a.pw; a.m_skx = 2; a.m_sc = 0; a.m_sq = 0;
    a.m_alo = 1u << 16;                                   // LBO = 16 B
    a.m_ahi = (uint32_t)a.pw | (1u << 14);                // SBO = pw*16 B, version 1
  } else if (a.swz) {
    const uint32_t rb16 = (uint32_t)a.swz >> 4;
    a.m_nky = g.KH; a.m_nkx = g.KW; a.m_nc = a.planes; a.m_nq = (g.C_in < 64 ? g.C_in : 64) / 16;
    a.m_sky = (uint32_t)a.pw * rb16; a.m_skx = rb16; a.m_sc = (uint32_t)a.plane_bytes >> 4; a.m_sq = 2;
    a.m_alo = 1u << 16;
    const uint32_t layout = a.swz == 128 ? 2u : (a.swz == 64 ? 4u : 6u);
    const uint32_t sbo16 = a.tw == HT_W ? (uint32_t)a.pw * rb16 : 8u * rb16;     // next 8-row group: next tile row / next 8 px
    a.m_ahi = sbo16 | (1u << 14) | (layout << 29);
  } else {
    a.m_nky = g.KH; a.m_nkx = g.KW; a.m_nc = 1; a.m_nq = g.C_in / 16;
    a.m_sky = a.pw; a.m_skx = 1; a.m_sc = 0; a.m_sq = 2u * ((uint32_t)a.plane_bytes >> 4);
    a.m_alo = ((uint32_t)a.plane_bytes >> 4) << 16;       // LBO = plane stride
    a.m_ahi = (uint32_t)a.pw | (1u << 14);
  }
  a.tiles_x = (g.OW + a.tw - 1) / a.tw;
  a.tiles_y = (g.OH + a.th - 1) / a.th;
  a.tiles_total = g.B * a.tiles_x * a.tiles_y;
  int cols = 32;
  // Two accumulators per MMA warp when TMEM allows (warp w owns accumulators w and w + 2): a warp can start its next
  // item while the epilogue still drains the previous one (~15 % on the 64-channel layers).
  a.nacc = 4 * n_tile <= 512 ? 4 : 2;
  while (cols < a.nacc * n_tile) cols <<= 1;
  if (cols > 512) return fail(CT_ERR_INVALID, "conv_halo: n_tile too large for double-buffered TMEM%s", "");
  a.tmem_cols = cols;
  const size_t halo_bytes = (size_t)a.planes * a.plane_bytes;
  auto smem_for = [&](int s) { return (size_t)((a.w_bytes + 1023) & ~1023u) + s * halo_bytes + 256 + 1024 + 2 * 160 * 4 + 1024; };
  // co-resident CTAs per SM with s halo stages: shared memory, TMEM columns, register file (2 x 352 threads x 80 registers)
  auto ctas_for = [&](int s) {
    int n = (int)((227 * 1024) / smem_for(s));
    if (n > 512 / cols) n = 512 / cols;
    return n > 2 ? 2 : n;
  };
  // Halo stages.  With two MMA warps taking alternate items, every stage must always be consumed by the SAME warp
  // (stage = item % S with S even): a warp that saw only every other phase of a stage's full-barrier could not tell
  // "my item has landed" from "the other warp's previous item has not landed yet" (same phase parity) and would
  // run its MMAs on a half-loaded tile -- observed as rare wrong tiles / hangs with S = 3.  Layers with few MMAs
  // per item (1x1 heads: TMA-latency bound, want three stages in flight) use ONE MMA warp and any S instead.
  a.mma_warps = a.nblk <= 16 ? 1 : 2;
  int stages;
  if (a.mma_warps == 2) {
    // as many (even) stages as keep the CTAs-per-SM count: the TMA of a thin-channel halo (32-byte rows) takes ~4200
    // cycles to land (tools/halo_trace.py, level0), so with two stages per MMA warp the item period WAS the TMA latency / 2
    stages = 2;
    for (int sdeep = 8; sdeep >= 4; sdeep -= 2)
      if (smem_for(sdeep) <= 220 * 1024 && ctas_for(sdeep) == ctas_for(2)) { stages = sdeep; break; }
  } else {
    stages = 3;
    while (stages > 2 && (smem_for(stages) > 220 * 1024 || ctas_for(stages) != ctas_for(2))) --stages;
  }
  if (a.mma_warps == 2 && (stages & 1))
    return fail(CT_ERR_INVALID, "conv_halo: two MMA warps need an even number of halo stages%s", "");
  if (smem_for(stages) > 227 * 1024)
    return fail(CT_ERR_UNSUPPORTED, "conv_halo: weights + halo do not fit in shared memory%s (%ld bytes)", "",
                (long)smem_for(stages));
  a.halo_stages = stages;
  const size_t smem = smem_for(stages);

  CUtensorMap tmap;
  int rc;
  if (a.merged_xc) {
    const cuuint64_t dims[3] = {(cuuint64_t)g.W * 8, (cuuint64_t)g.H, (cuuint64_t)g.B};
    const cuuint64_t strides[2] = {(cuuint64_t)g.W * 16, (cuuint64_t)g.H * g.W * 16};
    const cuuint32_t box[3] = {(cuuint32_t)a.pw * 8, (cuuint32_t)a.ph, 1};
    rc = encode_tmap_bf16(&tmap, d->x, 3, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_NONE, "conv_halo");
  } else {
    const CUtensorMapSwizzle sw = a.swz == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                                  : a.swz == 64 ? CU_TENSOR_MAP_SWIZZLE_64B
                                  : a.swz == 32 ? CU_TENSOR_MAP_SWIZZLE_32B : CU_TENSOR_MAP_SWIZZLE_NONE;
    rc = encode_tmap_nhwc_bf16(&tmap, d->x, g.B, g.H, g.W, g.C_in, g.ld_in, a.swz ? a.swz / 2 : 8, a.pw, a.ph, sw,
                               "conv_halo");
  }
  if (rc != CT_OK) return rc;

  CT_CUDA_OK(set_max_dynamic_smem_once((const void*)conv_halo_kernel, 227 * 1024));
  // persistent grid: a multiple of n_tiles_n, at most (SMs x CTAs that fit) and no more than the work
  long groups = (long)sm_count() * ctas_for(stages) / a.n_tiles_n;
  if (groups < 1) groups = 1;
  if (groups > a.tiles_total) groups = a.tiles_total;
  const int grid = (int)(groups * a.n_tiles_n);
  CT_CUDA_OK(launch_kernel(conv_halo_kernel, dim3(grid), dim3(H_THREADS), smem, st, true, a, tmap));
  return after_launch();
}

}  // namespace ctb
