// Fused heat-map decode: 3x3 max-equals NMS + per-class top-K + cross-class top-K + gather of every
// regression head + box assembly (+ pose keypoint refinement), ONE launch, ONE packed record buffer.
// Restates utils.py:16-26,52-87 and decode.py:11-182 of the reference.
//
// Ordering rule (the reference leaves ties to torch.topk, SURVEY hazard H1): value descending, then
// flat index ascending -- implemented as an exact radix select on the 64-bit key
//   key = (float_bits(value) << 32) | (0xFFFFFFFF - index)        (values are >= 0 after sigmoid)
// so indices are bit-exact with the oracle on every input, ties included.
//
// grid = (C + J planes, B); each CTA streams one class plane from HBM once, straight into registers (rolling
// 3-row NMS, 16-byte loads, neighbours by shuffle), compacts the kept positive peaks as 64-bit keys into shared
// memory and selects its top-K there; the last CTA of a batch element to finish merges the C*K candidates by
// (value, class, index) and writes the K records.
#include "common.cuh"
#include "sm100.cuh"

namespace ctb {

constexpr int DT = 512;          // threads per CTA (3 CTAs per SM: 40 registers, 37 KB of shared memory each)
constexpr int MAXK = 512;
constexpr int PEAK_CAP = 4096;   // compact list of kept positive peaks (64-bit keys), 32 KB
constexpr int PLANE_CAP = 65536; // bytes of one class plane staged in shared memory by bulk copies (128 x 128 fp32)
constexpr int DEC_NCH = 4;       // ... in this many row chunks, one mbarrier each

struct DecodeArgs {
  ct_decode_desc d;
  int* counters;
  unsigned long long* cand;      // [B][C+J][K]
  int kpad;                      // pow2 >= K
  int bulk;                      // 1: planes are staged in shared memory by cp.async.bulk (dynamic smem = PLANE_CAP + list)
  int key_cap;                   // 64-bit keys the dynamic shared memory can hold (phase-2 merge keys staged there)
  int dbg;                       // CTB_DEC_DEBUG (tools/decode_time.py): 1 = stop after the streaming NMS, 2 = skip the
                                 // per-image merge -- timing experiments only, results are then incomplete
};

struct SelState {
  unsigned long long prefix, mask;
  int k_rem;
  int digit;
  int done;
};

// Exact K-th largest of n distinct 64-bit keys.  On return every key with (key & mask) >= prefix
// belongs to the top-K set and there are exactly K of them.
template <typename KeyFn>
__device__ void radix_select(int n, int K, KeyFn keyfn, int* hist, SelState* ss) {
  const int tid = threadIdx.x, lane = tid & 31;
  if (tid == 0) { ss->prefix = 0ull; ss->mask = 0ull; ss->k_rem = K; ss->done = 0; }
  __syncthreads();
  const int n_round = (n + DT - 1) / DT * DT;
  for (int shift = 56; shift >= 0; shift -= 8) {
    if (tid < 256) hist[tid] = 0;
    __syncthreads();
    const unsigned long long prefix = ss->prefix, mask = ss->mask;
    for (int i = tid; i < n_round; i += DT) {
      bool part = false;
      int dg = 0;
      if (i < n) {
        const unsigned long long key = keyfn(i);
        part = (key & mask) == prefix;
        dg = (int)((key >> shift) & 255ull);
      }
      const unsigned m = __ballot_sync(0xffffffffu, part);
      if (part) {
        const unsigned peers = __match_any_sync(m, dg);
        if (lane == __ffs(peers) - 1) atomicAdd(&hist[dg], __popc(peers));
      }
    }
    __syncthreads();
    if (tid < 32) {
      int loc[8], s = 0;
#pragma unroll
      for (int q = 0; q < 8; ++q) { loc[q] = hist[lane * 8 + q]; s += loc[q]; }
      // exclusive suffix sum over lanes (bins above this lane's 8 bins)
      int incl = s;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_down_sync(0xffffffffu, incl, o);
        if (lane + o < 32) incl += v;
      }
      const int above = incl - s;
      const int k_rem = ss->k_rem;
      if (above < k_rem && k_rem <= above + s) {
        int acc = above;
        for (int q = 7; q >= 0; --q) {
          if (acc + loc[q] >= k_rem) {
            ss->digit = lane * 8 + q;
            ss->k_rem = k_rem - acc;
            ss->done = (loc[q] == k_rem - acc) ? 1 : 0;
            break;
          }
          acc += loc[q];
        }
      }
    }
    __syncthreads();
    if (tid == 0) {
      ss->prefix |= ((unsigned long long)ss->digit) << shift;
      ss->mask |= 255ull << shift;
    }
    __syncthreads();
    if (ss->done) break;
  }
}

// descending in-place bitonic sort of n (power of two) keys in shared memory
__device__ void bitonic_sort_desc(unsigned long long* a, int n) {
  for (int k = 2; k <= n; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int i = threadIdx.x; i < n; i += DT) {
        const int ixj = i ^ j;
        if (ixj > i) {
          const unsigned long long x = a[i], y = a[ixj];
          const bool up = (i & k) == 0;          // first half of each k-block sorted descending
          if (up ? (x < y) : (x > y)) { a[i] = y; a[ixj] = x; }
        }
      }
      __syncthreads();
    }
  }
}

__device__ __forceinline__ bool nms_keep(const float* sp, int i, int H, int W) {
  const int y = i / W, x = i - y * W;
  const float c = sp[i];
  float m = c;
#pragma unroll
  for (int dy = -1; dy <= 1; ++dy) {
    const int yy = y + dy;
    if (yy < 0 || yy >= H) continue;
#pragma unroll
    for (int dx = -1; dx <= 1; ++dx) {
      const int xx = x + dx;
      if (xx < 0 || xx >= W) continue;
      m = fmaxf(m, sp[yy * W + xx]);
    }
  }
  return m == c;
}

// BULK: planes staged in shared memory by bulk copies (PLANE_CAP + list = 96 KB: two CTAs per SM, 64 registers);
// otherwise streamed through registers (32 KB: three CTAs per SM, 40 registers).
template <bool BULK>
__global__ void __launch_bounds__(DT, BULK ? 2 : 3)
decode_kernel(DecodeArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __shared__ int hist[256];
  __shared__ SelState ss;
  __shared__ unsigned long long sel[MAXK];
  __shared__ int sel_n;
  __shared__ int peak_n;
  __shared__ int is_last;
  __shared__ __align__(8) unsigned long long pbar[DEC_NCH];

  const ct_decode_desc& d = a.d;
  const int tid = threadIdx.x;
  const int pl = blockIdx.x, b = blockIdx.y;
  const int H = d.H, W = d.W, HW = H * W, K = d.K, NP = d.C + d.J;

  // ------------------------------ phase 1: one plane ------------------------------
  // The plane is STREAMED from HBM exactly once, straight into registers (no shared-memory staging): each warp owns a
  // band of rows; a lane holds 4 consecutive pixels of a row (16-byte load), gets its row neighbours by shuffle, and
  // rolls the 3-wide row maxima of the rows above / at / below through registers -- the 3x3 max-equals NMS costs
  // ~0.45 instructions per pixel.  Kept positive peaks (~1 pixel in 10) are compacted as ready-made 64-bit keys
  // (value bits, ~index) into a shared list; the exact radix select runs over that list.
  {
    const float* src = pl < d.C ? d.hm + ((size_t)b * d.C + pl) * HW
                                : d.hm_hp + ((size_t)b * d.J + (pl - d.C)) * HW;
    // a.bulk: the plane is fetched by DEC_NCH cp.async.bulk copies into shared memory (one thread, no registers, the whole
    // 64 KB in flight at once: the register-streamed form keeps one 512-byte row per warp in flight and measured
    // 1.7 TB/s for the NMS alone) and the same rolling NMS reads its rows from there as the chunks land.
    float* plane = reinterpret_cast<float*>(smem_raw);
    unsigned long long* klist = reinterpret_cast<unsigned long long*>(smem_raw + (BULK ? PLANE_CAP : 0));
    const bool vec_ok = (W & 3) == 0 && (reinterpret_cast<size_t>(src) & 15) == 0;
    const bool bulk = BULK && vec_ok;
    const int chunk_rows = (H + DEC_NCH - 1) / DEC_NCH;
    if (tid == 0) {
      peak_n = 0; sel_n = 0;
      if (bulk) {
        for (int c = 0; c < DEC_NCH; ++c) mbarrier_init(smem_u32(&pbar[c]), 1);
        fence_mbarrier_init();
        for (int c = 0; c < DEC_NCH; ++c) {
          const int r0 = c * chunk_rows;
          if (r0 >= H) break;
          const uint32_t bytes = (uint32_t)((H - r0 < chunk_rows ? H - r0 : chunk_rows) * W) * 4u;
          mbarrier_arrive_expect_tx(smem_u32(&pbar[c]), bytes);
          cp_async_bulk(smem_u32(plane + (size_t)r0 * W), src + (size_t)r0 * W, bytes, smem_u32(&pbar[c]));
        }
      }
    }
    for (int i = tid; i < a.kpad; i += DT) sel[i] = 0ull;
    __syncthreads();
    if (vec_ok) {
      const int lane = tid & 31, warp = tid >> 5;
      constexpr int NW = DT / 32;
      const int rpw = (H + NW - 1) / NW;
      const int y0 = warp * rpw;
      const float NEG = __int_as_float(0xff800000);
      if (bulk) {                                       // rows y0-1 .. y0+rpw of this warp: wait for the chunks holding them
        const int y_hi = (y0 + rpw < H ? y0 + rpw : H - 1);
        if (y0 < H)
          for (int c = 0; c <= y_hi / chunk_rows; ++c) mbarrier_wait_parity(smem_u32(&pbar[c]), 0u);
      }
      const float* rows = bulk ? plane : src;           // generic pointer: shared or global
      for (int x0 = 0; x0 < W; x0 += 128) {
        const int x = x0 + 4 * lane;
        const bool xin = x < W;
        // One row ahead of its use.  Measured (32 x 80 x 128 x 128 per launch): this form at 3 CTAs/SM 133 us; raw rows
        // fetched three ahead at 2 CTAs/SM (64 registers), or 4 CTAs of 256 threads, 157 us -- occupancy beats depth here
        auto load_row = [&](int y, float4& v, float4& h) {
          const bool yin = y >= 0 && y < H;                                    // warp-uniform
          v = make_float4(NEG, NEG, NEG, NEG);
          if (yin && xin) v = bulk ? *reinterpret_cast<const float4*>(rows + (size_t)y * W + x)
                                   : __ldg(reinterpret_cast<const float4*>(src + (size_t)y * W + x));
          float l = __shfl_up_sync(0xffffffffu, v.w, 1), r = __shfl_down_sync(0xffffffffu, v.x, 1);
          if (lane == 0) l = (yin && x0 > 0) ? rows[(size_t)y * W + x0 - 1] : NEG;
          if (lane == 31) r = (yin && x + 4 < W) ? rows[(size_t)y * W + x + 4] : NEG;
          h.x = fmaxf(fmaxf(l, v.x), v.y); h.y = fmaxf(fmaxf(v.x, v.y), v.z);
          h.z = fmaxf(fmaxf(v.y, v.z), v.w); h.w = fmaxf(fmaxf(v.z, v.w), r);
        };
        float4 v_cur, h_up, h_cur, v_dn, h_dn;
        load_row(y0 - 1, v_cur, h_up);
        load_row(y0, v_cur, h_cur);
        for (int j = 0; j < rpw; ++j) {
          const int y = y0 + j;
          load_row(y + 1, v_dn, h_dn);
          if (y < H) {                                                         // warp-uniform
            const float vc[4] = {v_cur.x, v_cur.y, v_cur.z, v_cur.w};
            const float mx[4] = {fmaxf(fmaxf(h_up.x, h_cur.x), h_dn.x), fmaxf(fmaxf(h_up.y, h_cur.y), h_dn.y),
                                 fmaxf(fmaxf(h_up.z, h_cur.z), h_dn.z), fmaxf(fmaxf(h_up.w, h_cur.w), h_dn.w)};
            unsigned bits = 0;
#pragma unroll
            for (int c = 0; c < 4; ++c) bits |= (xin && vc[c] > 0.f && mx[c] == vc[c]) ? (1u << c) : 0u;
            // inclusive prefix of the per-lane peak counts (0..4) from three independent ballots of the count's bit planes
            // (a 5-step shuffle scan is a 5-deep dependent chain per row); rows without a peak skip everything
            const int cnt = __popc(bits);
            const unsigned b0 = __ballot_sync(0xffffffffu, cnt & 1), b1 = __ballot_sync(0xffffffffu, cnt & 2),
                           b2 = __ballot_sync(0xffffffffu, cnt & 4);
            const unsigned le = 0xffffffffu >> (31 - lane);
            const int incl = __popc(b0 & le) + 2 * __popc(b1 & le) + 4 * __popc(b2 & le);
            const int total = __popc(b0) + 2 * __popc(b1) + 4 * __popc(b2);
            if (total) {
              int base = 0;
              if (lane == 0) base = atomicAdd(&peak_n, total);
              base = __shfl_sync(0xffffffffu, base, 0);
              int slot = base + incl - cnt;
#pragma unroll
              for (int c = 0; c < 4; ++c)
                if (bits & (1u << c)) {
                  if (slot < PEAK_CAP)
                    klist[slot] = ((unsigned long long)__float_as_uint(vc[c]) << 32) |
                                  (unsigned long long)(0xFFFFFFFFu - (unsigned)(y * W + x + c));
                  ++slot;
                }
            }
          }
          h_up = h_cur; h_cur = h_dn; v_cur = v_dn;
        }
      }
    }
    __syncthreads();
    if (a.dbg & 1) return;
    const int npk = peak_n;
    // The list is exact whenever it holds at least K peaks and did not overflow (zeros, which the index-ordered tie
    // rule would otherwise have to rank, are then out of the race).  Degenerate planes (fewer than K positive peaks,
    // plateaus that overflow the list, odd widths) select over all H*W keys, evaluating the NMS from global memory.
    const bool fast = vec_ok && npk >= K && npk <= PEAK_CAP;
    if (fast) {
      auto keyfn_l = [&](int j) -> unsigned long long { return klist[j]; };
      radix_select(npk, K, keyfn_l, hist, &ss);
      const unsigned long long prefix = ss.prefix, mask = ss.mask;
      for (int j = tid; j < npk; j += DT) {
        const unsigned long long key = klist[j];
        if ((key & mask) >= prefix) {
          const int slot = atomicAdd(&sel_n, 1);
          if (slot < MAXK) sel[slot] = key;
        }
      }
    } else {
      auto keyfn = [&](int i) -> unsigned long long {
        const int y = i / W, x = i - y * W;
        const float c = __ldg(src + i);
        float m = c;
        for (int dy = -1; dy <= 1; ++dy) {
          const int yy = y + dy;
          if (yy < 0 || yy >= H) continue;
          for (int dx = -1; dx <= 1; ++dx) {
            const int xx = x + dx;
            if (xx >= 0 && xx < W) m = fmaxf(m, __ldg(src + yy * W + xx));
          }
        }
        // heat * keep as a sort key: -0.0 cannot occur for sigmoid outputs; negatives (not produced by the reference
        // path) are clamped to 0 so the unsigned key order stays valid
        const float v = (m == c) ? c : 0.f;
        const unsigned vb = v > 0.f ? __float_as_uint(v) : 0u;
        return ((unsigned long long)vb << 32) | (unsigned long long)(0xFFFFFFFFu - (unsigned)i);
      };
      radix_select(HW, K, keyfn, hist, &ss);
      const unsigned long long prefix = ss.prefix, mask = ss.mask;
      for (int i = tid; i < HW; i += DT) {
        const unsigned long long key = keyfn(i);
        if ((key & mask) >= prefix) {
          const int slot = atomicAdd(&sel_n, 1);
          if (slot < MAXK) sel[slot] = key;
        }
      }
    }
    __syncthreads();
    // Class planes leave their K survivors UNSORTED: the cross-class merge orders by (value, class, index), which is
    // the order of the reference's second top-K over the [C, K] array (ties: class, then rank = index within a class).
    // Joint planes (pose) are consumed in rank order by the keypoint refinement: those are sorted here.
    if (pl >= d.C) bitonic_sort_desc(sel, a.kpad);
    unsigned long long* dst = a.cand + ((size_t)b * NP + pl) * K;
    for (int i = tid; i < K; i += DT) dst[i] = sel[i];
  }
  __threadfence();
  __syncthreads();
  if (tid == 0) {
    const int old = atomicAdd(&a.counters[b], 1);
    is_last = (old == NP - 1);
    if (is_last) a.counters[b] = 0;
  }
  __syncthreads();
  if (!is_last || (a.dbg & 2)) return;
  __threadfence();

  // ------------------------------ phase 2: merge + gather ------------------------------
  const unsigned long long* candb = a.cand + (size_t)b * NP * K;
  const int n2 = d.C * K;
  auto key2 = [&](int i) -> unsigned long long {
    const unsigned long long c = __ldcg(candb + i);
    const unsigned idx = 0xFFFFFFFFu - (unsigned)(c & 0xFFFFFFFFull);
    const unsigned g = (unsigned)(i / K) * (unsigned)HW + idx;            // class-major global position
    return (c & 0xFFFFFFFF00000000ull) | (unsigned long long)(0xFFFFFFFFu - g);
  };
  // The merge keys are staged in shared memory when they fit (C*K <= key_cap): every radix pass then reads them at
  // shared-memory latency; from L2 (one dependent round trip per 512 keys per pass) the merge of one image took ~35 us,
  // serialised at the tail of the launch.
  unsigned long long* skeys = reinterpret_cast<unsigned long long*>(smem_raw);
  const bool keys_in_smem = n2 <= a.key_cap;
  if (keys_in_smem) {
    for (int i = tid; i < n2; i += DT) skeys[i] = key2(i);
    __syncthreads();
  }
  auto key2s = [&](int i) -> unsigned long long { return skeys[i]; };
  if (keys_in_smem) radix_select(n2, K, key2s, hist, &ss);
  else radix_select(n2, K, key2, hist, &ss);
  if (tid == 0) sel_n = 0;
  for (int i = tid; i < a.kpad; i += DT) sel[i] = 0ull;
  __syncthreads();
  {
    const unsigned long long prefix = ss.prefix, mask = ss.mask;
    for (int i = tid; i < n2; i += DT) {
      const unsigned long long key = keys_in_smem ? skeys[i] : key2(i);
      if ((key & mask) >= prefix) {
        const int slot = atomicAdd(&sel_n, 1);
        if (slot < MAXK) sel[slot] = key;
      }
    }
  }
  __syncthreads();
  bitonic_sort_desc(sel, a.kpad);

  const int F = d.rec_floats;
  float* recb = d.records + (size_t)b * K * F;
  // per-detection scalars kept in shared memory for the pose step
  float* s_score = reinterpret_cast<float*>(smem_raw);
  float* s_x0 = s_score + K;
  float* s_y0 = s_x0 + K;
  float* s_box = s_y0 + K;            // [K][4]
  float* s_pose = s_box + 4 * K;      // pose scratch (see below)

  for (int k = tid; k < K; k += DT) {
    const unsigned long long key = sel[k];
    const float score = __uint_as_float((unsigned)(key >> 32));
    const unsigned gpos = 0xFFFFFFFFu - (unsigned)(key & 0xFFFFFFFFull);
    const int cls = (int)(gpos / (unsigned)HW);
    const unsigned idx = gpos - (unsigned)cls * (unsigned)HW;
    const float xs0 = (float)(idx % (unsigned)W), ys0 = (float)(idx / (unsigned)W);
    float* rec = recb + (size_t)k * F;
    rec[CT_REC_SCORE] = score;
    rec[CT_REC_CLS] = (float)cls;
    rec[CT_REC_XS] = xs0;
    rec[CT_REC_YS] = ys0;
    rec[CT_REC_IND] = __int_as_float((int)idx);
    float xs = xs0 + 0.5f, ys = ys0 + 0.5f;
    // first pass: the center-offset head decides xs/ys for the wh boxes (decode.py:103-111)
    for (int h = 0; h < d.n_heads; ++h) {
      if (d.heads[h].role == CT_ROLE_REG) {
        const float* m = d.heads[h].map + (size_t)b * d.heads[h].channels * HW;
        xs = xs0 + __ldg(m + idx);
        ys = ys0 + __ldg(m + HW + idx);
      }
    }
    float bl = 0.f, bt = 0.f, br = 0.f, bb = 0.f;
    for (int h = 0; h < d.n_heads; ++h) {
      const ct_decode_head& hd = d.heads[h];
      const float* m = hd.map + (size_t)b * hd.channels * HW;
      float* o = rec + hd.rec_offset;
      if (hd.role == CT_ROLE_WH) {
        float w = __ldg(m + idx), hh = __ldg(m + HW + idx);
        w = w < 0.f ? 0.f : w; hh = hh < 0.f ? 0.f : hh;
        o[0] = w; o[1] = hh;
        bl = xs - w / 2; bt = ys - hh / 2; br = xs + w / 2; bb = ys + hh / 2;
      } else if (hd.role == CT_ROLE_LTRB || hd.role == CT_ROLE_LTRB_AMODAL) {
        const float l = __ldg(m + idx), t = __ldg(m + HW + idx);
        const float r = __ldg(m + 2 * HW + idx), bo = __ldg(m + 3 * HW + idx);
        o[0] = l; o[1] = t; o[2] = r; o[3] = bo;
        bl = xs0 + l; bt = ys0 + t; br = xs0 + r; bb = ys0 + bo;
      } else if (hd.role == CT_ROLE_HPS) {
        for (int c = 0; c < hd.channels; ++c)
          o[c] = __ldg(m + (size_t)c * HW + idx) + ((c & 1) ? ys0 : xs0);
      } else {
        for (int c = 0; c < hd.channels; ++c) o[c] = __ldg(m + (size_t)c * HW + idx);
      }
    }
    rec[CT_REC_BBOX + 0] = bl; rec[CT_REC_BBOX + 1] = bt;
    rec[CT_REC_BBOX + 2] = br; rec[CT_REC_BBOX + 3] = bb;
    s_score[k] = score; s_x0[k] = xs0; s_y0[k] = ys0;
    s_box[4 * k + 0] = bl; s_box[4 * k + 1] = bt; s_box[4 * k + 2] = br; s_box[4 * k + 3] = bb;
  }
  __syncthreads();
  if (d.hm_hp == nullptr || d.rec_hps < 0) return;

  // ------------------------------ pose refinement (decode.py:11-81) ------------------------------
  const int J = d.J;
  float* c_sc = s_pose;                 // [J][K] candidate score (masked)
  float* c_x = c_sc + J * K;            // [J][K]
  float* c_y = c_x + J * K;
  float* r_sc = c_y + J * K;            // [J][K] per (joint, det): score used in kps_score
  int hps_off = -1, reg_h = -1;
  for (int h = 0; h < d.n_heads; ++h) {
    if (d.heads[h].role == CT_ROLE_HPS) hps_off = d.heads[h].rec_offset;
    if (d.heads[h].role == CT_ROLE_REG) reg_h = h;
  }
  const float thresh = 0.2f;
  for (int i = tid; i < J * K; i += DT) {
    const int j = i / K;
    const unsigned long long ck = __ldcg(candb + (size_t)(d.C + j) * K + (i - j * K));
    float sc = __uint_as_float((unsigned)(ck >> 32));
    const unsigned idx = 0xFFFFFFFFu - (unsigned)(ck & 0xFFFFFFFFull);
    float hx = (float)(idx % (unsigned)W), hy = (float)(idx / (unsigned)W);
    if (d.hp_offset) {
      const float* m = d.hp_offset + (size_t)b * 2 * HW;
      hx = hx + __ldg(m + idx); hy = hy + __ldg(m + HW + idx);
    } else if (reg_h >= 0) {
      const float* m = d.heads[reg_h].map + (size_t)b * 2 * HW;
      hx = hx + __ldg(m + idx); hy = hy + __ldg(m + HW + idx);
    } else {
      hx = hx + 0.5f; hy = hy + 0.5f;
    }
    if (!(sc > thresh)) { sc = -1.f; hx = -10000.f; hy = -10000.f; }
    c_sc[i] = sc; c_x[i] = hx; c_y[i] = hy;
  }
  __syncthreads();
  for (int i = tid; i < J * K; i += DT) {
    const int j = i / K, k = i - j * K;
    float* rec = recb + (size_t)k * F;
    const float kx = rec[hps_off + 2 * j], ky = rec[hps_off + 2 * j + 1];
    float best = 0.f; int bi = 0;
    for (int c = 0; c < K; ++c) {
      const float dx = __fsub_rn(kx, c_x[j * K + c]), dy = __fsub_rn(ky, c_y[j * K + c]);
      const float dist = __fsqrt_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)));
      if (c == 0 || dist < best) { best = dist; bi = c; }
    }
    const float sc = c_sc[j * K + bi], hx = c_x[j * K + bi], hy = c_y[j * K + bi];
    const bool m = (sc < thresh) || (hx < s_box[4 * k + 0]) || (hx > s_box[4 * k + 2]) ||
                   (hy < s_box[4 * k + 1]) || (hy > s_box[4 * k + 3]);
    r_sc[i] = m ? s_score[k] : sc;
    rec[d.rec_hps + 2 * j] = m ? kx : hx;
    rec[d.rec_hps + 2 * j + 1] = m ? ky : hy;
  }
  __syncthreads();
  if (d.rec_kps_score >= 0) {
    for (int k = tid; k < K; k += DT) {
      float s = 0.f;
      for (int j = 0; j < J; ++j) s = __fadd_rn(s, r_sc[j * K + k]);
      recb[(size_t)k * F + d.rec_kps_score] = __fmul_rn(s_score[k], __fdiv_rn(s, (float)J));
    }
  }
}

}  // namespace ctb

using namespace ctb;

static inline int64_t align256(int64_t x) { return (x + 255) / 256 * 256; }

extern "C" int64_t ct_decode_workspace_bytes(int32_t B, int32_t C, int32_t J, int32_t K) {
  return align256((int64_t)4 * B) + (int64_t)8 * B * (C + J) * K;
}

extern "C" int ct_decode(const ct_decode_desc* d, void* stream) {
  CT_REQUIRE(d && d->hm && d->records && d->workspace, "null pointer");
  CT_REQUIRE(d->B > 0 && d->C > 0 && d->H > 0 && d->W > 0, "bad shape");
  CT_REQUIRE(d->K > 0 && d->K <= MAXK && d->K <= d->H * d->W, "K out of range (1..512, <= H*W)");
  CT_REQUIRE(d->n_heads >= 0 && d->n_heads <= CT_DECODE_MAX_HEADS, "too many heads");
  CT_REQUIRE(d->rec_floats >= CT_REC_HEADS, "record too small");
  CT_REQUIRE(d->hm_hp == nullptr || d->J > 0, "hm_hp without J");
  DecodeArgs a;
  a.d = *d;
  if (a.d.hm_hp == nullptr) a.d.J = 0;
  a.counters = reinterpret_cast<int*>(d->workspace);
  a.cand = reinterpret_cast<unsigned long long*>(reinterpret_cast<char*>(d->workspace) +
                                                 align256((int64_t)4 * d->B));
  int kpad = 1;
  while (kpad < d->K) kpad <<= 1;
  a.kpad = kpad;
  static const int dec_dbg = getenv("CTB_DEC_DEBUG") ? atoi(getenv("CTB_DEC_DEBUG")) : 0;
  a.dbg = dec_dbg;
  const int HW = d->H * d->W, K = d->K, J = a.d.J;
  CT_REQUIRE((long long)d->C * HW < (1ll << 31), "C*H*W must stay below 2^31 (class-major positions in the merge keys)");
  a.bulk = ((size_t)HW * 4 <= PLANE_CAP && (d->W & 3) == 0) ? 1 : 0;      // else: register-streamed planes
  size_t smem1 = (size_t)PEAK_CAP * 8 + (a.bulk ? PLANE_CAP : 0);
  size_t smem2 = (size_t)(7 * K + 4 * J * K) * 4;
  size_t smem = smem1 > smem2 ? smem1 : smem2;
  a.key_cap = (int)(smem / 8);
  if (smem > 200 * 1024)
    return fail(CT_ERR_UNSUPPORTED, "ct_decode: K x joints of %s%ld floats exceed the shared-memory scratch of the pose "
                                    "refinement", "", (long)(4 * J * K));
  cudaStream_t st = (cudaStream_t)stream;
  dim3 grid(d->C + J, d->B);
  if (a.bulk) {
    CT_CUDA_OK(cudaFuncSetAttribute(decode_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    decode_kernel<true><<<grid, DT, smem, st>>>(a);
  } else {
    CT_CUDA_OK(cudaFuncSetAttribute(decode_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    decode_kernel<false><<<grid, DT, smem, st>>>(a);
  }
  return after_launch();
}
