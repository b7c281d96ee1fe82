// Per-stream state kept on the device between frames (SURVEY 8f rows 1-3):
//   ct_track_step    generic_post_process's affine + Tracker.step's greedy displacement association
//                    (utils/post_process.py:21-91, utils/tracker.py:28-138) on the packed decode records, plus the
//                    (centre, radius) boxes of Detector._get_additional_inputs (detector.py:254-290) for the NEXT frame
//   ct_render_tracks the gaussian max-splat of those boxes into pre_hm (image.py:128-154)
//   ct_flip_merge    Detector._flip_output (detector.py:311-332; model/utils.py:28-50) for --flip_test
//   ct_warp_affine_normalize   Detector.pre_process's cv2.warpAffine(INTER_LINEAR) + (x/255 - mean)/std + HWC->CHW
//                    (detector.py:207-226), cv2's fixed-point bilinear restated
// All HBM-bound byte/index work: one pass over the data, coalesced, no tensor cores.
#include <math_constants.h>

#include "common.cuh"

namespace ctb {

// ------------------------------------------------------------------------------------------------------------------
// flip merge: out[c,y,x] = 0.5 * (in[0,c,y,x] + sign[c] * in[1,perm[c],y,W-1-x])
// ------------------------------------------------------------------------------------------------------------------
__global__ void flip_merge_kernel(const float* __restrict__ in2, float* __restrict__ out, int C, int H, int W,
                                  const int* __restrict__ perm, const float* __restrict__ sign) {
  const size_t total = (size_t)C * H * W;
  const size_t plane = (size_t)H * W;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int c = (int)(i / plane);
    const size_t r = i - (size_t)c * plane;
    const int y = (int)(r / W), x = (int)(r - (size_t)y * W);
    const int cs = perm ? perm[c] : c;
    const float sg = sign ? sign[c] : 1.f;
    const float a = in2[i];
    const float b = in2[total + (size_t)cs * plane + (size_t)y * W + (W - 1 - x)];
    // the reference adds the two maps and halves the sum: (a + s*b) / 2, in that order (division by 2 is exact)
    out[i] = __fmul_rn(__fadd_rn(a, __fmul_rn(sg, b)), 0.5f);
  }
}

// ------------------------------------------------------------------------------------------------------------------
// track step
// ------------------------------------------------------------------------------------------------------------------
constexpr int TRK_THREADS = 128;
constexpr int TF = CT_TRK_FLOATS;

struct TrackArgs {
  ct_track_desc d;
};

__device__ __forceinline__ float aff_f32(const float* t, float x, float y) {
  // np.dot(trans[2x3] f32, [x, y, 1] f32): x*t0 + y*t1 + t2 accumulated left to right in fp32
  return __fadd_rn(__fadd_rn(__fmul_rn(t[0], x), __fmul_rn(t[1], y)), t[2]);
}
__device__ __forceinline__ double aff_f64(const double* t, double x, double y) {
  return __dadd_rn(__dadd_rn(__dmul_rn(t[0], x), __dmul_rn(t[1], y)), t[2]);
}

// gaussian_radius(det_size=(h, w), min_overlap=0.7): utils/image.py:105-125, float64
__device__ double gaussian_radius_f64(double h, double w) {
  const double mo = 0.7;
  const double b1 = h + w;
  const double c1 = w * h * (1 - mo) / (1 + mo);
  const double r1 = (b1 + sqrt(b1 * b1 - 4 * c1)) / 2;
  const double b2 = 2 * (h + w);
  const double c2 = (1 - mo) * w * h;
  const double r2 = (b2 + sqrt(b2 * b2 - 16 * c2)) / 2;
  const double a3 = 4 * mo;
  const double b3 = -2 * mo * (h + w);
  const double c3 = (mo - 1) * w * h;
  const double r3 = (b3 + sqrt(b3 * b3 - 4 * a3 * c3)) / 2;
  return fmin(r1, fmin(r2, r3));
}

// dynamic shared memory of the greedy step (track table, detections, per-row bookkeeping) ...
__host__ __device__ inline size_t track_smem_greedy(int K, int T) {
  return ((size_t)T * TF + (size_t)K * TF + 3 * (size_t)K + T) * 4 + (2 * (size_t)K + 2 * (size_t)T) * 4 + 64;
}
// ... and the scratch of the assignment solver and the public-detection births behind it (8-byte aligned):
// doubles spc[T], v[T], u[K]; ints path[T], row4col[T], remaining[T], col_seen[T], col4row[K], row_seen[K],
// rejected[K], claimed[K], born[K].  Rows of the solver are the shorter side (<= K), columns the longer (<= T).
__host__ __device__ inline size_t track_smem_scratch_offset(int K, int T) {
  return (track_smem_greedy(K, T) + 7) & ~(size_t)7;
}
__host__ __device__ inline size_t track_smem_full(int K, int T) {
  return track_smem_scratch_offset(K, T) + (size_t)T * (2 * 8 + 4 * 4) + (size_t)K * (8 + 5 * 4);
}

// Gated association cost of (detection i, track j) as tracker.py::_gated_cost + hungarian_assignment build it:
// float64 of the float32 squared distance between the detection's predicted previous centre and the track centre,
// or exactly 1e18 when the pair is blocked (distance above either box area, or different classes).
struct GatedCost {
  const float* old; const float* det; const float* px; const float* py; const float* isz; const float* tsz;
  __device__ __forceinline__ double operator()(int i, int j) const {
    const float* t = old + (size_t)j * TF;
    const float dx = __fsub_rn(t[CT_TRK_CT], px[i]), dy = __fsub_rn(t[CT_TRK_CT + 1], py[i]);
    const float dist = __fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy));
    const bool blocked = dist > tsz[j] || dist > isz[i] || t[CT_TRK_CLASS] != det[(size_t)i * TF + CT_TRK_CLASS];
    return blocked ? 1e18 : (double)dist;
  }
};

// One candidate column of a Dijkstra round: reduced cost, position in `remaining`, column still unassigned.
struct LsapPick { double v; int pos; bool free; };

// scipy's tie rule (rectangular_lsap.cpp): the minimum reduced cost; among equal minima the LAST unassigned column in
// scan order if there is one, else the FIRST.  Commutative and associative over disjoint sets of positions, so it
// runs as a butterfly.
__device__ __forceinline__ LsapPick lsap_better(LsapPick a, LsapPick b) {
  if (b.pos < 0) return a;
  if (a.pos < 0) return b;
  if (b.v < a.v) return b;
  if (a.v < b.v) return a;
  if (a.free || b.free) {
    if (a.free && b.free) return b.pos > a.pos ? b : a;
    return a.free ? a : b;
  }
  return b.pos < a.pos ? b : a;
}

// Minimum-cost assignment of the N x M gated cost matrix by ONE warp, pair for pair what scipy's
// linear_sum_assignment returns: Crouse's shortest augmenting path (scipy/optimize/rectangular_lsap.cpp), restated
// in Python in tests/lsap_restated.py.  N > M solves the transpose (rows = tracks).  Each round the lanes relax their
// columns of `remaining` and pick the next column by warp shuffles, in the same float64 operation order as scipy.
// Results: s_match[det] = track of a kept pair (cost <= 1e16), s_rej[det] = track of a pair forced through a blocked
// cell, s_taken[track] = 1 for every paired track.
__device__ void lsap_warp(const GatedCost& cost, int N, int M, int lane, double* spc, double* v, double* u, int* path,
                          int* row4col, int* remaining, int* col_seen, int* col4row, int* row_seen, int* s_match,
                          int* s_rej, int* s_taken) {
  const unsigned full = 0xffffffffu;
  const bool tr = N > M;
  const int nr = tr ? M : N, nc = tr ? N : M;
  for (int c = lane; c < nc; c += 32) { v[c] = 0.0; row4col[c] = -1; }
  for (int r = lane; r < nr; r += 32) { u[r] = 0.0; col4row[r] = -1; }
  for (int i = lane; i < N; i += 32) s_rej[i] = -1;
  __syncwarp();
  for (int cur = 0; cur < nr; ++cur) {
    for (int c = lane; c < nc; c += 32) { remaining[c] = nc - 1 - c; spc[c] = CUDART_INF; col_seen[c] = 0; }
    for (int r = lane; r < nr; r += 32) row_seen[r] = 0;
    __syncwarp();
    double minVal = 0.0;
    int i = cur, sink = -1, nrem = nc;
    while (sink < 0) {
      if (lane == 0) row_seen[i] = 1;
      const double ui = u[i];
      LsapPick best = {CUDART_INF, -1, false};
      for (int it = lane; it < nrem; it += 32) {
        const int j = remaining[it];
        const double r = __dsub_rn(__dsub_rn(__dadd_rn(minVal, tr ? cost(j, i) : cost(i, j)), ui), v[j]);
        double s = spc[j];
        if (r < s) { path[j] = i; spc[j] = r; s = r; }
        const LsapPick p = {s, it, row4col[j] == -1};
        best = lsap_better(best, p);
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        LsapPick p;
        p.v = __shfl_xor_sync(full, best.v, o);
        p.pos = __shfl_xor_sync(full, best.pos, o);
        p.free = __shfl_xor_sync(full, (int)best.free, o) != 0;
        best = lsap_better(best, p);
      }
      minVal = best.v;
      const int j = remaining[best.pos];
      const int owner = row4col[j];
      __syncwarp();                                   // every lane is done with remaining / spc of this round
      if (lane == 0) { col_seen[j] = 1; remaining[best.pos] = remaining[nrem - 1]; }
      --nrem;
      if (owner == -1) sink = j; else i = owner;
      __syncwarp();
    }
    // dual update (u of the rows and v of the columns reached this augmentation), then flip the path
    for (int r = lane; r < nr; r += 32)
      if (row_seen[r] && r != cur) u[r] = __dadd_rn(u[r], __dsub_rn(minVal, spc[col4row[r]]));
    if (lane == 0) u[cur] = __dadd_rn(u[cur], minVal);
    for (int c = lane; c < nc; c += 32)
      if (col_seen[c]) v[c] = __dsub_rn(v[c], __dsub_rn(minVal, spc[c]));
    __syncwarp();
    if (lane == 0) {
      int j = sink;
      while (true) {
        const int r = path[j];
        row4col[j] = r;
        const int nxt = col4row[r];
        col4row[r] = j;
        j = nxt;
        if (r == cur) break;
      }
    }
    __syncwarp();
  }
  for (int r = lane; r < nr; r += 32) {
    const int c = col4row[r];
    const int det = tr ? c : r, trk = tr ? r : c;
    s_taken[trk] = 1;
    if (cost(det, trk) <= 1e16) s_match[det] = trk; else s_rej[det] = trk;
  }
}

// MOT public-detection births (tracker.py:83-103, host: tracker.py::_public_births) by one warp: each public
// detection in order claims the first nearest (float32 squared distance of the predicted previous centre) detection
// not yet matched or claimed, if that distance is below the detection's box area; a claimed detection confident enough
// to start a track is appended to born[].  Returns the number of births.  Runs only if some detection is unmatched.
__device__ int public_births_warp(const float* pub, int P, int N, int lane, const float* px, const float* py,
                                  const float* isz, const float* det, float new_thresh, const int* s_match,
                                  int* claimed, int* born) {
  const unsigned full = 0xffffffffu;
  bool any_free = false;
  for (int i = lane; i < N; i += 32) {
    claimed[i] = s_match[i] >= 0;
    any_free |= s_match[i] < 0;
  }
  __syncwarp();
  if (!__any_sync(full, any_free)) return 0;
  int nb = 0;
  for (int p = 0; p < P; ++p) {
    const float qx = pub[2 * p], qy = pub[2 * p + 1];
    float best = 3.0e38f;
    int bi = 0x7fffffff;
    for (int i = lane; i < N; i += 32) {
      const float dx = __fsub_rn(px[i], qx), dy = __fsub_rn(py[i], qy);
      const float c = claimed[i] ? 1e18f : __fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy));
      if (c < best) { best = c; bi = i; }              // ascending i per lane: first minimum kept
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ov = __shfl_xor_sync(full, best, o);
      const int oi = __shfl_xor_sync(full, bi, o);
      if (ov < best || (ov == best && oi < bi)) { best = ov; bi = oi; }
    }
    __syncwarp();
    if (bi < N && best < isz[bi]) {
      if (lane == 0) claimed[bi] = 1;
      if (det[(size_t)bi * TF + CT_TRK_SCORE] > new_thresh) {
        if (lane == 0) born[nb] = bi;
        ++nb;
      }
    }
    __syncwarp();
  }
  return nb;
}

__global__ void __launch_bounds__(TRK_THREADS)
track_step_kernel(const TrackArgs a) {
  extern __shared__ __align__(16) unsigned char tsm[];
  const ct_track_desc& d = a.d;
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int T = d.max_tracks, K = d.K;
  float* s_old = reinterpret_cast<float*>(tsm);                 // [T][TF]   previous tracks
  float* s_det = s_old + (size_t)T * TF;                        // [K][TF]   this frame's detections (image coords)
  float* s_px = s_det + (size_t)K * TF;                         // [K] predicted previous centre x (ct + tracking)
  float* s_py = s_px + K;                                       // [K]
  float* s_isz = s_py + K;                                      // [K] detection box area
  float* s_tsz = s_isz + K;                                     // [T] track box area
  int* s_match = reinterpret_cast<int*>(s_tsz + T);             // [K] matched track or -1
  int* s_taken = s_match + K;                                   // [T]
  int* s_pos_det = s_taken + T;                                 // [K] output slot of det or -1
  int* s_pos_trk = s_pos_det + K;                               // [T] output slot of a coasting track or -1
  // solver / public-birth scratch: only present (and only touched) with --hungarian or public detections
  double* s_spc = reinterpret_cast<double*>(tsm + track_smem_scratch_offset(K, T));   // [T]
  double* s_v = s_spc + T;                                      // [T]
  double* s_u = s_v + T;                                        // [K]
  int* s_path = reinterpret_cast<int*>(s_u + K);                // [T]
  int* s_row4col = s_path + T;                                  // [T]
  int* s_remaining = s_row4col + T;                             // [T]
  int* s_col_seen = s_remaining + T;                            // [T]
  int* s_col4row = s_col_seen + T;                              // [K]
  int* s_row_seen = s_col4row + K;                              // [K]
  int* s_rej = s_row_seen + K;                                  // [K] track of a rejected (forced) pair or -1
  int* s_claimed = s_rej + K;                                   // [K]
  int* s_born = s_claimed + K;                                  // [K] public births in claim order
  const bool hung = d.assign == CT_ASSIGN_HUNGARIAN;
  __shared__ float red_v[TRK_THREADS / 32];
  __shared__ int red_j[TRK_THREADS / 32];
  __shared__ int s_n, s_total, s_ids, s_nborn;

  int M = d.counts[b * 2 + 0];
  if (M > T) M = T;
  const int id_count = d.counts[b * 2 + 1];
  float* trk = d.tracks + (size_t)b * T * TF;
  for (int i = tid; i < M * TF; i += TRK_THREADS) s_old[i] = trk[i];
  if (tid == 0) s_n = 0;
  __syncthreads();

  // ---- detections of this frame: generic_post_process (post_process.py:21-91), merge_outputs (detector.py:371-377)
  const float* rec = d.records + (size_t)b * K * d.F;
  const float* to = d.trans_out_inv + b * 6;
  int cnt = 0;
  for (int i = tid; i < K; i += TRK_THREADS) cnt += rec[(size_t)i * d.F + CT_REC_SCORE] > d.out_thresh ? 1 : 0;
  atomicAdd(&s_n, cnt);
  __syncthreads();
  const int N = s_n;                     // records are sorted by score: the kept detections are a prefix
  for (int i = tid; i < N; i += TRK_THREADS) {
    const float* r = rec + (size_t)i * d.F;
    float* o = s_det + (size_t)i * TF;
    const float cx = r[CT_REC_XS], cy = r[CT_REC_YS];
    const float ctx = aff_f32(to, cx, cy), cty = aff_f32(to + 3, cx, cy);
    float tx = 0.f, ty = 0.f;
    if (d.rec_tracking >= 0) {
      const float px = __fadd_rn(r[d.rec_tracking], cx), py = __fadd_rn(r[d.rec_tracking + 1], cy);
      tx = __fsub_rn(aff_f32(to, px, py), ctx);
      ty = __fsub_rn(aff_f32(to + 3, px, py), cty);
    }
    const float bl = r[CT_REC_BBOX], bt = r[CT_REC_BBOX + 1], br = r[CT_REC_BBOX + 2], bb = r[CT_REC_BBOX + 3];
    o[CT_TRK_SCORE] = r[CT_REC_SCORE];
    o[CT_TRK_CLASS] = r[CT_REC_CLS] + 1.f;
    o[CT_TRK_CT] = ctx; o[CT_TRK_CT + 1] = cty;
    o[CT_TRK_TRACKING] = tx; o[CT_TRK_TRACKING + 1] = ty;
    o[CT_TRK_BBOX] = aff_f32(to, bl, bt); o[CT_TRK_BBOX + 1] = aff_f32(to + 3, bl, bt);
    o[CT_TRK_BBOX + 2] = aff_f32(to, br, bb); o[CT_TRK_BBOX + 3] = aff_f32(to + 3, br, bb);
    o[CT_TRK_ID] = 0.f; o[CT_TRK_AGE] = 1.f; o[CT_TRK_ACTIVE] = 0.f;
    s_px[i] = __fadd_rn(ctx, tx);
    s_py[i] = __fadd_rn(cty, ty);
    s_isz[i] = __fmul_rn(__fsub_rn(o[CT_TRK_BBOX + 2], o[CT_TRK_BBOX]), __fsub_rn(o[CT_TRK_BBOX + 3], o[CT_TRK_BBOX + 1]));
    s_match[i] = -1;
  }
  for (int j = tid; j < M; j += TRK_THREADS) {
    const float* t = s_old + (size_t)j * TF;
    s_tsz[j] = __fmul_rn(__fsub_rn(t[CT_TRK_BBOX + 2], t[CT_TRK_BBOX]), __fsub_rn(t[CT_TRK_BBOX + 3], t[CT_TRK_BBOX + 1]));
    s_taken[j] = 0;
  }
  __syncthreads();

  if (hung) {
    // ---- --hungarian (tracker.py:52-72): minimum-cost assignment by warp 0
    if (warp == 0) {
      const GatedCost cost = {s_old, s_det, s_px, s_py, s_isz, s_tsz};
      lsap_warp(cost, N, M, lane, s_spc, s_v, s_u, s_path, s_row4col, s_remaining, s_col_seen, s_col4row, s_row_seen,
                s_match, s_rej, s_taken);
    }
    __syncthreads();
  }
  // ---- greedy assignment (tracker.py:129-138): detections in score order take their nearest free, valid track;
  //      argmin ties -> lowest track index
  const float INF = 3.0e38f;
  for (int i = 0; i < N && M > 0 && !hung; ++i) {
    const float px = s_px[i], py = s_py[i], isz = s_isz[i], icls = s_det[(size_t)i * TF + CT_TRK_CLASS];
    float best = INF;
    int bj = 0x7fffffff;
    for (int j = tid; j < M; j += TRK_THREADS) {
      const float* t = s_old + (size_t)j * TF;
      const float dx = __fsub_rn(t[CT_TRK_CT], px), dy = __fsub_rn(t[CT_TRK_CT + 1], py);
      const float dist = __fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy));
      const bool ok = !s_taken[j] && !(dist > s_tsz[j]) && !(dist > isz) && t[CT_TRK_CLASS] == icls;
      if (ok && dist < best) { best = dist; bj = j; }       // ascending j per thread: first minimum kept
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, best, o);
      const int oj = __shfl_xor_sync(0xffffffffu, bj, o);
      if (ov < best || (ov == best && oj < bj)) { best = ov; bj = oj; }
    }
    if (lane == 0) { red_v[warp] = best; red_j[warp] = bj; }
    __syncthreads();
    if (tid == 0) {
      float v = red_v[0];
      int j = red_j[0];
      for (int w = 1; w < TRK_THREADS / 32; ++w)
        if (red_v[w] < v || (red_v[w] == v && red_j[w] < j)) { v = red_v[w]; j = red_j[w]; }
      if (v < 1e16f && j < M) { s_match[i] = j; s_taken[j] = 1; }
    }
    __syncthreads();
  }

  // ---- MOT public detections (tracker.py:83-103): births only on detections a public detection claims
  if (d.public_det) {
    if (warp == 0) {
      int P = min(d.public_count[b], d.max_public);
      P = P > 0 ? P : 0;
      const int nb = public_births_warp(d.public_det + (size_t)b * d.max_public * 2, P, N, lane, s_px, s_py, s_isz,
                                        s_det, d.new_thresh, s_match, s_claimed, s_born);
      if (lane == 0) s_nborn = nb;
    }
    __syncthreads();
  }

  // ---- output order (tracker.py:74-127): matched detections, then new tracks, then coasting tracks; with
  //      --hungarian the detections / tracks of rejected pairs follow the naturally unmatched ones, in pair order
  if (tid == 0) {
    int pos = 0, ids = id_count;
    for (int i = 0; i < N; ++i) {
      s_pos_det[i] = -1;
      if (s_match[i] >= 0) {
        float* o = s_det + (size_t)i * TF;
        const float* t = s_old + (size_t)s_match[i] * TF;
        o[CT_TRK_ID] = t[CT_TRK_ID]; o[CT_TRK_AGE] = 1.f; o[CT_TRK_ACTIVE] = t[CT_TRK_ACTIVE] + 1.f;
        if (pos < T) s_pos_det[i] = pos++;
      }
    }
    if (d.public_det) {
      for (int k = 0; k < s_nborn; ++k) {
        const int i = s_born[k];
        float* o = s_det + (size_t)i * TF;
        ++ids;
        o[CT_TRK_ID] = (float)ids; o[CT_TRK_AGE] = 1.f; o[CT_TRK_ACTIVE] = 1.f;
        if (pos < T) s_pos_det[i] = pos++;
      }
    } else {
      for (int i = 0; i < N; ++i) {
        if (s_match[i] >= 0 || (hung && s_rej[i] >= 0)) continue;
        float* o = s_det + (size_t)i * TF;
        if (o[CT_TRK_SCORE] > d.new_thresh) {
          ++ids;
          o[CT_TRK_ID] = (float)ids; o[CT_TRK_AGE] = 1.f; o[CT_TRK_ACTIVE] = 1.f;
          if (pos < T) s_pos_det[i] = pos++;
        }
      }
      for (int i = 0; i < N && hung; ++i) {
        if (s_rej[i] < 0) continue;
        float* o = s_det + (size_t)i * TF;
        if (o[CT_TRK_SCORE] > d.new_thresh) {
          ++ids;
          o[CT_TRK_ID] = (float)ids; o[CT_TRK_AGE] = 1.f; o[CT_TRK_ACTIVE] = 1.f;
          if (pos < T) s_pos_det[i] = pos++;
        }
      }
    }
    for (int j = 0; j < M; ++j) {
      s_pos_trk[j] = -1;
      if (s_taken[j]) continue;
      float* t = s_old + (size_t)j * TF;
      if (t[CT_TRK_AGE] < (float)d.max_age) {
        t[CT_TRK_AGE] += 1.f; t[CT_TRK_ACTIVE] = 0.f;
        if (pos < T) s_pos_trk[j] = pos++;
      }
    }
    for (int i = 0; i < N && hung; ++i) {
      const int j = s_rej[i];
      if (j < 0) continue;
      float* t = s_old + (size_t)j * TF;
      if (t[CT_TRK_AGE] < (float)d.max_age) {
        t[CT_TRK_AGE] += 1.f; t[CT_TRK_ACTIVE] = 0.f;
        if (pos < T) s_pos_trk[j] = pos++;
      }
    }
    s_total = pos;
    s_ids = ids;
  }
  __syncthreads();
  const int total = s_total;
  for (int e = tid; e < N * TF; e += TRK_THREADS) {
    const int i = e / TF, f = e - i * TF;
    if (s_pos_det[i] >= 0) trk[(size_t)s_pos_det[i] * TF + f] = s_det[e];
  }
  for (int e = tid; e < M * TF; e += TRK_THREADS) {
    const int j = e / TF, f = e - j * TF;
    if (s_pos_trk[j] >= 0) trk[(size_t)s_pos_trk[j] * TF + f] = s_old[e];
  }
  if (tid == 0) { d.counts[b * 2 + 0] = total; d.counts[b * 2 + 1] = s_ids; }
  __syncthreads();     // the table rows written above are re-read below by other threads
  __threadfence_block();

  // ---- boxes of the NEXT frame's prior heat-map (detector.py:254-290): image -> input coords, clip, radius, centre
  if (d.boxes) {
    const double* ti = d.trans_input + b * 6;
    float* bx = d.boxes + (size_t)b * T * 5;
    for (int r = tid; r < T; r += TRK_THREADS) {
      float radius = -1.f, cxo = 0.f, cyo = 0.f;
      if (r < total) {
        const float* t = trk + (size_t)r * TF;
        if (!(t[CT_TRK_SCORE] < d.pre_thresh) && t[CT_TRK_ACTIVE] != 0.f) {
          const float wmax = (float)(d.inp_w - 1), hmax = (float)(d.inp_h - 1);
          float x0 = (float)aff_f64(ti, (double)t[CT_TRK_BBOX], (double)t[CT_TRK_BBOX + 1]);
          float y0 = (float)aff_f64(ti + 3, (double)t[CT_TRK_BBOX], (double)t[CT_TRK_BBOX + 1]);
          float x1 = (float)aff_f64(ti, (double)t[CT_TRK_BBOX + 2], (double)t[CT_TRK_BBOX + 3]);
          float y1 = (float)aff_f64(ti + 3, (double)t[CT_TRK_BBOX + 2], (double)t[CT_TRK_BBOX + 3]);
          x0 = fminf(fmaxf(x0, 0.f), wmax); x1 = fminf(fmaxf(x1, 0.f), wmax);
          y0 = fminf(fmaxf(y0, 0.f), hmax); y1 = fminf(fmaxf(y1, 0.f), hmax);
          const float h = __fsub_rn(y1, y0), w = __fsub_rn(x1, x0);
          if (h > 0.f && w > 0.f) {
            const double rad = gaussian_radius_f64(ceil((double)h), ceil((double)w));
            const int ri = (int)rad;                 // int(): truncation
            radius = (float)(ri > 0 ? ri : 0);
            cxo = (float)(int)(__fadd_rn(x0, x1) * 0.5f);   // astype(np.int32): truncation
            cyo = (float)(int)(__fadd_rn(y0, y1) * 0.5f);
          }
        }
      }
      bx[r * 5 + 0] = (float)b; bx[r * 5 + 1] = cxo; bx[r * 5 + 2] = cyo; bx[r * 5 + 3] = radius; bx[r * 5 + 4] = 0.f;
    }
  }
}

// splat of the boxes written by track_step_kernel; rows with radius < 0 are skipped.  grid = B*T (fixed: graph-capturable)
__global__ void render_tracks_kernel(const float* __restrict__ boxes, int n, float* __restrict__ hm, int B, int H, int W) {
  const int i = blockIdx.x;
  if (i >= n) return;
  const float rf = boxes[i * 5 + 3];
  if (rf < 0.f) return;
  const int b = (int)boxes[i * 5 + 0], cx = (int)boxes[i * 5 + 1], cy = (int)boxes[i * 5 + 2], r = (int)rf;
  if (b < 0 || b >= B) return;
  const double sigma = (double)(2 * r + 1) / 6.0;
  const int left = min(cx, r), right = min(W - cx, r + 1), top = min(cy, r), bottom = min(H - cy, r + 1);
  const int w = left + right, h = top + bottom;
  if (w <= 0 || h <= 0) return;
  for (int j = threadIdx.x; j < w * h; j += blockDim.x) {
    const int yy = j / w - top, xx = j % w - left;
    double v = exp(-(double)(xx * xx + yy * yy) / (2.0 * sigma * sigma));
    if (v < 2.220446049250313e-16) v = 0.0;
    atomicMax(reinterpret_cast<int*>(hm + ((size_t)b * H + cy + yy) * W + cx + xx), __float_as_int((float)v));
  }
}

// ------------------------------------------------------------------------------------------------------------------
// pre_process: cv2.warpAffine(src u8 HWC, M, (ow, oh), INTER_LINEAR, BORDER_CONSTANT 0) then (v/255 - mean)/std, CHW.
// cv2's arithmetic (imgwarp.cpp warpAffine + remapBilinear): source coordinates in 1/1024 px fixed point rounded
// to 1/32 px, bilinear weights from a 32x32 table of int16 coefficients summing to 2^15, result (sum + 2^14) >> 15.
// ------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ int sat_int(double v) {        // cv::saturate_cast<int>(double) = cvRound, ties to even
  return __double2int_rn(v);
}

__global__ void warp_affine_norm_kernel(const unsigned char* __restrict__ src, int sh, int sw, int sstep,
                                        float* __restrict__ dst, int B, int oh, int ow,
                                        const double* __restrict__ minv /*[B][6] dst->src*/, float3 mean, float3 stdv) {
  const size_t total = (size_t)B * oh * ow;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int b = (int)(i / ((size_t)oh * ow));
    const size_t r = i - (size_t)b * oh * ow;
    const int y = (int)(r / ow), x = (int)(r - (size_t)y * ow);
    const double* M = minv + b * 6;
    const int AB_BITS = 10, AB_SCALE = 1 << AB_BITS, INTER_BITS = 5, INTER_TAB = 1 << INTER_BITS;
    const int round_delta = AB_SCALE / INTER_TAB / 2;
    const int adelta = sat_int(M[0] * x * AB_SCALE), bdelta = sat_int(M[3] * x * AB_SCALE);
    const int X0 = sat_int((M[1] * y + M[2]) * AB_SCALE) + round_delta;
    const int Y0 = sat_int((M[4] * y + M[5]) * AB_SCALE) + round_delta;
    const int X = (X0 + adelta) >> (AB_BITS - INTER_BITS), Y = (Y0 + bdelta) >> (AB_BITS - INTER_BITS);
    const int sx = X >> INTER_BITS, sy = Y >> INTER_BITS;          // arithmetic shifts: floor
    // BilinearTab_i: (1-fy|fy) x (1-fx|fx) in 1/32 steps, scaled by 2^15: exact integers (the table's one saturated
    // entry, fx = fy = 0, yields the same pixel as the exact weight 32768)
    const int fx = X & (INTER_TAB - 1), fy = Y & (INTER_TAB - 1);
    const int w[4] = {(32 - fy) * (32 - fx) * 32, (32 - fy) * fx * 32, fy * (32 - fx) * 32, fy * fx * 32};
    const unsigned char* img = src + (size_t)b * sh * sstep;
    float out[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      int acc = 0;
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        const int yy = sy + (t >> 1), xx = sx + (t & 1);
        const int v = ((unsigned)yy < (unsigned)sh && (unsigned)xx < (unsigned)sw) ? img[(size_t)yy * sstep + xx * 3 + c] : 0;
        acc += v * w[t];
      }
      const int pix = (acc + (1 << 14)) >> 15;
      const int p8 = pix < 0 ? 0 : (pix > 255 ? 255 : pix);
      // ((inp / 255. - mean) / std).astype(float32): float64 arithmetic, one final rounding
      out[c] = (float)p8;
    }
    const size_t plane = (size_t)oh * ow;
    float* o = dst + (size_t)b * 3 * plane + (size_t)y * ow + x;
    o[0] = (float)(((double)out[0] / 255.0 - (double)mean.x) / (double)stdv.x);
    o[plane] = (float)(((double)out[1] / 255.0 - (double)mean.y) / (double)stdv.y);
    o[2 * plane] = (float)(((double)out[2] / 255.0 - (double)mean.z) / (double)stdv.z);
  }
}

}  // namespace ctb

using namespace ctb;

static inline int sw_blocks(size_t total) {
  size_t b = (total + 255) / 256;
  return (int)(b < 148 * 16 ? (b ? b : 1) : 148 * 16);
}

extern "C" int ct_flip_merge(const float* in2, float* out, int32_t C, int32_t H, int32_t W, const int32_t* perm,
                             const float* sign, void* stream) {
  CT_REQUIRE(in2 && out, "null pointer");
  CT_REQUIRE(C > 0 && H > 0 && W > 0, "bad shape");
  flip_merge_kernel<<<sw_blocks((size_t)C * H * W), 256, 0, (cudaStream_t)stream>>>(in2, out, C, H, W, perm, sign);
  return after_launch();
}

extern "C" int64_t ct_track_smem_bytes(int32_t K, int32_t max_tracks) {
  return (int64_t)track_smem_full(K, max_tracks);
}

extern "C" int ct_track_step(const ct_track_desc* d, void* stream) {
  CT_REQUIRE(d && d->records && d->trans_out_inv && d->tracks && d->counts, "null pointer");
  CT_REQUIRE(d->B > 0 && d->K > 0 && d->F >= CT_REC_HEADS && d->max_tracks >= d->K, "bad shape");
  CT_REQUIRE(d->rec_tracking < 0 || d->rec_tracking + 2 <= d->F, "tracking offset outside the record");
  CT_REQUIRE(d->boxes == nullptr || (d->trans_input != nullptr && d->inp_h > 0 && d->inp_w > 0), "boxes need trans_input");
  CT_REQUIRE(d->assign == CT_ASSIGN_GREEDY || d->assign == CT_ASSIGN_HUNGARIAN, "unknown assign mode");
  CT_REQUIRE(d->public_det == nullptr || d->public_count != nullptr, "public_det needs public_count");
  CT_REQUIRE(d->max_public >= 0, "max_public < 0");
  // greedy with private births launches exactly as it did before the solver existed: no scratch
  const bool scratch = d->assign != CT_ASSIGN_GREEDY || d->public_det != nullptr;
  const size_t smem = scratch ? track_smem_full(d->K, d->max_tracks) : track_smem_greedy(d->K, d->max_tracks);
  CT_REQUIRE(smem <= 200 * 1024, "track table does not fit in shared memory (lower max_tracks)");
  if (smem > 48 * 1024)
    CT_CUDA_OK(cudaFuncSetAttribute(track_step_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  TrackArgs a;
  a.d = *d;
  track_step_kernel<<<d->B, TRK_THREADS, smem, (cudaStream_t)stream>>>(a);
  return after_launch();
}

extern "C" int ct_render_tracks(const float* boxes, int32_t n, float* pre_hm, int32_t B, int32_t H, int32_t W,
                                void* stream) {
  CT_REQUIRE(pre_hm && boxes && n > 0, "null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  CT_CUDA_OK(cudaMemsetAsync(pre_hm, 0, (size_t)B * H * W * sizeof(float), st));
  render_tracks_kernel<<<n, 128, 0, st>>>(boxes, n, pre_hm, B, H, W);
  return after_launch();
}

extern "C" int ct_warp_affine_normalize(const uint8_t* src, int32_t B, int32_t src_h, int32_t src_w, int32_t src_step,
                                        const double* minv, const float* mean, const float* std,
                                        float* dst, int32_t out_h, int32_t out_w, void* stream) {
  CT_REQUIRE(src && minv && mean && std && dst, "null pointer");
  CT_REQUIRE(B > 0 && src_h > 0 && src_w > 0 && src_step >= 3 * src_w && out_h > 0 && out_w > 0, "bad shape");
  warp_affine_norm_kernel<<<sw_blocks((size_t)B * out_h * out_w), 256, 0, (cudaStream_t)stream>>>(
      src, src_h, src_w, src_step, dst, B, out_h, out_w, minv, make_float3(mean[0], mean[1], mean[2]),
      make_float3(std[0], std[1], std[2]));
  return after_launch();
}
