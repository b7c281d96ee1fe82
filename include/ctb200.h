/* ctb200.h -- C ABI of libctb200.so: the B200 (sm_100a) implementation of CenterTrack's
 * per-frame inference hot path.  Plain C: raw device pointers, sizes, a cudaStream_t passed
 * as void*; every entry point returns 0 on success or a negative ct_status and never throws.
 * No ownership transfer: the caller (the Python shims in centertrack_b200/, which allocate
 * through torch) owns every buffer.  Thread-compatible: no global mutable state other than
 * the per-thread last-error string.
 *
 * Reference interfaces each entry point replaces (paths relative to the reference's src/lib):
 *   ct_conv_forward   nn.Conv2d+BatchNorm2d(+residual)+ReLU chains of DLA-34: dla.py:38-66
 *                     (BasicBlock), 154-172 (Root), 293-303 (_make_conv_level), 212-218
 *                     (Tree.project); head convs base_model.py:27-38; and, with
 *                     mode=CT_A_DCN, the absent DCNv2 extension's DCN.forward that
 *                     dla.py:513,516 calls (modulated deformable conv v2, 3x3/s1/p1/dg1).
 *   ct_stem_forward   DLA.forward's three 7x7 stems, dla.py:238-242,256-267,305-311.
 *   ct_maxpool2       nn.MaxPool2d(2,2) = Tree.downsample, dla.py:207.
 *   ct_upsample_add   IDAUp's depthwise ConvTranspose2d + skip add, dla.py:529-531,543-545.
 *   ct_decode         Detector.process's decode half: _nms + _topk + _tranpose_and_gather_feat
 *                     + generic_decode, utils.py:16-26,52-87 and decode.py:83-182
 *                     (+ _update_kps_with_hm decode.py:11-81 for the pose heads).
 *   ct_render_pre_hm  Detector._get_additional_inputs's gaussian splat, detector.py:254-290.
 *   ct_track_step     generic_post_process's affine (utils/post_process.py:21-91) + Tracker.step's association
 *                     (utils/tracker.py:28-138: greedy, --hungarian, --public_det births) + the (centre, radius) boxes
 *                     of _get_additional_inputs for the next frame, per stream, on the device;  ct_render_tracks
 *                     splats those boxes (image.py:128-154).
 *   ct_flip_merge     Detector._flip_output, detector.py:311-332 (flip_tensor / flip_lr / flip_lr_off, model/utils.py:28-50).
 *   ct_warp_affine_normalize   Detector.pre_process's cv2.warpAffine + normalise + HWC->CHW, detector.py:207-226.
 */
#ifndef CTB200_H_
#define CTB200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CTB200_ABI_VERSION 1

typedef enum {
  CT_OK = 0,
  CT_ERR_INVALID = -1,     /* bad argument / unsupported shape */
  CT_ERR_CUDA = -2,        /* a CUDA runtime call failed (see ct_last_error) */
  CT_ERR_UNSUPPORTED = -3  /* valid request this build cannot serve */
} ct_status;

typedef enum { CT_F32 = 0, CT_BF16 = 1 } ct_dtype;

/* How the A operand (rows = output pixels, K = taps x C_in) of the implicit GEMM is formed. */
typedef enum {
  CT_A_CONV = 0,  /* plain KxK window, stride/pad */
  CT_A_DCN = 1,   /* 3x3 s1 p1 modulated-deformable bilinear sampling driven by `om` */
  CT_A_DCN_WIN = 2 /* the same operator on the bf16 tcgen05 engine with the input neighbourhood of each 8x16-pixel
                      output patch staged in shared memory by TMA (samples displaced by more than the margin fall
                      back to global memory).  Needs C_in % 64 == 0 and weights packed 64-channel-chunk-major:
                      ct_pack_weights(engine, w', C_out, 64, 3 * C_in / 64, 3, ...) with
                      w'[o][c][chunk * 3 + ky][kx] = w[o][chunk * 64 + c][ky][kx] */
} ct_a_mode;

/* Epilogue / output format. */
typedef enum {
  CT_OUT_NHWC = 0,       /* out[p*ld_out + o], activation dtype */
  CT_OUT_NHWC_F32 = 1,   /* fp32 NHWC (DCN offset/mask map; sigmoid on channels >= sig_from) */
  CT_OUT_NCHW_F32 = 2,   /* fp32 [B,C_out,H,W] planes (head outputs, reference layout) */
  CT_OUT_NHWC_S2D = 3    /* CT_OUT_NHWC written space-to-depth: pixel (y, x) lands at pixel (y/2, x/2), channels
                            [((y&1)*2 + (x&1)) * ld_out, +C_out) of a [B, OH/2, OW/2, 4*ld_out] tensor -- the input
                            layout of a stride-2 3x3 consumer run as a stride-1 2x2 convolution over 4*C channels
                            (DLA stem -> level0 -> level1).  Halo engine only; OH, OW even; no residual. */
} ct_out_mode;

typedef enum {           /* per-launch transform applied to the fp32 NCHW head outputs */
  CT_HEAD_NONE = 0,
  CT_HEAD_SIGMOID = 1,   /* hm, hm_hp: detector.py:301-304 */
  CT_HEAD_DEPTH = 2      /* dep = 1/(sigmoid(x)+1e-6)-1, times depth_scale: detector.py:305-307 */
} ct_head_act;

typedef enum {
  CT_ENGINE_SIMT = 0,          /* fp32 FFMA implicit GEMM (reference accuracy; fp32 or bf16 activations) */
  CT_ENGINE_TCGEN05 = 1,       /* tcgen05 implicit GEMM, A gathered per tap (any stride, DCN) */
  CT_ENGINE_TCGEN05_HALO = 2,  /* tcgen05, TMA-loaded halo tile, taps by descriptor shift: stride-1 'same'
                                  convs with C_in in {8,16,32,48,64,128,192,256} whose weights fit in smem */
  CT_ENGINE_TCGEN05_X3 = 3     /* the gather engine on fp32 activations (dtype CT_F32) with bf16 hi/lo split operands:
                                  D += A_hi B_hi + A_hi B_lo + A_lo B_hi, fp32 accumulate -- ~1e-5 per layer, the
                                  tensor-core path that meets the reference's fp32 results to 1e-3 end to end */
} ct_engine;

/* One convolution-like layer.  Activations are NHWC with an explicit pixel stride (ld, in
 * elements) so that a producer can write straight into a channel slice of a concat buffer
 * (DLA Root nodes, dla.py:167) and a consumer can read a slice back. */
typedef struct {
  int32_t engine;        /* ct_engine */
  int32_t dtype;         /* ct_dtype of activations in/out (CT_ENGINE_TCGEN05 requires CT_BF16) */
  int32_t a_mode;        /* ct_a_mode */
  int32_t B, H, W;       /* input batch / spatial size */
  int32_t C_in, ld_in;   /* input channels used, input pixel stride */
  int32_t C_out;         /* real output channels */
  int32_t KH, KW, stride, pad;
  int32_t OH, OW;        /* output spatial size */
  int32_t ld_out;        /* output pixel stride (CT_OUT_NHWC*; CT_OUT_NHWC_S2D: stride of one of the four sub-pixels) */
  int32_t out_mode;      /* ct_out_mode */
  int32_t relu;          /* 1: ReLU after shift (+residual) */
  int32_t ld_res;        /* residual pixel stride (residual may be NULL) */
  int32_t head_act;      /* ct_head_act (CT_OUT_NCHW_F32 only) */
  int32_t sig_from;      /* CT_OUT_NHWC_F32: sigmoid applied to channels >= sig_from (DCN mask) */
  float   depth_scale;
  int32_t ld_om;         /* CT_A_DCN: pixel stride of `om` (fp32 NHWC, >= 27) */
  int32_t n_tile;        /* tcgen05: output-channel tile (multiple of 16, <= 256); 0 = auto */
  int32_t epilogue_sum3; /* HALO engine, C_out == 48: out16 = sum over present groups g (bit g set) of
                            relu(acc[16g..16g+15] + shift) -- the three DLA stems (dla.py:307-311) */
  int32_t pad_w1;        /* 0: horizontal padding = pad; else horizontal padding + 1 (the (k,1) / (1,k) convs of
                            GlobalConv, dla.py:477-503; SIMT and gather engines) */
  const void* x;         /* input activations */
  const void* w;         /* packed weights: see ct_pack_weights */
  const float* shift;    /* [C_out] folded BN shift / conv bias (may be NULL) */
  const void* residual;  /* [P_out, ld_res] same dtype as activations, or NULL */
  const float* om;       /* CT_A_DCN: offsets (ch 0..17, 2k=dy 2k+1=dx) + sigmoid'd mask (18..26) */
  void* out;
} ct_conv_desc;

/* Size in bytes of the packed weight blob ct_pack_weights produces for this engine/shape. */
int64_t ct_packed_weight_bytes(int32_t engine, int32_t C_out, int32_t C_in, int32_t KH, int32_t KW,
                               int32_t n_tile);
/* Host-side packing.  w_oihw: fp32 [C_out, C_in, KH, KW] (already BN-scale-folded).
 * SIMT engine : fp32 [KH*KW*C_in (k = tap*C_in + c)][C_out padded to 64].
 * tcgen05     : bf16 tiles [n_tiles][k_slices][n_tile rows x 64 k] in the 128B-swizzled
 *               shared-memory image the MMA descriptor expects (one bulk copy per tile).
 * tcgen05 x3  : the same with two tiles per K slice: [hi = bf16(w)][lo = bf16(w - hi)].
 * tcgen05 halo: bf16 [n_tiles][K=16 blocks][2 K-cores][n_tile/8][8 rows][8] (un-swizzled K-major core
 *               matrices); block = (tap, 16 channels), or (ky, tap pair) when C_in == 8. */
int ct_pack_weights(int32_t engine, const float* w_oihw, int32_t C_out, int32_t C_in, int32_t KH,
                    int32_t KW, int32_t n_tile, void* dst);

int ct_conv_forward(const ct_conv_desc* d, void* stream);

/* Three 7x7 stems on reference-layout inputs (fp32 NCHW):
 *   out = relu(bn(conv7(img))) + relu(bn(conv7(pre_img))) + relu(bn(conv7(pre_hm)))
 * w: fp32 [49 taps][7 in-ch (img0..2, pre0..2, hm)][16] BN-scale-folded; shift: [3][16].
 * pre_img / pre_hm may be NULL (dla.py:308-311).  out: NHWC [B,H,W,16] of `dtype`. */
int ct_stem_forward(const float* img, const float* pre_img, const float* pre_hm, const float* w,
                    const float* shift, void* out, int32_t dtype, int32_t B, int32_t H, int32_t W,
                    int32_t ld_out, void* stream);

/* (img, pre_img, pre_hm) fp32 NCHW -> bf16 NHWC [B,H,W,8] = (img0..2, pre0..2, hm, 0): the input of the
 * tensor-core stem (CT_ENGINE_TCGEN05_HALO, 7x7, C_in = 8, epilogue_sum3).  NULL inputs give zeros. */
int ct_pack_stem_input(const float* img, const float* pre_img, const float* pre_hm, void* out, int32_t B,
                       int32_t H, int32_t W, void* stream);

/* the same packing in fp32 (NHWC [B,H,W,8] floats): stem input of CT_ENGINE_TCGEN05_X3 */
int ct_pack_stem_input_f32(const float* img, const float* pre_img, const float* pre_hm, float* out, int32_t B,
                           int32_t H, int32_t W, void* stream);

int ct_maxpool2(const void* x, void* out, int32_t dtype, int32_t B, int32_t H, int32_t W, int32_t C,
                int32_t ld_in, int32_t ld_out, void* stream);

/* the same pooling of a tensor stored space-to-depth (CT_OUT_NHWC_S2D): x [B,H2,W2,(sy,sx,C)] -> out [B,H2,W2,C],
 * out[p][c] = max over the four C-channel groups of pixel p */
int ct_maxpool2_s2d(const void* x, void* out, int32_t dtype, int32_t B, int32_t H2, int32_t W2, int32_t C,
                    int32_t ld_in, int32_t ld_out, void* stream);

/* out[b,oy,ox,c] = skip[...] + sum_{ky,kx} x[b,(oy+pad-ky)/f,(ox+pad-kx)/f,c] * w[ky,kx,c]
 * (depthwise ConvTranspose2d, kernel 2f, stride f, pad f/2; w fp32 channel-last [2f][2f][C]). */
int ct_upsample_add(const void* x, const void* skip, const float* w, void* out, int32_t dtype,
                    int32_t B, int32_t H, int32_t W, int32_t C, int32_t f, int32_t ld_in,
                    int32_t ld_skip, int32_t ld_out, void* stream);

/* ---- decode ------------------------------------------------------------------------- */
#define CT_DECODE_MAX_HEADS 12
typedef enum {          /* role of a gathered regression map in generic_decode */
  CT_ROLE_RAW = 0,      /* copied as-is (tracking, dep, rot, dim, amodel_offset, ...) */
  CT_ROLE_REG = 1,      /* center offset: xs = xs0 + reg_x (decode.py:103-108) */
  CT_ROLE_WH = 2,       /* clamped >= 0, makes bboxes (decode.py:113-129) */
  CT_ROLE_LTRB = 3,     /* bboxes = ct0 + ltrb (decode.py:132-139) */
  CT_ROLE_LTRB_AMODAL = 4, /* bboxes_amodal, overrides bboxes (decode.py:150-159) */
  CT_ROLE_HPS = 5       /* keypoint offsets: += xs0/ys0 (decode.py:161-166) */
} ct_head_role;

typedef struct {
  const float* map;     /* fp32 [B, channels, H, W] */
  int32_t channels;
  int32_t role;         /* ct_head_role */
  int32_t rec_offset;   /* float offset inside a record where the raw gathered row is written */
} ct_decode_head;

typedef struct {
  int32_t B, C, H, W, K;
  const float* hm;          /* post-sigmoid fp32 [B,C,H,W] */
  int32_t n_heads;
  ct_decode_head heads[CT_DECODE_MAX_HEADS];
  /* pose refinement (decode.py:11-81); hm_hp == NULL disables */
  const float* hm_hp;       /* post-sigmoid [B,J,H,W] */
  const float* hp_offset;   /* [B,2,H,W] or NULL (then `reg` head map is used if present, else +0.5) */
  int32_t J;
  int32_t rec_hps;          /* float offset of the 2J refined keypoints, -1 if none */
  int32_t rec_kps_score;    /* float offset of kps_score, -1 if none */
  /* record layout: [score, cls, xs0, ys0, bbox l,t,r,b, ind (int32 bits), ... heads ...] */
  int32_t rec_floats;       /* floats per record (F) */
  int32_t has_bbox;
  float*  records;          /* out [B, K, F] */
  /* workspace: ct_decode_workspace_bytes(...) bytes, 256B aligned; contents need no init
   * except that the first 4*B bytes (per-batch arrival counters) are zeroed by the caller
   * once; the kernel resets them. */
  void* workspace;
} ct_decode_desc;

#define CT_REC_SCORE 0
#define CT_REC_CLS 1
#define CT_REC_XS 2
#define CT_REC_YS 3
#define CT_REC_BBOX 4
#define CT_REC_IND 8
#define CT_REC_HEADS 9

int64_t ct_decode_workspace_bytes(int32_t B, int32_t C, int32_t J, int32_t K);
int ct_decode(const ct_decode_desc* d, void* stream);

/* Gaussian splat of the previous frame's tracks into pre_hm (fp32 [B,1,H,W], zeroed here).
 * boxes: fp32 [n,5] rows (b, cx_int, cy_int, radius, unused) already in INPUT-resolution
 * pixel units -- the affine + gaussian_radius arithmetic stays on the host
 * (detector.py:264-276); the np.maximum splat of image.py:138-154 runs on the device. */
int ct_render_pre_hm(const float* boxes, int32_t n, float* pre_hm, int32_t B, int32_t H, int32_t W,
                     void* stream);

/* ---- per-stream state on the device (SURVEY 8f) ------------------------------------------ */
/* One track / result row: the fields Tracker.step reads and writes (utils/tracker.py), image coordinates. */
#define CT_TRK_SCORE 0
#define CT_TRK_CLASS 1      /* clses + 1 (post_process.py:47) */
#define CT_TRK_CT 2         /* ct x, y */
#define CT_TRK_TRACKING 4   /* tracking dx, dy (already in image coordinates) */
#define CT_TRK_BBOX 6       /* x0, y0, x1, y1 */
#define CT_TRK_ID 10        /* tracking_id (exact in fp32 below 2^24) */
#define CT_TRK_AGE 11
#define CT_TRK_ACTIVE 12
#define CT_TRK_FLOATS 13

typedef struct {
  int32_t B, K, F;            /* decode records [B,K,F] (ct_decode), sorted by score */
  int32_t rec_tracking;       /* float offset of the `tracking` head inside a record, -1 if absent */
  int32_t max_tracks;         /* T: rows of the per-stream track table (>= K; tracks beyond T are dropped) */
  float out_thresh;           /* detections with score > out_thresh survive (detector.py:371-377) */
  float new_thresh;           /* unmatched detections with score > new_thresh start a track (tracker.py:108-113) */
  float pre_thresh;           /* tracks with score >= pre_thresh and active != 0 are splatted (detector.py:262-263) */
  int32_t max_age;            /* unmatched tracks coast while age < max_age (tracker.py:115-126) */
  int32_t inp_h, inp_w;       /* network input size = pre_hm size */
  const float* records;
  const float* trans_out_inv; /* [B,6] fp32: output grid -> image, get_affine_transform(c,s,0,(w,h),inv=1).astype(f32) */
  const double* trans_input;  /* [B,6] fp64: image -> network input (meta['trans_input']); needed when boxes != NULL */
  float* tracks;              /* in/out [B,T,CT_TRK_FLOATS]: the stream's tracks == the results of this step */
  int32_t* counts;            /* in/out [B,2]: number of tracks, id_count */
  float* boxes;               /* out [B,T,5] rows (b, cx, cy, radius, 0) for ct_render_tracks, radius < 0 = skip; or NULL */
  /* Association mode (a zeroed tail = greedy matching, private births: the behaviour before these fields existed). */
  int32_t assign;             /* ct_track_assign */
  const float* public_det;    /* [B,max_public,2] image-coordinate centres of the public detections (MOT --public_det,
                                 tracker.py:83-103): a track may only start on a detection one of them claims; or NULL */
  const int32_t* public_count; /* [B] public detections of this frame per stream (clamped to max_public); needed with
                                  public_det */
  int32_t max_public;         /* row capacity of public_det per stream (>= 0) */
} ct_track_desc;

typedef enum {
  CT_ASSIGN_GREEDY = 0,       /* tracker.py:129-138: detections in score order take their nearest free track */
  CT_ASSIGN_HUNGARIAN = 1     /* --hungarian, tracker.py:52-72: minimum-cost assignment, pair for pair what scipy's
                                 linear_sum_assignment returns on the gated float64 cost (blocked pairs = 1e18); pairs
                                 forced through a blocked cell are handed back as unmatched */
} ct_track_assign;

/* Dynamic shared memory of the largest ct_track_step launch for (K, max_tracks): the track table, this frame's
 * detections and, for CT_ASSIGN_HUNGARIAN / public_det, the solver's per-column and per-row scratch. */
int64_t ct_track_smem_bytes(int32_t K, int32_t max_tracks);
int ct_track_step(const ct_track_desc* d, void* stream);
/* pre_hm (fp32 [B,1,H,W], zeroed here) <- max-splat of boxes [n,5] (rows with radius < 0 skipped); n is the grid size,
 * so the launch shape does not depend on the data (CUDA-graph capturable). */
int ct_render_tracks(const float* boxes, int32_t n, float* pre_hm, int32_t B, int32_t H, int32_t W, void* stream);

/* out[c,y,x] = (in2[0,c,y,x] + sign[c] * in2[1,perm[c],y,W-1-x]) / 2;  in2 fp32 [2,C,H,W], out [1,C,H,W];
 * perm (int32 [C], device) / sign (fp32 [C], device) may be NULL (identity / +1). */
int ct_flip_merge(const float* in2, float* out, int32_t C, int32_t H, int32_t W, const int32_t* perm,
                  const float* sign, void* stream);

/* dst fp32 [B,3,out_h,out_w] = ((warpAffine(src) / 255 - mean) / std), src uint8 [B,src_h,src_w,3] (row pitch src_step
 * bytes), minv fp64 [B,6] = the INVERTED 2x3 map (dst -> src) exactly as cv::warpAffine inverts it; mean/std host fp32[3].
 * Bilinear in cv2's fixed point (1/32 px, 15-bit weights), zero border. */
int ct_warp_affine_normalize(const uint8_t* src, int32_t B, int32_t src_h, int32_t src_w, int32_t src_step,
                             const double* minv, const float* mean, const float* std, float* dst, int32_t out_h,
                             int32_t out_w, void* stream);

/* ---- misc --------------------------------------------------------------------------- */
const char* ct_last_error(void);
int ct_abi_version(void);
/* Kernels launched by this library on the calling thread since the last reset. */
int64_t ct_launch_count(void);
void ct_reset_launch_count(void);
/* Debug: timeline trace of CTA 0 of the halo conv kernel into device_buf (>= 16 KB of uint64: 8 clock64()
 * stamps per work item, see csrc/conv_halo.cu); NULL switches it off (default). */
int ct_debug_trace(void* device_buf);
/* Debug: 4 uint32 of host-MAPPED memory; a stuck mbarrier wait in the halo kernel writes (site, item, block, warp)
 * there before trapping.  NULL = off (default). */
int ct_debug_watch(void* mapped_host_buf);

#ifdef __cplusplus
}
#endif
#endif /* CTB200_H_ */
