// Pieces shared by the SIMT (fp32-exact) and tcgen05 (bf16) implicit-GEMM engines: output-pixel decomposition, conv
// window addressing, DCNv2 bilinear sampling, and the tensor-core engines' host-side launch setup.
#pragma once
#include "common.cuh"
#include <cuda.h>
#include <utility>
#include <vector>

namespace ctb {

struct ConvGeom {
  int B, H, W, C_in, ld_in;
  int C_out, KH, KW, stride, pad, pad_w, OH, OW;
  int ld_out, out_mode, relu, ld_res, head_act, sig_from;
  float depth_scale;
  int ld_om;
  int P_out;      // B*OH*OW
  int K_total;    // KH*KW*C_in
};

inline ConvGeom make_geom(const ct_conv_desc* d) {
  ConvGeom g;
  g.B = d->B; g.H = d->H; g.W = d->W; g.C_in = d->C_in; g.ld_in = d->ld_in;
  g.C_out = d->C_out; g.KH = d->KH; g.KW = d->KW; g.stride = d->stride; g.pad = d->pad;
  g.pad_w = d->pad_w1 > 0 ? d->pad_w1 - 1 : d->pad;
  g.OH = d->OH; g.OW = d->OW; g.ld_out = d->ld_out; g.out_mode = d->out_mode;
  g.relu = d->relu; g.ld_res = d->ld_res; g.head_act = d->head_act; g.sig_from = d->sig_from;
  g.depth_scale = d->depth_scale; g.ld_om = d->ld_om;
  g.P_out = d->B * d->OH * d->OW;
  g.K_total = d->KH * d->KW * d->C_in;
  return g;
}

// Modulated-deformable sampling parameters of one (output pixel, tap):  SURVEY.md Appendix B.
//   py = y - 1 + i + dy_k,  px = x - 1 + j + dx_k ;  S = 0 unless -1 < py < H and -1 < px < W ;
//   bilinear over the integer neighbours that lie inside the image; the whole sample times mask.
struct DcnTap {
  int off[4];     // element offsets (relative to the image base) of the 4 corner pixels
  float w[4];     // bilinear weight x mask, 0 for corners outside the image
};

__device__ __forceinline__ DcnTap dcn_tap(const float* __restrict__ om_px, int tap, int oy, int ox,
                                          int H, int W, int ld_in) {
  DcnTap t;
  const float dy = om_px[2 * tap], dx = om_px[2 * tap + 1], m = om_px[18 + tap];
  const float py = (float)(oy - 1 + tap / 3) + dy;
  const float px = (float)(ox - 1 + tap % 3) + dx;
  const bool valid = (py > -1.f) && (py < (float)H) && (px > -1.f) && (px < (float)W);
  const float y0f = floorf(py), x0f = floorf(px);
  const float ly = py - y0f, lx = px - x0f, hy = 1.f - ly, hx = 1.f - lx;
  const int y0 = (int)y0f, x0 = (int)x0f;
  const bool y0ok = valid && y0 >= 0 && y0 <= H - 1, y1ok = valid && y0 + 1 >= 0 && y0 + 1 <= H - 1;
  const bool x0ok = x0 >= 0 && x0 <= W - 1, x1ok = x0 + 1 >= 0 && x0 + 1 <= W - 1;
  const int yc0 = min(max(y0, 0), H - 1), yc1 = min(max(y0 + 1, 0), H - 1);
  const int xc0 = min(max(x0, 0), W - 1), xc1 = min(max(x0 + 1, 0), W - 1);
  t.off[0] = (yc0 * W + xc0) * ld_in; t.w[0] = (y0ok && x0ok) ? hy * hx * m : 0.f;
  t.off[1] = (yc0 * W + xc1) * ld_in; t.w[1] = (y0ok && x1ok) ? hy * lx * m : 0.f;
  t.off[2] = (yc1 * W + xc0) * ld_in; t.w[2] = (y1ok && x0ok) ? ly * hx * m : 0.f;
  t.off[3] = (yc1 * W + xc1) * ld_in; t.w[3] = (y1ok && x1ok) ? ly * lx * m : 0.f;
  return t;
}

// Apply the per-channel epilogue transform of fp32 head planes.
__device__ __forceinline__ float head_transform(float v, int head_act, float depth_scale) {
  if (head_act == CT_HEAD_SIGMOID) return sigmoidf_ref(v);
  if (head_act == CT_HEAD_DEPTH) return (1.f / (sigmoidf_ref(v) + 1e-6f) - 1.f) * depth_scale;
  return v;
}

// ---- host-side launch setup shared by the tensor-core engines ----
// cuTensorMapEncodeTiled through the runtime's driver entry point (no -lcuda at link time); nullptr if unavailable
typedef CUresult (*TmapEncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                      const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                      CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
inline TmapEncodeTiledFn tmap_encode_tiled() {
  static TmapEncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<TmapEncodeTiledFn>(p);
  }
  return fn;
}

// Tensor map of a bf16 tensor (innermost dimension first, byte strides of the outer ones), unit element strides,
// zero fill outside the tensor.  `who` names the caller in the error message.
inline int encode_tmap_bf16(CUtensorMap* map, const void* x, cuuint32_t rank, const cuuint64_t* dims,
                            const cuuint64_t* strides, const cuuint32_t* box, CUtensorMapSwizzle swizzle,
                            const char* who) {
  const TmapEncodeTiledFn enc = tmap_encode_tiled();
  if (!enc) return fail(CT_ERR_CUDA, "%s: cuTensorMapEncodeTiled entry point unavailable", who);
  const cuuint32_t estr[4] = {1, 1, 1, 1};
  const CUresult cr = enc(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, rank, const_cast<void*>(x), dims, strides, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return cr == CUDA_SUCCESS ? CT_OK : fail(CT_ERR_CUDA, "%s: cuTensorMapEncodeTiled failed (%ld)", who, (long)cr);
}

// 4-D map {C, W, H, B} of a bf16 NHWC tensor whose pixel stride is `ld` elements; box {box_c, box_w, box_h, 1}
inline int encode_tmap_nhwc_bf16(CUtensorMap* map, const void* x, int B, int H, int W, int C, int ld, int box_c,
                                 int box_w, int box_h, CUtensorMapSwizzle swizzle, const char* who) {
  const cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B};
  const cuuint64_t strides[3] = {(cuuint64_t)ld * 2, (cuuint64_t)W * ld * 2, (cuuint64_t)H * W * ld * 2};
  const cuuint32_t box[4] = {(cuuint32_t)box_c, (cuuint32_t)box_w, (cuuint32_t)box_h, 1};
  return encode_tmap_bf16(map, x, 4, dims, strides, box, swizzle, who);
}

// Raises `kernel`'s dynamic shared-memory limit to `bytes`, once per (kernel, device): the attribute is per device, and
// a process may drive several GPUs from one thread.
inline cudaError_t set_max_dynamic_smem_once(const void* kernel, int bytes) {
  int dev = 0;
  cudaGetDevice(&dev);
  static thread_local std::vector<std::pair<const void*, int>> done;
  for (const auto& e : done)
    if (e.first == kernel && e.second == dev) return cudaSuccess;
  const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e == cudaSuccess) done.emplace_back(kernel, dev);
  return e;
}

// SM count of the current device, queried once per device (148 if the query fails)
inline int sm_count() {
  int dev = 0;
  cudaGetDevice(&dev);
  static thread_local std::vector<int> sms;
  if ((int)sms.size() <= dev) sms.resize(dev + 1, 0);
  if (sms[dev] == 0 && cudaDeviceGetAttribute(&sms[dev], cudaDevAttrMultiProcessorCount, dev) != cudaSuccess)
    sms[dev] = 0;
  return sms[dev] > 0 ? sms[dev] : 148;
}

int conv_forward_simt(const ct_conv_desc* d, cudaStream_t st);
int conv_forward_tc(const ct_conv_desc* d, cudaStream_t st);
int conv_forward_halo(const ct_conv_desc* d, cudaStream_t st);
int halo_blocks(int C_in, int KH, int KW);
int halo_set_trace(void* buf);
int tc_set_trace(void* buf);
int halo_set_watch(void* mapped_host_buf);

}  // namespace ctb
