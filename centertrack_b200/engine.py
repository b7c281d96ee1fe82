"""DLA-34 + DLAUp/IDAUp(DCNv2) + heads as a static plan of libctb200 launches.

The plan restates the dataflow of the reference's DLASeg (dla.py:594-640, Appendix A of SURVEY.md)
on NHWC activations:
  * every Conv2d+BatchNorm2d(+residual)+ReLU is ONE ct_conv_forward launch (BN folded into the
    weights / shift on the host, dla.py:38-66,154-172,293-303);
  * Root's torch.cat (dla.py:167) never happens: producers write straight into channel slices of a
    concat buffer (explicit pixel stride `ld`), the Root 1x1 conv reads the buffer;
  * the two dead `base.level{3,4}.project` convs (SURVEY hazard H4) are accepted in the
    state_dict and not executed;
  * DeformConv (dla.py:506-518) = offset/mask 3x3 conv (fp32 NHWC map, sigmoid fused on the mask
    channels) + the DCN implicit GEMM with BN+ReLU fused;
  * IDAUp's `up(proj(x)) + skip` (dla.py:543-545) is one fused depthwise-transposed-conv + add;
  * all heads' first 3x3 convs (base_model.py:27-38) run as one conv 64 -> 256*n_heads, then one
    1x1 per head writing the reference-layout fp32 NCHW map (sigmoid / depth transform of
    detector.py:300-308 optionally fused).

precision='bf16'   : bf16 activations, tcgen05 engines (fast path)
precision='bf16x3' : fp32 activations, tcgen05 gather engine with bf16 hi/lo split operands (three MMAs per product
                     term, fp32 accumulate): the tensor-core path that stays within 1e-3 of the reference
precision='fp32'   : fp32 activations, SIMT engine (reference-accuracy path, <= 1e-3 of the reference)
"""
import ctypes as C
import os

import numpy as np
import torch

from . import _lib as L

BN_EPS = 1e-5


class TV(object):
  """A channel slice [off, off+C) of an NHWC buffer [B,H,W,ld]."""

  def __init__(self, buf, off, Cn):
    self.buf, self.off, self.C = buf, off, Cn
    self.B, self.H, self.W, self.ld = buf.shape

  @property
  def ptr(self):
    return self.buf.data_ptr() + self.off * self.buf.element_size()

  def tensor(self):
    return self.buf[..., self.off:self.off + self.C]


def s2d_weights_3x3_s1(w):
  """3x3 stride-1 pad-1 conv [O, I, 3, 3] -> the same operator on the space-to-depth grid: [4 O, 4 I, 3, 3] acting on
  channels (sy, sx, c) of [B, 4 C, H/2, W/2].  Output sub-pixel sy' reads full-res row 2Y + sy' + ky - 1 = s2d row
  Y + ty - 1, sub-row sy, with 2 (ty - 1) + sy = sy' + ky - 1; same along x.  3/4 of the entries are structural zeros."""
  O, I = w.shape[:2]
  ws = torch.zeros((4 * O, 4 * I, 3, 3), dtype=w.dtype)
  for sy_o in range(2):
    for sx_o in range(2):
      o0 = (sy_o * 2 + sx_o) * O
      for ky in range(3):
        for kx in range(3):
          ry, rx = sy_o + ky - 1, sx_o + kx - 1
          ty, sy, tx, sx = ry // 2 + 1, ry % 2, rx // 2 + 1, rx % 2
          c0 = (sy * 2 + sx) * I
          ws[o0:o0 + O, c0:c0 + I, ty, tx] = w[:, :, ky, kx]
  return ws


def s2d_weights_3x3_s2(w):
  """3x3 stride-2 pad-1 conv [O, I, 3, 3] -> a 2x2 stride-1 conv [O, 4 I, 2, 2] over the space-to-depth input, padded on
  the top / left only: input row 2 oy - 1 + ky = s2d row oy + ty - 1, sub-row sy with (ty, sy) = (0, 1), (1, 0), (1, 1)
  for ky = 0, 1, 2; same along x."""
  O, I = w.shape[:2]
  ws = torch.zeros((O, 4 * I, 2, 2), dtype=w.dtype)
  tap = ((0, 1), (1, 0), (1, 1))
  for ky in range(3):
    for kx in range(3):
      (ty, sy), (tx, sx) = tap[ky], tap[kx]
      c0 = (sy * 2 + sx) * I
      ws[:, c0:c0 + I, ty, tx] = w[:, :, ky, kx]
  return ws


class DLA34Engine(object):

  def __init__(self, state_dict, heads, B, H, W, precision='bf16', device='cuda',
               depth_scale=1.0, has_pre_img=True, has_pre_hm=True, dla_node='dcn'):
    assert precision in ('bf16', 'fp32', 'bf16x3')
    assert dla_node in ('dcn', 'conv', 'gcn')
    self.dla_node = dla_node
    assert H % 32 == 0 and W % 32 == 0, 'DLA-34 needs input sizes divisible by 32'
    self.lib = L.lib()
    self.sd = {k: v.detach().to('cpu', torch.float64) for k, v in state_dict.items()
               if v.dtype.is_floating_point}
    self.heads = dict(heads)
    self.B, self.H, self.W = B, H, W
    self.precision = precision
    self.device = torch.device(device)
    self.dtype = torch.bfloat16 if precision == 'bf16' else torch.float32
    self.ct_dtype = L.CT_BF16 if precision == 'bf16' else L.CT_F32
    self.engine = {'bf16': L.CT_ENGINE_TCGEN05, 'fp32': L.CT_ENGINE_SIMT, 'bf16x3': L.CT_ENGINE_TCGEN05_X3}[precision]
    self.x3 = (precision == "bf16x3")
    self.depth_scale = float(depth_scale)
    self.has_pre_img = has_pre_img and ('base.pre_img_layer.0.weight' in self.sd)
    self.has_pre_hm = has_pre_hm and ('base.pre_hm_layer.0.weight' in self.sd)
    self.ops = []          # (kind, payload)
    self.keep = []         # device tensors referenced by raw pointers
    self.named = {}        # name -> TV (for per-stage parity tests)
    self.head_descs = {}   # head -> final ConvDesc (to toggle the fused activation)
    self.algo_flops = {}   # op name -> flops of the reference layer, where the launch shape carries structural zeros
    self.s2d_named = set() # named intermediates stored space-to-depth ([B, H/2, W/2, (sy, sx, 16)])
    self.n_sm = 148
    self.debug_sync = bool(int(os.environ.get('CTB_DEBUG_SYNC', '0')))
    self.use_halo = precision == 'bf16'
    self._build()
    self.graph = None

  # ------------------------------------------------------------------ helpers
  def _buf(self, h, w, c, dtype=None):
    t = torch.empty((self.B, h, w, c), dtype=dtype or self.dtype, device=self.device)
    self.keep.append(t)
    return t

  def _dev(self, t):
    t = t.to(self.device)
    self.keep.append(t)
    return t

  def _fold(self, conv, bn=None, bias_key=None):
    """-> (W' [O,I,kh,kw] float64, shift [O] float64): BN(eval) folded into conv."""
    w = self.sd[conv + '.weight']
    O = w.shape[0]
    b = self.sd[bias_key] if bias_key is not None and bias_key in self.sd else \
        self.sd.get(conv + '.bias', torch.zeros(O, dtype=torch.float64))
    if bn is None:
      return w, b
    s = self.sd[bn + '.weight'] / torch.sqrt(self.sd[bn + '.running_var'] + BN_EPS)
    shift = self.sd[bn + '.bias'] - self.sd[bn + '.running_mean'] * s + b * s
    return w * s.view(-1, 1, 1, 1), shift

  def _pick_n_tile(self, P, C_out):
    cpad = (C_out + 15) // 16 * 16
    cands = [c for c in (256, 128, 64, 32, 16) if c <= max(cpad, 16)]
    if cpad <= 256 and cpad not in cands:
      cands = [cpad] + cands
    m_tiles = (P + 127) // 128
    for c in cands:
      if m_tiles * ((C_out + c - 1) // c) >= self.n_sm:
        return c
    small = [c for c in cands if c >= 64]
    return small[-1] if small else cands[0]

  def _pack(self, w, n_tile, engine):
    """w: float64 [O,I,kh,kw] -> packed device blob for `engine`."""
    w32 = w.to(torch.float32).contiguous()
    O, I, kh, kw = w32.shape
    nbytes = self.lib.ct_packed_weight_bytes(engine, O, I, kh, kw, n_tile)
    assert nbytes > 0
    dst = torch.empty(nbytes, dtype=torch.uint8)
    L.check(self.lib.ct_pack_weights(engine, C.c_void_p(w32.data_ptr()), O, I, kh, kw, n_tile,
                                     C.c_void_p(dst.data_ptr())), 'ct_pack_weights')
    return self._dev(dst)

  def _conv(self, name, x, w, shift, out, k, stride=1, relu=True, residual=None, a_mode=L.CT_A_CONV,
            om=None, out_mode=L.CT_OUT_NHWC, head_act=L.CT_HEAD_NONE, sig_from=1 << 30, c_out=None, sum3=0,
            w_pack=None, out_hw=None):
    """Append one conv-like launch.  x: TV; out: TV (NHWC modes) or fp32 tensor (NCHW)."""
    C_in = x.C
    if w.shape[1] != C_in:      # input channels padded (never happens for DLA-34 tensors)
      raise ValueError('%s: C_in mismatch %d vs %d' % (name, w.shape[1], C_in))
    C_out = w.shape[0] if c_out is None else c_out
    kh, kw = (k, k) if isinstance(k, int) else k
    pad, pad_w = kh // 2, kw // 2
    OH = (x.H + 2 * pad - kh) // stride + 1
    OW = (x.W + 2 * pad_w - kw) // stride + 1
    if out_hw is not None:      # even kernels: padding on the top / left only (ctb200.h, OH / OW)
      OH, OW = out_hw
    P = self.B * OH * OW
    engine = self.engine
    n_tile = self._pick_n_tile(P, C_out) if engine in (L.CT_ENGINE_TCGEN05, L.CT_ENGINE_TCGEN05_X3) else 0
    if engine == L.CT_ENGINE_TCGEN05_X3 and n_tile > 128 and a_mode == L.CT_A_DCN:
      n_tile = 128            # x3 DCN: two 36 KB-table stages of (32 + 2 x n_tile/8) KB must fit
    if engine == L.CT_ENGINE_TCGEN05 and self.use_halo and a_mode == L.CT_A_CONV and stride == 1 and kh == kw and \
        (C_in in (16, 32, 48, 64, 128, 192, 256) or (C_in == 8 and sum3)):
      k = kh
      # stride-1 layer whose weights fit in smem: TMA halo tile + descriptor-shifted taps (csrc/conv_halo.cu)
      nblk = k * ((k + 1) // 2) if C_in == 8 else k * k * (C_in // 16)
      halo = C_in * 2 * (8 + k - 1 + (1 if C_in == 8 else 0)) * (16 + k - 1) + 1024 * max(1, C_in // 64)
      cpad = (C_out + 15) // 16 * 16
      for nt in ([48] if sum3 else [c for c in (128, 96, 80, 64, 48, 32, 16) if c <= cpad and (c == cpad or cpad % c == 0 or c >= 64)]):
        if nblk * nt * 32 + 2 * halo + 4096 <= 224 * 1024 and (nt >= 32 or cpad <= 16):
          engine, n_tile = L.CT_ENGINE_TCGEN05_HALO, nt
          break
    d = L.ConvDesc()
    d.engine, d.dtype, d.a_mode = engine, self.ct_dtype, a_mode
    d.epilogue_sum3 = sum3
    d.B, d.H, d.W, d.C_in, d.ld_in, d.C_out = self.B, x.H, x.W, C_in, x.ld, C_out
    d.KH, d.KW = kh, kw
    d.stride, d.pad, d.OH, d.OW = stride, pad, OH, OW
    d.pad_w1 = 0 if pad_w == pad else pad_w + 1
    d.out_mode, d.relu, d.head_act, d.sig_from = out_mode, int(relu), head_act, sig_from
    d.depth_scale = self.depth_scale
    d.n_tile = n_tile
    d.x = x.ptr
    d.w = self._pack(w if w_pack is None else w_pack, n_tile, engine).data_ptr()
    sh = self._dev(shift.to(torch.float32).contiguous())
    d.shift = sh.data_ptr()
    if residual is not None:
      d.residual, d.ld_res = residual.ptr, residual.ld
    if om is not None:
      d.om, d.ld_om = om.data_ptr(), om.shape[-1]
    if out_mode == L.CT_OUT_NCHW_F32:
      assert out.shape == (self.B, C_out, OH, OW) and out.dtype == torch.float32
      d.out, d.ld_out = out.data_ptr(), 0
    elif out_mode == L.CT_OUT_NHWC_F32:
      assert out.shape[:3] == (self.B, OH, OW) and out.dtype == torch.float32
      d.out, d.ld_out = out.data_ptr(), out.shape[-1]
    elif out_mode == L.CT_OUT_NHWC_S2D:
      co = 16 if sum3 else C_out
      assert engine == L.CT_ENGINE_TCGEN05_HALO and (out.H, out.W, out.C, out.ld) == (OH // 2, OW // 2, 4 * co, 4 * co)
      d.out, d.ld_out = out.ptr, co
      self.named[name] = out
    else:
      assert (out.H, out.W) == (OH, OW) and out.C == (16 if sum3 else C_out), (name, out.H, out.W, out.C, OH, OW, C_out)
      d.out, d.ld_out = out.ptr, out.ld
      self.named[name] = out
    self.ops.append(('conv', d, name))
    return d

  def _conv_bn(self, name, x, conv, bn, out, k, stride=1, relu=True, residual=None):
    w, shift = self._fold(conv, bn)
    return self._conv(name, x, w, shift, out, k, stride, relu, residual)

  def _maxpool(self, x, out):
    self.ops.append(('pool', (x, out), 'maxpool'))

  def _basic_block(self, p, x, out, stride, residual, x_s2d=False):
    """BasicBlock dla.py:38-66: conv1-bn1-relu-conv2-bn2-(+residual)-relu.  x_s2d: x is stored space-to-depth
    ([B, H/2, W/2, 4 C]) and stride is 2: conv1 runs as a 2x2 stride-1 convolution over it (s2d_weights_3x3_s2)."""
    if x_s2d:
      assert stride == 2
      oh, ow = x.H, x.W
      mid = TV(self._buf(oh, ow, out.C), 0, out.C)
      w, sh = self._fold(p + '.conv1', p + '.bn1')
      self._conv(p + '.conv1', x, s2d_weights_3x3_s2(w), sh, mid, 2, 1, out_hw=(oh, ow))
      self.algo_flops[p + '.conv1'] = 2.0 * self.B * oh * ow * w.shape[0] * 9 * w.shape[1]
    else:
      oh, ow = x.H // stride, x.W // stride
      mid = TV(self._buf(oh, ow, out.C), 0, out.C)
      self._conv_bn(p + '.conv1', x, p + '.conv1', p + '.bn1', mid, 3, stride, True)
    self._conv_bn(p, mid, p + '.conv2', p + '.bn2', out, 3, 1, True, residual)

  def _deform(self, p, x, out):
    """DeformConv dla.py:506-518 = DCN + BN + ReLU."""
    sd = self.sd
    om = self._buf(x.H, x.W, 32, torch.float32)
    self._conv(p + '.offset', x, sd[p + '.conv.conv_offset_mask.weight'],
               sd[p + '.conv.conv_offset_mask.bias'], om, 3, 1, relu=False,
               out_mode=L.CT_OUT_NHWC_F32, sig_from=18)
    w, shift = self._fold(p + '.conv', p + '.actf.0')
    if self.engine == L.CT_ENGINE_TCGEN05 and x.C % 64 == 0:
      # sample from a TMA-staged shared-memory window; K order = (64-channel chunk, tap, channel).  With the persistent
      # window kernel this also wins on 128 -> 128 at 64x64 (100 vs 124 us for the global-memory sampler)
      nch = x.C // 64
      w_cm = w.reshape(w.shape[0], nch, 64, 3, 3).permute(0, 2, 1, 3, 4).reshape(w.shape[0], 64, nch * 3, 3)
      self._conv(p, x, w, shift, out, 3, 1, relu=True, a_mode=L.CT_A_DCN_WIN, om=om, w_pack=w_cm.contiguous())
    else:
      self._conv(p, x, w, shift, out, 3, 1, relu=True, a_mode=L.CT_A_DCN, om=om)

  def _node(self, p, x, out, which):
    """IDAUp's proj (which=0) / node (which=1) module by --dla_node (dla.py:588-592): DeformConv | Conv | GlobalConv."""
    if self.dla_node == 'dcn':
      return self._deform(p, x, out)
    if self.dla_node == 'conv' or which == 0:             # Conv (dla.py:466-475): 1x1 conv + BN + ReLU
      return self._conv_bn(p, x, p + '.conv.0', p + '.conv.1', out, 1)
    # GlobalConv (dla.py:477-503): relu(bn((1xk o kx1)(x) + (kx1 o 1xk)(x))).  BN is affine, so its scale folds into
    # the second conv of each branch, its shift into the left branch, and the right branch adds the left as residual.
    sd = self.sd
    kk = sd[p + '.gcl.0.weight'].shape[2]
    s = sd[p + '.act.0.weight'] / torch.sqrt(sd[p + '.act.0.running_var'] + BN_EPS)
    t = sd[p + '.act.0.bias'] - sd[p + '.act.0.running_mean'] * s
    zero = torch.zeros(out.C, dtype=torch.float64)
    t1 = TV(self._buf(x.H, x.W, out.C), 0, out.C)
    left = TV(self._buf(x.H, x.W, out.C), 0, out.C)
    t2 = TV(self._buf(x.H, x.W, out.C), 0, out.C)
    self._conv(p + '.gcl.0', x, sd[p + '.gcl.0.weight'], zero, t1, (kk, 1), 1, relu=False)
    self._conv(p + '.gcl.1', t1, sd[p + '.gcl.1.weight'] * s.view(-1, 1, 1, 1), t, left, (1, kk), 1, relu=False)
    self._conv(p + '.gcr.0', x, sd[p + '.gcr.0.weight'], zero, t2, (1, kk), 1, relu=False)
    return self._conv(p, t2, sd[p + '.gcr.1.weight'] * s.view(-1, 1, 1, 1), zero, out, (kk, 1), 1, relu=True, residual=left)

  def _up_add(self, p, x, skip, out, f):
    w = self._dev(self.sd[p + '.weight'].to(torch.float32).reshape(x.C, 2 * f, 2 * f).permute(1, 2, 0).contiguous())
    self.ops.append(('up', (x, skip, w, out, f), p))
    self.named[p] = out

  def _ida(self, p, layers, startp, endp, o):
    """IDAUp.forward dla.py:539-545 on TVs."""
    for i in range(startp + 1, endp):
      j = i - startp
      src = layers[i]
      proj = TV(self._buf(src.H, src.W, o), 0, o)
      self._node('%s.proj_%d' % (p, j), src, proj, 0)
      upw = self.sd['%s.up_%d.weight' % (p, j)]
      f = upw.shape[2] // 2
      summed = TV(self._buf(src.H * f, src.W * f, o), 0, o)
      self._up_add('%s.up_%d' % (p, j), proj, layers[i - 1], summed, f)
      node = TV(self._buf(src.H * f, src.W * f, o), 0, o)
      self._node('%s.node_%d' % (p, j), summed, node, 1)
      layers[i] = node

  # ------------------------------------------------------------------ plan
  def _build(self):
    B, H, W = self.B, self.H, self.W
    sd = self.sd
    f32 = torch.float32
    # static inputs in the reference's layout (fp32 NCHW)
    self.in_img = torch.zeros((B, 3, H, W), dtype=f32, device=self.device)
    self.in_pre = torch.zeros((B, 3, H, W), dtype=f32, device=self.device)
    self.in_hm = torch.zeros((B, 1, H, W), dtype=f32, device=self.device)

    # ---- stems (dla.py:238-242,256-267,305-311) ----
    wst = torch.zeros((49, 7, 16), dtype=torch.float64)
    shst = torch.zeros((3, 16), dtype=torch.float64)
    for si, (pfx, c0, cn) in enumerate((('base.base_layer', 0, 3), ('base.pre_img_layer', 3, 3),
                                        ('base.pre_hm_layer', 6, 1))):
      if pfx + '.0.weight' not in sd:
        continue
      w, sh = self._fold(pfx + '.0', pfx + '.1')          # [16,cn,7,7]
      wst[:, c0:c0 + cn, :] = w.permute(2, 3, 1, 0).reshape(49, cn, 16)
      shst[si] = sh
    self.stem_w = self._dev(wst.to(f32).contiguous())
    self.stem_shift = self._dev(shst.to(f32).contiguous())
    s2d = self.use_halo and H % 2 == 0 and W % 2 == 0      # stem -> level0 -> level1 on the space-to-depth grid
    x0 = TV(self._buf(H // 2, W // 2, 64), 0, 64) if s2d else TV(self._buf(H, W, 16), 0, 16)
    if self.use_halo:
      # tensor-core stem: pack (img, pre, hm) -> bf16 NHWC [.,8], one 7x7 conv 8 -> 48 (block-diagonal over the
      # three stems) whose epilogue applies ReLU per stem and sums them (dla.py:307-311)
      x8 = TV(self._buf(H, W, 8), 0, 8)
      self.ops.append(('pack', x8, 'stem.pack'))
      w48 = torch.zeros((48, 8, 7, 7), dtype=torch.float64)
      for si, (c0, cn) in enumerate(((0, 3), (3, 3), (6, 1))):
        w48[16 * si:16 * si + 16, c0:c0 + cn] = wst[:, c0:c0 + cn, :].reshape(7, 7, cn, 16).permute(3, 2, 0, 1)
      self.stem_desc = self._conv('stem', x8, w48, shst.reshape(48), x0, 7, 1, relu=False, sum3=7,
                                  out_mode=L.CT_OUT_NHWC_S2D if s2d else L.CT_OUT_NHWC)
      if s2d:
        self.s2d_named.add('stem')
    elif self.x3:
      # bf16x3 stem: pack (img, pre, hm) -> fp32 NHWC [.,8], one 7x7 conv 8 -> 48 (block-diagonal over the three stems)
      # with shift + ReLU per stem; the sum of the three (dla.py:307-311) is folded into level0, whose 3x3 conv reads
      # the 48 channels with its weights tiled three times along the input (conv(a + b + c) = conv over [a|b|c])
      x8 = TV(self._buf(H, W, 8), 0, 8)
      self.ops.append(('pack32', x8, 'stem.pack'))
      w48 = torch.zeros((48, 8, 7, 7), dtype=torch.float64)
      sh48 = shst.clone()
      for si, (c0, cn) in enumerate(((0, 3), (3, 3), (6, 1))):
        w48[16 * si:16 * si + 16, c0:c0 + cn] = wst[:, c0:c0 + cn, :].reshape(7, 7, cn, 16).permute(3, 2, 0, 1)
      x0 = TV(self._buf(H, W, 48), 0, 48)
      self.stem48 = self._conv('stem48', x8, w48, sh48.reshape(48), x0, 7, 1, relu=True)
      # an absent input (pre_img / pre_hm is None, dla.py:308-311) must contribute nothing: its packed channels are
      # zero, so only its group's shift has to go -> one shift vector per presence mask
      self.stem48_shift = {}
      for mask in range(8):
        shm = sh48.clone()
        for gi in range(3):
          if not (mask >> gi) & 1:
            shm[gi] = 0
        self.stem48_shift[mask] = self._dev(shm.reshape(48).to(f32).contiguous())
    else:
      self.ops.append(('stem', x0, 'stem'))
    self.named['stem'] = x0

    # ---- level0 / level1 ----
    if not s2d:
      l1 = TV(self._buf(H // 2, W // 2, 32), 0, 32)
      l0 = TV(self._buf(H, W, 16), 0, 16)
      if self.x3:
        w0, sh0 = self._fold('base.level0.0', 'base.level0.1')
        self._conv('base.level0', x0, w0.repeat(1, 3, 1, 1), sh0, l0, 3, 1)
      else:
        self._conv_bn('base.level0', x0, 'base.level0.0', 'base.level0.1', l0, 3, 1)
      self._conv_bn('base.level1', l0, 'base.level1.0', 'base.level1.1', l1, 3, 2)
    else:
      # The 16-channel 512x512 layers on the space-to-depth grid [B, H/2, W/2, (sy, sx, 16)] (written in that layout by
      # the stem's epilogue, CT_OUT_NHWC_S2D): 128-byte pixel rows for the TMA instead of 32-byte ones (level0 was bound
      # by the TMA's row rate), N = 64 per MMA instead of 16 at the same MMA count, and level1's stride 2 disappears.
      #  level0 (3x3 s1 16 -> 16): output sub-pixel sy' reads full-res row 2Y + sy' + ky - 1 = s2d row Y + ty - 1, sub-row
      #    sy with 2 (ty - 1) + sy = sy' + ky - 1  ->  a 3x3 convolution 64 -> 64 whose weights are 3/4 structural zeros.
      #  level1 (3x3 s2 16 -> 32): input row 2 oy - 1 + ky = s2d row oy + ty - 1, sub-row sy with (ty, sy) = (0, 1), (1, 0),
      #    (1, 1) for ky = 0, 1, 2  ->  a 2x2 convolution 64 -> 32 padded on the top / left only.
      w0, sh0 = self._fold('base.level0.0', 'base.level0.1')
      w0s = s2d_weights_3x3_s1(w0)
      l0 = TV(self._buf(H // 2, W // 2, 64), 0, 64)          # (level0 is below first_level: not an input of DLAUp)
      self._conv('base.level0', x0, w0s, sh0.repeat(4), l0, 3, 1)
      self.s2d_named.add('base.level0')
      self.algo_flops['base.level0'] = 2.0 * B * H * W * 16 * 9 * 16
      w1, sh1 = self._fold('base.level1.0', 'base.level1.1')
      w1s = s2d_weights_3x3_s2(w1)
      # level1's own output goes out space-to-depth as well ([B, H/4, W/4, (sy, sx, 32)]): level2 reads it through a 2x2
      # max-pool (= a max over the four channel groups) and a 3x3 stride-2 conv (= a 2x2 conv over 128 channels)
      l1 = TV(self._buf(H // 4, W // 4, 128), 0, 128)
      self._conv('base.level1', l0, w1s, sh1, l1, 2, 1, out_hw=(H // 2, W // 2), out_mode=L.CT_OUT_NHWC_S2D)
      self.s2d_named.add('base.level1')
      self.algo_flops['base.level1'] = 2.0 * B * (H // 2) * (W // 2) * 32 * 9 * 16

    # ---- level2: Tree(1, 32->64, s2, level_root=False) ----
    h2, w2 = H // 4, W // 4
    cat2 = self._buf(h2, w2, 128)
    bottom2 = TV(self._buf(h2, w2, 32), 0, 32)
    if s2d:
      self.ops.append(('pool_s2d', (l1, bottom2), 'maxpool'))
    else:
      self._maxpool(l1, bottom2)
    res2 = TV(self._buf(h2, w2, 64), 0, 64)
    self._conv_bn('base.level2.project', bottom2, 'base.level2.project.0', 'base.level2.project.1',
                  res2, 1, 1, relu=False)
    x1 = TV(cat2, 64, 64)
    x2 = TV(cat2, 0, 64)
    self._basic_block('base.level2.tree1', l1, x1, 2, res2, x_s2d=s2d)
    self._basic_block('base.level2.tree2', x1, x2, 1, x1)
    l2 = TV(self._buf(h2, w2, 64), 0, 64)
    self._conv_bn('base.level2', TV(cat2, 0, 128), 'base.level2.root.conv', 'base.level2.root.bn', l2, 1)

    # ---- level3 / level4: Tree(2, c->2c, s2, level_root=True) ----
    def tree_l2(p, x, cin, cout):
      oh, ow = x.H // 2, x.W // 2
      catb = self._buf(oh, ow, 3 * cout + cin)            # [x2'' | x1'' | bottom(cin) | T1(cout)]
      bottom = TV(catb, 2 * cout, cin)
      self._maxpool(x, bottom)
      # outer project is dead compute (hazard H4): skipped
      # tree1 = Tree(1, cin->cout, s2)
      cata = self._buf(oh, ow, 2 * cout)
      resa = TV(self._buf(oh, ow, cout), 0, cout)
      self._conv_bn(p + '.tree1.project', bottom, p + '.tree1.project.0', p + '.tree1.project.1',
                    resa, 1, 1, relu=False)
      x1a, x2a = TV(cata, cout, cout), TV(cata, 0, cout)
      self._basic_block(p + '.tree1.tree1', x, x1a, 2, resa)
      self._basic_block(p + '.tree1.tree2', x1a, x2a, 1, x1a)
      t1 = TV(catb, 2 * cout + cin, cout)
      self._conv_bn(p + '.tree1', TV(cata, 0, 2 * cout), p + '.tree1.root.conv',
                    p + '.tree1.root.bn', t1, 1)
      # tree2 = Tree(1, cout->cout, s1), children = [bottom, t1]
      x1b, x2b = TV(catb, cout, cout), TV(catb, 0, cout)
      self._basic_block(p + '.tree2.tree1', t1, x1b, 1, t1)
      self._basic_block(p + '.tree2.tree2', x1b, x2b, 1, x1b)
      out = TV(self._buf(oh, ow, cout), 0, cout)
      self._conv_bn(p, TV(catb, 0, 3 * cout + cin), p + '.tree2.root.conv', p + '.tree2.root.bn',
                    out, 1)
      return out

    l3 = tree_l2('base.level3', l2, 64, 128)
    l4 = tree_l2('base.level4', l3, 128, 256)

    # ---- level5: Tree(1, 256->512, s2, level_root=True) ----
    h5, w5 = H // 32, W // 32
    cat5 = self._buf(h5, w5, 1280)                          # [x2 | x1 | bottom(256)]
    bottom5 = TV(cat5, 1024, 256)
    self._maxpool(l4, bottom5)
    res5 = TV(self._buf(h5, w5, 512), 0, 512)
    self._conv_bn('base.level5.project', bottom5, 'base.level5.project.0', 'base.level5.project.1',
                  res5, 1, 1, relu=False)
    x1, x2 = TV(cat5, 512, 512), TV(cat5, 0, 512)
    self._basic_block('base.level5.tree1', l4, x1, 2, res5)
    self._basic_block('base.level5.tree2', x1, x2, 1, x1)
    l5 = TV(self._buf(h5, w5, 512), 0, 512)
    self._conv_bn('base.level5', TV(cat5, 0, 1280), 'base.level5.root.conv', 'base.level5.root.bn', l5, 1)

    # ---- DLAUp (dla.py:549-574): ida_0 (o=256), ida_1 (o=128), ida_2 (o=64) ----
    layers = [l0, l1, l2, l3, l4, l5]
    out = [layers[-1]]
    chans = [64, 128, 256, 512]
    for i in range(3):
      o = chans[-i - 2]
      self._ida('dla_up.ida_%d' % i, layers, len(layers) - i - 2, len(layers), o)
      out.insert(0, layers[-1])
    # ---- ida_up on [out0, out1, out2] (dla.py:635-638; the .clone() is unnecessary here because the
    # plan never writes in place) ----
    y = [out[0], out[1], out[2]]
    self._ida('ida_up', y, 0, 3, 64)
    feat = y[-1]
    self.named['feat'] = feat

    # ---- heads (base_model.py:14-65,86-90) ----
    oh, ow = H // 4, W // 4
    self.out_hw = (oh, ow)
    self.outputs = {}
    first = []   # heads with >=1 hidden conv: fuse their first convs
    for h in self.heads:
      n_layers = len([k for k in sd if k.startswith(h + '.') and k.endswith('.weight')])
      first.append((h, n_layers))
    fused = [h for h, n in first if n >= 2]
    mid_c = {h: sd[h + '.0.weight'].shape[0] for h in fused}
    ks = {sd[h + '.0.weight'].shape[2] for h in fused}
    assert len(ks) <= 1, 'heads with different first-conv kernel sizes are not supported'
    if fused:
      kh = ks.pop()
      wcat = torch.cat([sd[h + '.0.weight'] for h in fused], 0)
      bcat = torch.cat([sd[h + '.0.bias'] for h in fused], 0)
      mid = self._buf(oh, ow, wcat.shape[0])
      self._conv('heads.0', feat, wcat, bcat, TV(mid, 0, wcat.shape[0]), kh, 1, relu=True)
    off = 0
    for h, n_layers in first:
      classes = self.heads[h]
      o = torch.empty((B, classes, oh, ow), dtype=f32, device=self.device)
      self.outputs[h] = o
      if n_layers >= 2:
        cur = TV(mid, off, mid_c[h])
        off += mid_c[h]
        idx = 2
        for _ in range(n_layers - 2):      # extra hidden 1x1 convs (num_head_conv > 1)
          wgt = sd['%s.%d.weight' % (h, idx)]
          nxt = TV(self._buf(oh, ow, wgt.shape[0]), 0, wgt.shape[0])
          self._conv('%s.%d' % (h, idx), cur, wgt, sd['%s.%d.bias' % (h, idx)], nxt, 1, 1, relu=True)
          cur = nxt
          idx += 2
        wgt, bias = sd['%s.%d.weight' % (h, idx)], sd['%s.%d.bias' % (h, idx)]
      else:
        cur = feat
        wgt, bias = sd[h + '.weight'], sd[h + '.bias']
      d = self._conv(h, cur, wgt, bias, o, wgt.shape[2], 1, relu=False, out_mode=L.CT_OUT_NCHW_F32)
      self.head_descs[h] = d
    self.set_fused_activations(False)

  # ------------------------------------------------------------------ run
  def set_fused_activations(self, on):
    """on=True: hm/hm_hp sigmoid and the dep transform (detector.py:300-308) run in the head epilogue."""
    for h, d in self.head_descs.items():
      act = L.CT_HEAD_NONE
      if on and h in ('hm', 'hm_hp'):
        act = L.CT_HEAD_SIGMOID
      elif on and h == 'dep':
        act = L.CT_HEAD_DEPTH
      d.head_act = act
    self.fused_act = on
    self.graph = None

  def _run_one(self, kind, pl, name, img_ptr, pre_ptr, hm_ptr, st):
    lib = self.lib
    if kind == 'conv':
      if pl.epilogue_sum3:          # stem: which of (img, pre_img, pre_hm) exist this call (dla.py:308-311)
        pl.epilogue_sum3 = 1 | (2 if pre_ptr.value else 0) | (4 if hm_ptr.value else 0)
      elif name == 'stem48':
        pl.shift = self.stem48_shift[1 | (2 if pre_ptr.value else 0) | (4 if hm_ptr.value else 0)].data_ptr()
      rc = lib.ct_conv_forward(C.byref(pl), st)
    elif kind == 'stem':
      rc = lib.ct_stem_forward(img_ptr, pre_ptr, hm_ptr, L.ptr(self.stem_w), L.ptr(self.stem_shift),
                               C.c_void_p(pl.ptr), self.ct_dtype, self.B, self.H, self.W, pl.ld, st)
    elif kind == 'pack':
      rc = lib.ct_pack_stem_input(img_ptr, pre_ptr, hm_ptr, C.c_void_p(pl.ptr), self.B, self.H, self.W, st)
    elif kind == 'pack32':
      rc = lib.ct_pack_stem_input_f32(img_ptr, pre_ptr, hm_ptr, C.c_void_p(pl.ptr), self.B, self.H, self.W, st)
    elif kind == 'pool_s2d':
      x, o = pl
      rc = lib.ct_maxpool2_s2d(C.c_void_p(x.ptr), C.c_void_p(o.ptr), self.ct_dtype, self.B, x.H, x.W, o.C, x.ld, o.ld, st)
    elif kind == 'pool':
      x, o = pl
      rc = lib.ct_maxpool2(C.c_void_p(x.ptr), C.c_void_p(o.ptr), self.ct_dtype, self.B, x.H, x.W, x.C,
                           x.ld, o.ld, st)
    else:
      x, skip, w, o, f = pl
      rc = lib.ct_upsample_add(C.c_void_p(x.ptr), C.c_void_p(skip.ptr), L.ptr(w), C.c_void_p(o.ptr),
                               self.ct_dtype, self.B, x.H, x.W, x.C, f, x.ld, skip.ld, o.ld, st)
    if rc != 0:
      L.check(rc, '%s (%s)' % (kind, name))
    if self.debug_sync:                  # CTB_DEBUG_SYNC=1: attribute an asynchronous kernel fault to its layer
      try:
        torch.cuda.synchronize()
      except Exception as e:
        raise RuntimeError('kernel fault in op %s (%s): %s' % (kind, name, e))

  def _run_ops(self, img_ptr, pre_ptr, hm_ptr):
    st = L.stream_ptr()
    for kind, pl, name in self.ops:
      self._run_one(kind, pl, name, img_ptr, pre_ptr, hm_ptr, st)

  @property
  def n_launches(self):
    return len(self.ops)

  def forward(self, images, pre_images=None, pre_hms=None):
    """images/pre_images [B,3,H,W], pre_hms [B,1,H,W]: fp32 CUDA NCHW contiguous.
    Returns {head: fp32 [B,c,H/4,W/4]} (buffers owned by the engine, overwritten by the next call)."""
    for t in (images, pre_images, pre_hms):
      if t is not None:
        assert t.is_cuda and t.dtype == torch.float32 and t.is_contiguous(), 'fp32 contiguous CUDA input'
    assert tuple(images.shape) == (self.B, 3, self.H, self.W), (images.shape, self.B, self.H, self.W)
    pre = pre_images if self.has_pre_img else None
    hm = pre_hms if self.has_pre_hm else None
    self._run_ops(L.ptr(images), L.ptr(pre), L.ptr(hm))
    return self.outputs

  # CUDA-graph replay: inputs are first copied into the engine's static buffers
  def capture(self):
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
      for _ in range(2):
        self._run_ops(L.ptr(self.in_img), L.ptr(self.in_pre if self.has_pre_img else None),
                      L.ptr(self.in_hm if self.has_pre_hm else None))
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
      self._run_ops(L.ptr(self.in_img), L.ptr(self.in_pre if self.has_pre_img else None),
                    L.ptr(self.in_hm if self.has_pre_hm else None))
    self.graph = g
    return g

  def replay(self):
    if self.graph is None:
      self.capture()
    self.graph.replay()
    return self.outputs

  def stage(self, name):
    """NCHW fp32 copy of a named intermediate (parity tests)."""
    t = self.named[name].tensor()
    if name in self.s2d_named:                            # stored space-to-depth (see _build)
      B, h, w, _ = t.shape
      c = t.shape[-1] // 4
      return t.reshape(B, h, w, 2, 2, c).permute(0, 5, 1, 3, 2, 4).reshape(B, c, 2 * h, 2 * w).float().contiguous()
    return t.permute(0, 3, 1, 2).float().contiguous()
