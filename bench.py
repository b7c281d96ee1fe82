#!/usr/bin/env python
"""bench.py -- CenterTrack per-frame inference hot path on B200 (contract: see DESIGN.md section 6).

  python bench.py --gpus N --steps K --warmup W [--batch B] [--config CFG] [--precision P] [--impl reference]
                   [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (default = BASELINE.json configs[1]): DLA-34 coco_tracking, 512x512, bf16, synthetic frame pairs, K=100.
--config mot | nuscenes_ddd | coco_pose selects BASELINE configs 3-5 (960x544 / 800x448 / 512x512 pose heads).
One step = the hot path over one batch of B frames (B independent streams) per GPU:
    prior heat-map splat from the streams' tracks -> DLA-34 + DCNv2 neck + heads (+ fused sigmoid) -> fused decode
    (NMS + top-K + gathers) -> greedy displacement association,   all on the device, one CUDA graph.
metric = frames/sec, whole job.  Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np
import torch

K = 100
# name -> (H, W, algorithmic GFLOP per frame (SURVEY 8d / BASELINE.md section 2), BASELINE.json config index)
CONFIGS = {'coco_tracking': (512, 512, 72.56, 1), 'mot': (544, 960, 143.23, 2),
           'nuscenes_ddd': (448, 800, 124.98, 3), 'coco_pose': (512, 512, 86.84, 4)}


def metric_name(cfg):
  H, W = CONFIGS[cfg][:2]
  return 'frames/sec (device-timed) DLA-34 %dx%d' % (W, H) if cfg != 'coco_tracking' else \
      'frames/sec (device-timed) DLA-34 512x512'


def workload_name(cfg):
  H, W, _, idx = CONFIGS[cfg]
  return 'DLA-34 %s %dx%d frame pairs + pre_hm, K=%d (BASELINE configs[%d])' % (cfg, W, H, K, idx)


def _peaks():
  p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
  if os.path.exists(p):
    d = json.load(open(p))
    return d.get('bf16_tflops_sustained', d.get('bf16_tflops')), d.get('hbm_gbs'), 'measured'
  return 1400.0, 6650.0, 'fallback'


class ClockSampler(threading.Thread):
  """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
  Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,'
       'clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
       'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

  def __init__(self, gpu):
    super().__init__(daemon=True)
    self.gpu, self.rows, self.stop_flag = gpu, [], False
    # NVML is set up HERE, before the timed region (import + nvmlInit take longer than a 0.2 s timed region on a cold
    # box); the thread then takes a sample every ~5 ms.  nvidia-smi (0.1 s per call) is the fall-back.
    self.nv = self.h = None
    try:
      import pynvml as nv
      nv.nvmlInit()
      try:
        h = nv.nvmlDeviceGetHandleByUUID('GPU-' + str(torch.cuda.get_device_properties(gpu).uuid))
      except Exception:
        h = nv.nvmlDeviceGetHandleByIndex(gpu)
      self.mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
      self.bits = (('hw_slowdown', nv.nvmlClocksEventReasonHwSlowdown), ('hw_thermal_slowdown', nv.nvmlClocksEventReasonHwThermalSlowdown),
                   ('sw_thermal_slowdown', nv.nvmlClocksEventReasonSwThermalSlowdown), ('sw_power_cap', nv.nvmlClocksEventReasonSwPowerCap))
      nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
      self.nv, self.h = nv, h
    except Exception:
      self.nv = self.h = None

  def _nvml(self):
    if self.nv is None:
      return False
    nv, h = self.nv, self.h
    while not self.stop_flag:
      try:
        sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
        try:
          r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
        except Exception:
          r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
        self.rows.append([str(self.gpu), str(sm), str(self.mx), '', ''] + ['Active' if r & b else 'Not Active' for _, b in self.bits])
      except Exception:
        pass
      time.sleep(0.005)
    return True

  def run(self):
    if self._nvml():
      return
    while not self.stop_flag:
      try:
        r = subprocess.run(['nvidia-smi', '-i', str(self.gpu), '--query-gpu=' + self.Q,
                            '--format=csv,noheader,nounits'], capture_output=True, text=True, timeout=5)
        if r.returncode == 0 and r.stdout.strip():
          self.rows.append([c.strip() for c in r.stdout.strip().split(',')])
      except Exception:
        pass
      time.sleep(0.1)

  def summary(self):
    self.stop_flag = True
    sm = [float(r[1]) for r in self.rows if r[1].replace('.', '').isdigit()]
    mx = [float(r[2]) for r in self.rows if r[2].replace('.', '').isdigit()]
    reasons = set()
    for r in self.rows:
      for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), r[5:9]):
        if v.lower().startswith('active'):
          reasons.add(name)
    return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
            'reasons': sorted(reasons), 'samples': len(self.rows)}


def _use_host_threads():
  """torch's own default thread count is kept (64 on the GPU box: oversubscribing its logical CPUs made the oracle
  several times slower); only when a launcher pinned it to one thread (torchrun exports OMP_NUM_THREADS=1) is it
  raised, to half the logical CPUs (= physical cores on an SMT-2 host).  CTB_CPU_THREADS overrides."""
  n = int(os.environ.get('CTB_CPU_THREADS', '0'))
  if n <= 0 and torch.get_num_threads() <= 1:
    n = max(1, (os.cpu_count() or 2) // 2)
  if n > 0:
    torch.set_num_threads(n)


def _oracle_step(cfg, n_frames=1, budget_s=None):
  """The CPU restatement of the reference path (oracle/), timed on this host: network + sigmoid + decode +
  post-process + greedy association for up to n_frames frame pairs of the config's size (stops early once budget_s
  seconds have elapsed).  Returns (seconds, threads, frames done)."""
  sys.path.insert(0, os.path.join(ROOT, 'oracle'))
  sys.path.insert(0, os.path.join(ROOT, 'tests'))
  import ct_oracle as co
  from centertrack_b200 import synthetic as wt
  from helpers import make_model
  H, W = CONFIGS[cfg][:2]
  opt, model, sd = make_model(cfg)
  orc = co.DLA34Oracle(sd, opt.heads)
  trk = co.TrackerOracle(opt.new_thresh)
  trk.init_track([])
  img, pre, hm = wt.synthetic_inputs(1, H, W)
  c = np.array([W / 2., H / 2.], np.float32)
  done = 0
  t0 = time.perf_counter()
  for _ in range(n_frames):
    out = co.sigmoid_output(orc.forward(img, pre, hm))
    dets = {k: v for k, v in co.generic_decode(out, K).items() if not k.startswith('_')}
    if 'dep' not in dets:                                   # ddd post-process needs calibration: association only for 2-D
      res = co.generic_post_process(dets, [c], [max(H, W) * 1.0], H // 4, W // 4, opt.out_thresh)[0]
      trk.step([r for r in res if r['score'] > opt.out_thresh])
    done += 1
    if budget_s is not None and time.perf_counter() - t0 > budget_s:
      break
  return time.perf_counter() - t0, torch.get_num_threads(), done


def run_reference(args, rank, world):
  """--impl reference: the reference's CPU implementation of the path (oracle port; the Python
  reference itself cannot travel to the GPU box) on all host threads.  Rank 0 only."""
  if rank != 0:
    return
  _use_host_threads()
  frames_per_step = 1
  for _ in range(min(args.warmup, 1)):
    _oracle_step(args.config, 1)
  t, thr = 0.0, 1
  steps = args.steps
  for _ in range(steps):
    dt, thr, _n = _oracle_step(args.config, frames_per_step)
    t += dt
  fps = steps * frames_per_step / t
  line = {'impl': 'reference', 'metric': metric_name(args.config), 'value': fps, 'unit': 'frames/s', 'n_gpus': args.gpus,
          'steps': steps, 'warmup': min(args.warmup, 1), 'ms_per_step': 1000 * t / steps,
          'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32',
          'data': 'synthetic',
          'config': {'workload': workload_name(args.config), 'frames_per_step': frames_per_step},
          'cpu_baseline': {'value': fps, 'unit': 'frames/s', 'cores': thr, 'kind': 'port',
                           'sample': '%d steps x %d frame (oracle/ct_oracle.py: torch-CPU fp32 convs + '
                                     'restated DCNv2/decode/association)' % (steps, frames_per_step)},
          'e2e': {'value': fps, 'unit': 'frames/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
  _emit(line)


_REAL_STDOUT = None


def _emit(line):
  data = (json.dumps(line) + '\n').encode()
  if _REAL_STDOUT is None:
    sys.stdout.write(data.decode())
    sys.stdout.flush()
  else:
    sys.stdout.flush()
    os.write(_REAL_STDOUT, data)


# ------------------------------------------------------------------------------------------------------------------
# per-kernel time inside the step (roofline shares)
# ------------------------------------------------------------------------------------------------------------------
def _op_flops(kind, pl, L, name=None, eng=None):
  """ALGORITHMIC flops of the reference layer the launch implements (layers run on a space-to-depth view carry
  structural zeros in their weights: those MACs are not counted)."""
  if kind != 'conv':
    return 0.0
  algo = getattr(eng, 'algo_flops', {}).get(name)
  if algo is not None:
    return float(algo)
  if pl.epilogue_sum3:
    return 2.0 * pl.B * pl.OH * pl.OW * 16 * 49 * 7            # the three stems: 16 x (3+3+1) x 7x7 MACs/pixel
  return 2.0 * pl.B * pl.OH * pl.OW * pl.C_out * pl.KH * pl.KW * pl.C_in


def _op_group(kind, pl, L):
  if kind != 'conv':
    return kind
  if pl.a_mode in (L.CT_A_DCN, L.CT_A_DCN_WIN):
    # window DCN with one N tile of <= 128 channels runs the persistent kernel (conv_tc.cu conv_forward_tc, CTB_DCN_PERSIST)
    persist = pl.a_mode == L.CT_A_DCN_WIN and pl.C_out <= 128 and os.environ.get('CTB_DCN_PERSIST', '1') != '0'
    return 'dcn_persist' if persist else 'dcn_tc'
  return {L.CT_ENGINE_TCGEN05: 'conv_tc', L.CT_ENGINE_TCGEN05_HALO: 'conv_halo', L.CT_ENGINE_SIMT: 'conv_simt',
          L.CT_ENGINE_TCGEN05_X3: 'conv_tc'}[pl.engine]


def per_op_times(runner, L, reps=5):
  """Per-launch device time of one step IN ITS REAL ORDER AND CACHE STATE: the step is captured once more into a CUDA
  graph with an (external, timing) event-record node after every launch; consecutive differences over `reps` replays.
  Falls back to the CUPTI kernel records of torch.profiler, then to one event pair per eager launch.
  -> (method, [ms per op of eng.ops], decode_ms, tracker_ms or None)"""
  eng = runner.eng
  n = len(eng.ops)
  slot = 1
  img, pre, hm = runner.img[slot], runner.img[(slot - 1) % 3], runner.hm[slot]
  img_p, pre_p, hm_p = L.ptr(img), L.ptr(pre if eng.has_pre_img else None), L.ptr(hm if eng.has_pre_hm else None)
  from centertrack_b200.decode import generic_decode

  def run_marked(marks):
    k = 0
    marks[k].record(); k += 1
    if runner.tracker is not None:
      runner.tracker.render(hm)
    marks[k].record(); k += 1
    st = L.stream_ptr()
    for kind, pl, name in eng.ops:
      eng._run_one(kind, pl, name, img_p, pre_p, hm_p, st)
      marks[k].record(); k += 1
    generic_decode(dict(eng.outputs), K=runner.K, records_out=runner.rec, workspace=runner.ws)
    marks[k].record(); k += 1
    if runner.tracker is not None:
      runner.tracker.step(runner.rec)
    marks[k].record(); k += 1

  def collect(marks):
    d = [marks[i].elapsed_time(marks[i + 1]) for i in range(len(marks) - 1)]
    return d[1:1 + n], d[1 + n], (d[0] + d[2 + n]) if runner.tracker is not None else None

  n_marks = n + 4
  try:
    marks = [torch.cuda.Event(enable_timing=True, external=True) for _ in range(n_marks)]
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
      run_marked([torch.cuda.Event(enable_timing=True) for _ in range(n_marks)])
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
      run_marked(marks)
    acc, dec, trk = np.zeros(n), 0.0, 0.0
    for _ in range(reps):
      g.replay()
      torch.cuda.synchronize()
      a, b, c = collect(marks)
      acc += np.array(a); dec += b; trk += (c or 0.0)
    return 'graph-event-nodes', list(acc / reps), dec / reps, (trk / reps if runner.tracker is not None else None)
  except Exception as e:                                      # noqa: BLE001
    sys.stderr.write('per_op_times: graph event nodes unavailable (%s); eager event pairs\n' % (e,))
  acc, dec, trk = np.zeros(n), 0.0, 0.0
  for _ in range(reps):
    marks = [torch.cuda.Event(enable_timing=True) for _ in range(n_marks)]
    run_marked(marks)
    torch.cuda.synchronize()
    a, b, c = collect(marks)
    acc += np.array(a); dec += b; trk += (c or 0.0)
  return 'eager-event-pairs', list(acc / reps), dec / reps, (trk / reps if runner.tracker is not None else None)


def parity_at_bench_shape(runner, cfg, B, H, W, precision, wt):
  """The engine that was just timed, at the shape it was timed at, against the reference's fp32 outputs
  (tests/golden/e2e_*.npz): errors of frames 0 and B-1 of a seeded batch (tests/parity.py metrics)."""
  sys.path.insert(0, os.path.join(ROOT, 'tests'))
  import parity as P
  gold = os.path.join(ROOT, 'tests', 'golden')
  if cfg == 'coco_tracking' and B == 32:
    cases = [('e2e_coco_tracking_512_b32f0', 0), ('e2e_coco_tracking_512_b32f31', 31)]
    seed, batch = 4242, 32
  else:
    stem = {'coco_tracking': 'e2e_coco_tracking_512', 'mot': 'e2e_mot_544x960', 'coco_pose': 'e2e_coco_pose_512'}.get(cfg)
    if stem is None:
      return None
    cases, seed, batch = [(stem, 0)], 317, 1
  img, pre, hm = wt.synthetic_inputs(batch, H, W, seed=seed)
  if batch < B:                                              # frame 0 is the golden's frame; the rest of the batch is filler
    rep = lambda t: t.expand(B, *t.shape[1:]).contiguous()
    img, pre, hm = rep(img), rep(pre), rep(hm)
  eng = runner.eng
  dev = runner.device
  from centertrack_b200.decode import generic_decode
  out = dict(eng.forward(img.to(dev), pre.to(dev), hm.to(dev)))
  dets = generic_decode(out, K=K, workspace=runner.ws)
  torch.cuda.synchronize(dev)
  d = {k: dets[k].cpu().numpy() for k in ('clses', 'xs', 'ys')}
  res = {'engine': precision, 'against': 'reference fp32 outputs, tests/golden (oracle/gen_golden.py)', 'frames': {}}
  worst = {}
  for stem, frame in cases:
    g = np.load(os.path.join(gold, stem + '.npz'))
    m = P.summarize(P.head_metrics(out, g, frame), P.peak_metrics(out, d, g, frame), P.stage_metrics(eng.stage, g, frame))
    res['frames'][stem] = m
    for k in ('score_max', 'bbox_max', 'tracking_max'):
      if k in m:
        worst[k] = max(worst.get(k, 0.0), m[k])
    worst['head_max'] = max(worst.get('head_max', 0.0), max(m['head_max'].values()))
    worst['stage_max'] = max(worst.get('stage_max', 0.0), max(m['stage_max'].values()))
    worst['topk_overlap'] = min(worst.get('topk_overlap', 1.0), m['topk_overlap'])
  res['worst'] = worst
  return res


def accurate_engine_leg(model, cfg, B, H, W, opt, dev, tracking, host_img, host_hm, wt, steps=8, warmup=3):
  """The same step on the tensor-core engine that meets north_star's 1e-3 (bf16x3: fp32 activations, bf16 hi/lo split
  operands), device-resident timing + its parity at this shape, so that ONE bench line says "Y frames/s at the bf16
  format's error, X frames/s within 1e-3 of the reference".  Runs after every headline measurement; a failure here is
  reported in the key and cannot touch the numbers above it."""
  from centertrack_b200.runner import NS, StreamRunner
  r = StreamRunner(model, B, H, W, K=K, precision='bf16x3', device=dev, opt=opt, device_tracking=tracking)
  for s in range(NS):
    r.load_device_inputs(host_img[s & 1].to(dev), host_hm[s & 1].to(dev), s)
  r.warm()
  for _ in range(warmup):
    r.step_device()
  torch.cuda.synchronize(dev)
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  e0.record()
  for _ in range(steps):
    r.step_device()
  e1.record()
  torch.cuda.synchronize(dev)
  ms = e0.elapsed_time(e1) / steps
  par = parity_at_bench_shape(r, cfg, B, H, W, 'bf16x3', wt)
  return {'engine': 'bf16x3', 'value': B / (ms / 1000.0), 'unit': 'frames/s', 'ms_per_step': ms, 'steps': steps,
          'warmup': warmup, 'what': 'same step (splat + network + decode + association, one CUDA graph, inputs resident) '
          'on the tcgen05 engine with bf16 hi/lo split operands and fp32 activations',
          'parity_worst': par['worst'] if par else None, 'tolerance': 'north_star: fp32 heat-maps / offsets within 1e-3'}


def stock_pytorch_leg(sd, heads, B, H, W, dev, wt, steps=3, warmup=2):
  """Context, not a target: the same graph through STOCK PyTorch on the same device -- cuDNN convolutions,
  torchvision.ops.deform_conv2d (the im2col + GEMM design of the DCNv2 op the reference calls, dla.py:513), ATen
  max_pool2d / topk for the decode's NMS and its two top-Ks (model/utils.py:52-87) -- eager, as the reference runs.
  The network is the oracle's functional restatement with its tensors moved to the device (the Python reference
  itself cannot travel to the GPU box); like `cpu_baseline` it is a reported baseline (kind "port"), run after every
  headline measurement."""
  import contextlib
  import torch.nn.functional as F
  from torchvision.ops import deform_conv2d
  sys.path.insert(0, os.path.join(ROOT, 'oracle'))
  import ct_oracle as co

  def dcn(x, w, b, wo, bo):
    o1, o2, m = torch.chunk(F.conv2d(x, wo, bo, 1, 1), 3, 1)
    return deform_conv2d(x, torch.cat((o1, o2), 1).float(), w, b, 1, 1, 1, torch.sigmoid(m).float())

  orc = co.DLA34Oracle(sd, heads, dcn_fn=dcn)
  orc.sd = {k: v.to(dev) for k, v in orc.sd.items()}
  img, pre, hm = wt.synthetic_inputs(1, H, W, seed=317)
  rep = lambda t: t.expand(B, *t.shape[1:]).contiguous().to(dev)
  img, pre, hm = rep(img), rep(pre), rep(hm)
  cuda = torch.device(dev).type == 'cuda'

  def step():
    out = orc.forward(img, pre, hm)
    heat = torch.sigmoid(out['hm'].float())
    heat = heat * (F.max_pool2d(heat, 3, 1, 1) == heat).float()
    b, c = heat.shape[:2]
    sc, _ = torch.topk(heat.view(b, c, -1), K)
    return torch.topk(sc.view(b, -1), K)[0]

  res = {'kind': 'port', 'frames_per_step': B, 'steps': steps, 'warmup': warmup, 'unit': 'frames/s',
         'what': 'oracle network restatement on the device through stock PyTorch (cuDNN, torchvision deform_conv2d) + '
                 'ATen NMS / top-K, eager; no association',
         'cudnn_allow_tf32': bool(torch.backends.cudnn.allow_tf32)}
  for name, ctx in (('fp32', contextlib.nullcontext),
                    ('bf16_autocast', lambda: torch.autocast(torch.device(dev).type, dtype=torch.bfloat16))):
    with torch.no_grad(), ctx():
      for _ in range(warmup):
        step()
      if cuda:
        torch.cuda.synchronize(dev)
      t0 = time.perf_counter()
      for _ in range(steps):
        step()
      if cuda:
        torch.cuda.synchronize(dev)
      dt = time.perf_counter() - t0
    res[name] = B * steps / dt
  return res


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, runner):
  """What a caller of StreamRunner.step_device holds after the last timed step, as DIR/<name>.npy: the packed decode
  records [B,K,F] and, with device tracking, the track table [B,T,CT_TRK_FLOATS] and the per-stream counts [B,2]."""
  arrays = {'records': runner.rec.cpu().numpy()}
  if runner.tracker is not None:
    arrays['tracks'] = runner.tracker.tracks.cpu().numpy()
    arrays['track_counts'] = runner.tracker.counts.cpu().numpy().astype(np.float64)
  total = sum(a.nbytes for a in arrays.values())
  assert total <= DUMP_LIMIT_BYTES, 'output dump of %d bytes exceeds %d' % (total, DUMP_LIMIT_BYTES)
  os.makedirs(out_dir, exist_ok=True)
  for name, a in arrays.items():
    np.save(os.path.join(out_dir, name + '.npy'), a)


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument('--gpus', type=int, default=1)
  ap.add_argument('--steps', type=int, default=30)
  ap.add_argument('--warmup', type=int, default=5)
  ap.add_argument('--batch', type=int, default=32, help='frames (independent streams) per GPU per step')
  ap.add_argument('--config', default='coco_tracking', choices=sorted(CONFIGS))
  ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
  ap.add_argument('--precision', default='bf16', choices=['bf16', 'fp32', 'bf16x3'])
  ap.add_argument('--no-cpu-baseline', action='store_true')
  ap.add_argument('--no-parity', action='store_true')
  ap.add_argument('--no-latency', action='store_true')
  ap.add_argument('--no-gpu-baseline', action='store_true', help='skip the stock-PyTorch-on-the-same-GPU context leg')
  ap.add_argument('--no-accurate', action='store_true', help='skip the bf16x3 (<= 1e-3) engine leg of the default run')
  ap.add_argument('--host-tracking', action='store_true',
                  help='round-1 mode: pre_hm supplied by the host, no association on the device')
  ap.add_argument('--dump-outputs', metavar='DIR',
                  help='write the records and track tables of the last timed step to DIR/<name>.npy (inputs are seeded: '
                       'the same arguments give the same inputs, so two builds can be compared output for output)')
  args = ap.parse_args()
  if args.dump_outputs and args.impl != 'b200':
    ap.error('--dump-outputs dumps the device path (--impl b200)')
  # stdout carries exactly ONE JSON line: everything any library writes to fd 1 during the run (NCCL prints a version
  # banner there) is sent to stderr, and the result line goes to the saved descriptor (see _emit)
  global _REAL_STDOUT
  sys.stdout.flush()
  _REAL_STDOUT = os.dup(1)
  os.dup2(2, 1)
  args.warmup = max(args.warmup, 3)

  rank = int(os.environ.get('RANK', 0))
  world = int(os.environ.get('WORLD_SIZE', 1))
  local = int(os.environ.get('LOCAL_RANK', 0))
  if args.impl == 'reference':
    return run_reference(args, rank, world)

  torch.cuda.set_device(local)
  dev = torch.device('cuda', local)
  dist = None
  if world > 1:
    import torch.distributed as dist
    dist.init_process_group('nccl', device_id=dev)

  sys.path.insert(0, os.path.join(ROOT, 'oracle'))
  sys.path.insert(0, os.path.join(ROOT, 'tests'))
  from centertrack_b200 import synthetic as wt
  from helpers import make_model
  from centertrack_b200 import _lib as L
  from centertrack_b200.runner import NS, StreamRunner

  cfg = args.config
  H, W, gflop_per_frame, _ = CONFIGS[cfg]
  B = args.batch
  opt, model, sd = make_model(cfg)
  model = model.to(dev)
  tracking = not args.host_tracking
  runner = StreamRunner(model, B, H, W, K=K, precision=args.precision, device=dev, opt=opt, device_tracking=tracking)
  # synthetic inputs: 2 distinct frames per stream (+ pre_hm in host-tracking mode); inputs alone are 2 x B x 3-4 MB
  # and one step streams ~0.3 GB of activations per frame, so nothing but the 40 MB of weights can live in the 126 MB L2
  img, pre, hm = wt.synthetic_inputs(2, H, W, seed=317 + rank)
  g = torch.Generator().manual_seed(rank)
  host_img = [(img[s:s + 1] + 0.05 * torch.randn(B, 3, H, W, generator=g)).pin_memory() for s in range(2)]
  host_hm = [hm[s:s + 1].expand(B, 1, H, W).contiguous().pin_memory() for s in range(2)]
  for s in range(NS):
    runner.load_device_inputs(host_img[s & 1].to(dev), host_hm[s & 1].to(dev), s)
  runner.warm()

  def barrier():
    if dist is not None:
      dist.barrier()
    torch.cuda.synchronize(dev)

  gather_src = runner.tracker.tracks if tracking else runner.rec
  gathered = torch.empty((world * B,) + tuple(gather_src.shape[1:]), device=dev) if world > 1 else None

  # ---------------- device-resident timing (value) ----------------
  def dev_step():
    runner.step_device()
    if gathered is not None:               # the one collective of the path: fixed-size result gather
      dist.all_gather_into_tensor(gathered, gather_src)

  sampler = ClockSampler(local) if rank == 0 else None      # NVML set up before the warm-up, sampling starts after it
  for _ in range(args.warmup):
    dev_step()
  barrier()
  if rank == 0:
    sampler.start()
  e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
  e0.record()
  for _ in range(args.steps):
    dev_step()
  e1.record()
  barrier()
  ms = e0.elapsed_time(e1)
  if dist is not None:
    t = torch.tensor([ms], device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
  clocks = sampler.summary() if rank == 0 else None
  if args.dump_outputs and rank == 0:
    dump_outputs(args.dump_outputs, runner)
  ms_per_step = ms / args.steps
  value = world * B * args.steps / (ms / 1000.0)

  # ---------------- end-to-end timing (host frames in, host records + tracks out) ----------------
  def host_step(i):
    if tracking:
      runner.step_host(host_img[i & 1])
    else:
      runner.step_host(host_img[i & 1], host_hm[i & 1])

  for i in range(args.warmup):
    host_step(i)
  runner.fetch()
  barrier()
  t0 = time.perf_counter()
  for i in range(args.steps):
    host_step(i)
  rec_last = runner.fetch()
  n_tracks_last = int(runner.fetch_tracks()[1][:, 0].sum()) if tracking else None
  barrier()
  e2e_s = time.perf_counter() - t0
  if dist is not None:
    t = torch.tensor([e2e_s], device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_s = float(t.item())
  e2e = world * B * args.steps / e2e_s

  if rank != 0:
    if dist is not None:
      dist.destroy_process_group()
    return

  # ---------------- roofline: per-kernel time inside the step, measured live ----------------
  # `traffic`: dram__bytes_read.sum + dram__bytes_write.sum from the committed ncu --set full capture of one step at
  # 32 frames/step (profiles/), scaled by frames per step; null for configs without a capture.
  eng = runner.eng
  method, op_ms, decode_ms, tracker_ms = per_op_times(runner, L)
  raw_sum = sum(op_ms) + decode_ms + (tracker_ms or 0.0)
  rescaled = False
  if raw_sum > 1.05 * ms_per_step:          # the marked replay ran slower than the plain one (event nodes, eager launch
    f = ms_per_step / raw_sum               # gaps): attribute the excess proportionally so that the shares add up
    op_ms, decode_ms = [x * f for x in op_ms], decode_ms * f
    tracker_ms = tracker_ms * f if tracker_ms is not None else None
    rescaled = True
  groups = {}
  for (kind, pl, name), dt in zip(eng.ops, op_ms):
    gname = _op_group(kind, pl, L)
    gr = groups.setdefault(gname, {'ms': 0.0, 'flop': 0.0, 'launches': 0})
    gr['ms'] += dt
    gr['flop'] += _op_flops(kind, pl, L, name, eng)
    gr['launches'] += 1
  sum_ms = sum(op_ms) + decode_ms + (tracker_ms or 0.0)
  peak_tf, peak_hbm, peak_src = _peaks()
  traffic_per_frame = {}
  tp = os.path.join(ROOT, 'profiles', 'traffic.json')
  if os.path.exists(tp):
    traffic_per_frame = json.load(open(tp)).get(cfg if args.precision == 'bf16' else '', {})

  def merged(keys):
    ms = sum(groups.get(k, {'ms': 0.0})['ms'] for k in keys)
    fl = sum(groups.get(k, {'flop': 0.0})['flop'] for k in keys)
    n = sum(groups.get(k, {'launches': 0})['launches'] for k in keys)
    tr = [traffic_per_frame.get({'conv_tc': 'conv_tc_plain'}.get(k, k)) for k in keys if groups.get(k)]
    if ms <= 0:
      return None
    ach = fl / (ms / 1000.0) / 1e12
    return {'bound': 'tensor', 'achieved': ach, 'peak': peak_tf, 'unit': 'TFLOP/s', 'frac': ach / peak_tf if peak_tf else None,
            'traffic': (sum(tr) * B) if tr and all(t is not None for t in tr) else None, 'ms_per_step': round(ms, 4),
            'share_of_step': ms / sum_ms, 'gflop_per_step': fl / 1e9, 'launches': n}

  # one entry per kernel FUNCTION; the headline is the function with the largest share of the step
  fn = {'conv_halo_kernel': merged(['conv_halo']), 'dcn_persist_kernel': merged(['dcn_persist']),
        'conv_tc_kernel': merged(['dcn_tc', 'conv_tc']), 'conv_simt_kernel': merged(['conv_simt'])}
  fn = {k: v for k, v in fn.items() if v}
  dcn = merged(['dcn_persist', 'dcn_tc'])                   # all 16 DCNv2 main launches, whichever kernel ran them
  tc = merged(['conv_tc'])                                  # plain gather launches of conv_tc_kernel
  halo = fn.get('conv_halo_kernel')
  simt = fn.get('conv_simt_kernel')
  hm_bytes = float(eng.outputs['hm'].numel() * 4 + (eng.outputs['hm_hp'].numel() * 4 if 'hm_hp' in eng.outputs else 0))
  dec_gbs = hm_bytes / (decode_ms * 1e-3) / 1e9 if decode_ms > 0 else 0.0
  top = max(fn, key=lambda k: fn[k]['ms_per_step'])
  roofline = dict(fn[top])
  roofline['kernel'] = '%s (%d launches of one step)' % (top, roofline.pop('launches'))
  roofline.update({
      'traffic_unit': 'bytes per step (all launches of the kernel), ncu capture at 32 frames/step scaled',
      'peak_source': peak_src, 'method': method,
      'kernels': dict(fn, dcn_main=dcn, conv_tc_plain=tc),
      'ms_by_group': {k: round(v['ms'], 4) for k, v in groups.items()},
      'top_ops_us': [[n, round(t * 1000, 1)] for t, n in sorted(((dt, name) for (kind, pl, name), dt in zip(eng.ops, op_ms)),
                                                             reverse=True)[:24]],
      'sum_kernel_ms': round(raw_sum, 4), 'ms_per_step': round(ms_per_step, 4),
      'sum_over_step': raw_sum / ms_per_step, 'rescaled_to_step': rescaled,
      'decode': {'us_per_launch': round(decode_ms * 1000, 1), 'frames': B, 'bound': 'hbm', 'achieved': dec_gbs,
                 'peak': peak_hbm, 'unit': 'GB/s', 'frac': dec_gbs / peak_hbm if peak_hbm else None},
      'whole_step_tflops': gflop_per_frame * B / ms_per_step,
      'whole_step_frac': gflop_per_frame * B / ms_per_step / peak_tf if peak_tf else None})
  if os.environ.get('CTB_BENCH_OPS_FILE'):                   # every op with its engine group, for tools / DESIGN tables
    with open(os.environ['CTB_BENCH_OPS_FILE'], 'w') as f:
      json.dump([[name, kind, round(dt * 1000, 1)] for (kind, pl, name), dt in zip(eng.ops, op_ms)], f)
  assert sum_ms <= 1.05 * ms_per_step, 'per-kernel times (%.3f ms) do not add up to the step (%.3f ms)' % (sum_ms, ms_per_step)

  # ---------------- parity of the engine that was timed, at the timed shape ----------------
  parity = None
  if not args.no_parity:
    try:
      parity = parity_at_bench_shape(runner, cfg, B, H, W, args.precision, wt)
    except Exception as e:                                    # noqa: BLE001
      parity = {'error': repr(e)}

  # ---------------- per-image latency: Detector.process at B=1 (the reference's only published figure) ----------------
  latency = None
  if not args.no_latency:
    from centertrack_b200.detector import Detector
    det = Detector.__new__(Detector)
    opt1 = make_model(cfg, extra=['--b200_precision', args.precision])[0]
    det.opt, det.model = opt1, model
    model.precision = args.precision
    i1, p1, h1 = wt.synthetic_inputs(1, H, W, seed=5)
    i1, p1, h1 = i1.to(dev), p1.to(dev), h1.to(dev)
    for _ in range(5):
      det.process(i1, p1, h1, None)
    t0 = time.perf_counter()
    n_lat = 30
    for _ in range(n_lat):
      det.process(i1, p1, h1, None)
    lat_ms = (time.perf_counter() - t0) / n_lat * 1000.0
    latency = {'ms_per_image': round(lat_ms, 3), 'what': 'Detector.process, 1 frame pair + pre_hm, inputs on device, '
               'graph replay + fused decode + one D2H of the records; wall clock incl. both synchronisations',
               'reference_published_ms': 30.0, 'reference_published_on': 'Titan Xp (BASELINE.md)'}

  # ---------------- the <= 1e-3 tensor-core engine on the same step (N=1, default precision only) ----------------
  accurate = None
  if args.precision == 'bf16' and world == 1 and not args.no_accurate:
    try:
      accurate = accurate_engine_leg(model, cfg, B, H, W, opt, dev, tracking, host_img, host_hm, wt)
    except Exception as e:                                    # noqa: BLE001
      accurate = {'engine': 'bf16x3', 'error': repr(e)}

  # ---------------- context: the same graph through stock PyTorch / cuDNN on this GPU (N=1 only) ----------------
  gpu_base = None
  if world == 1 and not args.no_gpu_baseline:
    try:
      gpu_base = stock_pytorch_leg(sd, opt.heads, B, H, W, dev, wt)
      torch.cuda.empty_cache()
    except Exception as e:                                    # noqa: BLE001
      gpu_base = {'kind': 'port', 'error': repr(e)}

  cpu = None
  if not args.no_cpu_baseline and world == 1:       # rank 0 at N=1 only
    _use_host_threads()
    _oracle_step(cfg, 1)                                # warm-up (oneDNN primitive caches)
    dt, thr, n = _oracle_step(cfg, 10, budget_s=15.0)   # ~10-15 s of wall clock on the box's host threads
    cpu = {'value': n / dt, 'unit': 'frames/s', 'cores': thr, 'kind': 'port',
           'sample': '%d frames %dx%d (oracle/ct_oracle.py, torch-CPU fp32 + restated decode/association)' % (n, W, H)}

  line = {'metric': metric_name(cfg), 'value': value, 'unit': 'frames/s', 'n_gpus': world, 'steps': args.steps,
          'warmup': args.warmup, 'ms_per_step': ms_per_step, 'higher_is_better': True, 'scaling': 'weak',
          'vs_baseline': None, 'dtype': args.precision, 'data': 'synthetic',
          'config': {'workload': workload_name(cfg),
                     'frames_per_step_per_gpu': B, 'global_batch': B * world,
                     'parallelism': 'stream-sharded replicas x%d, NCCL all_gather of the result tables' % world,
                     'step': ('prior heat-map splat from device-resident tracks + network + decode + greedy association '
                              '(one CUDA graph)') if tracking else 'network + decode, pre_hm given (one CUDA graph)',
                     'l2': 'no flush: per-step inputs %.0f MB in 3 rotating slots + ~%.1f GB of activations per '
                           'step exceed the 126 MB L2' % (2 * B * 3 * H * W * 4 / 1e6, 0.29 * B * H * W / 262144.),
                     'cuda_graph': True},
          'e2e': {'value': e2e, 'unit': 'frames/s', 'h2d_bytes_per_step': runner.h2d_bytes_per_step,
                  'd2h_bytes_per_step': runner.d2h_bytes_per_step,
                  'what': 'pinned host frames -> H2D -> step -> D2H of records + track tables, every step, '
                          'reference dependency chain (pre_hm(t) from tracks(t-1)) kept on the device'},
          'gpu_launches': int(runner.launches_per_step * args.steps),
          'decode_us': round(decode_ms * 1000, 1),
          'tracker_us': round(tracker_ms * 1000, 1) if tracker_ms is not None else None,
          'clocks': clocks, 'roofline': roofline, 'parity': parity, 'accurate_engine': accurate, 'latency': latency,
          'gpu_baseline': gpu_base, 'cpu_baseline': cpu,
          'check': {'top_score_frame0': float(rec_last[0, 0, 0]), 'tracks_last_step': n_tracks_last}}
  _emit(line)
  if dist is not None:
    dist.destroy_process_group()


if __name__ == '__main__':
  main()
