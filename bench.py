#!/usr/bin/env python
"""Benchmark of the TAPIR hot path (DESIGN.md section 6).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A "step" is one full inference pass  get_feature_grids + get_query_features +
estimate_trajectories (+ the per-level mean of forward)  over one synthetic clip.

Headline (`value`, `e2e`): BASELINE.json configs[1] = 256x256x48 video, 256 query points per GPU;
with N GPUs the job is ONE clip tracked for 256*N query points (weak scaling in queries): backbone
frames are sharded, one NCCL all-gather of the feature grids, queries sharded, no collective in
the refinement loop.  metric = query-points x frames / second, whole job.

The same JSON line carries one sub-record per other BASELINE config, each timed with the same
rules (warm-up >= 3, CUDA events, max over ranks, L2 flushed between steps, own clocks window):
  sub_records.c4_strong  configs[3]  256x256x96, 4096 queries IN TOTAL shared by the ranks (strong)
  sub_records.c3_stream  configs[2]  causal model, 250 single-frame steps, 1024 points (N = 1 only)
  sub_records.c5_hires   configs[4]  1024x1024x64, 8192 queries, three refinement levels
and `roofline_named` holds the per-kernel roofline objects of the two kernels BASELINE.json's
north star names (global cost volume, local correlation) next to `roofline` (largest share).

--dump-outputs DIR writes what the last timed headline step returned as .npy files; inputs and
weights come from fixed seeds, so two builds run with the same arguments can be compared output
for output.
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
  sys.path.insert(0, ROOT)

import torch  # noqa: E402

UNIT = 'point-frames/s'

# name -> (frames, resolution, queries_per_gpu or None, total_queries or None, scaling, config name)
WORKLOADS = {
    'c2': dict(frames=48, res=256, q_per_gpu=256, q_total=None, scaling='weak',
               config='BASELINE.json configs[1]'),
    'c4': dict(frames=96, res=256, q_per_gpu=None, q_total=4096, scaling='strong',
               config='BASELINE.json configs[3]'),
    'c5': dict(frames=64, res=1024, q_per_gpu=None, q_total=8192, scaling='strong',
               config='BASELINE.json configs[4]'),
}
C3 = dict(frames=250, warm_frames=10, res=256, points=1024, config='BASELINE.json configs[2]')


def metric_name(wl):
  return (f"query-points x frames / sec (TAPIR inference, {wl['res']}x{wl['res']}x{wl['frames']}"
          + (f", {wl['q_total']} queries" if wl['q_total'] else '') + ')')


def _peaks():
  path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
  if os.path.exists(path):
    with open(path) as fh:
      d = json.load(fh)
    return dict(hbm=d['hbm_gbs'], tf_burst=d['bf16_tflops'], tf_sustained=d['bf16_tflops_sustained'],
                source='measured (MEASURED_PEAKS.json)')
  return dict(hbm=6650.0, tf_burst=1590.0, tf_sustained=1400.0, source='fallback (B200_PROFILING.md)')


# bf16 MMAs issued per fp32-equivalent product term under each precision policy (DESIGN.md 2)
_MMA_TERMS = {'bf16': 1, 'bf16x3': 3, 'bf16x6': 6}


class ClockSampler:
  """nvidia-smi clocks / throttle reasons; one background process per run, any number of
  (begin, end) windows; samples are attributed to a window by their timestamp."""
  Q = ('timestamp,clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,'
       'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
       'clocks_event_reasons.sw_power_cap')
  NAMES = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']

  def __init__(self, index):
    self.index = index
    self.proc = None
    self.lines = []

  def start(self):
    try:
      self.proc = subprocess.Popen(
          ['nvidia-smi', '-i', str(self.index), f'--query-gpu={self.Q}', '--format=csv,noheader,nounits',
           '-lms', '20'], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
      self.thread = threading.Thread(target=self._read, daemon=True)
      self.thread.start()
    except OSError:
      self.proc = None

  def _read(self):
    for line in self.proc.stdout:
      self.lines.append((time.time(), line.strip()))

  def stop(self):
    if self.proc is None:
      return
    time.sleep(0.05)
    self.proc.terminate()
    try:
      self.proc.wait(timeout=5)
    except subprocess.TimeoutExpired:
      self.proc.kill()

  def window(self, t0, t1):
    if self.proc is None:
      return dict(sm_mhz=None, sm_max_mhz=None, reasons=['nvidia-smi unavailable'])

    def parse(use_window):
      sm, mx, reasons = [], None, set()
      for ts, ln in list(self.lines):
        if use_window and not (t0 - 0.02 <= ts <= t1 + 0.05):
          continue
        parts = [p.strip() for p in ln.split(',')]
        if len(parts) < 7:
          continue
        try:
          sm.append(float(parts[1]))
          mx = float(parts[2])
        except ValueError:
          continue
        for n, v in zip(self.NAMES, parts[3:7]):
          if v.lower().startswith('active'):
            reasons.add(n)
      return sm, mx, reasons

    time.sleep(0.03)  # let the sample that closes the window arrive
    sm, mx, reasons = parse(True)
    where = 'timed region'
    if not sm:  # region shorter than the sampling period: fall back to the whole run under load
      sm, mx, reasons = parse(False)
      sm = [v for v in sm if mx and v > 0.5 * mx] or sm
      where = 'whole run (timed region shorter than the sampling period)'
    return dict(sm_mhz=(statistics.median(sm) if sm else None), sm_max_mhz=mx,
                reasons=sorted(reasons), samples=len(sm), window=where)


def build_inputs(wl, world):
  from tapnet_b200 import synth  # seeded synthetic inputs
  n = wl['q_per_gpu'] * world if wl['q_per_gpu'] else wl['q_total']
  video = synth.make_video(wl['frames'], wl['res'], wl['res'], seed=1)
  queries = synth.make_queries(n, wl['frames'], wl['res'], wl['res'], seed=2)
  return video, queries


def to_uint8_frames(video):
  """[-1, 1] float clip -> the raw uint8 frames the reference's callers hold
  (pytorch_live_demo.py:30-41 is the inverse map)."""
  return ((video + 1) * 127.5).round().clamp(0, 255).to(torch.uint8)


# ----------------------------------------------------------------------------------- ours


class Runner:
  """Shared state of one bench process: model(s), flush buffer, clocks sampler, dist."""

  def __init__(self, args):
    import torch.distributed as dist
    from tapnet_b200 import _lib, synth, tapir_model
    self.args = args
    self.dist = dist
    self.world = int(os.environ.get('WORLD_SIZE', '1'))
    self.rank = int(os.environ.get('RANK', '0'))
    self.local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    if self.world != args.gpus and self.world == 1 and args.gpus > 1:
      raise SystemExit('launch with torch.distributed.run for --gpus > 1')
    torch.cuda.set_device(self.local_rank)
    self.dev = torch.device('cuda', self.local_rank)
    if self.world > 1:
      if os.environ.get('NCCL_DEBUG', 'VERSION').upper() == 'VERSION':
        os.environ['NCCL_DEBUG'] = 'WARN'  # keep stdout to the single JSON line
      dist.init_process_group('nccl', device_id=self.dev)
    self.lib = _lib.load()
    self.sd = synth.make_state_dict(0)
    self.tapir_model = tapir_model
    self.model = tapir_model.TAPIR(pyramid_level=1, precision=args.precision)
    self.model.load_state_dict(self.sd)
    self.model = self.model.to(self.dev).eval()
    self.flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=self.dev)  # > 126 MB L2
    self.sampler = ClockSampler(self.local_rank)
    if self.rank == 0:
      self.sampler.start()
    self.peaks = _peaks()

  def barrier(self):
    if self.world > 1:
      self.dist.barrier()
    torch.cuda.synchronize()

  def timed(self, fn, steps):
    """K steps inside one barrier+sync bracket; per-step CUDA events; L2 flushed between steps.
    Returns (ms per step = max over ranks of the per-rank mean, clocks window, what the last
    step's fn() returned)."""
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
           for _ in range(steps)]
    self.barrier()
    t0 = time.time()
    for a, b in evs:
      out = None  # release the previous step's outputs before the next step, as a caller would
      self.flush.zero_()
      a.record()
      out = fn()
      b.record()
    self.barrier()
    t1 = time.time()
    ms = sum(a.elapsed_time(b) for a, b in evs)
    t = torch.tensor([ms], dtype=torch.float64, device=self.dev)
    if self.world > 1:
      self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
    clocks = self.sampler.window(t0, t1) if self.rank == 0 else None
    return t.item() / steps, clocks, out

  def profile(self, fn, reps=2):
    """Per-kernel device time: CUDA events around every launch of the library on its stream."""
    self.lib.tapir_profile_enable(1)
    for _ in range(reps):
      fn()
    cbuf = ctypes.create_string_buffer(1 << 16)
    prof = None
    if self.lib.tapir_profile_report(cbuf, len(cbuf)) == 0:
      prof = json.loads(cbuf.value.decode())
    self.lib.tapir_profile_enable(0)
    if not prof:
      return None, None
    tot = sum(v['ms'] for v in prof.values()) or 1.0
    breakdown = {k: dict(ms_per_step=round(v['ms'] / reps, 4), launches_per_step=v['launches'] // reps,
                         share=round(v['ms'] / tot, 4),
                         tflops=round(v['flops'] / (v['ms'] * 1e-3) / 1e12, 2) if v['ms'] > 0 else 0,
                         gbs=round(v['bytes'] / (v['ms'] * 1e-3) / 1e9, 1) if v['ms'] > 0 else 0)
                 for k, v in sorted(prof.items(), key=lambda kv: -kv[1]['ms'])}
    return prof, breakdown


def _traffic(name):
  tpath = os.path.join(ROOT, 'profiles', 'roofline_traffic.json')
  if os.path.exists(tpath):
    with open(tpath) as fh:
      return json.load(fh).get(name)
  return None


def roofline_tensor(name, v, peaks, terms, note=None):
  ach = v['flops'] / (v['ms'] * 1e-3) / 1e12
  d = dict(kernel=name, bound='tensor', achieved=round(ach, 2), peak=peaks['tf_sustained'],
           unit='TFLOP/s', frac=round(ach / peaks['tf_sustained'], 4), traffic=_traffic(name),
           peak_source=peaks['source'] + ', sustained (kernel timed inside a long step)',
           launches=v['launches'], avg_launch_ms=round(v['ms'] / v['launches'], 4),
           mma_terms=terms, issued_mma_tflops=round(ach * terms, 1),
           issued_mma_frac_of_sustained_peak=round(ach * terms / peaks['tf_sustained'], 4),
           issued_mma_frac_of_burst_peak=round(ach * terms / peaks['tf_burst'], 4),
           hbm_view=dict(algorithmic_gbs=round(v['bytes'] / (v['ms'] * 1e-3) / 1e9, 1),
                         frac_of_hbm_peak=round(v['bytes'] / (v['ms'] * 1e-3) / 1e9 / peaks['hbm'], 4)),
           note=note or ('achieved counts ALGORITHMIC fp32-equivalent FLOPs (2*M*N*K); the kernel '
                         f'issues {terms} bf16 MMAs per product term (split-bf16, required by the '
                         'parity budget), so tensor-pipe work is that multiple of this figure'))
  return d


def roofline_hbm(name, v, peaks):
  ach = v['bytes'] / (v['ms'] * 1e-3) / 1e9
  return dict(kernel=name, bound='hbm', achieved=round(ach, 1), peak=peaks['hbm'], unit='GB/s',
              frac=round(ach / peaks['hbm'], 4), traffic=_traffic(name), peak_source=peaks['source'],
              launches=v['launches'], avg_launch_ms=round(v['ms'] / v['launches'], 4))


DUMP_LIMIT = 64 << 20


def dump_outputs(out_dir, out, num_queries, world, rank):
  """Writes what one call of the timed path returned as float32 `<key>.npy` files: `tracks`,
  `occlusion`, `expected_dist` ([1, N, T(, 2)]) and, where the call returns them, the
  per-iteration `unrefined_*` lists stacked on a new leading axis.  Query shards are gathered
  first (a collective when world > 1; rank 0 writes).  Above DUMP_LIMIT bytes in all, every array
  keeps the same seeded sample of query points, whose indices go to `query_index.npy`."""
  import numpy as np  # pylint: disable=g-import-not-at-top
  from tapnet_b200 import distributed as tdist  # pylint: disable=g-import-not-at-top
  arrays = {}
  for k, v in out.items():
    qaxis = 2 if isinstance(v, (list, tuple)) else 1
    t = torch.stack(list(v)) if qaxis == 2 else v
    if world > 1:
      t = tdist.gather_queries(t, num_queries, qaxis)
    arrays[k] = (t.float().cpu().numpy(), qaxis)
  if rank != 0:
    return
  total = sum(a.nbytes for a, _ in arrays.values())
  if total > DUMP_LIMIT:
    keep = DUMP_LIMIT // (total // num_queries + 8)  # + 8 bytes per query for query_index
    idx = np.sort(np.random.default_rng(0).choice(num_queries, keep, replace=False))
    arrays = {k: (np.take(a, idx, axis=qaxis), qaxis) for k, (a, qaxis) in arrays.items()}
    arrays['query_index'] = (idx.astype(np.float64), 0)
  os.makedirs(out_dir, exist_ok=True)
  for k, (a, _) in arrays.items():
    np.save(os.path.join(out_dir, k + '.npy'), a)


def run_offline_workload(R, name, steps, warmup, with_profile=True, legs=('device', 'e2e', 'e2e_u8'),
                         dump_dir=None):
  """One offline workload (c2 / c4 / c5) -> record dict (rank 0) or None.  With dump_dir, the
  outputs of the last timed device step are written there (dump_outputs)."""
  from tapnet_b200 import distributed as tdist
  wl = WORKLOADS[name]
  world, rank, dev, model = R.world, R.rank, R.dev, R.model
  video_h, queries_h = build_inputs(wl, world)
  N, T = queries_h.shape[1], wl['frames']
  frames_u8_pin = to_uint8_frames(video_h).pin_memory()
  queries_pin = queries_h.pin_memory()
  big = video_h.numel() * 4 > (1 << 30)  # c5: keep the clip on the device as uint8 only
  video_pin = None if big else video_h.pin_memory()
  video_d = frames_u8_pin.to(dev) if big else video_pin.to(dev)
  queries_d = queries_pin.to(dev)
  out_pin = {k: torch.empty(s, dtype=torch.float32).pin_memory() for k, s in
             (('tracks', (1, N, T, 2)), ('occlusion', (1, N, T)), ('expected_dist', (1, N, T)))}

  def fwd(v, q, gather):
    if world > 1:
      return tdist.sharded_forward(model, v, q, gather_outputs=gather)
    return model(v, q)

  def step_device():
    return fwd(video_d, queries_d, False)

  def make_e2e(src_pin):
    def step():
      # the public call with HOST buffers: the clip is streamed to the device in frame chunks
      # behind the stem convolution (TAPIR.get_feature_grids), queries copied, results read back
      out = fwd(src_pin, queries_pin, True)
      if rank == 0:
        for k in out_pin:
          out_pin[k].copy_(out[k], non_blocking=True)
      torch.cuda.current_stream().synchronize()
    return step

  for _ in range(max(warmup, 3)):
    step_device()
  R.barrier()
  launches0 = R.lib.tapir_launch_count()
  ms_step, clocks, last = R.timed(step_device, steps)
  launches = (R.lib.tapir_launch_count() - launches0) // max(steps, 1)
  if dump_dir:
    dump_outputs(dump_dir, last, N, world, rank)
  del last
  d2h = int(sum(t.numel() * 4 for t in out_pin.values()))
  e2e = e2e_u8 = None
  if 'e2e' in legs and video_pin is not None:
    f = make_e2e(video_pin)
    f()
    ms, _, _ = R.timed(f, steps)
    e2e = dict(value=round(N * T / (ms * 1e-3), 1), unit=UNIT, ms_per_step=round(ms, 3),
               h2d_bytes_per_step=int(video_h.numel() * 4 + queries_h.numel() * 4),
               d2h_bytes_per_step=d2h, frames='float32 [-1,1]')
  if 'e2e_u8' in legs:
    f = make_e2e(frames_u8_pin)
    f()
    ms, _, _ = R.timed(f, steps)
    e2e_u8 = dict(value=round(N * T / (ms * 1e-3), 1), unit=UNIT, ms_per_step=round(ms, 3),
                  h2d_bytes_per_step=int(video_h.numel() + queries_h.numel() * 4),
                  d2h_bytes_per_step=d2h,
                  frames='uint8 raw frames (what the reference callers hold, '
                         'pytorch_live_demo.py:30-41); preprocess_frames fused into the stem conv')
  prof = breakdown = None
  if with_profile:
    prof, breakdown = R.profile(step_device, 2)
  if rank != 0:
    return None
  rec = dict(
      metric=metric_name(wl), value=round(N * T / (ms_step * 1e-3), 1), unit=UNIT, n_gpus=world,
      steps=steps, warmup=max(warmup, 3), ms_per_step=round(ms_step, 3), scaling=wl['scaling'],
      config=dict(workload=f"TAPIR/BootsTAPIR inference {wl['res']}x{wl['res']}x{T}, "
                           + (f"{wl['q_per_gpu']} query points per GPU ({N} total)" if wl['q_per_gpu']
                              else f'{N} query points in total shared by {world} GPU(s)')
                           + f", {wl['config']}",
                  frames=T, resolution=wl['res'], queries=N,
                  refine_iterations=4 * (3 if wl['res'] == 1024 else 1),
                  parallelism=f'frame-shard backbone + all-gather + query-shard x{world}',
                  l2='256 MiB buffer written between timed steps (L2 flush)',
                  weights='seeded random init (no checkpoint reachable offline)',
                  device_resident_video='uint8' if big else 'float32'),
      clocks=clocks, gpu_launches=int(launches))
  # `e2e` = the clip as the reference's callers hold it: raw uint8 frames (pytorch_live_demo.py:
  # 30-41 normalises them on the device; here that is fused into the stem conv).  The same call
  # with an already-normalised float32 clip (4x the PCIe bytes) is reported next to it.
  if e2e_u8 is not None:
    rec['e2e'] = e2e_u8
  if e2e is not None:
    rec['e2e_float_frames'] = e2e
  if prof:
    rec['_prof'] = prof
    rec['kernel_breakdown'] = breakdown
  return rec


def run_c3_stream(R):
  """BASELINE config 3: causal model, per-frame online steps through OnlineTracker (CUDA-graph
  replay of pytorch_live_demo.py:62-85), 1024 points, 250 frames after 10 warm-up frames."""
  from tapnet_b200 import streaming, synth
  dev = R.dev
  cm = R.tapir_model.TAPIR(pyramid_level=1, use_casual_conv=True, precision=R.args.precision)
  cm.load_state_dict(R.sd)
  cm = cm.to(dev).eval()
  n, res, F, W = C3['points'], C3['res'], C3['frames'], C3['warm_frames']
  clip = synth.make_video(16, res, res, seed=1)  # frames are cycled; content does not affect timing
  clip_u8_pin = to_uint8_frames(clip)[0].pin_memory()   # [16, H, W, 3]
  clip_d = clip[0].to(dev)
  q = synth.make_queries(n, 1, res, res, seed=2, frame0_only=True).to(dev)

  def run(tracker, frames_src, host_io):
    tracker.init(frames_src[0].to(dev), q)
    trk_pin = torch.empty(1, n, 1, 2, dtype=torch.float32).pin_memory()
    vis_pin = torch.empty(1, n, 1, dtype=torch.bool).pin_memory()

    def one(t):
      tracks, vis = tracker.step(frames_src[t % 16])
      if host_io:  # a live consumer reads every frame's result before it grabs the next frame
        trk_pin.copy_(tracks, non_blocking=True)
        vis_pin.copy_(vis, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    for t in range(W):
      one(t)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    t0 = time.time()
    e0.record()
    for t in range(F):
      one(W + t)
    e1.record()
    torch.cuda.synchronize()
    t1 = time.time()
    return e0.elapsed_time(e1) / F, R.sampler.window(t0, t1)

  trk = streaming.OnlineTracker(cm, res, res, n)
  trk.init(clip_d[0], q)
  trk.step(clip_d[0])  # captures the graph (launch counter advances while capturing)
  ms_dev, clocks = run(trk, clip_d, False)
  trk.close()
  trk8 = streaming.OnlineTracker(cm, res, res, n, uint8_frames=True)
  ms_e2e, _ = run(trk8, clip_u8_pin, True)
  trk8.close()
  # launches of one frame + per-kernel time: eager steps (events cannot be read out of a graph)
  from tapnet_b200 import live
  qf = live.online_model_init(cm, clip_d[None, :1], q)
  state = [{k: v.to(dev) for k, v in d.items()}
           for d in cm.construct_initial_causal_state(n, len(qf.resolutions) - 1)]
  holder = {'s': state}

  def eager():
    _, _, holder['s'] = live.online_model_predict(cm, clip_d[None, :1], qf, holder['s'])

  for _ in range(3):
    eager()
  torch.cuda.synchronize()
  l0 = R.lib.tapir_launch_count()
  eager()
  per_frame_launches = int(R.lib.tapir_launch_count() - l0)
  _, breakdown = R.profile(eager, 4)
  return dict(
      metric='causal online tracking, ms per frame (1 frame per step, causal state carried)',
      config=dict(workload=f"causal BootsTAPIR streaming {res}x{res}, {n} points, {F} frames after "
                           f"{W} warm-up frames, {C3['config']}", points=n, frames=F,
                  path='tapnet_b200.streaming.OnlineTracker (CUDA-graph replay of the per-frame step)'),
      ms_per_frame=round(ms_dev, 4), frames_per_s=round(1e3 / ms_dev, 1),
      value=round(n * 1e3 / ms_dev, 1), unit=UNIT, higher_is_better=True, n_gpus=1,
      e2e=dict(ms_per_frame=round(ms_e2e, 4), frames_per_s=round(1e3 / ms_e2e, 1),
               value=round(n * 1e3 / ms_e2e, 1), unit=UNIT,
               h2d_bytes_per_step=int(res * res * 3), d2h_bytes_per_step=int(n * 2 * 4 + n),
               note='every frame: uint8 frame from pinned host memory in, tracks + visibility out, '
                    'host synchronised before the next frame (live-demo consumer)'),
      clocks=clocks, gpu_launches_per_frame=per_frame_launches, kernel_breakdown=breakdown)


def run_ours(args):
  R = Runner(args)
  world, rank = R.world, R.rank
  main = run_offline_workload(R, args.workload, args.steps, args.warmup, dump_dir=args.dump_outputs)
  sub = {}
  if not args.no_sub and args.workload == 'c2':
    sub_steps = max(2, min(args.steps, 5))
    r = run_offline_workload(R, 'c4', sub_steps, 3, legs=('device', 'e2e_u8'))
    if r:
      sub['c4_strong'] = r
    if world == 1:
      try:
        sub['c3_stream'] = run_c3_stream(R)
      except Exception as e:  # pylint: disable=broad-except
        sub['c3_stream'] = dict(error=repr(e)[:300])
    try:
      r = run_offline_workload(R, 'c5', 2, 3, with_profile=(world == 1), legs=('device', 'e2e_u8'))
      if r:
        sub['c5_hires'] = r
    except Exception as e:  # pylint: disable=broad-except
      if rank == 0:
        sub['c5_hires'] = dict(error=repr(e)[:300])
  if rank != 0:
    R.sampler.stop()
    if world > 1:
      R.dist.destroy_process_group()
    return
  R.sampler.stop()
  peaks = R.peaks
  prof = main.pop('_prof', None)
  for r in sub.values():
    r.pop('_prof', None)
  terms = _MMA_TERMS[args.precision]
  roofline = None
  named = {}
  if prof:
    per_step = {k: dict(v, launches=v['launches'] // 2) for k, v in prof.items()}
    name, v = max(prof.items(), key=lambda kv: kv[1]['ms'])
    is_gemm = v['flops'] > 0 and ('mixer.' in name or 'conv' in name or 'gemm' in name or 'proj' in name) \
        and name != 'mixer.dw'
    vv = dict(v, launches=max(v['launches'], 1))
    roofline = roofline_tensor(name, vv, peaks, terms) if is_gemm else roofline_hbm(name, vv, peaks)
    roofline['launches'] = per_step[name]['launches']
    if 'cost_volume.gemm' in prof:
      cv = roofline_tensor('cost_volume.gemm', prof['cost_volume.gemm'], peaks, 6,
                           note='global cost volume (tapir_model.py:720): 2*N*T*1024*256 FLOPs, computed '
                                'with three bf16 terms per operand = 6 MMAs per product (fp32-equivalent: '
                                'its arg-max must match the reference bit for bit); bytes = cost volume '
                                'written (fp32) + grid and query planes read (SURVEY.md 8(d), materialised)')
      cv['launches'] = per_step['cost_volume.gemm']['launches']
      named['cost_volume'] = cv
    if 'local_corr' in prof:
      lc = roofline_hbm('local_corr', prof['local_corr'], peaks)
      lc['launches'] = per_step['local_corr']['launches']
      lc['note'] = ('algorithmic bytes per SURVEY.md 8(d): N*T*(64 cells * (128+256+256) ch * 4 B + 2132 B) '
                    'per refinement iteration; most of them are served by L2 (frame-major CTA order), so '
                    'the figure can exceed the HBM copy peak')
      named['local_corr'] = lc
    if 'cost_volume.head' in prof:
      v = prof['cost_volume.head']
      named['cost_volume_head'] = dict(
          kernel='cost_volume.head', bound='cuda-core / shared memory',
          achieved=round(v['flops'] / (v['ms'] * 1e-3) / 1e12, 2), unit='TFLOP/s',
          avg_launch_ms=round(v['ms'] / max(v['launches'], 1), 4), launches=per_step['cost_volume.head']['launches'])
  wl = WORKLOADS[args.workload]
  cpu_baseline = None
  if world == 1 and not args.no_cpu:
    video_h, queries_h = build_inputs(wl, world)
    cpu_baseline = cpu_reference(R.sd, video_h, queries_h, wl, repeats=3)
  line = dict(
      metric=main['metric'], value=main['value'], unit=UNIT, n_gpus=world, steps=args.steps,
      warmup=max(args.warmup, 3), ms_per_step=main['ms_per_step'], higher_is_better=True,
      scaling=wl['scaling'], vs_baseline=None,
      dtype='bf16x3' if args.precision == 'bf16x3' else args.precision, data='synthetic',
      config=main['config'], clocks=main['clocks'], e2e=main.get('e2e'),
      e2e_float_frames=main.get('e2e_float_frames'), gpu_launches=main['gpu_launches'],
      roofline=roofline, roofline_named=named or None, cpu_baseline=cpu_baseline,
      sub_records=sub or None, kernel_breakdown=main.get('kernel_breakdown'))
  print(json.dumps(line))
  if world > 1:
    R.dist.destroy_process_group()


# ----------------------------------------------------------------------------------- CPU reference


def _load_reference_module():
  """The UNMODIFIED reference torch path, if it is installed in the tree: `baseline/_ref`
  (a git-ignored `pip install --target baseline/_ref` of the original tapnet package).
  Layout-only shims for its two absent dependencies (einshape, dm-tree) come from oracle/shims.
  Returns (the module `tapnet.torch.tapir_model`, its root) or (None, None)."""
  root = os.path.join(ROOT, 'baseline', '_ref')
  if not os.path.isfile(os.path.join(root, 'tapnet', 'torch', 'tapir_model.py')):
    return None, None
  for p in (root, os.path.join(ROOT, 'oracle', 'shims')):
    if p not in sys.path:
      sys.path.insert(0, p)
  try:
    from tapnet.torch import tapir_model as ref  # pylint: disable=g-import-not-at-top
    return ref, root
  except Exception:  # pylint: disable=broad-except
    return None, None


SAMPLE_FRAMES, SAMPLE_QUERIES = 4, 16


class CpuArm:
  """The reference's CPU implementation of the path, timed on a bounded sample of the workload.

  kind 'reference': the unmodified `tapnet.torch.tapir_model.TAPIR` (see _load_reference_module);
  kind 'port': oracle/tapir_oracle.py (the CPU restatement) when the reference is not importable.
  One sample = backbone on SAMPLE_FRAMES of the clip's frames (frames are independent: cost is
  linear in frames) + get_query_features / estimate_trajectories for SAMPLE_QUERIES of the
  queries over ALL frames (queries are independent: linear in queries).  The two per-unit costs
  are scaled to the full job:  value = N*T / (t_backbone * T/SAMPLE_FRAMES + t_track * N/SAMPLE_QUERIES).
  """

  def __init__(self, sd, video, queries, wl):
    self.video, self.queries, self.wl = video, queries, wl
    self.T, self.N = video.shape[1], queries.shape[1]
    self.res = wl['res']
    ref, root = _load_reference_module()
    self.kind = 'reference' if ref is not None else 'port'
    self.where = root
    g = torch.Generator().manual_seed(0)
    r = self.res
    levels = 3 if r == 1024 else 1
    sizes = [256] + ([256, 512, 1024][:levels] if r == 1024 else [r])
    # timing-only grids of the right shapes (unit-norm random features)
    lo = [torch.nn.functional.normalize(torch.randn(1, self.T, s // 8, s // 8, 256, generator=g), dim=-1)
          for s in sorted(set(sizes))]
    hi = [torch.nn.functional.normalize(torch.randn(1, self.T, s // 4, s // 4, 128, generator=g), dim=-1)
          for s in sorted(set(sizes))]
    idx = {s: i for i, s in enumerate(sorted(set(sizes)))}
    self.lo = tuple(lo[idx[s]] for s in sizes)
    self.hi = tuple(hi[idx[s]] for s in sizes)
    self.sizes = sizes
    if ref is not None:
      self.ref = ref
      self.model = ref.TAPIR(pyramid_level=1)
      self.model.load_state_dict(sd)
      self.model.eval()
    else:
      from oracle import tapir_oracle as O  # pylint: disable=g-import-not-at-top
      self.O, self.sd, self.cfg = O, sd, O.Config()

  def sample(self):
    """Seconds for the full job extrapolated from one sample."""
    v, q = self.video[:, :SAMPLE_FRAMES], self.queries[:, :SAMPLE_QUERIES]
    hw = (self.res, self.res)
    with torch.no_grad():
      if self.kind == 'reference':
        t0 = time.perf_counter()
        self.model.get_feature_grids(v, is_training=False)
        t_bb = time.perf_counter() - t0
        grids = self.ref.FeatureGrids(self.lo, self.hi, tuple(torch.Size([s, s]) for s in self.sizes))
        t0 = time.perf_counter()
        qf = self.model.get_query_features(self.video, False, q, grids)
        self.model.estimate_trajectories(hw, False, grids, qf, q, query_chunk_size=64)
        t_tr = time.perf_counter() - t0
      else:
        O = self.O
        t0 = time.perf_counter()
        O.get_feature_grids(self.sd, self.cfg, v)
        t_bb = time.perf_counter() - t0
        grids = O.Grids(self.lo, self.hi, tuple((s, s) for s in self.sizes))
        t0 = time.perf_counter()
        qf = O.get_query_features(self.cfg, self.video.shape, q, grids)
        O.estimate_trajectories(self.sd, self.cfg, hw, grids, qf, q, 64)
        t_tr = time.perf_counter() - t0
    return t_bb * (self.T / SAMPLE_FRAMES) + t_tr * (self.N / SAMPLE_QUERIES)

  def pick_threads(self):
    """torch's CPU kernels do not scale to very wide hosts on these small per-frame problems
    (128 threads were 40x slower than 8 on the GPU box): give the reference its best case.  The
    thread count is chosen from the median of 3 repetitions of THE SAMPLE ITSELF per candidate."""
    ncpu = os.cpu_count() or 1
    cands = sorted({c for c in (8, 16, 32, 64) if c <= ncpu} or {ncpu})
    best, best_t, table = cands[0], float('inf'), {}
    for c in cands:
      torch.set_num_threads(c)
      self.sample()  # warm (thread pool, allocator)
      ts = sorted(self.sample() for _ in range(3))
      table[c] = round(ts[1], 3)
      if ts[1] < best_t:
        best, best_t = c, ts[1]
      if ts[1] > 2.5 * best_t:
        break  # far past the optimum: wider counts only get slower
    torch.set_num_threads(best)
    self.threads, self.sweep = best, table
    return best

  def describe(self, seconds):
    n_units = self.N * self.T
    return dict(
        value=round(n_units / seconds, 1), unit=UNIT, cores=self.threads, kind=self.kind,
        sample=f'backbone on {SAMPLE_FRAMES}/{self.T} frames + get_query_features / '
               f'estimate_trajectories on {SAMPLE_QUERIES}/{self.N} queries x {self.T} frames; the two '
               f'per-unit costs scaled linearly to the full job (est. {seconds:.1f} s/step)',
        thread_sweep_s_per_step=self.sweep, logical_cores=os.cpu_count(),
        note=('unmodified reference tapnet.torch.tapir_model.TAPIR on the host cores '
              f'(imported from {os.path.relpath(self.where, ROOT) if self.where.startswith(ROOT) else self.where} '
              'through the layout-only einshape / dm-tree shims of oracle/shims)' if self.kind == 'reference'
              else 'CPU restatement of the reference torch path (oracle/tapir_oracle.py): the '
                   'reference itself is not importable on this box')
             + f'; torch {torch.__version__}; the reference JAX-CPU path cannot run (no jax in the image)')


def cpu_reference(sd, video, queries, wl, repeats=3):
  arm = CpuArm(sd, video, queries, wl)
  arm.pick_threads()
  ts = sorted(arm.sample() for _ in range(repeats))
  return arm.describe(ts[len(ts) // 2])


def run_reference(args):
  """--impl reference: the reference's own CPU implementation of the path on the host cores."""
  rank = int(os.environ.get('RANK', '0'))
  if rank != 0:
    return
  from tapnet_b200 import synth
  world = int(os.environ.get('WORLD_SIZE', str(args.gpus)))
  wl = WORKLOADS[args.workload]
  video, queries = build_inputs(wl, world)
  arm = CpuArm(synth.make_state_dict(0), video, queries, wl)
  arm.pick_threads()
  for _ in range(args.warmup):
    arm.sample()
  ts = [arm.sample() for _ in range(args.steps)]
  sec = statistics.median(ts)
  N, T = queries.shape[1], wl['frames']
  base = arm.describe(sec)
  base['spread'] = dict(min_s=round(min(ts), 3), max_s=round(max(ts), 3), samples=len(ts))
  v = base['value']
  line = dict(impl='reference', metric=metric_name(wl), value=v, unit=UNIT, n_gpus=world,
              steps=args.steps, warmup=args.warmup, ms_per_step=round(sec * 1e3, 1),
              higher_is_better=True, scaling=wl['scaling'], vs_baseline=None, dtype='f32',
              data='synthetic',
              config=dict(workload=f"TAPIR/BootsTAPIR inference {wl['res']}x{wl['res']}x{T}, "
                                   + (f"{wl['q_per_gpu']} query points per GPU ({N} total)" if wl['q_per_gpu']
                                      else f'{N} query points in total')
                                   + f", {wl['config']}",
                          frames=T, resolution=wl['res'], queries=N,
                          refine_iterations=4 * (3 if wl['res'] == 1024 else 1)),
              cpu_baseline=base,
              e2e=dict(value=v, unit=UNIT, h2d_bytes_per_step=0, d2h_bytes_per_step=0))
  print(json.dumps(line))


def main():
  ap = argparse.ArgumentParser()
  ap.add_argument('--gpus', type=int, default=1)
  ap.add_argument('--steps', type=int, default=20,
                  help='timed steps of each leg of the headline workload (sub-records keep their '
                       'own short budgets)')
  ap.add_argument('--warmup', type=int, default=3)
  ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
  ap.add_argument('--precision', default='bf16x3', choices=['bf16', 'bf16x3', 'bf16x6'])
  ap.add_argument('--no-cpu', action='store_true', help='skip the cpu_baseline leg')
  ap.add_argument('--no-sub', action='store_true', help='skip the c4 / c3 / c5 sub-records')
  ap.add_argument('--workload', default='c2', choices=['c2', 'c4', 'c5'],
                  help='headline workload: c2 = driver contract (default)')
  ap.add_argument('--dump-outputs', metavar='DIR',
                  help='write the outputs of the last timed headline step to DIR/<name>.npy')
  args = ap.parse_args()
  if args.steps < 1:
    ap.error('--steps must be at least 1')
  if args.impl == 'reference':
    run_reference(args)
  else:
    run_ours(args)


if __name__ == '__main__':
  main()
