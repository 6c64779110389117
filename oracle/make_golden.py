"""TEST INFRASTRUCTURE - generates tests/golden/*.npz by running the UNMODIFIED reference.

Run in the build container only (needs /root/reference):  python -m oracle.make_golden
The fixtures pin `oracle/tapir_oracle.py` (and through it the CUDA path) to the reference's
own outputs on seeded synthetic inputs; inputs are regenerated from the seeds recorded in
each file (`oracle/synth.py`), outputs are stored.
"""
import json
import os

import numpy as np
import torch

from oracle import reference_loader, synth

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                          'tests', 'golden')

CASES = {
    # name: (model kwargs, T, N, H, W, mode)
    'c1_bootstapir_256x8_n16': (dict(pyramid_level=1), 8, 16, 256, 256, 'offline'),
    'tapir_pl0_noextra_256x4_n8': (dict(pyramid_level=0, extra_convs=False), 4, 8, 256, 256,
                                   'offline'),
    'bootstapir_320x384x4_n12': (dict(pyramid_level=1), 4, 12, 320, 384, 'offline'),
    'causal_256x6_n16': (dict(pyramid_level=1, use_casual_conv=True), 6, 16, 256, 256,
                         'causal'),
    # BASELINE config 5's pyramid: 1024x1024 -> levels 256 / 512 / 1024, 12 refinement iterations
    'bootstapir_1024x2_n6': (dict(pyramid_level=1), 2, 6, 1024, 1024, 'offline'),
    # the README's live-demo shape (17 fps figure): 480x480, 8 points, two levels = 8 iterations
    'causal_480x3_n8': (dict(pyramid_level=1, use_casual_conv=True), 3, 8, 480, 480, 'causal'),
    # constructor argument initial_resolution (tapir_model.py:86): a 24 x 40 cost-volume map
    'bootstapir_ir192x320x3_n10': (dict(pyramid_level=1, initial_resolution=(192, 320)), 3, 10, 192,
                                   320, 'offline'),
    # constructor argument pyramid_level = 2: two pooled levels, four correlation levels (mixer in 584)
    'tapir_pl2_256x3_n6': (dict(pyramid_level=2), 3, 6, 256, 256, 'offline'),
}


def _np(x):
  return x.detach().cpu().numpy()


class _StageAProbe:
  """Records what `utils.soft_argmax_heatmap_batched` (utils.py:116-150) sees and decides: wraps
  the reference function, repeats its own arg-max expression on the same tensor (same op, same
  input -> same indices) and passes the call through unchanged."""

  def __init__(self):
    self.argmax, self.margin = [], []

  def __enter__(self):
    from tapnet.torch import utils as ref_utils  # the unmodified reference module
    self._mod = ref_utils
    self._orig = ref_utils.soft_argmax_heatmap_batched

    def wrapped(softmax_val, threshold=5):
      b, n, t = softmax_val.shape[:3]
      flat = softmax_val.reshape(b, n, t, -1)
      self.argmax.append(torch.argmax(flat, dim=-1)[0])
      top2 = torch.topk(flat, 2, dim=-1).values[0]
      self.margin.append(top2[..., 0] - top2[..., 1])
      return self._orig(softmax_val, threshold)

    ref_utils.soft_argmax_heatmap_batched = wrapped
    return self

  def __exit__(self, *exc):
    self._mod.soft_argmax_heatmap_batched = self._orig

  def result(self):
    return torch.cat(self.argmax, dim=0), torch.cat(self.margin, dim=0)


def run_case(name):
  kwargs, T, N, H, W, mode = CASES[name]
  sd = synth.make_state_dict(0, kwargs.get('pyramid_level', 1), kwargs.get('extra_convs', True))
  model = reference_loader.build(sd, **kwargs)
  video = synth.make_video(T, H, W, seed=1)
  queries = synth.make_queries(N, T, H, W, seed=2, frame0_only=(mode == 'causal'))
  out = {}
  meta = dict(name=name, model_kwargs=kwargs, T=T, N=N, H=H, W=W, mode=mode,
              weights_seed=0, video_seed=1, query_seed=2, torch=torch.__version__)
  with torch.no_grad():
    grids = model.get_feature_grids(video, is_training=False)
    qf = model.get_query_features(video, False, queries, grids)
    # strided sub-samples of the feature grids / query features (full grids are MBs)
    out['lowres_sub'] = _np(grids.lowres[-1][0, :, ::5, ::7, ::16])
    out['hires_sub'] = _np(grids.hires[-1][0, :, ::9, ::11, ::16])
    out['qfeat_lowres'] = _np(qf.lowres[-1][0, :, ::8])
    out['qfeat_hires'] = _np(qf.hires[-1][0, :, ::8])
    meta['resolutions'] = [list(map(int, r)) for r in grids.resolutions]
    torch.manual_seed(123)  # estimate_trajectories shuffles queries with torch.randperm
    perm = torch.randperm(N)  # the permutation the call below will draw (tapir_model.py:464)
    torch.manual_seed(123)
    with _StageAProbe() as probe:
      tr = model.estimate_trajectories(video.shape[-3:-1], False, grids, qf, queries,
                                       query_chunk_size=64)
    # stage-A arg-max cell of every (query, frame) heat map, exactly as the reference computed it
    # (utils.py:126), un-permuted to query order; plus the top-2 probability margin of each map
    am, mg = probe.result()
    inv = torch.empty_like(perm)
    inv[perm] = torch.arange(N)
    out['stage_a_argmax'] = _np(am[inv]).astype(np.int32)
    out['stage_a_margin'] = _np(mg[inv]).astype(np.float32)
    out['tracks_iters'] = np.stack([_np(t[0]) for t in tr['tracks']])
    out['occlusion_iters'] = np.stack([_np(t[0]) for t in tr['occlusion']])
    out['expected_dist_iters'] = np.stack([_np(t[0]) for t in tr['expected_dist']])
    torch.manual_seed(123)
    fw = model(video, queries)
    out['tracks'] = _np(fw['tracks'][0])
    out['occlusion'] = _np(fw['occlusion'][0])
    out['expected_dist'] = _np(fw['expected_dist'][0])
    if mode == 'causal':
      # streaming: frame by frame with causal state (pytorch_live_demo.py:44-85)
      g0 = model.get_feature_grids(video[:, :1], False)
      qf0 = model.get_query_features(video[:, :1], False, queries, g0)
      state = model.construct_initial_causal_state(N, len(qf0.resolutions) - 1)
      tr_l, oc_l, ex_l = [], [], []
      for t in range(T):
        g = model.get_feature_grids(video[:, t:t + 1], False)
        r = model.estimate_trajectories((H, W), False, g, qf0, None, query_chunk_size=64,
                                        causal_context=state, get_causal_context=True)
        state = r['causal_context']
        tr_l.append(_np(r['tracks'][-1][0]))
        oc_l.append(_np(r['occlusion'][-1][0]))
        ex_l.append(_np(r['expected_dist'][-1][0]))
      out['online_tracks'] = np.concatenate(tr_l, axis=1)
      out['online_occlusion'] = np.concatenate(oc_l, axis=1)
      out['online_expected_dist'] = np.concatenate(ex_l, axis=1)
      out['online_state_sub'] = _np(state[-1]['block_11_causal_2'][0, :, :, ::64])
  out['meta'] = np.frombuffer(json.dumps(meta).encode(), dtype=np.uint8)
  return out


# constructor keywords whose state_dict layout tests/test_schema.py pins
SCHEMA_KWARGS = {'pl1': dict(pyramid_level=1), 'pl0_noextra': dict(pyramid_level=0, extra_convs=False)}
# frame sizes whose generate_default_resolutions(size, (256, 256)) tests/test_host_logic.py pins
RESOLUTION_SIZES = [(256, 256), (240, 240), (480, 480), (480, 640), (360, 640), (512, 512),
                    (720, 1280), (1024, 1024), (1080, 1920), (264, 264), (250, 500), (2048, 1024)]


def run_interface():
  """The reference's host-side interface, no compute: state_dict key order and shapes per
  constructor, and the refinement resolutions it picks per frame size (utils.py:275-317)."""
  import contextlib  # pylint: disable=g-import-not-at-top
  import io  # pylint: disable=g-import-not-at-top
  ref = reference_loader.load()
  from tapnet.torch import utils as ref_utils  # pylint: disable=g-import-not-at-top
  schema = {k: [[name, list(v.shape)] for name, v in ref.TAPIR(**kw).state_dict().items()]
            for k, kw in SCHEMA_KWARGS.items()}
  with contextlib.redirect_stdout(io.StringIO()):   # the non-multiple-of-8 warning
    res = [[list(hw), [[int(v) for v in r] for r in ref_utils.generate_default_resolutions(hw, (256, 256))]]
           for hw in RESOLUTION_SIZES]
  meta = dict(name='reference_interface', schema=schema, schema_kwargs=SCHEMA_KWARGS,
              default_resolutions=res, torch=torch.__version__)
  return {'meta': np.frombuffer(json.dumps(meta).encode(), dtype=np.uint8)}


def main():
  import sys  # pylint: disable=g-import-not-at-top
  os.makedirs(GOLDEN_DIR, exist_ok=True)
  for name in (sys.argv[1:] or ['reference_interface', *CASES]):
    out = run_interface() if name == 'reference_interface' else run_case(name)
    path = os.path.join(GOLDEN_DIR, name + '.npz')
    np.savez_compressed(path, **out)
    print(name, os.path.getsize(path), 'bytes')


if __name__ == '__main__':
  main()
