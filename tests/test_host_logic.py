"""Host-side mirror of the reference interface (CPU only: no compute calls)."""
import pytest
import torch

from oracle import synth
from tapnet_b200 import schema, tapir_model


def test_state_dict_layout_and_load():
  m = tapir_model.TAPIR(pyramid_level=1)
  sd = m.state_dict()
  assert list(sd.keys()) == list(schema.state_dict_schema().keys())
  m.load_state_dict(synth.make_state_dict(0))  # strict load of a reference-layout dict
  m0 = tapir_model.TAPIR(pyramid_level=0, extra_convs=False)
  assert len(m0.state_dict()) == 188 and m0.extra_convs is None


def test_ctor_surface_matches_reference_keywords():
  m = tapir_model.TAPIR(bilinear_interp_with_depthwise_conv=False, num_pips_iter=4, pyramid_level=1,
                        mixer_hidden_dim=512, num_mixer_blocks=12, mixer_kernel_shape=3,
                        patch_size=7, softmax_temperature=20.0,
                        parallelize_query_extraction=False, initial_resolution=(256, 256),
                        blocks_per_group=(2, 2, 2, 2), feature_extractor_chunk_size=10,
                        extra_convs=True, use_casual_conv=True)
  assert m.use_casual_conv and m.initial_resolution == (256, 256)
  for name in ('forward', 'get_feature_grids', 'get_query_features', 'estimate_trajectories',
               'construct_initial_causal_state', 'update_query_features'):
    assert callable(getattr(m, name))


def test_errors_match_reference():
  m = tapir_model.TAPIR()
  with pytest.raises(ValueError, match='Get query feats not supported in TAPIR.'):
    m(torch.zeros(1, 2, 256, 256, 3), torch.zeros(1, 4, 3), get_query_feats=True)
  with pytest.raises(ValueError, match='multiple of 8'):
    m.get_feature_grids(torch.zeros(1, 1, 256, 256, 3), False, refinement_resolutions=[(250, 256)])
  with pytest.raises(RuntimeError, match='CUDA only'):
    m(torch.zeros(1, 2, 256, 256, 3), torch.zeros(1, 4, 3))


def test_causal_state_shape_and_aliasing():
  m = tapir_model.TAPIR(use_casual_conv=True)
  st = m.construct_initial_causal_state(5, 2)
  assert len(st) == 8 and st[0] is st[7]  # reference returns the same dict 4*L times
  assert st[0]['block_11_causal_2'].shape == (1, 5, 2, 2048)
  assert sorted(st[0])[0] == 'block_0_causal_1' and len(st[0]) == 24


def test_update_query_features_in_place():
  m = tapir_model.TAPIR(use_casual_conv=True)
  lo, hi = torch.zeros(1, 4, 256), torch.zeros(1, 4, 128)
  qf = tapir_model.QueryFeatures((lo, lo), (hi, hi), ((256, 256), (256, 256)))
  new = tapir_model.QueryFeatures((torch.ones(1, 1, 256),) * 2, (torch.ones(1, 1, 128),) * 2,
                                  ((256, 256), (256, 256)))
  st = m.construct_initial_causal_state(4, 1)
  for d in st:
    for v in d.values():
      v.fill_(3.0)
  qf2, st2 = m.update_query_features(qf, new, 2, st)
  assert lo[0, 2].eq(1).all() and lo[0, 1].eq(0).all() and qf2.lowres[0] is lo
  assert st2[0]['block_0_causal_1'][0, 2].eq(0).all() and st2[0]['block_0_causal_1'][0, 1].eq(3).all()


def test_default_resolutions():
  f = tapir_model.generate_default_resolutions
  assert f((256, 256), (256, 256)) == [(256, 256)]
  assert f((480, 480), (256, 256)) == [(256, 256), (480, 480)]
  assert f((1024, 1024), (256, 256)) == [(256, 256), (512, 512), (1024, 1024)]


def test_default_resolutions_sweep_matches_reference_and_oracle(golden):
  """generate_default_resolutions over a sweep of frame sizes: product == oracle restatement ==
  the reference's own function (utils.py:275-317), whose results
  `python -m oracle.make_golden reference_interface` stored."""
  import contextlib
  import io
  from oracle import tapir_oracle as O
  sweep = golden('reference_interface')['meta']['default_resolutions']
  assert len(sweep) == 12
  for hw, ref in sweep:
    hw = tuple(hw)
    with contextlib.redirect_stdout(io.StringIO()):   # the non-multiple-of-8 warning
      got = tapir_model.generate_default_resolutions(hw, (256, 256))
      want = O.default_resolutions(hw, (256, 256))
      assert [tuple(r) for r in got] == [tuple(r) for r in want], hw
      assert [tuple(r) for r in got] == [tuple(r) for r in ref], hw
    assert all(r[0] % 8 == 0 and r[1] % 8 == 0 for r in got)
    assert tuple(got[0]) == (256, 256)


def test_live_crop_window_matches_reference_slicing():
  """live.center_square_window == the slicing of get_frame (pytorch_live_demo.py:88-95) on a
  coordinate image, for landscape / portrait / square frames."""
  import numpy as np
  from tapnet_b200 import live
  for h, w in [(240, 320), (320, 240), (480, 480), (36, 53), (1080, 1920), (7, 3)]:
    yy, xx = np.meshgrid(np.arange(h), np.arange(w), indexing='ij')
    image = np.stack([yy, xx], -1)
    trunc = abs(w - h) // 2
    if w > h:
      want = image[:, trunc:-trunc]
    elif w < h:
      want = image[trunc:-trunc]
    else:
      want = image
    y0, x0, ch, cw = live.center_square_window(h, w)
    np.testing.assert_array_equal(image[y0:y0 + ch, x0:x0 + cw], want)


def test_build_model_dispatches_on_haiku_npy(tmp_path):
  """build_model('x.npy'): the Haiku tree goes through convert.py (ADVICE r1: bulk.track_many_points
  is handed such a path); constructor arguments are inferred from the tree."""
  import numpy as np
  from tapnet_b200 import convert
  sd = synth.make_state_dict(3, pyramid_level=0, extra_convs=False)
  tree = convert.to_haiku_params(sd, pyramid_level=0, extra_convs=False)
  path = tmp_path / 'ckpt.npy'
  np.save(path, {'params': tree}, allow_pickle=True)
  m = tapir_model.build_model(str(path), device='cpu')
  assert m.pyramid_level == 0 and m.extra_convs is None
  got = m.state_dict()
  assert list(got.keys()) == list(sd.keys())
  for k in sd:
    assert torch.equal(got[k], sd[k]), k


def test_workspace_is_grow_only_and_parked_while_pinned():
  """TAPIR._workspace: a captured CUDA graph holds raw pointers into these buffers (ADVICE r1), so
  an outgrown buffer is parked, not freed, while a tracker pins the model; the generation counter
  tells graph owners that their capture is stale."""
  m = tapir_model.TAPIR()
  cpu = torch.device('cpu')
  a = m._workspace('mixer', 100, cpu)
  g0 = m._ws_generation
  assert m._workspace('mixer', 50, cpu) is a and m._ws_generation == g0   # reuse, no growth
  m._ws_pins += 1                                                          # a tracker captured
  b = m._workspace('mixer', 1000, cpu)
  assert b is not a and m._ws_generation == g0 + 1
  assert any(t is a for t in m._ws_retired)                                # parked, still alive
  m._ws_pins -= 1
  c = m._workspace('mixer', 5000, cpu)
  assert c is not b and not any(t is b for t in m._ws_retired)             # unpinned: dropped


def test_param_signature_notices_in_place_updates_and_reload():
  m = tapir_model.TAPIR()
  s0 = m._param_sig()
  assert m._param_sig() == s0
  with torch.no_grad():
    next(m.parameters()).add_(1.0)
  s1 = m._param_sig()
  assert s1 != s0
  m.load_state_dict(synth.make_state_dict(1))
  assert m._param_sig() != s1
