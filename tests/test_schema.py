import pytest

from tapnet_b200 import schema


def test_param_counts():
  s = schema.state_dict_schema()
  n = sum(int(__import__('numpy').prod(v)) for v in s.values())
  assert len(s) == 218 and n == 54699335  # SURVEY.md 8(a1)
  s0 = schema.state_dict_schema(0, False)
  assert len(s0) == 188


@pytest.mark.parametrize('kw', [dict(pyramid_level=1), dict(pyramid_level=0, extra_convs=False)])
def test_schema_matches_reference_module(kw, golden):
  """Key order and shapes of the reference module's state_dict, as stored by
  `python -m oracle.make_golden reference_interface`."""
  meta = golden('reference_interface')['meta']
  (tag,) = [t for t, k in meta['schema_kwargs'].items() if k == kw]
  ref = [(name, tuple(shape)) for name, shape in meta['schema'][tag]]
  s = schema.state_dict_schema(kw.get('pyramid_level', 1), kw.get('extra_convs', True))
  assert [name for name, _ in ref] == list(s.keys())
  for k, shape in ref:
    assert shape == s[k], k
