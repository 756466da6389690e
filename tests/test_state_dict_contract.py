"""State-dict contract (SURVEY.md 8(b)): the hand-written spec equals the real reference's (recorded in tests/golden)."""
import pytest


@pytest.mark.parametrize("model", ["2M", "20M"])
def test_spec_matches_reference(model):
    from oracle import synth
    from oracle.state_dict_spec import state_dict_spec
    from tests.util import reference_state_dict

    cfg = synth.MODEL_CFGS[model]
    sd = reference_state_dict(f"VIMAPolicy/{model}", cfg)
    spec = state_dict_spec(**cfg)
    assert [k for k, _ in sd] == list(spec.keys())
    for k, shape in sd:
        assert shape == tuple(spec[k]), k
