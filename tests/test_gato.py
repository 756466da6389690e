"""VIMA-Gato decoder-only baseline (BASELINE.json configs[4]): oracle vs reference golden (CPU), CUDA path vs golden (GPU)."""
import numpy as np
import pytest
import torch

from oracle import detgen, synth, vima_oracle as O
from oracle.state_dict_spec import gato_state_dict_spec
from tests.util import assert_close, golden_pick, load_golden, reference_state_dict, rel_l2

NAME = "gato_small"


def _oracle_sd(model):
    sd = {}
    for k, shape in gato_state_dict_spec(**synth.GATO_CFGS[model]).items():
        w = detgen.weight_for(k, shape)
        if w is not None:
            sd[k] = w
    return sd


def test_gato_oracle_matches_reference_golden():
    case = synth.GATO_CASES[NAME]
    cfg = synth.GATO_CFGS[case.model]
    sd = _oracle_sd(case.model)
    g = load_golden(NAME)
    with torch.no_grad():
        pt, pm = O.gato_forward_prompt_assembly(sd, synth.make_gato_prompt(case))
        ot = O.gato_forward_obs_token(sd, synth.make_gato_obs(case))
        at = O.forward_action_token(sd, synth.make_actions(case, case.T))
        pred = O.gato_policy_forward(sd, ot, at, pt, pm, n_head=cfg["n_head"])
        logits = O.action_decoder_logits(sd, pred[-1:])
        modes = O.action_modes(logits)
    e, a = golden_pick(g, "prompt_masks", pm)
    assert np.array_equal(e, a)
    for key, val in [("prompt_tokens", pt), ("obs_tokens", ot), ("action_tokens", at), ("predicted", pred), ("logits_raw", logits)]:
        e, a = golden_pick(g, key, val)
        assert_close(f"{NAME}.{key}", e, a, 2e-5)
    for k, v in modes.items():
        e, a = golden_pick(g, f"mode.{k}", v)
        assert np.array_equal(e, a)


def test_gato_state_dict_contract():
    import vima_b200

    cfg = synth.GATO_CFGS["gato_tiny"]
    pol = vima_b200.VIMAGatoPolicy(**cfg)
    sd = pol.state_dict()
    spec = gato_state_dict_spec(**cfg)
    assert sorted(sd.keys()) == sorted(spec.keys())
    for k, v in sd.items():
        assert tuple(v.shape) == tuple(spec[k]), k
    # checkpoints written with transformers 4.x also carry the causal buffer: accepted and ignored
    sd2 = dict(sd)
    sd2["transformer.lm.h.0.attn.bias"] = torch.ones(1, 1, 512, 512)
    pol.load_state_dict(sd2, strict=True)


def test_gato_spec_matches_reference():
    cfg = synth.GATO_CFGS["gato_tiny"]
    sd = dict(reference_state_dict("VIMAGatoPolicy/gato_tiny", cfg))
    spec = gato_state_dict_spec(**cfg)
    assert sorted(sd.keys()) == sorted(spec.keys())
    for k, shape in sd.items():
        assert shape == tuple(spec[k]), k


@pytest.mark.gpu
def test_gato_policy_matches_reference_golden():
    import vima_b200
    from vima_b200.utils import DataDict
    from tests.policy_runner import to_dev

    vima_b200.set_precision("f16x3")
    case = synth.GATO_CASES[NAME]
    pol = vima_b200.VIMAGatoPolicy(**synth.GATO_CFGS[case.model])
    detgen.fill_module_(pol)
    pol = pol.cuda().eval()
    g = load_golden(NAME)
    with torch.no_grad():
        tt, wb, ib = synth.make_gato_prompt(case)
        pt, pm = pol.forward_prompt_assembly((tt, wb.cuda(), DataDict(to_dev(ib, "cuda"))))
        ot = pol.forward_obs_token(DataDict(to_dev(synth.make_gato_obs(case), "cuda")))
        at = pol.forward_action_token(to_dev(synth.make_actions(case, case.T), "cuda"))
        pred = pol.forward(obs_token=ot, action_token=at, prompt_token=pt, prompt_token_mask=pm)
        dists = pol.forward_action_decoder(pred[-1:])
        logits = torch.cat([dists[k].raw_logits for k in dists], dim=-1)
    e, a = golden_pick(g, "prompt_masks", pm)
    assert np.array_equal(e, a)
    errs = {}
    for key, val in [("prompt_tokens", pt), ("obs_tokens", ot), ("action_tokens", at), ("predicted", pred), ("logits_raw", logits)]:
        e, a = golden_pick(g, key, val)
        errs[key] = rel_l2(e, a)
    assert max(errs.values()) < 1e-3, errs
    for k in O.ACTION_DIMS:
        e, a = golden_pick(g, f"mode.{k}", dists[k].mode())
        assert np.array_equal(e, a), k
    print(errs)
