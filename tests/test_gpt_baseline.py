"""VIMA-GPT decoder-only baseline (one token per observation; vima/policy/vima_gpt_policy.py): oracle vs reference golden
(CPU), state-dict contract, CUDA path vs golden (GPU)."""
import numpy as np
import pytest
import torch

from oracle import detgen, synth, vima_oracle as O
from oracle.state_dict_spec import gpt_state_dict_spec
from tests.util import assert_close, golden_pick, load_golden, reference_state_dict, rel_l2

NAME = "gpt_small"


def _oracle_sd(model):
    sd = {}
    for k, shape in gpt_state_dict_spec(**synth.GATO_CFGS[model]).items():
        w = detgen.weight_for(k, shape)
        if w is not None:
            sd[k] = w
    return sd


def test_gpt_oracle_matches_reference_golden():
    case = synth.GPT_CASES[NAME]
    cfg = synth.GATO_CFGS[case.model]
    sd = _oracle_sd(case.model)
    g = load_golden(NAME)
    with torch.no_grad():
        pt, pm = O.gpt_forward_prompt_assembly(sd, synth.make_gato_prompt(case))
        ot = O.gpt_forward_obs_token(sd, synth.make_gato_obs(case))
        at = O.forward_action_token(sd, synth.make_actions(case, case.T))
        pred = O.gpt_policy_forward(sd, ot, at, pt, pm, n_head=cfg["n_head"])
        logits = O.action_decoder_logits(sd, pred[-1:])
        modes = O.action_modes(logits)
    assert ot.shape == (case.T, case.B, cfg["embed_dim"]) and pred.shape == ot.shape
    e, a = golden_pick(g, "prompt_masks", pm)
    assert np.array_equal(e, a)
    for key, val in [("prompt_tokens", pt), ("obs_tokens", ot), ("action_tokens", at), ("predicted", pred), ("logits_raw", logits)]:
        e, a = golden_pick(g, key, val)
        assert_close(f"{NAME}.{key}", e, a, 2e-5)
    for k, v in modes.items():
        e, a = golden_pick(g, f"mode.{k}", v)
        assert np.array_equal(e, a)


def test_gpt_state_dict_contract():
    import vima_b200

    cfg = synth.GATO_CFGS["gato_tiny"]
    pol = vima_b200.VIMAGPTPolicy(**cfg)
    sd = pol.state_dict()
    spec = gpt_state_dict_spec(**cfg)
    assert sorted(sd.keys()) == sorted(spec.keys())
    for k, v in sd.items():
        assert tuple(v.shape) == tuple(spec[k]), k
    # the alias package exports it like the reference's vima/policy/__init__.py:1-4 (checked in a fresh interpreter: other
    # tests of this session may have put the real reference under the name `vima`)
    import os
    import subprocess
    import sys

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = ("import vima, vima_b200; assert vima.policy.VIMAGPTPolicy is vima_b200.VIMAGPTPolicy; "
            "assert hasattr(vima.nn, 'MultiViewRGBEncoder') and hasattr(vima.nn, 'ViTEncoderRectangular')")
    subprocess.run([sys.executable, "-c", code], cwd=root, check=True, env={**os.environ, "PYTHONPATH": root})


def test_gpt_spec_matches_reference():
    cfg = synth.GATO_CFGS["gato_tiny"]
    sd = dict(reference_state_dict("VIMAGPTPolicy/gato_tiny", cfg))
    spec = gpt_state_dict_spec(**cfg)
    assert sorted(sd.keys()) == sorted(spec.keys())
    for k, shape in sd.items():
        assert shape == tuple(spec[k]), k


@pytest.mark.gpu
def test_gpt_policy_matches_reference_golden():
    import vima_b200
    from vima_b200.utils import DataDict
    from tests.policy_runner import to_dev

    vima_b200.set_precision("f16x3")
    case = synth.GPT_CASES[NAME]
    pol = vima_b200.VIMAGPTPolicy(**synth.GATO_CFGS[case.model])
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
        feat = pol.obj_encoder(rgb=to_dev(synth.make_gato_obs(case)["rgb"], "cuda"))  # module-level surface: (T,B,2E)
    assert feat.shape == (case.T, case.B, 2 * pol.embed_dim)
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
