"""VIMA-Flamingo baseline (XAttnGPT decoder over Perceiver-resampled image tokens; vima/policy/vima_flamingo_policy.py):
oracle vs reference golden and vs HF's PerceiverModel (CPU), state-dict contract, CUDA path vs golden (GPU)."""
import numpy as np
import pytest
import torch

from oracle import detgen, synth, vima_oracle as O
from oracle.state_dict_spec import flamingo_state_dict_spec
from tests.util import assert_close, golden_pick, load_golden, reference_state_dict, rel_l2

NAME = "flamingo_small"


def _oracle_sd(model):
    sd = {}
    for k, shape in flamingo_state_dict_spec(**synth.FLAMINGO_CFGS[model]).items():
        w = detgen.weight_for(k, shape)
        if w is not None:
            sd[k] = w
    return sd


def test_perceiver_oracle_matches_hf_model():
    """The resampler is third-party code (transformers PerceiverModel, unpinned by the reference): restatement == library."""
    pm = pytest.importorskip("transformers.models.perceiver.modeling_perceiver")
    torch.manual_seed(0)
    E = 64
    cfg = pm.PerceiverConfig(d_model=E, d_latents=E, num_latents=4, num_blocks=4, num_self_attends_per_block=4, num_self_attention_heads=8,
                             num_cross_attention_heads=8, attention_probs_dropout_prob=0.1)
    m = pm.PerceiverModel(cfg).eval()
    for p_ in m.parameters():
        torch.nn.init.normal_(p_, std=0.1)
    x = torch.randn(3, 16, E)
    with torch.no_grad():
        ref = m(inputs=x, attention_mask=torch.ones(3, 16, dtype=torch.bool)).last_hidden_state
        got = O.perceiver_forward({"pc.model." + k: v for k, v in m.state_dict().items()}, "pc.", x)
    assert rel_l2(ref, got) < 1e-6


def test_flamingo_oracle_matches_reference_golden():
    case = synth.FLAMINGO_CASES[NAME]
    cfg = synth.FLAMINGO_CFGS[case.model]
    sd = _oracle_sd(case.model)
    g = load_golden(NAME)
    with torch.no_grad():
        pt, pm = O.flamingo_forward_prompt_assembly(sd, synth.make_gato_prompt(case))
        ot = O.flamingo_forward_obs_token(sd, synth.make_gato_obs(case))
        at = O.forward_action_token(sd, synth.make_actions(case, case.T))
        pred = O.flamingo_policy_forward(sd, ot, at, pt, pm, n_head=cfg["dt_n_heads"], xattn_n_head=cfg["xattn_n_heads"])
        logits = O.action_decoder_logits(sd, pred[-1:])
        modes = O.action_modes(logits)
    assert ot.shape == (case.T, case.B, 4, cfg["embed_dim"])
    e, a = golden_pick(g, "prompt_masks", pm)
    assert np.array_equal(e, a)
    for key, val in [("prompt_tokens", pt), ("obs_tokens", ot), ("action_tokens", at), ("predicted", pred), ("logits_raw", logits)]:
        e, a = golden_pick(g, key, val)
        assert_close(f"{NAME}.{key}", e, a, 2e-5)
    for k, v in modes.items():
        e, a = golden_pick(g, f"mode.{k}", v)
        assert np.array_equal(e, a)


def test_flamingo_state_dict_contract():
    import vima_b200

    cfg = synth.FLAMINGO_CFGS["flamingo_tiny"]
    pol = vima_b200.VIMAFlamingoPolicy(**cfg)
    sd = pol.state_dict()
    spec = flamingo_state_dict_spec(**cfg)
    assert sorted(sd.keys()) == sorted(spec.keys())
    for k, v in sd.items():
        assert tuple(v.shape) == tuple(spec[k]), k


def test_flamingo_spec_matches_reference():
    cfg = synth.FLAMINGO_CFGS["flamingo_tiny"]
    sd = dict(reference_state_dict("VIMAFlamingoPolicy/flamingo_tiny", cfg))
    spec = flamingo_state_dict_spec(**cfg)
    assert sorted(sd.keys()) == sorted(spec.keys())
    for k, shape in sd.items():
        assert shape == tuple(spec[k]), k


@pytest.mark.gpu
def test_flamingo_policy_matches_reference_golden():
    import vima_b200
    from vima_b200.utils import DataDict
    from tests.policy_runner import to_dev

    vima_b200.set_precision("f16x3")
    case = synth.FLAMINGO_CASES[NAME]
    pol = vima_b200.VIMAFlamingoPolicy(**synth.FLAMINGO_CFGS[case.model])
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
