#!/usr/bin/env python
"""bench.py -- policy steps/sec of the VIMA policy forward pass on B200 (contract: see the task statement).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload cfg3|cfg2|cfg3x|cfg5]
                    [--precision f16f8] [--ragged] [--graph] [--dump-outputs DIR]
    python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N ...

One "step" = one policy step for every episode of the batch, exactly as scripts/example.py chains the policy's
public methods with a full-history re-forward (SURVEY.md 8(d)):
    forward_obs_token(new obs) -> forward(T obs steps, T-1 actions, prompt) -> forward_action_decoder(last row)
    -> .mode() -> forward_action_token(action)                       [prompt encode is once per episode: untimed, reported]

Workloads (BASELINE.json configs / SURVEY.md 8(d) rows):
    cfg3  (default, the headline)  VIMA-200M, 256 episodes/GPU, Q=32, Lp=256, T=8 (L=263)           configs[2] / row #3
    cfg2                            VIMA-20M, 64 episodes/GPU, Q=16, Lp=64, T=4 (L=67)               configs[1] / row #2
    cfg3x                           cfg3 with a 512-token prompt through XAttnGPT(xattn_n_positions=512) -- beyond the
                                    reference VIMAPolicy's cap (vima_policy.py:26-38), prompt tokens synthetic  row #3x
    cfg5                            VIMA-Gato 200M (22 layers, decoder-only), 256 episodes/GPU, L=392   configs[4] / row #5

`value`     : device-timed (CUDA events), inputs resident in HBM.
`e2e`       : wall-clock (perf_counter) over the same step through the same public methods, the new observation coming
              from pinned HOST memory (H2D inside the timed region), the action indices read back to the host every step.
`cpu_baseline` / `--impl reference`: the UNMODIFIED reference (oracle/_ref, staged by oracle/make_ref.py; the oracle port
              if it is not staged) on the box's host cores, fixed thread count, a bounded sample of the same workload.
              bench.py runs the same `--impl reference` code in a subprocess, so the two numbers share one code path.
`gpu_eager` : the same unmodified reference in PyTorch eager on the SAME GPU (fp32, and TF32-allowed), full batch, with the
              rel-L2 between its outputs and ours on identical inputs and weights.
`--dump-outputs DIR`: what the last device-timed step returned on rank 0 -- normalised and raw action logits [B, 700] in
              ActionDecoder key order (logits, logits_raw), the action indices per key (mode.<key>, as float64) and the next
              action token (action_token) -- as DIR/<name>.npy.  Inputs and weights are seeded, so two builds run with the same
              arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from dataclasses import replace

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "policy steps/sec (batched action decode)"
# Host threads of the CPU arm: fixed (no search).  torch's CPU GEMMs stop scaling well before the 100+ cores of a GPU
# box and collapse when oversubscribed, so the arm uses min(cores, CPU_THREADS) intra-op threads and says so.
CPU_THREADS = 32


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg3", choices=["cfg3", "cfg2", "cfg3x", "cfg5"])
    ap.add_argument("--precision", default="f16f8")
    ap.add_argument("--batch", type=int, default=0, help="episodes per GPU (default: the workload's)")
    ap.add_argument("--ragged", action="store_true", help="ragged prompts + random object masks (the masked attention branches)")
    ap.add_argument("--graph", action="store_true", help="(default) replay the policy step from a CUDA graph")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel of the step from Python instead of replaying a CUDA graph")
    ap.add_argument("--cpu-episodes", type=int, default=8, help="episodes in the CPU reference sample")
    ap.add_argument("--cpu-threads", type=int, default=0, help="override CPU_THREADS (probing only)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-eager", action="store_true")
    ap.add_argument("--no-incremental", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned (rank 0) as DIR/<name>.npy, for output-by-output comparison of two builds")
    args = ap.parse_args()
    if args.dump_outputs and args.steps < 1:
        ap.error("--dump-outputs needs at least one timed step")
    return args


# ------------------------------------------------------------------------------------------------------------
# workloads
# ------------------------------------------------------------------------------------------------------------
class Workload:
    def __init__(self, name: str, batch: int = 0, ragged: bool = False):
        from oracle import synth

        self.name = name
        self.kind = "gato" if name == "cfg5" else "vima"
        self.xattn_n_positions = None
        self.synthetic_prompt = False
        if name == "cfg5":
            case = synth.GATO_CASES["gato_cfg5"]
            self.cfg = dict(synth.GATO_CFGS[case.model])
            self.model_name = "VIMA-Gato 200M (22 layers, 24 heads, decoder-only)"
        elif name == "cfg3x":
            case = replace(synth.CASES["cfg3"], name="cfg3x", n_words=480, seed=18)  # Lp = 480 + 32 = 512
            self.cfg = dict(synth.MODEL_CFGS[case.model])
            self.xattn_n_positions, self.synthetic_prompt = 512, True
            self.model_name = "VIMA-200M with XAttnGPT(xattn_n_positions=512)"
        else:
            case = synth.CASES[name]
            self.cfg = dict(synth.MODEL_CFGS[case.model])
            self.model_name = f"VIMA-{case.model}"
        if batch:
            case = replace(case, B=batch)
        if ragged:
            case = replace(case, ragged=True)
        self.case = case
        self.E = self.cfg["embed_dim"]
        self.Q = 16 if self.kind == "gato" else case.Q  # Gato: 8 patch tokens per 64x128 view, two views
        self.T, self.Lp = case.T, case.Lp if self.kind == "vima" else case.n_words + case.n_imgs * 16
        self.Ls = self.T * self.Q + self.T - 1
        self.L = self.Ls if self.kind == "vima" else self.Lp + 1 + self.Ls

    def with_batch(self, B: int, seed_shift: int = 0) -> "Workload":
        w = Workload.__new__(Workload)
        w.__dict__.update(self.__dict__)
        w.case = replace(self.case, B=B, seed=self.case.seed + seed_shift)
        return w

    # SURVEY.md 8(d): algorithmic FLOPs (2MNK per GEMM, attention dense incl. the masked half) per episode-step
    def flops_per_episode_step(self) -> float:
        E, L, Lp = self.E, self.L, self.Lp
        heads = 12 * 2 * (512 * E + 512 * 512) + 2 * 512 * 700
        if self.kind == "gato":
            nl = self.cfg["n_layer"]
            dec = nl * (32 * L * E * E + 4 * L * L * E)
            # new observation: 2 views x (patch embed 8 x 3072 x 768 + 4 ViT layers x 24 S W^2) + fusion
            obj = 2 * (2 * 8 * 3072 * 768 + 4 * 24 * 8 * 768 * 768) + 2 * 16 * (E + 2) * E
            return dec + obj + heads
        nl = self.cfg["xf_n_layers"]
        dec = nl * (60 * L * E * E + 4 * Lp * E * E + 4 * L * Lp * E + 4 * L * L * E)
        obj = self.Q * (0.286e9 + 2.4e6 + 2 * 1536 * E)
        return dec + obj + heads

    def describe(self) -> str:
        c = self.case
        extra = ", ragged prompts + random object masks" if c.ragged else ""
        if self.kind == "gato":
            return (f"{self.name}: {self.model_name} policy step (full-history re-forward, one causal sequence prompt|sep|history), "
                    f"{c.B} episodes/GPU, Q={self.Q} image tokens/obs, Lp={self.Lp}, T={self.T} (L={self.L}){extra}")
        return (f"{self.name}: {self.model_name} policy step (full-history re-forward), {c.B} episodes/GPU, Q={self.Q} object tokens, "
                f"Lp={self.Lp} prompt tokens, T={self.T}-step history (L={self.L}){extra}")

    def config(self, world: int) -> dict:
        """Identical for both arms (the driver compares them)."""
        cfg = {"workload": self.describe(), "global_batch": world * self.case.B, "parallelism": f"dp{world}",
               "l2": "inputs larger than L2: activations and packed weights stream from HBM every step (L2 = 126 MB)"}
        if self.name == "cfg3":
            cfg["prompt_len_note"] = ("Lp=256 is BASELINE.md section 4 row #3 / SURVEY 8(d) #3: the reference VIMAPolicy caps prompts at "
                                      "xattn_n_positions=256 (vima_policy.py:26-38); the 512-token prompt is workload cfg3x")
        return cfg


def wrap_dd(DD, x):
    """nested dict -> nested DataDict (the reference's DataDict does not wrap inner dicts itself)."""
    if isinstance(x, dict):
        return DD({k: wrap_dd(DD, v) for k, v in x.items()})
    return x


def to_dev(x, dev, non_blocking=False):
    if isinstance(x, dict):
        return {k: to_dev(v, dev, non_blocking) for k, v in x.items()}
    return x.to(dev, non_blocking=non_blocking)


def pin(x):
    if isinstance(x, dict):
        return {k: pin(v) for k, v in x.items()}
    return x.pin_memory()


def nbytes(x):
    if isinstance(x, dict):
        return sum(nbytes(v) for v in x.values())
    return x.numel() * x.element_size()


def host_inputs(wl: Workload):
    """Seeded CPU tensors of one rank: history observations, past actions, the new observation."""
    from oracle import synth

    c = wl.case
    if wl.kind == "gato":
        return dict(hist=synth.make_gato_obs(c, T=c.T - 1, tag="hist"), acts=synth.make_actions(c, c.T), new=synth.make_gato_obs(c, T=1, tag="new"))
    return dict(hist=synth.make_obs(c, T=c.T - 1, tag="hist"), acts=synth.make_actions(c, c.T), new=synth.make_obs(c, T=1, tag="new"))


def synthetic_prompt(wl: Workload, dev):
    from oracle import detgen

    c = wl.case
    tok = detgen.uniform(f"bench.prompt.{wl.name}", (wl.Lp, c.B, wl.E), c.seed).to(dev)
    msk = torch.ones(c.B, wl.Lp, dtype=torch.bool, device=dev)
    if c.ragged:  # valid length ~U[Lp/2, Lp], episode 0 full
        n = detgen.randint(f"bench.prompt_len.{wl.name}", (c.B,), wl.Lp // 2, wl.Lp + 1, c.seed).to(dev)
        n[0] = wl.Lp
        msk = torch.arange(wl.Lp, device=dev)[None, :] < n[:, None]
    return tok, msk


class Stepper:
    """The policy step of scripts/example.py:125-198 over any object with the reference's public policy API (ours or the
    reference's own class, on any device)."""

    def __init__(self, policy, DD, wl: Workload, dev, inputs, prompt_tokens, prompt_masks):
        self.policy, self.DD, self.wl, self.dev = policy, DD, wl, dev
        self.gato = wl.kind == "gato"
        self.prompt_tokens, self.prompt_masks = prompt_tokens, prompt_masks
        hist = wrap_dd(DD, to_dev(inputs["hist"], dev))
        if self.gato:
            self.h_tok, self.h_msk = policy.forward_obs_token(hist), None
        else:
            self.h_tok, self.h_msk = policy.forward_obs_token(hist)
        self.a_tok = policy.forward_action_token(to_dev(inputs["acts"], dev))
        self.last_pred = None

    def __call__(self, obs_dev):
        p = self.policy
        if self.gato:
            n_tok = p.forward_obs_token(wrap_dd(self.DD, obs_dev))
            pred = p.forward(obs_token=torch.cat([self.h_tok, n_tok], dim=0), action_token=self.a_tok, prompt_token=self.prompt_tokens,
                             prompt_token_mask=self.prompt_masks)
        else:
            n_tok, n_msk = p.forward_obs_token(wrap_dd(self.DD, obs_dev))
            pred = p.forward(obs_token=torch.cat([self.h_tok, n_tok], dim=0), obs_mask=torch.cat([self.h_msk, n_msk], dim=0),
                             action_token=self.a_tok, prompt_token=self.prompt_tokens, prompt_token_mask=self.prompt_masks)
        self.last_pred = pred[-1:]
        dists = p.forward_action_decoder(pred[-1:])
        modes = {k: v.mode() for k, v in dists.items()}
        nxt = p.forward_action_token({k: v.clone() for k, v in modes.items()})
        return dists, modes, nxt


def raw_logits(dists) -> torch.Tensor:
    """[B, 700] un-normalised head outputs in ActionDecoder key order (ours expose them; the all-gather payload)."""
    return torch.cat([dists[k].raw_logits for k in dists], dim=-1).reshape(-1, 700).contiguous()


def norm_logits(dists) -> torch.Tensor:
    return torch.cat([d.logits for k in dists for d in dists[k]._dists], dim=-1).reshape(-1, 700)


DUMP_LIMIT_BYTES = 64 << 20


def step_outputs(dists, modes, nxt) -> dict:
    """What one policy step hands its caller, as host arrays: name -> (float32/float64 array, episode axis)."""
    out = {"logits": (norm_logits(dists).float().cpu().numpy(), 0), "logits_raw": (raw_logits(dists).float().cpu().numpy(), 0),
           "action_token": (nxt.float().cpu().numpy(), 1)}
    for k, v in modes.items():  # action indices, exact in float64
        out[f"mode.{k}"] = (v.cpu().numpy().astype("float64"), 1)
    return out


def dump_outputs(path: str, outputs: dict) -> None:
    """Writes path/<name>.npy.  Above DUMP_LIMIT_BYTES in all, every array keeps the same fixed, seeded sample of episodes
    (listed in episodes.npy), so that two runs with the same arguments still compare element for element."""
    import numpy as np

    total = sum(a.nbytes for a, _ in outputs.values())
    budget = DUMP_LIMIT_BYTES - 4096 * (len(outputs) + 1)  # .npy headers
    if total > budget:
        a0, ax0 = next(iter(outputs.values()))
        n_ep = a0.shape[ax0]
        per_episode = total / n_ep + 8  # + its float64 entry in episodes.npy
        keep = np.sort(np.random.default_rng(0).choice(n_ep, max(1, int(budget // per_episode)), replace=False))
        outputs = {k: (np.take(a, keep, axis=ax), ax) for k, (a, ax) in outputs.items()}
        outputs["episodes"] = (keep.astype("float64"), 0)
    os.makedirs(path, exist_ok=True)
    for k, (a, _) in outputs.items():
        np.save(os.path.join(path, f"{k}.npy"), a)


# ------------------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------------------
def sample_clocks(stop_evt, out):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    dev = os.environ.get("LOCAL_RANK", "0")
    try:
        pr = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", dev],
                              stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
    except Exception:
        return
    out["proc"] = pr

    def rd():
        for line in pr.stdout:
            out.setdefault("lines", []).append(line.strip())

    t = threading.Thread(target=rd, daemon=True)
    t.start()
    stop_evt.wait()
    pr.terminate()
    t.join(timeout=2)


def summarise_clocks(lines):
    sm, mx, reasons = [], [], set()
    for ln in lines or []:
        f = [x.strip() for x in ln.split(",")]
        if len(f) < 7:
            continue
        try:
            sm.append(float(f[0])); mx.append(float(f[1]))
        except ValueError:
            continue
        for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[3:7]):
            if v.lower().startswith("active"):
                reasons.add(name)
    if not sm:
        return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
    return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------------------------
# reference arm: the unmodified reference (oracle/_ref) on host cores; the oracle port when it is not staged
# ------------------------------------------------------------------------------------------------------------
def build_reference_policy(wl: Workload, dev):
    """The reference's own policy class, filled with the shared deterministic weights. Returns (policy, DataDict)."""
    from oracle import detgen
    from oracle.ref_shim import load_reference

    ref = load_reference()
    DD = sys.modules["vima.utils"].DataDict
    torch.manual_seed(0)
    if wl.kind == "gato":
        pol = ref.VIMAGatoPolicy(**wl.cfg)
    else:
        pol = ref.VIMAPolicy(**wl.cfg)
        if wl.xattn_n_positions is not None:  # cfg3x: same decoder class with the longer cross-attention position table
            import vima.nn as rnn

            pol.xattn_gpt = rnn.XAttnGPT(wl.E, n_layer=wl.cfg["xf_n_layers"], n_head=wl.cfg["sattn_n_heads"], dropout=0.1,
                                         xattn_n_head=wl.cfg["xattn_n_heads"], xattn_ff_expanding=4, xattn_n_positions=wl.xattn_n_positions,
                                         use_geglu=True)
    detgen.fill_module_(pol)
    return pol.to(dev).eval(), DD


def cpu_threads(args) -> int:
    return max(1, min(os.cpu_count() or 1, args.cpu_threads or CPU_THREADS))


def cpu_reference_steps(args, wl: Workload, n_episodes: int, warm: int, reps: int):
    """-> (seconds per step list, kind). One step = n_episodes policy steps on the CPU."""
    from oracle.ref_shim import reference_available

    torch.set_num_threads(cpu_threads(args))
    w = wl.with_batch(n_episodes)
    dev = torch.device("cpu")
    times = []
    with torch.no_grad():
        if reference_available():
            kind = "reference"
            pol, DD = build_reference_policy(w, dev)
            ptok, pmsk = synthetic_prompt(w, dev)
            inp = host_inputs(w)
            st = Stepper(pol, DD, w, dev, inp, ptok, pmsk)
            new = inp["new"]
            fn = lambda: st(new)
        else:  # the oracle restatement (VIMAPolicy workloads only)
            kind = "port"
            if w.kind != "vima" or w.xattn_n_positions:
                raise RuntimeError("the staged reference (oracle/_ref) is missing and the oracle port only covers the VIMAPolicy workloads")
            fn = _oracle_port_step(w)
        for i in range(warm + reps):
            t0 = time.perf_counter()
            fn()
            dt = time.perf_counter() - t0
            if i >= warm:
                times.append(dt)
    return times, kind


def _oracle_port_step(w: Workload):
    from oracle import detgen, synth, vima_oracle as O
    from oracle.state_dict_spec import state_dict_spec

    case, cfg = w.case, w.cfg
    skip = ("t5_prompt_encoder", "prompt_embedding", "prompt_obj_post_layer")  # prompt encode is outside the step
    sd = {}
    for k, shape in state_dict_spec(**cfg).items():
        if not k.startswith(skip):
            v = detgen.weight_for(k, shape)
            if v is not None:
                sd[k] = v
    ptok, pmsk = synthetic_prompt(w, torch.device("cpu"))
    hist = synth.make_obs(case, T=case.T - 1, tag="hist")
    h_tok, h_msk = O.forward_obs_token(sd, hist)
    a_tok = O.forward_action_token(sd, synth.make_actions(case, case.T))
    new_obs = synth.make_obs(case, T=1, tag="new")
    return lambda: O.policy_step(sd, obs=new_obs, history_obs_tokens=h_tok, history_obs_masks=h_msk, history_action_tokens=a_tok,
                                 prompt_tokens=ptok, prompt_masks=pmsk, n_head=cfg["sattn_n_heads"], xattn_n_head=cfg["xattn_n_heads"])


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", "1"))
    wl = Workload(args.workload, args.batch, args.ragged)
    n_ep = args.cpu_episodes
    t0 = time.perf_counter()
    times, kind = cpu_reference_steps(args, wl, n_ep, max(args.warmup, 1), max(args.steps, 1))
    ms = statistics.median(times) * 1e3
    val = n_ep / (ms / 1e3)
    spread = (max(times) - min(times)) / statistics.median(times)
    what = "the unmodified reference (oracle/_ref, vima.policy public API)" if kind == "reference" else "the oracle port (oracle/vima_oracle.py)"
    sample = (f"{n_ep} episodes x {len(times)} timed steps (median; spread {spread:.2f}) of {args.workload} (L={wl.L}, Lp={wl.Lp}) on {what}, "
              f"torch fp32, {torch.get_num_threads()} intra-op threads of {os.cpu_count()} logical cores, prompt tokens synthetic")
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": "steps/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": wl.config(world),
        "cpu_baseline": {"value": val, "unit": "steps/s", "cores": torch.get_num_threads(), "kind": kind, "sample": sample},
        "e2e": {"value": val, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "step_seconds": times, "wall_s": time.perf_counter() - t0,
    }
    print(json.dumps(line), flush=True)


def cpu_baseline_start(args):
    """Starts `bench.py --impl reference` (the code the driver's reference arm runs) in a fresh process: one code path, one number.
    The child sees no GPU and uses its own fixed thread count; it runs while this process does the GPU-resident `gpu_eager` leg (whose
    host side is confined to a few threads meanwhile), which takes about a minute off the default run."""
    cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--workload", args.workload, "--steps", "5", "--warmup", "2",
           "--cpu-episodes", str(args.cpu_episodes)] + (["--ragged"] if args.ragged else []) + (["--batch", str(args.batch)] if args.batch else []) \
        + (["--cpu-threads", str(args.cpu_threads)] if args.cpu_threads else [])
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")}
    env["CUDA_VISIBLE_DEVICES"] = ""
    try:
        return subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, env=env)
    except Exception as e:  # noqa: BLE001
        return {"error": repr(e)[:400]}


def cpu_baseline_collect(proc):
    if isinstance(proc, dict):
        return proc
    try:
        out, err = proc.communicate(timeout=900)
        for ln in reversed(out.strip().splitlines()):
            if ln.startswith("{"):
                return json.loads(ln)["cpu_baseline"]
        return {"error": (err or out)[-400:]}
    except Exception as e:  # noqa: BLE001
        proc.kill()
        return {"error": repr(e)[:400]}


# ------------------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------------------
class GemmTimer:
    """Wraps Context.gemm with CUDA events on the launching stream: per-launch durations + algorithmic FLOPs."""

    def __init__(self, ctx):
        self.ctx, self.orig, self.rec, self.on = ctx, ctx.gemm, [], False

        def timed(**kw):
            if not self.on:
                return self.orig(**kw)
            e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
            e0.record()
            self.orig(**kw)
            e1.record()
            n_eff = kw["N"]
            self.rec.append((e0, e1, 2.0 * kw["M"] * n_eff * kw["K"], (kw["M"], kw["N"], kw["K"])))

        ctx.gemm = timed

    def summary(self):
        tot_ms = sum(a.elapsed_time(b) for a, b, _, _ in self.rec)
        tot_fl = sum(f for _, _, f, _ in self.rec)
        return tot_ms, tot_fl, len(self.rec)


def build_our_policy(wl: Workload, dev):
    import vima_b200
    from oracle import detgen

    if wl.kind == "gato":
        pol = vima_b200.VIMAGatoPolicy(**wl.cfg)
    else:
        pol = vima_b200.VIMAPolicy(**wl.cfg)
        if wl.xattn_n_positions is not None:
            from vima_b200 import nn as vnn

            pol.xattn_gpt = vnn.XAttnGPT(wl.E, n_layer=wl.cfg["xf_n_layers"], n_head=wl.cfg["sattn_n_heads"], dropout=0.1,
                                         xattn_n_head=wl.cfg["xattn_n_heads"], xattn_ff_expanding=4, xattn_n_positions=wl.xattn_n_positions,
                                         use_geglu=True)
    detgen.fill_module_(pol)
    return pol.to(dev).eval()


def encode_prompt(policy, wl: Workload, dev):
    """-> (prompt_tokens, prompt_masks, ms per batch | None). Once per episode: outside the step."""
    from oracle import synth
    from vima_b200.utils import DataDict

    if wl.synthetic_prompt:
        tok, msk = synthetic_prompt(wl, dev)
        return tok, msk, None
    prompt = synth.make_gato_prompt(wl.case) if wl.kind == "gato" else synth.make_prompt(wl.case)
    pr_in = (prompt[0], prompt[1].to(dev), DataDict(to_dev(prompt[2], dev)))
    policy.forward_prompt_assembly(pr_in)  # warm (weight packing)
    torch.cuda.synchronize()
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    torch.cuda.nvtx.range_push("prompt")  # ncu --nvtx-include "prompt/": the once-per-episode prompt encode on its own
    e0.record()
    tok, msk = policy.forward_prompt_assembly(pr_in)
    e1.record(); torch.cuda.synchronize()
    torch.cuda.nvtx.range_pop()
    return tok, msk, e0.elapsed_time(e1)


def gpu_eager_leg(wl: Workload, dev, inputs, prompt_tokens, prompt_masks, our_pred, our_logits_norm, our_modes, new_obs_dev):
    """The unmodified reference in PyTorch eager on this GPU: fp32 and TF32-allowed, same batch, same inputs and weights."""
    from oracle.ref_shim import reference_available

    if not reference_available():
        return {"unavailable": "oracle/_ref is not staged"}
    out = {}
    pol, DD = build_reference_policy(wl, dev)
    with torch.no_grad():
        st = Stepper(pol, DD, wl, dev, inputs, prompt_tokens.contiguous(), prompt_masks)
        for mode, tf32 in (("fp32", False), ("tf32", True)):
            torch.backends.cuda.matmul.allow_tf32 = tf32
            torch.backends.cudnn.allow_tf32 = tf32
            for _ in range(2):
                dists, modes, _ = st(new_obs_dev)
            torch.cuda.synchronize()
            ts = []
            for _ in range(3):
                e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
                e0.record()
                dists, modes, _ = st(new_obs_dev)
                e1.record(); torch.cuda.synchronize()
                ts.append(e0.elapsed_time(e1))
            ms = statistics.median(ts)
            ref_pred = st.last_pred.float()
            ref_ln = norm_logits(dists).float()
            rl2 = lambda a, b: float((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30))
            agree = [float((modes[k] == our_modes[k]).float().mean()) for k in modes]
            out[mode] = {"ms_per_step": ms, "value": wl.case.B / (ms / 1e3), "unit": "steps/s",
                         "ours_vs_this_rel_l2": {"predicted_token": rl2(our_pred, ref_pred), "normalised_logits": rl2(our_logits_norm, ref_ln)},
                         "action_index_agreement": min(agree)}
        torch.backends.cuda.matmul.allow_tf32 = False
        torch.backends.cudnn.allow_tf32 = False
    out["what"] = ("unmodified reference (oracle/_ref) through its public policy API, PyTorch eager on the same GPU, same "
                   f"{wl.case.B}-episode batch, same weights/inputs; 3 timed steps (median) after 2 warm-ups")
    del st, pol
    torch.cuda.empty_cache()
    return out


def run_ours(args):
    import torch.distributed as dist

    import vima_b200
    from vima_b200 import _C
    from vima_b200.dist import all_gather_logits
    from vima_b200.utils import DataDict

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    vima_b200.set_precision(args.precision)
    wl0 = Workload(args.workload, args.batch, args.ragged)
    wl = wl0.with_batch(wl0.case.B, seed_shift=rank)  # independent episodes per rank
    B, T, Q = wl.case.B, wl.T, wl.Q
    t_setup = time.perf_counter()
    policy = build_our_policy(wl, dev)
    ctx = _C.Context.get(dev)

    with torch.no_grad():
        prompt_tokens, prompt_masks, prompt_ms = encode_prompt(policy, wl, dev)
        inputs = host_inputs(wl)
        step = Stepper(policy, DataDict, wl, dev, inputs, prompt_tokens, prompt_masks)
        new_obs_host = pin(inputs["new"])
        new_obs_dev = to_dev(new_obs_host, dev)
        gathered = torch.empty((world * B, 700), dtype=torch.float32, device=dev) if world > 1 else None

        use_graph = not args.no_graph
        policy_step = step
        graph_note = None
        if use_graph:  # the policy step (static shapes) is captured once and replayed; a failed capture falls back to eager launches
            from vima_b200.graphs import GraphedStep

            try:
                policy_step = GraphedStep(step, new_obs_dev, warmup=max(args.warmup, 3))
                graph_note = policy_step.describe()
            except Exception as e:  # noqa: BLE001
                use_graph, policy_step = False, step
                graph_note = {"capture_failed": repr(e)[:300], "note": "fell back to per-kernel launches"}
                torch.cuda.synchronize()

        def make_full_step(inner):
            def full_step(obs_dev):
                dists, modes, nxt = inner(obs_dev)
                if world > 1:  # the path's one exchange: all-gather of the action logits over NVLink (outside the graph)
                    all_gather_logits(raw_logits(dists), out=gathered)
                return dists, modes, nxt
            return full_step

        full_step = make_full_step(step)       # eager launches (instrumented GEMM pass, checks)
        run_step = make_full_step(policy_step)  # what the timed regions run

        def barrier():
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()

        gt = GemmTimer(ctx)
        for _ in range(max(args.warmup, 3)):
            run_step(new_obs_dev)
        barrier()
        setup_s = time.perf_counter() - t_setup

        # ---- timed: device-resident inputs ----
        stop = threading.Event(); clk = {}
        th = threading.Thread(target=sample_clocks, args=(stop, clk), daemon=True); th.start()
        time.sleep(0.3)
        launches0 = ctx.launches
        gt.on = not use_graph
        barrier()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        torch.cuda.nvtx.range_push("timed")
        e0.record()
        for _ in range(args.steps):
            last = run_step(new_obs_dev)
        e1.record()
        barrier()
        torch.cuda.nvtx.range_pop()
        gt.on = False
        if args.dump_outputs and rank == 0:  # now: the replays below overwrite the graph's static outputs
            dump_outputs(args.dump_outputs, step_outputs(*last))
        ms_total = e0.elapsed_time(e1)
        launches = ctx.launches - launches0
        if use_graph:
            launches = policy_step.kernels_per_replay * args.steps
        gemm_ms, gemm_fl, n_gemm = gt.summary()
        gemm_region_ms = ms_total
        if use_graph:
            # per-launch events cannot be recorded inside a replayed graph: the GEMM launches are timed in a second region of the
            # same K steps launched kernel by kernel (same kernels, same order, same stream); share_of_step refers to that region
            full_step(new_obs_dev)  # untimed: the eager path's buffers come from this stream's allocator pool from here on
            barrier()
            gt.on = True
            e2 = torch.cuda.Event(enable_timing=True); e3 = torch.cuda.Event(enable_timing=True)
            e2.record()
            for _ in range(args.steps):
                full_step(new_obs_dev)
            e3.record()
            barrier()
            gt.on = False
            gemm_region_ms = e2.elapsed_time(e3)
            gemm_ms, gemm_fl, n_gemm = gt.summary()

        # ---- timed: end to end, wall clock (pinned host obs -> device, action indices -> host, every step) ----
        h2d = nbytes(new_obs_host)
        d2h = 0
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            if use_graph:  # pinned host -> the graph's static input buffers (no intermediate device copy)
                obs_d = policy_step.load_inputs(new_obs_host)
            else:
                obs_d = to_dev(new_obs_host, dev, non_blocking=True)
            _, modes, _ = run_step(obs_d)
            host_modes = {k: v.cpu() for k, v in modes.items()}  # blocking read of the step's result
            d2h = sum(v.numel() * v.element_size() for v in host_modes.values())
        torch.cuda.synchronize()
        e2e_ms_total = (time.perf_counter() - t0) * 1e3
        barrier()
        stop.set(); th.join(timeout=3)

        # ---- on hardware: the gathered logits are what each rank computed (bit for bit) ----
        gather_check = None
        dists, modes, _ = full_step(new_obs_dev)
        our_pred = step.last_pred.float().clone()
        our_ln = norm_logits(dists).float().clone()
        our_modes = {k: v.clone() for k, v in modes.items()}
        if world > 1:
            mine = raw_logits(dists)
            own_ok = bool(torch.equal(gathered[rank * B:(rank + 1) * B], mine))
            ok_t = torch.tensor([1.0 if own_ok else 0.0], device=dev)
            dist.all_reduce(ok_t, op=dist.ReduceOp.MIN)
            gather_check = {"every_rank_finds_its_own_logits_in_its_slice_bit_exact": bool(ok_t.item() == 1.0)}
            if rank == 0:  # rank 1's episodes recomputed here from the same seed must equal rank 1's gathered slice
                wl1 = wl0.with_batch(B, seed_shift=1)
                pt1, pm1, _ = encode_prompt(policy, wl1, dev)
                st1 = Stepper(policy, DataDict, wl1, dev, host_inputs(wl1), pt1, pm1)
                d1, _, _ = st1(to_dev(host_inputs(wl1)["new"], dev))
                gather_check["rank1_slice_equals_single_gpu_recompute_bit_exact"] = bool(torch.equal(gathered[B:2 * B], raw_logits(d1)))
                del st1

        # ---- separately reported (SURVEY.md 8(d)): the same T-step episode decoded step by step through the K/V cache ----
        incr_ms = None
        if wl.kind == "vima" and not args.no_incremental:
            n_tok, n_msk = policy.forward_obs_token(DataDict(new_obs_dev))
            all_tok = torch.cat([step.h_tok, n_tok], dim=0)
            all_msk = torch.cat([step.h_msk, n_msk], dim=0)
            for rep in range(2):  # first repetition warms the allocator
                barrier()
                e4 = torch.cuda.Event(enable_timing=True); e5 = torch.cuda.Event(enable_timing=True)
                e4.record()
                cache = policy.start_decode(prompt_tokens, prompt_masks, max_tokens=T * (Q + 1) - 1)
                for t in range(T):
                    pred_t = policy.forward_step(cache, all_tok[t:t + 1], all_msk[t:t + 1], None if t == 0 else step.a_tok[t - 1:t])
                    policy.forward_action_token({k: v.mode() for k, v in policy.forward_action_decoder(pred_t).items()})
                e5.record(); barrier()
                incr_ms = e4.elapsed_time(e5)
                del cache

        # ---- the reference on the host cores (child process, no GPU), started now so that it overlaps the eager leg below ----
        cpu_proc = None
        if not args.no_cpu_baseline and world == 1:
            cpu_proc = cpu_baseline_start(args)
            torch.set_num_threads(4)  # this process's host work from here on is set-up code; the child owns its 32 threads

        # ---- same-GPU comparator: the unmodified reference in PyTorch eager (rank 0, N=1 only) ----
        eager = None
        if world == 1 and not args.no_gpu_eager:
            try:
                eager = gpu_eager_leg(wl, dev, inputs, prompt_tokens, prompt_masks, our_pred, our_ln, our_modes, new_obs_dev)
            except Exception as e:  # noqa: BLE001  (a reported baseline must not take the bench line down)
                eager = {"error": repr(e)[:500]}
                torch.cuda.empty_cache()

    def gather_floats(x):
        if world == 1:
            return [x]
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        outl = [torch.zeros_like(t) for _ in range(world)]
        dist.all_gather(outl, t)
        return [float(o.item()) for o in outl]

    per_rank_ms = gather_floats(ms_total / args.steps)
    per_rank_e2e = gather_floats(e2e_ms_total / args.steps)
    per_rank_gemm = gather_floats(gemm_ms / args.steps)
    ms_step = max(per_rank_ms)
    e2e_ms_step = max(per_rank_e2e)
    if incr_ms is not None:
        incr_ms = max(gather_floats(incr_ms))
    value = world * B / (ms_step / 1e3)
    e2e_value = world * B / (e2e_ms_step / 1e3)

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak_tf = peaks.get("bf16_tflops_sustained") or 1400.0  # the GEMMs run inside a long step -> sustained figure
        peak_src = "MEASURED_PEAKS.json bf16_tflops_sustained (of measured)" if peaks else "B200_PROFILING.md fallback 1.4 PF sustained (of fallback)"
        step_flops = wl.flops_per_episode_step() * B
        roof = {"bound": "tensor", "peak": peak_tf, "unit": "TFLOP/s", "kernel": "gemm_tc_kernel (tcgen05)", "peak_source": peak_src,
                "traffic": None, "traffic_note": "per-launch dram bytes of every kernel of the step: profiles/r2_kernel_metrics_step.txt (ncu)",
                "step_algorithmic_tflop": step_flops / 1e12, "step_tflops": step_flops / (ms_step / 1e3) / 1e12,
                "step_frac_of_peak": step_flops / (ms_step / 1e3) / 1e12 / peak_tf,
                "note": ("achieved = sum(2MNK) / sum(t) over every gemm_tc_kernel launch of the timed region (CUDA events on the launching stream); "
                         "in *x3 modes every product is 3 tensor passes, in f16f8 1 fp16 + 2 fp8 passes = 2 pass-equivalents")}
        if gemm_ms > 0:
            achieved = gemm_fl / (gemm_ms / 1e3) / 1e12
            roof.update({"achieved": achieved, "frac": achieved / peak_tf, "launches_per_step": n_gemm / args.steps,
                         "share_of_step": (gemm_ms / args.steps) / (ms_total / args.steps)})
            if use_graph:
                roof["timed_in"] = ("a second region of the same K steps launched kernel by kernel (events cannot be recorded inside the "
                                    f"replayed graph): {gemm_region_ms / args.steps:.3f} ms/step there vs {ms_step:.3f} ms/step replayed; "
                                    "share_of_step = GEMM device time per step / replayed step time (same kernels, same order)")
        else:  # graph replay: no per-launch events; the whole step against the peak
            roof.update({"achieved": roof["step_tflops"], "frac": roof["step_frac_of_peak"],
                         "note": roof["note"] + "; CUDA-graph replay: per-launch events unavailable, achieved = whole-step algorithmic rate"})
        dtype_txt = {"f16x3": "f16 hi/lo operand pairs (3-term products, fp32-equivalent), fp32 accumulate/softmax/LN",
                     "bf16x3": "bf16 hi/lo operand pairs (3-term), fp32 accumulate", "f16": "f16 operands, fp32 accumulate",
                     "bf16": "bf16 operands, fp32 accumulate",
                     "f16f8": "f16 hi*hi + e4m3 cross terms (2 tensor pass-equivalents), f16 3-term in attention, fp32 accumulate/softmax/LN"}[args.precision]
        line = {
            "metric": METRIC, "value": value, "unit": "steps/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": dtype_txt, "data": "synthetic",
            "config": wl0.config(world),
            "precision_mode": args.precision,
            "e2e": {"value": e2e_value, "unit": "steps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms_step,
                    "timer": "time.perf_counter around the loop (blocking .cpu() of the action indices every step)"},
            "gpu_launches": int(launches),
            "clocks": summarise_clocks(clk.get("lines")),
            "roofline": roof,
            "per_rank": {"ms_per_step": per_rank_ms, "e2e_ms_per_step": per_rank_e2e, "gemm_ms_per_step": per_rank_gemm},
            "setup_s": setup_s,
        }
        if prompt_ms is not None:
            line["prompt_encode"] = {"ms_per_batch": prompt_ms,
                                     "steps_per_s_with_prompt_amortised": world * B * T / ((prompt_ms + T * ms_step) / 1e3)}
        if graph_note:
            line["cuda_graph"] = graph_note
        if gather_check is not None:
            line["gather_check"] = gather_check
        if incr_ms is not None:
            line["incremental"] = {"value": world * B * T / (incr_ms / 1e3), "unit": "env steps/s", "episode_ms": incr_ms,
                                   "note": f"not the graded metric: {T}-step episode decoded through the K/V cache (start_decode/forward_step, "
                                           "decoder + heads + action embed per step; obs tokens precomputed); same predictions as the full re-forward"}
        if eager is not None:
            line["gpu_eager"] = eager
        if cpu_proc is not None:
            line["cpu_baseline"] = cpu_baseline_collect(cpu_proc)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
