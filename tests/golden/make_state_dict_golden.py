#!/usr/bin/env python
"""Record the state-dict layout of the UNMODIFIED reference policies (needs the reference importable through
`oracle/ref_shim.py`).

For each policy class and configuration the state-dict contract tests check, the reference class is instantiated and its
state dict's keys (in order) and shapes are written, with the configuration, to tests/golden/reference_state_dicts.json.
The tests compare `oracle/state_dict_spec.py` against this file, so they run without the reference."""
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

OUT = os.path.join(HERE, "reference_state_dicts.json")


def cases():
    """(entry name, reference class name under vima.policy, config) of every checked layout."""
    from oracle import synth

    out = [(f"VIMAPolicy/{m}", "VIMAPolicy", synth.MODEL_CFGS[m]) for m in ("2M", "20M")]
    out.append(("VIMAGatoPolicy/gato_tiny", "VIMAGatoPolicy", synth.GATO_CFGS["gato_tiny"]))
    out.append(("VIMAGPTPolicy/gato_tiny", "VIMAGPTPolicy", synth.GATO_CFGS["gato_tiny"]))
    out.append(("VIMAFlamingoPolicy/flamingo_tiny", "VIMAFlamingoPolicy", synth.FLAMINGO_CFGS["flamingo_tiny"]))
    return out


def main():
    from oracle import ref_shim

    ref_shim.load_reference()
    policies = sys.modules["vima.policy"]
    entries = []
    for name, cls, cfg in cases():
        sd = getattr(policies, cls)(**cfg).state_dict()
        rows = ",\n".join(json.dumps([k, list(v.shape)]) for k, v in sd.items())  # one key per line: reviewable diffs
        entries.append(f'{json.dumps(name)}: {{"cfg": {json.dumps(dict(cfg))}, "state_dict": [\n{rows}\n]}}')
    with open(OUT, "w") as fh:
        fh.write("{\n" + ",\n".join(entries) + "\n}\n")
    with open(OUT) as fh:
        print("wrote", os.path.basename(OUT), {k: len(v["state_dict"]) for k, v in json.load(fh).items()})


if __name__ == "__main__":
    main()
