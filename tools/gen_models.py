#!/usr/bin/env python3
"""Regenerate data/*.yaml (model INPUTS) from the reference's data directory.

The model inputs are data, not code: the basis description (number of spins, Hamming weight, spin
inversion, symmetry generators) and the Hamiltonian term list (expression + site tuples) of each
of the reference's data/*.yaml, kept verbatim in tests/golden/reference_models/.  This script extracts
that semantic content and re-emits it in a normalised layout (no anchors, no comments, no solver-only
keys such as `observables`, `number_vectors`, `output`, `max_primme_*`), the one tests, bench.py and
smoke() read.  tests/test_host.py (test_model_inputs_equal_the_reference_inputs) re-checks semantic
equality against tests/golden/reference_models/.

Usage:  python tools/gen_models.py [tests/golden/reference_models] [data]
"""
import glob
import os
import sys

import yaml


class _Flow(list):
    pass


def _flow_representer(dumper, data):
    return dumper.represent_sequence("tag:yaml.org,2002:seq", data, flow_style=True)


yaml.add_representer(_Flow, _flow_representer, Dumper=yaml.SafeDumper)


def normalise(conf: dict) -> dict:
    b = conf["basis"]
    basis = {
        "number_spins": int(b["number_spins"]),
        "hamming_weight": b.get("hamming_weight", None),
        "spin_inversion": b.get("spin_inversion", None),
        "symmetries": [
            {"permutation": _Flow(int(v) for v in g["permutation"]), "sector": int(g.get("sector", 0))}
            for g in (b.get("symmetries") or [])
        ],
    }
    terms = []
    for t in conf["hamiltonian"]["terms"]:
        entry = {}
        if "expression" in t:
            entry["expression"] = t["expression"]
        else:
            entry["matrix"] = [_Flow(row) for row in t["matrix"]]
        entry["sites"] = _Flow(_Flow(int(s) for s in tup) for tup in t["sites"])
        terms.append(entry)
    return {"basis": basis, "hamiltonian": {"name": conf["hamiltonian"].get("name", ""), "terms": terms}}


def main():
    root = os.path.join(os.path.dirname(__file__), "..")
    src = sys.argv[1] if len(sys.argv) > 1 else os.path.join(root, "tests", "golden", "reference_models")
    dst = sys.argv[2] if len(sys.argv) > 2 else os.path.join(root, "data")
    os.makedirs(dst, exist_ok=True)
    for path in sorted(glob.glob(os.path.join(src, "*.yaml"))):
        with open(path, "r", encoding="utf-8") as f:
            conf = yaml.safe_load(f)
        out = normalise(conf)
        name = os.path.basename(path)
        with open(os.path.join(dst, name), "w", encoding="utf-8") as f:
            f.write(f"# model input '{name}': normalised by tools/gen_models.py (see its docstring)\n")
            yaml.safe_dump(out, f, allow_unicode=True, sort_keys=False, width=120)
        print("wrote", name)


if __name__ == "__main__":
    main()
