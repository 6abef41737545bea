"""Writes tests/golden/fzn/: small FlatZinc models and, in pins.json, what the front-end builds of each (sha256 of the
TNF network) and the optimum found by brute force over the FlatZinc semantics.  tests/test_frontend.py rebuilds the
networks from the stored models and checks them against the pins, so a change of the front-end's output is seen.

  python tests/golden/make_frontend_pins.py

The models come from the seeded generators of tests/test_frontend.py (plain integer / Boolean models and set
variables) plus the syntax-subset model; they are stored as text so that the pins do not depend on a random generator.
"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from tests import test_frontend as tf  # noqa: E402
from turbo_b200.model import Model  # noqa: E402

OUT = os.path.join(HERE, "fzn")


def main():
    os.makedirs(OUT, exist_ok=True)
    models = {}
    for seed in range(16):
        models[f"random_{seed:02d}"] = tf.gen_model(np.random.default_rng(seed))
    for seed in range(6):
        models[f"sets_{seed:02d}"] = tf.gen_set_model(np.random.default_rng(1000 + seed))
    models["syntax_subset"] = (tf.SYNTAX_SUBSET, 3)
    pins = {}
    for name, (text, best) in sorted(models.items()):
        with open(os.path.join(OUT, name + ".fzn"), "w") as f:
            f.write(text if text.endswith("\n") else text + "\n")
        m = Model.from_fzn(os.path.join(OUT, name + ".fzn"))
        pins[name] = {"tnf_sha256": tf.network_sha(m), "optimum": best}
        print(f"{name:16s} V={m.problem.nvars:4d} P={m.problem.nprops:4d} optimum={best}")
    with open(os.path.join(OUT, "pins.json"), "w") as f:
        json.dump(pins, f, indent=1, sort_keys=True)
        f.write("\n")


if __name__ == "__main__":
    main()
