#!/usr/bin/env python
"""Generates tests/golden/reference_outputs.npz: what the REFERENCE'S OWN compiled objects return for the inputs of the tests
that compare with them.

Needs oracle/_ref/libref.so, which `make -C oracle ref` builds where the reference sources are present:
    python tests/golden/make_reference_outputs.py
Every record_<name>() of the modules below builds its test's inputs and returns the reference's outputs as arrays; they are
stored as "<name>.<field>" and read back by oracle_lib.recorded(name). Run it again whenever such a test changes its inputs."""
import importlib
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
import oracle_lib as ol  # noqa: E402

MODULES = ["test_oracle_kats", "test_oracle_vs_reference_blocks", "test_oracle_vs_reference_blocks_fuzz", "test_scan_policy", "test_recorder"]


def main():
    assert ol.have_ref_blocks(), "build oracle/_ref/libref.so first: make -C oracle ref"
    out = {}
    for m in MODULES:
        mod = importlib.import_module(m)
        for fn in sorted(f for f in dir(mod) if f.startswith("record_")):
            for field, a in getattr(mod, fn)().items():
                out[f"{fn[len('record_'):]}.{field}"] = np.asarray(a)
    np.savez_compressed(ol.REF_OUTPUTS, **out)
    print("wrote", ol.REF_OUTPUTS, os.path.getsize(ol.REF_OUTPUTS), "bytes,", len(out), "arrays")


if __name__ == "__main__":
    main()
