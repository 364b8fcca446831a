#!/usr/bin/env python
"""Regenerate the reference data under ``tests/golden/`` from the UNMODIFIED reference (``ref_loader.load()``).

* ``reference_nodes.txt``: the reference's node schemas (one set per number of visible CUDA devices, 0-8), display
  names and the device chains it builds, as a Python literal so tuples stay tuples;
* ``reference_differential.pt``: weights and inputs of ``tests/test_engine.py``'s ``Toy`` model and the reference's
  outputs and per-call batch sizes with it split over a 40/40/15/5 CPU chain.

    python baseline/make_golden.py
"""
from __future__ import annotations

import copy
import os
import pprint
import sys
from unittest import mock

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

from baseline import ref_loader  # noqa: E402

MAX_CUDA = 8
NODES = ("ParallelDevice", "ParallelDeviceList", "ParallelAnything")
ATTRS = ("RETURN_TYPES", "RETURN_NAMES", "FUNCTION", "CATEGORY")
BATCHES = (1, 3, 8, 21, 32)


def node_data(ref) -> dict:
    schemas = {}
    for n in range(MAX_CUDA + 1):
        with mock.patch.object(torch.cuda, "is_available", return_value=n > 0), \
                mock.patch.object(torch.cuda, "device_count", return_value=n):
            schemas[n] = {name: dict(INPUT_TYPES=ref.NODE_CLASS_MAPPINGS[name].INPUT_TYPES(),
                                     **{a: getattr(ref.NODE_CLASS_MAPPINGS[name], a) for a in ATTRS})
                          for name in NODES}
    chain = ref.ParallelDevice().add_device("cpu", 40)[0]
    chain = ref.ParallelDevice().add_device("cpu", 60, chain)[0]
    return {"schemas": schemas, "display_names": dict(ref.NODE_DISPLAY_NAME_MAPPINGS),
            "parallel_device_description": ref.ParallelDevice.DESCRIPTION, "add_device_chain": chain,
            "create_list": ref.ParallelDeviceList().create_list("cpu", 50, "cpu", 0, "cpu", 25)}


def differential(ref) -> dict:
    import test_engine as te
    torch.manual_seed(0)
    base = te.Toy()
    theirs = copy.deepcopy(base)
    ref.ParallelAnything().setup_parallel(theirs, te.chain_of(40, 40, 15, 5), True, False, True, False)
    cases = {}
    for B in BATCHES:
        x, t, c, y = te.inputs(B)
        theirs.calls.clear()
        with torch.no_grad():
            out = theirs(x, t, context=c, y=y)
        cases[B] = {"x": x, "t": t, "c": c, "y": y, "out": out.clone(), "calls": sorted(theirs.calls)}
    return {"state_dict": {k: v.clone() for k, v in base.state_dict().items()}, "cases": cases}


def main() -> None:
    ref = ref_loader.load()
    os.makedirs(GOLDEN, exist_ok=True)
    with open(os.path.join(GOLDEN, "reference_nodes.txt"), "w") as f:
        f.write(pprint.pformat(node_data(ref), width=200) + "\n")
    torch.save(differential(ref), os.path.join(GOLDEN, "reference_differential.pt"))


if __name__ == "__main__":
    main()
