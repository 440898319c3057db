#!/usr/bin/env python
"""Store what the parity tests compare against when the reference checkout is not at hand.

Runs the reference's own code (needs a checkout of hellojialee/Improved-Body-Parts at ``SPG_REFERENCE_ROOT``) and
writes, under ``reference/`` next to this file (kept apart from the ``*.npz`` grouping cases):

``fuzz.npz.xz``                  ``find_peaks -> find_connections -> find_people`` on the random parameter / dirt draws
                                 of ``tests/test_oracle_vs_reference.py::fuzz_cases``
``format_results.json``          the file ``format_results`` (evaluate.py:563-582) writes for the people lists of
                                 ``tests/test_wire.py::_golden_people``
``utils_config.json``            ``skeleton.read_reference_ini`` of the reference's ``utils/config``, which tests/test_launcher.py checks
``imhn.npz``                     the ``NetworkEval`` state dict's names and shapes, and a fixed sample of all ``nstack x 5``
                                 output maps for the deterministic weights of ``tests/test_imhn.py::seeded_state``

``python tests/golden/make_reference_outputs.py``
"""
from __future__ import annotations

import contextlib
import io
import json
import lzma
import os
import sys
import types

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
OUT = os.path.join(HERE, "reference")
TESTS = os.path.dirname(HERE)
ROOT = os.path.dirname(TESTS)
for p in (ROOT, TESTS, HERE):
    sys.path.insert(0, p)

from golden_io import flatten, stack  # noqa: E402
from oracle import ref_loader  # noqa: E402


def fuzz() -> None:
    from improved_body_parts_b200 import skeleton
    from test_oracle_vs_reference import N_TRIALS, candidate_from_peaks, fuzz_cases, input_crc

    ref = ref_loader.Reference()
    assert tuple(ref.limbs) == skeleton.LIMBS
    crcs, flats = [], []
    for trial, heat, paf, extent, params, _ in fuzz_cases(N_TRIALS):
        crcs.append(input_crc(heat, paf))
        for i in range(2):  # image-major within a draw: entry 2 * trial + i
            f = flatten(ref.group(np.ascontiguousarray(heat[i].transpose(1, 2, 0)),
                                  np.ascontiguousarray(paf[i].transpose(1, 2, 0)), extent, params))
            assert np.array_equal(f.pop("candidate"), candidate_from_peaks(f))  # not stored: the peaks in order
            flats.append(f)
    buf = io.BytesIO()  # xz packs these float64 tables a quarter tighter than the npz's own deflate
    np.savez(buf, input_crc=np.array(crcs, np.int64), **stack(flats))
    with lzma.open(os.path.join(OUT, "fuzz.npz.xz"), "wb", preset=9 | lzma.PRESET_EXTREME) as fh:
        fh.write(buf.getvalue())


def format_results() -> None:
    from test_wire import _golden_people

    path = os.path.join(OUT, "format_results.json")
    ref_loader.reference_function("format_results")(_golden_people(), path)


def utils_config() -> None:
    from improved_body_parts_b200 import skeleton

    param, model = skeleton.read_reference_ini(os.path.join(ref_loader.REFERENCE_ROOT, "utils", "config"))
    with open(os.path.join(OUT, "utils_config.json"), "w") as fh:
        model = {k: model[k] for k in ("boxsize", "padValue", "stride", "max_downsample")}
        json.dump({"param": param, "model": model}, fh, indent=1, sort_keys=True)
        fh.write("\n")


def imhn() -> None:
    import torch
    from test_imhn import imhn_input, map_sample, seeded_state

    sys.path.insert(0, ref_loader.REFERENCE_ROOT)
    with contextlib.redirect_stdout(io.StringIO()):
        from models.posenet import NetworkEval  # the reference's module, unmodified
    opt = types.SimpleNamespace(nstack=4, hourglass_inp_dim=256, increase=128)
    ref = NetworkEval(opt, types.SimpleNamespace(num_layers=50), bn=True).eval()
    entries = [(k, list(v.shape)) for k, v in ref.state_dict().items()]
    ref.load_state_dict(seeded_state(entries), strict=True)
    out = {"state": np.array(json.dumps(entries))}
    with torch.no_grad():
        want = ref(imhn_input())
    for i in range(4):
        for j in range(5):
            out[f"s{i}_{j}_absmax"] = np.float32(want[i][j].abs().max())
            out[f"s{i}_{j}_sample"] = map_sample(want[i][j])
    np.savez_compressed(os.path.join(OUT, "imhn.npz"), **out)


if __name__ == "__main__":
    if not ref_loader.reference_available():
        raise SystemExit(f"no reference checkout at {ref_loader.REFERENCE_ROOT} (set SPG_REFERENCE_ROOT)")
    for step in (format_results, utils_config, fuzz, imhn):
        step()
        print(step.__name__, "done")
