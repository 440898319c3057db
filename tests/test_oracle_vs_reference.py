"""CPU: the checker against the reference's own functions on random hyper-parameters and dirty-input knobs the fixed
golden cases do not enumerate.

The reference's outputs for these draws are stored in tests/golden/reference/fuzz.npz.xz (written by
tests/golden/make_reference_outputs.py, which runs the reference's functions unmodified); the inputs are regenerated
from their seeds and checked against the stored CRC before the comparison."""
import io
import lzma
import os
import zlib

import numpy as np

from golden_io import unflatten, unstack
from oracle import spg_oracle as so
from parity import diff_structures

N_TRIALS = 24  # the draws whose reference outputs are stored
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference", "fuzz.npz.xz")


def input_crc(heat, paf) -> int:
    return zlib.crc32(paf.tobytes(), zlib.crc32(heat.tobytes()))


def candidate_from_peaks(flat):
    """``candidate`` of the reference's ``find_people``: every peak's (x, y, score, id) in order."""
    return np.column_stack([flat["peak_xy"], flat["peak_score"], flat["peak_id"]]).astype(np.float64)


def fuzz_cases(n_trials, seed=20260921):
    """The draw sequence shared with tests/test_gpu_parity.py::test_random_parameters_and_dirt_against_the_checker."""
    from improved_body_parts_b200 import skeleton, synth

    rng = np.random.default_rng(seed)
    for trial in range(n_trials):
        H = int(rng.choice([48, 64, 72, 96, 128])); W = int(rng.choice([48, 64, 80, 96, 128]))
        persons = int(rng.integers(1, 14))
        kw = dict(drop_prob=float(rng.choice([0.0, 0.1, 0.3])), plateau=int(rng.integers(0, 4)), spikes=int(rng.integers(0, 20)),
                  colocate=int(rng.integers(0, 3)), edge=bool(rng.integers(0, 2)), stretch=int(rng.integers(0, 4)),
                  negative_bias=float(rng.choice([0.0, 0.0, 0.03])), heat_gain=float(rng.choice([1.0, 1.0, 0.5])),
                  paf_gain=float(rng.choice([1.0, 1.0, 0.6])))
        params = dict(skeleton.default_params(),
                      thre1=float(rng.choice([0.05, 0.1, 0.2, 0.3])), thre2=float(rng.choice([0.02, 0.05, 0.1, 0.3])),
                      connect_ration=float(rng.choice([0.5, 0.7, 0.8, 0.95, 1.0])), mid_num=int(rng.choice([1, 2, 5, 10, 20, 33, 40])),
                      len_rate=float(rng.choice([1.2, 4.0, 16.0])), connection_tole=float(rng.choice([0.3, 0.7, 1.3])),
                      offset_radius=int(rng.integers(0, 5)), remove_recon=int(rng.integers(0, 2)))
        f64 = bool(rng.integers(0, 4) == 0)
        heat, paf = synth.make_batch(31000 + trial, 3, H, W, persons, **kw)
        if f64:
            paf = paf.astype(np.float64) * (1.0 + 2.0 ** -27)
        extent = int(rng.choice([H, 40, 2 * H]))
        cap = int(rng.choice([64, 128]))
        yield trial, heat, paf, extent, params, cap


def test_checker_equals_live_reference_on_random_parameters():
    from improved_body_parts_b200 import skeleton

    with lzma.open(GOLDEN) as fh, np.load(io.BytesIO(fh.read()), allow_pickle=False) as z:
        ref = {k: z[k] for k in z.files}
    for trial, heat, paf, extent, params, _ in fuzz_cases(N_TRIALS):
        assert int(ref["input_crc"][trial]) == input_crc(heat, paf), f"trial {trial}: inputs differ from the stored draw"
        o = so.group_batch(heat, paf, skeleton.LIMBS, extent, params)
        assert (o.status == 0).all()
        for i in range(2):
            flat = unstack(ref, 2 * trial + i)
            want = unflatten(dict(flat, candidate=candidate_from_peaks(flat)))
            d = diff_structures(want, o.as_reference_structures(i), float_tol=0.0)
            assert not d, f"trial {trial} image {i} {params}:\n" + "\n".join(d)
