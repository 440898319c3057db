"""CPU: wire records (improved_body_parts_b200/wire.py) -- the ``format_results`` payload (evaluate.py:563-582).

The record layout is checked against the C header's formula, pack/unpack round-trips the reference's Python
structures (integer ``(0, 0)`` placeholders included), and the JSON written by ``wire.format_results`` is compared
byte for byte with the file the reference's own ``format_results`` wrote for the people lists its own ``process()``
tail builds on the goldens (tests/golden/reference/format_results.json, tests/golden/make_reference_outputs.py)."""
import json
import os
from pathlib import Path

import numpy as np
import pytest

from conftest import golden_paths
from golden_io import load_case


def _process_tail(subset, candidate, dt_gt_mapping):
    """evaluate.py:523-543, restated inline (as tests/test_oracle.py::test_to_coco_matches_process_tail does)."""
    keypoints = []
    for s in subset[..., 0]:
        coords = []
        for index in s[:18]:
            if index == -1:
                X, Y = 0, 0
            else:
                X, Y = candidate[index.astype(int)][:2]
            coords.append((X, Y))
        coco = [None] * 17
        for dt_index, gt_index in dt_gt_mapping.items():
            if gt_index is None:
                continue
            coco[gt_index] = coords[dt_index]
        keypoints.append((coco, 1 - 1.0 / s[18]))
    return keypoints


def _golden_people(names=("clean_p10_128", "dropout_p16", "weak_pruned_p10", "empty", "colocate_edge_p8")):
    from improved_body_parts_b200 import skeleton
    out = {}
    for i, p in enumerate(golden_paths()):
        name = os.path.basename(p)[:-4]
        if name in names:
            c = load_case(p)
            _, _, _, subset, candidate = c["structs"]
            out[1000 + i] = _process_tail(np.asarray(subset), np.asarray(candidate), skeleton.DT_GT_MAPPING)
    assert len(out) == len(names)
    return out


def test_record_layout_matches_the_header_formula():
    from improved_body_parts_b200 import wire
    for J, R in ((17, 64), (17, 1), (5, 128)):
        assert wire.record_dtype(J, R).itemsize == 8 + R * (2 * J + 2) * 8 == wire.record_bytes(J, R)
    dt = wire.record_dtype(17, 64)
    assert dt.fields["n_persons"][1] == 0 and dt.fields["status"][1] == 4 and dt.fields["rows"][1] == 8


def test_pack_unpack_round_trip_keeps_placeholders_and_bits():
    from improved_body_parts_b200 import wire
    people = _golden_people()
    ids = list(people)
    rec = wire.pack([people[i] for i in ids], rows=64, status=[0] * len(ids))
    raw = rec.tobytes()
    back = wire.unpack(wire.as_records(np.frombuffer(raw, np.uint8), 17, 64), ids)
    n_missing = 0
    for i in ids:
        assert len(back[i]) == len(people[i])
        for (pa, sa), (pb, sb) in zip(people[i], back[i]):
            assert sa == sb
            for a, b in zip(pa, pb):
                assert type(a[0]) is type(b[0]) or (isinstance(a[0], (int, np.integer)) == isinstance(b[0], (int, np.integer)))
                assert a[0] == b[0] and a[1] == b[1]
                n_missing += isinstance(b[0], int)
    assert n_missing > 0  # the fixtures contain persons with undetected joints
    with pytest.raises(ValueError):
        wire.pack([people[ids[0]]], rows=1)


def test_format_results_writes_the_reference_file(tmp_path):
    from improved_body_parts_b200 import wire
    people = _golden_people()
    a = Path(__file__).parent / "golden" / "reference" / "format_results.json"  # what the reference's format_results wrote
    b, c = tmp_path / "ours.json", tmp_path / "wire.json"
    wire.format_results(people, str(b))
    assert a.read_bytes() == b.read_bytes()
    # ... and through the binary records (what the GPU emits): same bytes again
    ids = list(people)
    rec = wire.pack([people[i] for i in ids], rows=64)
    json.dump(wire.coco_results_from_records(rec, ids), open(c, "w"))
    assert a.read_bytes() == c.read_bytes()
    assert len(json.load(open(a))) == sum(len(v) for v in people.values()) > 20
