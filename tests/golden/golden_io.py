"""Flat (npz-friendly) encoding of the reference's nested output structures, and back.

A fixture holds the inputs (``heat [K,H,W] f32``, ``paf [L,H,W] f32|f64``, channel-first), the limb table,
``image_extent``, the parameter dict, and the outputs of the reference's own functions flattened as below.
"""
from __future__ import annotations

import json

import numpy as np


def flatten(structs) -> dict:
    all_peaks, connection_all, special_k, subset, candidate = structs
    K, L = len(all_peaks), len(connection_all)
    part_count = np.array([len(p) for p in all_peaks], np.int32)
    flat = [t for part in all_peaks for t in part]
    n = len(flat)
    peak_xy = np.array([[float(t[0]), float(t[1])] for t in flat], np.float64).reshape(n, 2)
    peak_score = np.array([t[2] for t in flat], np.float32)
    peak_id = np.array([t[3] for t in flat], np.int64)
    peak_is_int = np.array([isinstance(t[0], (int, np.integer)) for t in flat], np.uint8)
    conn_count = np.array([-1 if isinstance(c, list) else c.shape[0] for c in connection_all], np.int32)
    rows = [c for c in connection_all if not isinstance(c, list) and c.shape[0]]
    conn_rows = np.concatenate(rows, 0) if rows else np.zeros((0, 6))
    return dict(part_count=part_count, peak_xy=peak_xy, peak_score=peak_score, peak_id=peak_id,
                peak_is_int=peak_is_int, conn_count=conn_count, conn_rows=np.asarray(conn_rows, np.float64),
                special_k=np.array(list(special_k), np.int32), subset=np.asarray(subset, np.float64),
                candidate=np.asarray(candidate, np.float64).reshape(-1, 4) if n else np.zeros((0, 4)))


def unflatten(d) -> tuple:
    part_count = d["part_count"]
    all_peaks, g = [], 0
    for c in range(len(part_count)):
        lst = []
        for _ in range(int(part_count[c])):
            if d["peak_is_int"][g]:
                xy = (np.int64(d["peak_xy"][g, 0]), np.int64(d["peak_xy"][g, 1]))
            else:
                xy = (np.float64(d["peak_xy"][g, 0]), np.float64(d["peak_xy"][g, 1]))
            lst.append(xy + (np.float32(d["peak_score"][g]), int(d["peak_id"][g])))
            g += 1
        all_peaks.append(lst)
    connection_all, r = [], 0
    for m in d["conn_count"]:
        if m < 0:
            connection_all.append([])
        else:
            connection_all.append(np.array(d["conn_rows"][r:r + m], np.float64).reshape(m, 6))
            r += int(m)
    cand = d["candidate"] if len(d["candidate"]) else np.zeros((0,))
    return all_peaks, connection_all, [int(v) for v in d["special_k"]], np.array(d["subset"]), np.array(cand)


def stack(flats) -> dict:
    """Several ``flatten`` dicts as one: each field concatenated along axis 0, its per-dict lengths in ``<field>_len``."""
    out = {}
    for k in flats[0]:
        out[k] = np.concatenate([f[k] for f in flats])
        out[k + "_len"] = np.array([len(f[k]) for f in flats], np.int64)
    return out


def unstack(d, j: int) -> dict:
    """The ``j``-th ``flatten`` dict of a ``stack`` result."""
    out = {}
    for k in d:
        if k + "_len" in d:
            n = d[k + "_len"]
            a = int(n[:j].sum())
            out[k] = d[k][a:a + int(n[j])]
    return out


def save_case(path, heat, paf, limbs, image_extent, params, structs, meta=None) -> None:
    np.savez_compressed(path, heat=heat, paf=paf, limbs=np.asarray(limbs, np.int32), image_extent=np.int64(image_extent),
                        params=np.array(json.dumps(params)), meta=np.array(json.dumps(meta or {})), **flatten(structs))


def load_case(path):
    with np.load(path, allow_pickle=False) as z:
        d = {k: z[k] for k in z.files}
    params = json.loads(str(d["params"]))
    meta = json.loads(str(d["meta"]))
    return dict(heat=d["heat"], paf=d["paf"], limbs=[tuple(int(v) for v in p) for p in d["limbs"]],
                image_extent=int(d["image_extent"]), params=params, meta=meta, structs=unflatten(d))
