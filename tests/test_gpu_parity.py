"""GPU: the CUDA path (through the C ABI, libspgroup.so) against the golden vectors and the CPU checker.

Bar (BASELINE.json north_star / SURVEY.md §8): integer content bit-exact; floats within 1e-4.  The kernels
reproduce the reference's arithmetic operation for operation, so these tests assert the stronger property --
floats bit-identical too (float_tol = 0) -- and would report a 1e-4-only agreement as a failure to look at.
"""
import os

import numpy as np
import pytest

from conftest import golden_paths
from golden_io import load_case
from parity import FLOAT_TOL, diff_structures, structure_stats

pytestmark = pytest.mark.gpu

GOLDENS = golden_paths()


@pytest.fixture(scope="module")
def env(cuda_device):
    import torch
    from improved_body_parts_b200 import skeleton, synth
    from improved_body_parts_b200.grouping import Grouper
    from oracle import spg_oracle as so

    class Env:
        pass

    e = Env()
    e.torch, e.skeleton, e.synth, e.Grouper, e.so, e.dev = torch, skeleton, synth, Grouper, so, cuda_device
    return e


def _run_gpu(env, heat, paf, extent, params, limbs=None, **cfg):
    t = env.torch
    N, K, H, W = heat.shape
    g = env.Grouper(limbs if limbs is not None else env.skeleton.LIMBS, max_batch=N, max_h=H, max_w=W, **cfg)
    try:
        g.group_device(t.from_numpy(heat).to(env.dev), t.from_numpy(paf).to(env.dev), extent, params)
        return g.fetch()
    finally:
        g.close()


def _assert_same(ref_structs, got_structs, what):
    d = diff_structures(ref_structs, got_structs, float_tol=0.0)
    if d:
        loose = diff_structures(ref_structs, got_structs, float_tol=FLOAT_TOL)
        pytest.fail(f"{what}: not bit-identical ({'within 1e-4' if not loose else 'ALSO outside 1e-4'}):\n" + "\n".join(d))


@pytest.mark.parametrize("path", GOLDENS, ids=[os.path.basename(p)[:-4] for p in GOLDENS])
def test_cuda_matches_reference_golden(env, path):
    case = load_case(path)
    H, W = case["heat"].shape[1:]
    r = _run_gpu(env, case["heat"][None], case["paf"][None], case["image_extent"], case["params"], limbs=case["limbs"],
                 max_peaks_per_part=128, max_person_rows=128)
    assert r.status[0] == 0, f"status {r.status[0]:#x}"
    got = r.as_reference_structures(0)
    _assert_same(case["structs"], got, os.path.basename(path))
    assert structure_stats(got) == structure_stats(case["structs"])


@pytest.mark.parametrize("persons,n,kw", [
    (10, 64, {}), (30, 64, {}),
    (25, 32, dict(drop_prob=0.15, stretch=6, spikes=30, plateau=3, colocate=4, edge=True)),
    (20, 16, dict(negative_bias=0.04, drop_prob=0.1))])
def test_cuda_matches_oracle_batches(env, persons, n, kw):
    heat, paf = env.synth.make_batch(7000 + persons, n, 128, 128, persons, **kw)
    params = env.skeleton.default_params()
    o = env.so.group_batch(heat, paf, env.skeleton.LIMBS, 128, params, threads=4)
    assert (o.status == 0).all()
    r = _run_gpu(env, heat, paf, 128, params, max_peaks_per_part=96, max_person_rows=128)
    assert (r.status == 0).all(), r.status
    for i in range(n):
        _assert_same(o.as_reference_structures(i), r.as_reference_structures(i), f"image {i}")


def test_full_size_batch_256_p30(env):
    """BASELINE.json configs[2] per-GPU shard: 256 images, 128x128, 30 persons -- every image vs the checker."""
    heat, paf = env.synth.make_batch(424242, 256, 128, 128, 30)
    params = env.skeleton.default_params()
    o = env.so.group_batch(heat, paf, env.skeleton.LIMBS, 128, params, threads=max(1, min(16, os.cpu_count() or 1)))
    r = _run_gpu(env, heat, paf, 128, params)
    assert (r.status == 0).all() and (o.status == 0).all()
    assert np.array_equal(r.n_persons, o.n_persons)
    for i in range(256):
        _assert_same(o.as_reference_structures(i), r.as_reference_structures(i), f"image {i}")
    # process() tail: COCO-ordered joints + person score
    for i in (0, 17, 255):
        kp, sc = o.to_coco(i, env.skeleton.COCO_FROM_PART)
        P = int(r.n_persons[i])
        assert np.array_equal(r.people_xy[i, :P], kp) and np.array_equal(r.people_score[i, :P], sc)


def test_f64_body_part_planes(env):
    heat, paf = env.synth.make_batch(99, 8, 96, 128, 12)
    paf64 = paf.astype(np.float64) * (1.0 + 2.0 ** -29) + 2.0 ** -41
    params = env.skeleton.default_params()
    o = env.so.group_batch(heat, paf64, env.skeleton.LIMBS, 96, params)
    r = _run_gpu(env, heat, paf64, 96, params)
    assert (r.status == 0).all()
    for i in range(8):
        _assert_same(o.as_reference_structures(i), r.as_reference_structures(i), f"image {i}")


@pytest.mark.parametrize("H,W", [(57, 61), (50, 70), (33, 130)])
def test_unaligned_widths_take_the_generic_loaders(env, H, W):
    heat, paf = env.synth.make_batch(5150, 4, H, W, 4, edge=True)
    params = env.skeleton.default_params()
    o = env.so.group_batch(heat, paf, env.skeleton.LIMBS, H, params)
    r = _run_gpu(env, heat, paf, H, params)
    assert (r.status == 0).all()
    for i in range(4):
        _assert_same(o.as_reference_structures(i), r.as_reference_structures(i), f"image {i}")


@pytest.mark.parametrize("H,W,persons", [(200, 260, 12), (150, 512, 10), (300, 132, 10)])
def test_planes_too_large_for_the_plane_ring_take_the_banded_nms(env, H, W, persons):
    """Keypoint planes that do not fit shared memory three times go through nms_peaks_banded_kernel: band heights that do
    not divide H, a last band of a few rows, widths whose bands hold 15 / 8 / 31 rows -- peaks on band borders use the halo rows."""
    t = env.torch
    heat, paf = env.synth.make_batch(2600 + H, 3, H, W, persons, scale_range=(1.5, 3.0), edge=True)
    params = env.skeleton.default_params()
    o = env.so.group_batch(heat, paf, env.skeleton.LIMBS, H, params)
    g = env.Grouper(max_batch=3, max_h=H, max_w=W)
    try:
        g.group_device(t.from_numpy(heat).to(env.dev), t.from_numpy(paf).to(env.dev), H, params)
        r = g.fetch()
        names = g.stage_kernels()
    finally:
        g.close()
    assert names[0] == "nms_peaks_banded_kernel", names
    assert (r.status == 0).all() and (o.status == 0).all()
    for i in range(3):
        _assert_same(o.as_reference_structures(i), r.as_reference_structures(i), f"image {i}")


@pytest.mark.parametrize("capP,capR", [(37, 41), (50, 47)])
def test_odd_capacities(env, capP, capR):
    """Capacities that break the 16-byte granularity of the bulk copies (peak arrays of 18 x 37 floats, connection tables
    of 30 x 37 words): the fused kernel's matchers stage the peaks themselves, the stand-alone assembler loads its tables
    with plain loads; record / slot / scratch layouts with odd counts."""
    t = env.torch
    heat, paf = env.synth.make_batch(3737, 6, 128, 128, 14, drop_prob=0.1, edge=True, colocate=1)
    params = env.skeleton.default_params()
    o = env.so.group_batch(heat, paf, env.skeleton.LIMBS, 128, params)
    hd, pd = t.from_numpy(heat).to(env.dev), t.from_numpy(paf).to(env.dev)
    for fused in ("1", "0"):
        os.environ["SPG_FUSE_MA"] = fused
        try:
            g = env.Grouper(max_batch=6, max_peaks_per_part=capP, max_person_rows=capR)
        finally:
            os.environ.pop("SPG_FUSE_MA", None)
        try:
            g.group_device(hd, pd, 128, params)
            r = g.fetch()
        finally:
            g.close()
        assert (r.status == 0).all() and (o.status == 0).all()
        for i in range(6):
            _assert_same(o.as_reference_structures(i), r.as_reference_structures(i), f"fused={fused} image {i}")


def test_512_planes_sample_through_l2(env):
    """BASELINE.json configs[3] shape: 512x512 maps do not fit shared memory (1 MiB / plane)."""
    heat, paf = env.synth.make_batch(31337, 2, 512, 512, 24, scale_range=(3.0, 5.0))
    params = env.skeleton.default_params()
    o = env.so.group_batch(heat, paf, env.skeleton.LIMBS, 512, params)
    r = _run_gpu(env, heat, paf, 512, params, max_peaks_per_part=96)
    assert (r.status == 0).all()
    for i in range(2):
        _assert_same(o.as_reference_structures(i), r.as_reference_structures(i), f"image {i}")


def test_network_layout_channel_slices(env):
    """The network's raw [N,50,h,w] tensor: body parts at channel 0, keypoints at 30 (config/config.py:101-103)."""
    t = env.torch
    heat, paf = env.synth.make_batch(2718, 6, 64, 64, 5)
    vol = np.zeros((6, 50, 64, 64), np.float32)
    vol[:, :30] = paf
    vol[:, 30:48] = heat
    vol[:, 48:] = 0.9  # background maps must never be read
    d = t.from_numpy(vol).to(env.dev)
    params = env.skeleton.default_params()
    g = env.Grouper(max_batch=6, max_h=64, max_w=64)
    g.group_device(d[:, 30:48], d[:, :30], 64, params)
    r = g.fetch()
    g.close()
    o = env.so.group_batch(heat, paf, env.skeleton.LIMBS, 64, params)
    for i in range(6):
        _assert_same(o.as_reference_structures(i), r.as_reference_structures(i), f"image {i}")


def test_stage_wise_entry_points(env):
    """spg_upload_* + single stages: each stage fed with the CHECKER's previous-stage output."""
    t = env.torch
    heat, paf = env.synth.make_batch(1234, 3, 96, 96, 9, drop_prob=0.1)
    params = env.skeleton.default_params()
    o = env.so.group_batch(heat, paf, env.skeleton.LIMBS, 96, params)
    g = env.Grouper(max_batch=3, max_h=96, max_w=96)
    # stage 2+3 from uploaded peaks
    for i in range(3):
        tot = int(o.part_count[i].sum())
        g.upload_peaks(i, o.part_count[i], o.px[i, :tot], o.py[i, :tot], o.pscore[i, :tot])
    g.limb_score(t.from_numpy(paf).to(env.dev), 96, params)
    g.limb_match(3, params)
    r = g.fetch(3)
    for i in range(3):
        assert np.array_equal(r.conn_count[i], o.conn_count[i])
        for k in range(30):
            m = int(o.conn_count[i, k])
            if m > 0:
                ij = r.conn_ij[i, k, :m].astype(np.int64)
                assert np.array_equal(np.stack([ij >> 16, ij & 0xffff], 1), o.conn_ij[i, k, :m])
                assert np.array_equal(r.conn_score[i, k, :m], o.conn_score[i, k, :m])
                assert np.array_equal(r.conn_norm[i, k, :m], o.conn_norm[i, k, :m])
    g.close()
    # stage 4 from uploaded peaks + connections
    g = env.Grouper(max_batch=3, max_h=96, max_w=96)
    for i in range(3):
        tot = int(o.part_count[i].sum())
        g.upload_peaks(i, o.part_count[i], o.px[i, :tot], o.py[i, :tot], o.pscore[i, :tot])
        rows_ij, rows_s, rows_n = [], [], []
        for k in range(30):
            m = max(int(o.conn_count[i, k]), 0)
            rows_ij.append(o.conn_ij[i, k, :m]); rows_s.append(o.conn_score[i, k, :m]); rows_n.append(o.conn_norm[i, k, :m])
        g.upload_connections(i, o.conn_count[i], np.concatenate(rows_ij), np.concatenate(rows_s), np.concatenate(rows_n))
    g.assemble(3, params)
    r = g.fetch(3)
    for i in range(3):
        P = int(o.n_persons[i])
        assert int(r.n_persons[i]) == P
        assert np.array_equal(r.subset[i, :P], o.subset[i, :P])
    g.close()


def test_host_entry_point_equals_device_entry_point(env):
    t = env.torch
    heat, paf = env.synth.make_batch(777, 40, 128, 128, 12)
    params = env.skeleton.default_params()
    g = env.Grouper(max_batch=40)
    g.group_device(t.from_numpy(heat).to(env.dev), t.from_numpy(paf).to(env.dev), 128, params)
    a = g.fetch()
    hp = t.from_numpy(heat).pin_memory().numpy()
    pp = t.from_numpy(paf).pin_memory().numpy()
    out = g.group_host(hp, pp, 128, params)
    b = g.fetch(40)
    g.close()
    assert np.array_equal(out["n_persons"], a.n_persons) and np.array_equal(out["status"], a.status)
    for i in range(40):
        P = int(a.n_persons[i])
        assert np.array_equal(out["people_xy"][i, :P], a.people_xy[i, :P])
        assert np.array_equal(out["people_score"][i, :P], a.people_score[i, :P])
        assert np.array_equal(b.subset[i, :P], a.subset[i, :P])


def test_capacity_overflows_are_flagged_not_fatal(env):
    from improved_body_parts_b200 import grouping as G

    heat, paf = env.synth.make_batch(4321, 2, 128, 128, 30)
    params = env.skeleton.default_params()
    r = _run_gpu(env, heat, paf, 128, params, max_peaks_per_part=8)
    assert (r.status & G.ST_PEAK_OVERFLOW).all()
    r = _run_gpu(env, heat, paf, 128, params, max_person_rows=4)
    assert (r.status & G.ST_ROW_OVERFLOW).all()
    r = _run_gpu(env, heat, paf, 128, params, max_cands_per_limb=4)
    assert (r.status & G.ST_CAND_OVERFLOW).all()


def test_invalid_arguments_fail_loudly(env):
    from improved_body_parts_b200.grouping import GroupingError

    t = env.torch
    g = env.Grouper(max_batch=2, max_h=64, max_w=64)
    with pytest.raises(GroupingError):
        g.group_device(t.zeros(3, 18, 64, 64, device=env.dev), t.zeros(3, 30, 64, 64, device=env.dev), 64)  # > max_batch
    with pytest.raises(GroupingError):
        g.group_device(t.zeros(1, 18, 128, 64, device=env.dev), t.zeros(1, 30, 128, 64, device=env.dev), 64)  # > max_h
    with pytest.raises(GroupingError):
        g.limb_match(1)  # no candidates yet
    with pytest.raises(GroupingError):
        g.group_device(t.zeros(1, 18, 64, 64, device=env.dev), t.zeros(1, 30, 64, 64, device=env.dev), 64,
                       dict(offset_radius=9))
    g.close()


def test_screen_is_conservative_and_effective(env, monkeypatch):
    """limb_score's f32 screen may only drop pairs the exact evaluation would drop: identical outputs with the
    screen disabled, survivors >= candidates, and on clean 30-person images it removes most of the nA*nB pairs."""
    t = env.torch
    heat, paf = env.synth.make_batch(8080, 16, 128, 128, 30)
    params = env.skeleton.default_params()
    hd, pd = t.from_numpy(heat).to(env.dev), t.from_numpy(paf).to(env.dev)
    g = env.Grouper(max_batch=16)
    g.group_device(hd, pd, 128, params)
    a = g.fetch()
    v = g.device_tensors()
    surv, cand = v["surv_count"][:16].cpu().numpy(), v["cand_count"][:16].cpu().numpy()
    g.close()
    monkeypatch.setenv("SPG_NO_SCREEN", "1")
    g = env.Grouper(max_batch=16)
    g.group_device(hd, pd, 128, params)
    b = g.fetch()
    surv_off = g.device_tensors()["surv_count"][:16].cpu().numpy()
    g.close()
    for f in ("conn_count", "cand_count", "conn_ij", "conn_score", "conn_norm", "n_persons", "subset", "people_xy"):
        assert np.array_equal(getattr(a, f), getattr(b, f)), f
    assert (surv >= cand).all()
    pairs = np.array([[a.peak_count[i, x] * a.peak_count[i, y] for x, y in env.skeleton.LIMBS] for i in range(16)])
    assert np.array_equal(surv_off, pairs)           # screen off: every pair is evaluated exactly
    frac = surv.sum() / pairs.sum()
    print(f"screen keeps {frac:.3f} of {pairs.sum()} pairs; candidates are {cand.sum() / pairs.sum():.3f}")
    assert frac < 0.5


def test_persistent_and_per_item_kernels_agree(env, monkeypatch):
    """nms_peaks and limb_score have two schedules (persistent ring for f32 planes that fit it, one CTA per item
    otherwise): same peaks and candidates, hence identical results downstream; both equal to the checker."""
    t = env.torch
    heat, paf = env.synth.make_batch(60606, 24, 128, 128, 22, drop_prob=0.1, stretch=4, spikes=10, edge=True, colocate=2)
    params = env.skeleton.default_params()
    hd, pd = t.from_numpy(heat).to(env.dev), t.from_numpy(paf).to(env.dev)
    outs = []
    for flag in ("1", "0"):
        monkeypatch.setenv("SPG_PERSIST", flag)
        g = env.Grouper(max_batch=24)
        g.group_device(hd, pd, 128, params)
        outs.append(g.fetch())
        assert ("persist" in g.stage_kernels()[0]) == (flag == "1") and ("persist" in g.stage_kernels()[1]) == (flag == "1")
        g.close()
    a, b = outs
    assert (a.status == 0).all() and (b.status == 0).all()
    for f in ("peak_count", "peak_x", "peak_y", "peak_score", "peak_anchor", "conn_count", "cand_count", "conn_ij",
              "conn_score", "conn_norm", "n_persons", "subset", "people_xy", "people_score"):
        x, y = getattr(a, f), getattr(b, f)
        if f.startswith("peak_") and f != "peak_count":  # slots beyond the count are undefined
            m = np.arange(x.shape[2])[None, None, :] < np.minimum(a.peak_count, x.shape[2])[:, :, None]
            x, y = np.where(m, x, 0), np.where(m, y, 0)
        assert np.array_equal(x, y), f
    o = env.so.group_batch(heat, paf, env.skeleton.LIMBS, 128, params, threads=4)
    for i in range(24):
        _assert_same(o.as_reference_structures(i), a.as_reference_structures(i), f"image {i}")


def test_survivor_list_overflow_is_evaluated_in_place(env, monkeypatch):
    """With the screen off every pair survives; 40 persons give ~1 600 pairs per limb, more than the persistent
    kernel's survivor list holds, so the screeners evaluate the excess themselves (from the staged plane) while the
    scorers read the rest back through L2.  Same results as the checker, and every pair accounted for."""
    t = env.torch
    heat, paf = env.synth.make_batch(515, 6, 128, 128, 40)
    params = env.skeleton.default_params()
    monkeypatch.setenv("SPG_NO_SCREEN", "1")
    g = env.Grouper(max_batch=6)
    g.group_device(t.from_numpy(heat).to(env.dev), t.from_numpy(paf).to(env.dev), 128, params)
    got = g.fetch()
    surv = g.device_tensors()["surv_count"][:6].cpu().numpy()
    assert "persist" in g.stage_kernels()[1]
    g.close()
    assert (got.status == 0).all()
    pairs = np.array([[got.peak_count[i, x] * got.peak_count[i, y] for x, y in env.skeleton.LIMBS] for i in range(6)])
    assert pairs.max() > 1024 and np.array_equal(surv, pairs)
    o = env.so.group_batch(heat, paf, env.skeleton.LIMBS, 128, params, threads=4)
    for i in range(6):
        _assert_same(o.as_reference_structures(i), got.as_reference_structures(i), f"image {i}")


@pytest.mark.parametrize("scorers", ["1", "5", "30"])
def test_role_split_does_not_change_results(env, monkeypatch, scorers):
    """The persistent limb_score kernel splits its 31 worker warps into screeners and scorers (SPG_EXACT_WARPS, a
    tuning knob): any split -- one scorer for everything, one screener for everything -- gives the checker's results."""
    t = env.torch
    heat, paf = env.synth.make_batch(31337, 12, 128, 128, 26, drop_prob=0.05, spikes=6, colocate=1)
    params = env.skeleton.default_params()
    monkeypatch.setenv("SPG_EXACT_WARPS", scorers)
    got = _run_gpu(env, heat, paf, 128, params)
    assert (got.status == 0).all()
    o = env.so.group_batch(heat, paf, env.skeleton.LIMBS, 128, params, threads=4)
    for i in range(12):
        _assert_same(o.as_reference_structures(i), got.as_reference_structures(i), f"scorers={scorers} image {i}")


def test_arbitrary_limb_tables(env):
    """The limb table is runtime data (the reference ships 24-, 30- and 49-limb skeletons): a random 40-limb table over
    the 18 parts, including repeated and reversed part pairs, against the checker."""
    rng = np.random.default_rng(5)
    limbs = []
    while len(limbs) < 40:
        a, b = (int(v) for v in rng.choice(18, size=2, replace=False))
        limbs.append((a, b))
    heat, paf = env.synth.make_batch(9001, 6, 96, 96, 7, limbs=limbs, drop_prob=0.05)
    params = env.skeleton.default_params()
    o = env.so.group_batch(heat, paf, limbs, 96, params)
    assert (o.status == 0).all()
    r = _run_gpu(env, heat, paf, 96, params, limbs=limbs)
    assert (r.status == 0).all()
    for i in range(6):
        _assert_same(o.as_reference_structures(i), r.as_reference_structures(i), f"image {i}")


def test_random_parameters_and_dirt_against_the_checker(env):
    """40 seeded draws of (hyper-parameters x dirty-input knobs x map shape): every combination the CUDA path can be
    configured with must reproduce the checker, floats included.  Covers offset_radius 0..4, mid_num 1..40 (per-m
    tables), connect_ration / thresholds that move maxfail, remove_recon, len_rate / connection_tole rejects."""
    from test_oracle_vs_reference import fuzz_cases  # the same draws are checked against the reference's outputs on CPU

    for trial, heat, paf, extent, params, cap in fuzz_cases(40):
        o = env.so.group_batch(heat, paf, env.skeleton.LIMBS, extent, params)
        r = _run_gpu(env, heat, paf, extent, params, max_peaks_per_part=cap, max_person_rows=128)
        what = f"trial {trial}: {heat.shape[2]}x{heat.shape[3]} {params} paf={paf.dtype} extent={extent} capP={cap}"
        assert (o.status == 0).all(), what
        assert (r.status == 0).all(), what + f" status {r.status}"
        for i in range(3):
            _assert_same(o.as_reference_structures(i), r.as_reference_structures(i), what + f" image {i}")


@pytest.mark.parametrize("mode", ["f32", "f64", "f32-as-f64"])
def test_512_planes_full_batch(env, mode):
    """VERDICT r1: parity at 512x512 rested on 2 images.  32 images of smooth 512x512 maps (bodies and blobs 4x, as the
    x4 bicubic up-sampling of predict() produces them), 14 persons each, all three body-part dtypes: the keypoint planes
    take the band kernel, the body-part planes (1 / 2 MiB each) are sampled through L2."""
    t = env.torch
    N = 32
    heat, paf = env.synth.make_batch(5120, N, 512, 512, 14, scale_range=(3.2, 5.2), sigma_scale=4.0, noise=0.0, drop_prob=0.05)
    params = env.skeleton.default_params()
    paf_ref = paf if mode == "f32" else paf.astype(np.float64)
    o = env.so.group_batch(heat, paf_ref, env.skeleton.LIMBS, 512, params, threads=8)
    g = env.Grouper(max_batch=N, max_h=512, max_w=512)
    try:
        hd = t.from_numpy(heat).to(env.dev)
        pd = t.from_numpy(paf_ref if mode == "f64" else paf).to(env.dev)
        g.group_device(hd, pd, 512, params, paf_as_f64=mode == "f32-as-f64")
        r = g.fetch()
        names = g.stage_kernels()
    finally:
        g.close()
    assert (o.status == 0).all() and (r.status == 0).all() and r.n_persons.sum() > 10 * N
    assert "false" in names[1], names
    for i in range(N):
        _assert_same(o.as_reference_structures(i), r.as_reference_structures(i), f"{mode} image {i}")


def test_f64_planes_full_batch(env):
    """VERDICT r1: f64 parity rested on 8 images.  64 dirty 30-person images with float64 body-part maps whose values
    are not float32-representable (what a multi-scale predict() returns)."""
    t = env.torch
    N = 64
    heat, paf = env.synth.make_batch(6400, N, 128, 128, 30, drop_prob=0.08, spikes=6, colocate=1, edge=True)
    paf64 = paf.astype(np.float64) * (1.0 + 2.0 ** -30) + 2.0 ** -40
    params = env.skeleton.default_params()
    o = env.so.group_batch(heat, paf64, env.skeleton.LIMBS, 128, params, threads=8)
    r = _run_gpu(env, heat, paf64, 128, params)
    assert (o.status == 0).all() and (r.status == 0).all()
    for i in range(N):
        _assert_same(o.as_reference_structures(i), r.as_reference_structures(i), f"image {i}")
