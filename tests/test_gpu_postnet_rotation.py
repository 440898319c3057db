"""GPU: the post-network stage with rotation search (spg_postnet_rotated, csrc/postnet_rot.cuh -- evaluate.py:90-161
with rotation_search != [0]) against its CPU checker tests/rotation_port.py, which tests/test_postnet_rotation_port.py
pins to cv2 (the warp bit for bit).

The kernel spells out the port's float32 / fixed-point operations one by one, so the bar is BIT-IDENTICAL maps."""
import numpy as np
import pytest

from test_gpu_postnet import CASES, _network_like_output

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def env(cuda_device):
    import torch
    import rotation_port as rp
    from improved_body_parts_b200 import skeleton, synth
    from improved_body_parts_b200.grouping import Grouper, GroupingError
    from oracle import postnet_port as pp
    from oracle import spg_oracle as so

    class Env:
        pass

    e = Env()
    e.torch, e.skeleton, e.synth, e.Grouper, e.GroupingError, e.pp, e.rp, e.so, e.dev = \
        torch, skeleton, synth, Grouper, GroupingError, pp, rp, so, cuda_device
    return e


def _port_maps(env, outs, crops, angles, stride, image_hw, nan_scrub=False):
    """The checker: evaluate.py:126-161 per (scale, angle) item through tests/rotation_port.py -> float64 maps
    (heat [N,K,H,W], paf [N,L,H,W]); ``nan_scrub`` is demo_image.py:179-180 after every item."""
    sk = env.skeleton
    N = outs[0].shape[0]
    H, W = image_hw
    heat_avg = np.zeros((N, H, W, 18))
    paf_avg = np.zeros((N, H, W, 30))
    for o, (ch, cw), ang in zip(outs, crops, angles):
        h, w = o.shape[3:]
        padded = (h * stride, w * stride)
        pad = [0, 0, padded[0] - ch, padded[1] - cw]
        for i in range(N):
            hm, pf = env.rp.post_network_scale(o[i].astype(np.float32), stride, padded, pad, (H, W), 30, 48,
                                               sk.FLIP_PAF_ORD, sk.FLIP_HEAT_ORD[:18], angle=ang)
            heat_avg[i] = env.pp.accumulate(heat_avg[i], hm, len(outs))
            paf_avg[i] = env.pp.accumulate(paf_avg[i], pf, len(outs))
            if nan_scrub:
                heat_avg[i][np.isnan(heat_avg[i])] = 0
                paf_avg[i][np.isnan(paf_avg[i])] = 0
    return heat_avg.transpose(0, 3, 1, 2), paf_avg.transpose(0, 3, 1, 2)


def _run(env, outs, crops, angles, image_hw, **kw):
    t = env.torch
    g = env.Grouper(max_batch=outs[0].shape[0], max_h=image_hw[0], max_w=image_hw[1])
    try:
        heat, paf = g.postnet([t.from_numpy(o).to(env.dev) for o in outs], crops, image_hw, angles=angles, **kw)
        return heat.cpu().numpy(), paf.cpu().numpy(), g.postnet_kernel(), g.launch_count
    finally:
        g.close()


GEOMS = ["identity_128_to_512", "padded_ratio_1.25", "odd_sizes", "tiny"]


@pytest.mark.parametrize("name", GEOMS)
@pytest.mark.parametrize("angle", [5.0, -5.0, 22.5, 90.0, 180.0])
def test_single_rotated_item_is_the_ports(env, name, angle):
    sizes, crops, image_hw = CASES[name]
    outs = [_network_like_output(env, 700 + len(name), 2, sizes[0][0], sizes[0][1], 4)]
    ref_heat, ref_paf = _port_maps(env, outs, crops, [angle], 4, image_hw)
    heat, paf, kernel, _ = _run(env, outs, crops, [angle], image_hw, paf_dtype=env.torch.float64)
    assert kernel == "postnet_rot_kernel"
    assert np.array_equal(heat, ref_heat.astype(np.float32)), "keypoint maps differ from the checker"
    assert np.array_equal(paf, ref_paf), "body-part maps differ from the checker"
    if not (name == "tiny" and angle in (90.0, 180.0)):  # there the swapped centre turns the crop out of the map: all 0
        assert np.abs(ref_heat).max() > 0.3 and np.abs(ref_paf).max() > 0.3


def test_single_rotated_item_with_float32_body_part_planes(env):
    """One item divides by 1: float32 planes hold the reference's float64 values, as for spg_postnet."""
    sizes, crops, image_hw = CASES["padded_ratio_1.25"]
    outs = [_network_like_output(env, 41, 2, sizes[0][0], sizes[0][1], 4)]
    ref_heat, ref_paf = _port_maps(env, outs, crops, [-5.0], 4, image_hw)
    heat, paf, _, _ = _run(env, outs, crops, [-5.0], image_hw)
    assert paf.dtype == np.float32
    assert np.array_equal(heat, ref_heat.astype(np.float32)) and np.array_equal(paf.astype(np.float64), ref_paf)


def test_three_scales_by_three_angles(env):
    """[0.5, 1, 2] x [-5, 0, 5]: nine items in the loop's order (scale-major, angle-minor); angle-0 items take the
    stride-4 kernel between rotated launches, the float64 sums carry over through memory."""
    image_hw = (60, 76)
    nets = [(8, 12), (16, 20), (32, 40)]
    crops_s = [(30, 38), (60, 76), (120, 152)]
    outs, crops, angles = [], [], []
    for k, ((h, w), crop) in enumerate(zip(nets, crops_s)):
        for a in (-5.0, 0.0, 5.0):
            outs.append(_network_like_output(env, 900 + len(outs), 2, h, w, 3))
            crops.append(crop)
            angles.append(a)
    ref_heat, ref_paf = _port_maps(env, outs, crops, angles, 4, image_hw)
    heat, paf, kernel, launches = _run(env, outs, crops, angles, image_hw)
    assert kernel == "postnet_rot_kernel" and launches == 9 and paf.dtype == np.float64
    assert np.array_equal(heat, ref_heat.astype(np.float32)) and np.array_equal(paf, ref_paf)


@pytest.mark.parametrize("stride,crop", [(4, (64, 78)), (2, (32, 39))])
@pytest.mark.parametrize("angles", [[0.0, 22.5], [5.0, 0.0, 0.0, 0.0, 0.0, 0.0, -5.0]])
def test_zero_angle_groups_and_the_generic_stride(env, angles, stride, crop):
    """Zero-angle groups longer than one fused launch, and stride 2 (the generic kernel) beside rotated items."""
    image_hw = (50, 61)
    outs = [_network_like_output(env, 60 + k, 1, 16, 20, 3) for k in range(len(angles))]
    crops = [crop] * len(angles)
    ref_heat, ref_paf = _port_maps(env, outs, crops, angles, stride, image_hw)
    heat, paf, _, _ = _run(env, outs, crops, angles, image_hw, stride=stride)
    assert np.array_equal(heat, ref_heat.astype(np.float32)) and np.array_equal(paf, ref_paf)


def test_f16_and_strided_network_output(env):
    t = env.torch
    sizes, crops, image_hw = CASES["padded_ratio_1.25"]
    out = _network_like_output(env, 55, 2, sizes[0][0], sizes[0][1], 4)
    angles = [5.0, 0.0, -37.3]
    outs16 = [out.astype(np.float16)] * 3
    ref_heat, ref_paf = _port_maps(env, outs16, crops * 3, angles, 4, image_hw)
    heat, paf, _, _ = _run(env, outs16, crops * 3, angles, image_hw)
    assert np.array_equal(heat, ref_heat.astype(np.float32)) and np.array_equal(paf, ref_paf)
    # a [N,2,50,h,w] view into a larger buffer: arbitrary channel / pair / image strides
    big = t.zeros((2, 2, 64) + out.shape[3:], device=env.dev)
    big[:, :, 7:57] = t.from_numpy(out).to(env.dev)
    ref_heat, ref_paf = _port_maps(env, [out], crops, [22.5], 4, image_hw)
    g = env.Grouper(max_batch=2, max_h=image_hw[0], max_w=image_hw[1])
    try:
        heat, paf = g.postnet([big[:, :, 7:57]], crops, image_hw, angles=[22.5], paf_dtype=t.float64)
        assert np.array_equal(heat.cpu().numpy(), ref_heat.astype(np.float32)) and np.array_equal(paf.cpu().numpy(), ref_paf)
    finally:
        g.close()


@pytest.mark.parametrize("angles", [[22.5], [0.0, 5.0]])
def test_nan_scrub(env, angles):
    """NaN inputs spread through the taps as in the port.  The image is not the crop's size: a resize to the same size
    is a copy in cv2 and skipped by the kernels, while the port's resize multiplies the neighbours by weight 0 and so
    spreads NaNs one step further."""
    out = _network_like_output(env, 78, 1, 16, 16, 2)
    out[0, 0, 3, 5, 5] = np.nan
    out[0, 0, 35, 2, 9] = np.nan
    outs, crops, image_hw = [out] * len(angles), [(64, 64)] * len(angles), (56, 60)
    ref_heat, ref_paf = _port_maps(env, outs, crops, angles, 4, image_hw, nan_scrub=True)
    heat, paf, _, _ = _run(env, outs, crops, angles, image_hw, nan_scrub=True, paf_dtype=env.torch.float64)
    _, paf_raw, _, _ = _run(env, outs, crops, angles, image_hw, paf_dtype=env.torch.float64)
    assert np.isnan(paf_raw).any() and not np.isnan(paf).any() and not np.isnan(heat).any()
    assert np.array_equal(heat, ref_heat.astype(np.float32)) and np.array_equal(paf, ref_paf)


def test_all_zero_angles_are_spg_postnet_byte_for_byte(env):
    t = env.torch
    sizes, crops, image_hw = CASES["three_scales"]
    outs = [t.from_numpy(_network_like_output(env, 31 + k, 2, h, w, 3)).to(env.dev) for k, (h, w) in enumerate(sizes)]
    g = env.Grouper(max_batch=2, max_h=image_hw[0], max_w=image_hw[1])
    try:
        h0, p0 = g.postnet(outs, crops, image_hw)
        k0 = g.postnet_kernel()
        h1, p1 = g.postnet(outs, crops, image_hw, angles=[0.0, -0.0, 0.0])
        assert g.postnet_kernel() == k0
        assert t.equal(h0.view(t.int32), h1.view(t.int32)) and t.equal(p0.view(t.int64), p1.view(t.int64))
    finally:
        g.close()


@pytest.mark.parametrize("bad", [float("nan"), float("inf"), -float("inf")])
def test_non_finite_angles_are_rejected(env, bad):
    t = env.torch
    out = t.from_numpy(_network_like_output(env, 5, 1, 8, 8, 1)).to(env.dev)
    g = env.Grouper(max_batch=1, max_h=32, max_w=32)
    try:
        with pytest.raises(env.GroupingError, match="not finite"):
            g.postnet([out, out], [(32, 32)] * 2, (32, 32), angles=[5.0, bad])
    finally:
        g.close()


@pytest.mark.parametrize("angle", [5.0, -22.5])
def test_rotated_postnet_then_grouping_equals_the_checkers_pipeline(env, angle):
    """Network output -> spg_postnet_rotated -> grouping (float32 planes, float64 arithmetic) on the device, against
    rotation_port (float64 maps, as predict() returns them) -> C checker."""
    from parity import diff_structures
    t = env.torch
    n, h, w = 4, 32, 40
    out = _network_like_output(env, 1200 + int(angle), n, h, w, 6, noise=0.004)
    image_hw = (4 * h, 4 * w)
    ref_heat, ref_paf = _port_maps(env, [out], [image_hw], [angle], 4, image_hw)
    params = env.skeleton.default_params()
    o = env.so.group_batch(ref_heat.astype(np.float32), np.ascontiguousarray(ref_paf), env.skeleton.LIMBS, image_hw[0], params)
    g = env.Grouper(max_batch=n, max_h=image_hw[0], max_w=image_hw[1], max_peaks_per_part=128, max_person_rows=128)
    try:
        heat, paf = g.postnet([t.from_numpy(out).to(env.dev)], [image_hw], image_hw, angles=[angle])
        g.group_device(heat, paf, image_hw[0], params, paf_as_f64=True)
        r = g.fetch()
    finally:
        g.close()
    assert (r.status == 0).all() and (o.status == 0).all() and r.n_persons.sum() >= n
    for i in range(n):
        d = diff_structures(o.as_reference_structures(i), r.as_reference_structures(i), float_tol=0.0)
        assert not d, f"image {i}:\n" + "\n".join(d)


def test_device_predict_with_rotation_search(env):
    """dropin.predict with rotation_search = [-5, 0, 5]: the network sees cv2.warpAffine(padded / 255, M) and its
    mirror for every item, and the maps are the checker's three-item average."""
    import cv2
    t = env.torch
    from improved_body_parts_b200 import dropin
    rng = np.random.default_rng(9)
    image = rng.integers(0, 255, size=(150, 210, 3), dtype=np.uint8)
    params = dict(env.skeleton.default_params(), scale_search=[1.0], rotation_search=[-5.0, 0.0, 5.0])
    model_params = dict(boxsize=160, stride=4, max_downsample=64, padValue=128)
    scale = 1.0 * 160 / 150
    resized = cv2.resize(image, (0, 0), fx=scale, fy=scale, interpolation=cv2.INTER_CUBIC)
    padded, pad = dropin.pad_right_down_corner(resized, 64, 128)
    base = np.float32(padded / 255)
    h, w = padded.shape[0] // 4, padded.shape[1] // 4
    outs = [_network_like_output(env, 4400 + k, 1, h, w, 5, noise=0.004)[0] for k in range(3)]
    seen = []

    def model(x):
        seen.append(x.cpu().numpy())
        return [[t.from_numpy(outs[len(seen) - 1]).to(x.device)]]

    dropin.configure(device=0, limbs=env.skeleton.LIMBS)
    try:
        heatmap, paf = dropin.predict(image, params, model, model_params, 20, 30, "synthetic")
    finally:
        dropin.configure()
    assert len(seen) == 3
    for x, angle in zip(seen, (-5.0, 0.0, 5.0)):
        want = base if angle == 0 else cv2.warpAffine(
            base, cv2.getRotationMatrix2D((base.shape[0] / 2, base.shape[1] / 2), angle, 1), (0, 0))
        assert np.array_equal(x[0], want) and np.array_equal(x[1], want[:, ::-1])
    ref_heat, ref_paf = _port_maps(env, [o[None] for o in outs], [resized.shape[:2]] * 3, [-5.0, 0.0, 5.0], 4,
                                   image.shape[:2])
    assert heatmap.shape == (150, 210, 18) and not paf.as_f64
    assert np.array_equal(heatmap.numpy(), ref_heat[0].transpose(1, 2, 0).astype(np.float32).astype(np.float64))
    assert np.array_equal(paf.numpy(), ref_paf[0].transpose(1, 2, 0))


def test_wire_signal_survives_a_postnet_that_grows_its_workspace(env):
    """Arm the in-kernel wire signal, run a five-scale postnet (it allocates the float64 keypoint sums), then the fused
    match + assemble: the signal lands and the records are the checker's."""
    from improved_body_parts_b200 import wire
    t = env.torch
    n, H = 3, 64
    sizes, crops, image_hw = CASES["five_scales"]
    outs = [t.from_numpy(_network_like_output(env, 808 + k, n, a, b, 3)).to(env.dev) for k, (a, b) in enumerate(sizes)]
    heat, paf = env.synth.make_batch(818, n, H, H, 5)
    params = env.skeleton.default_params()
    o = env.so.group_batch(heat, paf, env.skeleton.LIMBS, H, params)
    g = env.Grouper(max_batch=n, max_h=H, max_w=H)
    try:
        buf = t.zeros((n, g.wire_record_bytes()), dtype=t.uint8, device=env.dev)
        word = t.zeros((1,), dtype=t.int64, device=env.dev)
        g.set_wire_output(buf.data_ptr())
        g.arm_wire_signal(word.data_ptr(), 41)
        g.postnet(outs, crops, image_hw, angles=[0.0, 5.0, 0.0, 0.0, 0.0])
        g.group_device(t.from_numpy(heat).to(env.dev), t.from_numpy(paf).to(env.dev), H, params)
        t.cuda.synchronize()
        assert word.tolist() == [41]
        rec = wire.as_records(buf.cpu().numpy(), 17, g.capR)
    finally:
        g.close()
    for i in range(n):
        P = int(o.n_persons[i])
        xy, sc = o.to_coco(i, env.skeleton.COCO_FROM_PART)
        assert int(rec[i]["n_persons"]) == P and np.array_equal(rec[i]["rows"]["xy"][:P], xy) and \
            np.array_equal(rec[i]["rows"]["score"][:P], sc)
