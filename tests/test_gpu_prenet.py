"""GPU: the pre-network stage (spg_prenet, csrc/prenet.cuh -- evaluate.py:98-116) against its CPU checker
tests/prenet_port.py, which tests/test_prenet_port.py pins to cv2 (IPP off) bit for bit.

The kernels spell out the port's integer / float32 / fixed-point operations one by one, so the bar is BIT-IDENTICAL
network inputs."""
import ctypes as C

import numpy as np
import pytest

import prenet_port as P
from test_gpu_postnet import _network_like_output
from test_prenet_port import GEOMETRIES, _image

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def env(cuda_device):
    import torch
    from improved_body_parts_b200 import skeleton, synth
    from improved_body_parts_b200.grouping import Grouper, GroupingError
    from oracle import spg_oracle as so

    class Env:
        pass

    e = Env()
    e.torch, e.skeleton, e.synth, e.Grouper, e.GroupingError, e.so, e.dev = \
        torch, skeleton, synth, Grouper, GroupingError, so, cuda_device
    e.g = Grouper(max_batch=1, max_h=64, max_w=64)
    yield e
    e.g.close()


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def _check(env, img, scale, angles, md=64, pv=128, dev_img=None):
    t = env.torch
    want, crop = P.network_inputs(img, scale, angles, md, pv)
    got, got_crop = env.g.prenet(t.from_numpy(img).to(env.dev) if dev_img is None else dev_img, scale, angles,
                                 max_downsample=md, pad_value=pv)
    assert got_crop == crop and tuple(got.shape) == want.shape
    got = got.cpu().numpy()
    for k in range(len(angles)):
        d = int((_bits(got[k]) != _bits(want[k])).sum())
        assert d == 0, f"angle {angles[k]}: {d} values differ from the port"


@pytest.mark.parametrize("h,w,scale", GEOMETRIES)
def test_prenet_equals_the_port(env, h, w, scale):
    _check(env, _image(h * 7 + w, h, w), scale, [0.0])


def test_several_angles_in_one_call(env):
    _check(env, _image(11, 150, 210), 160 / 150, [-5.0, 0.0, 5.0, 22.5, 90.0, 180.0, -37.3])


@pytest.mark.parametrize("md,pv", [(64, 0), (64, 255), (8, 128), (8, 0)])
def test_max_downsample_and_pad_value(env, md, pv):
    _check(env, _image(md + pv, 333, 500), 0.5 * 640 / 333, [0.0, 5.0], md=md, pv=pv)


@pytest.mark.parametrize("h,w,scale", [(120, 90, 1.7), (37, 51, 0.45), (1, 9, 1.6)])
def test_strided_input_rows(env, h, w, scale):
    """A crop of a larger frame: row stride (w + 37) * 3 bytes, starting 11 pixels in."""
    t = env.torch
    frame = _image(5, h + 10, w + 37)
    dev_frame = t.from_numpy(frame).to(env.dev)
    crop = dev_frame[5:5 + h, 11:11 + w]
    assert crop.stride(0) == (w + 37) * 3
    _check(env, np.ascontiguousarray(frame[5:5 + h, 11:11 + w]), scale, [0.0, -5.0], dev_img=crop)


def test_the_workspace_grows_and_shrinks_without_harm(env):
    """A large scale after small ones and a small one after the large: each call equals the port."""
    img = _image(21, 90, 120)
    for s in (0.5, 6.0, 0.8):
        _check(env, img, s, [0.0, 5.0])


def test_bad_arguments_are_rejected(env):
    t, g = env.torch, env.g
    img = t.zeros((40, 50, 3), dtype=t.uint8, device=env.dev)
    for kw in (dict(scale=0.0), dict(scale=-1.0), dict(scale=float("nan")), dict(scale=float("inf")),
               dict(scale=1.0, angles=[0.0, float("nan")]), dict(scale=1.0, angles=[float("inf")]),
               dict(scale=1000.0), dict(scale=1.0, max_downsample=0), dict(scale=1.0, max_downsample=-8),
               dict(scale=1.0, pad_value=256), dict(scale=1.0, pad_value=-1), dict(scale=0.001)):
        with pytest.raises(env.GroupingError):
            g.prenet(img, **kw)
    with pytest.raises(env.GroupingError):
        g.prenet(t.zeros((40, 50, 4), dtype=t.uint8, device=env.dev), 1.0)
    with pytest.raises(env.GroupingError):
        g.prenet(img.float(), 1.0)
    # the C entry point itself: channels != 3 and a short row stride
    out = t.empty((1, 2, 64, 64, 3), dtype=t.float32, device=env.dev)
    ang = (C.c_double * 1)(0.0)
    args = lambda ch, rs: (g._h, C.c_void_p(img.data_ptr()), C.c_int64(rs), 40, 50, ch, C.c_double(1.0), ang, 1, 64, 128,
                           C.c_void_p(out.data_ptr()), C.c_int64(out[0].numel()), None)
    assert g._lib.spg_prenet(*args(4, 200)) == -1 and b"channels" in g._lib.spg_last_error(g._h)
    assert g._lib.spg_prenet(*args(1, 50)) == -1
    assert g._lib.spg_prenet(*args(3, 149)) == -1
    assert g._lib.spg_prenet(*args(3, 150)) == 0
    t.cuda.synchronize()


def test_wire_signal_survives_a_prenet_that_grows_its_workspace(env):
    """Arm the in-kernel wire signal, run a prenet on a fresh handle (it allocates the padded-image workspace), then the
    fused match + assemble: the signal lands and the records are the checker's."""
    from improved_body_parts_b200 import wire
    t = env.torch
    n, H = 3, 64
    heat, paf = env.synth.make_batch(828, n, H, H, 5)
    params = env.skeleton.default_params()
    o = env.so.group_batch(heat, paf, env.skeleton.LIMBS, H, params)
    g = env.Grouper(max_batch=n, max_h=H, max_w=H)
    try:
        buf = t.zeros((n, g.wire_record_bytes()), dtype=t.uint8, device=env.dev)
        word = t.zeros((1,), dtype=t.int64, device=env.dev)
        g.set_wire_output(buf.data_ptr())
        g.arm_wire_signal(word.data_ptr(), 43)
        g.prenet(t.from_numpy(_image(1, 200, 300)).to(env.dev), 2.0, [0.0, 5.0])
        g.prenet(t.from_numpy(_image(2, 200, 300)).to(env.dev), 4.0, [0.0])  # grows it again
        g.group_device(t.from_numpy(heat).to(env.dev), t.from_numpy(paf).to(env.dev), H, params)
        t.cuda.synchronize()
        assert word.tolist() == [43]
        rec = wire.as_records(buf.cpu().numpy(), 17, g.capR)
    finally:
        g.close()
    for i in range(n):
        P_ = int(o.n_persons[i])
        xy, sc = o.to_coco(i, env.skeleton.COCO_FROM_PART)
        assert int(rec[i]["n_persons"]) == P_ and np.array_equal(rec[i]["rows"]["xy"][:P_], xy) and \
            np.array_equal(rec[i]["rows"]["score"][:P_], sc)


def _predict(env, image, params, model_params, device_input, outs):
    """dropin.predict with a recording model stub that answers item k with ``outs[k]``."""
    from improved_body_parts_b200 import dropin
    t = env.torch
    seen = []

    def model(x):
        seen.append(x.cpu().numpy())
        return [[t.from_numpy(outs[len(seen) - 1]).to(x.device)]]

    dropin.configure(device=0, limbs=env.skeleton.LIMBS, device_input=device_input)
    try:
        heat, paf = dropin.predict(image, params, model, model_params, 20, 30, "synthetic")
    finally:
        dropin.configure(device_input=False)
    return seen, heat, paf


def test_device_input_predict_feeds_the_ports_tensors_and_matches_the_host_path(env):
    """scale_search [0.5, 1, 2] x rotation_search [-5, 0, 5]: the model sees exactly the port's pairs, in the loop's order;
    with the same network answers the maps equal those of the host-input path."""
    import cv2
    image = _image(77, 150, 210)
    params = dict(env.skeleton.default_params(), scale_search=[0.5, 1.0, 2.0], rotation_search=[-5.0, 0.0, 5.0])
    model_params = dict(boxsize=160, stride=4, max_downsample=64, padValue=128)
    want = []
    for x in params["scale_search"]:
        pairs, _ = P.network_inputs(image, x * 160 / 150, params["rotation_search"], 64, 128)
        want.extend(pairs)
    outs = [_network_like_output(env, 4500 + k, 1, p.shape[1] // 4, p.shape[2] // 4, 4, noise=0.004)[0]
            for k, p in enumerate(want)]
    seen, heat, paf = _predict(env, image, params, model_params, True, outs)
    assert len(seen) == 9
    for k, (x, y) in enumerate(zip(seen, want)):
        assert x.dtype == np.float32 and np.array_equal(_bits(x), _bits(y)), f"item {k}"
    # a CUDA uint8 tensor is taken as it is
    seen_t, heat_t, paf_t = _predict(env, env.torch.from_numpy(image).to(env.dev), params, model_params, True, outs)
    assert all(np.array_equal(_bits(x), _bits(y)) for x, y in zip(seen_t, want))
    seen_h, heat_h, paf_h = _predict(env, image, params, model_params, False, outs)
    assert [x.shape for x in seen_h] == [x.shape for x in seen]
    saved = cv2.ipp.useIPP()
    try:  # the host path is cv2's: with IPP off it feeds the model the same tensors
        cv2.ipp.setUseIPP(False)
        seen_off, _, _ = _predict(env, image, params, model_params, False, outs)
    finally:
        cv2.ipp.setUseIPP(saved)
    assert all(np.array_equal(_bits(x), _bits(y)) for x, y in zip(seen_off, want))
    for a, b in ((heat, heat_h), (paf, paf_h), (heat_t, heat_h), (paf_t, paf_h)):
        assert a.shape == b.shape and a.as_f64 == b.as_f64 and np.array_equal(a.numpy(), b.numpy())


def test_install_device_input(env):
    from improved_body_parts_b200 import dropin
    import types
    mod = types.SimpleNamespace(limbSeq=env.skeleton.LIMBS, posenet=None)
    with pytest.raises(ValueError):
        dropin.install(mod, device_input=True)
    try:
        dropin.install(mod, device_predict=True, device_input=True)
        assert dropin._device_input and mod.predict is not None
    finally:
        dropin.configure(device_input=False)
