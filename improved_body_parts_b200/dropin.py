"""Drop-in replacements for the reference's grouping call sites (evaluate.py:509-511).

The reference has no plugin interface: ``process()`` resolves three module-level functions by name,

    all_peaks                  = find_peaks(heatmap, params)                                  # evaluate.py:169
    connection_all, special_k  = find_connections(all_peaks, paf, oriImg.shape[0], params)    # evaluate.py:206
    subset, candidate          = find_people(connection_all, special_k, all_peaks, params)    # evaluate.py:279

so the boundary is "same names, same arguments, same Python return structures".  The functions below honour it
and run every stage on the GPU through ``libspgroup.so``; ``install(evaluate)`` rebinds the three names in an
already imported ``evaluate`` module (INTEGRATION.md shows the launcher).  Argument meaning and quirks follow
the reference: ``image_width`` is really the image height (evaluate.py:510), border peaks come back as integer
coordinates, ``special_k`` limbs get ``[]``, ``candidate`` is the flattened peak table.

Each stage is self-contained (it uploads what it is given), so the functions can be swapped in one at a time;
``group()`` is the fused call for code that owns the call site and wants one device round trip.
There is no CPU path: without the CUDA library / an sm_100 GPU these functions raise ``GroupingError``.
"""
from __future__ import annotations

from itertools import product
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np

from .grouping import Grouper, GroupingError, GroupResult
from .skeleton import COCO_FROM_PART, LIMBS, NUM_PARTS, GroupParams

_limbs: Tuple[Tuple[int, int], ...] = LIMBS
_device = 0
_variant = "evaluate"
_device_input = False
_groupers: Dict[int, Grouper] = {}
CAP_PEAKS, CAP_CANDS, CAP_ROWS = 128, 4096, 128
MAX_DIM = 32767  # the C ABI's limit; the workspace does not depend on the map size, so ONE handle serves every image size


def configure(limbs: Optional[Sequence[Tuple[int, int]]] = None, device: Optional[int] = None,
              variant: Optional[str] = None, device_input: Optional[bool] = None) -> None:
    """Select the limb table (default: the Canonical ``limbs_conn``, config/config.py:94), the CUDA device, the
    behavioural variant: ``"evaluate"`` (evaluate.py, the default) or ``"demo"`` (demo_image.py's inlined copy, which
    differs at :288, :414-415 and :533 -- SURVEY.md 3.2), and where ``predict`` builds the network input:
    ``device_input=True`` on the GPU (``Grouper.prenet``), ``False`` (the default) with cv2 on the host as the reference."""
    global _limbs, _device, _variant, _device_input
    if device_input is not None:
        _device_input = bool(device_input)
    if limbs is not None:
        _limbs = tuple((int(a), int(b)) for a, b in limbs)
    if device is not None:
        _device = int(device)
    if variant is not None:
        if variant not in ("evaluate", "demo"):
            raise ValueError("variant must be 'evaluate' or 'demo'")
        _variant = variant
    for g in _groupers.values():
        g.close()
    _groupers.clear()


def _grouper(H: int = 0, W: int = 0) -> Grouper:
    """The one native handle of the current device (evaluate.py runs over images of hundreds of different sizes: a
    handle per size, as in round 1, grew device memory and streams without bound)."""
    g = _groupers.get(_device)
    if g is None:
        g = Grouper(_limbs, NUM_PARTS, COCO_FROM_PART, max_batch=1, max_h=MAX_DIM, max_w=MAX_DIM,
                    max_peaks_per_part=CAP_PEAKS, max_cands_per_limb=CAP_CANDS, max_person_rows=CAP_ROWS, device=_device)
        _groupers[_device] = g
    return g


def _params(params):
    """The reference's params dict -> what the library runs with (the demo variant adds its three deviations)."""
    if isinstance(params, GroupParams):
        return params
    return GroupParams.demo(params) if _variant == "demo" else params


def _check(r: GroupResult) -> None:
    if r.status[0]:
        raise GroupingError(f"grouping capacity exceeded or invalid sample index (status {int(r.status[0]):#x}); "
                            f"capacities: {CAP_PEAKS} peaks/part, {CAP_CANDS} candidates/limb, {CAP_ROWS} person rows")


def _maps_to_device(hwc: np.ndarray, channels: int, dtype):
    """``[H, W, C]`` host maps (what predict() returns) -> ``[1, channels, H, W]`` device planes of ``dtype``.

    The array goes up as it is and is transposed / cast on the device: a numpy transpose of a 512x512x30 float64 array
    alone cost 40 ms per image (round 2 measurement).  The float64 -> float32 cast rounds to nearest even on both sides."""
    import torch
    arr = np.asarray(hwc)
    if arr.dtype not in (np.float32, np.float64):
        arr = arr.astype(np.float64)
    t = torch.from_numpy(np.ascontiguousarray(arr)).to(f"cuda:{_device}")
    want = torch.float32 if dtype == np.float32 else torch.float64
    return t[:, :, :channels].permute(2, 0, 1).to(want).contiguous()[None]


class DeviceMaps:
    """Averaged maps that stay on the GPU between ``predict`` and the grouping functions (what ``dropin.predict``
    returns in place of the reference's ``[H, W, C]`` float64 host arrays).  ``numpy()`` gives the reference's array."""

    def __init__(self, tensor, as_f64: bool):
        self.tensor, self.as_f64 = tensor, as_f64  # [1, C, H, W]; as_f64: float32 storage of the float64 values
        self.shape = (int(tensor.shape[2]), int(tensor.shape[3]), int(tensor.shape[1]))

    def numpy(self) -> np.ndarray:
        return self.tensor[0].permute(1, 2, 0).double().cpu().numpy()


#: what the last stage left on the device, so that the next stage does not upload it again when it is handed the very
#: objects the previous stage returned (the call sequence of evaluate.py:509-511)
_state: Dict[str, object] = {}


def pad_right_down_corner(img: np.ndarray, stride: int, pad_value: int) -> Tuple[np.ndarray, list]:
    """utils/util.py:44-64: pad below / to the right up to a multiple of ``stride`` with ``pad_value``."""
    h, w = img.shape[:2]
    pad = [0, 0, 0 if h % stride == 0 else stride - h % stride, 0 if w % stride == 0 else stride - w % stride]
    return np.pad(img, ((0, pad[2]), (0, pad[3]), (0, 0)), constant_values=pad_value), pad


def predict(image, params, model, model_params, heat_layers=None, paf_layers=None, input_image_path=None):
    """evaluate.py:83-166 with everything after the forward pass on the device.

    Same arguments as the reference's ``predict``.  By default the image is scaled and padded exactly as there (cv2,
    host) and, for an item of ``rotation_search`` with a non-zero angle, rotated with ``cv2.warpAffine`` (:108-111,
    host): the network input is bit-identical to the reference's with cv2 as it comes (IPP on).  With
    ``configure(device_input=True)`` the image goes up once as uint8 (a CUDA uint8 ``[H, W, 3]`` tensor is taken as it
    is) and ``Grouper.prenet`` builds every item on the GPU: bit-identical to the reference's input with cv2's IPP off
    (``cv2.ipp.setUseIPP(False)``); with IPP on, cv2's uint8 resize differs by at most 1 in a few percent of the values.
    The network runs on the image and its mirror (:116-124), and the flip ensemble, both bicubic resizes, the warp
    back, the crop and the float64 average over ``product(scale_search, rotation_search)`` (:126-161) happen in
    ``spg_postnet`` / ``spg_postnet_rotated`` -- the maps never visit the host.
    Returns two ``DeviceMaps`` (heatmap, paf) that ``find_peaks`` / ``find_connections`` / ``group`` accept directly."""
    import torch
    if _device_input:
        return _predict_device_input(image, params, model, model_params)
    import cv2
    g = _grouper()
    multiplier = [x * model_params["boxsize"] / image.shape[0] for x in params["scale_search"]]
    outs, crops, angles = [], [], []
    for scale, angle in product(multiplier, params["rotation_search"]):  # evaluate.py:89-90
        if scale * image.shape[0] > 2600 or scale * image.shape[1] > 3800:  # evaluate.py:94-96
            scale = min(2600 / image.shape[0], 3800 / image.shape[1])
        image_to_test = cv2.resize(image, (0, 0), fx=scale, fy=scale, interpolation=cv2.INTER_CUBIC)
        padded, _ = pad_right_down_corner(image_to_test, model_params["max_downsample"], model_params["padValue"])
        input_img = np.float32(padded / 255)
        if angle != 0:  # evaluate.py:108-111; the maps are warped back on the device
            rotate_matrix = cv2.getRotationMatrix2D((input_img.shape[0] / 2, input_img.shape[1] / 2), angle, 1)
            input_img = cv2.warpAffine(input_img, rotate_matrix, (0, 0))
        pair = np.concatenate((input_img[None, ...], input_img[:, ::-1, :].copy()[None, ...]), axis=0)
        outs.append(_forward(model, torch.from_numpy(pair).to(f"cuda:{_device}")))
        crops.append(image_to_test.shape[:2])
        angles.append(float(angle))
    return _postnet(g, outs, crops, image.shape[:2], model_params, angles)


def _forward(model, pair):
    """The forward pass of one item (:116-126): the last stack's finest-scale output, ``[1, 2, C, h, w]``."""
    import torch
    with torch.no_grad():
        out = model(pair)[-1][0]
    if out.dtype not in (torch.float32, torch.float16):
        out = out.float()
    return out[None].contiguous()


def _postnet(g: Grouper, outs, crops, image_hw, model_params, angles):
    import torch
    heat, paf = g.postnet(outs, crops, image_hw, stride=int(model_params["stride"]), nan_scrub=_variant == "demo",
                          angles=angles)
    return DeviceMaps(heat, False), DeviceMaps(paf, paf.dtype == torch.float32)


def _predict_device_input(image, params, model, model_params):
    """``predict`` with the network input built on the device: one upload, one ``prenet`` per scale."""
    import torch
    g = _grouper()
    dev = torch.device("cuda", _device)
    if torch.is_tensor(image):
        img = image.to(dev)
    else:
        img = torch.from_numpy(np.ascontiguousarray(image)).to(dev)
    h, w = int(img.shape[0]), int(img.shape[1])
    rotation = [float(a) for a in params["rotation_search"]]
    outs, crops, angles = [], [], []
    for scale in (x * model_params["boxsize"] / h for x in params["scale_search"]):  # evaluate.py:89-90
        if scale * h > 2600 or scale * w > 3800:  # evaluate.py:94-96
            scale = min(2600 / h, 3800 / w)
        pairs, crop = g.prenet(img, scale, rotation, max_downsample=int(model_params["max_downsample"]),
                               pad_value=int(model_params["padValue"]))
        for k, angle in enumerate(rotation):  # product(multiplier, rotate_angle): scale-major, angle-minor
            outs.append(_forward(model, pairs[k]))
            crops.append(crop)
            angles.append(angle)
    return _postnet(g, outs, crops, (h, w), model_params, angles)


def _upload_peaks(g: Grouper, all_peaks) -> None:
    if _state.get("peaks") is all_peaks and _state.get("handle") is g:
        return  # still on the device from our own find_peaks
    _state.clear()
    counts = [len(p) for p in all_peaks]
    flat = [t for part in all_peaks for t in part]
    g.upload_peaks(0, counts, [float(t[0]) for t in flat], [float(t[1]) for t in flat], [np.float32(t[2]) for t in flat])


# ---- the three reference functions ---------------------------------------------------------------------
def find_peaks(heatmap_avg, params):
    """evaluate.py:169-203.  ``heatmap_avg [H,W,>=18]`` -> list[18] of [(x, y, score, id), ...]."""
    H, W = heatmap_avg.shape[:2]
    g = _grouper(H, W)
    heat = heatmap_avg.tensor if isinstance(heatmap_avg, DeviceMaps) else _maps_to_device(heatmap_avg, NUM_PARTS, np.float32)
    g.nms_peaks(heat, _params(params))  # the cast is evaluate.py:173
    r = g.fetch(1)
    _check(r)
    all_peaks = r.as_reference_structures(0)[0]
    _state.clear()
    _state.update(peaks=all_peaks, handle=g)
    return all_peaks


def find_connections(all_peaks, paf_avg, image_width, params):
    """evaluate.py:206-276.  ``paf_avg [H,W,L]`` float32 or float64 -> (connection_all, special_k)."""
    H, W = paf_avg.shape[:2]
    g = _grouper(H, W)
    _upload_peaks(g, all_peaks)
    if isinstance(paf_avg, DeviceMaps):
        g.limb_score(paf_avg.tensor, image_width, _params(params), paf_as_f64=paf_avg.as_f64)
    else:
        dtype = np.float64 if np.asarray(paf_avg).dtype == np.float64 else np.float32
        g.limb_score(_maps_to_device(paf_avg, len(_limbs), dtype), image_width, _params(params))
    g.limb_match(1, _params(params))
    r = g.fetch(1)
    _check(r)
    # ids in the rows are those of the caller's all_peaks (:267), not positions in our tables
    _, conns, special, _, _ = r.as_reference_structures(0)
    for k, rows in enumerate(conns):
        if isinstance(rows, list) or not len(rows):
            continue
        a, b = _limbs[k]
        rows[:, 0] = np.array([t[3] for t in all_peaks[a]], np.float64)[rows[:, 3].astype(np.int64)]
        rows[:, 1] = np.array([t[3] for t in all_peaks[b]], np.float64)[rows[:, 4].astype(np.int64)]
    _state.update(conns=conns, special=special)
    return conns, special


def find_people(connection_all, special_k, all_peaks, params):
    """evaluate.py:279-498 -> (subset [P,20,2] float64, candidate [N,4] float64)."""
    g = _grouper()  # assembly does not depend on the map size
    if _state.get("conns") is connection_all and _state.get("special") is special_k and _state.get("peaks") is all_peaks \
            and _state.get("handle") is g:  # evaluate.py:509-511 handing our own objects back: everything is still on the device
        g.assemble(1, _params(params))
        r = g.fetch(1)
        _check(r)
        return r.subset[0, :int(r.n_persons[0])].copy(), np.array([item for sublist in all_peaks for item in sublist])
    _upload_peaks(g, all_peaks)
    special = set(int(k) for k in special_k)
    counts, ij, sc, nm = [], [], [], []
    for k, rows in enumerate(connection_all):
        if k in special:
            counts.append(-1)
            continue
        rows = np.asarray(rows, np.float64).reshape(-1, 6)
        counts.append(len(rows))
        ij.append(rows[:, 3:5].astype(np.int32))
        sc.append(rows[:, 2])
        nm.append(rows[:, 5])
    g.upload_connections(0, counts, np.concatenate(ij) if ij else np.zeros((0, 2), np.int32),
                         np.concatenate(sc) if sc else np.zeros(0), np.concatenate(nm) if nm else np.zeros(0))
    g.assemble(1, _params(params))
    r = g.fetch(1)
    _check(r)
    subset = r.subset[0, :int(r.n_persons[0])].copy()
    candidate = np.array([item for sublist in all_peaks for item in sublist])  # evaluate.py:283, verbatim semantics
    # subset holds positions in the flattened table; the reference stores the peaks' own ids there (equal unless
    # the caller renumbered all_peaks)
    flat_ids = [t[3] for part in all_peaks for t in part]
    if flat_ids != list(range(len(flat_ids))):
        ids = np.asarray(flat_ids, np.float64)
        sel = subset[:, :-2, 0] >= 0
        subset[:, :-2, 0][sel] = ids[subset[:, :-2, 0][sel].astype(int)]
    return subset, candidate


def group(heatmap_avg, paf_avg, image_extent, params):
    """Fused peaks -> connections -> people: one upload, four kernels, one download.

    Returns ``(all_peaks, connection_all, special_k, subset, candidate)`` exactly as the three calls would."""
    H, W = heatmap_avg.shape[:2]
    g = _grouper(H, W)
    _state.clear()
    if isinstance(heatmap_avg, DeviceMaps):
        g.group_device(heatmap_avg.tensor, paf_avg.tensor, image_extent, _params(params), paf_as_f64=paf_avg.as_f64)
    else:
        dtype = np.float64 if np.asarray(paf_avg).dtype == np.float64 else np.float32
        g.group_device(_maps_to_device(heatmap_avg, NUM_PARTS, np.float32), _maps_to_device(paf_avg, len(_limbs), dtype),
                       image_extent, _params(params))
    r = g.fetch(1)
    _check(r)
    return r.as_reference_structures(0)


def keypoints(subset, candidate):
    """Tail of process() (evaluate.py:523-543): [(17 x (x, y) in COCO order, score)]."""
    out = []
    for row in subset:
        pts = []
        for part in COCO_FROM_PART:
            idx = row[part, 0]
            pts.append((0, 0) if idx == -1 else tuple(candidate[int(idx)][:2]))
        out.append((pts, 1 - 1.0 / row[-2, 0]))
    return out


def keypoint_heatmap_nms(heat, kernel: int = 3, thre: float = 0.1):
    """utils/util.py:177-183 -- the one seam demo_image.py offers (:213).  ``heat [1,C,H,W]`` tensor -> ``heat * keep``.

    Peaks come from the CUDA NMS kernel; the masked map is rebuilt from them (zeros elsewhere)."""
    import torch
    if kernel != 3:
        raise GroupingError("only the 3x3 NMS the reference uses is implemented")
    if heat.dim() != 4 or heat.shape[0] != 1:
        raise GroupingError("expected a [1,C,H,W] tensor")
    C, H, W = heat.shape[1:]
    g = Grouper(((0, 0),), C, (0,), max_batch=1, max_h=MAX_DIM, max_w=MAX_DIM, max_peaks_per_part=CAP_PEAKS,
                device=_device) if C != NUM_PARTS else _grouper(H, W)
    src = heat.to(f"cuda:{_device}", torch.float32).contiguous()
    _state.clear()
    g.nms_peaks(src, dict(thre1=float(thre), offset_radius=0))
    r = g.fetch(1)
    _check(r)
    out = torch.zeros_like(src)
    for c in range(C):
        n = int(min(r.peak_count[0, c], r.peak_anchor.shape[2]))
        if n:
            a = r.peak_anchor[0, c, :n].astype(np.int64)
            ys = torch.as_tensor((a >> 16) & 0x7fff, device=src.device)
            xs = torch.as_tensor(a & 0xffff, device=src.device)
            out[0, c, ys, xs] = src[0, c, ys, xs]
    if C != NUM_PARTS:
        g.close()
    return out.to(heat.device)


def install(evaluate_module, device_predict: bool = False, device_input: bool = False) -> None:
    """Rebind ``find_peaks / find_connections / find_people`` of an imported reference ``evaluate`` module.

    ``limbSeq`` is taken from the module (evaluate.py:54) so alternative skeletons keep working.  With
    ``device_predict`` the module's ``predict`` (:83-166) is replaced as well: the network of the module (the global
    ``posenet`` the reference's own predict uses, :124) feeds the device post-network stage and the maps stay on the GPU.
    ``device_input`` (with ``device_predict``) builds the network input on the GPU too -- equal to the reference's
    with cv2's IPP off, see ``predict``."""
    if device_input and not device_predict:
        raise ValueError("device_input needs device_predict")
    configure(limbs=getattr(evaluate_module, "limbSeq", _limbs), device_input=device_input)
    evaluate_module.find_peaks = find_peaks
    evaluate_module.find_connections = find_connections
    evaluate_module.find_people = find_people
    if device_predict:
        def _predict(image, params, model, model_params, heat_layers, paf_layers, input_image_path):
            return predict(image, params, getattr(evaluate_module, "posenet", model), model_params, heat_layers,
                           paf_layers, input_image_path)
        evaluate_module.predict = _predict
