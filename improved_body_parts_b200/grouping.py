"""ctypes binding of ``libspgroup.so`` (include/spgroup.h) -- the B200 grouping path.

This module is the host-side mirror of the reference's grouping interface: ``Grouper`` owns one native
handle (one per GPU / stream) and exposes the whole path (``group_device`` / ``group_host``) and the four
stages.  There is no CPU implementation behind it: if the CUDA library is missing or no sm_100 device is
present, construction raises.  PyTorch is used only as plumbing (device memory, streams, NCCL).
"""
from __future__ import annotations

import ctypes as C
import dataclasses
import os
from typing import Optional, Sequence, Tuple

import numpy as np

from .skeleton import COCO_FROM_PART, LIMBS, NUM_PARTS, GroupParams

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libspgroup.so")
ABI_VERSION = 2

ST_PEAK_OVERFLOW, ST_CAND_OVERFLOW, ST_ROW_OVERFLOW, ST_SAMPLE_INDEX, ST_ASSERT, ST_WIRE_OVERFLOW = 1, 2, 4, 8, 16, 32
F32, F64, F32_AS_F64, F16 = 0, 1, 2, 3

#: every symbol include/spgroup.h declares (checked by tests/test_abi.py against the built library)
EXPORTS = (
    "spg_create", "spg_destroy", "spg_last_error", "spg_abi_version", "spg_get_device_view", "spg_group_batch",
    "spg_group_host", "spg_host_alloc", "spg_host_free", "spg_nms_peaks", "spg_limb_score", "spg_limb_match",
    "spg_assemble", "spg_upload_peaks", "spg_upload_connections", "spg_download_peaks", "spg_download_connections",
    "spg_download_people", "spg_download_status", "spg_launch_count", "spg_stage_kernel", "spg_wire_record_bytes",
    "spg_set_wire_output", "spg_wire_create", "spg_wire_open", "spg_wire_close", "spg_wire_destroy", "spg_wire_signal",
    "spg_wire_wait", "spg_postnet", "spg_match_assemble", "spg_wire_signal_many", "spg_arm_wire_signal",
    "spg_postnet_rotated", "spg_prenet_size", "spg_prenet")


class GroupingError(RuntimeError):
    pass


class _Config(C.Structure):
    _fields_ = [("abi_version", C.c_int32), ("device", C.c_int32), ("n_parts", C.c_int32), ("n_limbs", C.c_int32),
                ("limbs", C.POINTER(C.c_int32)), ("n_out_joints", C.c_int32), ("out_from_part", C.POINTER(C.c_int32)),
                ("max_batch", C.c_int32), ("max_h", C.c_int32), ("max_w", C.c_int32),
                ("max_peaks_per_part", C.c_int32), ("max_cands_per_limb", C.c_int32), ("max_person_rows", C.c_int32)]


class _Params(C.Structure):
    _fields_ = [("thre1", C.c_double), ("thre2", C.c_double), ("connect_ration", C.c_double),
                ("len_rate", C.c_double), ("connection_tole", C.c_double), ("min_mean_score", C.c_double),
                ("mid_num", C.c_int32), ("offset_radius", C.c_int32), ("remove_recon", C.c_int32),
                ("min_parts", C.c_int32), ("crit1_strict", C.c_int32), ("refresh_len_check", C.c_int32)]


class _PostnetScale(C.Structure):
    _fields_ = [("net_out", C.c_void_p), ("dtype", C.c_int32), ("image_stride", C.c_int64), ("pair_stride", C.c_int64),
                ("chan_stride", C.c_int64), ("h", C.c_int32), ("w", C.c_int32), ("crop_h", C.c_int32), ("crop_w", C.c_int32)]


class _PostnetDesc(C.Structure):
    _fields_ = [("n_scales", C.c_int32), ("scales", C.POINTER(_PostnetScale)), ("stride", C.c_int32),
                ("paf_chan0", C.c_int32), ("heat_chan0", C.c_int32), ("flip_paf_ord", C.POINTER(C.c_int32)),
                ("flip_heat_ord", C.POINTER(C.c_int32)), ("nan_scrub", C.c_int32)]


class _DeviceView(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("max_batch", "n_parts", "n_limbs", "n_out_joints", "cap_peaks", "cap_cands",
                                          "cap_rows")] + \
               [(n, C.c_void_p) for n in ("peak_x", "peak_y", "peak_score", "peak_anchor", "peak_count", "conn_ij",
                                          "conn_score", "conn_norm", "conn_count", "cand_count", "surv_count", "subset",
                                          "n_persons", "people_xy", "people_score", "status")]


_lib = None


def load_library() -> C.CDLL:
    """Load ``libspgroup.so`` from the package directory.  Fails loudly; there is no fallback."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise GroupingError(f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; "
                                f"g.build()'` (or `make -C improved_body_parts_b200/csrc`).  There is no CPU fallback.")
        lib = C.CDLL(LIB_PATH)
        lib.spg_last_error.restype = C.c_char_p
        lib.spg_last_error.argtypes = [C.c_void_p]
        lib.spg_launch_count.restype = C.c_int64
        lib.spg_launch_count.argtypes = [C.c_void_p]
        lib.spg_stage_kernel.restype = C.c_char_p
        lib.spg_stage_kernel.argtypes = [C.c_void_p, C.c_int32]
        lib.spg_create.argtypes = [C.POINTER(_Config), C.POINTER(C.c_void_p)]
        lib.spg_destroy.argtypes = [C.c_void_p]
        lib.spg_destroy.restype = None
        lib.spg_wire_record_bytes.restype = C.c_int64
        lib.spg_wire_record_bytes.argtypes = [C.c_void_p]
        lib.spg_set_wire_output.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32]
        lib.spg_arm_wire_signal.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64]
        lib.spg_wire_create.argtypes = [C.c_int32, C.c_uint64, C.POINTER(C.c_void_p), C.c_char_p]
        lib.spg_wire_open.argtypes = [C.c_int32, C.c_char_p, C.POINTER(C.c_void_p)]
        lib.spg_wire_close.argtypes = [C.c_void_p]
        lib.spg_wire_destroy.argtypes = [C.c_int32, C.c_void_p]
        lib.spg_wire_signal.argtypes = [C.c_int32, C.c_void_p, C.c_uint64, C.c_void_p]
        lib.spg_wire_wait.argtypes = [C.c_int32, C.c_void_p, C.c_uint64, C.c_void_p]
        lib.spg_prenet_size.argtypes = [C.c_int32, C.c_int32, C.c_double, C.c_int32] + [C.POINTER(C.c_int32)] * 4
        lib.spg_prenet.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_double,
                                   C.POINTER(C.c_double), C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p]
        if lib.spg_abi_version() != ABI_VERSION:
            raise GroupingError("libspgroup.so ABI version mismatch")
        _lib = lib
    return _lib


def params_struct(params) -> _Params:
    """``params``: the reference's dict (utils/config keys), a GroupParams, or None for the defaults."""
    if params is None:
        gp = GroupParams()
    elif isinstance(params, GroupParams):
        gp = params
    else:
        gp = GroupParams.from_dict(dict(params))
    return _Params(gp.thre1, gp.thre2, gp.connect_ration, gp.len_rate, gp.connection_tole, gp.min_mean_score,
                   gp.mid_num, gp.offset_radius, gp.remove_recon, gp.min_parts, gp.crit1_strict, gp.refresh_len_check)


def _vp(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class _CudaView:
    """Zero-copy torch view of handle-owned device memory (``__cuda_array_interface__``)."""

    def __init__(self, ptr: int, shape: Tuple[int, ...], typestr: str):
        self.__cuda_array_interface__ = {"shape": tuple(int(s) for s in shape), "typestr": typestr,
                                         "data": (int(ptr), False), "version": 2, "strides": None}


@dataclasses.dataclass
class GroupResult:
    """Host copy of everything one call produced (dense arrays with the handle's capacities)."""
    K: int
    L: int
    limbs: np.ndarray
    peak_count: np.ndarray   # [N,K]
    peak_x: np.ndarray       # [N,K,capP] f64
    peak_y: np.ndarray
    peak_score: np.ndarray   # f32
    peak_anchor: np.ndarray  # u32: (y<<16)|x, bit 31 = border peak
    conn_count: np.ndarray   # [N,L], -1 = special_k
    cand_count: np.ndarray   # [N,L]
    conn_ij: np.ndarray      # [N,L,capP] u32 (i<<16)|j
    conn_score: np.ndarray
    conn_norm: np.ndarray
    n_persons: np.ndarray    # [N]
    subset: np.ndarray       # [N,capR,K+2,2]
    people_xy: np.ndarray    # [N,capR,J,2]
    people_score: np.ndarray  # [N,capR]
    status: np.ndarray       # [N] u32

    def as_reference_structures(self, n: int):
        """(all_peaks, connection_all, special_k, subset, candidate) exactly as evaluate.py:203,276,498 return them."""
        K, L = self.K, self.L
        capP = self.peak_x.shape[2]
        cnt = np.minimum(self.peak_count[n], capP)
        off = np.concatenate([[0], np.cumsum(cnt)])
        all_peaks, flat = [], []
        for c in range(K):
            lst = []
            for q in range(int(cnt[c])):
                anchor = int(self.peak_anchor[n, c, q])
                gid = int(off[c] + q)
                if anchor >> 31:
                    xy = (np.int64(anchor & 0xffff), np.int64((anchor >> 16) & 0x7fff))
                else:
                    xy = (np.float64(self.peak_x[n, c, q]), np.float64(self.peak_y[n, c, q]))
                lst.append(xy + (np.float32(self.peak_score[n, c, q]), gid))
                flat.append((float(self.peak_x[n, c, q]), float(self.peak_y[n, c, q]),
                             float(self.peak_score[n, c, q]), float(gid)))
            all_peaks.append(lst)
        connection_all, special_k = [], []
        for k in range(L):
            m = int(self.conn_count[n, k])
            if m < 0:
                special_k.append(k)
                connection_all.append([])
                continue
            a, b = (int(v) for v in self.limbs[k])
            ij = self.conn_ij[n, k, :m].astype(np.int64)
            rows = np.zeros((m, 6))
            rows[:, 3] = ij >> 16
            rows[:, 4] = ij & 0xffff
            rows[:, 0] = off[a] + rows[:, 3]
            rows[:, 1] = off[b] + rows[:, 4]
            rows[:, 2] = self.conn_score[n, k, :m]
            rows[:, 5] = self.conn_norm[n, k, :m]
            connection_all.append(rows)
        P = int(self.n_persons[n])
        subset = self.subset[n, :P].copy()
        candidate = np.array(flat, np.float64).reshape(-1, 4) if flat else np.zeros((0,))
        return all_peaks, connection_all, special_k, subset, candidate

    def keypoints(self, n: int):
        """process() tail (evaluate.py:523-543): list of ([17 x (x, y)], score)."""
        P = int(self.n_persons[n])
        return [([tuple(xy) for xy in self.people_xy[n, j]], float(self.people_score[n, j])) for j in range(P)]


# ---- peer memory + stream-ordered signalling (the NVLink gather; sharding.py drives it) ------------------------
def wire_create(device: int, nbytes: int) -> Tuple[int, bytes]:
    """Zero-filled device buffer other processes can map: ``(device address, 64-byte IPC handle)``."""
    lib = load_library()
    ptr, hd = C.c_void_p(), C.create_string_buffer(64)
    if lib.spg_wire_create(C.c_int32(device), C.c_uint64(nbytes), C.byref(ptr), hd) != 0:
        raise GroupingError("spg_wire_create failed: " + (lib.spg_last_error(None) or b"").decode())
    return int(ptr.value), hd.raw


def wire_open(device: int, ipc_handle: bytes) -> int:
    lib = load_library()
    ptr = C.c_void_p()
    if lib.spg_wire_open(C.c_int32(device), C.c_char_p(ipc_handle), C.byref(ptr)) != 0:
        raise GroupingError("spg_wire_open failed: " + (lib.spg_last_error(None) or b"").decode())
    return int(ptr.value)


def wire_close(peer_ptr: int) -> None:
    load_library().spg_wire_close(C.c_void_p(peer_ptr))


def wire_destroy(device: int, dev_ptr: int) -> None:
    load_library().spg_wire_destroy(C.c_int32(device), C.c_void_p(dev_ptr))


def wire_signal(device: int, word_ptr: int, value: int, stream) -> None:
    """Release-store ``value`` into a 64-bit word (local or peer memory) after everything earlier on ``stream``."""
    if load_library().spg_wire_signal(C.c_int32(device), C.c_void_p(word_ptr), C.c_uint64(value),
                                      C.c_void_p(int(getattr(stream, "cuda_stream", stream)))) != 0:
        raise GroupingError("spg_wire_signal failed")


def wire_signal_many(device: int, word_ptrs: Sequence[int], value: int, stream) -> None:
    """One launch that release-stores ``value`` into every word of ``word_ptrs`` (<= 32, local or peer memory)."""
    arr = (C.c_void_p * len(word_ptrs))(*[C.c_void_p(p) for p in word_ptrs])
    if load_library().spg_wire_signal_many(C.c_int32(device), arr, C.c_int32(len(word_ptrs)), C.c_uint64(value),
                                           C.c_void_p(int(getattr(stream, "cuda_stream", stream)))) != 0:
        raise GroupingError("spg_wire_signal_many failed")


def wire_wait(device: int, word_ptr: int, value: int, stream) -> None:
    """Make ``stream`` wait until the LOCAL 64-bit word is >= ``value`` (a stream memory operation, no SM involved)."""
    if load_library().spg_wire_wait(C.c_int32(device), C.c_void_p(word_ptr), C.c_uint64(value),
                                    C.c_void_p(int(getattr(stream, "cuda_stream", stream)))) != 0:
        raise GroupingError("spg_wire_wait failed")


def device_bytes_view(ptr: int, nbytes: int, device: int):
    """Zero-copy uint8 torch view of raw device memory."""
    import torch
    return torch.as_tensor(_CudaView(ptr, (int(nbytes),), "|u1"), device=torch.device("cuda", device))


def prenet_size(height: int, width: int, scale: float, max_downsample: int = 64):
    """``spg_prenet_size``: ``((crop_h, crop_w), (Hp, Wp))`` -- ``imageToTest``'s and ``imageToTest_padded``'s sizes
    for a ``height x width`` image at ``scale`` (evaluate.py:98-100)."""
    lib = load_library()
    v = [C.c_int32() for _ in range(4)]
    rc = lib.spg_prenet_size(int(height), int(width), float(scale), int(max_downsample), *(C.byref(x) for x in v))
    if rc != 0:
        raise GroupingError(f"spg_prenet_size failed ({rc}): {(lib.spg_last_error(None) or b'').decode()}")
    return (v[0].value, v[1].value), (v[2].value, v[3].value)


class Grouper:
    """One native grouping handle.  Not thread-safe; use one per stream / GPU."""

    def __init__(self, limbs: Sequence[Tuple[int, int]] = LIMBS, n_parts: int = NUM_PARTS,
                 out_from_part: Sequence[int] = COCO_FROM_PART, *, max_batch: int = 256, max_h: int = 128,
                 max_w: int = 128, max_peaks_per_part: int = 64, max_cands_per_limb: int = 1024,
                 max_person_rows: int = 96, device: int = 0):
        self._lib = load_library()
        self._h = C.c_void_p()
        self.limbs = np.ascontiguousarray(np.asarray(limbs, np.int32).reshape(-1, 2))
        self.out_from_part = np.ascontiguousarray(np.asarray(out_from_part, np.int32))
        self.K, self.L, self.J = int(n_parts), int(self.limbs.shape[0]), int(self.out_from_part.shape[0])
        self.max_batch, self.max_h, self.max_w = int(max_batch), int(max_h), int(max_w)
        self.capP, self.capC, self.capR = int(max_peaks_per_part), int(max_cands_per_limb), int(max_person_rows)
        self.device = int(device)
        cfg = _Config(ABI_VERSION, self.device, self.K, self.L, self.limbs.ctypes.data_as(C.POINTER(C.c_int32)), self.J,
                      self.out_from_part.ctypes.data_as(C.POINTER(C.c_int32)), self.max_batch, self.max_h, self.max_w,
                      self.capP, self.capC, self.capR)
        rc = self._lib.spg_create(C.byref(cfg), C.byref(self._h))
        if rc != 0:
            msg = self._lib.spg_last_error(None)
            self._h = C.c_void_p()
            raise GroupingError(f"spg_create failed ({rc}): {msg.decode() if msg else ''}")

    # -- lifetime ------------------------------------------------------------------------------
    def close(self) -> None:
        if getattr(self, "_h", None) and self._h.value:
            self._lib.spg_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def _check(self, rc: int, what: str) -> None:
        if rc != 0:
            msg = self._lib.spg_last_error(self._h)
            raise GroupingError(f"{what} failed ({rc}): {msg.decode() if msg else ''}")

    @property
    def launch_count(self) -> int:
        return int(self._lib.spg_launch_count(self._h))

    def stage_kernels(self):
        """Names of the kernel variants the last launches used: (nms_peaks, limb_score, limb_match, assemble)."""
        return tuple((self._lib.spg_stage_kernel(self._h, i) or b"").decode() for i in range(4))

    def postnet_kernel(self) -> str:
        """Name of the kernel the last ``postnet`` call launched."""
        return (self._lib.spg_stage_kernel(self._h, 4) or b"").decode()

    # -- wire records (include/spgroup.h; wire.py is the host-side view) -------------------------------
    def wire_record_bytes(self, rows: Optional[int] = None) -> int:
        """Bytes of one image's record with ``rows`` person rows (default: ``max_person_rows``)."""
        return 8 + int(self.capR if rows is None else rows) * (2 * self.J + 2) * 8

    def set_wire_output(self, dev_ptr: Optional[int], first_record: int = 0, rows: Optional[int] = None) -> None:
        """Make the assemble stage also write one wire record per image to ``dev_ptr`` (a raw device address: local
        memory or a peer GPU's buffer opened with ``wire_open``); ``None`` switches it off."""
        rc = self._lib.spg_set_wire_output(self._h, C.c_void_p(dev_ptr or 0), C.c_int64(first_record),
                                           C.c_int32(self.capR if rows is None else rows))
        self._check(rc, "spg_set_wire_output")

    def arm_wire_signal(self, word_ptr: Optional[int], value: int = 0) -> None:
        """The next single-launch assemble stage release-stores ``value`` into the 64-bit word at ``word_ptr`` (local or
        peer memory) when its last CTA is done: the "records landed" signal without a separate kernel.  One shot."""
        rc = self._lib.spg_arm_wire_signal(self._h, C.c_void_p(word_ptr or 0), C.c_uint64(value))
        self._check(rc, "spg_arm_wire_signal")

    # -- helpers ---------------------------------------------------------------------------------
    def _stream_ptr(self, stream) -> C.c_void_p:
        if stream is None:
            import torch
            stream = torch.cuda.current_stream(self.device)  # the handle's device, not torch's current one
        return C.c_void_p(int(getattr(stream, "cuda_stream", stream)))

    def _check_maps(self, t, name: str, channels: int, dtypes) -> None:
        """Shape / dtype / channel checks shared by the whole-path and the stage entry points."""
        import torch
        self._dev_tensor(t, name)
        if t.device.index != self.device:
            raise GroupingError(f"{name} lives on cuda:{t.device.index}, the handle on cuda:{self.device}")
        if t.dtype not in dtypes:
            raise GroupingError(f"{name} must be " + " or ".join(str(d).replace("torch.", "") for d in dtypes))
        if t.shape[1] < channels:
            raise GroupingError(f"{name} has {t.shape[1]} channels, the skeleton needs {channels}")
        if t.shape[0] > self.max_batch:
            raise GroupingError(f"{name} holds {t.shape[0]} images, the handle was created for {self.max_batch}")

    @staticmethod
    def _dev_tensor(t, name: str):
        if not t.is_cuda:
            raise GroupingError(f"{name} must be a CUDA tensor")
        if t.dim() != 4 or t.stride(3) != 1 or t.stride(2) != t.shape[3]:
            raise GroupingError(f"{name} must be [N,C,H,W] with contiguous rows (pixel stride 1, row stride W)")
        return t

    def _paf_dtype(self, paf, as_f64: bool = False) -> int:
        import torch
        if paf.dtype == torch.float32:
            return F32_AS_F64 if as_f64 else F32
        if paf.dtype == torch.float64:
            return F64
        raise GroupingError("body-part maps must be float32 or float64")

    # -- whole path --------------------------------------------------------------------------------
    def group_device(self, heat, paf, image_extent: float, params=None, stream=None, paf_as_f64: bool = False) -> None:
        """peaks -> connections -> people on device-resident maps; asynchronous on ``stream``.

        ``heat [N,>=K,H,W] float32`` (first K channels are used) and ``paf [N,>=L,H,W] float32|float64`` CUDA
        tensors; channel slices of the network's [N,50,h,w] output work without copies.  ``image_extent`` is the
        reference's ``oriImg.shape[0]`` (evaluate.py:510).
        """
        import torch
        self._check_maps(heat, "heat", self.K, (torch.float32,))  # find_peaks casts to float32, evaluate.py:173
        self._check_maps(paf, "paf", self.L, (torch.float32, torch.float64))
        N, _, H, W = heat.shape
        if paf.shape[0] != N or tuple(paf.shape[2:]) != (H, W):
            raise GroupingError("heat/paf shapes do not agree")
        p = params_struct(params)
        rc = self._lib.spg_group_batch(self._h, C.c_void_p(heat.data_ptr()), C.c_int64(heat.stride(0)),
                                       C.c_int64(heat.stride(1)), C.c_void_p(paf.data_ptr()),
                                       C.c_int32(self._paf_dtype(paf, paf_as_f64)), C.c_int64(paf.stride(0)), C.c_int64(paf.stride(1)),
                                       C.c_int32(N), C.c_int32(H), C.c_int32(W), C.c_double(float(image_extent)),
                                       C.byref(p), self._stream_ptr(stream))
        self._check(rc, "spg_group_batch")
        self._peaks_shape = (N, H, W)
        self._last_n = N

    def group_host(self, heat: np.ndarray, paf: np.ndarray, image_extent: float, params=None, out=None) -> dict:
        """Host maps in, person lists out (H2D / kernels / D2H pipelined inside the library).  Synchronous.

        ``heat [N,K,H,W] float32`` and ``paf [N,L,H,W] float32|float64`` C-contiguous numpy arrays (pinned memory
        gives full copy/compute overlap).  ``out`` may carry preallocated result arrays to reuse.
        """
        if heat.dtype != np.float32 or not heat.flags.c_contiguous or heat.ndim != 4 or heat.shape[1] != self.K:
            raise GroupingError("heat must be a C-contiguous float32 [N,K,H,W] array")
        if paf.dtype not in (np.float32, np.float64) or not paf.flags.c_contiguous or paf.ndim != 4 or paf.shape[1] != self.L:
            raise GroupingError("paf must be a C-contiguous float32/float64 [N,L,H,W] array")
        N, _, H, W = heat.shape
        if paf.shape[0] != N or paf.shape[2:] != (H, W):
            raise GroupingError("heat/paf shapes differ")
        if out is None:
            out = {}
        o_n = out.setdefault("n_persons", np.zeros((N,), np.int32))
        o_xy = out.setdefault("people_xy", np.zeros((N, self.capR, self.J, 2), np.float64))
        o_sc = out.setdefault("people_score", np.zeros((N, self.capR), np.float64))
        o_st = out.setdefault("status", np.zeros((N,), np.uint32))
        p = params_struct(params)
        rc = self._lib.spg_group_host(self._h, _vp(heat), _vp(paf), C.c_int32(F64 if paf.dtype == np.float64 else F32),
                                      C.c_int32(N), C.c_int32(H), C.c_int32(W), C.c_double(float(image_extent)),
                                      C.byref(p), _vp(o_n), _vp(o_xy), _vp(o_sc), _vp(o_st))
        self._check(rc, "spg_group_host")
        self._last_n = N
        return out

    # -- pre-network stage ----------------------------------------------------------------------------
    def prenet(self, image, scale: float, angles=(0.0,), *, max_downsample: int = 64, pad_value: int = 128, out=None,
               stream=None):
        """What the network sees for every angle of one scale of ``predict()``'s loop (evaluate.py:98-116), built on
        the device: bicubic resize of the uint8 image, padding to a multiple of ``max_downsample`` with ``pad_value``,
        ``/ 255``, the rotation by each angle, and the mirrored copy.

        ``image``: CUDA uint8 ``[H, W, 3]`` (BGR, as cv2 reads it) on the handle's device with contiguous pixels; any
        row stride, so a crop of a larger frame works.  Returns ``(pairs [n_angles, 2, Hp, Wp, 3] float32,
        (crop_h, crop_w))``: ``pairs[k]`` is the network input of ``angles[k]`` and ``(crop_h, crop_w)`` the
        ``imageToTest`` size ``postnet`` crops to.  The values equal the reference's with cv2's IPP off, bit for bit;
        with IPP on (cv2's default) the uint8 resize differs by at most 1 in a few percent of the values."""
        import torch
        if not torch.is_tensor(image) or not image.is_cuda or image.device.index != self.device:
            raise GroupingError(f"image must be a CUDA tensor on cuda:{self.device}")
        if image.dtype != torch.uint8 or image.dim() != 3 or image.shape[2] != 3:
            raise GroupingError("image must be a uint8 [H, W, 3] tensor")
        if image.stride(2) != 1 or image.stride(1) != 3:
            raise GroupingError("image pixels must be contiguous (pixel stride 3, channel stride 1)")
        H, W = int(image.shape[0]), int(image.shape[1])
        (ch, cw), (hp, wp) = prenet_size(H, W, scale, max_downsample)
        ang = np.ascontiguousarray(np.asarray(angles, np.float64).reshape(-1))
        if out is None:
            out = torch.empty((len(ang), 2, hp, wp, 3), dtype=torch.float32, device=torch.device("cuda", self.device))
        elif out.dtype != torch.float32 or tuple(out.shape) != (len(ang), 2, hp, wp, 3) or not out.is_contiguous() \
                or not out.is_cuda or out.device.index != self.device:
            raise GroupingError(f"out must be a contiguous float32 [{len(ang)}, 2, {hp}, {wp}, 3] tensor on cuda:{self.device}")
        rc = self._lib.spg_prenet(self._h, C.c_void_p(image.data_ptr()), C.c_int64(image.stride(0)), C.c_int32(H),
                                  C.c_int32(W), C.c_int32(3), C.c_double(float(scale)),
                                  ang.ctypes.data_as(C.POINTER(C.c_double)), C.c_int32(len(ang)), C.c_int32(int(max_downsample)),
                                  C.c_int32(int(pad_value)), C.c_void_p(out.data_ptr()), C.c_int64(2 * hp * wp * 3),
                                  self._stream_ptr(stream))
        self._check(rc, "spg_prenet")
        return out, (ch, cw)

    # -- post-network stage ---------------------------------------------------------------------------
    def postnet(self, net_outs, crops, out_hw, *, stride: int = 4, paf_dtype=None, heat_out=None, paf_out=None,
                paf_chan0: int = 0, heat_chan0: Optional[int] = None, flip_paf_ord=None, flip_heat_ord=None,
                nan_scrub: bool = False, stream=None, angles=None):
        """The scale loop of ``predict()`` after the forward pass (evaluate.py:126-161) on the device.

        ``net_outs``: one CUDA tensor ``[N, 2, C, h, w]`` (float32 / float16; image, mirrored image) per scale;
        ``crops``: per scale ``(crop_h, crop_w)`` = ``imageToTest.shape[:2]``; ``out_hw``: the image size.
        ``angles``: with rotation search, one angle in degrees per entry -- the entries are then the items of
        ``product(multiplier, rotation_search)`` in that order, each network output computed on the input warped with
        ``cv2.getRotationMatrix2D((Hp / 2, Wp / 2), angle, 1)`` (evaluate.py:108-111).  All zeros is the same as ``None``.
        Returns ``(heat [N,K,H,W] float32, paf [N,L,H,W])`` -- ``paf`` float32 for a single scale (pass
        ``paf_as_f64=True`` to the grouping calls: the reference's float64 values are exactly these), float64 otherwise.
        """
        import torch
        from .skeleton import FLIP_HEAT_ORD, FLIP_PAF_ORD, NUM_LIMBS
        if len(net_outs) != len(crops) or not net_outs:
            raise GroupingError("one crop size per scale expected")
        H, W = (int(v) for v in out_hw)
        N = int(net_outs[0].shape[0])
        dev = torch.device("cuda", self.device)
        single = len(net_outs) == 1
        if paf_dtype is None:
            paf_dtype = torch.float32 if single else torch.float64
        if paf_dtype == torch.float32 and not single:
            raise GroupingError("float32 body-part planes hold the reference's float64 values only for a single scale")
        heat_chan0 = self.L if heat_chan0 is None else heat_chan0
        fp = np.ascontiguousarray(np.asarray(FLIP_PAF_ORD if flip_paf_ord is None else flip_paf_ord, np.int32)[:self.L])
        fh = np.ascontiguousarray(np.asarray(FLIP_HEAT_ORD if flip_heat_ord is None else flip_heat_ord, np.int32)[:self.K])
        if flip_paf_ord is None and self.L != NUM_LIMBS:
            raise GroupingError("flip_paf_ord is needed for a non-canonical skeleton")
        scales = (_PostnetScale * len(net_outs))()
        for t, (o, (ch, cw)) in enumerate(zip(net_outs, crops)):
            if not o.is_cuda or o.device.index != self.device or o.dim() != 5 or o.shape[0] != N or o.shape[1] != 2:
                raise GroupingError("network output must be a [N,2,C,h,w] CUDA tensor on the handle's device")
            if o.stride(4) != 1 or o.stride(3) != o.shape[4]:
                raise GroupingError("network output rows must be contiguous")
            if o.dtype not in (torch.float32, torch.float16):
                raise GroupingError("network output must be float32 or float16")
            if o.shape[2] < max(heat_chan0 + self.K, paf_chan0 + self.L):
                raise GroupingError("network output has too few channels")
            scales[t] = _PostnetScale(o.data_ptr(), F32 if o.dtype == torch.float32 else F16, o.stride(0), o.stride(1),
                                      o.stride(2), o.shape[3], o.shape[4], int(ch), int(cw))
        if heat_out is None:
            heat_out = torch.empty((N, self.K, H, W), dtype=torch.float32, device=dev)
        if paf_out is None:
            paf_out = torch.empty((N, self.L, H, W), dtype=paf_dtype, device=dev)
        if not (heat_out.is_contiguous() and paf_out.is_contiguous()) or paf_out.dtype != paf_dtype:
            raise GroupingError("heat_out / paf_out must be contiguous tensors of the requested dtype")
        desc = _PostnetDesc(len(net_outs), scales, int(stride), int(paf_chan0), int(heat_chan0),
                            fp.ctypes.data_as(C.POINTER(C.c_int32)), fh.ctypes.data_as(C.POINTER(C.c_int32)), int(bool(nan_scrub)))
        out_args = (C.c_int32(N), C.c_int32(H), C.c_int32(W), C.c_void_p(heat_out.data_ptr()), C.c_void_p(paf_out.data_ptr()),
                    C.c_int32(F32 if paf_dtype == torch.float32 else F64), self._stream_ptr(stream))
        if angles is None:
            rc = self._lib.spg_postnet(self._h, C.byref(desc), *out_args)
            self._check(rc, "spg_postnet")
        else:
            ang = np.ascontiguousarray(np.asarray(angles, np.float64).reshape(-1))
            if ang.shape[0] != len(net_outs):
                raise GroupingError("one angle per network output expected")
            rc = self._lib.spg_postnet_rotated(self._h, C.byref(desc), ang.ctypes.data_as(C.POINTER(C.c_double)), *out_args)
            self._check(rc, "spg_postnet_rotated")
        return heat_out, paf_out

    # -- stages -------------------------------------------------------------------------------------
    def nms_peaks(self, heat, params=None, stream=None) -> None:
        """find_peaks (evaluate.py:169-203) on ``heat [N,>=K,H,W]`` float32 CUDA."""
        import torch
        self._check_maps(heat, "heat", self.K, (torch.float32,))
        N, _, H, W = heat.shape
        self._peaks_shape = (N, H, W)
        p = params_struct(params)
        rc = self._lib.spg_nms_peaks(self._h, C.c_void_p(heat.data_ptr()), C.c_int64(heat.stride(0)),
                                     C.c_int64(heat.stride(1)), C.c_int32(N), C.c_int32(H), C.c_int32(W), C.byref(p),
                                     self._stream_ptr(stream))
        self._check(rc, "spg_nms_peaks")
        self._last_n = N

    def limb_score(self, paf, image_extent: float, params=None, stream=None, paf_as_f64: bool = False) -> None:
        """Scoring half of find_connections (evaluate.py:211-255) for peaks already on the device."""
        import torch
        self._check_maps(paf, "paf", self.L, (torch.float32, torch.float64))
        N, _, H, W = paf.shape
        ps = getattr(self, "_peaks_shape", None)  # peaks from spg_nms_peaks: the maps must agree (uploaded peaks carry no shape)
        if ps is not None and (ps[0] < N or ps[1:] != (H, W)):
            raise GroupingError(f"paf is {N}x{H}x{W} but the peaks on the device come from {ps[0]}x{ps[1]}x{ps[2]} heat maps")
        p = params_struct(params)
        rc = self._lib.spg_limb_score(self._h, C.c_void_p(paf.data_ptr()), C.c_int32(self._paf_dtype(paf, paf_as_f64)),
                                      C.c_int64(paf.stride(0)), C.c_int64(paf.stride(1)), C.c_int32(N), C.c_int32(H),
                                      C.c_int32(W), C.c_double(float(image_extent)), C.byref(p), self._stream_ptr(stream))
        self._check(rc, "spg_limb_score")
        self._last_n = N

    def limb_match(self, n_images: int, params=None, stream=None) -> None:
        """Matching half of find_connections (evaluate.py:259-274)."""
        p = params_struct(params)
        self._check(self._lib.spg_limb_match(self._h, C.c_int32(n_images), C.byref(p), self._stream_ptr(stream)),
                    "spg_limb_match")

    def assemble(self, n_images: int, params=None, stream=None) -> None:
        """find_people + process() tail (evaluate.py:279-498, 523-543)."""
        p = params_struct(params)
        self._check(self._lib.spg_assemble(self._h, C.c_int32(n_images), C.byref(p), self._stream_ptr(stream)),
                    "spg_assemble")

    def match_assemble(self, n_images: int, params=None, stream=None) -> None:
        """limb_match + assemble fused in one kernel (what the whole-path calls run)."""
        p = params_struct(params)
        self._check(self._lib.spg_match_assemble(self._h, C.c_int32(n_images), C.byref(p), self._stream_ptr(stream)),
                    "spg_match_assemble")

    # -- state transfer ---------------------------------------------------------------------------------
    def upload_peaks(self, image_index: int, part_count, x, y, score, stream=None) -> None:
        self._peaks_shape = None
        pc = np.ascontiguousarray(part_count, np.int32)
        x = np.ascontiguousarray(x, np.float64)
        y = np.ascontiguousarray(y, np.float64)
        s = np.ascontiguousarray(score, np.float32)
        self._check(self._lib.spg_upload_peaks(self._h, C.c_int32(image_index), _vp(pc), _vp(x), _vp(y), _vp(s),
                                               self._stream_ptr(stream)), "spg_upload_peaks")

    def upload_connections(self, image_index: int, conn_count, ij, score, norm, stream=None) -> None:
        cc = np.ascontiguousarray(conn_count, np.int32)
        ij = np.ascontiguousarray(ij, np.int32).reshape(-1, 2)
        sc = np.ascontiguousarray(score, np.float64)
        nm = np.ascontiguousarray(norm, np.float64)
        self._check(self._lib.spg_upload_connections(self._h, C.c_int32(image_index), _vp(cc), _vp(ij), _vp(sc), _vp(nm),
                                                     self._stream_ptr(stream)), "spg_upload_connections")

    def fetch(self, n_images: Optional[int] = None, stream=None) -> GroupResult:
        """Synchronise and copy every result of the last call to the host."""
        N = int(self._last_n if n_images is None else n_images)
        K, L, J, cP, cR = self.K, self.L, self.J, self.capP, self.capR
        st = self._stream_ptr(stream)
        r = GroupResult(
            K=K, L=L, limbs=self.limbs, peak_count=np.zeros((N, K), np.int32), peak_x=np.zeros((N, K, cP)),
            peak_y=np.zeros((N, K, cP)), peak_score=np.zeros((N, K, cP), np.float32),
            peak_anchor=np.zeros((N, K, cP), np.uint32), conn_count=np.zeros((N, L), np.int32),
            cand_count=np.zeros((N, L), np.int32), conn_ij=np.zeros((N, L, cP), np.uint32),
            conn_score=np.zeros((N, L, cP)), conn_norm=np.zeros((N, L, cP)), n_persons=np.zeros((N,), np.int32),
            subset=np.zeros((N, cR, K + 2, 2)), people_xy=np.zeros((N, cR, J, 2)), people_score=np.zeros((N, cR)),
            status=np.zeros((N,), np.uint32))
        self._check(self._lib.spg_download_peaks(self._h, C.c_int32(N), _vp(r.peak_count), _vp(r.peak_x), _vp(r.peak_y),
                                                 _vp(r.peak_score), _vp(r.peak_anchor), st), "spg_download_peaks")
        self._check(self._lib.spg_download_connections(self._h, C.c_int32(N), _vp(r.conn_count), _vp(r.cand_count),
                                                       _vp(r.conn_ij), _vp(r.conn_score), _vp(r.conn_norm), st),
                    "spg_download_connections")
        self._check(self._lib.spg_download_people(self._h, C.c_int32(N), _vp(r.n_persons), _vp(r.subset), _vp(r.people_xy),
                                                  _vp(r.people_score), st), "spg_download_people")
        self._check(self._lib.spg_download_status(self._h, C.c_int32(N), _vp(r.status), st), "spg_download_status")
        return r

    def device_tensors(self) -> dict:
        """Zero-copy torch views of the device-resident person lists (what the NCCL gather sends)."""
        import torch
        v = _DeviceView()
        self._check(self._lib.spg_get_device_view(self._h, C.byref(v)), "spg_get_device_view")
        dev = torch.device("cuda", self.device)
        N, cR, J, K = self.max_batch, self.capR, self.J, self.K

        def view(ptr, shape, typestr):
            return torch.as_tensor(_CudaView(ptr, shape, typestr), device=dev)

        return {"n_persons": view(v.n_persons, (N,), "<i4"),
                "people_xy": view(v.people_xy, (N, cR, J, 2), "<f8"),
                "people_score": view(v.people_score, (N, cR), "<f8"),
                "subset": view(v.subset, (N, cR, K + 2, 2), "<f8"),
                "status": view(v.status, (N,), "<i4"),
                "cand_count": view(v.cand_count, (N, self.L), "<i4"),
                "surv_count": view(v.surv_count, (N, self.L), "<i4")}
