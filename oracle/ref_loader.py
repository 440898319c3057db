"""Load the reference's grouping functions UNMODIFIED, for pinning the oracle.

TEST INFRASTRUCTURE ONLY.  This module works only where ``/root/reference``
exists (the build container); it never travels to the GPU box.  It is used by
``tests/golden/make_golden.py`` and ``tests/golden/make_reference_outputs.py``
(fixture generation).

``import evaluate`` cannot work here (pycocotools / matplotlib / configobj /
apex are missing and the module body parses ``sys.argv`` and pins
``CUDA_VISIBLE_DEVICES``), so the three hot-path functions are lifted out of
the source with ``ast`` and exec'd verbatim:

    find_peaks        /root/reference/evaluate.py:169-203
    find_connections  /root/reference/evaluate.py:206-276
    find_people       /root/reference/evaluate.py:279-498

with the globals they resolve at call time: ``np``, ``math``, ``torch``,
``util`` (= the reference's own ``utils/util.py``, imported unmodified, which
provides ``keypoint_heatmap_nms`` :177-183 and ``refine_centroid`` :186-211) and
``limbSeq`` (= ``config.limbs_conn``, /root/reference/config/config.py:94).
On a CPU-only host ``Tensor.cuda`` is patched to the identity for the duration
of the call (evaluate.py:176 calls ``.cuda()`` unconditionally).
"""
from __future__ import annotations

import ast
import contextlib
import importlib.util
import math
import os
import sys

REFERENCE_ROOT = os.environ.get("SPG_REFERENCE_ROOT", "/root/reference")
_WANTED = ("find_peaks", "find_connections", "find_people")


def reference_available() -> bool:
    return os.path.isfile(os.path.join(REFERENCE_ROOT, "evaluate.py"))


def _load_module(name: str, path: str):
    spec = importlib.util.spec_from_file_location(name, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


@contextlib.contextmanager
def _cuda_identity_if_needed():
    import torch

    if torch.cuda.is_available():
        yield
        return
    orig = torch.Tensor.cuda
    torch.Tensor.cuda = lambda self, *a, **k: self
    try:
        yield
    finally:
        torch.Tensor.cuda = orig


class Reference:
    """The reference's three functions bound to a limb table."""

    def __init__(self, limbs=None):
        import numpy as np
        import torch

        if not reference_available():
            raise FileNotFoundError(f"reference not present at {REFERENCE_ROOT}")
        util = _load_module("_spg_ref_util", os.path.join(REFERENCE_ROOT, "utils", "util.py"))
        if limbs is None:
            # config/config.py imports only numpy; GetConfig('Canonical') is the
            # skeleton evaluate.py uses (evaluate.py:51-54).
            import io
            with contextlib.redirect_stdout(io.StringIO()):  # GetConfig prints the whole layer table
                cfg = _load_module("_spg_ref_config", os.path.join(REFERENCE_ROOT, "config", "config.py"))
                limbs = cfg.GetConfig("Canonical").limbs_conn
        src = open(os.path.join(REFERENCE_ROOT, "evaluate.py"), encoding="utf-8").read()
        tree = ast.parse(src)
        body = [n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name in _WANTED]
        assert len(body) == len(_WANTED), "reference layout changed"
        ns = {"np": np, "math": math, "torch": torch, "util": util,
              "limbSeq": [tuple(int(v) for v in p) for p in limbs]}
        code = compile(ast.Module(body=body, type_ignores=[]), os.path.join(REFERENCE_ROOT, "evaluate.py"), "exec")
        exec(code, ns)
        self._ns = ns
        self.util = util
        self.limbs = ns["limbSeq"]

    def find_peaks(self, heatmap_avg, params):
        with _cuda_identity_if_needed():
            return self._ns["find_peaks"](heatmap_avg, params)

    def find_connections(self, all_peaks, paf_avg, image_width, params):
        return self._ns["find_connections"](all_peaks, paf_avg, image_width, params)

    def find_people(self, connection_all, special_k, all_peaks, params):
        import warnings

        with warnings.catch_warnings():
            warnings.simplefilter("ignore")  # int(np.where(...)[0]) deprecation, evaluate.py:437-438
            return self._ns["find_people"](connection_all, special_k, all_peaks, params)

    def group(self, heat_hwc, paf_hwc, image_extent, params):
        """peaks -> connections -> people, the window evaluate.py:509-511 times."""
        peaks = self.find_peaks(heat_hwc, params)
        conns, special = self.find_connections(peaks, paf_hwc, image_extent, params)
        subset, candidate = self.find_people(conns, special, peaks, params)
        return peaks, conns, special, subset, candidate


def reference_function(name: str, extra_globals: dict = None):
    """Any top-level function of /root/reference/evaluate.py, lifted verbatim (e.g. ``format_results`` :563-582)."""
    import json

    import numpy as np

    src = open(os.path.join(REFERENCE_ROOT, "evaluate.py"), encoding="utf-8").read()
    node = next(n for n in ast.parse(src).body if isinstance(n, ast.FunctionDef) and n.name == name)
    ns = {"np": np, "math": math, "json": json, "os": os}
    ns.update(extra_globals or {})
    exec(compile(ast.Module(body=[node], type_ignores=[]), os.path.join(REFERENCE_ROOT, "evaluate.py"), "exec"), ns)
    return ns[name]


class DemoReference:
    """The grouping code INLINED in ``demo_image.py``'s ``process()`` (``/root/reference/demo_image.py:185-536``), lifted
    statement for statement: everything from ``all_peaks = []`` (:185) to the final prune
    ``subset = np.delete(subset, deleteIdx, axis=0)`` (:536), minus the matplotlib call ``show_color_vector(...)`` (:191).
    It differs from evaluate.py in three decisions (SURVEY.md 3.2: ``>`` at :288, the length check at :414-415,
    ``count < 4`` at :533); this class is what pins ``GroupParams.demo()`` to it."""

    def __init__(self, limbs=None):
        import numpy as np
        import torch

        base = Reference(limbs)
        path = os.path.join(REFERENCE_ROOT, "demo_image.py")
        tree = ast.parse(open(path, encoding="utf-8").read())
        proc = next(n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name == "process")
        def is_assign_to(n, name):
            return isinstance(n, ast.Assign) and len(n.targets) == 1 and isinstance(n.targets[0], ast.Name) and n.targets[0].id == name
        start = next(i for i, n in enumerate(proc.body) if is_assign_to(n, "all_peaks"))
        ends = [i for i, n in enumerate(proc.body) if is_assign_to(n, "subset") and "np.delete" in ast.unparse(n)]
        assert ends and ends[-1] > start, "demo_image.py layout changed"
        body = [n for n in proc.body[start:ends[-1] + 1]
                if not (isinstance(n, ast.Expr) and isinstance(n.value, ast.Call) and "show_color_vector" in ast.unparse(n.value.func))]
        ret = ast.parse("return all_peaks, connection_all, special_k, subset, candidate").body[0]
        fn = ast.FunctionDef(name="demo_group", args=ast.arguments(
            posonlyargs=[], args=[ast.arg(arg=a) for a in ("heatmap_avg", "paf_avg", "oriImg", "params")], kwonlyargs=[],
            kw_defaults=[], defaults=[]), body=body + [ret], decorator_list=[], type_params=[])
        mod = ast.fix_missing_locations(ast.Module(body=[fn], type_ignores=[]))
        ns = {"np": np, "math": math, "torch": torch, "util": base.util, "limbSeq": base.limbs}
        exec(compile(mod, path, "exec"), ns)
        self._fn, self.limbs = ns["demo_group"], base.limbs

    def group(self, heat_hwc, paf_hwc, image_extent, params):
        import warnings

        import numpy as np

        class _Img:  # only oriImg.shape[0] is read (demo_image.py:282)
            shape = (int(image_extent), 0, 3)

        with _cuda_identity_if_needed(), warnings.catch_warnings():
            warnings.simplefilter("ignore")
            return self._fn(np.asarray(heat_hwc), np.asarray(paf_hwc), _Img, params)


if __name__ == "__main__":
    print("reference available:", reference_available())
    if reference_available():
        r = Reference()
        print("limbs:", r.limbs)
