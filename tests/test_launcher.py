"""CPU: the launcher that runs ``evaluate.py`` unchanged (tools/run_evaluate_b200.py) against the REAL module, where a
reference checkout is present -- import with stubbed third-party modules, CUDA_VISIBLE_DEVICES restored after the
module pins it (evaluate.py:28), the three call-site names rebound (:509-511), ``limbSeq`` picked up (:54), ``params``
read from the reference's own utils/config, and ``format_results`` replaceable -- and the INI reader against what it
made of that utils/config."""
import importlib.util
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get("SPG_REFERENCE_ROOT", "/root/reference")


_CHILD = r'''
import json, os, sys
sys.path.insert(0, {root!r})
os.environ["CUDA_VISIBLE_DEVICES"] = "3,5"
spec_path = os.path.join({root!r}, "tools", "run_evaluate_b200.py")
import importlib.util
spec = importlib.util.spec_from_file_location("run_evaluate_b200", spec_path)
L = importlib.util.module_from_spec(spec); spec.loader.exec_module(L)
ev = L.prepare({ref!r}, replace_format_results=True)
from improved_body_parts_b200 import dropin, skeleton, wire
import inspect
out = dict(
    file=ev.__file__, visible=os.environ.get("CUDA_VISIBLE_DEVICES"),
    rebound=[ev.find_peaks is dropin.find_peaks, ev.find_connections is dropin.find_connections, ev.find_people is dropin.find_people],
    limbs_equal=[tuple(int(v) for v in p) for p in ev.limbSeq] == list(dropin._limbs) == list(skeleton.LIMBS),
    params={{k: ev.params[k] for k in ("thre1", "thre2", "connect_ration", "mid_num", "len_rate", "connection_tole", "offset_radius", "remove_recon", "scale_search", "rotation_search")}},
    model={{k: ev.model_params[k] for k in ("boxsize", "stride", "max_downsample", "padValue")}},
    process_resolves_by_name="find_peaks(heatmap, params)" in inspect.getsource(ev.process),
    fmt=ev.format_results is wire.format_results, stubbed=ev.__spg_stubbed__,
    has_predict=callable(ev.predict) and callable(ev.validation), dt_gt=ev.dt_gt_mapping == skeleton.DT_GT_MAPPING,
    flip=[list(ev.flip_heat_ord) == list(skeleton.FLIP_HEAT_ORD), list(ev.flip_paf_ord) == list(skeleton.FLIP_PAF_ORD)])
print("RESULT " + json.dumps(out))
'''


@pytest.mark.skipif(not os.path.isfile(os.path.join(REF, "evaluate.py")), reason="needs the reference checkout's evaluate.py")
def test_launcher_imports_the_real_evaluate_and_rebinds_it():
    import json
    r = subprocess.run([sys.executable, "-c", _CHILD.format(root=ROOT, ref=REF)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-3000:]
    out = json.loads(next(l for l in r.stdout.splitlines() if l.startswith("RESULT "))[7:])
    assert os.path.samefile(out["file"], os.path.join(REF, "evaluate.py"))
    assert out["visible"] == "3,5", "CUDA_VISIBLE_DEVICES must be restored after evaluate.py:28 pins it"
    assert out["rebound"] == [True, True, True] and out["limbs_equal"] and out["process_resolves_by_name"]
    assert out["params"] == {"thre1": 0.1, "thre2": 0.1, "connect_ration": 0.8, "mid_num": 20, "len_rate": 16.0,
                             "connection_tole": 0.7, "offset_radius": 2, "remove_recon": 0, "scale_search": [1.0],
                             "rotation_search": [0.0]}
    assert out["model"] == {"boxsize": 640, "stride": 4, "max_downsample": 64, "padValue": 128}
    assert out["fmt"] and out["has_predict"] and out["dt_gt"] and out["flip"] == [True, True]


def test_ini_reader_agrees_with_the_reference_config_file():
    import json
    sys.path.insert(0, ROOT)
    from improved_body_parts_b200 import skeleton
    # what the reader made of the reference's own utils/config (tests/golden/make_reference_outputs.py)
    stored = json.load(open(os.path.join(ROOT, "tests", "golden", "reference", "utils_config.json")))
    param, model = stored["param"], stored["model"]
    fixture = skeleton.read_reference_ini(os.path.join(ROOT, "tests", "golden", "reference_utils_config.ini"))
    assert param == fixture[0]
    assert {k: model[k] for k in ("boxsize", "padValue", "stride", "max_downsample")} == \
           {k: fixture[1][k] for k in ("boxsize", "padValue", "stride", "max_downsample")}
    d = skeleton.default_params()
    assert all(param[k] == d[k] for k in d)
