"""CPU: the inference IMHN (improved_body_parts_b200/imhn.py, SURVEY.md §8 f-3) against the reference's own module.

The reference's ``NetworkEval`` (models/posenet.py:175-193) state dict names and shapes, and its outputs for fixed
deterministic weights, are stored in tests/golden/reference/imhn.npz (tests/golden/make_reference_outputs.py).  The
same weights are loaded into ours with ``strict=True`` (same parameter names and shapes: reference checkpoints load,
evaluate.py:629-630) and the outputs are compared: all ``nstack x 5`` maps of ``forward_all`` and the single tensor
``forward`` returns (= ``output_tuple[-1][0]``, evaluate.py:126).  The self-consistency checks (BatchNorm folding,
pruned vs full forward) need no stored data."""
import math
import os

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _small(nstack=2):
    from improved_body_parts_b200.imhn import IMHN
    torch.manual_seed(0)
    m = IMHN(nstack=nstack)
    with torch.no_grad():  # non-trivial BatchNorm statistics, weights large enough for visible outputs
        for mod in m.modules():
            if isinstance(mod, torch.nn.BatchNorm2d):
                mod.running_mean.uniform_(-0.2, 0.2)
                mod.running_var.uniform_(0.5, 1.5)
                mod.weight.uniform_(0.5, 1.5)
                mod.bias.uniform_(-0.1, 0.1)
            elif isinstance(mod, torch.nn.Conv2d):
                mod.weight.normal_(0, (2.0 / (mod.weight[0].numel())) ** 0.5)
    return m.eval()


def test_pruned_forward_is_the_last_stacks_finest_map_and_bn_folding_is_exact_enough():
    m = _small(2)
    x = torch.rand(2, 64, 64, 3)
    with torch.no_grad():
        full = m.forward_all(x)
        one = m(x)
        assert len(full) == 2 and len(full[0]) == 5 and [tuple(p.shape[1:]) for p in full[-1]] == \
            [(50, 16, 16), (50, 8, 8), (50, 4, 4), (50, 2, 2), (50, 1, 1)]
        assert torch.equal(one, full[-1][0])
        n_bn = sum(isinstance(mod, torch.nn.BatchNorm2d) for mod in m.modules())
        m.fold_batchnorm_()
        assert n_bn > 100 and not any(isinstance(mod, torch.nn.BatchNorm2d) for mod in m.modules())
        folded = m(x)
    assert one.abs().max() > 1e-3
    assert torch.allclose(folded, one, rtol=1e-4, atol=1e-5 * float(one.abs().max()))


def seeded_state(entries, seed=1):
    """Deterministic values for a state dict given as ``(name, shape)`` pairs: weight matrices and kernels uniform in
    +-1/sqrt(fan_in) (PyTorch's default bound), BatchNorm scales and statistics away from the identity, small biases."""
    g = torch.Generator().manual_seed(seed)
    out = {}
    for name, shape in entries:
        leaf = name.rsplit(".", 1)[-1]
        if leaf == "num_batches_tracked":
            out[name] = torch.zeros(shape, dtype=torch.long)
            continue
        if leaf == "running_mean":
            lo, hi = -0.2, 0.2
        elif leaf == "running_var" or (leaf == "weight" and len(shape) == 1):
            lo, hi = 0.5, 1.5
        elif len(shape) > 1:
            hi = math.prod(shape[1:]) ** -0.5
            lo = -hi
        else:
            lo, hi = -0.1, 0.1
        out[name] = torch.rand(shape, generator=g) * (hi - lo) + lo
    return out


def imhn_input():
    return torch.rand(2, 64, 64, 3, generator=torch.Generator().manual_seed(2))


def map_sample(t, n=256):
    """A fixed, evenly strided sample of at most about ``n`` values of a map, as float32."""
    flat = t.detach().reshape(-1)
    return flat[::max(1, flat.numel() // n)].numpy().astype(np.float32)


def test_reference_state_dict_loads_strictly_and_outputs_agree():
    """The reference's ``NetworkEval`` state dict (names and shapes) loads with ``strict=True`` and, for the same
    deterministic weights, every map of ``forward_all`` and the tensor ``forward`` returns agree with the reference's
    outputs (tests/golden/reference/imhn.npz: a fixed sample of each map and the map's largest magnitude)."""
    import json

    from improved_body_parts_b200.imhn import IMHN
    with np.load(os.path.join(ROOT, "tests", "golden", "reference", "imhn.npz"), allow_pickle=False) as z:
        ref = {k: z[k] for k in z.files}
    entries = json.loads(str(ref["state"]))
    ours = IMHN(nstack=4)
    missing = ours.load_state_dict(seeded_state(entries), strict=True)  # same names, same shapes
    assert not missing.missing_keys and not missing.unexpected_keys
    assert sum(p.numel() for p in ours.parameters()) == sum(math.prod(s) for k, s in entries if "running" not in k
                                                            and "num_batches" not in k) > 100e6
    x = imhn_input()
    with torch.no_grad():
        got = ours.forward_all(x)
        worst = 0.0
        for i in range(4):
            for j in range(5):
                scale = float(ref[f"s{i}_{j}_absmax"])
                assert scale > 1e-3
                worst = max(worst, float(np.abs(map_sample(got[i][j]) - ref[f"s{i}_{j}_sample"]).max()) / scale)
        # same float32 network; only the association of a few sums differs (x + (a + b) vs (x + a) + b, mean vs avg-pool)
        assert worst < 2e-5, worst
        assert float(np.abs(map_sample(ours(x)) - ref["s3_0_sample"]).max()) / float(ref["s3_0_absmax"]) < 2e-5
