#!/usr/bin/env python
"""Small run for compute-sanitizer (memcheck / synccheck): dirty images through every kernel of the library --
pre-network stage (strided image, rotated and not), post-network stage (identity, single- and multi-scale, non-identity
second resize, rotation search), persistent, banded and per-item nms / limb_score
(f32, f32-as-f64, f64), fused match+assemble with wire records and the armed signal, the stand-alone match / assemble."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from improved_body_parts_b200 import synth, skeleton
from improved_body_parts_b200.grouping import Grouper

dev = torch.device("cuda:0")
prm = skeleton.default_params()
heat, paf = synth.make_batch(99, 6, 128, 128, 12, drop_prob=0.1, edge=True, spikes=10, colocate=2)
g = Grouper(max_batch=6)
hd, pd = torch.from_numpy(heat).to(dev), torch.from_numpy(paf).to(dev)
wire_buf = torch.zeros((6, g.wire_record_bytes()), dtype=torch.uint8, device=dev)
word = torch.zeros((1,), dtype=torch.int64, device=dev)
g.set_wire_output(wire_buf.data_ptr())
g.arm_wire_signal(word.data_ptr(), 7)
g.group_device(hd, pd, 128, prm)                                  # persistent kernels + fused match_assemble
k1 = g.stage_kernels()
g.group_device(hd, pd, 128, prm, paf_as_f64=True)                 # f32 storage, f64 arithmetic
g.group_device(hd, pd.double(), 128, prm)                         # f64 planes: per-item kernel
g.nms_peaks(hd, prm); g.limb_score(pd, 128, prm); g.limb_match(6, prm); g.assemble(6, prm)   # stand-alone kernels
r = g.fetch()
torch.cuda.synchronize()
assert int(word.item()) == 7
# post-network stage: single scale with a non-identity second resize, and three fused scales
outs = [torch.from_numpy(np.stack([synth.make_network_output(5 + i, int(24 * f), int(32 * f), 4, body_scale=f, base_hw=(24, 32))
                                   for i in range(2)])).to(dev) for f in (0.5, 1.0, 2.0)]
g2 = Grouper(max_batch=2, max_h=160, max_w=200)
h1, p1 = g2.postnet([outs[1]], [(90, 120)], (77, 101))
h3, p3 = g2.postnet(outs, [(48, 64), (96, 128), (192, 256)], (96, 128))
hi, pi = g2.postnet([outs[1]], [(96, 128)], (96, 128))             # crop == image: the identity kernel
hr, pr = g2.postnet([outs[1]], [(90, 120)], (77, 101), angles=[22.5])                  # rotation search: one rotated item
hr3, pr3 = g2.postnet(outs, [(48, 64), (96, 128), (192, 256)], (96, 128), angles=[5.0, 0.0, -90.0])  # rotated / angle-0 launches
g2.group_device(h3, p3, 96, prm)
# pre-network stage: a strided crop of a larger frame, angle 0 and rotated items, a copy (dsize == ssize) and a down-scale
frame = torch.from_numpy(np.random.default_rng(3).integers(0, 256, (130, 190, 3), dtype=np.uint8)).to(dev)
crop = frame[7:127, 13:173]
pairs, _ = g2.prenet(crop, 1.37, [0.0, -5.0, 22.5])
pairs1, _ = g2.prenet(crop, 1.0, [0.0], max_downsample=8, pad_value=0)
pairs2, _ = g2.prenet(crop, 0.21, [90.0])
# planes that do not fit shared memory three times: banded nms, body-part planes sampled through L2
heat3, paf3 = synth.make_batch(7, 2, 150, 260, 8, scale_range=(1.5, 3.0), edge=True)
g3 = Grouper(max_batch=2, max_h=150, max_w=260)
g3.group_device(torch.from_numpy(heat3).to(dev), torch.from_numpy(paf3).to(dev), 150, prm)
k3 = g3.stage_kernels()
torch.cuda.synchronize()
print("persons", r.n_persons.tolist(), "status", r.status.tolist(), "kernels", k1, g.stage_kernels(), "postnet", tuple(h1.shape), tuple(p3.shape), tuple(hi.shape), "large planes", k3, "prenet", tuple(pairs.shape))
