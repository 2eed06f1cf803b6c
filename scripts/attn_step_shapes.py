"""Per-call times of the native attention forward and backward at the four shapes of the GPS pre-training step, with the
key-padding masks of bench.py's synthetic batch (64 scenes) and the step's dropout (p = 0.1, none on the gated spatial
attention).  CUDA events over 50 calls after 5 warm-up calls.  Usage: python scripts/attn_step_shapes.py [out.json]"""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import bench
from sceneverse_b200 import native, ops, synthetic

B, H, E = bench.SCENES, 12, 768
dev = torch.device("cuda", 0)
d = synthetic.scene_batch(42, B=B, O=bench.OBJS, P=8, L=bench.TXT, Ls=bench.SCENE_TXT)
txt_pad = torch.from_numpy(d["txt_masks"] == 0).to(dev)
cap_pad = torch.from_numpy(d["scene_txt_masks"] == 0).to(dev)
obj_pad = torch.from_numpy(~d["obj_masks"]).to(dev)
g = torch.Generator(device=dev).manual_seed(0)


def rnd(*s, scale=1.0):
    return torch.randn(*s, device=dev, generator=g) * scale


def timed(fn, n=50):
    for _ in range(5):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / n * 1e3


locs = ops.calc_pairwise_locs(rnd(B, bench.OBJS, 3, scale=2.0), None)
shapes = [("bert_text_50", txt_pad, 0.1, None), ("bert_caption_300", cap_pad, 0.1, None),
          ("joint_130", torch.cat([txt_pad, obj_pad], 1), 0.1, None),
          ("spatial_80_gated", obj_pad, 0.0, rnd(B, bench.OBJS, H * 6))]
res = {"gpu": torch.cuda.get_device_name(dev), "scenes": B, "unit": "us per call"}
for name, mask, p, sw in shapes:
    L = mask.shape[1]
    q, k, v, go = (rnd(B, L, E).bfloat16() for _ in range(4))
    kw = dict(key_padding_mask=mask, dropout_p=p, seed=7)
    if sw is not None:
        kw.update(spatial_w=sw, pairwise_locs=locs)
    o, lse = native.attention(q, k, v, H, return_lse=True, spatial_heads=H if sw is not None else 0, **kw)
    t_f = timed(lambda: native.attention(q, k, v, H, return_lse=True, spatial_heads=H if sw is not None else 0, **kw))
    t_b = timed(lambda: native.attention_backward(q, k, v, o, go, lse, H, **kw))
    res[name] = {"fwd_us": round(t_f, 1), "bwd_us": round(t_b, 1)}
    print(name, res[name], flush=True)
if len(sys.argv) > 1:
    json.dump(res, open(sys.argv[1], "w"), indent=1)
