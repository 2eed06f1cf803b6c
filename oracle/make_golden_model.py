"""ORACLE — TEST INFRASTRUCTURE ONLY.  Run IN THE BUILD CONTAINER (needs /root/reference):
    python oracle/make_golden_model.py
Runs the UNMODIFIED reference Python modules on CPU (fp32) through oracle/ref_shims.py, with the CPU
restatement of the CUDA ops as `_ext`, on seeded synthetic inputs and name-keyed synthetic weights
(sceneverse_b200/weights.py — reproducible anywhere without the reference), and writes small
fixtures to tests/golden/model_*.npz / *.json.
"""
import json
import os
import sys
import tempfile

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref_shims  # noqa: E402
from sceneverse_b200 import synthetic, weights  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")


def golden_pointnetpp():
    from modules.layers.pointnet import PointNetPP
    net = PointNetPP(sa_n_points=[32, 16, None], sa_n_samples=[32, 32, None], sa_radii=[0.2, 0.4, None],
                     sa_mlps=[[3, 64, 64, 128], [128, 128, 128, 256], [256, 256, 512, 768]]).eval()
    net.load_state_dict(weights.synthetic_state_dict(net, seed=0))
    x = torch.from_numpy(synthetic.object_batch(3, 8, 1024, pad_fraction=0.25))
    inter = {}
    hooks = [net.encoder[i].register_forward_hook(lambda m, a, o, i=i: inter.__setitem__(i, o)) for i in range(3)]
    with torch.no_grad():
        y = net(x)
    for h in hooks:
        h.remove()
    np.savez_compressed(os.path.join(OUT, "model_pointnetpp.npz"),
                        input_seed=3, n_clouds=8, pad_fraction=0.25, weight_seed=0,
                        new_xyz1=inter[0][0].numpy(), feat1=inter[0][1].numpy(),
                        new_xyz2=inter[1][0].numpy(), feat2=inter[1][1].numpy(),
                        feat3=inter[2][1].numpy(), out=y.numpy())
    return {k: list(v.shape) for k, v in net.state_dict().items()}


def _load(m, seed=0):
    m.load_state_dict(weights.synthetic_state_dict(m, seed=seed))
    return m.eval()


def golden_gps_stack():
    """Config-1-like parity gate (BASELINE.json configs[0]): B=2 scenes x 32 object slots (second scene padded),
    P=1024, L=50; language features are seeded random (BERT is upstream of the path)."""
    import tempfile
    from modules.build import GROUNDING_REGISTRY, HEADS_REGISTRY, VISION_REGISTRY
    import importlib
    import types
    CL = importlib.import_module("optim.loss.contra_loss")
    LL = importlib.import_module("optim.loss.loss")
    og3d_loss, lm_cls_loss = LL.og3d_loss, LL.lm_cls_loss
    d = synthetic.scene_batch(21, B=2, O=32, P=1024, L=50, Ls=300, min_obj=12)
    t = {k: torch.from_numpy(v) for k, v in d.items()}
    g = torch.Generator().manual_seed(5)
    txt = torch.randn(2, 50, 768, generator=g) * 0.5
    scene_txt = torch.randn(2, 768, generator=g) * 0.5
    out = {}
    with tempfile.TemporaryDirectory() as tmp, torch.no_grad(), ref_shims.cpu_cuda_identity():
        ref_shims.write_text_features(tmp, weights.synthetic_tensor("text_features", (607, 768)))
        enc = _load(VISION_REGISTRY.get("PointOpenVocabEncoder")(None, lang_path=tmp, freeze=True))
        obj, obj_pre, sem = enc(t["obj_fts"], t["obj_locs"], t["obj_masks"], t["obj_sem_masks"], t["obj_labels"], 1, 1)
        out.update(vis_obj=obj.numpy(), vis_obj_pre=obj_pre.numpy(), vis_sem_cls=sem.numpy()[:, :, :64],
                   vis_sem_cls_argmax=sem.argmax(-1).numpy())
        v2 = _load(GROUNDING_REGISTRY.get("UnifiedSpatialCrossEncoderV2")(None), 1)
        t2, o2 = v2(txt, t["txt_masks"], obj, t["obj_locs"], t["obj_masks"])
        out.update(v2_txt=t2.numpy(), v2_obj=o2.numpy())
        v1 = _load(GROUNDING_REGISTRY.get("UnifiedSpatialCrossEncoderV1")(None), 2)
        t1, o1 = v1(txt, t["txt_masks"], obj, t["obj_locs"], t["obj_masks"])
        out.update(v1_txt=t1.numpy(), v1_obj=o1.numpy())
        en = _load(GROUNDING_REGISTRY.get("EntitySpatialCrossEncoder")(None), 3)
        _, oe = en(txt, t["txt_masks"], obj, t["obj_locs"], t["obj_masks"])
        out.update(entity_obj=oe.numpy())
        gh = _load(HEADS_REGISTRY.get("GroundHeadV1")(None, input_size=768, hidden_size=384, sem_cls_size=607), 4)
        a, b, c, dd = gh(t2, o2, obj_pre, t["obj_masks"])
        out.update(gh_txt_cls=a.numpy(), gh_obj_cls=b.numpy()[:, :, :64], gh_obj_cls_pre=c.numpy()[:, :, :64], gh_og3d=dd.numpy())
        ph = _load(HEADS_REGISTRY.get("OVPretrainHead")(None), 5)
        lm, ol = ph(t2, o2)
        out.update(ph_txt_lm_slice=lm.numpy()[:, :, :128], ph_txt_lm_rowsum=lm.sum(-1).numpy(), ph_obj_lm=ol.numpy()[:, :, :64])
        # losses (num_gpu = 1 -> no gather), data_dict keys as OpenVocab.forward fills them (openvocab.py:52-74)
        dd_ = dict(t)
        dd_.update(intra_obj_embeds=o2, intra_text_embed=t2[:, 0], inter_obj_embeds=obj, inter_text_embed=txt[:, 0],
                   scene_embed=obj.mean(dim=1), scene_text_embed=scene_txt, og3d_logits=dd.clone(),
                   txt_lm_cls_logits=lm)
        cfg = types.SimpleNamespace(num_gpu=1, task="Pretrain")
        out.update(loss_within=CL.TextObjWithinBatch(cfg)(dict(dd_, intra_obj_embeds=o2.clone())).numpy(),
                   loss_obj_between=CL.TextObjBetweenBatch(cfg)(dd_).numpy(),
                   loss_scene_between=CL.TextSceneBetweenBatch(cfg)(dd_).numpy(),
                   loss_og3d=og3d_loss(dd_).numpy(), loss_lm=lm_cls_loss(dd_).numpy())
    np.savez_compressed(os.path.join(OUT, "model_gps_stack.npz"), data_seed=21, txt_seed=5, **out)
    print({k: (v.shape if hasattr(v, "shape") else v) for k, v in out.items()})


def golden_gps_backward():
    """Backward parity fixture: the UNMODIFIED reference vision encoder (frozen PointNet++, trainable spatial layers) ->
    UnifiedSpatialCrossEncoderV2 -> GroundHeadV1 + OVPretrainHead -> lm + within + obj-between + scene-between + og3d
    losses, eval mode (no dropout), fp32 CPU; stores the loss, the gradient norm of EVERY trainable parameter and a few
    gradient slices.  tests/test_gps_modules.py replays it with the B200 classes."""
    import importlib
    import types
    from modules.build import GROUNDING_REGISTRY, HEADS_REGISTRY, VISION_REGISTRY
    CL = importlib.import_module("optim.loss.contra_loss")
    LL = importlib.import_module("optim.loss.loss")
    d = synthetic.scene_batch(33, B=2, O=16, P=1024, L=50, Ls=300, min_obj=6)
    t = {k: torch.from_numpy(v) for k, v in d.items()}
    g = torch.Generator().manual_seed(7)
    txt = torch.randn(2, 50, 768, generator=g) * 0.5
    scene_txt = torch.randn(2, 768, generator=g) * 0.5
    cfg = types.SimpleNamespace(num_gpu=1, task="Pretrain")
    with tempfile.TemporaryDirectory() as tmp, ref_shims.cpu_cuda_identity():
        ref_shims.write_text_features(tmp, weights.synthetic_tensor("text_features", (607, 768)))
        mods = {
            "enc": _load(VISION_REGISTRY.get("PointOpenVocabEncoder")(None, lang_path=tmp, freeze=True)),
            "v2": _load(GROUNDING_REGISTRY.get("UnifiedSpatialCrossEncoderV2")(None), 1),
            "gh": _load(HEADS_REGISTRY.get("GroundHeadV1")(None, input_size=768, hidden_size=384, sem_cls_size=607), 4),
            "ph": _load(HEADS_REGISTRY.get("OVPretrainHead")(None), 5),
            "l_within": CL.TextObjWithinBatch(cfg), "l_obj": CL.TextObjBetweenBatch(cfg), "l_scene": CL.TextSceneBetweenBatch(cfg),
        }
        pn = {}
        hk = mods["enc"].point_feature_extractor.register_forward_hook(lambda m, a, o: pn.__setitem__("out", o.detach()))
        obj, obj_pre, sem = mods["enc"](t["obj_fts"], t["obj_locs"], t["obj_masks"], t["obj_sem_masks"], t["obj_labels"], 1, 1)
        hk.remove()
        t2, o2 = mods["v2"](txt, t["txt_masks"], obj, t["obj_locs"], t["obj_masks"])
        _, _, _, og = mods["gh"](t2, o2, obj_pre, t["obj_masks"])
        lm, _ = mods["ph"](t2, o2)
        dd = dict(t)
        dd.update(intra_obj_embeds=o2, intra_text_embed=t2[:, 0], inter_obj_embeds=obj, inter_text_embed=txt[:, 0],
                  scene_embed=obj.mean(dim=1), scene_text_embed=scene_txt, og3d_logits=og, txt_lm_cls_logits=lm)
        parts = {"lm": LL.lm_cls_loss(dd), "within": mods["l_within"](dd), "obj_between": mods["l_obj"](dd),
                 "scene_between": mods["l_scene"](dd), "og3d": LL.og3d_loss(dd)}
        total = sum(parts.values())
        total.backward()
    norms, slices = {}, {}
    for mname, m in mods.items():
        for n, p in m.named_parameters():
            if p.grad is not None:
                norms[f"{mname}.{n}"] = float(p.grad.double().norm())
    for key in ["v2.unified_encoder.0.self_attn.in_proj_weight", "enc.spatial_encoder.0.self_attn.lang_cond_fc.weight",
                "ph.lm_pred_head.transform.dense.weight", "gh.og3d_head.0.weight", "enc.spatial_encoder.3.norm2.bias"]:
        mname, n = key.split(".", 1)
        slices[key] = dict(mods[mname].named_parameters())[n].grad.reshape(-1)[:96].numpy()
    np.savez_compressed(os.path.join(OUT, "model_gps_grads.npz"), data_seed=33, txt_seed=7, total=total.detach().numpy(),
                        pn_out=pn["out"].numpy(),   # frozen PointNet++ features: lets a CPU test skip the CUDA-only backbone
                        **{"loss_" + k: v.detach().numpy() for k, v in parts.items()},
                        **{"slice:" + k: v for k, v in slices.items()})
    json.dump(norms, open(os.path.join(OUT, "model_gps_grad_norms.json"), "w"), indent=0, sort_keys=True)
    print("backward golden:", float(total), len(norms), "parameter gradients")


def golden_qa_head():
    """QAHeadV1 (modules/heads/qa_head.py) with name-keyed synthetic weights (seed 11) on seeded object / text features."""
    import importlib
    ref = importlib.import_module("modules.heads.qa_head").QAHeadV1(None, num_answers=200).eval()
    ref.load_state_dict(weights.synthetic_state_dict(ref, seed=11))
    g = torch.Generator().manual_seed(0)
    obj, txt = torch.randn(3, 20, 768, generator=g), torch.randn(3, 12, 768, generator=g)
    om = torch.rand(3, 20, generator=g) > 0.3
    om[:, 0] = True
    tm = torch.arange(12)[None, :] < torch.tensor([12, 5, 9])[:, None]
    with torch.no_grad():
        out = ref(obj, om, txt, tm)
    shapes = json.dumps({k: list(v.shape) for k, v in ref.state_dict().items()})
    np.savez_compressed(os.path.join(OUT, "model_qa_head.npz"), weight_seed=11, input_seed=0, state_dict_shapes=shapes,
                        out=out.numpy())
    print("qa head golden:", tuple(out.shape))


def main():
    ref_shims.install()
    torch.manual_seed(0)
    golden_gps_stack()
    golden_gps_backward()
    golden_qa_head()
    shapes = {"PointNetPP": golden_pointnetpp()}
    # state_dict contracts of the registry classes (SURVEY.md §8b): key -> shape
    from modules.build import GROUNDING_REGISTRY, HEADS_REGISTRY, VISION_REGISTRY
    import modules.vision.pcd_openvocab_encoder  # noqa: F401
    import modules.grounding.unified_encoder  # noqa: F401
    import modules.heads.grounding_head  # noqa: F401
    import modules.heads.pretrain_head  # noqa: F401
    with tempfile.TemporaryDirectory() as d:
        ref_shims.write_text_features(d, weights.synthetic_tensor("text_features", (607, 768)))
        enc = VISION_REGISTRY.get("PointOpenVocabEncoder")(None, lang_path=d, freeze=True)
    shapes["PointOpenVocabEncoder"] = {k: list(v.shape) for k, v in enc.state_dict().items()}
    for name in ["UnifiedSpatialCrossEncoderV2", "UnifiedSpatialCrossEncoderV1", "EntitySpatialCrossEncoder"]:
        m = GROUNDING_REGISTRY.get(name)(None)
        shapes[name] = {k: list(v.shape) for k, v in m.state_dict().items()}
    for name, kw in [("GroundHeadV1", dict(input_size=768, hidden_size=384, sem_cls_size=607)), ("GroundHead", {}),
                     ("PretrainHeadV1", {}), ("OVPretrainHead", {})]:
        m = HEADS_REGISTRY.get(name)(None, **kw)
        shapes[name] = {k: list(v.shape) for k, v in m.state_dict().items()}
    json.dump(shapes, open(os.path.join(OUT, "state_dict_shapes.json"), "w"), indent=0, sort_keys=True)
    print({k: len(v) for k, v in shapes.items()})


if __name__ == "__main__":
    main()
