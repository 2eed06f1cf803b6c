"""ORACLE — TEST INFRASTRUCTURE ONLY.  Run on a B200:  python oracle/make_golden_gpu.py OUT_DIR

Runs the REFERENCE's own CUDA kernels (oracle/_ref/_ext_ref.so = the reference's
_ext_src/src/*.cu compiled for sm_100a by oracle/build_ref_ext.py) on seeded inputs and writes
small .npz fixtures to OUT_DIR; they are then committed under tests/golden/:
  * pointops_*.npz (inputs + reference outputs) pin both the CPU oracle (tests/test_oracle.py) and the
    CUDA library (tests/test_pointops_gpu.py).  The CPU oracle is cross-checked on every one of them.
  * reference_cuda_cases.npz: reference outputs only, for the seeded inputs of tests/cases.py that
    tests/test_pointops_gpu.py compares bit for bit (a seeded sample of rows of the largest ball queries).
"""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import build_ref_ext, pointops_ref  # noqa: E402
from tests import cases  # noqa: E402


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def reference_cuda_cases(ref, out):
    z = {}
    for name, (xyz, m) in {**cases.fps_cases(), **cases.fps_cases_large()}.items():
        z["fps__" + name] = ref.furthest_point_sampling(dev(xyz), m).cpu().numpy()
    for name, (new_xyz, xyz, r, ns) in cases.bq_cases().items():
        z["bq__" + name] = ref.ball_query(dev(new_xyz), dev(xyz), r, ns).cpu().numpy()
    for j, (u, k, _, _, _) in enumerate(cases.three_nn_cases()):
        d, i = ref.three_nn(dev(u), dev(k))
        z[f"three_nn__{j}__dist2"], z[f"three_nn__{j}__idx"] = d.cpu().numpy(), i.cpu().numpy()
    for B, N in cases.SWEEP_SHAPES:
        xyz, m, r = cases.sweep_case(B, N)
        x = dev(xyz)
        idx = ref.furthest_point_sampling(x, m)
        cen = torch.gather(x, 1, idx.long()[..., None].expand(-1, -1, 3)).contiguous()
        bq = ref.ball_query(cen, x, r, 32).cpu().numpy().reshape(B * m, 32)
        rows = np.sort(np.random.default_rng(0).choice(B * m, size=min(B * m, 1024), replace=False))
        z[f"sweep__{B}x{N}__fps"] = idx.cpu().numpy()
        z[f"sweep__{B}x{N}__bq_rows"], z[f"sweep__{B}x{N}__bq"] = rows, bq[rows]
    np.savez_compressed(os.path.join(out, "reference_cuda_cases.npz"), **z)
    print("reference_cuda_cases:", len(z), "arrays,", sum(v.nbytes for v in z.values()), "bytes")


def main(out):
    ref = build_ref_ext.load_prebuilt()
    assert ref is not None, "oracle/_ref/_ext_ref.so missing"
    os.makedirs(out, exist_ok=True)
    reference_cuda_cases(ref, out)
    bad = 0
    fps = cases.fps_cases()
    keep = ["sa1_objects", "sa2_shape", "ball_n3", "ball_n80", "ball_n100", "ball_n513", "ball_n1000",
            "adversarial_n32", "adversarial_n80", "adversarial_n1024", "m_gt_n"]
    for name in keep:
        xyz, m = fps[name]
        idx = ref.furthest_point_sampling(dev(xyz), m).cpu().numpy()
        np.savez_compressed(os.path.join(out, f"pointops_fps_{name}.npz"), op="fps", xyz=xyz, m=m, idx=idx)
        ok = np.array_equal(pointops_ref.furthest_point_sampling(xyz, m), idx)
        bad += not ok
        print("fps", name, "oracle==reference:", ok)
    big = cases.fps_cases_large()
    for name in ["ball_n2048", "adversarial_n2048"]:
        xyz, m = big[name]
        idx = ref.furthest_point_sampling(dev(xyz), m).cpu().numpy()
        np.savez_compressed(os.path.join(out, f"pointops_fps_{name}.npz"), op="fps", xyz=xyz, m=m, idx=idx)
        ok = np.array_equal(pointops_ref.furthest_point_sampling(xyz, m), idx)
        bad += not ok
        print("fps", name, "oracle==reference:", ok)
    for name, (new_xyz, xyz, r, ns) in cases.bq_cases().items():
        if name in ("many_centres",):
            continue
        idx = ref.ball_query(dev(new_xyz), dev(xyz), r, ns).cpu().numpy()
        np.savez_compressed(os.path.join(out, f"pointops_bq_{name}.npz"), op="ball_query", new_xyz=new_xyz, xyz=xyz,
                            radius=r, nsample=ns, idx=idx)
        ok = np.array_equal(pointops_ref.ball_query(new_xyz, xyz, r, ns), idx)
        bad += not ok
        print("ball_query", name, "oracle==reference:", ok)
    rng = np.random.default_rng(1)
    u = rng.standard_normal((2, 200, 3)).astype(np.float32)
    k = rng.standard_normal((2, 48, 3)).astype(np.float32)
    d, i = ref.three_nn(dev(u), dev(k))
    d, i = d.cpu().numpy(), i.cpu().numpy()
    np.savez_compressed(os.path.join(out, "pointops_three_nn.npz"), op="three_nn", unknown=u, known=k, dist2=d, idx=i)
    od, oi = pointops_ref.three_nn(u, k)
    ok = np.array_equal(od, d) and np.array_equal(oi, i)
    bad += not ok
    print("three_nn oracle==reference:", ok)
    feats = rng.standard_normal((2, 6, 48)).astype(np.float32)
    w = rng.random((2, 200, 3)).astype(np.float32)
    o = ref.three_interpolate(dev(feats), dev(i), dev(w)).cpu().numpy()
    np.savez_compressed(os.path.join(out, "pointops_three_interpolate.npz"), op="three_interpolate", points=feats,
                        idx=i, weight=w, out=o)
    ok = np.array_equal(pointops_ref.three_interpolate(feats, i, w), o)
    bad += not ok
    print("three_interpolate oracle==reference:", ok)
    pts = rng.standard_normal((2, 6, 256)).astype(np.float32)
    gi = rng.integers(0, 256, size=(2, 8, 16)).astype(np.int32)
    o = ref.group_points(dev(pts), dev(gi)).cpu().numpy()
    np.savez_compressed(os.path.join(out, "pointops_group_points.npz"), op="group_points", points=pts, idx=gi, out=o)
    ok = np.array_equal(pointops_ref.group_points(pts, gi), o)
    bad += not ok
    print("group_points oracle==reference:", ok)
    print("GOLDEN_MISMATCHES", bad)
    return bad


if __name__ == "__main__":
    sys.exit(1 if main(sys.argv[1]) else 0)
