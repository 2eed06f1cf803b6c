"""Seeded input cases shared by the CPU (oracle) and GPU (parity) tests."""
import numpy as np

from sceneverse_b200 import synthetic


def fps_cases():
    """name -> (xyz (B,N,3) float32, m)"""
    cases = {}
    objs = synthetic.object_batch(7, 12, P=1024, pad_fraction=0.2)
    cases["sa1_objects"] = (np.ascontiguousarray(objs[:, :, :3]), 32)
    cases["sa2_shape"] = (synthetic.unit_ball_clouds(11, 9, 32), 16)
    for n, m in [(1, 1), (2, 2), (3, 2), (16, 5), (31, 7), (33, 9), (64, 16), (80, 20), (100, 25), (255, 17),
                 (512, 24), (513, 24), (1000, 32), (1023, 31), (1024, 40)]:
        cases[f"ball_n{n}"] = (synthetic.unit_ball_clouds(100 + n, 3, n), m)
    for n in (32, 80, 1024):
        adv = synthetic.adversarial_clouds(200 + n, n)
        cases[f"adversarial_n{n}"] = (np.stack([adv[k] for k in sorted(adv)]), min(n, 32))
    cases["m_gt_n"] = (synthetic.unit_ball_clouds(5, 2, 8), 12)
    return cases


def fps_cases_large():
    cases = {}
    for n, m in [(1025, 16), (2048, 32), (3000, 20), (4096, 16), (8192, 12), (8193, 8), (20000, 10)]:
        cases[f"ball_n{n}"] = (synthetic.unit_ball_clouds(300 + n, 2, n), m)
    adv = synthetic.adversarial_clouds(9, 2048)
    cases["adversarial_n2048"] = (np.stack([adv[k] for k in sorted(adv)]), 24)
    adv = synthetic.adversarial_clouds(10, 9000)
    cases["adversarial_n9000"] = (np.stack([adv[k] for k in sorted(adv)]), 12)
    cases["ball_n65536"] = (synthetic.unit_ball_clouds(77, 3, 65536), 40)          # 16 CTAs per cloud
    cases["ball_n300000_b2"] = (synthetic.unit_ball_clouds(78, 2, 300000), 6)      # 74 CTAs per cloud, 2 waves of clouds
    adv = synthetic.adversarial_clouds(11, 16384)
    cases["adversarial_n16384"] = (np.stack([adv[k] for k in sorted(adv)]), 16)
    return cases


def three_nn_cases():
    """[(unknown (B,n,3), known (B,m,3), feats (B,c,m), weight (B,n,3), grad_out (B,c,n))], one seeded stream"""
    rng = np.random.default_rng(1)
    out = []
    for (B, n, m, c) in [(2, 300, 64, 8), (1, 17, 2, 3), (2, 1024, 2500, 4)]:
        u = rng.standard_normal((B, n, 3)).astype(np.float32)
        k = rng.standard_normal((B, m, 3)).astype(np.float32)
        feats = rng.standard_normal((B, c, m)).astype(np.float32)
        w = rng.random((B, n, 3)).astype(np.float32)
        g = rng.standard_normal((B, c, n)).astype(np.float32)
        out.append((u, k, feats, w, g))
    return out


# BASELINE.json configs[4] shapes: (batch, points); m = N/32, r = 0.2 (1024/N)^(1/3), nsample 32
SWEEP_SHAPES = [(2, 16384), (1, 65536), (1, 262144)]


def sweep_case(B, N):
    """(xyz (B,N,3), m, radius) of one sweep shape"""
    return synthetic.unit_ball_clouds(11, B, N), N // 32, float(0.2 * (1024.0 / N) ** (1.0 / 3.0))


def bq_cases():
    """name -> (new_xyz (B,M,3), xyz (B,N,3), radius, nsample)"""
    rng = np.random.default_rng(3)
    cases = {}
    objs = synthetic.object_batch(8, 10, P=1024, pad_fraction=0.2)
    xyz = np.ascontiguousarray(objs[:, :, :3])
    ctr = xyz[:, rng.permutation(1024)[:32]]
    cases["sa1"] = (np.ascontiguousarray(ctr), xyz, 0.2, 32)
    x2 = synthetic.unit_ball_clouds(12, 7, 32)
    cases["sa2"] = (np.ascontiguousarray(x2[:, :16]), x2, 0.4, 32)
    x3 = synthetic.unit_ball_clouds(13, 3, 3000)
    cases["big_tile"] = (np.ascontiguousarray(x3[:, ::40]), x3, 0.15, 16)       # 75 centres, 2 tiles
    cases["many_centres"] = (np.ascontiguousarray(x3[:, :300]), x3, 0.3, 64)   # >8 warps of centres
    cases["no_hits"] = (np.ascontiguousarray(x2[:, :5] + 10.0), x2, 0.1, 8)
    cases["nsample1"] = (np.ascontiguousarray(x2[:, :7]), x2, 0.5, 1)
    cases["nsample_odd"] = (np.ascontiguousarray(x2[:, :33 % 32 + 3]), x2, 0.6, 13)
    lat = synthetic.adversarial_clouds(14, 512)["lattice"][None]
    cases["lattice_ties"] = (np.ascontiguousarray(lat[:, :40]), lat, 0.25, 20)  # d2 == r2 exactly -> excluded
    return cases
