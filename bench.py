#!/usr/bin/env python
"""bench.py — one JSON line on rank 0 (contract in the task statement).

Workload (config.workload):
  gps_pretrain  (default)  BASELINE.json configs[3] on one node: the full GPS pre-training step of
      configs/final/all_pretrain.yaml (+TextObjBetweenBatch): B = 64 scenes/GPU x 80 object slots x 1024 points,
      50-token captions + 300-token scene captions; BERT-4L -> PointNet++ (frozen, native fused path) -> 4 spatial
      layers -> 4 joint layers -> OVPretrainHead -> lm_cls + 3 contrastive losses -> backward -> clip -> AdamW,
      bf16 autocast, data-parallel over scenes (NCCL gradient all-reduce + embedding all-gather).
      Metric: scenes/s (whole job).  `e2e` = the same step fed from pinned HOST buffers (H2D of the whole data_dict
      inside the timed region) with the loss read back.
  scanrefer     (--workload scanrefer)     BASELINE.json configs[2]: the same encoders with GroundHeadV1 (hidden 384) and
      og3d_loss (configs/final/finetune/scanrefer_finetune.yaml), B = 64 scenes/GPU, no scene captions.
  objcls        (--workload objcls)        BASELINE.json configs[1]: object-level pre-training, 64 objects x 1024 points, bf16,
      PointNet++ TRAINABLE with train-mode BatchNorm (model/objcls.py) on the native point operators (+ their gradients).
  pointops_sa1  (--workload pointops_sa1)  the FPS+ball_query front alone at the model shape (5120 x 1024), Mpts/s.
  pointops_sweep (--workload pointops_sweep) BASELINE.json configs[4]: FPS + ball query, 16 K - 1 M points, batch 1 - 256.

Every default run also measures the two gated kernels in isolation (CUDA events) and reports their rooflines:
  roofline           sa2_mlp tcgen05 kernel, tensor bound, vs measured bf16 TFLOP/s
  roofline_pointops  sa_sample kernel (FPS + ball query), HBM bound, vs measured copy GB/s
`--impl reference` times the CPU path (host cores) on a bounded sample: the same modules on CPU with the CPU oracle
standing in for the CUDA-only point ops (the reference has no CPU implementation of them, sampling.cpp:34).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SCENES, OBJS, PTS, TXT, SCENE_TXT = 64, 80, 1024, 50, 300
NPOINT, RADIUS, NSAMPLE = 32, 0.2, 32
# SURVEY.md §8(d): unfused accounting, fixed definition: FPS (12N+4m) + ball query (12N+12M+4*M*ns) = 29,184 B / cloud
ALG_BYTES_PER_CLOUD = (12 * PTS + 4 * NPOINT) + (12 * PTS + 12 * NPOINT + 4 * NPOINT * NSAMPLE)
SA2_FLOPS_PER_CLOUD = 2 * 512 * (131 * 128 + 128 * 128 + 128 * 256)  # algorithmic (unpadded K) flops of the SA2 MLP
METRIC = "GPS pre-train scenes/sec"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), float(d["bf16_tflops"]), "measured (MEASURED_PEAKS.json: copy GB/s, cuBLAS bf16 burst)"
    return 6650.0, 1590.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.stop = index, [], threading.Event()
        self.t = threading.Thread(target=self.run, daemon=True)

    def run(self):
        while not self.stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                parts = [x.strip() for x in out.strip().split(",")]
                if len(parts) >= 7:
                    self.rows.append(parts)
            except Exception:
                pass
            self.stop.wait(0.05)

    def __enter__(self):
        self.t.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        self.t.join(timeout=6)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        sm = sorted(float(r[0]) for r in self.rows)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[3 + i].lower().startswith("active") for r in self.rows)]
        pw = [float(r[2]) for r in self.rows if r[2].replace(".", "", 1).isdigit()]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.rows[0][1]), "reasons": reasons,
                "samples": len(self.rows), "power_w_max": max(pw) if pw else None}


DUMP_PARAM_SAMPLE = 4 << 20   # trainable parameters written by --dump-outputs (16 MB of float32)


def dump_outputs(out_dir, ps, loss):
    """What the last timed step hands its caller, as .npy files: the loss (float64), the L2 norm of every trainable parameter
    tensor after the update (float64, named_parameters order) and a fixed seeded sample of DUMP_PARAM_SAMPLE trainable
    parameter values (float32, positions in the concatenation of those tensors, ascending).  Inputs and initial weights are
    seeded, but the split-K weight gradients are summed with atomic adds in whatever order the CTAs finish, so two runs agree
    to float rounding, not bit for bit: compare with a tolerance."""
    import torch
    module = ps.module if hasattr(ps, "module") else ps.model
    params = [p.detach() for p in module.parameters() if p.requires_grad]
    flat = torch.cat([p.reshape(-1).float() for p in params])
    idx = np.unique(np.random.default_rng(0).integers(0, flat.numel(), size=min(flat.numel(), DUMP_PARAM_SAMPLE)))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "loss.npy"), np.array(loss, np.float64))
    np.save(os.path.join(out_dir, "param_norms.npy"),
            torch.stack([torch.linalg.vector_norm(p.double()) for p in params]).cpu().numpy())
    np.save(os.path.join(out_dir, "param_sample.npy"), flat[torch.from_numpy(idx).to(flat.device)].cpu().numpy())


def cpu_threads():
    """Threads for the CPU arm: every core up to 32 (beyond that the small ops of the step only get slower)."""
    return min(os.cpu_count() or 1, 32)


def make_scene_batches(n_batches, scenes, seed0):
    """Distinct synthetic batches; object clouds are drawn from a pool of 512 synthetic objects (generation cost)."""
    from sceneverse_b200 import synthetic
    out = []
    for i in range(n_batches):
        d = synthetic.scene_batch(seed0 + 1000 * i, B=scenes, O=OBJS, P=8, L=TXT, Ls=SCENE_TXT)  # layout only (P=8 is a stub)
        pool = synthetic.object_batch(seed0 + 1000 * i + 7, 512, PTS)
        rng = np.random.default_rng(seed0 + i)
        fts = np.ones((scenes, OBJS, PTS, 6), np.float32)
        pick = rng.integers(0, 512, size=(scenes, OBJS))
        m = d["obj_masks"]
        fts[m] = pool[pick[m]]
        d["obj_fts"] = fts
        out.append(d)
    return out


def cpu_reference_step_fn(scenes):
    """The GPS step on CPU: same host modules, CPU oracle as `_ext` (bench-only use of oracle/)."""
    import torch
    from oracle import pointops_ref
    from sceneverse_b200 import model as M, pointnet2_utils, train, weights
    pointops_ref.build()
    pointnet2_utils._ext = pointops_ref.RefExt()  # CPU stand-in for the CUDA-only operators, this process only
    torch.set_num_threads(cpu_threads())
    tf = weights.synthetic_tensor("text_features", (607, 768))
    ps = train.PretrainStep(M.pretrain_config(1, text_features=tf), "cpu", dtype=torch.float32)
    batch = {k: torch.from_numpy(v) for k, v in make_scene_batches(1, scenes, 42)[0].items()}
    return lambda: float(ps.step(dict(batch)))


def run_reference(args, config):
    scenes = 2
    step = cpu_reference_step_fn(scenes)
    steps = max(1, min(args.steps, 3))
    step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = (time.perf_counter() - t0) / steps
    val = scenes / dt
    cb = {"value": val, "unit": "scenes/s", "cores": cpu_threads(), "kind": "port",
          "sample": f"{scenes} scenes x {OBJS} objects x {PTS} pts per step (scenes/s extrapolated from {scenes} of the {SCENES} "
                    "scenes of a GPU step), full fwd+bwd+AdamW step in fp32 on "
                    "CPU: sceneverse_b200 host modules + oracle/pointops_ref.c as the point-op `_ext`, torch threads = min(cores, 32)"}
    print(json.dumps({"impl": "reference", "metric": METRIC, "value": val, "unit": "scenes/s", "n_gpus": 0, "steps": steps,
                      "warmup": 1, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
                      "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config, "cpu_baseline": cb,
                      "e2e": {"value": val, "unit": "scenes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def kernel_rooflines(torch, device):
    """The two gated kernels timed in isolation (CUDA events on the current stream, inputs rotated beyond L2)."""
    from sceneverse_b200 import _lib, synthetic, weights
    from sceneverse_b200.modules.pointnet import GPS_SPEC, PointNetPP
    from sceneverse_b200.pointnet2 import _ext
    hbm, tfl, src = peaks()
    B = SCENES * OBJS
    base = synthetic.object_batch(5, 512, PTS, 0.3)
    xs = [torch.from_numpy(np.ascontiguousarray(np.tile(base, (B // 512, 1, 1))[np.random.default_rng(i).permutation(B)]))
          .to(device) for i in range(3)]
    xyzs = [x[..., :3].contiguous() for x in xs]

    def timed(fn, n=20):
        for i in range(5):
            fn(i)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for i in range(n):
            fn(i)
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / n

    t_s = timed(lambda i: _ext.fps_ballquery(xyzs[i % 3], NPOINT, RADIUS, NSAMPLE))
    ach = ALG_BYTES_PER_CLOUD * B / (t_s * 1e-3) / 1e9
    # the meaningful "before": the reference's own CUDA kernels (sampling_gpu.cu / ball_query_gpu.cu compiled unmodified for
    # sm_100a into oracle/_ref, measurement only) on the same clouds: FPS -> gather -> ball query, as pointnet2_modules.py:54-58
    ref_ms = None
    try:
        from oracle import build_ref_ext
        ref = build_ref_ext.load_prebuilt()
        if ref is not None:
            def ref_chain(i):
                x = xyzs[i % 3]
                idx = ref.furthest_point_sampling(x, NPOINT)
                new = ref.gather_points(x.transpose(1, 2).contiguous(), idx).transpose(1, 2).contiguous()
                return ref.ball_query(new, x, RADIUS, NSAMPLE)
            ref_ms = timed(ref_chain, n=5)
    except Exception:
        ref_ms = None
    traffic = None
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    tj = json.load(open(tp)) if os.path.exists(tp) else {}
    rp = {"bound": "hbm", "kernel": "sa_sample_kernel<32> (FPS + ball query, one warp per cloud)", "ms": t_s,
          "mpts_per_s": B * PTS / (t_s * 1e-3) / 1e6, "achieved": ach, "peak": hbm, "unit": "GB/s", "frac": ach / hbm,
          "traffic": tj.get("sa_sample_kernel_dram_bytes_per_launch", traffic), "algorithmic_bytes_per_launch": ALG_BYTES_PER_CLOUD * B,
          "peak_source": src, "note": "binding bound is fp32 instruction issue, not HBM (DESIGN.md)",
          "ref_cuda_ms": ref_ms, "ref_cuda_what": "reference furthest_point_sampling + gather_points (+2 transposes) + ball_query, "
                                                  "its own sm_100a build (oracle/_ref), same 5120 x 1024 clouds"}
    net = PointNetPP(**GPS_SPEC).eval()
    net.load_state_dict(weights.synthetic_state_dict(net, 0))
    net = net.to(device)
    pk = net._pack()
    lib = _lib.gps()
    st = torch.cuda.current_stream().cuda_stream
    outs = [_ext.sa_sample2(xyz, 32, 0.2, 32, 16, 0.4, 32) for xyz in xyzs]
    feat1 = [torch.empty((B, 32, 128), dtype=torch.bfloat16, device=device) for _ in range(3)]
    feat2 = torch.empty((B, 16, 256), dtype=torch.bfloat16, device=device)
    for i in range(3):
        _lib.check(lib, lib.sv_sa1_mlp_bf16(xs[i].data_ptr(), outs[i][1].data_ptr(), outs[i][2].data_ptr(),
                                            pk["sa1"].data_ptr(), B, PTS, 32, feat1[i].data_ptr(), st), "sa1")

    def sa2(i):
        o = outs[i % 3]
        _lib.check(lib, lib.sv_sa2_mlp_bf16(o[1].data_ptr(), feat1[i % 3].data_ptr(), o[4].data_ptr(), o[5].data_ptr(),
                                            pk["sa2"].data_ptr(), B, 32, 32, feat2.data_ptr(), st), "sa2")
    t_m = timed(sa2)
    ach_t = SA2_FLOPS_PER_CLOUD * B / (t_m * 1e-3) / 1e12
    rt = {"bound": "tensor", "kernel": "sa_mlp_kernel<SA2> (gather + 3 tcgen05 GEMMs + max, 131->128->128->256)", "ms": t_m,
          "achieved": ach_t, "peak": tfl, "unit": "TFLOP/s", "frac": ach_t / tfl,
          "traffic": tj.get("sa2_mlp_kernel_dram_bytes_per_launch"), "algorithmic_flops_per_launch": SA2_FLOPS_PER_CLOUD * B,
          "peak_source": src}
    return rt, rp


def attention_rooflines(torch, device):
    """Attention kernels timed in isolation at the step's shapes (CUDA events): the attention CORE (4 B H Lq Lk 64 flops
    forward, 2.5x that backward) and, for the language-object cross-attention of the V1 / Entity stacks, the whole block
    projection GEMMs + core + output projection (SURVEY.md §8d: 2 (Lq + 2 Lk) D^2 + 2 Lq D^2 + 4 H Lq Lk dh per scene)."""
    from sceneverse_b200 import native
    _, tfl, src = peaks()
    B, H, D = SCENES, 12, 768
    g = torch.Generator(device=device).manual_seed(3)

    def rnd(*s_):
        return (torch.randn(*s_, device=device, generator=g) * 0.5).bfloat16()

    def timed(fn, n=20):
        for _ in range(5):
            fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(n):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / n
    out = {"peak": tfl, "unit": "TFLOP/s", "peak_source": src, "bound": "tensor"}
    for name, Lq, Lk in [("cross_80x50", 80, 50), ("joint_130", 130, 130), ("bert_300", 300, 300)]:
        q, k, v = rnd(B, Lq, D), rnd(B, Lk, D), rnd(B, Lk, D)
        go = rnd(B, Lq, D)
        o, lse = native.attention(q, k, v, H, return_lse=True)
        t_f = timed(lambda: native.attention(q, k, v, H, return_lse=True))
        t_b = timed(lambda: native.attention_backward(q, k, v, o, go, lse, H))
        fl = 4.0 * B * H * Lq * Lk * 64
        out[name] = {"fwd_ms": t_f, "bwd_ms": t_b, "fwd_tflops": fl / (t_f * 1e-3) / 1e12, "bwd_tflops": 2.5 * fl / (t_b * 1e-3) / 1e12,
                     "fwd_frac": fl / (t_f * 1e-3) / 1e12 / tfl, "bwd_frac": 2.5 * fl / (t_b * 1e-3) / 1e12 / tfl}
    # cross-attention block, forward: q-projection, packed k|v projection, core, output projection — all native kernels
    Lq, Lk = 80, 50
    xq, xkv = rnd(B * Lq, D), rnd(B * Lk, D)
    wq, wkv, wo = rnd(D, D), rnd(2 * D, D), rnd(D, D)
    bq, bkv, bo = torch.zeros(D, device=device), torch.zeros(2 * D, device=device), torch.zeros(D, device=device)

    def block():
        qq = native.linear_fwd(xq, wq, bq).view(B, Lq, D)
        kv = native.linear_fwd(xkv, wkv, bkv).view(B, Lk, 2 * D)
        oo = native.attention(qq, kv[..., :D], kv[..., D:], H)
        return native.linear_fwd(oo.view(B * Lq, D), wo, bo)
    t_blk = timed(block)
    fl_blk = B * (2.0 * (Lq + 2 * Lk) * D * D + 2.0 * Lq * D * D + 4.0 * H * Lq * Lk * 64)
    out["cross_80x50_block"] = {"fwd_ms": t_blk, "flops": fl_blk, "fwd_tflops": fl_blk / (t_blk * 1e-3) / 1e12,
                                "fwd_frac": fl_blk / (t_blk * 1e-3) / 1e12 / tfl,
                                "what": "q-proj GEMM + k|v-proj GEMM + attention core + out-proj GEMM (4 native launches)"}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="gps_pretrain",
                    choices=["gps_pretrain", "scanrefer", "objcls", "pointops_sa1", "pointops_sweep"])
    ap.add_argument("--overlap", action="store_true", help="N > 1: split the gradient all-reduce and capture it in the step graph (experimental)")
    ap.add_argument("--no-equal-work", action="store_true", help="N = 1: skip the extra run with distributed autograd semantics")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="run the step eagerly instead of replaying the captured CUDA graph")
    ap.add_argument("--no-kernel-rooflines", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="training-step workloads: after the timed steps, write what the last one computed to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.workload.startswith("pointops")):
        ap.error("--dump-outputs needs --impl b200 and a training-step workload (gps_pretrain, scanrefer, objcls)")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    warmup = max(args.warmup, 3)
    config = {"workload": args.workload, "scenes_per_gpu": SCENES, "objects_per_scene": OBJS, "points": PTS,
              "txt_len": TXT, "scene_txt_len": SCENE_TXT, "global_batch": SCENES * max(world, 1),
              "losses": ["lm_cls_loss", "TextObjWithinBatch", "TextObjBetweenBatch", "TextSceneBetweenBatch"],
              "optimizer": "AdamW + clip 5.0 + warmup-cosine", "backbone": "PointNet++ frozen (all_pretrain.yaml)",
              "l2": "3 distinct input batches rotated (3 x 126 MB of points > 126 MB L2)", "parallelism": f"dp{world}"}

    if args.impl == "reference":
        if rank == 0:
            run_reference(args, config)
        return 0

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
    from sceneverse_b200 import _lib, model as M, train, weights
    from sceneverse_b200.pointnet2 import _ext
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    stream = torch.cuda.current_stream()

    if args.workload == "pointops_sweep":
        # BASELINE.json configs[4]: FPS (m = N/32) + ball query (M = m centres, r = 0.2*(1024/N)^(1/3), nsample 32) on
        # unit-ball clouds, batch sharded over the ranks; Mpts/s = B*N / t, roofline = 28.5 algorithmic bytes per point
        from sceneverse_b200 import synthetic
        hbm, _, src = peaks()
        rows = []
        for (Bt, N) in [(256, 16384), (64, 16384), (16, 65536), (4, 262144), (1, 1048576)]:
            Bl = max(1, Bt // world)
            x = torch.from_numpy(synthetic.unit_ball_clouds(7 + rank, min(Bl, 8), N)).to(device)
            x = x.repeat((Bl + x.shape[0] - 1) // x.shape[0], 1, 1)[:Bl].contiguous()
            m, r = N // 32, 0.2 * (1024.0 / N) ** (1.0 / 3.0)
            idx = _ext.furthest_point_sampling(x, m)
            cen = torch.gather(x, 1, idx.long()[..., None].expand(-1, -1, 3)).contiguous()
            for _ in range(max(1, min(warmup, 3)) - 1):          # warm-up (the first call above was one)
                _ext.furthest_point_sampling(x, m)
                _ext.ball_query(cen, x, r, 32)
            torch.cuda.synchronize()
            iters = max(1, min(args.steps, 5))
            tf_ = tb_ = 0.0
            for _ in range(iters):
                e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
                e[0].record(stream)
                idx = _ext.furthest_point_sampling(x, m)
                e[1].record(stream)
                _ext.ball_query(cen, x, r, 32)
                e[2].record(stream)
                torch.cuda.synchronize()
                tf_ += e[0].elapsed_time(e[1]) / iters
                tb_ += e[1].elapsed_time(e[2]) / iters
            t = torch.tensor([tf_, tb_], device=device, dtype=torch.float64)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            tf_, tb_ = float(t[0]), float(t[1])
            pts = Bl * world * N
            ach = pts * 28.5 / ((tf_ + tb_) * 1e-3) / 1e9
            rows.append({"batch": Bl * world, "N": N, "m": m, "radius": r, "fps_ms": tf_, "ball_query_ms": tb_,
                         "mpts_per_s": pts / ((tf_ + tb_) * 1e-3) / 1e6, "hbm_frac": ach / hbm})
        if world > 1:
            dist.destroy_process_group()
        if rank == 0:
            best = max(rows, key=lambda r_: r_["mpts_per_s"])
            print(json.dumps({"metric": "FPS+ball_query Mpts/s (sweep 16K-1M points)", "value": best["mpts_per_s"], "unit": "Mpts/s",
                              "n_gpus": world, "steps": max(1, min(args.steps, 5)), "warmup": max(1, min(warmup, 3)),
                              "ms_per_step": best["fps_ms"] + best["ball_query_ms"],
                              "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
                              "data": "synthetic", "config": {"workload": "pointops_sweep", "parallelism": f"dp{world}"},
                              "sweep": rows, "roofline": {"bound": "hbm", "peak": hbm, "unit": "GB/s", "peak_source": src,
                                                          "achieved": best["hbm_frac"] * hbm, "frac": best["hbm_frac"], "traffic": None,
                                                          "note": "FPS is bound by the m-1 serial arg-max steps (one L2 exchange per step for N > 8192), not by HBM"},
                              "gpu_launches": 2 * len(rows)}))
        return 0

    if args.workload == "pointops_sa1":
        rt, rp = kernel_rooflines(torch, device)
        if rank == 0:
            print(json.dumps({"metric": "FPS+ball_query Mpts/s (model shape)", "value": rp["mpts_per_s"] * world, "unit": "Mpts/s",
                              "n_gpus": world, "steps": 20, "warmup": 5, "ms_per_step": rp["ms"], "higher_is_better": True,
                              "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                              "roofline": rp, "gpu_launches": 20}))
        return 0

    NBUF = 3
    tf = weights.synthetic_tensor("text_features", (607, 768))
    if args.workload == "objcls":
        # BASELINE.json configs[1]: 64 objects x 1024 points per step (one "scene" of 64 valid objects), labels for the CE
        from sceneverse_b200 import synthetic
        OBJ = 64
        np_batches = []
        for i in range(NBUF):
            d = synthetic.scene_batch(42 + rank + 1000 * i, B=1, O=OBJ, P=PTS, all_valid=True)
            np_batches.append({k: d[k] for k in ("obj_fts", "obj_labels", "obj_masks")})
        config.update(workload="objcls", objects_per_step=OBJ, scenes_per_gpu=None, objects_per_scene=None, global_batch=OBJ * max(world, 1),
                      txt_len=None, scene_txt_len=None, losses=["obj_cls_loss (label smoothing 0.3)"], optimizer="AdamW",
                      backbone="PointNet++ trainable, train-mode BatchNorm (model/objcls.py)",
                      l2="3 distinct input batches rotated (working set of one step: ~1 GB of grouped activations > L2)")
        ps = train.ObjClsStep(device, tf.to(device), dtype=torch.bfloat16, seed=1234, cuda_graph=not args.no_graph, num_gpu=1)
        units_per_step, unit = OBJ, "objects/s"
        metric = "ObjCls pre-train objects/sec (PointNet++ trainable)"
    else:
        np_batches = make_scene_batches(NBUF, SCENES, 42 + rank)
        if args.workload == "scanrefer":
            mcfg = M.scanrefer_config(world, text_features=tf)
            for b_ in np_batches:
                b_.pop("scene_txt_ids", None), b_.pop("scene_txt_masks", None)
            config.update(workload="scanrefer", scene_txt_len=None, losses=["og3d_loss"],
                          heads="GroundHeadV1 hidden 384 (configs/final/finetune/scanrefer_finetune.yaml)")
            metric = "ScanRefer grounding fine-tune scenes/sec"
        else:
            mcfg = M.pretrain_config(world, text_features=tf)
            metric = METRIC
        ps = train.PretrainStep(mcfg, device, dtype=torch.bfloat16, seed=1234, cuda_graph=not args.no_graph,
                                overlap_allreduce=args.overlap)
        units_per_step, unit = SCENES, "scenes/s"
    pinned = [{k: torch.from_numpy(v).pin_memory() for k, v in b.items()} for b in np_batches]
    resident = [{k: v.to(device) for k, v in p.items()} for p in pinned]
    h2d_bytes = sum(v.numel() * v.element_size() for v in pinned[0].values())
    config["cuda_graph"] = bool(ps.graph_mode)
    host_loss = torch.zeros((), dtype=torch.float32).pin_memory()

    def step_resident(i):
        return ps.step(dict(resident[i % NBUF]))

    # e2e: every step's inputs travel host -> device inside the timed region; the copy of step i+1 is issued on a
    # side stream while step i computes (two device-side staging slots), the loss is read back to pinned host memory
    copy_stream = torch.cuda.Stream(device=device)
    slots = [{k: torch.empty_like(v, device=device) for k, v in pinned[0].items()} for _ in range(2)]
    ready = [torch.cuda.Event() for _ in range(2)]
    consumed = [torch.cuda.Event() for _ in range(2)]
    state = {"primed": -1}

    def upload(i):
        s = i % 2
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[s])
            for k, v in pinned[i % NBUF].items():
                slots[s][k].copy_(v, non_blocking=True)
            ready[s].record(copy_stream)

    def step_e2e(i):
        if state["primed"] != i:   # first call of a timed loop: nothing was prefetched for it
            upload(i)
        upload(i + 1)
        state["primed"] = i + 1
        s = i % 2
        stream.wait_event(ready[s])
        loss = ps.step(dict(slots[s]))
        consumed[s].record(stream)
        host_loss.copy_(loss.float(), non_blocking=True)
        return loss

    def timed(fn, steps, warm):
        for i in range(warm):
            fn(i)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = _lib.launch_count()
        e0.record(stream)
        last = None
        for i in range(steps):
            last = fn(i)
        e1.record(stream)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        launches = _lib.launch_count() - l0
        if ps.graph_mode and hasattr(ps, "native_launches_per_step"):
            launches = steps * ps.native_launches_per_step   # replayed kernel nodes bypass the C-ABI launch counter
        t = torch.tensor([e0.elapsed_time(e1)], device=device, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), launches, float(last)

    with ClockSampler(local_rank) as cs:
        total_ms, launches, loss = timed(step_resident, args.steps, warmup)
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, ps, loss)   # before the e2e steps below move the parameters on
        e2e_ms, _, _ = timed(step_e2e, args.steps, warmup)
    clocks = cs.summary()
    ms_per_step = total_ms / args.steps
    value = world * units_per_step / (ms_per_step * 1e-3)
    e2e_value = world * units_per_step / (e2e_ms / args.steps * 1e-3)
    phases = equal_work = None
    if world > 1 and getattr(ps, "dp_graph", False) and ps.graph_opt is not None:
        # where the data-parallel step goes when nothing is overlapped: graph(forward+backward) | NCCL all-reduce | graph(clip+AdamW)
        pt = torch.tensor(ps.phase_times(dict(resident[0]), steps=10), device=device, dtype=torch.float64)
        dist.all_reduce(pt, op=dist.ReduceOp.MAX)
        phases = {"ms_fwd_bwd": float(pt[0]), "ms_allreduce": float(pt[1]), "ms_opt": float(pt[2]),
                  "note": "un-overlapped path, 3 + 10 extra steps after the timed region, CUDA events, max over ranks; the exchange kernel inside "
                          "forward+backward waits for the slowest peer, so rank skew shows up there"}
    if world == 1 and args.workload == "gps_pretrain" and not args.no_equal_work and not args.no_graph:
        # the step ONE rank of a data-parallel job executes (distributed autograd semantics of common/dist_utils.py:131-149: the
        # between-batch negatives carry no gradient, so the scene-caption text-encoder backward disappears) — the equal-work
        # N = 1 baseline of the scaling curve
        ps.close()
        mcfg2 = M.pretrain_config(1, text_features=tf)
        mcfg2["emulate_dist"] = True
        ps2 = train.PretrainStep(mcfg2, device, dtype=torch.bfloat16, seed=1234, cuda_graph=True)
        t2, _, _ = (lambda f: timed(f, args.steps, warmup))(lambda i: ps2.step(dict(resident[i % NBUF])))
        equal_work = {"ms_per_step": t2 / args.steps, "value": units_per_step / (t2 / args.steps * 1e-3), "unit": unit,
                      "what": "N = 1 with the autograd semantics of the N > 1 step (detached between-batch negatives)"}
        ps2.close()
    rt = rp = ra = None
    if rank == 0 and not args.no_kernel_rooflines:
        rt, rp = kernel_rooflines(torch, device)
        ra = attention_rooflines(torch, device)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return 0
    from sceneverse_b200 import ops
    launch_kind = ("one CUDA graph per step: forward + backward + all-reduce(behind the text encoder, overlapped) + all-reduce(text "
                   "encoder) + clip/AdamW" if getattr(ps, "overlapped", False) else
                   "CUDA graphs (forward+backward | NCCL all-reduce | clip+AdamW)" if getattr(ps, "dp_graph", False) else
                   "whole step captured in one CUDA graph" if ps.graph_mode else "eager")
    out = {"metric": metric, "value": value, "unit": unit, "n_gpus": world, "steps": args.steps, "warmup": warmup,
           "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
           "data": "synthetic", "config": config, "final_loss": loss,
           "e2e": {"value": e2e_value, "unit": unit, "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 4},
           "gpu_launches": int(launches), "clocks": clocks,
           "native_kernels_in_step": ["sa_sample_kernel (FPS + ball query, 2 SA levels)", "sa_mlp_kernel<SA1>", "sa_mlp_kernel<SA2>",
                                      "gemm_kernel<BN, FWD|DGRAD|WGRAD, 1|2 CTAs>: every nn.Linear of the step in all three directions "
                                      "(bias / ReLU / GELU / dropout / activation-derivative epilogues, split-K wgrad + bias gradient "
                                      "accumulated into the flat gradient buffer), SA3 chain + fc, LM-head decoder",
                                      "pairwise_locs_kernel",
                                      "attn_fwd_kernel / attn_bwd_kernel x16 (spatial gate x4, joint MHA x4, BERT self-attention x8; packed "
                                      "QKV, in-kernel attention dropout)",
                                      "ln_fwd / ln_bwd_dx / ln_bwd_dgb kernels x44 (dropout + residual + LayerNorm)",
                                      "ce_fwd_bwd_kernel + scale_inplace_kernel (masked-LM CE on the padded vocabulary)",
                                      "embedding_bwd_kernel / colsum kernels (BERT embedding gradients)",
                                      "sqnorm_partial_kernel + adamw_flat_kernel (clip + AdamW + bf16 shadows over the flat buffers)",
                                      "norm_allgather_kernel (N > 1: contrastive exchange over NVLink peer memory)"],
           "library_ops_in_step": ["residual / positional adds, dtype casts, softmax of the 64x64 contrastive logits, masked fills (ATen "
                                   "elementwise, ~14 % of the step)", "two 64x768x64 InfoNCE logit matmuls + the 607-class object head (cuBLAS, "
                                   "0.5 %)", "gradient all-reduce (NCCL, N > 1)"],
           "launch": launch_kind}
    if phases is not None:
        out["phases_unoverlapped"] = phases
    if equal_work is not None:
        out["equal_work_n1"] = equal_work
    if world > 1:
        out["allreduce_overlapped"] = bool(getattr(ps, "overlapped", False))
    if rt is not None:
        out["roofline"], out["roofline_pointops"] = rt, rp
    if ra is not None:
        out["roofline_attention"] = ra
    if not args.no_cpu_baseline and args.workload == "gps_pretrain":
        scenes = 2
        step = cpu_reference_step_fn(scenes)
        step()
        t0 = time.perf_counter()
        step()
        dt = time.perf_counter() - t0
        out["cpu_baseline"] = {"value": scenes / dt, "unit": "scenes/s", "cores": cpu_threads(), "kind": "port",
                               "sample": f"1 step of {scenes} scenes (of the {SCENES} of a GPU step: scenes/s EXTRAPOLATED from "
                                         f"{scenes}/{SCENES} of the batch) x {OBJS} x {PTS}, fp32, same modules on CPU with "
                                         "oracle/pointops_ref.c as `_ext`"}
    print(json.dumps(out))
    return 0


if __name__ == "__main__":
    sys.exit(main())
