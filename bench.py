#!/usr/bin/env python
"""bench.py -- frames/sec of the per-frame keypoint-voting hot path on synthetic 12288-pt RGB-D clouds.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--config linemod|ycb]
                    [--ms-mode certified|early_exit|strict] [--quick] [--dump-outputs DIR]

Metric / config (BASELINE.json): frames/sec; headline workload = configs[1]: LineMOD-shape synthetic,
12288 pts, 1 instance, 8 kps, batch 32 per GPU.  A step = one pass of hot path A (Pointnet2MSG.forward)
+ hot path B (cal_frame_poses_lm) over one batch.  N > 1 (launched by torchrun): every rank owns its
own frames (weak scaling, frames sharded across ranks, no data-path collective) and a step ends with
ONE NCCL all_gather of the poses.  Timing: CUDA events around exactly K steps, barrier + synchronize
on both sides, max over ranks.  Inputs: 4 rotating device-resident batches (252 MB > the 126 MB L2).

The ONE JSON line also carries (rank 0):
  e2e                 same metric through FramePipeline.run_host (pinned host in, H2D + D2H inside the
                      timed region)
  roofline            the dominant kernel family of the step (shared-MLP engine), HBM-bound: algorithmic
                      bytes (SURVEY section 8d) / event-timed duration vs MEASURED_PEAKS.json
  rooflines           every kernel family ON the step (timed live with CUDA events inside an
                      instrumented pass) + the stand-alone fused ball-query+group API call
  frames_per_s_hbm_frac   value / (HBM peak / 196.5 MB per frame)  (north_star: "fraction of the HBM roofline")
  meanshift_modes     the same step with the all-seeds modes (early_exit, strict = reference iteration counts)
  configs             BASELINE configs[2] (YCB b16/GPU; with --gpus 8 this is configs[3]: b128 sharded) and
                      configs[4] (49152 pts, 10 instances, bandwidth sweep), each with its own clock sample
  cpu_baseline        the CPU port of the path on the host cores (bounded sample, see its `sample`)
  stock_gpu_baseline  the UNMODIFIED reference on this GPU: reference `_ext` (oracle/_ref/_ext.so) under the
                      reference Pointnet2MSG + reference cal_frame_poses_lm / MeanShiftTorch on CUDA tensors
`--impl reference` times the CPU implementation of the same path (oracle port; the reference's
PointNet++ ops have no CPU path and /root/reference is absent on the GPU box) on the host cores.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_POINTS = 12288
CONFIGS = {
    "linemod": dict(batch=32, shape="linemod", config_id=2, n_points=12288, n_inst=None,
                    label="LineMOD-shape synthetic, 12288 pts, 1 instance, 8 kps"),
    "ycb": dict(batch=16, shape="ycb", config_id=3, n_points=12288, n_inst=None,
                label="YCB-shape synthetic, 12288 pts, 21 classes, 5 instances, 8 kps/obj"),
    "stress": dict(batch=8, shape="ycb", config_id=5, n_points=49152, n_inst=10,
                   label="dense-cloud stress, 49152 pts, 10 instances, 8 kps/obj"),
}
FRAME_HBM_BYTES = 196.5e6      # SURVEY section 8d: whole frame, path A, at reference op boundaries
MLP_IO_BYTES = 100.2e6         # SURVEY section 8d: MLP stage I/O per frame with every SharedMLP(+pool) one fused kernel
MLP_FLOPS = 17.45e9            # SURVEY section 8d: SA + FP shared MLPs per frame
GOLDEN_LM = os.path.join(ROOT, "tests", "golden", "poses_lm_big.npz")   # reference sweep counts of bench frame 0


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md copy bandwidth)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING a timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.rows, self.proc, self.th = [], None, None
        self.idx = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50", "-i", str(self.idx)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return self

        def pump():
            for line in self.proc.stdout:
                self.rows.append(line.strip())
        self.th = threading.Thread(target=pump, daemon=True)
        self.th.start()
        return self

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "samples": 0, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); smax.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        load = [s for s in sm if s > 0]
        return {"sm_mhz": statistics.median(load) if load else None,
                "sm_max_mhz": max(smax) if smax else None, "samples": len(load), "reasons": sorted(reasons)}


def qg_algorithmic_bytes(b, n, m, c, ns):
    """fused ball-query+group, one (level, scale): read xyz + new_xyz + feats; write idx + grouped
    (SURVEY section 8d, DESIGN.md section 4)."""
    return b * (12 * n + 12 * m + 4 * c * n + 4 * m * ns + 4 * (3 + c) * m * ns)


# ------------------------------------------------------------------------------------------------
# CPU port of the path (oracle/) -- the `cpu_baseline` leg and the `--impl reference` arm
# ------------------------------------------------------------------------------------------------
def reference_sweep_counts():
    """T per fit (centre + 8 keypoints) the REFERENCE needed on the first frame of the LineMOD bench
    batch, recorded from the reference itself (tests/golden/make_golden_big.py).  Shipped as a fixture so
    that both arms scale the CPU sample by the same counts."""
    if os.path.exists(GOLDEN_LM):
        z = np.load(GOLDEN_LM)
        return [int(x) for x in z["raw_fit_iters"]], int(z["n_c"])
    return [98, 134, 152, 237, 137, 117, 123, 104, 162], 3348     # the same numbers, should the fixture be absent


_THREAD_PROBE = {}


def best_thread_count(votes, candidates):
    """torch CPU mean-shift sweeps are memory-bound on [n,n,3] temporaries: more threads are not always
    faster on a many-core host.  Probe (3 sweeps each, once per process) and keep the fastest."""
    import torch
    from oracle.meanshift_oracle import MeanShiftOracle

    key = (int(votes.shape[0]), tuple(candidates))
    if key in _THREAD_PROBE:
        torch.set_num_threads(_THREAD_PROBE[key][0])
        return _THREAD_PROBE[key]
    res = {}
    for nt in candidates:
        torch.set_num_threads(nt)
        MeanShiftOracle(0.08, max_iter=0).fit(votes)        # warm: thread pool + allocator at this size
        ms = MeanShiftOracle(0.08, max_iter=2)
        t0 = time.perf_counter()
        ms.fit(votes)
        res[nt] = (time.perf_counter() - t0) / 4.0          # 3 sweeps + the density/label pass
    best = min(res, key=res.get)
    torch.set_num_threads(best)
    _THREAD_PROBE[key] = (best, {str(k): round(v * 1e3, 1) for k, v in res.items()})
    return _THREAD_PROBE[key]


def cpu_path_sample(frame, sd, sweep_budget_s, complete_fit):
    """Bounded CPU sample of one LineMOD bench frame.
    hot path A: Pointnet2MSG.forward of the frame in full (C oracle ops + torch-CPU MLPs), warm, best of 2.
    hot path B: mean-shift on the frame's real centre votes (n_c = 3348): `complete_fit` runs the first
    fit of the frame to its end (98 sweeps by the reference's count); otherwise as many sweeps as fit in
    `sweep_budget_s`.  The per-sweep cost is scaled to the frame's 9 fits with the reference's recorded
    sweep counts.  Returns (seconds per frame, description dict)."""
    import torch
    from oracle import pointnet2_cpu
    from oracle.meanshift_oracle import MeanShiftOracle, best_fit_transform

    cores = os.cpu_count() or 1
    counts, n_c_ref = reference_sweep_counts()
    sel = frame.labels == frame.cls_ids[0]
    votes = torch.from_numpy(frame.pcld[sel] - frame.ctr_of[0][sel])
    cands = sorted({c for c in (cores, 64, 32, 16, 8) if c <= cores}, reverse=True)
    nt, probe = best_thread_count(votes, cands)
    t_sweep_probe = float(probe[str(nt)]) * 1e-3
    # hot path A (first call builds / loads the C oracle and spins the thread pools up: not timed)
    pointnet2_cpu.forward(frame.cld_rgb_nrm[None], sd, threads=cores)
    t_a = []
    for _ in range(2):
        t0 = time.perf_counter()
        pointnet2_cpu.forward(frame.cld_rgb_nrm[None], sd, threads=cores)
        t_a.append(time.perf_counter() - t0)
    # hot path B
    full = complete_fit and t_sweep_probe * (counts[0] + 1) <= 90.0
    n_iter = counts[0] if full else max(2, int(sweep_budget_s / max(t_sweep_probe, 1e-3)) - 1)
    ms = MeanShiftOracle(0.08, max_iter=300 if full else n_iter - 1)
    t0 = time.perf_counter()
    ms.fit(votes)
    t_fit = time.perf_counter() - t0
    sweeps_timed = ms.n_iter + 1                                   # + the density / label pass
    t_sweep = t_fit / sweeps_timed
    total_sweeps = sum(t + 1 for t in counts)
    t0 = time.perf_counter()
    best_fit_transform(np.random.rand(9, 3).astype(np.float32), np.random.rand(9, 3).astype(np.float32))
    t_b = total_sweeps * t_sweep + (time.perf_counter() - t0)
    info = {"path_a_s": [round(x, 3) for x in t_a], "threads_meanshift": nt, "ms_per_sweep_by_threads": probe,
            "sweeps_timed": sweeps_timed, "complete_fit": bool(full and ms.n_iter == counts[0]),
            "ms_per_sweep": round(t_sweep * 1e3, 1), "sweeps_per_frame": total_sweeps, "n_c": int(sel.sum())}
    desc = (f"1 frame of the workload: hot path A in full (best of 2 warm runs: {min(t_a):.2f}s); hot path B = "
            f"{'one COMPLETE fit' if info['complete_fit'] else 'a capped fit'} of {sweeps_timed} torch-CPU mean-shift sweeps at "
            f"n_c={int(sel.sum())} on {nt} threads ({t_sweep * 1e3:.0f} ms/sweep), scaled to the {total_sweeps} sweeps the "
            f"reference needs for the frame's 9 fits (recorded counts, tests/golden/poses_lm_big.npz)")
    return min(t_a) + t_b, desc, info


def reference_arm(args, json_out, rank):
    """`--impl reference`: the CPU implementation of the path on the host cores (rank 0 only)."""
    if rank != 0:
        return 0
    import torch  # noqa: F401
    from pvn3d_b200 import synth, testing

    cfg = CONFIGS["linemod"]
    frames = synth.make_batch(cfg["shape"], 1, n_points=cfg["n_points"], config_id=cfg["config_id"], lm_obj_id=1)
    sd = testing.seeded_pointnet2msg(0, 1).state_dict()
    times, desc, info = [], "", {}
    n = max(1, args.steps) + max(0, args.warmup)
    budget = max(1.5, min(6.0, 150.0 / n))        # the whole run stays within a few minutes
    for s in range(n):
        t, desc, info = cpu_path_sample(frames[0], sd, sweep_budget_s=budget, complete_fit=False)
        if s >= args.warmup:
            times.append(t)
    sec = statistics.median(times)
    value = 1.0 / sec
    cores = os.cpu_count() or 1
    line = {"metric": "frames/sec", "value": value, "unit": "frames/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "impl": "reference",
            "config": {"workload": workload_name(cfg), "n_points": cfg["n_points"], "parallelism": "host cores",
                       "note": "per-frame time is EXTRAPOLATED from a bounded sample: one frame of the reference's CPU path "
                               "takes ~10 minutes (9 fits x ~140 sweeps over n_c^2 = 1.1e7 pairs)"},
            "cpu_baseline": {"value": value, "unit": "frames/s", "cores": cores, "kind": "port", "sample": desc,
                             "detail": info, "spread_s_per_frame": [round(min(times), 2), round(max(times), 2)]},
            "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    json_out.write(json.dumps(line) + "\n")
    json_out.flush()
    return 0


def cpu_pose_path_ycb(frame, gpu_ms_per_frame):
    """north_star: ">= 200x the reference CPU MeanShift wall-clock on 12288-point YCB-shape clouds at 1 GPU".
    One COMPLETE YCB frame of hot path B on the host cores through the CPU port (oracle/frame_poses_oracle.py =
    pvn3d_eval_utils.py:37-110 on CPU tensors: centre-cluster filter pass, 5 classes x (1 + 8) fits, Kabsch)."""
    import torch
    from oracle import frame_poses_oracle
    from pvn3d_b200 import fixtures

    torch.set_num_threads(min(16, os.cpu_count() or 1))
    args = (torch.from_numpy(frame.pcld), torch.from_numpy(frame.labels), torch.from_numpy(frame.ctr_of),
            torch.from_numpy(frame.kp_of))
    r = fixtures.ycb_r_lst()
    t0 = time.perf_counter()
    frame_poses_oracle.cal_frame_poses(*args, True, 22, True, lambda c: fixtures.get_kps(c), lambda c: fixtures.get_ctr(c), r)
    sec = time.perf_counter() - t0
    return {"cpu_s_per_frame": sec, "threads": torch.get_num_threads(), "gpu_ms_per_frame": gpu_ms_per_frame,
            "speedup": sec * 1e3 / gpu_ms_per_frame, "kind": "port",
            "sample": "hot path B of ONE complete YCB frame (5 instances, 50 fits) on the CPU port, wall clock"}


def workload_name(cfg):
    return f"{cfg['label']}, batch {cfg['batch']}/GPU"


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
class Runner:
    """one configuration: frames, pipeline, rotating device / pinned host batches, timed loops"""

    def __init__(self, torch, cfg, dev, rank, world, ms_mode, overlap=True, engine="fused", bandwidth=0.08, n_rot=4,
                 lookahead=True):
        from pvn3d_b200 import synth
        from pvn3d_b200.pipeline import FramePipeline

        self.torch, self.cfg, self.dev, self.rank, self.world = torch, cfg, dev, rank, world
        #: the loop names the next batch, so its coordinate-only work (FPS, ball query, 3-NN) runs under this batch's MLPs
        self.lookahead = bool(lookahead and overlap)
        B = self.B = cfg["batch"]
        kw = dict(lm_obj_id=1) if cfg["shape"] == "linemod" else {}
        if cfg.get("n_inst"):
            kw["n_instances"] = cfg["n_inst"]
        self.frames = synth.make_batch(cfg["shape"], B, n_points=cfg["n_points"], config_id=cfg["config_id"],
                                       first_frame=rank * B, **kw)
        self.pipe = FramePipeline(cfg["shape"], B, n_points=cfg["n_points"], device=dev, lm_obj_id=1, ms_mode=ms_mode,
                                  engine=engine, overlap=overlap, bandwidth=bandwidth,
                                  pose_stream=os.environ.get("PVN3D_POSE_STREAM", "1") != "0")
        host = synth.stack(self.frames)
        self.n_rot = n_rot
        self.host_rot = [FramePipeline.pin_batch({k: np.roll(v, (B // n_rot) * r, axis=0) for k, v in host.items()})
                         for r in range(n_rot)]
        self.dev_rot = [{k: v.to(dev) for k, v in hb.items()} for hb in self.host_rot]
        self.rot_bytes = sum(v.numel() * v.element_size() for v in self.dev_rot[0].values()) * n_rot
        self.gather_buf = (torch.empty((world * B * self.pipe.n_cls * 12,), dtype=torch.float32, device=dev)
                           if world > 1 else None)

    def step_device(self, i):
        d = self.dev_rot[i % self.n_rot]
        nxt = self.dev_rot[(i + 1) % self.n_rot]["cld_rgb_nrm"] if self.lookahead else None
        poses, present = self.pipe.run_device(d["cld_rgb_nrm"], d["pcld"], d["labels"], d["ctr_of"], d["kp_of"],
                                              next_cloud=nxt)
        self.last = poses, present
        if self.world > 1:   # the single collective of the path: ~1.5 kB per frame
            self.torch.distributed.all_gather_into_tensor(self.gather_buf, poses.reshape(-1))

    def outputs(self, n_feature_points=1024):
        """What the last device step computed, on the host as float32: poses [B,n_cls,3,4], present [B,n_cls] and hot
        path A's features [B,128,N] at a fixed seeded sample of n_feature_points points (the poses do not depend on
        the features: the votes are inputs).  Call right after the step: later steps reuse the output buffers."""
        poses, present = self.last
        pts = np.sort(np.random.default_rng(0).choice(self.cfg["n_points"], n_feature_points, replace=False))
        feats = self.pipe.features.index_select(2, self.torch.from_numpy(pts).to(self.dev))
        return {"poses": poses.float().cpu().numpy(), "present": present.float().cpu().numpy(),
                "features_sample": feats.float().cpu().numpy()}

    def step_host(self, i):
        self.pipe.run_host(self.host_rot[i % self.n_rot], self.host_rot[(i + 1) % self.n_rot] if self.lookahead else None)
        if self.world > 1:
            self.torch.distributed.all_gather_into_tensor(self.gather_buf, self.pipe.solver.poses.reshape(-1))

    def barrier(self):
        if self.world > 1:
            self.torch.distributed.barrier()
        self.torch.cuda.synchronize(self.dev)

    def timed(self, fn, steps, lib=None):
        from pvn3d_b200 import dist as pdist

        torch = self.torch
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = lib.pvn3d_launch_count() if lib is not None else 0
        e0.record()
        for i in range(steps):
            fn(i)
        e1.record()
        self.barrier()
        ms = e0.elapsed_time(e1)
        return pdist.max_over_ranks(ms, self.dev), (lib.pvn3d_launch_count() - l0 if lib is not None else 0)

    def measure(self, steps, warmup, lib, e2e=True, clocks=True, keep_outputs=False):
        # W untimed steps of exactly the loop that is timed next (indices -W..-1, so that the look-ahead of the
        # last warm-up step names the first timed batch), then K timed steps; first the device-resident loop,
        # then the same for the host loop
        for i in range(-warmup, 0):
            self.step_device(i)
        sampler = ClockSampler(self.dev.index or 0).start() if (clocks and self.rank == 0) else None
        ms_dev, launches = self.timed(self.step_device, steps, lib)
        kept = self.outputs() if keep_outputs else None
        ms_e2e = None
        if e2e:
            for i in range(-warmup, 0):
                self.step_host(i)
            ms_e2e = self.timed(self.step_host, steps)[0]
        ck = sampler.stop() if sampler is not None else None
        frames = self.B * self.world * steps
        out = {"value": frames / (ms_dev * 1e-3), "unit": "frames/s", "ms_per_step": ms_dev / steps,
               "global_batch": self.B * self.world, "gpu_launches": int(launches), "clocks": ck}
        if kept is not None:
            out["outputs"] = kept
        if e2e:
            out["e2e"] = {"value": frames / (ms_e2e * 1e-3), "unit": "frames/s", "h2d_bytes_per_step": self.pipe.h2d_bytes(),
                          "d2h_bytes_per_step": self.pipe.d2h_bytes(), "ms_per_step": ms_e2e / steps}
        return out

    def set_mode(self, mode, bandwidth=0.08):
        from pvn3d_b200.eval_utils import FramePoseSolver

        s = self.pipe.solver
        self.pipe.solver = FramePoseSolver(s.b, s.n, s.k, s.n_cls, s.mesh_kps.cpu().numpy(),
                                           None if s.cls_radius is None else s.cls_radius.cpu().numpy(),
                                           s.use_filter, device=self.dev, mode=mode, bandwidth=bandwidth)

    def median_ms(self, fn, reps=5, warm=2):
        torch = self.torch
        for _ in range(warm):
            fn()
        out = []
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize(self.dev)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize(self.dev)
            out.append(e0.elapsed_time(e1))
        return statistics.median(out)

    def path_a_ms(self, i=0):
        d = self.dev_rot[i % self.n_rot]
        eng = self.pipe.fused if self.pipe.fused is not None else self.pipe.model
        with self.torch.no_grad():
            return self.median_ms(lambda: eng(d["cld_rgb_nrm"]))

    def path_b_ms(self, i=0):
        d = self.dev_rot[i % self.n_rot]
        return self.median_ms(lambda: self.pipe.solver.solve(d["pcld"], d["labels"], d["ctr_of"], d["kp_of"]))


def meanshift_work(torch, runner):
    """pair evaluations of one batch in strict mode (sum over fits of T * n_c^2), from the solver's outputs"""
    from pvn3d_b200.meanshift import MeanShiftTorch

    d = runner.dev_rot[0]
    ms = MeanShiftTorch(0.08, mode="strict")
    pairs, dens_pairs, sweeps0 = 0.0, 0.0, None
    for b in range(runner.B):
        labels = d["labels"][b]
        for c in torch.unique(labels[labels > 0]).tolist():
            sel = labels == c
            n_c = int(sel.sum())
            clouds = [d["pcld"][b][sel] - d["ctr_of"][b][sel]] + [d["pcld"][b][sel] - d["kp_of"][b][k][sel]
                                                                   for k in range(d["kp_of"].shape[1])]
            ms.fit_many(clouds)
            its = [int(x) for x in ms.last_iters.tolist()]
            if sweeps0 is None:
                sweeps0 = its
            pairs += float(n_c) * n_c * sum(its)
            dens_pairs += float(n_c) * n_c * (len(its) + 1)      # exact pass: centre fits twice (labels first), keypoints once
    return pairs, dens_pairs, sweeps0


def roofline_query_group(torch, _ext, dev, B, cloud, peak, peak_kind):
    """The stand-alone fused ball-query+group API (pvn3d_query_and_group2: what QueryAndGroup.forward maps to in
    the module-graph engine; the fused step gathers inside the MLP producer instead and never materialises the
    grouped tensor).  8 (level, scale) pairs of one batch with real level geometry, every call event-timed on the
    launching stream with the L2 flushed in between."""
    from pvn3d_b200.pointnet2 import SA_SPEC

    xyz = cloud[..., :3].contiguous()
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)
    total_bytes = total_ms = 0.0
    per = []
    chans = [6, 96, 256, 512]
    for li, (npoint, radii, nsamples, _) in enumerate(SA_SPEC):
        n = xyz.size(1)
        idx = _ext.furthest_point_sampling(xyz, npoint)
        new_xyz = torch.gather(xyz, 1, idx.long().unsqueeze(-1).expand(-1, -1, 3)).contiguous()
        if li == 0:
            fp, ld, cc = cloud[..., 3:].contiguous(), 6, 6
        else:
            cc = chans[li]
            fp, ld = torch.randn(B, n, cc, device=dev), cc
        ms_l = []
        for rep in range(3):
            flush.fill_(float(rep))
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            _ext.query_and_group2(xyz, new_xyz, fp, radii, nsamples, ldf=ld, c=cc, want_idx=True)
            e1.record()
            torch.cuda.synchronize(dev)
            ms_l.append(e0.elapsed_time(e1))
        ms_k = statistics.median(ms_l)
        nbytes = sum(qg_algorithmic_bytes(B, n, npoint, cc, ns) for ns in nsamples)
        per.append({"level": li + 1, "nsamples": list(nsamples), "MB": nbytes / 1e6, "us": ms_k * 1e3,
                    "GBps": nbytes / ms_k / 1e6, "frac": nbytes / ms_k / 1e6 / peak})
        total_bytes += nbytes
        total_ms += ms_k
        xyz = new_xyz
    achieved = total_bytes / total_ms / 1e6
    return {"kernel": "pvn3d_query_and_group2 = ball_scan_kernel + group_write_kernel (fused ball-query+group, both radii "
                      "of a level per call: 4 calls of one batch)",
            "on_timed_step": False, "where": "module-graph API (QueryAndGroup.forward); the fused step never writes the grouped tensor",
            "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "peak_kind": peak_kind,
            # dram bytes of the same four calls (8 kernels) from one `ncu --set full` capture (profiles/ncu_qgsplit_r01u.md,
            # kernels unchanged since): below the algorithmic bytes -- the descriptor tables are L2 hits
            "traffic": 2005.4 if B == 32 else None, "traffic_unit": "MB per batch (ncu, profiles/ncu_qgsplit_r01u.md)",
            "algorithmic_MB_per_batch": total_bytes / 1e6, "us_per_batch": total_ms * 1e3, "per_launch": per}


def heads_timing(torch, runner, dev):
    """SURVEY section 8 f3 (not part of the frame metric): DenseFusion + the three heads of PVN3D (pvn3d.py:157-182,
    245-267) on the layer kernel, random-init modules of this package's layout, random CNN embedding, the batch's
    PointNet++ features.  198.3 GFLOP per 12288-point frame as the reference executes it."""
    from pvn3d_b200 import heads as H

    b, n = runner.B, runner.cfg["n_points"]
    torch.manual_seed(0)
    mods = H.reference_layout_modules(n_classes=22, n_kps=8)
    eng = H.FusedHeads(*mods, device=dev)
    g = torch.Generator().manual_seed(1)
    rgb_emb = torch.randn(b, 128, n, generator=g).to(dev)
    cld_emb = runner.pipe.features if runner.pipe.features is not None else torch.randn(b, 128, n, generator=g).abs().to(dev)
    ms = runner.median_ms(lambda: eng(rgb_emb, cld_emb), reps=3, warm=1)
    flops = 198.3e9 * b * n / 12288
    return {"ms_per_batch": ms, "ms_per_frame": ms / b, "nominal_TFLOPs": flops / ms / 1e9,
            "what": "DenseFusion + SEG/KpOF/CtrOf heads, TF32 tensor cores; conv4 only ever averaged (32-row partial sums in the "
                    "epilogue), the broadcast global feature folded into a per-frame bias of every head's first layer (K 768 of 1792)"}


def stock_gpu_baseline(torch, runner, dev):
    """The unmodified reference on this GPU (BASELINE.md section 3.2): reference Python (staged under oracle/_ref/py)
    with its own compiled `_ext` (oracle/_ref/_ext.so): Pointnet2MSG.forward on the whole batch, and
    cal_frame_poses_lm with the reference MeanShiftTorch on CUDA tensors for ONE frame (the reference processes frames
    one at a time in a Python loop, pvn3d_eval_utils.py:373-387) scaled to the batch."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    try:
        from helpers import load_ref_ext, load_reference_python
    except Exception as e:
        return {"unavailable": f"tests/helpers.py not importable: {e!r}"}
    ref_ext = load_ref_ext()
    ref = load_reference_python()
    if ref_ext is None or ref is None:
        return {"unavailable": "oracle/_ref/_ext.so or oracle/_ref/py missing (built where /root/reference exists)"}
    from pvn3d_b200 import _ext as our_ext, testing

    d = runner.dev_rot[0]
    torch.manual_seed(0)
    model = ref.pvn3d.Pointnet2MSG(input_channels=6)
    testing.randomize_bn_(model, 1)
    model = model.to(dev).eval()
    ref.pn2_utils._ext = ref_ext
    try:
        with torch.no_grad():
            ms_a = runner.median_ms(lambda: model(d["cld_rgb_nrm"]), reps=3, warm=1)
    finally:
        ref.pn2_utils._ext = our_ext
    pcld, mask = d["pcld"][0], d["labels"][0].long()
    ctr_of, kp_of = d["ctr_of"][0][None], d["kp_of"][0]
    ref.eval_utils.cal_frame_poses_lm(pcld, mask, ctr_of, kp_of, True, 2, False, 1)       # warm
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    ref.eval_utils.cal_frame_poses_lm(pcld, mask, ctr_of, kp_of, True, 2, False, 1)
    torch.cuda.synchronize(dev)
    s_b = time.perf_counter() - t0
    B = runner.B
    ms_step = ms_a + B * s_b * 1e3
    return {"value": B / (ms_step * 1e-3), "unit": "frames/s", "ms_per_step": ms_step,
            "path_a_ms_per_batch": ms_a, "path_b_s_per_frame": s_b,
            "what": "UNMODIFIED reference: reference _ext kernels (compiled -O2 for sm_100a) + cuDNN (TF32 allowed, torch default) "
                    "under the reference Pointnet2MSG on the whole batch; reference cal_frame_poses_lm + MeanShiftTorch on CUDA "
                    "tensors, one complete frame timed (wall clock around a synchronised call) and scaled by the batch size"}


def b200_arm(args, json_out):
    import torch
    from pvn3d_b200 import _ext, _lib
    from pvn3d_b200 import dist as pdist

    rank, local_rank, world = pdist.init_from_env()
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    dev = torch.device(f"cuda:{local_rank}")
    torch.cuda.set_device(dev)
    lib = _lib.load()
    cfg = CONFIGS[args.config]
    peak, peak_kind = load_peaks()
    overlap = not args.no_overlap

    la = not args.no_lookahead
    run = Runner(torch, cfg, dev, rank, world, args.ms_mode, overlap=overlap, engine=args.engine, lookahead=la)
    head = run.measure(args.steps, args.warmup, lib, keep_outputs=bool(args.dump_outputs) and rank == 0)
    if "outputs" in head:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, arr in head.pop("outputs").items():
            np.save(os.path.join(args.dump_outputs, f"{name}.npy"), arr)
    B = run.B
    line = None
    if rank == 0:
        line = {"metric": "frames/sec", "value": head["value"], "unit": "frames/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32 (shared-MLP operands rounded to TF32, fp32 accumulate)", "data": "synthetic",
                "config": {"workload": workload_name(cfg), "n_points": cfg["n_points"], "global_batch": B * world,
                           "parallelism": (f"frame-sharded x{world}, one NCCL all_gather of poses per step" if world > 1 else "1 GPU"),
                           "l2": f"{run.n_rot} rotating device-resident input batches ({run.rot_bytes / 1e6:.0f} MB) > L2",
                           "mlp": ("tcgen05.mma kind::tf32 shared-MLP layers, grouping/interpolation fused into the operand producer"
                                   if args.engine == "fused" else "cuDNN/cuBLAS 1x1 conv (TF32 allowed, the reference's torch default)"),
                           "meanshift": {"certified": "certified (headline): returned seed + witness seeds, provably within 1e-5*bandwidth of "
                                                      "the reference's centre; iteration count not computed (include/pvn3d_b200.h)",
                                         "early_exit": "early_exit: all seeds, reference stop rule or stationary returned seed",
                                         "strict": "strict: all seeds, the reference's global stop rule (reference iteration counts)",
                                         "no_freeze": "no_freeze: literal reference schedule"}[args.ms_mode],
                           "overlap": ("hot path B on its own stream under hot path A" if overlap else "single stream")
                                      + ("; look-ahead: furthest-point sampling of batch i+1 on a high-priority third stream under "
                                         "the shared MLPs of batch i (whose first SA levels leave it one SM per frame)"
                                         if (la and overlap) else "")},
                "e2e": head["e2e"], "gpu_launches": head["gpu_launches"], "clocks": head["clocks"],
                "frames_per_s_hbm_frac": {"value": head["value"] / world / (peak * 1e9 / FRAME_HBM_BYTES),
                                          "per_gpu_roofline_frames_per_s": peak * 1e9 / FRAME_HBM_BYTES,
                                          "bytes_per_frame": FRAME_HBM_BYTES, "peak_GBps": peak, "peak_kind": peak_kind}}

    # ---- the same step in the all-seeds modes (every rank: the loops contain the collective) ---------------------
    modes = {}
    if not args.quick:
        for mode in ("early_exit", "strict"):
            if mode == args.ms_mode:
                continue
            run.set_mode(mode)
            m = run.measure(max(3, args.steps // 2), 2, lib, e2e=False, clocks=False)
            modes[mode] = {"value": m["value"], "unit": "frames/s", "ms_per_step": m["ms_per_step"]}
        run.set_mode(args.ms_mode)

    # ---- rank-0 diagnostics on the headline config (no collectives) ---------------------------------------------
    if rank == 0:
        line["meanshift_modes"] = modes
        d = run.dev_rot[0]
        ms_a = run.path_a_ms()
        ms_b = run.path_b_ms()
        line["stage_ms_per_batch"] = {"hot_path_A_pointnet2msg": ms_a, "hot_path_B_votes_to_poses": ms_b,
                                      "note": "each path alone on one stream, median of 5 warmed passes; the step overlaps them"}
        line["meanshift_ms_per_frame"] = ms_b / B
        certified = run.pipe.solver.certified_fits() if args.ms_mode == "certified" else None
        fam = None
        if run.pipe.fused is not None:
            fam = run.pipe.fused.profile(d["cld_rgb_nrm"], reps=3)
        rooflines = []
        if fam is not None:
            t_mlp = fam["mlp"]
            mlp_roof = {"kernel": "mlp_layer_kernel (all shared-MLP launches of one batch: 8 SA scales x (per-point first layer, "
                                  "gather + second layer, third layer + max-pool), 4 FP modules, the last one storing [B,128,N] directly) + factor tables",
                        "on_timed_step": True, "bound": "hbm", "achieved": MLP_IO_BYTES * B / t_mlp / 1e6, "peak": peak,
                        "unit": "GB/s", "frac": MLP_IO_BYTES * B / t_mlp / 1e6 / peak, "peak_kind": peak_kind,
                        # dram__bytes_read.sum + dram__bytes_write.sum over the 33 launches of one batch, `ncu --set full`
                        # (profiles/ncu_mlp_r02c.md): 1.5x the algorithmic bytes -- the second-layer activations
                        "traffic": 4964.1 if (B == 32 and cfg["shape"] == "linemod" and run.pipe.fused.factor) else None,
                        "traffic_unit": "MB per batch (ncu, profiles/ncu_mlp_r02c.md)",
                        "ms_per_batch": t_mlp, "algorithmic_MB_per_batch": MLP_IO_BYTES * B / 1e6,
                        "useful_TFLOPs": MLP_FLOPS * B / t_mlp / 1e9,
                        "note": "algorithmic bytes = SURVEY 8d MLP stage I/O with every SharedMLP(+max-pool) fused (100.2 MB/frame); "
                                "inter-layer activations that still round-trip HBM are NOT counted as useful"}
            rooflines.append(mlp_roof)
            n_iter = sum(s[0] for s in __import__("pvn3d_b200.pointnet2", fromlist=["SA_SPEC"]).SA_SPEC)
            rooflines.append({"kernel": "fps_regs_kernel (4 levels)", "on_timed_step": True, "bound": "latency",
                              "ms_per_batch": fam["fps"], "us_per_iteration": fam["fps"] * 1e3 / n_iter,
                              "iterations": n_iter, "note": "dependent arg-max iterations, one CTA per frame"})
            rooflines.append({"kernel": "ball_scan_kernel (4 levels, both radii per pass)", "on_timed_step": True,
                              "bound": "issue", "ms_per_batch": fam["ball"]})
            rooflines.append({"kernel": "three_nn_kernel + nn_weights_kernel (4 levels)", "on_timed_step": True,
                              "bound": "issue", "ms_per_batch": fam["three_nn"]})
            rooflines.append({"kernel": "glue (xyz split, new_xyz gathers)", "on_timed_step": True,
                              "ms_per_batch": fam["glue"]})
            line["roofline"] = mlp_roof
        # mean-shift: pair evaluations per second against the MUFU bound
        if not args.quick:
            pairs, dens_pairs, sweeps0 = meanshift_work(torch, run)
            run.set_mode("strict")
            ms_b_strict = run.path_b_ms()
            run.set_mode("early_exit")
            ms_b_early = run.path_b_ms()
            run.set_mode(args.ms_mode)
            sm_clock = (head["clocks"] or {}).get("sm_mhz") or 1965.0
            mufu_peak = 148 * 16 * sm_clock * 1e6
            rooflines.append({"kernel": "ms_iterate_kernel + ms_density_kernel, strict mode (all seeds, reference iteration counts)",
                              "on_timed_step": args.ms_mode == "strict", "bound": "mufu (16 ex2/clk/SM)",
                              "pair_evaluations_per_batch": pairs, "ms_per_batch_path_b": ms_b_strict,
                              "achieved_pairs_per_s": pairs / (ms_b_strict * 1e-3), "peak_pairs_per_s": mufu_peak,
                              "frac": pairs / (ms_b_strict * 1e-3) / mufu_peak,
                              "note": "whole path B time as the denominator (density pass, compaction, Kabsch included)"})
            line["meanshift_path_b_ms_per_batch"] = {"certified" if args.ms_mode == "certified" else args.ms_mode: ms_b,
                                                     "early_exit": ms_b_early, "strict": ms_b_strict}
            line["meanshift_sweeps_frame0"] = sweeps0
            line["meanshift_reference_sweeps_frame0"] = reference_sweep_counts()[0] if cfg["shape"] == "linemod" else None
        if certified is not None:
            nf = B * (run.pipe.n_cls - 1 if cfg["shape"] == "linemod" else run.pipe.n_cls) * (run.pipe.k + 1)
            line["meanshift_certified_fits"] = {"certified": certified, "launched": nf,
                                                "note": "fits closed by the witness kernel in the last launch (absent classes are empty fits)"}
        if not args.quick:
            rooflines.append(roofline_query_group(torch, _ext, dev, B, d["cld_rgb_nrm"], peak, peak_kind))
        line["rooflines"] = rooflines
        if "roofline" not in line:
            line["roofline"] = rooflines[-1] if rooflines else None

    # ---- the other BASELINE configs (every rank; frames sharded, same collective) -------------------------------
    if not args.quick and args.config == "linemod":
        subs = {}
        del run
        torch.cuda.empty_cache()
        r2 = Runner(torch, CONFIGS["ycb"], dev, rank, world, args.ms_mode, overlap=overlap, engine=args.engine, n_rot=4,
                    lookahead=la)
        m = r2.measure(max(5, args.steps // 2), 3, lib)
        key = f"ycb_b{CONFIGS['ycb']['batch']}" if world == 1 else f"ycb_b{CONFIGS['ycb']['batch'] * world}_sharded_x{world}"
        if rank == 0:
            m["workload"] = workload_name(CONFIGS["ycb"]) + (f", {world} GPUs" if world > 1 else "")
            m["path_b_ms_per_batch"] = r2.path_b_ms()
            m["meanshift_ms_per_frame"] = m["path_b_ms_per_batch"] / r2.B
            m["certified_fits"] = r2.pipe.solver.certified_fits() if args.ms_mode == "certified" else None
            r2.set_mode("strict")
            m["path_b_ms_per_batch_strict"] = r2.path_b_ms()
            if world == 1 and not args.no_cpu_baseline:
                m["cpu_meanshift"] = cpu_pose_path_ycb(r2.frames[0], m["meanshift_ms_per_frame"])
            subs[key] = m
        del r2
        torch.cuda.empty_cache()
        r3 = Runner(torch, CONFIGS["stress"], dev, rank, world, args.ms_mode, overlap=overlap, engine=args.engine, n_rot=2,
                    lookahead=la)
        m = r3.measure(max(3, args.steps // 4), 3, lib, e2e=True)
        if rank == 0:
            m["workload"] = workload_name(CONFIGS["stress"]) + (f", {world} GPUs" if world > 1 else "")
            m["path_a_ms_per_batch"] = r3.path_a_ms()
            sweep = {}
            for bw in (0.02, 0.04, 0.08, 0.16):
                r3.set_mode(args.ms_mode, bandwidth=bw)
                t_c = r3.path_b_ms()
                r3.set_mode("strict", bandwidth=bw)
                t_s = r3.path_b_ms()
                sweep[f"bw{bw}"] = {"meanshift_ms_per_frame": t_c / r3.B, "meanshift_ms_per_frame_strict": t_s / r3.B}
            m["bandwidth_sweep_path_b"] = sweep
            subs["stress_49152"] = m
        del r3
        torch.cuda.empty_cache()
        if rank == 0:
            line["configs"] = subs

    # ---- baselines timed beside it (rank 0, single GPU) ----------------------------------------------------------
    if rank == 0:
        if world == 1 and not args.no_cpu_baseline and not args.quick:
            from pvn3d_b200 import synth, testing
            c = CONFIGS["linemod"]
            frame = synth.make_batch(c["shape"], 1, n_points=c["n_points"], config_id=c["config_id"], lm_obj_id=1)[0]
            sd = testing.seeded_pointnet2msg(0, 1).state_dict()
            sec, desc, info = cpu_path_sample(frame, sd, sweep_budget_s=20.0, complete_fit=True)
            line["cpu_baseline"] = {"value": 1.0 / sec, "unit": "frames/s", "cores": os.cpu_count() or 1, "kind": "port",
                                    "sample": desc, "detail": info}
            try:
                rs = Runner(torch, CONFIGS["linemod"], dev, rank, 1, args.ms_mode, overlap=overlap, n_rot=1)
                line["stock_gpu_baseline"] = stock_gpu_baseline(torch, rs, dev)
                rs.step_device(0)
                line["densefusion_heads"] = heads_timing(torch, rs, dev)
                del rs
            except Exception as e:           # the stock leg must never take the bench line down
                line["stock_gpu_baseline"] = {"unavailable": repr(e)[:300]}
        else:
            line["cpu_baseline"] = None
        json_out.write(json.dumps(line) + "\n")
        json_out.flush()
    if world > 1:
        torch.distributed.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10,
                    help="timed steps K of the headline loop (the frames/s value and e2e); without --quick the other "
                         "loops run max(3, K/2) steps (other mean-shift modes), max(5, K/2) (YCB) and max(3, K/4) (stress)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="linemod", choices=["linemod", "ycb"])
    ap.add_argument("--ms-mode", default="certified", choices=["certified", "early_exit", "strict", "no_freeze"])
    ap.add_argument("--no-overlap", action="store_true", help="run hot path B after hot path A on one stream")
    ap.add_argument("--no-lookahead", action="store_true",
                    help="do not compute the next batch's geometry plan under this batch's MLPs")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--quick", action="store_true", help="headline + stage split only (development runs, ncu)")
    ap.add_argument("--engine", default="fused", choices=["fused", "modules"],
                    help="hot path A: fused tcgen05 engine (default) or module graph with cuDNN/cuBLAS MLPs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed (rank 0) as DIR/<name>.npy, float32: poses, present "
                         "and a fixed seeded sample of 1024 points of the [B,128,N] features (16 MB at batch 32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the GPU path: it needs --impl b200")
    # stdout carries exactly ONE line (the JSON): everything any library prints to fd 1 from here on
    # (NCCL prints its version there) goes to stderr; the JSON is written to the saved descriptor
    sys.stdout.flush()
    json_out = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    args.warmup = max(args.warmup, 5 if args.impl == "b200" else 0)   # the first steps of a loop grow the allocator pools
    if args.impl == "reference":
        rank = int(os.environ.get("RANK", "0"))
        return reference_arm(args, json_out, rank)
    return b200_arm(args, json_out)


if __name__ == "__main__":
    sys.exit(main())
