#!/usr/bin/env python
"""bench.py — headline benchmark of the hot path (BASELINE.json): pose-hypotheses/sec of one
FoundationPose `register` hot loop — 252 hypotheses x 5 refine iterations + scoring + arg-max — on a
synthetic 640x480 RGB-D frame and a random-textured 20 480-triangle mesh, random-init weights of the
reference architectures.

    python bench.py --gpus 1 --steps 10 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      # the reference networks on the host CPU cores
    python bench.py --impl torch-cuda ...     # GPU STAND-IN for the reference's CUDA build (not the reference arm):
                                              # the oracle port of its networks on CUDA under fp16 autocast
    python bench.py --gpus 1 --steps 10 --warmup 3 --dump-outputs DIR   # + what the last timed step returned, as .npy

A step = one pass of the hot path over one frame.  `value` = hypotheses / step time with the frame,
mesh and weights resident in HBM (device-timed with CUDA events, max over ranks); `e2e` = the same
metric through the public API `FoundationPose.register()` with HOST numpy buffers (frame upload, the
depth read-back for the translation guess, pose upload and result read-back inside the timed region).
At N > 1 the 252 hypotheses are sharded over the ranks (BASELINE.json configs[3]) with one NCCL
all-gather of per-hypothesis features before the replicated cross-hypothesis attention: "strong".
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_HYP = 252
N_ITER = 5
GFLOP_REFINE = 23.946  # per hypothesis per refine iteration (BASELINE.md §2)
GFLOP_SCORE = 21.94  # per hypothesis scored
METRIC = "pose-hypotheses/sec at 640x480 RGB-D, 252 hyp, 5 refine iters"


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            p = json.load(fh)
        return dict(hbm_gbs=p["hbm_gbs"], tf_burst=p["bf16_tflops"], tf_sustained=p["bf16_tflops_sustained"], source="measured")
    except Exception:
        return dict(hbm_gbs=6650.0, tf_burst=1590.0, tf_sustained=1400.0, source="fallback")


class ClockSampler:
    """SM clock / throttle-reason sampling during the timed region (B200_PROFILING.md): NVML every 20 ms when
    nvidia-ml-py is importable (an nvidia-smi process per sample is too slow for a 0.3 s loop), else nvidia-smi."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.rows = []  # (sm_mhz, max_mhz, {reasons})
        self._stop = threading.Event()
        self._t = threading.Thread(target=self._run, daemon=True)
        self._nvml = None
        try:
            import pynvml

            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[index]) if vis and all(x.strip().isdigit() for x in vis.split(",")) else index
            self._h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self._nvml = pynvml
        except Exception:
            self._nvml = None

    def _sample_nvml(self):
        n = self._nvml
        sm = n.nvmlDeviceGetClockInfo(self._h, n.NVML_CLOCK_SM)
        mx = n.nvmlDeviceGetMaxClockInfo(self._h, n.NVML_CLOCK_SM)
        bits = n.nvmlDeviceGetCurrentClocksThrottleReasons(self._h)
        names = set()
        for name, const in (("hw_slowdown", "nvmlClocksThrottleReasonHwSlowdown"), ("hw_thermal_slowdown", "nvmlClocksThrottleReasonHwThermalSlowdown"),
                            ("sw_thermal_slowdown", "nvmlClocksThrottleReasonSwThermalSlowdown"), ("sw_power_cap", "nvmlClocksThrottleReasonSwPowerCap")):
            if bits & getattr(n, const, 0):
                names.add(name)
        self.rows.append((float(sm), float(mx), names))

    def _sample_smi(self):
        out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=5).stdout.strip()
        if out:
            r = [x.strip() for x in out.split(",")]
            names = {nm for nm, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]) if v.lower().startswith("active")}
            self.rows.append((float(r[0]), float(r[1]), names))

    def _run(self):
        while not self._stop.is_set():
            try:
                self._sample_nvml() if self._nvml else self._sample_smi()
            except Exception:
                pass
            self._stop.wait(0.02 if self._nvml else 0.2)

    def __enter__(self):
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=5)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        reasons = set().union(*[r[2] for r in self.rows])
        return {"sm_mhz": float(np.median([r[0] for r in self.rows])), "sm_max_mhz": float(max(r[1] for r in self.rows)),
                "reasons": sorted(reasons), "samples": len(self.rows), "source": "nvml" if self._nvml else "nvidia-smi"}


def physical_cores_one_socket():
    """Physical cores of socket 0 (from /proc/cpuinfo); falls back to os.cpu_count()."""
    try:
        cores, phys, cur = set(), None, {}
        for line in open("/proc/cpuinfo"):
            if ":" in line:
                k, v = [x.strip() for x in line.split(":", 1)]
                cur[k] = v
            elif cur:
                if cur.get("physical id", "0") == "0":
                    cores.add(cur.get("core id", cur.get("processor")))
                cur = {}
        if cur and cur.get("physical id", "0") == "0":
            cores.add(cur.get("core id", cur.get("processor")))
        return max(1, len(cores))
    except Exception:
        return os.cpu_count() or 1


def pick_cpu_threads(fn):
    """torch's intra-op pool oversubscribes badly on many-core hosts for these small batches, and crossing sockets or
    using SMT siblings makes it worse (round 1: 128 threads on the 8-GPU box gave the slowest result).  Fixed candidate
    set capped at the physical cores of ONE socket; per candidate 2 warm-ups, then the median of 3 timed calls; the
    fastest wins.  Returns (threads, seconds per call)."""
    cap = min(physical_cores_one_socket(), os.cpu_count() or 1)
    cands = sorted({c for c in (8, 16, 32, cap) if c <= cap}) or [cap]
    best = (None, float("inf"))
    for c in cands:
        torch.set_num_threads(c)
        fn()
        fn()
        ts = []
        for _ in range(3):
            t0 = time.perf_counter()
            fn()
            ts.append(time.perf_counter() - t0)
        dt = sorted(ts)[1]
        if dt < best[1]:
            best = (c, dt)
    torch.set_num_threads(best[0])
    return best


def cpu_nets_rate(budget_s=20.0):
    """The reference networks (oracle port of RefineNet / ScoreNetMultiPair, fp32, torch CPU, all host
    threads) on pre-built crops: hypotheses/sec of a 5-iteration register, extrapolated from a bounded
    sample.  Returns (hyp_per_s, cores, sample description)."""
    from foundationpose_b200.weights import random_state_dict
    from oracle import nets

    sd_r, sd_s = random_state_dict("refine", 0), random_state_dict("score", 0)
    g = torch.Generator().manual_seed(0)
    n = 4
    A, B = torch.rand(n, 6, 160, 160, generator=g), torch.rand(n, 6, 160, 160, generator=g)
    cores, t_probe = pick_cpu_threads(lambda: nets.refine_forward(sd_r, A, B))
    t_probe /= n
    n = int(max(4, min(64, budget_s / (2.0 * max(t_probe, 1e-3)))))
    A, B = torch.rand(n, 6, 160, 160, generator=g), torch.rand(n, 6, 160, 160, generator=g)
    t0 = time.perf_counter()
    nets.refine_forward(sd_r, A, B)
    t_ref = (time.perf_counter() - t0) / n
    t0 = time.perf_counter()
    nets.score_forward(sd_s, A, B, L=n)
    t_sc = (time.perf_counter() - t0) / n
    rate = 1.0 / (N_ITER * t_ref + t_sc)
    return rate, cores, (f"RefineNet + ScoreNetMultiPair (oracle port, fp32 torch CPU, {cores} threads = best of 8/16/32/one socket's physical cores) on {n} pre-built 160x160 crop pairs; "
                         f"{t_ref * 1e3:.1f} ms/hyp-iter refine, {t_sc * 1e3:.1f} ms/hyp score; extrapolated to {N_ITER} iters + 1 score; raster/warp not included")


def dump_outputs(out_dir, poses, scores, best):
    """The arrays ShardedRegister.run hands its caller, as float32 / float64 .npy files (12 KB in all at 252 hypotheses)."""
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "poses.npy"), poses.detach().float().cpu().numpy())      # (252, 4, 4) refined poses
    np.save(os.path.join(out_dir, "scores.npy"), scores.detach().float().cpu().numpy())    # (252,) scorer logits + 100
    np.save(os.path.join(out_dir, "best.npy"), np.asarray(int(best.item()), dtype=np.float64))  # index of the selected pose


_REAL_STDOUT = None


def claim_stdout():
    """Keep fd 1 for the ONE JSON line: everything else that writes to stdout (NCCL's version banner comes from C
    code and ignores NCCL_DEBUG_FILE on some boxes) is sent to stderr."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    sys.stdout.flush()
    os.write(_REAL_STDOUT if _REAL_STDOUT is not None else 1, (json.dumps(line) + "\n").encode())


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path (its own networks; the
    raster/warp stage has no CPU implementation in the reference) on the host cores."""
    if rank != 0:
        return
    from foundationpose_b200.weights import random_state_dict
    from oracle import nets

    sd_r, sd_s = random_state_dict("refine", 0), random_state_dict("score", 0)
    g = torch.Generator().manual_seed(0)
    A1, B1 = torch.rand(4, 6, 160, 160, generator=g), torch.rand(4, 6, 160, 160, generator=g)
    cores, t_pass = pick_cpu_threads(lambda: nets.refine_forward(sd_r, A1, B1))
    t_pass /= 4
    # bounded sample per step: ~4 s of CPU work (6 network passes per hypothesis)
    n = int(max(1, min(16, 4.0 / (6 * max(t_pass, 1e-3)))))
    A, B = torch.rand(n, 6, 160, 160, generator=g), torch.rand(n, 6, 160, 160, generator=g)

    def step():
        for _ in range(N_ITER):
            nets.refine_forward(sd_r, A, B)
        nets.score_forward(sd_s, A, B, L=n)

    for _ in range(min(args.warmup, 1)):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = (time.perf_counter() - t0) / args.steps
    value = n / dt
    sample = (f"{n} hypotheses per step through RefineNet x{N_ITER} + ScoreNetMultiPair (oracle port of the reference modules, fp32 torch CPU, "
              f"{cores} threads) on pre-built 160x160 crops; the reference has no CPU raster/warp")
    emit({
        "impl": "reference", "metric": METRIC, "value": value, "unit": "hyp/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": "register: 252 hyp x 5 refine iters + score, 640x480 RGB-D (CPU arm: bounded sample of the same networks)",
                   "hypotheses_per_step": n},
        "cpu_baseline": {"value": value, "unit": "hyp/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "hyp/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    })


def load_traffic():
    """DRAM bytes per launch of the roofline kernels, measured by `ncu --set full` and committed by
    tools/ncu_summary.py as profiles/r02_ncu_traffic.json (kernel-name prefix -> dram read + write bytes of ONE launch)."""
    try:
        with open(os.path.join(ROOT, "profiles", "r02_ncu_traffic.json")) as fh:
            return json.load(fh)
    except Exception:
        return {}


class TorchCudaStandin:
    """GPU STAND-IN for the reference's nvdiffrast + PyTorch CUDA build, which cannot be installed here (SURVEY.md §8d
    last row): the oracle port of the reference networks as plain torch ops on CUDA under fp16 autocast with
    cudnn.benchmark = False / deterministic = True (what register()'s set_seed(0) leaves, Utils.py:222-229), fed with
    crops from THIS repository's producer because nvdiffrast / kornia are absent.  Clearly a stand-in: it is never the
    `--impl reference` arm."""

    def __init__(self, eng, sd_r, sd_s, diameter):
        from oracle import geometry, nets

        self.eng, self.nets, self.geometry, self.d = eng, nets, geometry, diameter
        self.sd_r = {k: v.cuda() for k, v in sd_r.items()}
        self.sd_s = {k: v.cuda() for k, v in sd_s.items()}
        torch.backends.cudnn.benchmark = False
        torch.backends.cudnn.deterministic = True

    def crops(self, poses, mode):
        _, dbg, _ = self.eng.make_crops(poses, mode=mode, want_crops=False, want_dbg=True)
        A = dbg[:, 0].permute(0, 3, 1, 2).contiguous()
        B = dbg[:, 1].permute(0, 3, 1, 2).contiguous()
        return A, B

    def refine_once(self, poses, autocast=True):
        A, B = self.crops(poses, 0)
        with torch.autocast("cuda", dtype=torch.float16, enabled=autocast):
            out = self.nets.refine_forward(self.sd_r, A, B)
        return self.geometry.pose_update(poses, out["trans"].float(), out["rot"].float(), self.d, 0.3490658503988659)

    def step(self, poses, iters, autocast=True):
        for _ in range(iters):
            poses, _, _ = self.refine_once(poses, autocast)
        A, B = self.crops(poses, 1)
        with torch.autocast("cuda", dtype=torch.float16, enabled=autocast):
            logits = self.nets.score_forward(self.sd_s, A, B, L=len(A)).reshape(-1).float()
        return poses, logits + 100


def run_torch_cuda(args, rank, world):
    """--impl torch-cuda: the stand-in alone, same metric / config, one JSON line with "impl": "torch-cuda"."""
    if rank != 0:
        return
    from foundationpose_b200 import hypotheses, synth
    from foundationpose_b200.engine import Engine
    from foundationpose_b200.estimater import make_mesh_tensors
    from foundationpose_b200.weights import random_state_dict

    torch.cuda.set_device(0)
    mesh, gt_pose, K, rgb, depth, mask = synth.default_scene(subdivisions=5, seed=0)
    mt = make_mesh_tensors(mesh)
    d = synth.mesh_diameter(mesh.vertices)
    eng = Engine()
    eng.set_mesh(mt["pos"], mt["normals"], mt["faces"], d, uv=mt["uv"], tex=mt["tex"])
    eng.set_frame(torch.from_numpy(rgb).cuda(), torch.from_numpy(depth).cuda(), K, filter_depth=True)
    center = hypotheses.guess_translation(eng.get_depth()[0].cpu().numpy(), mask, K)
    poses0 = torch.from_numpy(hypotheses.make_rotation_grid()).float().cuda()
    poses0[:, :3, 3] = torch.as_tensor(center, dtype=torch.float32, device="cuda")
    st = TorchCudaStandin(eng, random_state_dict("refine", 0), random_state_dict("score", 0), d)
    with torch.inference_mode():
        for _ in range(max(1, min(args.warmup, 2))):
            st.step(poses0, N_ITER)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            _, scores = st.step(poses0, N_ITER)
        e1.record()
        torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / args.steps
    emit({"impl": "torch-cuda", "metric": METRIC, "value": N_HYP / (ms * 1e-3), "unit": "hyp/s", "n_gpus": 1, "steps": args.steps,
          "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f16",
          "data": "synthetic", "best_index": int(scores.argmax().item()),
          "config": {"workload": "register: 252 hyp x 5 refine iters + score; GPU STAND-IN for the reference's CUDA build: oracle port of its "
                                 "networks as torch ops on CUDA, fp16 autocast, cudnn.benchmark=False; crops from this repository's producer "
                                 "(nvdiffrast / kornia are not installable here)"}})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference", "torch-cuda"])
    ap.add_argument("--no-standin", action="store_true", help="skip the torch-cuda stand-in / parity legs of the native line")
    ap.add_argument("--no-track", action="store_true", help="skip the track_one (BASELINE.json configs[2]) leg")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned (refined poses, scores, best index) to DIR/<name>.npy; "
                         "the inputs are seeded, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "native":
        ap.error("--dump-outputs applies to the native path only")
    args.warmup = max(args.warmup, 3) if args.impl == "native" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    claim_stdout()

    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if args.impl == "torch-cuda":
        run_torch_cuda(args, rank, world)
        return

    import torch.distributed as dist

    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # keep stdout for the ONE JSON line: NCCL's version / debug banner goes to stderr
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    from foundationpose_b200 import _lib, hypotheses, synth
    from foundationpose_b200.engine import Engine
    from foundationpose_b200.estimater import FoundationPose, PoseRefinePredictor, ScorePredictor
    from foundationpose_b200.parallel import ShardedRegister
    from foundationpose_b200.weights import random_state_dict

    peaks = load_peaks()
    # ---------------------------------------------------------------- synthetic workload (SURVEY.md §8d)
    mesh, gt_pose, K, rgb, depth, mask = synth.default_scene(subdivisions=5, seed=0)
    eng = Engine()
    refiner = PoseRefinePredictor(engine=eng, state_dict=random_state_dict("refine", 0))
    scorer = ScorePredictor(engine=eng, state_dict=random_state_dict("score", 0))
    est = FoundationPose(model_pts=mesh.vertices, model_normals=mesh.vertex_normals, mesh=mesh, scorer=scorer, refiner=refiner)
    sharded = ShardedRegister(eng)

    # device-resident inputs for `value`
    eng.set_frame(torch.from_numpy(rgb).cuda(), torch.from_numpy(depth).cuda(), K, filter_depth=True)
    d_f, _ = eng.get_depth()
    center = hypotheses.guess_translation(d_f.cpu().numpy(), mask, K)
    poses0 = est.rot_grid.clone()
    poses0[:, :3, 3] = torch.as_tensor(center, dtype=torch.float32, device="cuda")
    assert poses0.shape[0] == N_HYP

    def step_device():
        return sharded.run(poses0, N_ITER)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------------------------------------------------------- e2e through the public API (host buffers)
    rgb_h = np.ascontiguousarray(rgb)
    depth_h = np.ascontiguousarray(depth)

    def step_e2e():
        if world == 1:
            return est.register(K=K, rgb=rgb_h, depth=depth_h, ob_mask=mask, iteration=N_ITER)
        # sharded register: every rank uploads the frame and the mask, derives the start poses on the device,
        # refines its slice; one all-gather; same result everywhere
        eng.set_frame(rgb_h, depth_h, K, filter_depth=True)
        p, info = eng.start_poses(mask, est.rot_grid)
        po, sc, b = sharded.run(p, N_ITER)
        return (po[int(b.item())] @ est.get_tf_to_centered_mesh()).cpu().numpy()

    def time_e2e():
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            step_e2e()
        barrier()
        dt = (time.perf_counter() - t0) / args.steps * 1e3
        if world > 1:
            t = torch.tensor([dt], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        return dt

    # The GPU runs under its power cap for the whole benchmark and its clock sinks while the die heats up, so whichever
    # of the two measurements runs second looks slower.  Order: warm-up (both paths, graphs captured) -> e2e loop ->
    # device loop (`value`) -> e2e loop again; `e2e` is the mean of the two e2e loops, which brackets `value` in time.
    for _ in range(args.warmup):
        step_device()
    for _ in range(2):
        step_e2e()
    e2e_before = time_e2e()
    for _ in range(args.warmup):
        step_device()
    barrier()
    launches0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as clk:
        barrier()
        e0.record()
        for _ in range(args.steps):
            poses_out, scores, best = step_device()
        e1.record()
        barrier()
    ms = e0.elapsed_time(e1) / args.steps
    launches = (_lib.launch_count() - launches0) // args.steps
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, poses_out, scores, best)
    if world > 1:
        t = torch.tensor([ms], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item())
    value = N_HYP / (ms * 1e-3)
    for _ in range(2):
        step_e2e()
    e2e_after = time_e2e()
    e2e_ms = 0.5 * (e2e_before + e2e_after)
    # per step and rank: frame + mask up; (tx, ty, tz, n_valid) and the best pose down
    h2d = rgb_h.nbytes + depth_h.nbytes + mask.nbytes
    d2h = 16 + 64

    # ---------------------------------------------------------------- roofline of the dominant kernel (dedicated pass)
    _lib.prof_enable(True)
    for _ in range(2):
        step_device()
    g_ms, g_flops, g_n = _lib.prof_collect(0)
    c_ms, c_bytes, c_n = _lib.prof_collect(1)
    _lib.prof_enable(False)
    tf_ach = g_flops / (g_ms * 1e-3) / 1e12 if g_ms > 0 else 0.0
    gb_ach = c_bytes / (c_ms * 1e-3) / 1e9 if c_ms > 0 else 0.0
    roofline = {"kernel": "tcgen05 implicit-GEMM kernels: gemm_tile_kernel<BN,CG,SLABS,PATCH>, gemm_swap(_patch)_kernel, stem_conv_kernel (15 conv + linear layers)", "bound": "tensor",
                "achieved": tf_ach, "peak": peaks["tf_sustained"], "unit": "TFLOP/s", "frac": tf_ach / peaks["tf_sustained"],
                "peak_source": f"MEASURED_PEAKS.json bf16_tflops_sustained ({peaks['source']}); kernel timed inside a long step",
                "launches_timed": g_n, "avg_launch_ms": g_ms / max(g_n, 1), "share_of_step": (g_ms / 2) / ms,
                "traffic": None}
    traffic = load_traffic()  # measured by ncu --set full, committed under profiles/ (never a literal in this file)
    tg = traffic.get("gemm_tile_kernel")
    if tg:
        roofline["traffic"] = tg["dram_bytes"]
        roofline["traffic_note"] = (f"dram read+write of ONE launch of {tg['kernel']} ({tg.get('what', '')}) from {tg['source']}; "
                                    f"algorithmic bytes of that launch: {tg.get('algorithmic_bytes')}")
    roofline_raster = {"kernel": "crop producer: crop_tile_kernel<TILE> (meshlet binning + raster + shade + warp + normalise, one launch per pass)",
                       "bound": "hbm", "achieved": gb_ach, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": gb_ach / peaks["hbm_gbs"],
                       "launches_timed": c_n, "avg_launch_ms": c_ms / max(c_n, 1), "share_of_step": (c_ms / 2) / ms, "traffic": None}
    tc = traffic.get("crop_tile_kernel")
    if tc:
        roofline_raster["traffic"] = tc["dram_bytes"]
        roofline_raster["traffic_note"] = f"dram read+write of ONE launch at N = {tc.get('n_hyp')} from {tc['source']}; algorithmic bytes: {tc.get('algorithmic_bytes')}"
        if tc.get("issue_active_pct") is not None:
            roofline_raster["issue_active_pct"] = tc["issue_active_pct"]

    # ---------------------------------------------------------------- ranking margin of this run (SURVEY.md §7 hard part v)
    sc_sorted = torch.sort(scores.float(), descending=True).values
    top2_margin = float((sc_sorted[0] - sc_sorted[1]).item())
    score_spread = float(scores.float().std().item())

    # ---------------------------------------------------------------- track_one leg (BASELINE.json configs[2]), rank 0, N = 1
    track = None
    if rank == 0 and world == 1 and not args.no_track:
        seq = synth.track_sequence(20, gt_pose)
        frames = [synth.make_scene(mesh.visual.image, p_, seed=1 + i)[:2] for i, p_ in enumerate(seq)]
        est.register(K=K, rgb=frames[0][0], depth=frames[0][1], ob_mask=mask, iteration=N_ITER)
        n_frames = 1000
        for i in range(20):
            est.track_one(rgb=frames[i % 20][0], depth=frames[i % 20][1], K=K, iteration=2)
        lat = []
        for i in range(n_frames):
            k40 = i % 40
            f_rgb, f_depth = frames[k40 if k40 < 20 else 39 - k40]  # forwards, then backwards: no jumps
            t0 = time.perf_counter()
            est.track_one(rgb=f_rgb, depth=f_depth, K=K, iteration=2)
            lat.append((time.perf_counter() - t0) * 1e3)
        lat = np.sort(np.asarray(lat))
        track = {"ms_p50": float(lat[len(lat) // 2]), "ms_p99": float(lat[int(len(lat) * 0.99)]), "ms_mean": float(lat.mean()),
                 "frames": n_frames, "refine_iters": 2, "hypotheses": 1,
                 "api": "FoundationPose.track_one(rgb, depth, K, iteration=2) with host numpy frames (one CUDA-graph launch per frame: upload, "
                        "depth filters, xyz map, 2 refiner passes, pose read-back); wall clock per call",
                 "sequence": "20 distinct synthetic frames (object moving <= 5 mm / 2 deg per frame) played forwards and backwards 25 times"}

    # ---------------------------------------------------------------- GPU stand-in + parity numbers (rank 0, N = 1)
    standin = parity = None
    if rank == 0 and world == 1 and not args.no_standin:
        try:
            eng.set_frame(torch.from_numpy(rgb).cuda(), torch.from_numpy(depth).cuda(), K, filter_depth=True)
            st = TorchCudaStandin(eng, random_state_dict("refine", 0), random_state_dict("score", 0), est.diameter)
            with torch.inference_mode():
                st.step(poses0, N_ITER)
                torch.cuda.synchronize()
                s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s0.record()
                for _ in range(3):
                    _, st_scores = st.step(poses0, N_ITER)
                s1.record()
                torch.cuda.synchronize()
                st_ms = s0.elapsed_time(s1) / 3
                # parity of the first refine iteration's SE(3) deltas on the 252 start poses, same crops for all three
                torch.backends.cuda.matmul.allow_tf32 = False
                torch.backends.cudnn.allow_tf32 = False
                _, t32, r32 = st.refine_once(poses0, autocast=False)
                _, t16, r16 = st.refine_once(poses0, autocast=True)
                _, tn, rn = eng.refine(poses0, 1)
            standin = {"value": N_HYP / (st_ms * 1e-3), "unit": "hyp/s", "ms_per_step": st_ms, "best_index": int(st_scores.argmax().item()),
                       "what": "GPU STAND-IN for the reference's nvdiffrast + PyTorch CUDA build (not installable here): oracle port of its "
                               "networks as torch ops on CUDA, fp16 autocast, cudnn.benchmark=False, crops from this repository's producer; "
                               "NOT the --impl reference arm"}
            parity = {"what": "first refine iteration on the 252 start poses: max |delta| difference of the predicted SE(3) update "
                              "(translation in metres / rotation-matrix entries); fp32 oracle = the reference networks as fp32 torch ops on the same crops",
                      "native_vs_fp32_oracle": {"trans": float((tn - t32).abs().max()), "rot": float((rn - r32).abs().max())},
                      "autocast_oracle_vs_fp32_oracle": {"trans": float((t16 - t32).abs().max()), "rot": float((r16 - r32).abs().max())},
                      "native_vs_autocast_oracle": {"trans": float((tn - t16).abs().max()), "rot": float((rn - r16).abs().max())}}
        except Exception as ex:
            standin = {"value": None, "what": f"stand-in failed: {ex}"}

    # ---------------------------------------------------------------- CPU baseline (rank 0, N = 1 only)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            rate, cores, sample = cpu_nets_rate()
            cpu = {"value": rate, "unit": "hyp/s", "cores": cores, "kind": "port", "sample": sample}
        except Exception as ex:  # the oracle is test infrastructure; never let it break the bench line
            cpu = {"value": None, "unit": "hyp/s", "cores": os.cpu_count(), "kind": "port", "sample": f"failed: {ex}"}

    if rank == 0:
        flops_step = N_HYP * (N_ITER * GFLOP_REFINE + GFLOP_SCORE) * 1e9
        line = {
            "metric": METRIC, "value": value, "unit": "hyp/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f16",
            "data": "synthetic",
            "config": {"workload": "model-based register (BASELINE.json configs[1]; configs[3] sharding at N>1): icosphere-5 ellipsoid mesh "
                                   "(10242 v / 20480 f, 1024^2 texture), 640x480 synthetic RGB-D, 252 hyp, 5 refine iters + score + argmax",
                       "hypotheses": N_HYP, "refine_iters": N_ITER, "parallelism": f"hyp-shard x{world}",
                       "weights": "seeded random init of RefineNet/ScoreNetMultiPair (no checkpoints offline)",
                       "l2": "working set per step ~3.5 GB of activations >> 126 MB L2 (no flush needed)"},
            "whole_path_tflops": flops_step / (ms * 1e-3) / 1e12,
            "e2e": {"value": N_HYP / (e2e_ms * 1e-3), "unit": "hyp/s", "ms_per_step": e2e_ms, "h2d_bytes_per_step": int(h2d),
                    "d2h_bytes_per_step": int(d2h), "api": "FoundationPose.register(K, rgb, depth, ob_mask, iteration=5) with host numpy buffers",
                    "ms_per_step_before_value_loop": e2e_before, "ms_per_step_after_value_loop": e2e_after,
                    "note": "mean of two timed loops of `steps` calls, one before and one after the device-timed loop (the power-capped clock drifts while the die heats up)"},
            "gpu_launches": int(launches),
            "clocks": clk.summary(),
            "roofline": roofline,
            "roofline_raster": roofline_raster,
            "best_index": int(best.item()),
            "top2_margin": top2_margin,
            "score_spread": score_spread,
        }
        if track is not None:
            line["track_one"] = track
        if standin is not None:
            line["gpu_standin"] = standin
        if parity is not None:
            line["parity"] = parity
        if cpu is not None:
            line["cpu_baseline"] = cpu
        emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
