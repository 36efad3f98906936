#!/usr/bin/env python
"""bench.py -- BA iterations/sec and tracks-triangulated/sec at 400 frames x 4096 tracks (BASELINE.json).

    python bench.py --gpus 1 --steps 5 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference --steps 2 --warmup 1      # CPU arm (oracle port of the reference's BA)

One "step" = one bundle-adjustment solve of ITERS Levenberg-Marquardt iterations (residual/Jacobian ->
Schur -> Cholesky -> back-substitution -> candidate evaluation -> accept/reject) on configuration C3
(400 x 4096, SIMPLE_RADIAL, shared camera), starting from the same perturbed state every step.
value = steps*ITERS / seconds.  Tracks/s of the fused LORANSAC triangulation is timed in a second region
of the same run and reported as `tracks_per_s`.  With N>1 ranks the tracks are sharded and the reduced
camera system is all-reduced over NCCL once per iteration (strong scaling: total problem fixed).
"""
from __future__ import annotations

import os
import sys

if "reference" in sys.argv:
    # The CPU arm uses every host core -- also under torchrun, which exports OMP_NUM_THREADS=1 for its workers; the
    # BLAS / OpenMP runtimes read these at import time, so this has to happen before numpy is imported.
    for _k in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[_k] = str(os.cpu_count() or 1)

import argparse
import json
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

S_FRAMES, N_TRACKS = 400, 4096
CAMERA = "SIMPLE_RADIAL"
ITERS = 10                      # LM iterations per step
WORKLOAD = "C3: 400 frames x 4096 tracks, SIMPLE_RADIAL shared_camera, dense visibility (SURVEY 8d)"
METRIC = "BA iterations/sec"


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def load_tensor_peak():
    """Measured dense bf16 TFLOP/s of this pool's B200s (burst: a kernel timed alone), else the profiling recipe's figure."""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        if "bf16_tflops" in d:
            return float(d["bf16_tflops"]), "measured cuBLAS bf16 (MEASURED_PEAKS.json)"
    return 1650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock and throttle reasons DURING the timed region (B200_PROFILING.md recipe), sampled in-process through
    NVML every 250 ms (an `nvidia-smi -lms` child process was measured to slow the timed region by ~30 %)."""

    def __init__(self, index=0):
        self.index, self.rows, self._stop, self.th = index, [], threading.Event(), None
        self.err = None

    def prepare(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            pynvml.nvmlDeviceGetClockInfo(self.h, pynvml.NVML_CLOCK_SM)     # first query pays the one-time cost here
        except Exception as e:       # NVML missing: report it, do not fail the bench
            self.err = str(e)[:100]
            self.nv = None

    def start(self):
        if getattr(self, "nv", None) is None:
            return
        self.th = threading.Thread(target=self._run, daemon=True)
        self.th.start()

    def _run(self):
        nv = self.nv
        if self._stop.wait(0.04):          # first sample 40 ms into the region, then every 250 ms
            return
        while not self._stop.is_set():
            try:
                sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                mx = nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)
                rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.rows.append((sm, mx, rs))
            except Exception as e:
                self.err = str(e)[:100]
            self._stop.wait(0.25)

    def stop(self):
        if self.th is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable: %s" % self.err]}
        self._stop.set()
        self.th.join(timeout=2)
        nv = self.nv
        names = {"hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
        reasons = sorted(k for k, bit in names.items() if any(r[2] & bit for r in self.rows))
        sm = [r[0] for r in self.rows]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(r[1] for r in self.rows) if sm else None,
                "reasons": reasons, "samples": len(sm)}


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """Write each output of the last timed step as out_dir/<name>.npy: float64 stays float64, everything else
    (float32 tracks, integer counts and indices, boolean masks) becomes float32.  At the C3 size the whole set is a
    few MB, far under DUMP_LIMIT_BYTES, so every array is written in full."""
    host = {}
    for name, a in arrays.items():
        a = a.detach().cpu().numpy() if hasattr(a, "detach") else np.asarray(a)
        host[name] = a if a.dtype == np.float64 else a.astype(np.float32)
    total = sum(a.nbytes for a in host.values())
    if total > DUMP_LIMIT_BYTES:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT_BYTES}-byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in host.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def make_problem():
    from vggsfm_b200.synthetic import make_scene, perturb
    sc = make_scene(S_FRAMES, N_TRACKS, CAMERA, seed=0)
    extr, K, extra, pts = perturb(sc, seed=1)
    return sc, extr, K, extra, pts


# --------------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference's BA (pycolmap/Ceres are absent -> "port"), all host threads
# --------------------------------------------------------------------------------------------------

def cpu_ba_sample(sc, extr, K, extra, pts, iters):
    """`iters` LM iterations of oracle.ba_oracle.lm_solve at the full C3 size; returns (it/s, seconds), the time of
    the solve's initial residual/Jacobian evaluation (which is not an LM iteration) excluded from both."""
    from oracle import ba_oracle as bo
    S = extr.shape[0]
    intr = np.zeros((S, 4))
    intr[:, 0], intr[:, 1], intr[:, 2], intr[:, 3] = K[:, 0, 0], K[:, 0, 2], K[:, 1, 2], extra[:, 0]
    intr[:] = intr[0]
    opt = bo.LMOptions()
    opt.max_num_iterations = iters
    opt.gradient_tolerance = 0.0
    t0 = time.perf_counter()
    _, _, _, summ = bo.lm_solve(extr, intr, pts, sc.tracks.astype(np.float64), sc.mask, bo.SIMPLE_RADIAL,
                                bo.INTR_SHARED, options=opt, use_c=bo._load_c() is not None)
    dt = time.perf_counter() - t0 - summ.get("initial_eval_s", 0.0)
    return summ["iterations"] / dt, dt


def cpu_tri_sample(sc, ntracks):
    """CPU triangulate_tracks (256 hypotheses) on the first `ntracks` tracks of C3; returns (tracks/s, seconds, kind).
    kind = "port": oracle/tri_oracle.py (numpy restatement pinned to the reference's goldens)."""
    import torch
    from oracle import tri_oracle as to
    tn = to.cam_from_img(sc.tracks[:, :ntracks].astype(np.float64), sc.intrinsics, sc.extra_params)
    torch.manual_seed(0)
    pairs = to.draw_pairs(S_FRAMES, 256)
    t0 = time.perf_counter()
    to.triangulate_tracks(sc.extrinsics, tn, pairs, sc.vis[:, :ntracks], sc.score[:, :ntracks])
    dt = time.perf_counter() - t0
    return ntracks / dt, dt, "port"


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sc, extr, K, extra, pts = make_problem()
    cores = os.cpu_count()
    REF_ITERS = 3
    for _ in range(args.warmup):
        cpu_ba_sample(sc, extr, K, extra, pts, 1)
    its = 0
    dt = 0.0
    wall0 = time.perf_counter()
    for _ in range(args.steps):
        v, d = cpu_ba_sample(sc, extr, K, extra, pts, REF_ITERS)
        its += REF_ITERS
        dt += d
    wall = time.perf_counter() - wall0
    value = its / dt
    tri_v, _, tri_kind = cpu_tri_sample(sc, 16)
    sample = (f"each step = one oracle/ba_oracle.lm_solve of {REF_ITERS} LM iterations (C/OpenMP Jacobians + numpy/BLAS Schur and "
              "Cholesky, float64) at full C3 size; it/s counts the LM iterations only (the solve's initial evaluation is timed "
              f"and excluded, like the GPU arm's fixed setup); triangulation: {tri_kind} on 16 of 4096 tracks")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "it/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * wall / max(1, args.steps), "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD, "lm_iterations_per_step": REF_ITERS,
                   "note": "pycolmap/pyceres absent: oracle port of COLMAP/Ceres BA on host cores"},
        "cpu_baseline": {"value": value, "unit": "it/s", "cores": cores, "kind": "port", "sample": sample},
        "tracks_per_s": tri_v, "tracks_per_s_kind": tri_kind,
        "e2e": {"value": value, "unit": "it/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------------------

def syrk_roofline(D, K3, dev, clocks):
    import torch
    from vggsfm_b200 import _lib
    """Times vgg_syrk_ozaki (slice + tcgen05 SYRK) at this rank's Schur shape with CUDA events.  Algorithmic work =
    28 int8 GEMM pairs x 2 K Dpad (Dpad+128)/2 ops on the lower tiles; peak = 148 SMs x 8192 MAC/clk (the kind::i8 rate
    measured with N=256, tools/syrk_i8_check.py rate) x 2 x the SM clock sampled during the run."""
    import ctypes
    L = _lib.lib()
    Dpad = (D + 2 + 127) // 128 * 128
    Kpad = (K3 + 15) // 16 * 16
    slices = 7
    g = torch.Generator(device=dev).manual_seed(0)
    Zt = torch.randn(Kpad, Dpad, dtype=torch.float64, device=dev, generator=g)
    Zt[:, D:] = 0
    C = torch.zeros(Dpad, Dpad, dtype=torch.float64, device=dev)
    nb = ctypes.c_size_t()
    _lib.check(L.vgg_syrk_ozaki_workspace_bytes(Kpad, Dpad, slices, ctypes.byref(nb)), "vgg_syrk_ozaki_workspace_bytes")
    ws = torch.empty(nb.value, dtype=torch.uint8, device=dev)
    st = torch.cuda.current_stream().cuda_stream
    call = lambda: _lib.check(L.vgg_syrk_ozaki(Kpad, Dpad, Zt.data_ptr(), C.data_ptr(), slices, ws.data_ptr(), ws.numel(), st),
                              "vgg_syrk_ozaki")
    for _ in range(3):
        call()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 10
    a.record()
    for _ in range(reps):
        call()
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b) / reps
    pairs = slices * (slices + 1) // 2
    ops = pairs * 2.0 * Kpad * Dpad * (Dpad + 128) / 2
    sm_mhz = (clocks or {}).get("sm_mhz") or 1965.0
    peak = 148 * 8192 * 2 * sm_mhz * 1e6 / 1e12
    ach = ops / (ms * 1e-3) / 1e12
    return {"kernel": "oz_slice_kernel + oz_syrk_kernel (tcgen05.mma kind::i8, 7 Ozaki slices)", "bound": "tensor",
            "achieved": ach, "peak": peak, "unit": "TOP/s", "frac": ach / peak, "ms_per_call": ms,
            "peak_source": "148 SMs x 8192 int8 MAC/clk/SM (measured kind::i8 N=256 issue rate) x sampled SM clock",
            "fp64_equivalent_tflops": 2.0 * Kpad * Dpad * (Dpad + 128) / 2 / (ms * 1e-3) / 1e12,
            "note": "time includes the column-max and slicing kernels; in the LM loop the column max is fused into z_build"}


def corr_section(dev, hbm_peak):
    """C4 (BASELINE.json configs[3]): one correlation + sampling pass of the tracker's refinement loop, fused CUDA kernel
    vs the reference's GPU path restated with stock PyTorch ops (oracle.corr_oracle.TorchCorrBlock: fp16 matmul of the
    full volume + grid_sample) on the same device.  Coarse: fmaps [1,128,128,128,128], one 1024-query chunk, 5 levels,
    r = 4.  Fine: [1024,128,32,31,31] patches, one query each, 3 levels, r = 3.  Algorithmic bytes of the fused kernel =
    the (2r+2)^2 footprint positions x C x 2 B per level + the target vector + coordinates + outputs."""
    import torch
    from vggsfm_b200.corr import CorrBlock
    from oracle.corr_oracle import TorchCorrBlock
    out = {}

    def timeit(fn, reps, warm=2):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            fn()
        b.record()
        torch.cuda.synchronize()
        return a.elapsed_time(b) / reps

    for name, (B, S, C, H, W, N, L, r) in {"coarse": (1, 128, 128, 128, 128, 1024, 5, 4), "fine": (1024, 128, 32, 31, 31, 1, 3, 3)}.items():
        try:
            g = torch.Generator(device=dev).manual_seed(0)
            fm = torch.randn(B, S, C, H, W, device=dev, dtype=torch.float16, generator=g)
            tg = torch.randn(B, S, N, C, device=dev, dtype=torch.float32, generator=g)
            co = torch.rand(B, S, N, 2, device=dev, generator=g) * torch.tensor([W - 9.0, H - 9.0], device=dev) + 4.0
            K = 2 * r + 1
            ours = CorrBlock(fm, num_levels=L, radius=r, half=True)
            torch.cuda.synchronize()

            def run_ours():
                ours.corr(tg)
                return ours.sample(co)
            ms = timeit(run_ours, 5)
            foot = sum(min((2 * r + 2), H >> l) * min((2 * r + 2), W >> l) for l in range(L)) * C * 2
            ab = B * S * N * (foot + C * 4 + 8 + L * K * K * 4)
            rec = {"shape": [B, S, C, H, W], "queries": N, "levels": L, "radius": r, "ms_fused": ms,
                   "pairs_per_s": B * S * N / (ms * 1e-3)}
            if getattr(ours._pyr, "tc_tiles", None) is not None:
                # tcgen05 path (csrc/corr_tc.cu): the dense per-level correlation runs on the tensor cores (kind::f16,
                # fp32 accumulators in TMEM) and is sampled from TMEM -- tensor-bound, not HBM-bound
                fl = 2.0 * B * S * N * C * sum((H >> l) * (W >> l) for l in range(L))
                tpk, tsrc = load_tensor_peak()
                rec.update({"kernel": "corr_tc_kernel (tcgen05.mma kind::f16, M=128 N=256, TMEM accumulators)", "bound": "tensor",
                            "flops": fl, "achieved_tflops": fl / (ms * 1e-3) / 1e12, "tensor_peak_tflops": tpk,
                            "tensor_peak_source": tsrc, "frac_of_tensor_peak": fl / (ms * 1e-3) / 1e12 / tpk,
                            "ncu": "profiles/r02_ncu_corr_tc8.txt: sm__pipe_tensor_subpipe_hmma_cycles_active 38.7 %"})
            else:
                rec.update({"kernel": ("corr_sample_c32_kernel (CUDA cores, one footprint position per lane)" if C == 32
                                       else "corr_sample_kernel (CUDA cores, channels across lanes)"),
                            "bound": "hbm", "algorithmic_bytes": ab,
                            "achieved_gbs": ab / (ms * 1e-3) / 1e9, "frac_of_hbm_peak": ab / (ms * 1e-3) / 1e9 / hbm_peak})
            res = run_ours()
            del ours
            try:
                with torch.autocast("cuda", dtype=torch.float16):
                    base = TorchCorrBlock(fm, num_levels=L, radius=r)

                    def run_base():
                        base.corr(tg)
                        return base.sample(co)
                    rec["ms_torch_reference_path"] = timeit(run_base, 2, warm=1)
                    ref = run_base().float()
                rec["speedup_vs_torch_path"] = rec["ms_torch_reference_path"] / ms
                rec["max_abs_diff_vs_torch_path"] = float((res - ref).abs().max())
                rec["flops_torch_path"] = 2.0 * B * S * N * C * sum((H >> l) * (W >> l) for l in range(L))
                del base, ref
            except Exception as e:      # the full volume does not fit next to the bench tensors: report ours only
                rec["torch_reference_path_error"] = str(e)[:160]
            out[name] = rec
            del fm, tg, co, res
            torch.cuda.empty_cache()
        except Exception as e:
            out[name] = {"error": str(e)[:200]}
    return out


def small_problem_section(dev):
    """LM it/s at the sizes the real pipeline runs most (SURVEY 8d): C1 (8 x 256, SIMPLE_PINHOLE), C2 (50 x 2048,
    SIMPLE_PINHOLE), and the video runner's window BA (17 frames x 3072 points, first frame and the first 1024 points
    constant, intrinsics constant; video_runner.py:813-829).  These are launch- and sync-bound, not bandwidth-bound."""
    import torch
    from vggsfm_b200 import bundle_adjustment as ba
    from vggsfm_b200.synthetic import make_scene, perturb
    out = {}
    t = lambda a, dt=None: (torch.from_numpy(np.ascontiguousarray(a)).to(dt) if dt else torch.from_numpy(np.ascontiguousarray(a))).to(dev).contiguous()
    for name, S, N, window in (("C1_8x256", 8, 256, False), ("C2_50x2048", 50, 2048, False), ("window_17x3072", 17, 3072, True)):
        sc = make_scene(S, N, "SIMPLE_PINHOLE", seed=3, invisible_frac=0.2)
        extr, K, _, pts = perturb(sc, seed=4)
        intr = np.zeros((S, 4))
        intr[:, 0], intr[:, 1], intr[:, 2] = K[:, 0, 0], K[:, 0, 2], K[:, 1, 2]
        model = ba.SIMPLE_PINHOLE
        mode = ba.INTR_CONST if window else ba.INTR_PER_FRAME
        uv, mask = t(sc.tracks, torch.float32), t(sc.mask.astype(np.uint8))
        p0, i0, x0 = t(extr), t(intr), t(pts)
        pc = None
        if window:
            cp = torch.zeros(S, dtype=torch.bool, device=dev)
            cp[0] = True
            param_const = ba.default_param_const(S, model, mode, dev, False, False, gauge=False, const_pose=cp)
            pc = (torch.arange(N, device=dev) < 1024).to(torch.uint8)
        else:
            param_const = ba.default_param_const(S, model, mode, dev)
        opt = ba.default_options()
        opt.max_num_iterations = 10
        opt.gradient_tolerance = 0.0
        run = lambda: ba.lm_solve(uv, mask, p0.clone(), i0.clone(), x0.clone(), model, mode, param_const, pc, opt)
        for _ in range(3):
            s_ = run()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps, its = 10, 0
        a.record()
        for _ in range(reps):
            its += run().iterations
        b.record()
        torch.cuda.synchronize()
        ms = a.elapsed_time(b)
        out[name] = {"it_per_s": its / (ms * 1e-3), "ms_per_iteration": ms / max(1, its), "launches_per_solve": s_.kernel_launches}
    return out


def run_gpu(args):
    import torch
    import torch.distributed as dist
    from vggsfm_b200 import bundle_adjustment as ba
    from vggsfm_b200 import triangulation as tri
    from vggsfm_b200 import _lib
    from vggsfm_b200.dist import AllReduceHook, shard_range

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a GPU (no CPU fallback for the product path)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)        # NCCL_DEBUG is left as the launcher set it
    _lib.lib()

    sc, extr, K, extra, pts = make_problem()
    lo, hi = shard_range(N_TRACKS, rank, world)
    n_loc = hi - lo
    model, mode = ba.SIMPLE_RADIAL, ba.INTR_SHARED
    intr_np = np.zeros((S_FRAMES, 4))
    intr_np[:, 0], intr_np[:, 1], intr_np[:, 2], intr_np[:, 3] = K[0, 0, 0], K[0, 0, 2], K[0, 1, 2], extra[0, 0]
    t = lambda a, dt=None: (torch.from_numpy(np.ascontiguousarray(a)).to(dt) if dt else torch.from_numpy(np.ascontiguousarray(a))).to(dev).contiguous()
    uv = t(sc.tracks[:, lo:hi], torch.float32)
    mask = t(sc.mask[:, lo:hi].astype(np.uint8))
    poses0, intr0, pts0 = t(extr), t(intr_np), t(pts[lo:hi])
    param_const = ba.default_param_const(S_FRAMES, model, mode, dev)
    opt = ba.default_options()
    opt.max_num_iterations = ITERS
    opt.gradient_tolerance = 0.0          # run exactly ITERS iterations every step
    hook = None
    reduction = "none (1 GPU)"
    if world > 1:
        fabric = None
        if os.environ.get("VGG_FABRIC", "1") != "0":
            try:
                from vggsfm_b200.dist import FabricBuffer
                fabric = FabricBuffer(S_FRAMES, model, mode, dev)
            except Exception as e:       # no symmetric memory / multicast on this box: NCCL all-reduce instead
                if rank == 0:
                    print(f"[bench] fabric reduction unavailable ({str(e)[:120]}); using NCCL all-reduce", file=sys.stderr)
                fabric = None
        hook = AllReduceHook(fabric=fabric)
        if hook.fabric is None:
            reduction = "NCCL all-reduce of the reduced system"
        elif hook.fabric.v2 and os.environ.get("VGG_FABRIC", "2") != "1":
            reduction = ("fabric v2: reduce-scatter of the lower triangle by red.add.f64 into the owning rank's rows from the "
                         "SYRK epilogue, gather by peer loads, in-kernel barriers and mailbox all-reduce of the small vectors "
                         "(csrc/fabric.cu; no NCCL call and no host callback inside the LM loop)")
        else:
            reduction = "fabric v1: multimem.red all-reduce fused into the Schur kernels (NVSwitch multicast) + host-hook barriers"
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)   # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def ba_step():
        poses, intr, X = poses0.clone(), intr0.clone(), pts0.clone()
        s = ba.lm_solve(uv, mask, poses, intr, X, model, mode, param_const, None, opt, hook)
        return s, {"ba_poses": poses, "ba_intrinsics": intr, "ba_points3d": X}

    # ---- timed region 1: BA
    launches = 0
    sampler = ClockSampler(local)
    if rank == 0 and os.environ.get("VGG_BENCH_NOCLOCKS") != "1":
        sampler.prepare()                  # NVML init + device handle outside the timed region
    for _ in range(args.warmup):
        flush.fill_(1.0)                   # also loads the fill kernel's module before the timed region
        ba_step()
    barrier()
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    its = 0
    for _ in range(args.steps):
        flush.fill_(1.0)
        s, ba_out = ba_step()
        its += s.iterations
        launches += s.kernel_launches
    e1.record()
    barrier()
    ba_ms = e0.elapsed_time(e1)
    clocks = sampler.stop() if rank == 0 else None
    tms = torch.tensor([ba_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
    ba_ms = float(tms.item())
    value = its / (ba_ms * 1e-3)
    final_cost = s.final_cost

    # ---- timed region 2: triangulation (tracks sharded, no collective)
    E = t(sc.extrinsics)
    Kt = t(sc.intrinsics)
    ext = t(sc.extra_params)
    trk = t(sc.tracks[:, lo:hi])
    vis, score = t(sc.vis[:, lo:hi]), t(sc.score[:, lo:hi])
    torch.manual_seed(0)
    pairs = tri.draw_ransac_pairs(S_FRAMES, 256)

    def tri_pass():
        # what the pipeline does per pass for SIMPLE_RADIAL (triangulator.py:379-391): cam_from_img with the reference's
        # iterative undistortion, then the 256+50+10-hypothesis LORANSAC
        tn = tri.cam_from_img(trk, Kt, ext)
        return tri.triangulate_tracks(E, tn, track_vis=vis, track_score=score, ransac_pairs=pairs)

    for _ in range(args.warmup):
        tri_pass()
    barrier()
    e0.record()
    for _ in range(args.steps):
        flush.fill_(1.0)
        p3, num, inl = tri_pass()
        launches += 6
    e1.record()
    barrier()
    tms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
    tri_ms = float(tms.item())
    tracks_per_s = N_TRACKS * args.steps / (tri_ms * 1e-3)
    tri_median_err = float(np.median(np.linalg.norm(p3.cpu().numpy() - sc.points3d[lo:hi], axis=1)))

    # ---- e2e: public API with host (pinned) buffers, copies inside the timed region
    h_tracks = torch.from_numpy(sc.tracks[:, lo:hi].copy()).pin_memory()
    h_masks = torch.from_numpy(sc.mask[:, lo:hi].copy()).pin_memory()
    h_pts = torch.from_numpy(pts[lo:hi].copy()).pin_memory()
    h_extr = torch.from_numpy(extr.copy()).pin_memory()
    h_K = torch.from_numpy(K.copy()).pin_memory()
    h_extra = torch.from_numpy(extra.copy()).pin_memory()
    h2d = sum(x.numel() * x.element_size() for x in (h_tracks, h_masks, h_pts, h_extr, h_K, h_extra))

    def e2e_step():
        out = ba.bundle_adjustment(h_pts.to(dev, non_blocking=True), h_extr.to(dev, non_blocking=True),
                                   h_K.to(dev, non_blocking=True), h_extra.to(dev, non_blocking=True),
                                   h_tracks.to(dev, non_blocking=True), h_masks.to(dev, non_blocking=True),
                                   shared_camera=True, camera_type=CAMERA, options=opt, allreduce=hook)
        res = [out[0].cpu(), out[1].cpu(), out[2].cpu(), out[3].cpu()]
        return out[5], sum(x.numel() * x.element_size() for x in res), res + [out[4]]

    for _ in range(min(args.warmup, 2)):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    e2e_its = 0
    d2h = 0
    for _ in range(args.steps):
        s2, d2h, e2e_out = e2e_step()
        e2e_its += s2.iterations
        launches += s2.kernel_launches
    barrier()
    e2e_s = time.perf_counter() - t0
    ts = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ts, op=dist.ReduceOp.MAX)
    e2e_value = e2e_its / float(ts.item())

    if rank == 0 and args.dump_outputs:
        names = ("e2e_points3d", "e2e_extrinsics", "e2e_intrinsics", "e2e_extra_params", "e2e_valid_idx")
        dump_outputs(args.dump_outputs, {**ba_out, "tri_points3d": p3, "tri_inlier_num": num, "tri_inlier_mask": inl,
                                         **dict(zip(names, e2e_out))})

    # ---- roofline of the fused residual+Jacobian+block kernel (the HBM-bound kernel of the path), live
    roof = None
    roof_syrk = None
    cpu_base = None
    corr = None
    small = None
    c5 = None
    if rank == 0:
        peak, peak_src = load_peaks()
        dc, ns = ba.dims(model, mode)
        obs = S_FRAMES * n_loc

        def algo_bytes(S, N):
            KR = _lib.lib().vgg_ba_camrec_len(model, mode)
            return S * N * (8 + 1) + S * (12 + 4) * 8 + N * 3 * 8 + S * KR * 8 + N * 9 * 8 + (S * dc + ns) * N * 3 * 8

        def time_blocks(uv_, mask_, poses_, intr_, X_, reps):
            """(kernel ms, call ms): the kernel alone from the event pair the library records on its stream directly
            around the ba_blocks_kernel launch (csrc/dev_probes.h), and the whole build_blocks call (accumulator memset,
            W-tail memset2D, kernel) from torch events on the same stream.  L2 is flushed before every launch."""
            import ctypes
            L = _lib.lib()
            for _ in range(3):
                ba.build_blocks(uv_, mask_, poses_, intr_, X_, model, mode)
            torch.cuda.synchronize()
            _lib.check(L.vgg_dev_blocks_timing(1), "blocks timing")
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            tot = 0.0
            tot_k = 0.0
            k_ms = ctypes.c_double(0.0)
            try:
                for _ in range(reps):
                    flush.fill_(1.0)
                    a.record()
                    out = ba.build_blocks(uv_, mask_, poses_, intr_, X_, model, mode)
                    b.record()
                    torch.cuda.synchronize()
                    tot += a.elapsed_time(b)
                    _lib.check(L.vgg_dev_blocks_last_ms(ctypes.byref(k_ms)), "blocks timing")
                    tot_k += k_ms.value
                    del out
            finally:
                L.vgg_dev_blocks_timing(0)
            return tot_k / reps, tot / reps

        ms, ms_call = time_blocks(uv, mask, poses0, intr0, pts0, 10)
        ab = algo_bytes(S_FRAMES, n_loc)
        ach = ab / (ms * 1e-3) / 1e9
        roof = {"kernel": "ba_blocks_kernel<SIMPLE_RADIAL,INTR_SHARED,TMA>", "bound": "hbm", "achieved": ach,
                "peak": peak, "peak_source": peak_src, "unit": "GB/s", "frac": ach / peak,
                # dram__bytes_read.sum + dram__bytes_write.sum of this launch from the ncu --set full capture
                # profiles/r02_ncu_blocks_c3b.txt (16.0 MB + 176.7 MB; part of W is still in the 126 MB L2 when the counters stop)
                "traffic": 1.927e8 if n_loc == N_TRACKS else None,
                "bytes_per_launch": ab, "ms_per_launch": ms, "ms_per_call": ms_call, "observations": obs,
                "note": "ms_per_launch: CUDA event pair on the launching stream directly around the kernel; ms_per_call adds "
                        "the accumulator memset and the W-tail memset2D of one build_blocks call; 256 MB L2 flush before each"}
        # scaled synthetic (SURVEY 8d): 400 x 131072 tracks = 52 M observations, 8 GB of coupling blocks
        try:
            NS_ = 131072
            rng = np.random.default_rng(0)
            rep = NS_ // n_loc + 1
            uv_s = uv.repeat(1, rep, 1)[:, :NS_].contiguous()
            mk_s = mask.repeat(1, rep)[:, :NS_].contiguous()
            X_s = pts0.repeat(rep, 1)[:NS_].contiguous()
            ms_s, ms_s_call = time_blocks(uv_s, mk_s, poses0, intr0, X_s, 5)
            ab_s = algo_bytes(S_FRAMES, NS_)
            ach_s = ab_s / (ms_s * 1e-3) / 1e9
            roof["scaled"] = {"workload": "400 x 131072 tracks", "achieved": ach_s, "frac": ach_s / peak,
                              "bytes_per_launch": ab_s, "ms_per_launch": ms_s, "ms_per_call": ms_s_call,
                              # dram__bytes_read.sum + dram__bytes_write.sum of this launch shape from the ncu --set full
                              # capture kept in profiles/r01_ncu_full_summary_k1_scaled.txt (0.58 GB + 7.51 GB)
                              "traffic": 8.09e9}
            del uv_s, mk_s, X_s
        except Exception as e:     # out of memory on a shared box: keep the C3-size number
            roof["scaled"] = {"error": str(e)[:200]}
        # ---- tensor-core roofline of the Schur SYRK (the largest of this library's kernels per LM iteration), live
        try:
            roof_syrk = syrk_roofline(S_FRAMES * dc + ns, 3 * n_loc, dev, clocks)
        except Exception as e:
            roof_syrk = {"error": str(e)[:200]}
        if world == 1:
            try:
                small = small_problem_section(dev)
            except Exception as e:
                small = {"error": str(e)[:200]}
        if world == 1 and not args.no_corr:
            torch.cuda.empty_cache()
            corr = corr_section(dev, peak)
        if world == 1 and not args.no_c5:
            # C5 (BASELINE.json configs[4]): the synthetic 1000-frame sequential run of tools/video_c5.py, and its last joint
            # BA alone (second of two solves: the first one pays the CUDA-graph captures and the work-list plans)
            try:
                torch.cuda.empty_cache()
                sys.path.insert(0, os.path.join(ROOT, "tools"))
                import video_c5
                seq = video_c5.run(dev=dev)
                fin = video_c5.final_problem(dev=dev, reps=2)
                c5 = {"sequence": {k: seq[k] for k in ("workload", "frames", "seconds", "frames_per_s", "split_seconds", "windows",
                                                         "joint_bas", "joint_iterations", "window_iterations",
                                                         "camera_centre_rmse_vs_gt", "trajectory_length")},
                      "final_joint_ba": {"workload": fin["workload"], "seconds": fin["seconds"][-1],
                                         "lm_iterations": fin["lm_iterations"][-1], "lm_it_per_s": fin["lm_it_per_s"][-1]}}
            except Exception as e:
                c5 = {"error": str(e)[:200]}
        if world == 1:
            v, dt = cpu_ba_sample(sc, extr, K, extra, pts, 3)
            tv, tdt, tkind = cpu_tri_sample(sc, 16)
            cpu_base = {"value": v, "unit": "it/s", "cores": os.cpu_count(), "kind": "port",
                        "sample": f"3 LM iterations of oracle/ba_oracle.lm_solve (C/OpenMP Jacobians + numpy/BLAS Schur and Cholesky, float64) at full C3 size, {dt:.1f} s "
                                  f"(initial evaluation excluded); triangulation: {tkind} on 16 of 4096 tracks, {tdt:.1f} s",
                        "tracks_per_s": tv, "tracks_per_s_kind": tkind}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "it/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ba_ms / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD, "lm_iterations_per_step": ITERS, "parallelism": f"track-shard x{world}",
                       "reduction": reduction,
                       "tracks_per_rank": n_loc, "l2": "256 MB flush write between steps; working set ~0.8 GB > 126 MB L2",
                       "final_cost": final_cost},
            "tracks_per_s": tracks_per_s, "tri_ms_per_pass": tri_ms / args.steps, "tri_median_point_error": tri_median_err,
            "e2e": {"value": e2e_value, "unit": "it/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roof, "roofline_syrk": roof_syrk,
            "cpu_baseline": cpu_base, "corr": corr, "small_problems": small, "c5": c5,
        }
        line["config"]["syrk"] = os.environ.get("VGG_SYRK", "ozaki:7") + " (default: tcgen05 kind::i8, 7 Ozaki slices, FP64-equivalent)"
        if hook is not None:
            line["config"]["allreduce_calls"] = hook.calls
            line["config"]["allreduce_bytes"] = hook.bytes
            line["config"]["fabric_barriers"] = hook.barriers
            line["config"]["nccl_nranks"] = dist.get_world_size()
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-corr", action="store_true", help="skip the C4 correlation section (rank 0, N=1 only)")
    ap.add_argument("--no-c5", action="store_true", help="skip the C5 sequential-video section (rank 0, N=1 only)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last BA, triangulation and end-to-end steps returned as "
                         "DIR/<name>.npy (float32/float64; rank 0's shard of the tracks when N>1)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
