"""CUDA-event micro-benchmarks for A/B runs (env switches are read once per process):
   python tools/microbench.py chol | ba | blocks [N] | pose [S N] | pipeline [S N]"""
import ctypes
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from vggsfm_b200 import _lib, bundle_adjustment as ba       # noqa: E402
from vggsfm_b200.synthetic import make_scene, perturb       # noqa: E402

dev = torch.device("cuda:0")
mode = sys.argv[1] if len(sys.argv) > 1 else "ba"
tag = " ".join(f"{k}={v}" for k, v in os.environ.items() if k.startswith("VGG_"))


def timeit(fn, reps=10, warm=3):
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


if mode in ("pose", "pipeline"):
    from vggsfm_b200 import pose_refinement as pr
    from vggsfm_b200.synthetic import project_np
    from vggsfm_b200.triangulator import Triangulator
    S = int(sys.argv[2]) if len(sys.argv) > 2 else 400
    N = int(sys.argv[3]) if len(sys.argv) > 3 else 4096
    cam, shared = "SIMPLE_RADIAL", True
    sc = make_scene(S, N, cam, seed=3, invisible_frac=0.2, outlier_frac=0.02)
    extr0, K0, ex0, _ = perturb(sc, rot_deg=0.4, trans_frac=0.01, focal_frac=0.02, seed=4)
    T = lambda a, dt=None: torch.from_numpy(np.ascontiguousarray(a)).to(dev) if dt is None else torch.from_numpy(np.ascontiguousarray(a)).to(dev, dt)
    if mode == "pose":
        E, K, ex = T(extr0), T(K0), T(ex0)
        X, tracks, inl = T(sc.points3d), T(sc.tracks), T(sc.mask)
        valid = torch.ones(N, dtype=torch.bool, device=dev)
        isz = torch.tensor([1024, 1024], device=dev)
        for sh in (False, True):
            ms = timeit(lambda: pr.refine_pose(E, K, ex, inl, X, tracks, valid, isz, shared_camera=sh, camera_type=cam), reps=5, warm=2)
            its = pr.last_report.iterations.float()
            print(f"[{tag}] refine_pose {S}x{N} shared={sh}: {ms:.3f} ms  ({S / ms * 1e3:.0f} frames/s; LM its mean {its.mean():.1f} max {int(its.max())})")
        sys.exit(0)

    class Cams:
        pass
    c = Cams()
    c.focal_length = T(np.stack([K0[:, 0, 0], K0[:, 1, 1]], -1) * 2.0 / 1024, torch.float32)
    c.R, c.T = T(extr0[:, :, :3], torch.float32), T(extr0[:, :, 3], torch.float32)
    uv_gt, _ = project_np(sc.extrinsics, 1000.0, np.array([512.0, 512.0]), 0.05, sc.points3d)
    ok = np.linalg.norm(sc.tracks - uv_gt, axis=-1) < 3.0
    prelim = {"fmat_inlier_mask": T(ok[:1] & ok[1:])[None]}
    images = torch.zeros(1, S, 3, 64, 64, device=dev)
    tr = Triangulator()
    tracks, vis, score = T(sc.tracks)[None], T(sc.vis)[None], T(sc.score)[None]
    # images are only read for their shape and the colour lookup; use a 1024x1024 canvas without allocating it per call
    images = torch.zeros(1, S, 3, 1024, 1024, device=dev) if S <= 64 else torch.zeros(1, 1, 3, 1024, 1024, device=dev).expand(1, S, 3, 1024, 1024)

    def run():
        torch.manual_seed(0)
        return tr(c, tracks, vis, images, prelim, pred_score=score, BA_iters=2, shared_camera=shared, robust_refine=2,
                  camera_type=cam, extract_color=S <= 64)
    tr.verbose = True
    out = run()
    tr.verbose = False
    ms = timeit(run, reps=3, warm=1)
    print(f"[{tag}] Triangulator.forward {S}x{N} ({cam}, shared): {ms:.1f} ms  valid tracks {int(out[8].sum())} "
          f"valid frames {int(out[6].sum())}")
    sys.exit(0)

if mode == "trsv":
    import ctypes
    from vggsfm_b200 import _lib
    L = _lib.lib()
    n = int(sys.argv[2]) if len(sys.argv) > 2 else 2402
    lda = (n + 2 + 127) // 128 * 128
    rng = np.random.default_rng(0)
    U = np.triu(rng.normal(size=(n, n)) * 0.05) + np.eye(n)
    A = np.zeros((n + 1, lda))
    A[:n, :n] = U
    y = rng.normal(size=n)
    A[n, :n] = y                                     # like the LM: the right-hand side is the row below the triangle
    Ad = torch.from_numpy(A).to(dev)
    yd = Ad[n]
    xd = torch.empty(n, dtype=torch.float64, device=dev)
    nb = (n + 63) // 64
    st = np.zeros(6 * nb, dtype=np.int64)
    for _ in range(3):
        _lib.check(L.vgg_dev_trsv_probe(n, lda, Ad.data_ptr(), yd.data_ptr(), xd.data_ptr(), st.ctypes.data), "probe")
    x = xd.cpu().numpy()
    print(f"[{tag}] trsv n={n}: |Ux-y|/|y| = {np.linalg.norm(U @ x - y) / np.linalg.norm(y):.2e}")
    ent, lod, inv, see, pub, rhs = st[0::6], st[1::6], st[2::6], st[3::6], st[4::6], st[5::6]
    t0 = pub[nb - 1]
    print(f"  start-up of the last block row: entry -> block loaded {(lod[nb-1]-ent[nb-1])/1e3:.2f} us, -> inverse ready {(inv[nb-1]-lod[nb-1])/1e3:.2f} us, "
          f"-> published {(pub[nb-1]-inv[nb-1])/1e3:.2f} us; entry spread over CTAs {(ent.max()-ent.min())/1e3:.2f} us; "
          f"block row 0: inverse ready {(inv[0]-ent[0])/1e3:.2f} us after entry")
    print("  per block row, us since its own kernel entry: diagonal block loaded / inverse ready / rhs in shared memory / saw-all / published")
    for b in range(nb - 1, -1, -1):
        print(f"    {b:3d}  {(lod[b]-ent[b])/1e3:7.2f} {(inv[b]-ent[b])/1e3:7.2f} rhs {(rhs[b]-ent[b])/1e3:7.2f} {(see[b]-ent[b])/1e3:8.2f} {(pub[b]-ent[b])/1e3:8.2f}")
    print("  block  saw-all(us)  published(us)  compute(us)  hand-off to next(us)")
    for b in range(nb - 1, -1, -1):
        hand = (see[b - 1] - pub[b]) / 1e3 if b > 0 else float("nan")
        print(f"  {b:5d}  {(see[b] - t0) / 1e3:10.2f}  {(pub[b] - t0) / 1e3:12.2f}  {(pub[b] - see[b]) / 1e3:10.2f}  {hand:10.2f}")
    print(f"  total chain {(pub[0] - t0) / 1e3:.1f} us after the last block row published")
    sys.exit(0)

if mode == "chol128":
    import ctypes
    from vggsfm_b200 import _lib
    L = _lib.lib()
    rng = np.random.default_rng(0)
    B = rng.standard_normal((128, 160))
    A = np.ascontiguousarray(B @ B.T / 160 + 0.5 * np.eye(128))
    names = ["leaf(0)", "trsm(b)", "lookahead work", "lookahead wait", "dmma rank-32", "leaf(t0)"]
    Lo = np.zeros((128, 128))
    prof = np.zeros(13, dtype=np.int64)
    _lib.check(L.vgg_dev_chol128_probe(5, A.ctypes.data, Lo.ctypes.data, prof.ctypes.data), "probe")
    err = np.abs(Lo @ Lo.T - A).max() / np.abs(A).max()
    print(f"[{tag}] POTRF128: {prof[12]} cycles  |LL^T-A|/|A| = {err:.2e}")
    for w in (0, 1):
        print("    warp %d: " % w + "  ".join(f"{n} {prof[w * 6 + i]}" for i, n in enumerate(names)))
    sys.exit(0)

if mode == "chol":
    n = int(sys.argv[2]) if len(sys.argv) > 2 else 2403
    rng = np.random.default_rng(0)
    B = rng.normal(size=(n, n + 8))
    A = np.tril(B @ B.T + n * 1e-3 * np.eye(n))
    lda = (n + 127) // 128 * 128
    src = torch.zeros(n, lda, dtype=torch.float64, device=dev)
    src[:, :n] = torch.from_numpy(A).to(dev)
    buf = src.clone()
    ws = torch.empty(((n + 127) // 128) * 131072 + 1024, dtype=torch.uint8, device=dev)
    L = _lib.lib()
    st = torch.cuda.current_stream().cuda_stream

    def run():
        buf.copy_(src)
        _lib.check(L.vgg_cholesky_lower(n, lda, buf.data_ptr(), ws.data_ptr(), ws.numel(), None, st), "chol")
    t_all = timeit(run)
    t_copy = timeit(lambda: buf.copy_(src))
    Afull = src[:, :n] + torch.tril(src[:, :n], -1).T
    t_torch = timeit(lambda: torch.linalg.cholesky(Afull))
    run()
    torch.cuda.synchronize()
    got = torch.tril(buf[:, :n])
    err = (got @ got.T - Afull).abs().max().item() / Afull.abs().max().item()
    print(f"[{tag}] cholesky n={n}: own {t_all - t_copy:.3f} ms   torch.linalg.cholesky {t_torch:.3f} ms   |LL^T-A|/|A| = {err:.2e}")
else:
    S = 400
    N = int(sys.argv[2]) if len(sys.argv) > 2 else 4096
    sc = make_scene(S, N, "SIMPLE_RADIAL", seed=0)
    extr, K, extra, pts = perturb(sc, seed=1)
    t = lambda a, dt=None: (torch.from_numpy(np.ascontiguousarray(a)).to(dt) if dt else torch.from_numpy(np.ascontiguousarray(a))).to(dev).contiguous()
    intr = np.zeros((S, 4))
    intr[:, 0], intr[:, 1], intr[:, 2], intr[:, 3] = K[0, 0, 0], K[0, 0, 2], K[0, 1, 2], extra[0, 0]
    uv, mask = t(sc.tracks, torch.float32), t(sc.mask.astype(np.uint8))
    poses, intr_t, X = t(extr), t(intr), t(pts)
    model, mode_i = ba.SIMPLE_RADIAL, ba.INTR_SHARED
    if mode == "blocks":
        ms = timeit(lambda: ba.build_blocks(uv, mask, poses, intr_t, X, model, mode_i), reps=10)
        nbytes = S * N * 153
        import ctypes
        from vggsfm_b200 import _lib
        L = _lib.lib()
        L.vgg_dev_blocks_timing(1)
        flush = torch.empty(64 << 20, dtype=torch.float32, device=dev)
        k = ctypes.c_double(0.0)
        tot = 0.0
        for _ in range(10):
            flush.fill_(1.0)
            ba.build_blocks(uv, mask, poses, intr_t, X, model, mode_i)
            _lib.check(L.vgg_dev_blocks_last_ms(ctypes.byref(k)), "timing")
            tot += k.value
        L.vgg_dev_blocks_timing(0)
        kms = tot / 10
        print(f"[{tag}] build_blocks 400x{N}: call {ms:.4f} ms  {nbytes / ms / 1e6:.0f} GB/s;  kernel alone (L2 flushed) {kms:.4f} ms  {nbytes / kms / 1e6:.0f} GB/s (153 B/obs)")
    else:
        opt = ba.default_options()
        opt.max_num_iterations = 10
        opt.gradient_tolerance = 0.0
        res = []

        def run():
            res.append(ba.lm_solve(uv, mask, poses.clone(), intr_t.clone(), X.clone(), model, mode_i, options=opt))
        ms = timeit(run, reps=5)
        s = res[-1]
        print(f"[{tag}] lm_solve 400x{N} 10 its: {ms:.2f} ms/solve -> {10e3 / ms:.1f} it/s  cost={s.final_cost:.6f} launches={s.kernel_launches}")
