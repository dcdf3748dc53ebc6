#!/usr/bin/env python
"""Record what the GPU tests used to compare against live -- the REFERENCE's own CUDA operators and tracker (oracle/_ref/libkt_ref_*.so)
-- so that those tests run without the reference on the box.  The inputs are the tests' own seeded synthetic inputs; what is stored
is the reference's side of each comparison: small arrays as they are, large bit-exact results as digests (oracle/golden.py), large
tolerance-based results as a fixed, seeded sample.

Run on a GPU box with oracle/_ref built:   python tools/make_golden_live.py [OUT_DIR]   (writes OUT_DIR/ref_*.npz, default tests/golden)

The ICP replay of tests/test_gpu_baseline_configs.py fuses the PRODUCT's pose sequence with the reference's operators, so this tool
also runs the product tracker and stores the pose sequence it replayed next to the result.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402
import kintinuous_b200 as kb  # noqa: E402
from kintinuous_b200 import synth  # noqa: E402
from oracle import refbind  # noqa: E402
from oracle.golden import digest, canon_points, sample_touched  # noqa: E402

OUT = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "tests", "golden")
SIZE = 6.0


def zeros(shape, dt):
    return torch.zeros(shape, dtype=dt, device="cuda")


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def rot_y(ang):
    return np.array([[np.cos(ang), 0, np.sin(ang)], [0, 1, 0], [-np.sin(ang), 0, np.cos(ang)]], np.float32)


def ops_fixtures():
    """tests/test_gpu_ops.py and test_gpu_baseline_configs.py::test_wrap_beyond_one_volume_length (operators on identical buffers)."""
    V = 256
    ref = refbind.RefCuda(V)
    g = {}
    # ---- test_bilateral_full_resolution_vs_reference: bilateral + 3 pyrDown levels of five 640x480 inputs ----
    rng = np.random.default_rng(20260922)
    inputs = [synth.render(k)[0] for k in (0, 7)]
    noisy = inputs[0].astype(np.int64) + rng.integers(-40, 41, inputs[0].shape)
    noisy[rng.random(noisy.shape) < 0.05] = 0
    inputs.append(np.clip(noisy, 0, 65535).astype(np.uint16))
    far = inputs[0].copy()
    far[100:140, 200:300] = 65535; far[300:330, 10:50] = 50000; far[0:8, 600:640] = 47000
    inputs.append(far)
    inputs.append(rng.integers(0, 65536, inputs[0].shape).astype(np.uint16))
    rows_d = []
    for d in inputs:
        b = zeros((480, 640), torch.int16); ref.bilateral(dev(d.view(np.int16)), b, 480, 640)
        ds = [digest(b)]
        src = b
        for l in range(1, 4):
            r, c = 480 >> (l - 1), 640 >> (l - 1)
            pb = zeros((r // 2, c // 2), torch.int16); ref.pyrdown(src, pb, r, c)
            ds.append(digest(pb)); src = pb
        rows_d.append(ds)
    g["bilateral_full"] = np.array(rows_d)

    # ---- test_volume_ops_vs_reference_cuda_on_identical_buffers: 640x480 into a wrapped 256^3 volume ----
    rows, cols = 480, 640
    intr = np.array(synth.intrinsics(cols, rows), np.float32)
    d, c = synth.render(3)
    dd = dev(d.view(np.int16)); cc = dev(c)
    fb = zeros((rows, cols), torch.int16); ref.bilateral(dd, fb, rows, cols)
    vm = zeros((3 * rows, cols), torch.float32); nm = zeros((3 * rows, cols), torch.float32)
    ref.vmap(fb, vm, rows, cols, intr); ref.nmap(vm, nm, rows, cols)
    g["volops_inputs"] = np.array([digest(fb), digest(vm, "map"), digest(nm, "map")])
    R0 = np.eye(3, dtype=np.float32); t0 = np.array([3, 3, 3], np.float32)
    R1 = rot_y(0.03); t1 = t0 + np.array([0.02, -0.01, 0.03], np.float32)
    voxel = np.float32(SIZE) / np.float32(V)
    trunc = float(max(np.float32(max(0.01, SIZE / 100.0)), np.float32(2.1) * voxel))
    tb = zeros((V ** 3,), torch.int16); cb = zeros((V ** 3 * 4,), torch.uint8); dsb = zeros((rows, cols), torch.float32)
    vs = [SIZE] * 3
    steps = []
    for wrap, R, tt in [((0, 0, 0), R0, t0), ((250, 14, 3), R1, t1), ((250, 14, 3), R1.T.copy(), t1 + np.float32(0.05))]:
        Rinv = np.linalg.inv(R.astype(np.float64)).astype(np.float32)
        ref.integrate(dd, rows, cols, intr, vs, Rinv, tt, trunc, tb, cb, wrap, cc, nm, 1, dsb)
        vb = zeros((3 * rows, cols), torch.float32); nb = zeros((3 * rows, cols), torch.float32); xb = zeros((rows, cols, 4), torch.uint8)
        ref.raycast(intr, R, tt, trunc, vs, tb, vb, nb, rows, cols, wrap, xb, cb)
        torch.cuda.synchronize()
        steps.append([digest(tb), digest(cb), digest(vb, "map"), digest(nb, "map"), digest(xb)])
    g["volops_steps"] = np.array(steps)

    # ---- test_generate_image_and_depth_vs_reference_cuda: GUI taps on a ray-cast surface, 160x120 ----
    rows, cols = 120, 160
    intr = np.array(synth.intrinsics(cols, rows), np.float32)
    d, c = synth.render(0, cols, rows)
    dd = dev(d.view(np.int16)); cc = dev(c)
    fb = zeros((rows, cols), torch.int16); ref.bilateral(dd, fb, rows, cols)
    vm = zeros((3 * rows, cols), torch.float32); nm = torch.zeros_like(vm)
    ref.vmap(fb, vm, rows, cols, intr); ref.nmap(vm, nm, rows, cols)
    ts = zeros((V ** 3,), torch.int16); cs = zeros((V ** 3 * 4,), torch.uint8); ds = zeros((rows, cols), torch.float32)
    R = np.eye(3, dtype=np.float32); t = np.array([3, 3, 3], np.float32)
    for _ in range(3):
        ref.integrate(dd, rows, cols, intr, [6.0] * 3, R, t, 0.06, ts, cs, (0, 0, 0), cc, nm, 1, ds)
    R1g = rot_y(0.02); t1g = t + np.array([0.01, 0.0, 0.02], np.float32)
    va = torch.zeros_like(vm); na = torch.zeros_like(vm); xa = zeros((rows, cols, 4), torch.uint8)
    ref.raycast(intr, R1g, t1g, 0.06, [6.0] * 3, ts, va, na, rows, cols, (0, 0, 0), xa, cs)
    light = [-18.0, -18.0, -18.0]
    ib = zeros((rows, cols, 3), torch.uint8); cb2 = torch.zeros_like(ib)
    ref.generate_image(va, na, xa, light, 1, ib, cb2, rows, cols)
    Rinv = np.linalg.inv(R1g.astype(np.float64)).astype(np.float32)
    db = zeros((rows, cols), torch.int16); ref.generate_depth(Rinv, t1g, va, na, db, rows, cols)
    torch.cuda.synchronize()
    g["genimage_inputs"] = np.array([digest(fb), digest(vm, "map"), digest(nm, "map"), digest(ts), digest(cs), digest(va), digest(na), digest(xa)])
    g["genimage_outputs"] = np.array([digest(ib), digest(cb2), digest(db)])

    # ---- test_wrap_beyond_one_volume_length: offsets beyond one volume length, 160x120 ----
    d, c = synth.render(0, cols, rows)
    dd = dev(d.view(np.int16)); cc = dev(c)
    fb = zeros((rows, cols), torch.int16); ref.bilateral(dd, fb, rows, cols)
    vm = zeros((3 * rows, cols), torch.float32); nm = torch.zeros_like(vm)
    ref.vmap(fb, vm, rows, cols, intr); ref.nmap(vm, nm, rows, cols)
    g["wrap_inputs"] = np.array([digest(fb), digest(vm, "map"), digest(nm, "map")])
    vs = [SIZE] * 3; trunc = 0.06
    R = rot_y(0.05); Rinv = np.linalg.inv(R.astype(np.float64)).astype(np.float32)
    t = np.array([3.02, 2.99, 3.01], np.float32)
    wd, wn = [], []
    for wrap in ((V + 88, 2 * V + 3, 3 * V - 1), (V, 2 * V, 0), (5 * V + 17, 31, V + 200)):
        tb = zeros((V ** 3,), torch.int16); cb = zeros((V ** 3 * 4,), torch.uint8); ds = zeros((rows, cols), torch.float32)
        ref.integrate(dd, rows, cols, intr, vs, Rinv, t, trunc, tb, cb, wrap, cc, nm, 1, ds)
        vb = torch.zeros_like(vm); nb = torch.zeros_like(vm); xb = zeros((rows, cols, 4), torch.uint8)
        ref.raycast(intr, R, t, trunc, vs, tb, vb, nb, rows, cols, wrap, xb, cb)
        cap = 400000
        ob = zeros((cap * 32,), torch.uint8)
        n_b = ref.extract(tb, vs, ob, cap, wrap, cb, (0, V, 0, V, 225, 242), 1, tuple(int(w) for w in wrap))
        torch.cuda.synchronize()
        row = [digest(tb), digest(cb), digest(vb), digest(nb), digest(xb), digest(canon_points(ob[:n_b * 32]))]
        for axis in range(3):
            ref.clear(axis, 0, tb, cb, wrap[axis], wrap[axis] + 14)
        torch.cuda.synchronize()
        row += [digest(tb), digest(cb)]
        wd.append(row); wn.append([n_b, int((cb.view(-1, 4)[:, 3] != 0).sum())])
    g["wrap_steps"] = np.array(wd); g["wrap_counts"] = np.array(wn, np.int64)
    return g


def tracker_fixtures():
    """tests/test_gpu_tracker.py: the reference tracker's poses, volume and model maps on the live tests' input (640x480 into 256^3)."""
    V = 256
    ref = refbind.RefCuda(V)
    frames = [synth.render(k) for k in range(10)]
    g = {}
    # ---- test_tracker_vs_reference_cuda_live ----
    cfg = kb.Config.default(vol=V)
    rt = ref.tracker(refbind.TrackerConfig.from_kt(cfg))
    poses = []
    for k, (d, c) in enumerate(frames):
        rt.process(d, c, k)
        R, t, gc, w = rt.pose()
        poses.append(np.concatenate([R.reshape(-1), t, gc, w.astype(np.float32)]))
    g["live_poses"] = np.array(poses, np.float32)
    tb, cb = rt.export_volume()
    idx = sample_touched(cb[..., 3], 20000, 1)
    g["live_touched"] = np.int64((cb[..., 3] != 0).sum())
    g["live_vol_idx"] = idx; g["live_vol_tsdf"] = tb.reshape(-1)[idx]; g["live_vol_weight"] = cb[..., 3].reshape(-1)[idx]
    # model maps: level 2 (160x120) whole, levels 0 and 1 as a seeded sample of 16384 pixels each
    rng = np.random.default_rng(2)
    for lvl in range(3):
        vb = rt.download_map(2, lvl).reshape(3, -1)
        pix = np.arange(vb.shape[1]) if lvl == 2 else np.sort(rng.choice(vb.shape[1], 16384, replace=False))
        g[f"live_map{lvl}_pix"] = pix.astype(np.int32); g[f"live_map{lvl}"] = vb[:, pix]
    rt.close()
    # ---- test_degenerate_frames_vs_reference_cuda_live ----
    for odometry in (0, 2):
        rng = np.random.default_rng(11)
        seq = []
        for k in range(8):
            d, c = synth.render(k, noise=True) if k in (1, 2) else frames[k]
            d = d.copy()
            if k == 3:
                d[:] = 0
            if k == 4:
                d[:, 320:] = 0
            if k == 5:
                d[rng.random(d.shape) < 0.3] = 0
            if k == 6:
                d, c = seq[-1]
            seq.append((d, c))
        rt = ref.tracker(refbind.TrackerConfig.from_kt(kb.Config.default(vol=V, odometry=odometry)))
        poses = []
        for k, (d, c) in enumerate(seq):
            rt.process(d, c, k)
            R, t, gc, w = rt.pose()
            poses.append(np.concatenate([R.reshape(-1), t, gc, w.astype(np.float32)]))
        g[f"degen{odometry}_poses"] = np.array(poses, np.float32)
        tb, cb = rt.export_volume()
        g[f"degen{odometry}_touched"] = np.int64((cb[..., 3] != 0).sum())
        if odometry == 0:
            idx = sample_touched(cb[..., 3], 20000, 3)
            g["degen0_vol_idx"] = idx; g["degen0_vol_tsdf"] = tb.reshape(-1)[idx]
        rt.close()
    return g


def baseline_fixtures():
    """tests/test_gpu_baseline_configs.py::test_baseline_config_512_live_replay_exact at 640x480 into 512^3."""
    V, ROWS, COLS = 512, 480, 640
    ref = refbind.RefCuda(V)
    frames = [synth.render(k) for k in range(72)]
    intr = np.array(synth.intrinsics(COLS, ROWS), np.float32)
    vs = [SIZE] * 3
    g = {}
    # the reference's front end on persistent buffers, frame by frame (identical for the three runs: same stream)
    fb = zeros((ROWS, COLS), torch.int16); vm = zeros((3 * ROWS, COLS), torch.float32); nm = torch.zeros_like(vm)
    fe = []
    for d, c in frames:
        ref.bilateral(dev(d.view(np.int16)), fb, ROWS, COLS); ref.vmap(fb, vm, ROWS, COLS, intr); ref.nmap(vm, nm, ROWS, COLS)
        torch.cuda.synchronize()
        fe.append([digest(fb), digest(vm, "values"), digest(nm, "values")])
    g["frontend"] = np.array(fe)

    def vwrap_nonneg(w):
        return [int(x) if x >= 0 else V - ((-int(x)) % V) for x in w]

    for odometry, nframes in ((0, 72), (2, 22), (1, 26)):
        p = f"o{odometry}_"
        cfg = kb.Config.default(vol=V, odometry=odometry)
        mine = kb.Tracker(cfg)
        rt = ref.tracker(refbind.TrackerConfig.from_kt(cfg))
        rp = ref.tracker(refbind.TrackerConfig.from_kt(cfg)) if odometry == 0 else None
        g[p + "trunc"] = np.float32(rt.trunc_dist)
        poses, seq = [], []
        horizon, worst_self = -1, 0.0
        for k in range(nframes):
            d, c = frames[k]
            pm = mine.process_frame(d, c, k); rt.process(d, c, k)
            R, t, gc, w = rt.pose()
            poses.append(np.concatenate([R.reshape(-1), t, gc, w.astype(np.float32)]))
            if rp is not None:
                dp = d
                if k == 1:
                    dp = d.copy(); dp[ROWS // 2, COLS // 2] += 1
                rp.process(dp, c, k)
                _, _, gp, wp = rp.pose()
                self_dev = float(np.abs(gp - gc).max())
                if horizon < 0 and (self_dev > 2e-5 or not (wp == w).all()):
                    horizon = k
                if horizon < 0:
                    worst_self = max(worst_self, self_dev)
            Rinv, tint, wint = mine.last_integrate()
            seq.append(np.concatenate([np.array(pm.voxel_wrap, np.float64), Rinv.reshape(-1).astype(np.float64), tint.astype(np.float64), wint.astype(np.float64)]))
        g[p + "poses"] = np.array(poses, np.float32)
        g[p + "horizon"] = np.int64(horizon); g[p + "worst_self"] = np.float64(worst_self)
        g[p + "slices"] = np.array([(rt.get_slice(i)[1], len(rt.get_slice(i)[0])) for i in range(rt.num_slices())], np.int64).reshape(-1, 2)
        tb_, cb_ = rt.export_volume()
        idx = sample_touched(cb_[..., 3], 20000, 5 + odometry)
        g[p + "ref_vol_idx"] = idx; g[p + "ref_vol_tsdf"] = tb_.reshape(-1)[idx]
        mine.close(); rt.close()
        if rp is not None:
            rp.close()
        # replay of the product's pose sequence with the reference's operators
        seq = np.array(seq)
        g[p + "replay_seq"] = seq
        ts = zeros((V ** 3,), torch.int16); cs = zeros((V ** 3 * 4,), torch.uint8); ref.init_volume(ts, cs)
        fb.zero_(); vm.zero_(); nm.zero_()
        ds = zeros((ROWS, COLS), torch.float32)
        cap = 3 * ROWS * COLS
        ob = zeros((cap * 32,), torch.uint8)
        cur = [0, 0, 0]
        shifts = []
        for k in range(nframes):
            d, c = frames[k]
            dd = dev(d.view(np.int16)); cc = dev(c)
            ref.bilateral(dd, fb, ROWS, COLS); ref.vmap(fb, vm, ROWS, COLS, intr); ref.nmap(vm, nm, ROWS, COLS)
            wa = seq[k, 0:3].astype(np.int64)
            for axis in range(3):
                n = int(wa[axis]) - cur[axis]
                if n == 0:
                    continue
                lo, hi = [0, 0, 0], [V, V, V]
                if n > 0:
                    lo[axis], hi[axis] = 0, n + 1 + cfg.overlap
                elif axis < 2:
                    lo[axis], hi[axis] = V + (n - cfg.overlap), V
                else:
                    lo[axis], hi[axis] = V + (n - cfg.overlap) - 1, V - 1
                box = (lo[0], hi[0], lo[1], hi[1], lo[2], hi[2])
                cnt = ref.extract(ts, vs, ob, cap, vwrap_nonneg(cur), cs, box, 1, cur)
                shifts.append([k, axis, n, cnt])
                g[p + f"shift{len(shifts) - 1}"] = np.array([digest(canon_points(ob[:cnt * 32]))])
                ref.clear(axis, 1 if n < 0 else 0, ts, cs, cur[axis], cur[axis] + n)
                cur[axis] += n
            Rinv = seq[k, 3:12].astype(np.float32).reshape(3, 3); tint = seq[k, 12:15].astype(np.float32); wint = seq[k, 15:18].astype(np.int64)
            ref.integrate(dd, ROWS, COLS, intr, vs, Rinv, tint, float(g[p + "trunc"]), ts, cs, [int(x) for x in wint], cc, nm, 1, ds)
        g[p + "shifts"] = np.array(shifts, np.int64).reshape(-1, 4)
        if odometry == 0:
            wall = int((5.5 - cur[2] * SIZE / V) / (SIZE / V))
            box = (0, V, 0, V, max(0, wall - 15), min(V - 1, wall + 15))
            n_b = ref.extract(ts, vs, ob, cap, vwrap_nonneg(cur), cs, box, 1, cur)
            g[p + "backwall"] = np.array(list(box) + [n_b], np.int64)
            g[p + "backwall_digest"] = np.array([digest(canon_points(ob[:n_b * 32]))])
        torch.cuda.synchronize()
        g[p + "replay_volume"] = np.array([digest(ts), digest(cs)])
        g[p + "replay_touched"] = np.int64((cs.view(-1, 4)[:, 3] != 0).sum().item())
        print(f"baseline odometry={odometry}: horizon {horizon}, {len(shifts)} shifts", flush=True)
        del ts, cs
        torch.cuda.empty_cache()
    return g


def main():
    os.makedirs(OUT, exist_ok=True)
    np.savez_compressed(os.path.join(OUT, "ref_ops_live.npz"), **ops_fixtures())
    print("ops done", flush=True)
    np.savez_compressed(os.path.join(OUT, "ref_tracker_live_256.npz"), **tracker_fixtures())
    print("tracker done", flush=True)
    np.savez_compressed(os.path.join(OUT, "ref_baseline_512.npz"), **baseline_fixtures())
    print("golden written to", OUT)


if __name__ == "__main__":
    main()
