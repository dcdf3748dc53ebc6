"""GPU parity at BASELINE.json's OWN configurations -- 640x480 frames into a 512^3 volume, the default -t 14 shift threshold, all three
odometry modes -- against the reference's CUDA path compiled for VOL=512, recorded on a B200 (tools/make_golden_live.py ->
tests/golden/ref_baseline_512.npz: the reference's poses, its front end and its replay as digests, a sample of its volume).

Three statements per run, each exact or with its tolerance written here:

1. POSES (north_star: <= 1e-4 m / 1e-4 rad).  Frame by frame against the reference tracker (KintinuousTracker.cpp:444-915 restated in
   oracle/kt_host_logic.hpp driving the reference's own kernels).  The tracker is a closed loop (pose -> fused volume -> predicted
   surface -> next pose), so a long sequence can only be compared while the REFERENCE ITSELF is stable; that horizon is measured, not
   assumed: a second reference instance ("ref'") gets the same stream with ONE depth pixel of frame 1 raised by 1 mm (the smallest
   possible input change), and the stable horizon K* is the first frame where ref' has moved more than 2e-5 m away from ref.  On this
   synthetic stream (tools/pose_sensitivity.py, B200): through frame 45 -- three -t 14 shifts -- ref' stays within 6e-6 m of ref and the
   product within 8.1e-6 m; from frame 46 the camera has left the sphere and the cube behind, only the back wall is in view, x (the
   direction of travel) is unconstrained, and at the shift of frame 51 ref' jumps 7.5 cm away from ref (the product 4 cm): no two
   implementations -- nor two runs of the reference on inputs differing by one LSB -- agree beyond that point.
   ICP-only: for every frame k < K* (K* >= 40 is asserted): translation <= 1e-4 m, rotation <= 1e-4 rad, per-frame increment of the
   global position <= 2e-5 m, identical shift events.  For k >= K* only statements 2 and 3 (which do not depend on the reference's
   trajectory) and a gross sanity bound continue.  The photometric modes (-r, -ri) pick discrete correspondences, so the reference
   amplifies 1e-7 differences from the start (DESIGN.md section 5): the first frames are held to 1e-4, later ones to 2e-3; shift
   events identical throughout.

2. VOLUME, EXACT.  The sequence-level TSDF bar cannot be "every voxel within 1 LSB of the reference's run": the two trackers' poses differ
   in the 7th digit, which moves a handful of voxel projections across a pixel boundary, and such a voxel fuses a DIFFERENT pixel's depth
   -- its difference is bounded by |D(u,v) - D(u',v')| / mu per frame (a depth edge: the full TSDF range), not by 1 LSB.  What can be
   demanded exactly is stronger: replay the product's own pose sequence through the operators (bilateral, createVMap/NMap, scaleDepth +
   tsdf23, clearVolume*) on a second volume, frame by frame, and require the product's volume -- TSDF, weights AND colours, every voxel,
   after a real shift -- to be BIT-IDENTICAL to it: 0 LSB.  Pose closeness is statement 1; given the poses, fusion is exact.  The replay
   runs the product's operators; that they are the REFERENCE's is checked on the same sequence: the product's operators replaying the
   pose sequence recorded with the reference must give the reference replay's volume and slabs, digest for digest.

3. SLICES, EXACT.  At each shift the slab the product hands out must equal, as a multiset of 32-byte points, what the reference's
   extractCloudSlice returns on the replayed volume for the same box (extract.cu:325-419; slab boxes from KintinuousTracker.cpp:675-831)
   -- again through the product's extraction operator on the replay, pinned to the reference's by the recorded replay.
"""
import os

import numpy as np
import pytest

from conftest import GOLDEN

pytestmark = pytest.mark.gpu

V = 512
ROWS, COLS = 480, 640
SIZE = 6.0


def rot_angle(Ra, Rb):
    d = Ra.astype(np.float64) @ Rb.astype(np.float64).T
    w = np.array([d[2, 1] - d[1, 2], d[0, 2] - d[2, 0], d[1, 0] - d[0, 1]]) * 0.5
    return float(np.linalg.norm(w))


def canon(pts):
    a = np.ascontiguousarray(pts).view(np.uint64).reshape(len(pts), 4)
    return a[np.lexsort(a.T[::-1])] if len(a) else a


def vwrap_nonneg(w):                      # KintinuousTracker::vWrapCopyUpdate (.cpp:1075-1085)
    return [int(x) if x >= 0 else V - ((-int(x)) % V) for x in w]


def shift_box(axis, n, overlap):          # KintinuousTracker.cpp:680,695 / 735,750 / 790,805 (kt_shift.hpp::shift_box)
    lo, hi = [0, 0, 0], [V, V, V]
    if n > 0:
        lo[axis], hi[axis] = 0, n + 1 + overlap
    elif axis < 2:
        lo[axis], hi[axis] = V + (n - overlap), V
    else:
        lo[axis], hi[axis] = V + (n - overlap) - 1, V - 1
    return (lo[0], hi[0], lo[1], hi[1], lo[2], hi[2])


@pytest.fixture(scope="module")
def frames26():
    """72 frames: the synthetic camera moves 1 cm per frame in +x, a -t 14 shift (16.4 cm at 512^3 / 6 m) happens every ~17 frames; the
    room wall at x = -2.5 m sits 43 voxels inside the volume, so the FOURTH +x shift is the first whose leaving slab contains surface."""
    from concurrent.futures import ProcessPoolExecutor
    from kintinuous_b200 import synth
    try:
        with ProcessPoolExecutor(max_workers=min(16, os.cpu_count() or 1)) as ex:
            return list(ex.map(synth.render, range(72), chunksize=2))
    except Exception:
        return [synth.render(k) for k in range(72)]


def _replay(frames26, seq, cfg, trunc):
    """Fuse a pose sequence with the product's OPERATORS (kt_op_*) on a volume of their own.  Per frame: the front end on persistent
    buffers (Q7 staleness of invalid map pixels), the frame's shift events (slab extraction, clear), integrate.  A row of seq is the
    tracker's voxel wrap after the frame, then Rinv (9), t (3) and wrap (3) of its integration.  Returns the volume, the final signed
    voxel wrap and the extracted slabs as (frame, axis, n, canonical points)."""
    import torch
    import kintinuous_b200 as kb
    from kintinuous_b200 import synth
    from oracle.golden import canon_points
    ops = kb.ops
    intr = np.array(synth.intrinsics(COLS, ROWS), np.float32)
    vs = [SIZE] * 3
    ts = torch.zeros(V ** 3, dtype=torch.int16, device="cuda"); cs = torch.zeros(V ** 3 * 4, dtype=torch.uint8, device="cuda")
    ops.init_volume(ts, cs, V)
    fb = torch.zeros((ROWS, COLS), dtype=torch.int16, device="cuda")
    vm = torch.zeros((3 * ROWS, COLS), dtype=torch.float32, device="cuda"); nm = torch.zeros_like(vm)
    ds = torch.zeros((ROWS, COLS), dtype=torch.float32, device="cuda")
    cap = 3 * ROWS * COLS
    ob = torch.zeros(cap * 32, dtype=torch.uint8, device="cuda")
    cur = [0, 0, 0]                                                     # signed voxelWrap of the replay
    slabs = []
    for k in range(len(seq)):
        d, c = frames26[k]
        dd = torch.from_numpy(d.view(np.int16)).cuda(); cc = torch.from_numpy(c).cuda()
        ops.bilateral(dd, fb, ROWS, COLS); ops.create_vmap(intr, fb, vm, ROWS, COLS); ops.create_nmap(vm, nm, ROWS, COLS)
        for axis in range(3):                                           # x, then y, then z (.cpp:675-831)
            n = int(seq[k][axis]) - cur[axis]
            if n == 0:
                continue
            assert abs(n) == cfg.voxel_shift
            box = shift_box(axis, n, cfg.overlap)
            cnt = ops.extract_slice(ts, vs, V, ob, cap, vwrap_nonneg(cur), cs, box, 1, tuple(cur))
            slabs.append((k, axis, n, canon_points(ob[:cnt * 32])))
            ops.clear_volume(axis, 1 if n < 0 else 0, ts, cs, V, cur[axis], cur[axis] + n)
            cur[axis] += n
        Rinv = seq[k][3:12].astype(np.float32).reshape(3, 3); tint = seq[k][12:15].astype(np.float32); wint = [int(x) for x in seq[k][15:18]]
        assert wint == (vwrap_nonneg(cur) if k > 0 else [0, 0, 0])
        ops.integrate(dd, ROWS, COLS, intr, vs, Rinv, tint, trunc, ts, cs, V, wint, cc, nm, 1, ds)
    torch.cuda.synchronize()
    return ts, cs, cur, slabs


@pytest.mark.parametrize("odometry,nframes", [(0, 72), (2, 22), (1, 26)])
def test_baseline_config_512_live_replay_exact(built, frames26, odometry, nframes):
    import torch
    import kintinuous_b200 as kb
    from oracle.golden import digest, canon_points
    G = np.load(os.path.join(GOLDEN, "ref_baseline_512.npz"))
    p = f"o{odometry}_"
    cfg = kb.Config.default(vol=V, odometry=odometry)                  # voxel_shift 14, overlap 2: BASELINE configs[1] / configs[2]
    assert cfg.voxel_shift == 14 and cfg.overlap == 2
    mine = kb.Tracker(cfg)
    trunc = mine.trunc_dist
    assert abs(trunc - float(G[p + "trunc"])) == 0.0
    # K*: first frame where the reference is unstable under a 1-LSB input change (ref' of the module docstring, recorded)
    horizon = int(G[p + "horizon"]) if odometry == 0 and int(G[p + "horizon"]) >= 0 else None
    if horizon is not None:
        print(f"stable horizon K* = {horizon}: the reference moved > 2e-5 m under a 1-LSB change of one depth pixel of frame 1")
    seq = []
    prev = None
    worst_t = worst_inc = 0.0
    for k in range(nframes):
        d, c = frames26[k]
        pm = mine.process_frame(d, c, k)
        Ra, ta, ga, wa = pm.as_tuple()
        gp = G[p + "poses"][k]
        Rb, tb, gb, wb = gp[:9].reshape(3, 3), gp[9:12], gp[12:15], gp[15:18].astype(np.int32)
        stable = horizon is None or k < horizon
        # ---- 1. poses ----
        dt = float(np.abs(ta - tb).max())
        if odometry == 0:
            if stable:
                assert (wa == wb).all(), (odometry, k, wa, wb)          # identical shift events
                worst_t = max(worst_t, dt)
                assert rot_angle(Ra, Rb) <= 1e-4, (k, rot_angle(Ra, Rb))
                assert dt <= 1e-4 and np.abs(ga - gb).max() <= 1e-4, (k, dt)
                if prev is not None:
                    inc = float(np.abs((ga - prev[0]) - (gb - prev[1])).max()); worst_inc = max(worst_inc, inc)
                    assert inc <= 2e-5, (k, inc)
            else:
                assert np.abs(ga - gb).max() <= 0.25, (k, ga, gb)       # gross sanity only: see the module docstring
        else:
            assert (wa == wb).all(), (odometry, k, wa, wb)
            worst_t = max(worst_t, dt)
            tol = 1e-4 if k < 4 else 2e-3
            assert dt <= tol and rot_angle(Ra, Rb) <= tol, (odometry, k, dt, rot_angle(Ra, Rb))
            assert np.abs(ga - gb).max() <= tol
        prev = (ga.copy(), gb.copy())
        # the product's fused front end (kt_frontend.cu) against the reference's operators on this frame: filtered depth, vertex and
        # normal maps of level 0, bit for bit (NaNs in the same places)
        # (values compared as floats: a normal component that is exactly zero may carry either sign -- x - x and 0 * y products, invisible to
        # every consumer)
        fe = G["frontend"][k]
        assert digest(mine.download_map(4, 0).view(np.int16)) == fe[0], (odometry, k, "bilateral")
        assert digest(mine.download_map(0, 0), "values") == fe[1], (odometry, k, "vmap")
        assert digest(mine.download_map(1, 0), "values") == fe[2], (odometry, k, "nmap")
        Rinv, tint, wint = mine.last_integrate()
        seq.append(np.concatenate([wa, Rinv.reshape(-1), tint, wint]).astype(np.float64))
    seq = np.array(seq)
    # ---- 2./3. replay the product's own pose sequence: its volume and its slices, exactly ----
    ts, cs, cur, slabs = _replay(frames26, seq, cfg, trunc)
    n_slices = len(slabs)
    assert mine.num_slices() == n_slices
    slice_points = 0
    for i, (k, axis, n, want) in enumerate(slabs):
        pts, dim, cam_t = mine.get_slice(i)
        got = canon(pts)
        assert dim == (2 * axis + (0 if n > 0 else 1))
        assert got.shape == want.shape and (got == want).all(), (odometry, k, axis, got.shape, want.shape)
        slice_points += len(pts)
    shifted_frames = [s[0] for s in slabs]
    ta_, ca_ = mine.export_volume()
    tr_ = ts.cpu().numpy().reshape(V, V, V); cr_ = cs.cpu().numpy().reshape(V, V, V, 4)
    touched = int((cr_[..., 3] != 0).sum())
    assert touched > 1_000_000
    bad_t = int((ta_ != tr_).sum()); bad_c = int((ca_ != cr_).any(-1).sum())
    if bad_c:
        idx = np.argwhere((ca_ != cr_).any(-1))
        print("colour mismatches:", bad_c, "first", idx[:8].tolist(), "mine", ca_[tuple(idx[:8].T)].tolist(), "replay", cr_[tuple(idx[:8].T)].tolist(),
              "z range", idx[:, 0].min(), idx[:, 0].max(), "y range", idx[:, 1].min(), idx[:, 1].max(), "x range", idx[:, 2].min(), idx[:, 2].max())
    assert bad_t == 0 and bad_c == 0, (odometry, "voxels differing from the replay", bad_t, bad_c, touched)
    del ta_, ca_, tr_, cr_
    # ---- the replay's operators are the reference's: replaying the recorded pose sequence gives the reference replay's results ----
    rec = G[p + "replay_seq"]
    if not np.array_equal(seq, rec):
        del ts, cs
        torch.cuda.empty_cache()
        ts, cs, cur, slabs = _replay(frames26, rec, cfg, trunc)
    shifts = G[p + "shifts"]
    assert len(slabs) == len(shifts)
    for i, (k, axis, n, pts) in enumerate(slabs):
        assert [k, axis, n, len(pts)] == shifts[i].tolist() and digest(pts) == G[p + f"shift{i}"][0], (odometry, i)
    assert [digest(ts), digest(cs)] == G[p + "replay_volume"].tolist(), (odometry, "replay volume differs from the reference's")
    if odometry == 0:
        n_cmp = n_slices if horizon is None else sum(1 for k in shifted_frames if k < horizon)
    else:
        n_cmp = n_slices
        assert len(G[p + "slices"]) == n_slices
    assert n_slices >= 1, "the run must cross the -t 14 shift threshold"
    if odometry == 0:
        assert horizon is None or horizon >= 40, horizon               # the synthetic scene is well conditioned for at least 40 frames
        assert n_slices >= 4, n_slices
        assert n_cmp >= 3, n_cmp                                        # three shifts inside the stable horizon
        # 3b. the leaving slabs of this stream are mostly free space (the camera moves away from what it saw), so a slab that certainly
        # contains surface is extracted as well: 30 z planes around the room's back wall, on the replayed volume at the final cyclic
        # offset, product operator against the reference's extractCloudSlice -- the same multiset of points.
        wall = int((5.5 - cur[2] * SIZE / V) / (SIZE / V))
        box = (0, V, 0, V, max(0, wall - 15), min(V - 1, wall + 15))
        assert list(box) == G[p + "backwall"][:6].tolist()
        cap = 3 * ROWS * COLS
        oa = torch.zeros(cap * 32, dtype=torch.uint8, device="cuda")
        n_a = kb.ops.extract_slice(ts, [SIZE] * 3, V, oa, cap, vwrap_nonneg(cur), cs, box, 1, tuple(cur))
        n_b = int(G[p + "backwall"][6])
        assert n_a == n_b and n_a > 20000, (n_a, n_b, box)
        assert digest(canon_points(oa[:n_a * 32])) == G[p + "backwall_digest"][0]
        print(f"back-wall slab {box}: {n_a} points, multiset identical to the reference's extraction")
    for i in range(n_cmp):                                              # the reference tracker's own slices: same events, same sizes to 1 %
        a, dim_a, _ = mine.get_slice(i); dim_b, n_b = G[p + "slices"][i]
        assert dim_a == dim_b and abs(len(a) - n_b) <= 0.01 * n_b + 5, (i, len(a), n_b)
    # the reference tracker's own volume, for the record (a seeded sample of its touched voxels): differences come only from its 1e-6
    # different poses
    ta_, _ = mine.export_volume(color=False)
    dlsb = np.abs(ta_.reshape(-1)[G[p + "ref_vol_idx"]].astype(np.int32) - G[p + "ref_vol_tsdf"].astype(np.int32))
    frac = float((dlsb <= 1).mean())
    print(f"cfg odometry={odometry}: stable horizon {horizon}, worst |dt| {worst_t:.3e} m (reference vs its 1-LSB-perturbed self: {float(G[p + 'worst_self']):.3e} m), worst per-frame increment difference {worst_inc:.3e} m; {nframes} frames, shifts at {shifted_frames} ({slice_points} slice points), touched {touched}, replay mismatches 0/0, "
          f"vs reference tracker: {frac:.6f} of sampled touched voxels within 1 LSB, worst {int(dlsb.max())} LSB")
    if odometry == 0 and horizon is None:
        assert frac >= 0.999
    mine.close()


_PI_SCRIPT = r"""
import sys
import numpy as np
import kintinuous_b200 as kb
from kintinuous_b200 import synth
odo = int(sys.argv[1])
trk = kb.Tracker(kb.Config.default(vol=256, odometry=odo))
out = []
for k in range(6):
    d, c = synth.render(k)
    p = trk.process_frame(d, c, k)
    out.append(list(p.R) + list(p.t))
    if k == 1:
        tr = trk.trace()
np.save(sys.argv[2], np.array(out, np.float64)); np.save(sys.argv[2] + ".trace.npy", tr)
"""


@pytest.mark.parametrize("odometry", [0, 1, 2])
def test_per_iteration_path_matches_whole_frame_path_and_golden(built, tmp_path, odometry):
    """The per-iteration kernels (icp_kernel / residual_kernel / rgb_step_kernel, last-CTA solve) are what the tracker falls back to when an
    image does not fit the whole-frame kernels' shared-memory stage.  KT_FORCE_PER_ITERATION=1 takes them on a 640x480 image; poses and
    the per-iteration normal equations must agree with the whole-frame path (different, fixed summation trees: 1e-5) and with the
    reference's golden run."""
    import subprocess
    import sys
    from conftest import ROOT, GOLDEN
    res = {}
    for tag, extra in (("frame", {}), ("iter", {"KT_FORCE_PER_ITERATION": "1"})):
        out = str(tmp_path / f"{tag}_{odometry}.npy")
        env = dict(os.environ, PYTHONPATH=ROOT, **extra)
        r = subprocess.run([sys.executable, "-c", _PI_SCRIPT, str(odometry), out], env=env, capture_output=True, text=True, timeout=900, cwd=ROOT)
        assert r.returncode == 0, r.stderr[-2000:]
        res[tag] = (np.load(out), np.load(out + ".trace.npy"))
    name = {0: "icp", 1: "rgbd", 2: "icp_rgbd"}[odometry]
    g = np.load(os.path.join(GOLDEN, f"tracker_{name}_256.npz"))
    pf, tf = res["frame"]; pi, ti = res["iter"]
    assert tf.shape == ti.shape == g["trace1"].shape
    rel = np.abs(tf[:, :42] - ti[:, :42]).max(1) / np.abs(tf[:, :42]).max(1)
    # first iteration: same inputs, different fixed summation orders; later iterations of the photometric modes re-pick discrete
    # correspondences from poses that differ in the 7th digit (the same sensitivity the reference has, DESIGN.md section 5)
    assert rel[0] < 1e-5, rel[0]
    assert rel.max() < (1e-4 if odometry == 0 else 5e-3), rel.max()
    for k in range(6):
        tol = 1e-4 if (odometry == 0 or k < 4) else 2e-3
        gp = g["poses"][k]
        for p in (pf[k], pi[k]):
            assert np.abs(p[9:12] - gp[9:12]).max() <= tol, (odometry, k)
            assert rot_angle(p[:9].reshape(3, 3), gp[:9].reshape(3, 3)) <= tol
        if odometry == 0 or k < 3:
            assert np.abs(pf[k] - pi[k]).max() <= 2e-5, (odometry, k, np.abs(pf[k] - pi[k]).max())


def test_rgb_only_tracker_vs_golden_reference_cuda(built):
    """odometry = 1 (-r): rgbd_frame_kernel<false>, against the reference's golden run (tests/golden/tracker_rgbd_256.npz)."""
    import kintinuous_b200 as kb
    from kintinuous_b200 import synth
    from conftest import GOLDEN
    g = np.load(os.path.join(GOLDEN, "tracker_rgbd_256.npz"))
    trk = kb.Tracker(kb.Config.default(vol=256, odometry=1))
    for k in range(6):
        d, c = synth.render(k)
        p = trk.process_frame(d, c, k)
        R, t, gc, w = p.as_tuple()
        gp = g["poses"][k]
        tol = 1e-4 if k < 4 else 2e-3
        assert np.abs(t - gp[9:12]).max() <= tol and rot_angle(R, gp[:9].reshape(3, 3)) <= tol, (k, np.abs(t - gp[9:12]).max())
        assert (w == gp[15:18].astype(np.int32)).all()
        if k in (1, 2):
            tr = trk.trace(); gt = g[f"trace{k}"]
            assert len(tr) == len(gt) == 31                             # {10, 7, 7, 7} iterations, RGBDOdometry.cpp:76-107
            if k == 1:
                # photometric normal equations of every iteration (sigma, count in the last two columns are integers: exact)
                # iteration 0 starts from identical inputs: the photometric normal equations agree to summation-order rounding and the
                # integer correspondence count / sigma exactly; later iterations of the RGB-only mode re-pick discrete correspondences
                # from poses that differ in the 7th digit (no ICP term to damp it), so they are held to the correspondence COUNT (1 %)
                rel = np.abs(tr[:, :42] - gt[:, :42]).max(1) / np.abs(gt[:, :42]).max(1)
                assert rel[0] < 1e-5, rel[0]
                assert tr[0, 43] == gt[0, 43] and tr[0, 42] == gt[0, 42]
                assert (np.abs(tr[:, 43] - gt[:, 43]) <= 0.01 * gt[:, 43] + 2).all(), float(np.abs(tr[:, 43] - gt[:, 43]).max())
                assert np.median(rel) < 2e-3, np.median(rel)
    trk.close()


def test_wrap_beyond_one_volume_length(built):
    """voxelWrap grows without bound while the volume travels in +x/+y/+z (vWrapCopy only folds negative values,
    KintinuousTracker.cpp:1075-1085); the reference kernels reduce it with % VOLUME per access.  Offsets > V, a multiple of V, and
    negative ones must address the same storage as their residue: integrate, raycast, extract and clear against the reference's
    kernels on identical buffers, bit-exact (by digest: tests/golden/ref_ops_live.npz)."""
    import torch
    import kintinuous_b200 as kb
    from kintinuous_b200 import synth
    from oracle.golden import digest, canon_points
    live = np.load(os.path.join(GOLDEN, "ref_ops_live.npz"))
    Vs = 256
    ops = kb.ops
    rows, cols = 120, 160
    intr = np.array(synth.intrinsics(cols, rows), np.float32)
    d, c = synth.render(0, cols, rows)
    dd = torch.from_numpy(d.view(np.int16)).cuda(); cc = torch.from_numpy(c).cuda()
    fb = torch.zeros((rows, cols), dtype=torch.int16, device="cuda"); ops.bilateral(dd, fb, rows, cols)
    vm = torch.zeros((3 * rows, cols), dtype=torch.float32, device="cuda"); nm = torch.zeros_like(vm)
    ops.create_vmap(intr, fb, vm, rows, cols); ops.create_nmap(vm, nm, rows, cols)
    assert [digest(fb), digest(vm, "map"), digest(nm, "map")] == live["wrap_inputs"].tolist()      # the reference's input maps
    vs = [SIZE] * 3; trunc = 0.06
    ang = 0.05
    R = np.array([[np.cos(ang), 0, np.sin(ang)], [0, 1, 0], [-np.sin(ang), 0, np.cos(ang)]], np.float32)
    Rinv = np.linalg.inv(R.astype(np.float64)).astype(np.float32)
    t = np.array([3.02, 2.99, 3.01], np.float32)
    for i, wrap in enumerate(((Vs + 88, 2 * Vs + 3, 3 * Vs - 1), (Vs, 2 * Vs, 0), (5 * Vs + 17, 31, Vs + 200))):
        want = live["wrap_steps"][i]
        ta = torch.zeros(Vs ** 3, dtype=torch.int16, device="cuda"); ca = torch.zeros(Vs ** 3 * 4, dtype=torch.uint8, device="cuda")
        ds = torch.zeros((rows, cols), dtype=torch.float32, device="cuda")
        ops.integrate(dd, rows, cols, intr, vs, Rinv, t, trunc, ta, ca, Vs, wrap, cc, nm, 1, ds)
        torch.cuda.synchronize()
        assert int((ca.view(-1, 4)[:, 3] != 0).sum()) > 10000
        assert digest(ta) == want[0] and digest(ca) == want[1], wrap
        va = torch.zeros_like(vm); na = torch.zeros_like(vm); xa = torch.zeros((rows, cols, 4), dtype=torch.uint8, device="cuda")
        ops.raycast(intr, R, t, trunc, vs, ta, Vs, va, na, rows, cols, wrap, xa, ca)
        torch.cuda.synchronize()
        assert digest(va) == want[2] and digest(na) == want[3] and digest(xa) == want[4], wrap
        cap = 400000
        oa = torch.zeros(cap * 32, dtype=torch.uint8, device="cuda")
        box = (0, Vs, 0, Vs, 225, 242)                             # the back wall of the room (z = 5.5 m -> voxel 234)
        real = tuple(int(w) for w in wrap)
        n_a = ops.extract_slice(ta, vs, Vs, oa, cap, wrap, ca, box, 1, real)
        assert n_a == int(live["wrap_counts"][i][0]) and n_a > 100
        assert digest(canon_points(oa[:n_a * 32])) == want[5], wrap
        for axis in range(3):
            ops.clear_volume(axis, 0, ta, ca, Vs, wrap[axis], wrap[axis] + 14)
        torch.cuda.synchronize()
        assert digest(ta) == want[6] and digest(ca) == want[7], ("clear", wrap)


def test_tracker_tracks_ground_truth_across_repeated_shifts(built):
    """Tracker level, small and quick: 40 frames of the synthetic trajectory into a 128^3 volume with a 2-voxel shift threshold (several
    +x shifts): the global camera position keeps following the generator's ground truth across the shifts.  (Offsets beyond one volume
    length are covered exactly, per operator, by test_wrap_beyond_one_volume_length.)"""
    import kintinuous_b200 as kb
    from kintinuous_b200 import synth
    Vs = 128
    rows, cols = 120, 160
    trk = kb.Tracker(kb.Config.default(rows=rows, cols=cols, vol=Vs, odometry=0, voxel_shift=2))
    last = None
    for k in range(40):
        d, c = synth.render(k, cols, rows)
        p = trk.process_frame(d, c, k)
        R, t, gc, w = p.as_tuple()
        Rg, tg = synth.pose(k)
        assert np.abs(gc - tg).max() < 0.03, (k, gc, tg)
        last = w
    assert last[0] >= 6
    trk.close()
