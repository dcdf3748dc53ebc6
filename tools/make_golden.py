#!/usr/bin/env python
"""Generate tests/golden/*.npz by running the REFERENCE's own CUDA operators (oracle/_ref/libkt_ref_256.so, built
from /root/reference by oracle/build_ref.sh) on a B200.  The reference ships no golden vectors (SURVEY.md section 4),
so these fixtures are what pins the CPU oracle: they are outputs of the reference itself on seeded synthetic input.

Run on a GPU box:   python tools/make_golden.py           (writes gpurun_out/golden/*.npz; copy to tests/golden/)
Inputs are re-derivable from kintinuous_b200/synth.py (seed 20260922), so only outputs + a few parameters are stored.
"""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402
import kintinuous_b200 as kb  # noqa: E402
from kintinuous_b200 import synth  # noqa: E402
from oracle import refbind  # noqa: E402

OUT = os.environ.get("KT_GOLDEN_OUT", "gpurun_out/golden")
V = 256
SIZE = 6.0


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def main():
    os.makedirs(OUT, exist_ok=True)
    ref = refbind.RefCuda(V)
    # ---------------- operator fixtures at 160 x 120 ----------------
    rows, cols = 120, 160
    fx, fy, cx, cy = synth.intrinsics(cols, rows)
    intr = np.array([fx, fy, cx, cy], np.float32)
    depth0, rgb0 = synth.render(0, cols, rows)
    depth3, _ = synth.render(12, cols, rows)          # frame 12 at quarter resolution ~ 3 px of motion
    d0 = dev(depth0.view(np.int16)); d3 = dev(depth3.view(np.int16)); c0 = dev(rgb0)
    g = {}
    fb = torch.zeros_like(d0); ref.bilateral(d0, fb, rows, cols); g["bilateral"] = fb.cpu().numpy().view(np.uint16)
    p1 = torch.zeros((rows // 2, cols // 2), dtype=torch.int16, device="cuda"); ref.pyrdown(fb, p1, rows, cols); g["pyrdown"] = p1.cpu().numpy().view(np.uint16)
    vm = torch.zeros((3 * rows, cols), dtype=torch.float32, device="cuda"); nm = torch.zeros_like(vm)
    ref.vmap(fb, vm, rows, cols, intr); ref.nmap(vm, nm, rows, cols)
    g["vmap"] = vm.cpu().numpy(); g["nmap"] = nm.cpu().numpy()
    R0 = np.eye(3, dtype=np.float32); t0 = np.array([3, 3, 3], np.float32)
    ang = 0.03
    R1 = np.array([[np.cos(ang), 0, np.sin(ang)], [0, 1, 0], [-np.sin(ang), 0, np.cos(ang)]], np.float32)
    t1 = t0 + np.array([0.02, -0.01, 0.03], np.float32)
    gv = torch.zeros_like(vm); gn = torch.zeros_like(vm)
    ref.transform_maps(vm, nm, R1, t1, gv, gn, rows, cols); g["transform_v"] = gv.cpu().numpy(); g["transform_n"] = gn.cpu().numpy()
    rv = torch.zeros((3 * rows // 2, cols // 2), dtype=torch.float32, device="cuda"); rn = torch.zeros_like(rv)
    ref.resize_vmap(gv, rv, rows, cols); ref.resize_nmap(gn, rn, rows, cols); g["resize_v"] = rv.cpu().numpy(); g["resize_n"] = rn.cpu().numpy()
    # icp step: model = frame 0 in the volume frame, current = later frame
    mv = torch.zeros_like(vm); mn = torch.zeros_like(vm); ref.transform_maps(vm, nm, R0, t0, mv, mn, rows, cols)
    f3 = torch.zeros_like(d0); ref.bilateral(d3, f3, rows, cols)
    cv = torch.zeros_like(vm); cn = torch.zeros_like(vm); ref.vmap(f3, cv, rows, cols, intr); ref.nmap(cv, cn, rows, cols)
    A, b, res = ref.icp_step(R0, t0, cv, cn, R0, t0, intr, mv, mn, rows, cols)
    g["icp_A"] = A; g["icp_b"] = b; g["icp_res"] = res
    # integrate two frames (second with a wrapped volume and rotated pose), then raycast / extract / clear
    voxel = np.float32(SIZE) / np.float32(V)
    trunc = float(max(np.float32(max(0.01, SIZE / 100.0)), np.float32(2.1) * voxel))
    vs = [SIZE] * 3
    ts = torch.zeros(V ** 3, dtype=torch.int16, device="cuda"); cs = torch.zeros(V ** 3 * 4, dtype=torch.uint8, device="cuda")
    ref.init_volume(ts, cs)
    ds = torch.zeros((rows, cols), dtype=torch.float32, device="cuda")
    wrap = (14, 3, 250)
    ref.integrate(d0, rows, cols, intr, vs, R0, t0, trunc, ts, cs, wrap, c0, nm, 1, ds)
    g["depth_scaled"] = ds.cpu().numpy()
    ref.integrate(d3, rows, cols, intr, vs, np.linalg.inv(R1.astype(np.float64)).astype(np.float32), t1, trunc, ts, cs, wrap, c0, cn, 1, ds)
    torch.cuda.synchronize()
    tsdf = ts.cpu().numpy().reshape(V, V, V); col = cs.cpu().numpy().reshape(V, V, V, 4)
    nz_all = np.flatnonzero(col[..., 3].reshape(-1))              # every voxel ever touched (weight != 0)
    g["vol_touched"] = np.int64(len(nz_all))
    nz = nz_all[::4]                                              # every 4th touched voxel keeps the fixture small
    g["vol_idx"] = nz.astype(np.int32); g["vol_tsdf"] = tsdf.reshape(-1)[nz]; g["vol_color"] = col.reshape(-1, 4)[nz]
    va = torch.zeros_like(vm); na = torch.zeros_like(vm); cc = torch.zeros((rows, cols, 4), dtype=torch.uint8, device="cuda")
    ref.raycast(intr, R1, t1, trunc, vs, ts, va, na, rows, cols, wrap, cc, cs)
    # kept in a file of their own: every golden file stays under 1 MB
    np.savez_compressed(os.path.join(OUT, "ops_160x120_raycast.npz"), raycast_v=va.cpu().numpy(), raycast_n=na.cpu().numpy(), raycast_c=cc.cpu().numpy())
    cap = 400000
    ob = torch.zeros(cap * 32, dtype=torch.uint8, device="cuda")
    real = (14, 3, 250 - V)
    for name, box in {"zslab": (0, V, 0, V, 225, 242), "xplus": (0, 120, 0, V, 0, V), "yslab": (0, V, 180, 197, 0, V)}.items():
        n = ref.extract(ts, vs, ob, cap, wrap, cs, box, 1, real)
        pts = ob.cpu().numpy().view(refbind.POINT_DTYPE)[:n]
        arr = np.ascontiguousarray(pts).view(np.uint64).reshape(n, 4)
        g[f"extract_{name}"] = arr[np.lexsort(arr.T[::-1])] if n else arr
    # clear: sentinel-filled volumes, record which storage planes along the axis end up zero
    sent_t = torch.full((V ** 3,), 7, dtype=torch.int16, device="cuda"); sent_c = torch.full((V ** 3 * 4,), 9, dtype=torch.uint8, device="cuda")
    for axis in range(3):
        for back, (cur, n) in ((0, (14, 14)), (1, (-3, -14)), (0, (40, 16)), (1, (5, -16)), (0, (250, 14)), (1, (3, -14)), (0, (-20, 1)), (1, (0, -2))):
            x, y = sent_t.clone(), sent_c.clone()
            ref.clear(axis, back, x, y, cur, cur + n); torch.cuda.synchronize()
            zt = (x.view(V, V, V) == 0); zc = (y.view(V, V, V, 4) == 0).all(-1)
            assert bool((zt == zc).all())
            ax = {0: (0, 1), 1: (0, 2), 2: (1, 2)}[axis]          # tensor dims are (z, y, x)
            full = zt.all(dim=ax[1]).all(dim=ax[0]); part = zt.any(dim=ax[1]).any(dim=ax[0])
            assert bool((full == part).all())                     # planes are cleared completely or not at all
            g[f"clear_a{axis}_b{back}_c{cur}_n{n}"] = torch.nonzero(full).flatten().cpu().numpy().astype(np.int32)
    g["params"] = np.array([rows, cols, V, SIZE, trunc, ang], np.float64)
    np.savez_compressed(os.path.join(OUT, "ops_160x120.npz"), **g)

    # ---------------- RGB-D operator fixtures ----------------
    h = {}
    depth1, rgb1 = synth.render(4, cols, rows)
    d1 = dev(depth1.view(np.int16)); c1 = dev(rgb1)
    fd0 = torch.zeros((rows, cols), dtype=torch.float32, device="cuda"); fd1 = torch.zeros_like(fd0)
    ref.short_depth_to_metres(d0, fd0, rows, cols, 6000); ref.short_depth_to_metres(d1, fd1, rows, cols, 6000)
    i0 = torch.zeros((rows, cols), dtype=torch.uint8, device="cuda"); i1 = torch.zeros_like(i0)
    ref.bgr_to_intensity(c0, i0, rows, cols); ref.bgr_to_intensity(c1, i1, rows, cols)
    h["depth_f"] = fd1.cpu().numpy(); h["intensity"] = i1.cpu().numpy()
    pf = torch.zeros((rows // 2, cols // 2), dtype=torch.float32, device="cuda"); ref.pyrdown_gauss_f(fd1, pf, rows, cols); h["pyr_f"] = pf.cpu().numpy()
    pu = torch.zeros((rows // 2, cols // 2), dtype=torch.uint8, device="cuda"); ref.pyrdown_uchar_gauss(i1, pu, rows, cols); torch.cuda.synchronize(); h["pyr_u"] = pu.cpu().numpy()
    dx = torch.zeros((rows, cols), dtype=torch.int16, device="cuda"); dy = torch.zeros_like(dx)
    ref.derivative_images(i1, dx, dy, rows, cols); h["dIdx"] = dx.cpu().numpy(); h["dIdy"] = dy.cpu().numpy()
    cl = torch.zeros((rows, cols, 3), dtype=torch.float32, device="cuda")
    kd = np.array([float(np.float32(fx)), float(np.float32(fy)), float(np.float32(cx)), float(np.float32(cy))], np.float64)
    ref.project_to_point_cloud(fd0, cl, rows, cols, kd, 0); h["cloud"] = cl.cpu().numpy()
    K = np.array([[kd[0], 0, kd[2]], [0, kd[1], kd[3]], [0, 0, 1]])
    Rw = np.array([[np.cos(0.004), 0, np.sin(0.004)], [0, 1, 0], [-np.sin(0.004), 0, np.cos(0.004)]])
    tw = np.array([-0.01, 0.001, -0.004])
    krk = (K @ Rw @ np.linalg.inv(K)).astype(np.float32); kt = (K @ tw).astype(np.float32)
    cor = torch.zeros(rows * cols * 16, dtype=torch.uint8, device="cuda")
    sigma, count = ref.rgb_residual(float(3.0 ** 2 / (1 / 8.0) ** 2), dx, dy, fd0, fd1, i0, i1, cor, rows, cols, 0.07, kt, krk)
    h["corres"] = cor.cpu().numpy().reshape(rows * cols, 16); h["sigma_count"] = np.array([sigma, count], np.int64)
    h["krk"] = krk; h["kt"] = kt
    sig = float(np.sqrt(count))
    A, b = ref.rgb_step(cor, sig, cl, kd[0], kd[1], dx, dy, 1 / 8.0, rows, cols)
    h["rgb_A"] = A; h["rgb_b"] = b
    np.savez_compressed(os.path.join(OUT, "rgbd_160x120.npz"), **h)

    # ---------------- tracker fixtures: 640x480 into 256^3, three odometry modes + a shifting run ----------------
    rows, cols = 480, 640
    frames = [synth.render(k, cols, rows) for k in range(10)]
    # NOTE the shifting run goes FIRST: the reference's extract kernel publishes its point count from the first warp of the
    # last CTA while other warps may still be appending (extract.cu:290-305), so a full-volume extraction (finalise) can leak a
    # few counts into the NEXT extractCloudSlice call of the same process (observed: 71 phantom points).  DESIGN.md, R1.
    for name, kw in {"icp_shift": dict(odometry=0, voxel_shift=2), "icp": dict(odometry=0), "rgbd": dict(odometry=1), "icp_rgbd": dict(odometry=2)}.items():
        cfg = kb.Config.default(rows=rows, cols=cols, vol=V, **kw)
        rt = ref.tracker(refbind.TrackerConfig.from_kt(cfg))
        poses = []; traces = []
        for k, (d, c) in enumerate(frames):
            rt.process(d, c, k)
            R, t, gcam, w = rt.pose()
            poses.append(np.concatenate([R.reshape(-1), t, gcam, w.astype(np.float32)]))
            if k in (1, 2):
                traces.append(rt.trace())
        ts_, cs_ = rt.export_volume()
        touched = np.flatnonzero(cs_[..., 3].reshape(-1))
        rt.finalise()
        nsl = rt.num_slices()
        sl = [(rt.get_slice(i)[1], len(rt.get_slice(i)[0])) for i in range(nsl)]
        np.savez_compressed(os.path.join(OUT, f"tracker_{name}_256.npz"), poses=np.array(poses, np.float32), trace1=traces[0], trace2=traces[1],
                            touched=np.int64(len(touched)), tsdf_hist=np.bincount((ts_.reshape(-1)[touched].astype(np.int32) + 32768) >> 8, minlength=256),
                            weight_hist=np.bincount(cs_[..., 3].reshape(-1)[touched], minlength=256), slices=np.array(sl, np.int64).reshape(-1, 2))
        print(name, "done; slices", sl, flush=True)
        rt.close()
    print("golden written to", OUT)


if __name__ == "__main__":
    main()
