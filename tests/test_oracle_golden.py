"""Pin the CPU oracle (oracle/kt_oracle_cpu.cpp) against golden vectors produced by the REFERENCE's own CUDA operators
on a B200 (tools/make_golden.py -> tests/golden/*.npz).  The reference ships no fixtures of its own (SURVEY.md section 4).

Tolerances (stated per test): the oracle uses IEEE division / sqrt / expf where the reference's build uses the approximate
instructions (--prec-div=false --prec-sqrt=false, __expf, rsqrtf), so floating-point maps agree to a few ulp, integer images
can differ by 1 LSB at rounding boundaries on a small fraction of pixels, and a reduction differs by its summation order."""
import ctypes as C
import os

import numpy as np
import pytest

from conftest import GOLDEN


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _f(a):
    return np.ascontiguousarray(np.asarray(a, np.float32).reshape(-1))


@pytest.fixture(scope="module")
def G():
    p = os.path.join(GOLDEN, "ops_160x120.npz")
    if not os.path.exists(p):
        pytest.skip("tests/golden/ops_160x120.npz missing (generate with tools/make_golden.py on a GPU box)")
    return np.load(p)


@pytest.fixture(scope="module")
def scene():
    from kintinuous_b200 import synth
    rows, cols = 120, 160
    intr = np.array(synth.intrinsics(cols, rows), np.float32)
    d0, c0 = synth.render(0, cols, rows)
    d3, _ = synth.render(12, cols, rows)
    ang = 0.03
    R0 = np.eye(3, dtype=np.float32); t0 = np.array([3, 3, 3], np.float32)
    R1 = np.array([[np.cos(ang), 0, np.sin(ang)], [0, 1, 0], [-np.sin(ang), 0, np.cos(ang)]], np.float32)
    t1 = t0 + np.array([0.02, -0.01, 0.03], np.float32)
    return dict(rows=rows, cols=cols, intr=intr, d0=d0, c0=c0, d3=d3, R0=R0, t0=t0, R1=R1, t1=t1)


def map_close(a, b, rows, cols, rtol, atol, max_mask_mismatch=0):
    a = a.reshape(3, rows, cols); b = b.reshape(3, rows, cols)
    na, nb = np.isnan(a[0]), np.isnan(b[0])
    assert int((na != nb).sum()) <= max_mask_mismatch
    ok = ~na & ~nb
    assert np.allclose(a[:, ok], b[:, ok], rtol=rtol, atol=atol), float(np.abs(a[:, ok] - b[:, ok]).max())


def test_bilateral_and_pyrdown(cpu_oracle, G, scene):
    rows, cols = scene["rows"], scene["cols"]
    out = np.zeros((rows, cols), np.uint16)
    cpu_oracle.lib.ktoracle_bilateral(_p(scene["d0"]), _p(out), rows, cols)
    d = np.abs(out.astype(int) - G["bilateral"].astype(int))
    assert d.max() <= 1 and (d != 0).mean() < 2e-3            # 1 mm at a rounding tie, on < 0.2 % of pixels
    p = np.zeros((rows // 2, cols // 2), np.uint16)
    cpu_oracle.lib.ktoracle_pyrdown(_p(G["bilateral"]), _p(p), rows, cols)
    d = np.abs(p.astype(int) - G["pyrdown"].astype(int))
    assert d.max() <= 1 and (d != 0).mean() < 2e-3


def test_vertex_normal_maps(cpu_oracle, G, scene):
    rows, cols = scene["rows"], scene["cols"]
    fb = np.ascontiguousarray(G["bilateral"])
    vm = np.zeros((3 * rows, cols), np.float32); nm = np.zeros_like(vm)
    cpu_oracle.lib.ktoracle_vmap(_p(fb), _p(vm), rows, cols, _p(scene["intr"]))
    cpu_oracle.lib.ktoracle_nmap(_p(np.ascontiguousarray(G["vmap"])), _p(nm), rows, cols)
    map_close(vm, G["vmap"], rows, cols, rtol=2e-6, atol=1e-7)
    map_close(nm, G["nmap"], rows, cols, rtol=0, atol=2e-5)   # rsqrtf: 2 ulp of a unit vector component, amplified by flat cross products
    gv = np.zeros_like(vm); gn = np.zeros_like(vm)
    cpu_oracle.lib.ktoracle_transform_maps(_p(np.ascontiguousarray(G["vmap"])), _p(np.ascontiguousarray(G["nmap"])), _p(_f(scene["R1"])), _p(_f(scene["t1"])), _p(gv), _p(gn), rows, cols)
    map_close(gv, G["transform_v"], rows, cols, rtol=1e-6, atol=1e-6)
    map_close(gn, G["transform_n"], rows, cols, rtol=0, atol=1e-6)
    rv = np.zeros((3 * rows // 2, cols // 2), np.float32); rn = np.zeros_like(rv)
    cpu_oracle.lib.ktoracle_resize_vmap(_p(np.ascontiguousarray(G["transform_v"])), _p(rv), rows, cols)
    cpu_oracle.lib.ktoracle_resize_nmap(_p(np.ascontiguousarray(G["transform_n"])), _p(rn), rows, cols)
    map_close(rv, G["resize_v"], rows // 2, cols // 2, rtol=1e-6, atol=1e-6)
    map_close(rn, G["resize_n"], rows // 2, cols // 2, rtol=0, atol=1e-6)


def test_icp_normal_equations(cpu_oracle, G, scene):
    """Inputs rebuilt with the oracle itself from the golden filtered depth; A, b within 1e-4 relative of the reference's
    float tree reduction (summation order + approximate division in the projection)."""
    rows, cols = scene["rows"], scene["cols"]
    lib = cpu_oracle.lib
    intr = scene["intr"]
    vm = np.ascontiguousarray(G["vmap"]); nm = np.ascontiguousarray(G["nmap"])
    mv = np.zeros_like(vm); mn = np.zeros_like(vm)
    lib.ktoracle_transform_maps(_p(vm), _p(nm), _p(_f(scene["R0"])), _p(_f(scene["t0"])), _p(mv), _p(mn), rows, cols)
    f3 = np.zeros((rows, cols), np.uint16); lib.ktoracle_bilateral(_p(scene["d3"]), _p(f3), rows, cols)
    cv = np.zeros_like(vm); cn = np.zeros_like(vm)
    lib.ktoracle_vmap(_p(f3), _p(cv), rows, cols, _p(intr)); lib.ktoracle_nmap(_p(cv), _p(cn), rows, cols)
    A = np.zeros(36, np.float32); b = np.zeros(6, np.float32); res = np.zeros(2, np.float32)
    lib.ktoracle_icp_step(_p(_f(scene["R0"])), _p(_f(scene["t0"])), _p(cv), _p(cn), _p(_f(scene["R0"])), _p(_f(scene["t0"])), _p(intr), _p(mv), _p(mn), rows, cols,
                          C.c_float(0.10), C.c_float(float(np.sin(np.float32(20.0) * np.float32(3.14159254) / np.float32(180.0)))), _p(A), _p(b), _p(res))
    gA, gb, gres = G["icp_A"], G["icp_b"], G["icp_res"]
    assert abs(res[1] - gres[1]) <= 0.002 * gres[1]                       # inlier count: threshold ties on a few pixels
    assert np.abs(A.reshape(6, 6) - gA).max() <= 2e-3 * np.abs(gA).max()
    assert np.abs(b - gb).max() <= 2e-3 * np.abs(gb).max() + 1e-3


def _integrate_twice(lib, scene, G, V, trunc):
    rows, cols = scene["rows"], scene["cols"]
    vs = _f([6.0] * 3)
    tsdf = np.zeros(V ** 3, np.int16); color = np.zeros(V ** 3 * 4, np.uint8)
    wrap = np.array([14, 3, 250], np.int32)
    ds = np.zeros((rows, cols), np.float32)
    nm = np.ascontiguousarray(G["nmap"])
    lib.ktoracle_integrate(_p(scene["d0"]), rows, cols, _p(scene["intr"]), _p(vs), _p(_f(scene["R0"])), _p(_f(scene["t0"])), C.c_float(trunc), _p(tsdf), _p(color), V, _p(wrap),
                           _p(np.ascontiguousarray(scene["c0"])), _p(nm), 1, _p(ds))
    ds0 = ds.copy()
    # second frame: current normals from the oracle's own pipeline on frame 12
    f3 = np.zeros((rows, cols), np.uint16); lib.ktoracle_bilateral(_p(scene["d3"]), _p(f3), rows, cols)
    cv = np.zeros((3 * rows, cols), np.float32); cn = np.zeros_like(cv)
    lib.ktoracle_vmap(_p(f3), _p(cv), rows, cols, _p(scene["intr"])); lib.ktoracle_nmap(_p(cv), _p(cn), rows, cols)
    Rinv = np.linalg.inv(scene["R1"].astype(np.float64)).astype(np.float32)
    lib.ktoracle_integrate(_p(scene["d3"]), rows, cols, _p(scene["intr"]), _p(vs), _p(_f(Rinv)), _p(_f(scene["t1"])), C.c_float(trunc), _p(tsdf), _p(color), V, _p(wrap),
                           _p(np.ascontiguousarray(scene["c0"])), _p(cn), 1, _p(ds))
    return tsdf, color, ds0, wrap, vs


def test_integrate_raycast_extract(cpu_oracle, G, scene):
    lib = cpu_oracle.lib
    rows, cols = scene["rows"], scene["cols"]
    V = int(G["params"][2]); trunc = float(G["params"][4])
    tsdf, color, ds0, wrap, vs = _integrate_twice(lib, scene, G, V, trunc)
    assert np.allclose(ds0, G["depth_scaled"], rtol=3e-7, atol=0)          # scaleDepth: sqrt.approx / div.approx vs IEEE
    touched = np.flatnonzero(color.reshape(-1, 4)[:, 3])
    assert abs(len(touched) - int(G["vol_touched"])) <= 2e-4 * int(G["vol_touched"])
    idx = G["vol_idx"]
    dt = np.abs(tsdf[idx].astype(np.int32) - G["vol_tsdf"].astype(np.int32))
    # TSDF: <= 1 LSB on >= 99.9 % of the reference's touched voxels (a voxel whose projection lands on a pixel boundary may read
    # the neighbouring depth pixel under IEEE vs approximate arithmetic)
    assert (dt <= 1).mean() >= 0.999, float((dt <= 1).mean())
    dw = color.reshape(-1, 4)[idx, 3].astype(int) - G["vol_color"][:, 3].astype(int)
    assert (dw == 0).mean() >= 0.9995
    drgb = np.abs(color.reshape(-1, 4)[idx, :3].astype(int) - G["vol_color"][:, :3].astype(int)).max(1)
    assert (drgb <= 1).mean() >= 0.995

    # raycast the ORACLE volume and compare with the reference's raycast of the REFERENCE volume
    va = np.zeros((3 * rows, cols), np.float32); na = np.zeros_like(va); cc = np.zeros((rows, cols, 4), np.uint8)
    lib.ktoracle_raycast(_p(scene["intr"]), _p(_f(scene["R1"])), _p(_f(scene["t1"])), C.c_float(trunc), _p(vs), _p(tsdf), V, _p(va), _p(na), rows, cols, _p(wrap), _p(cc), _p(color))
    GR = np.load(os.path.join(GOLDEN, "ops_160x120_raycast.npz"))
    gv = GR["raycast_v"].reshape(3, rows, cols); v = va.reshape(3, rows, cols)
    ma, mb = np.isnan(v[0]), np.isnan(gv[0])
    assert (ma != mb).mean() < 2e-3
    ok = ~ma & ~mb
    err = np.abs(v[:, ok] - gv[:, ok]).max(0)
    # sub-0.1 mm, except the rare ray whose zero crossing is bracketed at a different march step or whose
    # interpolation denominator (F(t+dt) - F(t)) is nearly zero
    assert np.quantile(err, 0.999) < 1e-4 and (err > 1e-3).mean() < 1e-3
    gn = GR["raycast_n"].reshape(3, rows, cols); n = na.reshape(3, rows, cols)
    okn = ~np.isnan(n[0]) & ~np.isnan(gn[0])
    assert np.quantile(np.abs(n[:, okn] - gn[:, okn]).max(0), 0.99) < 2e-3

    # extraction: same multiset of points up to the volume differences above (compare counts and point sets by position)
    cap = 400000
    out = np.zeros(cap * 32, np.uint8)
    real = np.array([14, 3, 250 - V], np.int32)
    for name, box in {"zslab": (0, V, 0, V, 225, 242), "xplus": (0, 120, 0, V, 0, V), "yslab": (0, V, 180, 197, 0, V)}.items():
        key = f"extract_{name}"
        if key not in G.files:
            continue
        lib.ktoracle_extract.restype = C.c_size_t
        n_pts = lib.ktoracle_extract(_p(tsdf), _p(vs), V, _p(out), C.c_size_t(cap), _p(wrap), _p(color), *box, 1, _p(real))
        g = G[key]
        assert abs(int(n_pts) - len(g)) <= max(3, 0.002 * len(g)), (name, n_pts, len(g))


def test_clear_planes(cpu_oracle, G):
    """clearVolume{X,Y,Z}[Back]: exactly the storage planes the reference's kernels zero (including the launch-width quirk, Q13)."""
    lib = cpu_oracle.lib
    V = 64                                                        # plane sets are compared modulo the volume side
    keys = [k for k in G.files if k.startswith("clear_")]
    if not keys or all(len(G[k]) == 0 for k in keys):
        pytest.skip("golden file predates the sentinel clear fixtures")
    Vg = int(G["params"][2])
    for k in keys:
        _, a, b, c, n = k.split("_")
        axis, back, cur, nn = int(a[1:]), int(b[1:]), int(c[1:]), int(n[1:])
        t = np.full(Vg ** 3, 7, np.int16); col = np.full(Vg ** 3 * 4, 9, np.uint8)
        lib.ktoracle_clear(axis, back, _p(t), _p(col), Vg, cur, cur + nn)
        z = (t.reshape(Vg, Vg, Vg) == 0)
        ax = {0: (0, 1), 1: (0, 2), 2: (1, 2)}[axis]
        planes = np.flatnonzero(z.all(axis=ax))
        assert planes.tolist() == G[k].tolist(), (k, planes.tolist(), G[k].tolist())
        assert int(z.sum()) == len(planes) * Vg * Vg
    assert V == 64


@pytest.mark.parametrize("name,odometry,kw", [("icp", 0, {}), ("icp_rgbd", 2, {}), ("icp_shift", 0, {"voxel_shift": 2})])
def test_tracker_poses_against_reference_cuda(cpu_oracle, name, odometry, kw):
    """CPU oracle tracker (same host logic, CPU kernels) vs the reference-CUDA tracker's recorded poses: 640x480 into 256^3.
    Bar: BASELINE.json north_star -- pose <= 1e-4 m / 1e-4 rad per frame."""
    p = os.path.join(GOLDEN, f"tracker_{name}_256.npz")
    if not os.path.exists(p):
        pytest.skip("golden tracker file missing")
    g = np.load(p)
    import kintinuous_b200 as kb
    from kintinuous_b200 import synth
    from oracle import refbind
    n = 5
    cfg = kb.Config.default(rows=480, cols=640, vol=256, odometry=odometry, **kw)
    t = cpu_oracle.tracker(refbind.TrackerConfig.from_kt(cfg))
    for k in range(n):
        d, c = synth.render(k)
        t.process(d, c, k)
        R, tt, gc, w = t.pose()
        gp = g["poses"][k]
        assert np.abs(R.reshape(-1) - gp[:9]).max() <= 1e-4, (k, np.abs(R.reshape(-1) - gp[:9]).max())
        assert np.abs(tt - gp[9:12]).max() <= 1e-4, (k, np.abs(tt - gp[9:12]).max())
        assert (w == gp[15:18].astype(np.int32)).all()
        if k == 1:
            tr = t.trace(); gt = g["trace1"]
            assert len(tr) == len(gt)
            rel = np.abs(tr[:, :42] - gt[:, :42]).max(1) / np.abs(gt[:, :42]).max(1)
            assert rel.max() < 5e-3, rel.max()
    t.close()
