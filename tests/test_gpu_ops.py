"""GPU parity tests, operator level, through the C ABI (kt_op_*): the product's sm_100a kernels vs the golden vectors the
reference's OWN CUDA operators produced on the same inputs -- arrays (tests/golden/ops_160x120*.npz) and, where a bit-exact result is
too large to store, its digest (tests/golden/ref_ops_live.npz, tools/make_golden_live.py, oracle/golden.py).
Bar: bit-exact for every per-pixel / per-voxel operator (same nvcc numerics flags, same expression order); 1e-5 relative for the
29-float normal-equation reduction (different, deterministic summation tree)."""
import os

import numpy as np
import pytest

from conftest import GOLDEN

pytestmark = pytest.mark.gpu

V = 256
SIZE = 6.0


@pytest.fixture(scope="module")
def env(built):
    import torch
    import kintinuous_b200 as kb
    from kintinuous_b200 import synth
    assert kb.cuda_available(), "GPU test on a box without CUDA"
    g = np.load(os.path.join(GOLDEN, "ops_160x120.npz"))
    live = np.load(os.path.join(GOLDEN, "ref_ops_live.npz"))
    rows, cols = 120, 160
    intr = np.array(synth.intrinsics(cols, rows), np.float32)
    d0, c0 = synth.render(0, cols, rows)
    d3, _ = synth.render(12, cols, rows)
    ang = 0.03
    R0 = np.eye(3, dtype=np.float32); t0 = np.array([3, 3, 3], np.float32)
    R1 = np.array([[np.cos(ang), 0, np.sin(ang)], [0, 1, 0], [-np.sin(ang), 0, np.cos(ang)]], np.float32)
    t1 = t0 + np.array([0.02, -0.01, 0.03], np.float32)
    voxel = np.float32(SIZE) / np.float32(V)
    trunc = float(max(np.float32(max(0.01, SIZE / 100.0)), np.float32(2.1) * voxel))
    return dict(torch=torch, kb=kb, ops=kb.ops, g=g, live=live, rows=rows, cols=cols, intr=intr, d0=d0, c0=c0, d3=d3, R0=R0, t0=t0, R1=R1, t1=t1, trunc=trunc)


def dev(e, a):
    return e["torch"].from_numpy(np.ascontiguousarray(a)).cuda()


def zeros(e, shape, dtype):
    return e["torch"].zeros(shape, dtype=dtype, device="cuda")


def same_map(a, b, rows, cols):
    a = a.reshape(3, rows, cols); b = b.reshape(3, rows, cols)
    na, nb = np.isnan(a[0]), np.isnan(b[0])
    assert (na == nb).all()
    ok = ~na
    assert (a[:, ok].view(np.uint32) == b[:, ok].view(np.uint32)).all(), float(np.abs(a[:, ok] - b[:, ok]).max())


def test_pyramid_bit_exact_vs_golden(env):
    e = env; t = e["torch"]; rows, cols, g = e["rows"], e["cols"], e["g"]
    d0 = dev(e, e["d0"].view(np.int16))
    fb = zeros(e, (rows, cols), t.int16); e["ops"].bilateral(d0, fb, rows, cols)
    assert (fb.cpu().numpy().view(np.uint16) == g["bilateral"]).all()
    p1 = zeros(e, (rows // 2, cols // 2), t.int16); e["ops"].pyrdown(fb, p1, rows, cols)
    assert (p1.cpu().numpy().view(np.uint16) == g["pyrdown"]).all()
    vm = zeros(e, (3 * rows, cols), t.float32); nm = zeros(e, (3 * rows, cols), t.float32)
    e["ops"].create_maps(e["intr"], fb, vm, nm, rows, cols)
    same_map(vm.cpu().numpy(), g["vmap"], rows, cols); same_map(nm.cpu().numpy(), g["nmap"], rows, cols)
    v2 = zeros(e, (3 * rows, cols), t.float32); n2 = zeros(e, (3 * rows, cols), t.float32)
    e["ops"].create_vmap(e["intr"], fb, v2, rows, cols); e["ops"].create_nmap(v2, n2, rows, cols)
    same_map(v2.cpu().numpy(), g["vmap"], rows, cols); same_map(n2.cpu().numpy(), g["nmap"], rows, cols)
    gv = zeros(e, (3 * rows, cols), t.float32); gn = zeros(e, (3 * rows, cols), t.float32)
    e["ops"].transform_maps(vm, nm, e["R1"], e["t1"], gv, gn, rows, cols)
    same_map(gv.cpu().numpy(), g["transform_v"], rows, cols); same_map(gn.cpu().numpy(), g["transform_n"], rows, cols)
    rv = zeros(e, (3 * rows // 2, cols // 2), t.float32); rn = zeros(e, (3 * rows // 2, cols // 2), t.float32)
    e["ops"].resize_vmap(gv, rv, rows, cols); e["ops"].resize_nmap(gn, rn, rows, cols)
    same_map(rv.cpu().numpy(), g["resize_v"], rows // 2, cols // 2); same_map(rn.cpu().numpy(), g["resize_n"], rows // 2, cols // 2)


def test_bilateral_full_resolution_vs_reference(env):
    """640x480 exercises the interior (unrolled) and border code paths of the bilateral / pyrDown kernels."""
    e = env; t = e["torch"]
    from kintinuous_b200 import synth
    from oracle.golden import digest
    want = e["live"]["bilateral_full"]
    rng = np.random.default_rng(20260922)
    inputs = [synth.render(k)[0] for k in (0, 7)]
    noisy = inputs[0].astype(np.int64) + rng.integers(-40, 41, inputs[0].shape)          # sensor-like noise: weights far from 0 and 1
    noisy[rng.random(noisy.shape) < 0.05] = 0                                              # holes
    inputs.append(np.clip(noisy, 0, 65535).astype(np.uint16))
    far = inputs[0].copy()                                                                 # depths whose squared difference overflows
    far[100:140, 200:300] = 65535; far[300:330, 10:50] = 50000; far[0:8, 600:640] = 47000  # int32 in the reference (kept bit-exact)
    inputs.append(far)
    inputs.append(rng.integers(0, 65536, inputs[0].shape).astype(np.uint16))              # white noise over the whole u16 range
    for i, d in enumerate(inputs):
        dd = dev(e, d.view(np.int16))
        a = zeros(e, (480, 640), t.int16)
        e["ops"].bilateral(dd, a, 480, 640)
        assert digest(a) == want[i, 0], i
        src = a
        for l in range(1, 4):
            r, c = 480 >> (l - 1), 640 >> (l - 1)
            pa = zeros(e, (r // 2, c // 2), t.int16)
            e["ops"].pyrdown(src, pa, r, c)
            assert digest(pa) == want[i, l], (i, l)
            src = pa


def _model_and_current(e):
    t = e["torch"]; rows, cols, g = e["rows"], e["cols"], e["g"]
    vm = dev(e, g["vmap"]); nm = dev(e, g["nmap"])
    mv = zeros(e, (3 * rows, cols), t.float32); mn = zeros(e, (3 * rows, cols), t.float32)
    e["ops"].transform_maps(vm, nm, e["R0"], e["t0"], mv, mn, rows, cols)
    d3 = dev(e, e["d3"].view(np.int16))
    f3 = zeros(e, (rows, cols), t.int16); e["ops"].bilateral(d3, f3, rows, cols)
    cv = zeros(e, (3 * rows, cols), t.float32); cn = zeros(e, (3 * rows, cols), t.float32)
    e["ops"].create_maps(e["intr"], f3, cv, cn, rows, cols)
    return vm, nm, mv, mn, cv, cn, d3


def test_icp_step_vs_golden(env):
    e = env; g = e["g"]
    vm, nm, mv, mn, cv, cn, _ = _model_and_current(e)
    A, b, res = e["ops"].icp_step(e["R0"], e["t0"], cv, cn, e["R0"], e["t0"], e["intr"], mv, mn, e["rows"], e["cols"])
    assert res[1] == g["icp_res"][1]                                        # identical inlier set
    assert np.abs(A - g["icp_A"]).max() <= 1e-5 * np.abs(g["icp_A"]).max()
    assert np.abs(b - g["icp_b"]).max() <= 1e-5 * np.abs(g["icp_b"]).max()
    assert abs(res[0] - g["icp_res"][0]) <= 1e-5 * g["icp_res"][0]
    A2, b2, res2 = e["ops"].icp_step(e["R0"], e["t0"], cv, cn, e["R0"], e["t0"], e["intr"], mv, mn, e["rows"], e["cols"])
    assert (A == A2).all() and (b == b2).all()                              # deterministic reduction tree


def _integrated_volume(e):
    t = e["torch"]; rows, cols, g = e["rows"], e["cols"], e["g"]
    vm, nm, mv, mn, cv, cn, d3 = _model_and_current(e)
    d0 = dev(e, e["d0"].view(np.int16)); c0 = dev(e, e["c0"])
    ts = zeros(e, (V ** 3,), t.int16); cs = zeros(e, (V ** 3 * 4,), t.uint8)
    e["ops"].init_volume(ts, cs, V)
    ds = zeros(e, (rows, cols), t.float32)
    wrap = (14, 3, 250)
    vs = [SIZE] * 3
    e["ops"].integrate(d0, rows, cols, e["intr"], vs, e["R0"], e["t0"], e["trunc"], ts, cs, V, wrap, c0, nm, 1, ds)
    ds0 = ds.cpu().numpy().copy()
    e["ops"].integrate(d3, rows, cols, e["intr"], vs, np.linalg.inv(e["R1"].astype(np.float64)).astype(np.float32), e["t1"], e["trunc"], ts, cs, V, wrap, c0, cn, 1, ds)
    return ts, cs, ds0, wrap, vs


def test_integrate_raycast_extract_clear_bit_exact_vs_golden(env):
    e = env; t = e["torch"]; rows, cols, g = e["rows"], e["cols"], e["g"]
    ts, cs, ds0, wrap, vs = _integrated_volume(e)
    assert (ds0.view(np.uint32) == g["depth_scaled"].view(np.uint32)).all()
    tsdf = ts.cpu().numpy(); col = cs.cpu().numpy().reshape(-1, 4)
    assert int((col[:, 3] != 0).sum()) == int(g["vol_touched"])
    idx = g["vol_idx"]
    assert (tsdf[idx] == g["vol_tsdf"]).all()                               # TSDF: 0 LSB on every sampled voxel
    assert (col[idx] == g["vol_color"]).all()                               # colour + weight
    va = zeros(e, (3 * rows, cols), t.float32); na = zeros(e, (3 * rows, cols), t.float32); cc = zeros(e, (rows, cols, 4), t.uint8)
    e["ops"].raycast(e["intr"], e["R1"], e["t1"], e["trunc"], vs, ts, V, va, na, rows, cols, wrap, cc, cs)
    gr = np.load(os.path.join(GOLDEN, "ops_160x120_raycast.npz"))
    same_map(va.cpu().numpy(), gr["raycast_v"], rows, cols); same_map(na.cpu().numpy(), gr["raycast_n"], rows, cols)
    hit = ~np.isnan(gr["raycast_v"].reshape(3, rows, cols)[0])
    assert (cc.cpu().numpy()[hit] == gr["raycast_c"][hit]).all()
    cap = 400000
    out = zeros(e, (cap * 32,), t.uint8)
    real = (14, 3, 250 - V)
    for name, box in {"zslab": (0, V, 0, V, 225, 242), "xplus": (0, 120, 0, V, 0, V), "yslab": (0, V, 180, 197, 0, V)}.items():
        n = e["ops"].extract_slice(ts, vs, V, out, cap, wrap, cs, box, 1, real)
        arr = out.cpu().numpy()[: n * 32].view(np.uint64).reshape(n, 4)
        arr = arr[np.lexsort(arr.T[::-1])] if n else arr
        assert arr.shape == g[f"extract_{name}"].shape and (arr == g[f"extract_{name}"]).all(), name
    # capacity clamp: never writes past the caller's buffer (the reference does, extract.cu:268-288)
    small = 1000
    guard = t.full(((small + 16) * 32,), 0xAB, dtype=t.uint8, device="cuda")
    n = e["ops"].extract_slice(ts, vs, V, guard, small, wrap, cs, (0, 120, 0, V, 0, V), 1, real)
    assert n == small and bool((guard[small * 32:] == 0xAB).all())
    for key in [k for k in g.files if k.startswith("clear_")]:
        _, a, b, c, nn = key.split("_")
        axis, back, cur, n = int(a[1:]), int(b[1:]), int(c[1:]), int(nn[1:])
        x = t.full((V ** 3,), 7, dtype=t.int16, device="cuda"); y = t.full((V ** 3 * 4,), 9, dtype=t.uint8, device="cuda")
        e["ops"].clear_volume(axis, back, x, y, V, cur, cur + n)
        zt = (x.view(V, V, V) == 0); zc = (y.view(V, V, V, 4) == 0).all(-1)
        assert bool((zt == zc).all())
        ax = {0: (0, 1), 1: (0, 2), 2: (1, 2)}[axis]
        full = zt.all(dim=ax[1]).all(dim=ax[0])
        assert t.nonzero(full).flatten().cpu().numpy().tolist() == g[key].tolist(), key
        assert int(zt.sum().item()) == int(full.sum().item()) * V * V


def test_volume_ops_vs_reference_cuda_on_identical_buffers(env):
    """The reference's operators on the same buffers (640x480, wrapped volume): integrate, raycast -- bit-exact, by digest."""
    e = env; t = e["torch"]
    from kintinuous_b200 import synth
    from oracle.golden import digest
    live = e["live"]
    rows, cols = 480, 640
    intr = np.array(synth.intrinsics(cols, rows), np.float32)
    d, c = synth.render(3)
    dd = dev(e, d.view(np.int16)); cc = dev(e, c)
    fb = zeros(e, (rows, cols), t.int16); e["ops"].bilateral(dd, fb, rows, cols)
    vm = zeros(e, (3 * rows, cols), t.float32); nm = zeros(e, (3 * rows, cols), t.float32)
    e["ops"].create_vmap(intr, fb, vm, rows, cols); e["ops"].create_nmap(vm, nm, rows, cols)
    assert [digest(fb), digest(vm, "map"), digest(nm, "map")] == live["volops_inputs"].tolist()       # the reference's input maps
    ta = zeros(e, (V ** 3,), t.int16); ca = zeros(e, (V ** 3 * 4,), t.uint8)
    dsa = zeros(e, (rows, cols), t.float32)
    vs = [SIZE] * 3
    for i, (wrap, R, tt) in enumerate([((0, 0, 0), e["R0"], e["t0"]), ((250, 14, 3), e["R1"], e["t1"]), ((250, 14, 3), e["R1"].T.copy(), e["t1"] + np.float32(0.05))]):
        want = live["volops_steps"][i]
        Rinv = np.linalg.inv(R.astype(np.float64)).astype(np.float32)
        e["ops"].integrate(dd, rows, cols, intr, vs, Rinv, tt, e["trunc"], ta, ca, V, wrap, cc, nm, 1, dsa)
        t.cuda.synchronize()
        assert digest(ta) == want[0] and digest(ca) == want[1], i
        va = zeros(e, (3 * rows, cols), t.float32); na = zeros(e, (3 * rows, cols), t.float32); xa = zeros(e, (rows, cols, 4), t.uint8)
        e["ops"].raycast(intr, R, tt, e["trunc"], vs, ta, V, va, na, rows, cols, wrap, xa, ca)
        t.cuda.synchronize()
        assert digest(va, "map") == want[2] and digest(na, "map") == want[3], i
        assert digest(xa) == want[4], i


def test_rgbd_operators_vs_golden(env):
    e = env; t = e["torch"]; rows, cols = e["rows"], e["cols"]
    g = np.load(os.path.join(GOLDEN, "rgbd_160x120.npz"))
    from kintinuous_b200 import synth
    d1, c1 = synth.render(4, cols, rows)
    d0 = dev(e, e["d0"].view(np.int16)); dd1 = dev(e, d1.view(np.int16)); c0 = dev(e, e["c0"]); cc1 = dev(e, c1)
    fd0 = zeros(e, (rows, cols), t.float32); fd1 = zeros(e, (rows, cols), t.float32)
    e["ops"].short_depth_to_metres(d0, fd0, rows, cols, 6000); e["ops"].short_depth_to_metres(dd1, fd1, rows, cols, 6000)
    i0 = zeros(e, (rows, cols), t.uint8); i1 = zeros(e, (rows, cols), t.uint8)
    e["ops"].bgr_to_intensity(c0, i0, rows, cols); e["ops"].bgr_to_intensity(cc1, i1, rows, cols)
    assert (fd1.cpu().numpy().view(np.uint32) == g["depth_f"].view(np.uint32)).all() and (i1.cpu().numpy() == g["intensity"]).all()
    pf = zeros(e, (rows // 2, cols // 2), t.float32); e["ops"].pyrdown_gauss_f(fd1, pf, rows, cols)
    a, b = pf.cpu().numpy(), g["pyr_f"]
    assert (np.isnan(a) == np.isnan(b)).all() and (a[~np.isnan(a)].view(np.uint32) == b[~np.isnan(b)].view(np.uint32)).all()
    pu = zeros(e, (rows // 2, cols // 2), t.uint8); e["ops"].pyrdown_uchar_gauss(i1, pu, rows, cols)
    assert (pu.cpu().numpy() == g["pyr_u"]).all()
    dx = zeros(e, (rows, cols), t.int16); dy = zeros(e, (rows, cols), t.int16)
    e["ops"].derivative_images(i1, dx, dy, rows, cols)
    assert (dx.cpu().numpy() == g["dIdx"]).all() and (dy.cpu().numpy() == g["dIdy"]).all()
    cl = zeros(e, (rows, cols, 3), t.float32)
    fx, fy, cx, cy = [float(np.float32(v)) for v in synth.intrinsics(cols, rows)]
    e["ops"].project_to_point_cloud(fd0, cl, rows, cols, [fx, fy, cx, cy], 0)
    a, b = cl.cpu().numpy(), g["cloud"]
    ok = ~np.isnan(b)
    assert (np.isnan(a) == np.isnan(b)).all() and (a[ok].view(np.uint32) == b[ok].view(np.uint32)).all()
    cor = zeros(e, (rows * cols * 16,), t.uint8)
    sigma, count = e["ops"].rgb_residual(float(3.0 ** 2 / (1 / 8.0) ** 2), dx, dy, fd0, fd1, i0, i1, cor, rows, cols, 0.07, g["kt"], g["krk"])
    assert (sigma, count) == tuple(int(v) for v in g["sigma_count"])
    mine = cor.cpu().numpy().reshape(-1, 16); gold = g["corres"]
    valid = gold[:, 12] != 0
    assert ((mine[:, 12] != 0) == valid).all() and (mine[valid, :12] == gold[valid, :12]).all()
    A, b = e["ops"].rgb_step(cor, float(np.sqrt(count)), cl, fx, fy, dx, dy, 1 / 8.0, rows, cols)
    assert np.abs(A - g["rgb_A"]).max() <= 1e-5 * np.abs(g["rgb_A"]).max() and np.abs(b - g["rgb_b"]).max() <= 1e-5 * np.abs(g["rgb_b"]).max()


@pytest.mark.parametrize("rows,cols,variant", [(480, 640, "clean"), (480, 640, "holes"), (120, 160, "noise"), (96, 96, "holes")])
def test_fused_frontend_equals_the_operator_chain(built, rows, cols, variant):
    """The tracker's per-frame front end is two fused launches (kt_frontend.cu); the operator-level kernels are what the golden vectors
    pin against the reference.  Same inputs through both: every output -- filtered depth pyramid, vertex / normal maps of all four levels,
    scaled depth, colour-integration inputs, metric depth / intensity pyramids, gradients -- must be bit-identical.  Inputs with holes
    (NaN handling, the integer weight count Q2, stale planes Q7), sensor noise and far depths (the bilateral filter's integer path),
    and a size that is not a multiple of the 64 x 32 tile."""
    import torch
    import kintinuous_b200 as kb
    from kintinuous_b200 import synth
    ops = kb.ops
    d, c = synth.render(3, cols, rows, noise=(variant == "noise"))
    d = d.copy()
    rng = np.random.default_rng(4)
    if variant == "holes":
        d[rng.random(d.shape) < 0.15] = 0
        d[10:30, 20:50] = 0
        d[rows // 2:rows // 2 + 9, cols // 3:cols // 3 + 40] = 52000          # beyond 46 340 mm: the reference's int32 overflow path, and > 6 m cut-off
    intr = np.array(synth.intrinsics(cols, rows), np.float32)
    dd = torch.from_numpy(d.view(np.int16)).cuda(); cc = torch.from_numpy(c).cuda()
    L = 4
    def mk(dt, mult=1):
        return [torch.zeros((mult * (rows >> l), cols >> l), dtype=dt, device="cuda") for l in range(L)]
    # ---- operator chain (the kernels pinned by the golden vectors) ----
    rd, rv, rn = mk(torch.int16), mk(torch.float32, 3), mk(torch.float32, 3)
    ops.bilateral(dd, rd[0], rows, cols)
    for l in range(1, L):
        ops.pyrdown(rd[l - 1], rd[l], rows >> (l - 1), cols >> (l - 1))
    for l in range(L):
        kl = intr / (1 << l)
        ops.create_vmap(kl, rd[l], rv[l], rows >> l, cols >> l); ops.create_nmap(rv[l], rn[l], rows >> l, cols >> l)
    rm, ri, rx, ry = mk(torch.float32), mk(torch.uint8), mk(torch.int16), mk(torch.int16)
    ops.short_depth_to_metres(dd, rm[0], rows, cols, 6000); ops.bgr_to_intensity(cc, ri[0], rows, cols)
    for l in range(1, L):
        ops.pyrdown_gauss_f(rm[l - 1], rm[l], rows >> (l - 1), cols >> (l - 1)); ops.pyrdown_uchar_gauss(ri[l - 1], ri[l], rows >> (l - 1), cols >> (l - 1))
    for l in range(L):
        ops.derivative_images(ri[l], rx[l], ry[l], rows >> l, cols >> l)
    # scaleDepth through the integrate operator's own launch (1-voxel dummy volume is not possible: use a small one)
    Vs = 32
    ts = torch.zeros(Vs ** 3, dtype=torch.int16, device="cuda"); cs = torch.zeros(Vs ** 3 * 4, dtype=torch.uint8, device="cuda")
    rs = torch.zeros((rows, cols), dtype=torch.float32, device="cuda")
    ops.integrate(dd, rows, cols, intr, [6.0] * 3, np.eye(3, dtype=np.float32), np.array([3, 3, 3], np.float32), 0.4, ts, cs, Vs, (0, 0, 0), cc, rn[0], 1, rs)
    # ---- fused ----
    fd, fv, fn = mk(torch.int16), mk(torch.float32, 3), mk(torch.float32, 3)
    fm, fi, fx, fy = mk(torch.float32), mk(torch.uint8), mk(torch.int16), mk(torch.int16)
    fs = torch.zeros((rows, cols), dtype=torch.float32, device="cuda")
    cw = torch.zeros((rows, cols), dtype=torch.float32, device="cuda"); rgbf = torch.zeros((rows, cols, 4), dtype=torch.float32, device="cuda")
    ops.frontend(dd, cc, rows, cols, intr, 1, fd, fv, fn, fs, cw, rgbf, fm, fi, fx, fy)
    torch.cuda.synchronize()
    def same(a, b):
        if a.dtype != torch.float32:
            return torch.equal(a, b)
        # floats: identical values with NaNs in the same places (an exactly-zero normal component may carry either sign)
        return bool((torch.isnan(a) == torch.isnan(b)).all()) and bool((a[~torch.isnan(a)] == b[~torch.isnan(b)]).all())
    assert same(fs, rs), "scaled depth"
    for l in range(L):
        assert same(fd[l], rd[l]), ("depth", l)
        # Q7: an invalid pixel only has NaN in its x plane; its y / z planes keep what the buffer held (zeros here, on both sides)
        assert same(fv[l], rv[l]), ("vmap", l)
        assert same(fn[l], rn[l]), ("nmap", l)
        assert same(fm[l], rm[l]), ("depth_m", l)
        assert same(fi[l], ri[l]), ("intensity", l)
        assert same(fx[l], rx[l]) and same(fy[l], ry[l]), ("gradient", l)
    # colour-integration inputs: the definition (tsdf_volume.cu:601-622) on the reference-pinned normal map
    nx = rn[0][:rows]; nz = rn[0][2 * rows:].abs()
    w = torch.clamp(nz / 0.75, max=1.0) * 2.0
    want = torch.where(torch.isnan(nx), -w, w)
    # (the kernels divide by the constant 0.75 with the reference's approximate division: last-bit differences against torch's true division)
    assert torch.equal(torch.signbit(cw) & (want != 0), torch.signbit(want) & (want != 0)) and torch.allclose(cw, want, rtol=3e-7, atol=0), "colour weight"
    assert torch.equal(rgbf[..., :3], cc.to(torch.float32))
    # without the photometric set (ICP-only instance of the kernel): same maps
    gd, gv, gn = mk(torch.int16), mk(torch.float32, 3), mk(torch.float32, 3)
    ops.frontend(dd, cc, rows, cols, intr, 1, gd, gv, gn, None, None, None)
    torch.cuda.synchronize()
    for l in range(L):
        assert same(gd[l], rd[l]) and same(gv[l], rv[l]) and same(gn[l], rn[l]), ("icp-only instance", l)


def test_generate_image_and_depth_vs_reference_cuda(built):
    """The GUI taps (generateImage / generateDepth, image_generator.cu:161-230; getImage / getModelDepth in KintinuousTracker.cpp:960-981)
    against the reference's kernels on identical buffers: a surface predicted by ray casting a fused frame, the tracker's light
    (volume size * -3), bit-exact images and depth (by digest: tests/golden/ref_ops_live.npz)."""
    import torch
    import kintinuous_b200 as kb
    from kintinuous_b200 import synth
    from oracle.golden import digest
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
    ts = torch.zeros(Vs ** 3, dtype=torch.int16, device="cuda"); cs = torch.zeros(Vs ** 3 * 4, dtype=torch.uint8, device="cuda")
    ds = torch.zeros((rows, cols), dtype=torch.float32, device="cuda")
    R = np.eye(3, dtype=np.float32); t = np.array([3, 3, 3], np.float32)
    for _ in range(3):                                             # weights 3: a heat value between two palette entries
        ops.integrate(dd, rows, cols, intr, [6.0] * 3, R, t, 0.06, ts, cs, Vs, (0, 0, 0), cc, nm, 1, ds)
    ang = 0.02
    R1 = np.array([[np.cos(ang), 0, np.sin(ang)], [0, 1, 0], [-np.sin(ang), 0, np.cos(ang)]], np.float32)
    t1 = t + np.array([0.01, 0.0, 0.02], np.float32)
    va = torch.zeros_like(vm); na = torch.zeros_like(vm); xa = torch.zeros((rows, cols, 4), dtype=torch.uint8, device="cuda")
    ops.raycast(intr, R1, t1, 0.06, [6.0] * 3, ts, Vs, va, na, rows, cols, (0, 0, 0), xa, cs)
    torch.cuda.synchronize()
    # the inputs of the GUI taps are the reference's own, bit for bit
    assert [digest(fb), digest(vm, "map"), digest(nm, "map"), digest(ts), digest(cs), digest(va), digest(na), digest(xa)] == live["genimage_inputs"].tolist()
    light = [-18.0, -18.0, -18.0]                                  # KintinuousTracker::getImage: size * -3
    ia = torch.zeros((rows, cols, 3), dtype=torch.uint8, device="cuda"); ca = torch.zeros_like(ia)
    ops.generate_image(va, na, xa, light, 1, ia, ca, rows, cols)
    Rinv = np.linalg.inv(R1.astype(np.float64)).astype(np.float32)
    da = torch.zeros((rows, cols), dtype=torch.int16, device="cuda")
    ops.generate_depth(Rinv, t1, va, na, da, rows, cols)
    torch.cuda.synchronize()
    assert int((ia != 0).any(-1).sum()) > 0.8 * rows * cols          # the view really shows the room
    assert [digest(ia), digest(ca), digest(da)] == live["genimage_outputs"].tolist()
    zd = da.cpu().numpy().view(np.uint16)
    assert abs(float(np.median(zd[zd > 0])) - float(np.median(d[d > 0]))) < 60      # model depth ~ input depth (mm)
