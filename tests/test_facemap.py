"""Face maps on the B200 (dfb_facemap_create, dfb_interp_to_cells, dfb_interp_to_host): the apply kernel against numpy applying the
same taps (read through the host shim of tests/test_facemap_host.py) to the library's own fields, faces at cell centres bit for bit,
16-aligned widened slabs and batches bit for bit against the whole-plane handle, host delivery, stride, argument errors, and no effect
on the step, its state or its statistics."""
import ctypes as C

import numpy as np
import pytest

from test_facemap_host import AREA, POINT, Map, shim  # noqa: F401  (shim: the fixture)

pytestmark = pytest.mark.gpu
FLUCS = (0, 1, 2, 3, 4)
DTS = (2e-7, 1e-7, 3e-7)


def torch_dev():
    import torch
    return torch, torch.device("cuda", 0)


def plane(W):
    return W.plane_profile(64, 128, 8, 6)


def make(dfb, W, nplanes=1, **kw):
    df = dfb.DIGITAL_FILTER(dfb.DFConfig.from_plane(plane(W), seed=77, device=0, **kw), fetch=False, nplanes=nplanes)
    for dt in DTS:
        df.filter(dt)
    df.sync()
    return df


def faces(m, n, rng, kind, periodic=False):
    """n random faces over the plane (point maps: some beyond its edges); periodic: none across the seam"""
    vy, vz, zc = m.vy, m.vz, m.zc
    yf = rng.uniform(vy[0] - 0.02 * (vy[-1] - vy[0]), vy[-1], n)
    if kind == POINT:
        zf = rng.uniform(zc[0], zc[-1], n) if periodic else rng.uniform(vz[0] - 1e-5, vz[-1] + 1e-5, n)
        return dict(yf=yf, zf=zf)
    hy = rng.uniform(0.3, 2.5, n) * np.diff(vy).mean()
    hz = rng.uniform(0.3, 2.5, n) * np.diff(vz).mean()
    zf = vz[0] + 0.5 * hz + rng.uniform(0, 1, n) * (vz[-1] - vz[0] - hz) if periodic else rng.uniform(vz[0], vz[-1], n)
    return dict(yf=yf, zf=zf, hy=hy, hz=hz)


def host_map(shim, dfb, W, f, kind, **kw):  # noqa: F811
    return Map(shim, dfb, dfb.DFConfig.from_plane(plane(W), **kw), kind, f["yf"], f["zf"], f.get("hy"), f.get("hz"))


def fma_sum(m, F):
    """the kernel's sum, tap by tap in the map's order, each step a fused multiply-add (emulated in extended precision)"""
    out = np.zeros(m.n)
    for i in np.nonzero(m.served)[0]:
        jk, w = m.taps(i)
        acc = 0.0
        for (j, k), wt in zip(jk, w):
            acc = float(np.longdouble(wt) * np.longdouble(F[j, k]) + np.longdouble(acc))
        out[i] = acc
    return out


@pytest.mark.parametrize("kind", [POINT, AREA])
def test_apply_against_numpy(dfb, W, shim, kind):  # noqa: F811
    torch, dev = torch_dev()
    rng = np.random.default_rng(1 + kind)
    df = make(dfb, W)
    n = 3000
    probe = host_map(shim, dfb, W, dict(yf=[0.0], zf=[0.0]), POINT)
    f = faces(probe, n, rng, kind)
    m = host_map(shim, dfb, W, f, kind)
    fm = df.facemap(f["yf"], f["zf"], f.get("hy"), f.get("hz"))
    assert np.array_equal(fm.served, m.served) and fm.served.all()
    fields = [df.get(i) for i in FLUCS]
    ref = [fma_sum(m, F) for F in fields]
    rms = [float(np.sqrt(np.mean(F * F))) for F in fields]
    perm = torch.as_tensor(rng.permutation(n).astype(np.int32), device=dev)
    for mask in range(1, 32):
        sel = [i for i in FLUCS if mask >> i & 1]
        for variant in ("mean", "own", "scaled_stride"):
            stride = 3 if variant == "scaled_stride" else 1
            scale = [2.5 - 0.75 * r for r in range(len(sel))] if variant == "scaled_stride" else None
            init = [torch.as_tensor(rng.standard_normal(n * stride), device=dev) for _ in sel]
            dst = [t.clone() for t in init]
            mean = [torch.as_tensor(rng.standard_normal(n), device=dev) for _ in sel] if variant == "mean" else None
            torch.cuda.synchronize()                           # the handle's stream does not wait for torch's
            fm.to_cells(dst, perm, mean, scale, fields=sel, stride=stride)
            torch.cuda.synchronize()
            p = perm.cpu().numpy().astype(np.int64) * stride
            for r, i in enumerate(sel):
                got = dst[r].cpu().numpy()
                base = (mean[r].cpu().numpy() if mean is not None else init[r].cpu().numpy()[p])
                s = scale[r] if scale is not None else 1.0
                want = base + s * ref[i]
                err = np.abs(got[p] - want)
                assert np.all(err <= 1e-15 * abs(s) * rms[i] + 4e-16 * np.abs(want)), (mask, variant, i, float(err.max()))
                untouched = np.ones(n * stride, dtype=bool)
                untouched[p] = False
                assert np.array_equal(got[untouched], init[r].cpu().numpy()[untouched])
    host = fm.to_host()                                        # host delivery equals the device path with mean 0 and scale 1
    dst = [torch.zeros(n, dtype=torch.float64, device=dev) for _ in FLUCS]
    torch.cuda.synchronize()
    fm.to_cells(dst)
    torch.cuda.synchronize()
    for i in FLUCS:
        assert np.array_equal(host[i], dst[i].cpu().numpy())
        assert np.all(np.abs(host[i] - ref[i]) <= 1e-15 * rms[i])
    fm.close()
    df.close()


def test_faces_at_cell_centres_bitwise(dfb, W, shim):  # noqa: F811
    df = make(dfb, W)
    probe = host_map(shim, dfb, W, dict(yf=[0.0], zf=[0.0]), POINT)
    jj, kk = np.meshgrid(np.arange(df.Ny), np.arange(df.Nz), indexing="ij")
    j, k = jj.ravel(), kk.ravel()
    vy, vz = probe.vy, probe.vz
    pt = df.facemap(probe.yc[j], probe.zc[k])
    ar = df.facemap(0.5 * (vy[j] + vy[j + 1]), 0.5 * (vz[k] + vz[k + 1]), vy[j + 1] - vy[j], vz[k + 1] - vz[k])
    for fm in (pt, ar):
        out = fm.to_host()
        for i in FLUCS:
            assert np.array_equal(out[i], df.get(i).ravel()), i
    df.close()


def slab_layouts(NzG):
    for cuts in ([0, 64, 128], [0, 32, 64, 96, 128]):
        yield [(max(0, a - 16), min(NzG, b + 16), a, b) for a, b in zip(cuts[:-1], cuts[1:])]


@pytest.mark.parametrize("periodic", [0, 1])
def test_widened_slabs_equal_whole_plane(dfb, W, shim, periodic):  # noqa: F811
    rng = np.random.default_rng(40 + periodic)
    whole = make(dfb, W, periodic_z=periodic)
    probe = host_map(shim, dfb, W, dict(yf=[0.0], zf=[0.0]), POINT, periodic_z=periodic)
    for kind in (POINT, AREA):
        f = faces(probe, 4000, rng, kind, periodic=bool(periodic))
        ref = whole.facemap(**f).to_host()
        for layout in slab_layouts(whole.Nz):
            got = np.full_like(ref, np.nan)
            count = np.zeros(len(f["yf"]), dtype=int)
            for k0, k1, o0, o1 in layout:
                s = make(dfb, W, periodic_z=periodic, k_begin=k0, k_end=k1)
                for i in FLUCS:                                 # premise: 16-aligned slabs compute the whole plane's bits
                    assert np.array_equal(s.get(i), whole.get(i)[:, k0:k1]), (k0, k1, i)
                fm = s.facemap(**f, own=(o0, o1))
                fm.to_host(out=got)
                count += fm.served
                s.close()
            assert np.all(count == 1)
            assert np.array_equal(got, ref), (kind, layout)
    whole.close()


def test_batch_planes_equal_single_planes(dfb, W, shim):  # noqa: F811
    rng = np.random.default_rng(9)
    batch = make(dfb, W, nplanes=3)
    probe = host_map(shim, dfb, W, dict(yf=[0.0], zf=[0.0]), POINT)
    for kind in (POINT, AREA):
        f = faces(probe, 2000, rng, kind)
        fb = batch.facemap(**f)
        for p in range(3):
            single = make(dfb, W, plane_id=p)
            for i in FLUCS:                                     # premise: batch plane p is the single-plane handle's plane
                assert np.array_equal(batch.get(i, plane=p), single.get(i)), (p, i)
            assert np.array_equal(fb.to_host(plane=p), single.facemap(**f).to_host()), (kind, p)
            single.close()
    batch.close()


def snapshot(df):
    fo, step = df.get_state()
    out = [df.get(i) for i in range(8)] + [fo, np.array([step])]
    out += [df.stats(i)[0] for i in range(6)]
    out += [df.corr(fld, d, normalized=False)[0] for fld in range(3) for d in range(3)]
    return out


def test_maps_have_no_side_effects_and_survive_restart(dfb, W, tmp_path):
    torch, dev = torch_dev()
    a, b = make(dfb, W), make(dfb, W)
    for df in (a, b):
        df.stats_enable(True)
        df.corr_enable(z=4, y=3, t=2)
    probe_y, probe_z = a.table(8), np.linspace(0.0, a.table(13, n=a.Nz + 1)[-1], 50)
    yf, zf = np.repeat(probe_y[::8], 50), np.tile(probe_z, len(probe_y[::8]))
    for s, dt in enumerate(DTS):
        a.filter(dt)
        b.filter(dt)
        if s == 1:                                              # maps created, applied and destroyed on a only
            pm = a.facemap(yf, zf, wall_zero=True)
            am = a.facemap(yf, zf, np.full(len(yf), 3e-5), np.full(len(yf), 2e-5))
            dst = [torch.zeros(len(yf), dtype=torch.float64, device=dev) for _ in FLUCS]
            torch.cuda.synchronize()
            pm.to_cells(dst)
            am.to_host()
            pm.close()
        for x, y in zip(snapshot(a), snapshot(b)):
            assert np.array_equal(x, y, equal_nan=True)
    path = str(tmp_path / "a.dfbr")
    a.save_restart(path)
    a.filter(1e-7)
    a.load_restart(path)                                        # the map stays valid across a load: a resumes where b is
    a.filter(2e-7)
    b.filter(2e-7)
    bm = b.facemap(yf, zf, np.full(len(yf), 3e-5), np.full(len(yf), 2e-5))
    assert np.array_equal(am.to_host(), bm.to_host())
    a.close()
    b.close()


def test_argument_errors(dfb, W):
    df = make(dfb, W)
    fm = df.facemap([df.table(8)[3]], [1e-5])
    L = dfb.lib()
    out = np.zeros(5)
    d = out.ctypes.data_as(dfb.c_dp)
    for mid, plane, mask in ((fm.id + 7, 0, 1), (-1, 0, 1), (fm.id, 1, 1), (fm.id, -1, 1), (fm.id, 0, 0), (fm.id, 0, 32)):
        assert L.dfb_interp_to_host(df._h, mid, plane, mask, d) == dfb.ERR_ARG, (mid, plane, mask)
    d5 = (C.c_void_p * 5)()
    assert L.dfb_interp_to_cells(df._h, fm.id, 0, 1, None, None, None, d5, 1) == dfb.ERR_ARG        # dst[0] NULL
    assert L.dfb_interp_to_cells(df._h, fm.id, 0, 1, None, None, None, d5, 0) == dfb.ERR_ARG        # stride 0
    with pytest.raises(dfb.DfbError) as e:
        df.facemap([np.nan], [0.0])
    assert e.value.code == dfb.ERR_ARG
    # while a pipelined copy is outstanding: DFB_ERR_STATE, as for restart files
    host = [np.zeros((df.Ny, df.Nz)) for _ in range(5)]
    assert L.dfb_filter_to_host_begin(df._h, 1e-7, *[h.ctypes.data for h in host]) == dfb.OK
    assert L.dfb_interp_to_host(df._h, fm.id, 0, 1, d) == dfb.ERR_STATE
    assert L.dfb_facemap_create(df._h, 0, 0, None, None, None, None, 0, 0, 0, C.byref(C.c_int())) == dfb.ERR_STATE
    assert L.dfb_filter_to_host_end(df._h) == dfb.OK
    fm.to_host()
    mid = fm.id
    fm.close()
    assert L.dfb_interp_to_host(df._h, mid, 0, 1, d) == dfb.ERR_ARG                                 # destroyed
    df.close()
