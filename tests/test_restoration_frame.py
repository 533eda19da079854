"""GPU parity of the a13 restoration drivers: svt_b200_lr_save_boundary_lines_dev and svt_b200_lr_filter_frame_dev
against the reference's own svt_aom_save_tile_row_boundary_lines (restoration.c:1606) and
svt_av1_loop_restoration_filter_unit (:1067) run over every unit of a plane (oracle/ref_driver.c ref_lr_filter_plane),
for luma and chroma geometry, 8 and 10 bit, normal and optimized_lr stripes, pictures whose height is not a multiple of
the stripe / unit size (last unit absorbs the remainder, last stripe short, a stripe ending one row above the crop
border), a mix of RESTORE_NONE / WIENER / SGRPROJ units; plus the per-unit SSE (sse_restoration_unit)."""
import ctypes as ct

import numpy as np
import pytest

from helpers import rng

pytestmark = pytest.mark.gpu

PAD = 16


def _plane(r, w, h, bd, smooth):
    mx = (1 << bd) - 1
    dt = np.uint8 if bd == 8 else np.uint16
    if smooth:
        yy, xx = np.mgrid[0:h, 0:w]
        base = (np.sin(xx / 17.0) + np.cos(yy / 11.0) + 2.0) / 4.0 * mx
        v = np.clip(base + r.normal(0, mx / 60.0, (h, w)), 0, mx)
    else:
        v = r.integers(0, mx + 1, (h, w))
    buf = np.zeros((h + 2 * PAD, w + 2 * PAD + 5), dt)  # odd pitch on purpose
    buf[PAD:PAD + h, PAD:PAD + w] = v.astype(dt)
    return buf


def _units(r, n, b200):
    u = np.zeros(n, dtype=b200.LR_UNIT_DTYPE)
    for k in range(n):
        t = (1, 2, 0, 1, 2)[k % 5]
        u["restoration_type"][k] = t
        t0, t1, t2 = int(r.integers(-5, 11)), int(r.integers(-23, 9)), int(r.integers(-17, 47))
        taps = np.array([t0, t1, t2, -2 * (t0 + t1 + t2), t2, t1, t0, 0], np.int16)
        u["hfilter"][k] = taps
        u["vfilter"][k] = taps[::-1].copy() if k % 2 else taps
        if k % 2:
            u["vfilter"][k] = np.array([t2, t1, t0, -2 * (t0 + t1 + t2), t0, t1, t2, 0], np.int16)
        ep = int(r.integers(0, 16))
        u["sgr_ep"][k] = ep
        xqd = [int(r.integers(-96, 32)), int(r.integers(-32, 96))]
        u["sgr_xqd"][k] = xqd
    return u


CASES = [  # (luma width, luma height, bit depth, luma unit size)
    (328, 200, 8, 64), (328, 200, 10, 128), (256, 121, 8, 64), (200, 57, 10, 64), (640, 360, 8, 256), (1920, 1080, 8, 256), (1920, 1080, 10, 128)]


@pytest.mark.parametrize("case", CASES, ids=lambda c: "%dx%d_b%d_ru%d" % c)
def test_lr_frame_matches_reference(b200, oracle, golden, case):
    import torch
    W, H, bd, us = case
    r = rng(1300 + W + H + bd)
    psz = 1 if bd == 8 else 2
    tdt = torch.uint8 if bd == 8 else torch.int16
    refc = oracle.ref
    if refc is not None:
        refc.ref_lr_save_boundaries.restype = None
        refc.ref_lr_filter_plane.restype = None
    planes = (b200.LrPlane * 3)()
    keep, checks = [], []
    for p in range(3):
        ss = 1 if p else 0
        w, h, usp = (W + ss) >> ss, (H + ss) >> ss, us >> ss
        deb, cdf, src = _plane(r, w, h, bd, p == 1), _plane(r, w, h, bd, p != 2), _plane(r, w, h, bd, True)
        pitch = deb.shape[1]
        nst = b200.lib.svt_b200_lr_num_stripes(h, ss)
        bstride = b200.lib.svt_b200_lr_boundary_stride(w)
        hu, vu = b200.lib.svt_b200_lr_units_per_dim(w, usp), b200.lib.svt_b200_lr_units_per_dim(h, usp)
        units = _units(r, hu * vu, b200)
        # ---- reference: boundary lines of both passes, then every unit of the plane ----
        ab = bl = None
        want = {0: None, 1: None}
        if refc is not None:
            ab = np.full(2 * nst * bstride, 77, deb.dtype)
            bl = np.full(2 * nst * bstride, 77, deb.dtype)
            org = (PAD * pitch + PAD) * psz
            V = lambda a, o=0: ct.c_void_p(a.ctypes.data + o)  # noqa: E731
            refc.ref_lr_save_boundaries(V(deb, org), pitch, w, h, bd, p, W, H, 0, V(ab), V(bl), bstride)
            refc.ref_lr_save_boundaries(V(cdf, org), pitch, w, h, bd, p, W, H, 1, V(ab), V(bl), bstride)
            for opt in (0, 1):
                data = cdf.copy()
                out = np.zeros_like(cdf)
                refc.ref_lr_filter_plane(V(data, org), pitch, V(out, org), pitch, w, h, ss, ss, bd, usp, V(units), V(ab), V(bl), bstride, opt)
                want[opt] = out[PAD:PAD + h, PAD:PAD + w].copy()
        # ---- device ----
        T = lambda a: torch.from_numpy(a.view(np.int16) if a.dtype == np.uint16 else a).cuda()  # noqa: E731
        d_deb, d_cdf, d_src = T(deb[PAD:PAD + h, PAD:PAD + w].copy()), T(cdf[PAD:PAD + h, PAD:PAD + w].copy()), T(src[PAD:PAD + h, PAD:PAD + w].copy())
        d_dst = torch.zeros((h, w), dtype=tdt, device="cuda")
        d_ab = torch.full((2 * nst * bstride,), 77, dtype=tdt, device="cuda")
        d_bl = torch.full((2 * nst * bstride,), 77, dtype=tdt, device="cuda")
        d_units = torch.from_numpy(units.view(np.uint8)).cuda()
        d_sse = torch.zeros(hu * vu, dtype=torch.int64, device="cuda")
        planes[p] = b200.LrPlane(d_deb.data_ptr(), d_cdf.data_ptr(), d_dst.data_ptr(), d_src.data_ptr(), d_ab.data_ptr(), d_bl.data_ptr(), w, w, w, w,
                                 bstride, w, h, ss, ss, usp, 0)
        keep.append((d_deb, d_cdf, d_src, d_dst, d_ab, d_bl, d_units, d_sse))
        checks.append((w, h, usp, hu, vu, ab, bl, want, src[PAD:PAD + h, PAD:PAD + w].astype(np.int64)))
    s = torch.cuda.current_stream().cuda_stream
    assert b200.lib.svt_b200_lr_save_boundary_lines_dev(planes, 3, 0, bd, s) == 0
    assert b200.lib.svt_b200_lr_save_boundary_lines_dev(planes, 3, 1, bd, s) == 0
    torch.cuda.synchronize()
    for p in range(3):
        w, h, usp, hu, vu, ab, bl, want, src = checks[p]
        dt = np.uint8 if bd == 8 else np.uint16
        golden.check(keep[p][4].cpu().numpy().view(dt), ab, "above lines", p)
        golden.check(keep[p][5].cpu().numpy().view(dt), bl, "below lines", p)
    unit_ptrs = (ct.c_void_p * 3)(*[k[6].data_ptr() for k in keep])
    sse_ptrs = (ct.c_void_p * 3)(*[k[7].data_ptr() for k in keep])
    for opt in (0, 1):
        for k in keep:
            k[3].zero_()
        assert b200.lib.svt_b200_lr_filter_frame_dev(planes, 3, unit_ptrs, opt, bd, s) == 0
        assert b200.lib.svt_b200_lr_unit_sse_dev(planes, 3, sse_ptrs, bd, s) == 0
        torch.cuda.synchronize()
        for p in range(3):
            w, h, usp, hu, vu, ab, bl, want, src = checks[p]
            got = keep[p][3].cpu().numpy().view(np.uint8 if bd == 8 else np.uint16)
            golden.check(got, want[opt], "restored plane", p, opt)
            # sse_restoration_unit over each unit's limits
            off = 8 >> (1 if p else 0)
            sse = keep[p][7].cpu().numpy()
            d2 = (got.astype(np.int64) - src) ** 2
            for ur in range(vu):
                vs, ve = max(0, ur * usp - off), (h if ur == vu - 1 else (ur + 1) * usp - off)
                for uc in range(hu):
                    hs, he = uc * usp, (w if uc == hu - 1 else (uc + 1) * usp)
                    assert int(sse[ur * hu + uc]) == int(d2[vs:ve, hs:he].sum()), (p, ur, uc)


def test_lr_frame_rejects_bad_arguments(b200):
    planes = (b200.LrPlane * 3)()
    assert b200.lib.svt_b200_lr_filter_frame_dev(planes, 0, None, 0, 8, None) == -4
    assert b200.lib.svt_b200_lr_filter_frame_dev(planes, 1, None, 0, 9, None) == -4
    assert b200.lib.svt_b200_lr_num_stripes(1080, 0) == 17 and b200.lib.svt_b200_lr_num_stripes(540, 1) == 17
    assert b200.lib.svt_b200_lr_units_per_dim(1080, 256) == 4 and b200.lib.svt_b200_lr_units_per_dim(100, 256) == 1
