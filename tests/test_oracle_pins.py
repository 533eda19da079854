"""Pin the C restatement (oracle/port) against the UNMODIFIED reference objects (oracle/_ref),
on the reference's own test matrices (through the recorded digests of tests/golden/reference_digests.json
where oracle/_ref is not built, tests/reference_golden.py).  CPU only."""
import ctypes as ct

import numpy as np
import pytest

from helpers import rng, sad_loop_call, sad_pattern

BLOCKS = [(16, 16), (32, 32), (64, 64), (16, 8), (64, 32), (24, 24), (31, 7), (4, 4), (48, 64), (5, 11), (128, 128)]
AREAS = [(8, 3), (16, 31), (15, 6), (48, 40), (64, 25)]


@pytest.mark.parametrize("pattern", ["REF_MAX", "SRC_MAX", "RANDOM", "FLAT"])
def test_port_sad_loop_matches_reference(oracle, golden, pattern):
    r = rng(1)
    for (bw, bh) in BLOCKS:
        for (sa_w, sa_h) in AREAS:
            for skip in (0, 1):
                ref_stride = sa_w + bw + 9
                src_stride = bw + 3
                src, ref = sad_pattern(pattern, r, src_stride * bh, ref_stride * (sa_h + bh))
                a = sad_loop_call(oracle.port, "port_sad_loop", src, 0, src_stride, ref, 0, ref_stride, bh, bw, ref_stride,
                                  skip, sa_w, sa_h, -7, -9)
                b = sad_loop_call(oracle.ref, "svt_sad_loop_kernel_c", src, 0, src_stride, ref, 0, ref_stride, bh, bw,
                                  ref_stride, skip, sa_w, sa_h, -7, -9) if oracle.ref is not None else None
                golden.check(a, b, bw, bh, sa_w, sa_h, skip)


# ---- transforms: restatement vs unmodified reference, every size x valid type ------------------
from txfm_helpers import (TX_H, TX_W, coeff_input, mask_written, port_fwd, port_inv, ref_fwd, ref_inv,  # noqa: E402
                          residual_input, valid)


def test_port_txfm_valid_table(oracle):
    for sz in range(19):
        for ty in range(16):
            assert bool(oracle.port.port_txfm_valid(sz, ty)) == valid(sz, ty)


@pytest.mark.parametrize("kind", ["random", "max", "min"])
def test_port_fwd_txfm_matches_reference(oracle, golden, kind):
    r = rng(10)
    for sz in range(19):
        for ty in range(16):
            if not valid(sz, ty):
                continue
            for bd in (8, 10):
                res, stride = residual_input(r, sz, bd, kind)
                a = port_fwd(oracle.port, res, stride, ty, sz)
                b = ref_fwd(oracle.ref, res, stride, ty, sz, bd) if oracle.ref is not None else None
                golden.check(a, b, sz, ty, bd)


@pytest.mark.parametrize("kind", ["real", "sparse", "dc", "extreme", "zero"])
def test_port_inv_txfm_matches_reference(oracle, golden, kind):
    r = rng(11)
    for sz in range(19):
        for ty in range(16):
            if not valid(sz, ty):
                continue
            for bd in (8, 10):
                w, h = TX_W[sz], TX_H[sz]
                # the coefficients: the reference's forward transform (== the restatement's, test_port_fwd_txfm_matches_reference)
                fwd = (lambda res, st: ref_fwd(oracle.ref, res, st, ty, sz, bd)) if oracle.ref is not None else (lambda res, st: port_fwd(oracle.port, res, st, ty, sz))
                c = coeff_input(r, sz, bd, kind, fwd)
                pred = r.integers(0, 1 << bd, h * (w + 5)).astype(np.uint16)
                a = port_inv(oracle.port, c, pred, w + 5, w + 2, ty, sz, bd)
                b = mask_written(ref_inv(oracle.ref, c, pred, w + 5, w + 2, ty, sz, bd), w + 2, w, h) if oracle.ref is not None else None
                golden.check(mask_written(a, w + 2, w, h), b, sz, ty, bd)


# ---- quantizers -----------------------------------------------------------------------------------
import quant_helpers as qh  # noqa: E402


def test_port_quantizers_match_reference(oracle, golden):
    r = rng(30)
    n = 0
    for v, c, t, sc, qm, iqm, ls in qh.cases(r):
        a = qh.call_port(oracle.port, v[2], c, t, sc, qm, iqm, ls)
        b = qh.call_ref(oracle.ref, v[1], c, t, sc, qh.ref_extra(v, qm, iqm, ls)) if oracle.ref is not None else None
        golden.check(a, b, v[0], c.size, ls, qm is not None)
        n += 1
    assert n > 1000


# ---- Hadamard / SATD / SAD pyramid ---------------------------------------------------------------
import me_helpers as mh  # noqa: E402


def test_port_hadamard_matches_reference(oracle, golden):
    r = rng(40)
    for n in (4, 8, 16, 32):
        for kind in ("random", "max", "min"):
            stride = n + 7
            if kind == "random":
                src = r.integers(-255, 256, n * stride).astype(np.int16)
            else:
                src = np.full(n * stride, 255 if kind == "max" else -255, np.int16)
            a = mh.hadamard_call(oracle.port, "port_hadamard", src, stride, n)
            live = oracle.ref is not None
            golden.check(a, mh.hadamard_call(oracle.ref, "svt_aom_hadamard_%dx%d_c" % (n, n), src, stride, n) if live else None, n, kind)
            golden.check(oracle.port.port_satd(oracle.p(a), a.size), oracle.ref.svt_aom_satd_c(oracle.p(a), a.size) if live else None)


def test_port_fullpel_matches_reference_kernels(oracle, golden):
    r = rng(41)
    for (sa_w, sa_h, sub) in [(8, 3, 0), (16, 9, 0), (11, 4, 0), (8, 3, 1), (13, 2, 1), (3, 3, 0)]:
        ss, rs = 64 + 16, 64 + sa_w + 9
        src = r.integers(0, 256, ss * 64, dtype=np.uint8)
        ref = r.integers(0, 256, rs * (64 + sa_h), dtype=np.uint8)
        if sa_w == 16:  # force ties: flat content
            src[:] = 100
            ref[:] = 103
        a = mh.port_fullpel(oracle.port, src, 0, ss, ref, 0, rs, sa_w, sa_h, -5, 7, sub)
        b = mh.ref_fullpel(oracle.ref, src, 0, ss, ref, 0, rs, sa_w, sa_h, -5, 7, sub) if oracle.ref is not None else None
        golden.check(a, b, sa_w, sa_h, sub)


# ---- CDEF ----------------------------------------------------------------------------------------
import cdef_helpers as ch  # noqa: E402


@pytest.mark.parametrize("bd,subs", [(8, 1), (8, 4), (10, 2)])
def test_port_cdef_search_matches_reference(oracle, golden, bd, subs):
    r = rng(60 + bd + subs)
    W, H = 208, 136  # not multiples of 64: partial filter blocks on the right / bottom (last ones >= 16x8 luma)
    rec, src, skip = ch.make_frame(r, W, H, bd)
    sy = [0, 4, 9, 17, 35, 63, 2]
    su = [0, 4, -1, 17, 20, 63, 3]
    a = ch.port_cdef_search(oracle.port, rec, src, skip, W, H, bd, 5, subs, sy, su)
    b = ch.ref_cdef_search(oracle.ref, rec, src, skip, W, H, bd, 5, subs, sy, su) if oracle.ref is not None else None
    golden.check(a, b)


# ---- Wiener --------------------------------------------------------------------------------------
import rest_helpers as rh  # noqa: E402


def test_port_wiener_convolve_matches_reference(oracle, golden):
    r = rng(80)
    for bd in (8, 10, 12):
        dt = np.uint8 if bd == 8 else np.uint16
        for (w, h) in [(64, 64), (48, 56), (16, 8), (64, 20)]:
            ss = w + 16
            src = r.integers(0, 1 << bd, ss * (h + 16)).astype(dt)
            if w == 48:
                src[:] = (1 << bd) - 1
            fx, fy = rh.wiener_taps(r), rh.wiener_taps(r)
            off = 5 * ss + 6
            a = rh.port_wiener(oracle.port, src.astype(np.uint16), off, ss, w, h, fx, fy, bd, 1 if bd == 8 else 0)
            b = rh.ref_wiener(oracle.ref, src, off, ss, w, h, fx, fy, bd) if oracle.ref is not None else None
            golden.check(a, b, bd, w, h)


def test_port_compute_stats_matches_reference(oracle, golden):
    r = rng(81)
    for bd in (8, 10, 12):
        dt = np.uint8 if bd == 8 else np.uint16
        for win in (7, 5, 3):
            W, Hh = 72, 56
            dgd = r.integers(0, 1 << bd, W * Hh).astype(dt); src = r.integers(0, 1 << bd, W * Hh).astype(dt)
            a = rh.port_stats(oracle.port, win, dgd.astype(np.uint16), src.astype(np.uint16), 5, 61, 4, 50, W, W, bd)
            b = rh.ref_stats(oracle.ref, win, dgd, src, 5, 61, 4, 50, W, W, bd) if oracle.ref is not None else None
            golden.check(a, b, bd, win)


# ---- self-guided filter + projection ----------------------------------------------------------
def _sgr_inputs(r, bd, w, h, kind):
    dt = np.uint8 if bd == 8 else np.uint16
    stride = w + 14
    n = stride * (h + 8)
    if kind == "random":
        a = r.integers(0, 1 << bd, n)
    elif kind == "smooth":
        yy, xx = np.mgrid[0:h + 8, 0:stride]
        a = np.clip((np.sin(xx / 9.0) + np.cos(yy / 6.0)) * (40 << (bd - 8)) + (128 << (bd - 8)) + r.integers(-3, 4, (h + 8, stride)), 0,
                    (1 << bd) - 1).reshape(-1)
    else:
        a = np.full(n, (1 << bd) - 1)
    return a.astype(dt), stride, 4 * stride + 5


def test_port_selfguided_and_projection_match_reference(oracle, golden):
    r = rng(100)
    refc = oracle.ref
    live = refc is not None
    if live:
        ppe8 = refc.svt_av1_lowbd_pixel_proj_error_c; ppe8.restype = ct.c_int64
        ppe16 = refc.svt_av1_highbd_pixel_proj_error_c; ppe16.restype = ct.c_int64
        gps = refc.svt_get_proj_subspace_c; gps.restype = None
        app = refc.svt_apply_selfguided_restoration_c; app.restype = None
    oracle.port.port_pixel_proj_error.restype = ct.c_int64
    for bd in (8, 10, 12):
        for (w, h) in [(64, 64), (48, 33), (8, 8), (96, 21)]:
            for kind in ("random", "smooth", "max"):
                dgd, stride, off = _sgr_inputs(r, bd, w, h, kind)
                src, _, _ = _sgr_inputs(r, bd, w, h, "smooth")
                for idx in (0, 5, 9, 10, 13, 14, 15):
                    a = rh.port_selfguided(oracle.port, dgd.astype(np.uint16), off, w, h, stride, idx, bd)
                    b = rh.ref_selfguided(refc, dgd, off, w, h, stride, idx, bd) if live else None
                    prm = np.array(rh.SGR_PARAMS[idx], np.int32)
                    if prm[0] > 0:
                        golden.check(a[0], b and b[0], bd, w, h, kind, idx)
                    if prm[1] > 0:
                        golden.check(a[1], b and b[1], bd, w, h, kind, idx)
                    flt = b if live else a  # the filter outputs the projection works on (equal where the filter is used)
                    # projection subspace + error on these filter outputs
                    xq_a = np.zeros(2, np.int32); xq_b = np.zeros(2, np.int32)
                    if live:
                        gps(rh.bptr(src, off), w, h, stride, rh.bptr(dgd, off), stride, int(bd > 8), rh.P(flt[0]), w, rh.P(flt[1]), w, rh.P(xq_b),
                            rh.P(prm))
                    s16, d16 = src.astype(np.uint16), dgd.astype(np.uint16)
                    oracle.port.port_get_proj_subspace(rh.P(s16, off), w, h, stride, rh.P(d16, off), stride, rh.P(flt[0]), w, rh.P(flt[1]), w,
                                                       rh.P(xq_a), rh.P(prm))
                    golden.check(xq_a, xq_b if live else None, bd, w, h, kind, idx)
                    xq = np.array([int(r.integers(-96, 32)), int(r.integers(-32, 96))], np.int32)
                    eb = (ppe8 if bd == 8 else ppe16)(rh.bptr(src, off), w, h, stride, rh.bptr(dgd, off), stride, rh.P(flt[0]), w, rh.P(flt[1]),
                                                      w, rh.P(xq), rh.P(prm)) if live else None
                    ea = oracle.port.port_pixel_proj_error(rh.P(s16, off), w, h, stride, rh.P(d16, off), stride, rh.P(flt[0]), w, rh.P(flt[1]),
                                                           w, rh.P(xq), rh.P(prm), int(bd > 8))
                    golden.check(ea, eb, bd, w, h, kind, idx)
                # apply
                xqd = np.array([-32, 31], np.int32)
                da = np.zeros(h * w, np.uint16); db = np.zeros(h * w, dgd.dtype)
                tmp = np.zeros(2 * 161 * 161 * 4 + 1024, np.int32)
                if live:
                    app(rh.bptr(dgd, off), w, h, stride, 3, rh.P(xqd), rh.bptr(db), w, rh.P(tmp), bd, int(bd > 8))
                oracle.port.port_sgr_apply.restype = None
                oracle.port.port_sgr_apply(rh.P(dgd.astype(np.uint16), off), w, h, stride, 3, rh.P(xqd), rh.P(da), w, bd)
                golden.check(da, db if live else None, bd, w, h, kind)


# ---- picture-level reference drivers (oracle/ref_driver.c) ---------------------------------------
def test_ref_driver_me_matches_numpy_driver_and_avx2_tier(oracle, refc):
    from test_me_picture import _content
    r = rng(130)
    W, H = 320, 200
    ME_PAD = (16, 32, 72)
    shapes = []
    for lvl in range(3):
        w, h, pad = W >> (2 - lvl), H >> (2 - lvl), ME_PAD[lvl]
        shapes.append((h + 2 * pad, (w + 2 * pad + 15) & ~15, pad, w, h))
    cur = mh.build_pyramid_np(_content(r, W, H, (0, 0)), W, H, shapes)
    refs = [mh.build_pyramid_np(_content(r, W, H, (5, -3)), W, H, shapes), mh.build_pyramid_np(_content(r, W, H, (-19, 9)), W, H, shapes)]
    params = [dict(hme_l0_sa_w=16, hme_l0_sa_h=8, hme_l1_sa_w=8, hme_l1_sa_h=3, hme_l2_sa_w=8, hme_l2_sa_h=3, me_sa_w=8, me_sa_h=3,
                   hme_sub_sad=0, me_sub_sad=0, check_zero_centre=1),
              dict(hme_l0_sa_w=32, hme_l0_sa_h=12, hme_l1_sa_w=8, hme_l1_sa_h=3, hme_l2_sa_w=8, hme_l2_sa_h=3, me_sa_w=16, me_sa_h=5,
                   hme_sub_sad=1, me_sub_sad=1, check_zero_centre=0)]
    refc.ref_set_tier(0)
    a = mh.ref_me_picture(refc, cur, refs, shapes, W, H, params)
    b = mh.ref_me_picture_c(refc, cur, refs, shapes, W, H, params)
    for x, y in zip(a, b):
        assert np.array_equal(x, y)
    if refc.ref_set_tier(1) == 1:  # the intrinsics-only AVX2 tier must agree with the C tier
        c = mh.ref_me_picture_c(refc, cur, refs, shapes, W, H, params)
        for x, y in zip(b, c):
            assert np.array_equal(x, y)
    refc.ref_set_tier(0)


def test_committed_golden_fixtures_are_what_the_reference_computes(oracle, golden):
    """tests/golden/frame_*.json (used by the GPU tests and smoke() where oracle/_ref may be absent) against the reference run here"""
    import json
    import os
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, os.path.join(root, "tools"))
    import make_golden
    for name in sorted(n for n in os.listdir(os.path.join(root, "tests", "golden")) if n.startswith("frame_")):
        g = json.load(open(os.path.join(root, "tests", "golden", name)))
        now = make_golden.golden_for(g["width"], g["height"], g["seed"], g.get("bit_depth", 8), g.get("preset", 8)) if oracle.ref is not None else None
        golden.check(sorted(g["sha256"].items()), now and sorted(now["sha256"].items()), name)


def _lr_case(lib, kind, seed=34):
    """a fixed set of restoration units (luma and chroma geometry, both optimized_lr modes, interior / edge units) through
    lib.ref_lr_filter_unit_{wiener,sgrproj}_8bit -- i.e. the reference's svt_av1_loop_restoration_filter_unit with whatever
    the dispatch pointers of `lib` currently hold.  Returns the filtered planes."""
    import ctypes as ct
    r = np.random.default_rng(seed)
    fn = getattr(lib, "ref_lr_filter_unit_%s_8bit" % kind)
    fn.restype = None
    PAD, outs = 32, []
    for ss in (0, 1):
        W, Hh = (328 >> ss), (200 >> ss)
        stride = W + 2 * PAD
        plane = r.integers(0, 256, (Hh + 2 * PAD) * stride).astype(np.uint8)
        origin = PAD * stride + PAD
        nstripes = (Hh + (8 >> ss) + (64 >> ss) - 1) // (64 >> ss) + 1
        bstride = ((W + 8 + 31) // 32) * 32
        above = r.integers(0, 256, 2 * nstripes * bstride).astype(np.uint8)
        below = r.integers(0, 256, 2 * nstripes * bstride).astype(np.uint8)
        tile = np.array([0, 0, W, Hh], np.int32)
        ru = 128 >> ss
        for opt in (0, 1):
            for (hs, he, vs, ve) in [(0, min(ru, W), 0, min(ru + (ru // 2), Hh)), (ru, W, 0, Hh), (0, W, (ru - (8 >> ss)), Hh)]:
                limits = np.array([hs, he, vs, ve], np.int32)
                src, dst = plane.copy(), np.full_like(plane, 7)
                V = lambda a, o=0: ct.c_void_p(a.ctypes.data + o)  # noqa: E731
                if kind == "wiener":
                    t0, t1, t2 = int(r.integers(-5, 11)), int(r.integers(-23, 9)), int(r.integers(-17, 47))
                    taps = np.array([t0, t1, t2, -2 * (t0 + t1 + t2), t2, t1, t0, 0], np.int16)
                    fn(V(src, origin), stride, V(dst, origin), stride, V(limits), V(taps), V(taps), V(above), V(below), bstride, V(tile), 0, ss, ss, opt)
                else:
                    ep = int(r.integers(0, 14))
                    xqd = np.array([int(r.integers(-96, 32)), int(r.integers(-32, 96))], np.int32)
                    fn(V(src, origin), stride, V(dst, origin), stride, V(limits), ep, V(xqd), V(above), V(below), bstride, V(tile), 0, ss, ss, opt)
                assert np.array_equal(src, plane)
                outs.append(dst)
    return outs


def test_port_lr_unit_with_stripe_boundaries_matches_reference(oracle, golden):
    """SURVEY 8 a13 groundwork: one restoration unit filtered stripe by stripe with the saved boundary lines
    (svt_av1_loop_restoration_filter_unit, restoration.c:1067-1135) -- our restatement against the reference."""
    import ctypes as ct
    r = np.random.default_rng(33)
    refc = oracle.ref
    live = refc is not None
    oracle.port.port_lr_filter_unit_wiener_8bit.restype = None
    oracle.port.port_lr_filter_unit_sgrproj_8bit.restype = None
    if live:
        refc.ref_lr_filter_unit_wiener_8bit.restype = None
        refc.ref_lr_filter_unit_sgrproj_8bit.restype = None
    PAD = 32
    for ss in (0, 1):
        W, Hh = (328 >> ss), (200 >> ss)
        stride = W + 2 * PAD
        plane = r.integers(0, 256, (Hh + 2 * PAD) * stride).astype(np.uint8)
        origin = PAD * stride + PAD
        nstripes = (Hh + (8 >> ss) + (64 >> ss) - 1) // (64 >> ss) + 1
        bstride = ((W + 8 + 31) // 32) * 32
        above = r.integers(0, 256, 2 * nstripes * bstride).astype(np.uint8)
        below = r.integers(0, 256, 2 * nstripes * bstride).astype(np.uint8)
        tile = np.array([0, 0, W, Hh], np.int32)
        ru = 128 >> ss
        for opt in (0, 1):
            for (hs, he, vs, ve) in [(0, min(ru, W), 0, min(ru + (ru // 2), Hh)), (ru, W, 0, Hh), (0, W, (ru - (8 >> ss)), Hh),
                                     (ru, min(2 * ru, W), ru - (8 >> ss), min(2 * ru - (8 >> ss), Hh))]:
                t0, t1, t2 = int(r.integers(-5, 11)), int(r.integers(-23, 9)), int(r.integers(-17, 47))
                taps = np.array([t0, t1, t2, -2 * (t0 + t1 + t2), t2, t1, t0, 0], np.int16)
                limits = np.array([hs, he, vs, ve], np.int32)
                outs = []
                for fn in ([refc.ref_lr_filter_unit_wiener_8bit] if live else []) + [oracle.port.port_lr_filter_unit_wiener_8bit]:
                    src = plane.copy()
                    dst = np.full_like(plane, 7)
                    fn(ct.c_void_p(src.ctypes.data + origin), stride, ct.c_void_p(dst.ctypes.data + origin), stride,
                       ct.c_void_p(limits.ctypes.data), ct.c_void_p(taps.ctypes.data), ct.c_void_p(taps.ctypes.data),
                       ct.c_void_p(above.ctypes.data), ct.c_void_p(below.ctypes.data), bstride, ct.c_void_p(tile.ctypes.data), 0, ss, ss, opt)
                    assert np.array_equal(src, plane), "the picture must be left as it was"
                    outs.append(dst)
                golden.check(outs[-1], outs[0] if live else None, ss, opt, hs, he, vs, ve)
                # the self-guided filter through the same stripe machinery
                ep = int(r.integers(0, 16))
                xqd = np.array([int(r.integers(-96, 32)), int(r.integers(-32, 96))], np.int32)
                if ep >= 14:
                    xqd[1] = 0 if ep == 14 else xqd[1]  # r1 == 0 sets are legal with any xqd; keep the draw simple
                outs = []
                for fn in ([refc.ref_lr_filter_unit_sgrproj_8bit] if live else []) + [oracle.port.port_lr_filter_unit_sgrproj_8bit]:
                    src = plane.copy()
                    dst = np.full_like(plane, 7)
                    fn(ct.c_void_p(src.ctypes.data + origin), stride, ct.c_void_p(dst.ctypes.data + origin), stride,
                       ct.c_void_p(limits.ctypes.data), ep, ct.c_void_p(xqd.ctypes.data), ct.c_void_p(above.ctypes.data),
                       ct.c_void_p(below.ctypes.data), bstride, ct.c_void_p(tile.ctypes.data), 0, ss, ss, opt)
                    assert np.array_equal(src, plane)
                    outs.append(dst)
                golden.check(outs[-1], outs[0] if live else None, "sgr", ss, opt, hs, he, vs, ve, ep)


def test_me_controls_json_is_the_references_derivation(oracle, golden):
    """svt-av1-psy_b200/me_controls.json (what the workload hands to svt_b200_me_b64_picture_dev) == svt_aom_sig_deriv_me of the
    reference for every (preset, resolution class), re-derived here; and the two ctypes mirrors of the control struct agree"""
    import json
    import os
    from oracle import support as sp
    from oracle.frame_ref import load_workload_module
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    assert sp.ME_CONTROL_FIELDS == load_workload_module().dsp.ME_CONTROL_FIELDS
    committed = json.load(open(os.path.join(root, "svt-av1-psy_b200", "me_controls.json")))
    fresh = None
    if oracle.ref is not None:
        import importlib.util
        spec = importlib.util.spec_from_file_location("dump_me_controls", os.path.join(root, "tools", "dump_me_controls.py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        fresh = mod.all_controls()
    golden.check(sorted(committed), fresh and sorted(fresh))
    for key in sorted(committed):
        got = dict(committed[key])
        # picture distances of reference slots beyond n_ref are never read (the glue leaves them 0, the committed file carries the
        # workload's nominal distances there)
        n0, n1 = got["n_ref"]
        got["dist"] = [d if (i < 4 and i < n0) or (i >= 4 and i - 4 < n1) else 0 for i, d in enumerate(got["dist"])]
        golden.check(json.dumps(got, sort_keys=True), fresh and json.dumps(fresh[key], sort_keys=True), key)


def test_committed_av1_tables_and_resolution_classes_are_the_references(oracle, golden):
    """av1_tables.npz (scan orders, quantization matrices) == a fresh dump from the compiled reference; the workload's
    resolution classes == svt_aom_derive_input_resolution over a sweep of picture sizes"""
    import ctypes as ct
    import os
    import numpy as np
    from oracle.frame_ref import load_workload_module
    wlm = load_workload_module()
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    z = np.load(os.path.join(root, "svt-av1-psy_b200", "av1_tables.npz"))
    refc = oracle.ref
    live = refc is not None
    i16p, u8p = ct.POINTER(ct.c_int16), ct.POINTER(ct.c_uint8)
    if live:
        refc.ref_scan_order.restype = ct.c_int
        refc.ref_scan_order.argtypes = [ct.c_int, ct.c_int, i16p, i16p]
        refc.ref_qm_matrix.restype = ct.c_int
        refc.ref_qm_matrix.argtypes = [ct.c_int, ct.c_int, ct.c_int, u8p, u8p]
        refc.ref_input_resolution_class.restype = ct.c_int
        refc.ref_input_resolution_class.argtypes = [ct.c_uint32]
    for sz in range(19):
        n = int(z["scan_len"][sz])
        for ty in range(16):
            s, i = np.zeros(n, np.int16), np.zeros(n, np.int16)
            if live:
                assert refc.ref_scan_order(sz, ty, s.ctypes.data_as(i16p), i.ctypes.data_as(i16p)) == n
            o = int(z["scan_off"][sz, ty])
            golden.check((z["scan"][o:o + n], z["iscan"][o:o + n]), (s, i) if live else None, sz, ty)
        for lv in (0, 8, 11, 14):
            for pl in range(2):
                q, iq = np.zeros(n, np.uint8), np.zeros(n, np.uint8)
                if live:
                    assert refc.ref_qm_matrix(lv, pl, sz, q.ctypes.data_as(u8p), iq.ctypes.data_as(u8p)) == n
                o = int(z["qm_off"][sz])
                golden.check((z["qm"][lv, pl, o:o + n], z["iqm"][lv, pl, o:o + n]), (q, iq) if live else None, sz, lv, pl)
    for (w, h) in [(64, 64), (352, 288), (416, 240), (640, 360), (640, 480), (854, 480), (1024, 576), (1280, 720), (1920, 1080), (2560, 1440),
                   (3840, 2160), (4096, 2304), (7680, 4320)]:
        golden.check(wlm.input_resolution_class(w, h), refc.ref_input_resolution_class(w * h) if live else None, w, h)
