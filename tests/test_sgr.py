"""GPU parity: self-guided filter, apply, pixel-projection error and projection subspace vs the
reference C functions (fixtures after test/selfguided_filter_test.cc and SelfGuidedUtilTest.cc; the
subspace test asserts the integer xq pair is identical, as the reference test does)."""
import ctypes as ct

import numpy as np
import pytest

import rest_helpers as rh
from helpers import rng
from test_oracle_pins import _sgr_inputs

pytestmark = pytest.mark.gpu


def test_selfguided_filter_and_projection(b200, oracle, golden):
    r = rng(110)
    refc = oracle.ref
    live = refc is not None
    if live:
        ppe8 = refc.svt_av1_lowbd_pixel_proj_error_c; ppe8.restype = ct.c_int64
        ppe16 = refc.svt_av1_highbd_pixel_proj_error_c; ppe16.restype = ct.c_int64
        gps = refc.svt_get_proj_subspace_c; gps.restype = None
        app = refc.svt_apply_selfguided_restoration_c; app.restype = None
    for bd in (8, 10, 12):
        for (w, h) in [(64, 64), (48, 33), (8, 8), (96, 21), (32, 17)]:
            for kind in ("random", "smooth", "max"):
                dgd, stride, off = _sgr_inputs(r, bd, w, h, kind)
                src, _, _ = _sgr_inputs(r, bd, w, h, "smooth")
                for idx in (0, 3, 9, 10, 13, 14, 15):
                    want = rh.ref_selfguided(refc, dgd, off, w, h, stride, idx, bd) if live else None
                    f0 = np.full(w * h, -12345, np.int32); f1 = np.full(w * h, -12345, np.int32)
                    b200.lib.svt_b200_av1_selfguided_restoration(rh.P(dgd, off), w, h, stride, rh.P(f0), rh.P(f1), w, idx, bd, int(bd > 8))
                    golden.check((f0, f1), want, bd, w, h, kind, idx)
                    prm = np.array(rh.SGR_PARAMS[idx], np.int32)
                    xq_w = np.zeros(2, np.int32); xq_g = np.zeros(2, np.int32)
                    if live:
                        gps(rh.bptr(src, off), w, h, stride, rh.bptr(dgd, off), stride, int(bd > 8), rh.P(f0), w, rh.P(f1), w, rh.P(xq_w), rh.P(prm))
                    b200.lib.svt_b200_get_proj_subspace(rh.P(src, off), w, h, stride, rh.P(dgd, off), stride, int(bd > 8), rh.P(f0), w,
                                                        rh.P(f1), w, rh.P(xq_g), rh.P(prm))
                    golden.check(xq_g, xq_w if live else None, bd, w, h, kind, idx)
                    xq = np.array([int(r.integers(-96, 32)), int(r.integers(-32, 96))], np.int32)
                    ew = (ppe8 if bd == 8 else ppe16)(rh.bptr(src, off), w, h, stride, rh.bptr(dgd, off), stride, rh.P(f0), w, rh.P(f1), w,
                                                      rh.P(xq), rh.P(prm)) if live else None
                    fn = b200.lib.svt_b200_av1_lowbd_pixel_proj_error if bd == 8 else b200.lib.svt_b200_av1_highbd_pixel_proj_error
                    eg = fn(rh.P(src, off), w, h, stride, rh.P(dgd, off), stride, rh.P(f0), w, rh.P(f1), w, rh.P(xq), rh.P(prm))
                    golden.check(eg, ew, bd, w, h, kind, idx)
                xqd = np.array([-32, 31], np.int32)
                dw = np.zeros(h * w, dgd.dtype); dg = np.zeros(h * w, dgd.dtype)
                tmp = np.zeros(2 * 161 * 161 * 4 + 1024, np.int32)
                if live:
                    app(rh.bptr(dgd, off), w, h, stride, 3, rh.P(xqd), rh.bptr(dw), w, rh.P(tmp), bd, int(bd > 8))
                b200.lib.svt_b200_apply_selfguided_restoration(rh.P(dgd, off), w, h, stride, 3, rh.P(xqd), rh.P(dg), w, None, bd, int(bd > 8))
                golden.check(dg, dw if live else None, bd, w, h, kind)
