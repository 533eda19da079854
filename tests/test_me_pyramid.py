"""GPU parity: Hadamard/SATD (picture_operators_c.c:188-330), the SAD pyramid T1 kernels
(motion_estimation.c:98-427; fixtures modelled on test/SadTest.cc:731-1306) and the T2 85-PU
full-pel search against the reference kernels driven in the reference's own loop order."""
import ctypes as ct

import numpy as np
import pytest

import me_helpers as mh
from helpers import rng

pytestmark = pytest.mark.gpu


def test_hadamard_and_satd(b200, oracle):
    r = rng(50)
    for n in (4, 8, 16, 32):
        for kind in ("random", "max", "min", "zero"):
            stride = n + 5
            src = {"random": r.integers(-255, 256, n * stride), "max": np.full(n * stride, 255), "min": np.full(n * stride, -255),
                   "zero": np.zeros(n * stride)}[kind].astype(np.int16)
            if oracle.ref is not None:
                want = mh.hadamard_call(oracle.ref, "svt_aom_hadamard_%dx%d_c" % (n, n), src, stride, n)
            else:
                want = mh.hadamard_call(oracle.port, "port_hadamard", src, stride, n)
            got = b200.svt_aom_hadamard(src, stride, n)
            assert np.array_equal(got, want), (n, kind)
            assert b200.svt_aom_satd(got) == int(np.abs(want.astype(np.int64)).sum())


@pytest.mark.parametrize("sub", [0, 1])
def test_ext_all_sad_and_32x32_t1(b200, oracle, golden, sub):
    """T1 kernels with carried state (Allsad8x8_CalculationTest / Allsad32x32_CalculationTest)."""
    r = rng(51)
    refc = oracle.ref
    live = refc is not None
    for trial in range(6):
        ss, rs = 64 + 8 * (trial % 2), 96
        src = r.integers(0, 256, ss * 64, dtype=np.uint8)
        ref = r.integers(0, 256, rs * 64 + 16, dtype=np.uint8)
        if trial == 0:
            src[:] = 255; ref[:] = 0
        init = lambda n: r.integers(0, 20000 if trial % 3 else mh.MAX_SAD, n).astype(np.uint32)  # noqa: E731
        st = [init(64), init(16), r.integers(0, 1 << 32, 64, dtype=np.uint64).astype(np.uint32),
              r.integers(0, 1 << 32, 16, dtype=np.uint64).astype(np.uint32)]
        mv = int(r.integers(0, 1 << 32))
        a = [x.copy() for x in st]; e16a = np.zeros(128, np.uint32); e8 = np.zeros(512, np.uint32)
        if live:
            f = refc.svt_ext_all_sad_calculation_8x8_16x16_c; f.restype = None
            f(mh.P(src), ct.c_uint32(ss), mh.P(ref), ct.c_uint32(rs), ct.c_uint32(mv), mh.P(a[0]), mh.P(a[1]), mh.P(a[2]), mh.P(a[3]),
              mh.P(e16a), mh.P(e8), ct.c_bool(bool(sub)))
        b = [x.copy() for x in st]; e16b = np.zeros(128, np.uint32)
        b200.lib.svt_b200_ext_all_sad_calculation_8x8_16x16(mh.P(src), ss, mh.P(ref), rs, mv, mh.P(b[0]), mh.P(b[1]), mh.P(b[2]),
                                                            mh.P(b[3]), mh.P(e16b), mh.P(e8), sub)
        golden.check(b + [e16b], (a + [e16a]) if live else None)
        # 32x32 / 64x64 stage on top of the eight 16x16 SADs
        s2 = [init(4), init(1), init(4), init(1)]
        a2 = [x.copy() for x in s2]; e32a = np.zeros(32, np.uint32)
        if live:
            g = refc.svt_ext_eight_sad_calculation_32x32_64x64_c; g.restype = None
            g(mh.P(e16a), mh.P(a2[0]), mh.P(a2[1]), mh.P(a2[2]), mh.P(a2[3]), ct.c_uint32(mv), mh.P(e32a))
        b2 = [x.copy() for x in s2]; e32b = np.zeros(32, np.uint32)
        b200.lib.svt_b200_ext_eight_sad_calculation_32x32_64x64(mh.P(e16b), mh.P(b2[0]), mh.P(b2[1]), mh.P(b2[2]), mh.P(b2[3]), mv,
                                                                mh.P(e32b))
        golden.check(b2 + [e32b], (a2 + [e32a]) if live else None)
        # 1-point variants
        s3 = [init(4), init(1), init(4), init(1)]
        a3 = [x.copy() for x in s3]; o16a = np.zeros(1, np.uint32); o8a = np.zeros(4, np.uint32)
        if live:
            h = refc.svt_ext_sad_calculation_8x8_16x16_c; h.restype = None
            h(mh.P(src), ct.c_uint32(ss), mh.P(ref), ct.c_uint32(rs), mh.P(a3[0]), mh.P(a3[1]), mh.P(a3[2]), mh.P(a3[3]), ct.c_uint32(mv),
              mh.P(o16a), mh.P(o8a), ct.c_bool(bool(sub)))
        b3 = [x.copy() for x in s3]; o16b = np.zeros(1, np.uint32); o8b = np.zeros(4, np.uint32)
        b200.lib.svt_b200_ext_sad_calculation_8x8_16x16(mh.P(src), ss, mh.P(ref), rs, mh.P(b3[0]), mh.P(b3[1]), mh.P(b3[2]),
                                                        mh.P(b3[3]), mv, mh.P(o16b), mh.P(o8b), sub)
        golden.check(b3 + [o16b, o8b], (a3 + [o16a, o8a]) if live else None)
        s16 = init(16); s4 = [init(4), init(1), init(4), init(1)]
        a4 = [x.copy() for x in s4]; o32a = np.zeros(4, np.uint32)
        if live:
            k = refc.svt_ext_sad_calculation_32x32_64x64_c; k.restype = None
            k(mh.P(s16), mh.P(a4[0]), mh.P(a4[1]), mh.P(a4[2]), mh.P(a4[3]), ct.c_uint32(mv), mh.P(o32a))
        b4 = [x.copy() for x in s4]; o32b = np.zeros(4, np.uint32)
        b200.lib.svt_b200_ext_sad_calculation_32x32_64x64(mh.P(s16), mh.P(b4[0]), mh.P(b4[1]), mh.P(b4[2]), mh.P(b4[3]), mv, mh.P(o32b))
        golden.check(b4 + [o32b], (a4 + [o32a]) if live else None)
    buf = np.zeros(85, np.uint32)
    b200.lib.svt_b200_initialize_buffer_32bits(mh.P(buf), 21, 1, mh.MAX_SAD)
    assert (buf == mh.MAX_SAD).all()


def test_fullpel_search_batch(b200, oracle):
    """T2: many (b64, search area) items over one padded picture in one launch."""
    r = rng(52)
    W, H, pad = 256, 128, 72
    pitch = W + 2 * pad
    cur = r.integers(0, 256, pitch * (H + 2 * pad), dtype=np.uint8)
    refp = np.roll(cur, 2 * pitch - 3) ^ r.integers(0, 8, cur.size, dtype=np.uint8)
    refp[: pitch * 80] = 90   # flat band: forces ties in the top row of blocks
    cur[: pitch * 80] = 90
    lst = []
    cfgs = [(8, 3, 0), (16, 9, 0), (11, 4, 1), (21, 6, 0), (8, 4, 1), (3, 1, 0)]
    k = 0
    for by in range(0, H, 64):
        for bx in range(0, W, 64):
            sa_w, sa_h, sub = cfgs[k % len(cfgs)]; k += 1
            ox, oy = -(sa_w // 2) + (k % 5) - 2, -(sa_h // 2) + (k % 3) - 1
            lst.append(((pad + by) * pitch + pad + bx, (pad + by + oy) * pitch + pad + bx + ox, pitch, pitch, sa_w, sa_h, ox, oy, sub, 0, 0, 0,
                        [0, 0]))
    items = np.array(lst, dtype=b200.FULLPEL_ITEM_DTYPE)
    sad, mv = b200.fullpel_search_batch_host(cur, refp, items)
    for i, it in enumerate(items):
        args = (cur, int(it["src_off"]), pitch, refp, int(it["ref_off"]), pitch, int(it["sa_w"]), int(it["sa_h"]), int(it["org_x"]),
                int(it["org_y"]), int(it["sub_sad"]))
        want = mh.ref_fullpel(oracle.ref, *args) if oracle.ref is not None else mh.port_fullpel(oracle.port, *args)
        assert np.array_equal(sad[i], want[0]), i
        assert np.array_equal(mv[i], want[1]), i


def test_hadamard_path_fwht_and_cul_level(b200, oracle, golden):
    """the remaining dispatched helpers of the SATD / transform / quantiser group against the reference's C functions:
    hadamard_path_c (enc_mode_config.c:2147, all 22 block sizes, incl. the residual / coefficients it leaves behind),
    svt_av1_fwht4x4_c (transforms.c:3099) and svt_av1_compute_cul_level_c (full_loop.c:1449)"""
    import ctypes as ct
    r = rng(61)
    refc = oracle.ref
    live = refc is not None

    class Buf2D(ct.Structure):
        _fields_ = [("buf", ct.c_void_p), ("buf0", ct.c_void_p), ("width", ct.c_int), ("height", ct.c_int), ("stride", ct.c_int)]
    if live:
        refc.hadamard_path_c.argtypes = [Buf2D] * 4 + [ct.c_uint8]
        refc.hadamard_path_c.restype = ct.c_uint32
    wide = [4, 4, 8, 8, 8, 16, 16, 16, 32, 32, 32, 64, 64, 64, 128, 128, 4, 16, 8, 32, 16, 64]
    for bsize in range(22):
        side, stride = wide[bsize], 160
        inp = r.integers(0, 256, stride * 130, dtype=np.uint8)
        prd = r.integers(0, 256, stride * 130, dtype=np.uint8)
        if bsize % 3 == 0:
            inp[:], prd[:] = 255, 0  # largest residuals
        outs = []
        for fn, B in ([(refc.hadamard_path_c, Buf2D)] if live else []) + [(b200.lib.svt_b200_hadamard_path, b200.Buf2D)]:
            res = np.full(40 * 40, -77, np.int16)
            cof = np.full(32 * 32, -77, np.int32)
            cost = fn(B(res.ctypes.data, None, 0, 0, 40), B(cof.ctypes.data, None, 0, 0, side), B(inp.ctypes.data, None, 0, 0, stride),
                      B(prd.ctypes.data, None, 0, 0, stride), bsize)
            outs.append((int(cost), res, cof))
        golden.check(outs[-1], outs[0] if live else None, bsize)
    if live:
        refc.svt_av1_fwht4x4_c.restype = None
    for k in range(40):
        stride = 4 + (k % 5)
        src = r.integers(-1023 if k % 2 else -255, 1024 if k % 2 else 256, 4 * stride).astype(np.int16)
        want = np.zeros(16, np.int32); got = np.zeros(16, np.int32)
        if live:
            refc.svt_av1_fwht4x4_c(mh.P(src), mh.P(want), ct.c_uint32(stride))
        b200.lib.svt_b200_av1_fwht4x4(mh.P(src), mh.P(got), stride)
        golden.check(got, want if live else None, k)
    if live:
        refc.svt_av1_compute_cul_level_c.restype = ct.c_uint8
    for k in range(60):
        n = [16, 64, 256, 1024][k % 4]
        scan = r.permutation(n).astype(np.int16)
        q = np.zeros(n, np.int32)
        nz = r.integers(0, n, max(1, n // (2 + k % 7)))
        q[nz] = r.integers(-3 if k % 3 else -200, 4 if k % 3 else 200, nz.size)
        if k % 5 == 0:
            q[0] = 0
        for eob in (0, 1, n // 2, n):
            e1, e2 = ct.c_uint16(eob), ct.c_uint16(eob)
            want = refc.svt_av1_compute_cul_level_c(mh.P(scan), mh.P(q), ct.byref(e1)) if live else None
            got = b200.lib.svt_b200_av1_compute_cul_level(mh.P(scan), mh.P(q), ct.byref(e2))
            golden.check(got, want, k, eob)
