"""GPU parity for CDEF: T1 kernels vs the reference C functions (fixtures after test/CdefTest.cc) and
the T2 whole-picture strength search / apply vs the reference functions driven in the order of
cdef_seg_search (cdef_process.c:106-352)."""
import ctypes as ct

import numpy as np
import pytest

import cdef_helpers as ch
from helpers import rng

pytestmark = pytest.mark.gpu
BS, VL = 144, 0x7f7f


def test_find_dir_and_filter_block_t1(b200, oracle, golden):
    r = rng(70)
    refc = oracle.ref
    if refc is not None:
        fd = refc.svt_aom_cdef_find_dir_c; fd.restype = ct.c_uint8
        fb = refc.svt_cdef_filter_block_c; fb.restype = None
    for bd in (8, 10, 12):
        cs = bd - 8
        for trial in range(12):
            tile = r.integers(0, 1 << bd, 70 * BS).astype(np.uint16)
            if trial % 4 == 1:  # directional content
                yy, xx = np.mgrid[0:70, 0:BS]
                tile = (((xx + yy * (trial - 5)) // 3 % 2) * ((1 << bd) - 1)).astype(np.uint16).reshape(-1)
            if trial % 4 == 2:  # frame-edge sentinels around the block
                t2 = tile.reshape(70, BS); t2[:12] = VL; t2[:, :18] = VL; tile = t2.reshape(-1)
            off = 12 * BS + 18
            va, vb = ct.c_int32(0), ct.c_int32(0)
            want = (fd(ch.P(tile, off), BS, ct.byref(va), cs), va.value) if refc is not None else None
            db = b200.lib.svt_b200_aom_cdef_find_dir(ch.P(tile, off), BS, ct.byref(vb), cs)
            golden.check((db, vb.value), want)
            v1, v2, o1, o2 = ct.c_int32(0), ct.c_int32(0), ct.c_uint8(0), ct.c_uint8(0)
            b200.lib.svt_b200_aom_cdef_find_dir_dual(ch.P(tile, off), ch.P(tile, off + 8), BS, ct.byref(v1), ct.byref(v2), cs,
                                                     ct.byref(o1), ct.byref(o2))
            assert (o1.value, v1.value) == (db, vb.value)
            for bsize in (0, 1, 2, 3):
                for subs in (1, 2):
                    pri = int(r.integers(0, 16)) << cs
                    sec = int([0, 1, 2, 4][int(r.integers(0, 4))]) << cs
                    d = int(r.integers(0, 8)); pd = int(r.integers(3, 7)) + cs; sd = int(r.integers(3, 7)) + cs
                    w = 4 << (bsize in (2, 3)); h = 4 << (bsize in (1, 3))
                    a = np.full(h * 16, 0xabcd, np.uint16); b = a.copy()
                    if refc is not None:
                        fb(None, ch.P(a), 16, ch.P(tile, off), pri, sec, d, pd, sd, bsize, cs, ct.c_uint8(subs))
                    b200.lib.svt_b200_cdef_filter_block(None, ch.P(b), 16, ch.P(tile, off), pri, sec, d, pd, sd, bsize, cs, subs)
                    golden.check(b, a if refc is not None else None, bd, trial, bsize, subs)
                    if bd == 8:
                        a8 = np.full(h * 16, 0xcd, np.uint8); b8 = a8.copy()
                        if refc is not None:
                            fb(ch.P(a8), None, 16, ch.P(tile, off), pri, sec, d, pd, sd, bsize, cs, ct.c_uint8(subs))
                        b200.lib.svt_b200_cdef_filter_block(ch.P(b8), None, 16, ch.P(tile, off), pri, sec, d, pd, sd, bsize, cs, subs)
                        golden.check(b8, a8 if refc is not None else None)


def test_compute_cdef_dist_t1(b200, oracle, golden):
    r = rng(71)
    refc = oracle.ref
    if refc is not None:
        f16 = refc.svt_aom_compute_cdef_dist_c; f16.restype = ct.c_uint64
        f8 = refc.svt_aom_compute_cdef_dist_8bit_c; f8.restype = ct.c_uint64
    for bd in (8, 10):
        cs = bd - 8
        for bsize in (0, 1, 2, 3):
            for pli in (0, 1):
                for subs in (1, 2):
                    cnt = int(r.integers(1, 40))
                    dl = np.stack([r.integers(0, 8, cnt), r.integers(0, 8, cnt)], 1).astype(np.uint8).reshape(-1)
                    dst = r.integers(0, 1 << bd, 64 * 80).astype(np.uint16)
                    src = np.clip(r.integers(0, 1 << bd, 64 * 64), 0, (1 << bd) - 1).astype(np.uint16)
                    a = f16(ch.P(dst), 80, ch.P(src), ch.P(dl), cnt, bsize, cs, pli, ct.c_uint8(subs)) if refc is not None else None
                    b = b200.lib.svt_b200_compute_cdef_dist_16bit(ch.P(dst), 80, ch.P(src), ch.P(dl), cnt, bsize, cs, pli, subs)
                    golden.check(b, a, bd, bsize, pli, subs)
                    if bd == 8:
                        d8, s8 = dst.astype(np.uint8), src.astype(np.uint8)
                        a = f8(ch.P(d8), 80, ch.P(s8), ch.P(dl), cnt, bsize, cs, pli, ct.c_uint8(subs)) if refc is not None else None
                        b = b200.lib.svt_b200_compute_cdef_dist_8bit(ch.P(d8), 80, ch.P(s8), ch.P(dl), cnt, bsize, cs, pli, subs)
                        golden.check(b, a)


def test_search_one_dual_t1(b200, oracle, golden):
    r = rng(72)
    refc = oracle.ref
    if refc is not None:
        f = refc.svt_search_one_dual_c; f.restype = ct.c_uint64
    for (sb, ng, nb, start) in [(37, 8, 0, 0), (60, 16, 2, 0), (11, 64, 3, 0), (25, 12, 1, 4)]:
        m = r.integers(0, 1 << 30, (2, sb, 64)).astype(np.uint64)
        m[0, :, 3] = m[0, :, 5]  # ties
        rows = [(ct.c_void_p * sb)(*[m[p, i].ctypes.data for i in range(sb)]) for p in range(2)]
        mse = (ct.c_void_p * 2)(ct.cast(rows[0], ct.c_void_p), ct.cast(rows[1], ct.c_void_p))
        la = np.zeros(8, np.int32); lb = np.zeros(8, np.int32)
        la[:nb] = r.integers(start, ng, nb); lb[:nb] = r.integers(start, ng, nb)
        la2, lb2 = la.copy(), lb.copy()
        want = (f(ch.P(la), ch.P(lb), nb, mse, sb, start, ng), la, lb) if refc is not None else None
        b = b200.lib.svt_b200_search_one_dual(ch.P(la2), ch.P(lb2), nb, mse, sb, start, ng)
        golden.check((b, la2, lb2), want)


@pytest.mark.parametrize("bd,subs", [(8, 1), (8, 4), (10, 2)])
def test_cdef_search_frame_t2(b200, oracle, bd, subs):
    import torch
    r = rng(73 + bd + subs)
    W, H = 208, 136
    rec, src, skip = ch.make_frame(r, W, H, bd)
    sy = [0, 4, 9, 17, 35, 63, 2]
    su = [0, 4, -1, 17, 20, 63, 3]
    if oracle.ref is not None:
        want = ch.ref_cdef_search(oracle.ref, rec, src, skip, W, H, bd, 5, subs, sy, su)
    else:
        want = ch.port_cdef_search(oracle.port, rec, src, skip, W, H, bd, 5, subs, sy, su)
    dt = np.uint8 if bd == 8 else np.int16
    drec = [torch.from_numpy(p.astype(dt)).cuda() for p in rec]
    dsrc = [torch.from_numpy(p.astype(dt)).cuda() for p in src]
    dskip = torch.from_numpy(skip).cuda()
    dsy = torch.tensor(sy, dtype=torch.int32).cuda(); dsu = torch.tensor(su, dtype=torch.int32).cuda()
    nfb = ((W + 63) // 64) * ((H + 63) // 64)
    dmse = torch.zeros((2, nfb, len(sy)), dtype=torch.int64).cuda()
    ddir = torch.zeros((nfb, 64), dtype=torch.uint8).cuda(); dvar = torch.zeros((nfb, 64), dtype=torch.int32).cuda()
    fr = b200.cdef_frame_desc(drec, dsrc, W, H, bd, 5, subs)
    rc = b200.lib.svt_b200_cdef_search_frame_dev(ct.byref(fr), dskip.data_ptr(), dsy.data_ptr(), dsu.data_ptr(), len(sy), dmse.data_ptr(),
                                                 ddir.data_ptr(), dvar.data_ptr(), None)
    assert rc == 0
    torch.cuda.synchronize()
    got = dmse.cpu().numpy().astype(np.uint64)
    assert np.array_equal(ddir.cpu().numpy(), want[1])
    assert np.array_equal(dvar.cpu().numpy(), want[2])
    assert np.array_equal(got, want[0])
