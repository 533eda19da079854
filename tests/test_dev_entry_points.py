"""GPU parity of the device-resident T2 batch entry points that only had `_host` twins (or nothing) tested:
svt_b200_sad_search_batch_dev, svt_b200_fullpel_search_batch_dev, svt_b200_hadamard_satd_batch_dev and
svt_b200_sgr_units_dev -- device pointers + a stream, results compared with per-item reference calls
(svt_sad_loop_kernel_c, the reference full-pel kernels, svt_aom_hadamard_NxN_c + svt_aom_satd_c,
svt_av1_selfguided_restoration_c at 8 / 10 / 12 bit)."""
import ctypes as ct

import numpy as np
import pytest

import me_helpers as mh
import rest_helpers as rh
from helpers import rng, sad_loop_call

pytestmark = pytest.mark.gpu


def _dev(torch, a):
    return torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1)).cuda()


def test_sad_search_batch_dev(b200, oracle):
    import torch
    lib, fn = (oracle.ref, "svt_sad_loop_kernel_c") if oracle.ref is not None else (oracle.port, "port_sad_loop")
    r = rng(206)
    W, H, pad = 448, 256, 80
    pitch = W + 2 * pad
    cur = r.integers(0, 256, pitch * (H + 2 * pad), dtype=np.uint8)
    refp = np.roll(cur, 2 * pitch + 7) ^ r.integers(0, 4, cur.size, dtype=np.uint8)
    lst = []
    for by in range(0, H - 63, 64):
        for bx in range(0, W - 63, 64):
            # the HME shapes (block, area), one SUB_SAD item (doubled block pitch, halved rows), one skip_search_line item
            for (bw, bh, sa_w, sa_h, mult, skip) in [(64, 64, 8, 3, 1, 0), (32, 32, 16, 9, 1, 0), (16, 16, 48, 40, 1, 0), (64, 32, 8, 3, 2, 0),
                                                      (16, 16, 24, 12, 1, 1)]:
                ox, oy = bx - sa_w // 2, by - sa_h // 2
                lst.append(((pad + by) * pitch + pad + bx, (pad + oy) * pitch + pad + ox, pitch * mult, pitch * mult, pitch, bw, bh, sa_w, sa_h,
                            skip, 0))
    items = np.array(lst, dtype=b200.SAD_ITEM_DTYPE)
    d_cur, d_ref, d_items = _dev(torch, cur), _dev(torch, refp), _dev(torch, items)
    d_res = torch.zeros(len(items) * 8, dtype=torch.uint8, device="cuda")
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        rc = b200.lib.svt_b200_sad_search_batch_dev(d_cur.data_ptr(), d_ref.data_ptr(), d_items.data_ptr(), len(items), d_res.data_ptr(), 64, 64, 48, 40,
                                                    2, st.cuda_stream)
    assert rc == 0
    st.synchronize()
    res = d_res.cpu().numpy().view(b200.SAD_RESULT_DTYPE)
    # the host twin of the same call must agree too
    host = b200.sad_search_batch_host(cur, refp, items)
    for it, rr, hh in zip(items, res, host):
        mult = int(it["src_stride"]) // pitch
        want = sad_loop_call(lib, fn, cur, int(it["src_off"]), pitch * mult, refp, int(it["ref_off"]), pitch * mult, int(it["block_h"]),
                             int(it["block_w"]), pitch, int(it["skip_search_line"]), int(it["sa_w"]), int(it["sa_h"]))
        assert (int(rr["best_sad"]), int(rr["x"]), int(rr["y"])) == want
        assert (int(hh["best_sad"]), int(hh["x"]), int(hh["y"])) == want


def test_fullpel_search_batch_dev(b200, oracle):
    import torch
    r = rng(207)
    W, H, pad = 320, 192, 72
    pitch = W + 2 * pad
    cur = r.integers(0, 256, pitch * (H + 2 * pad), dtype=np.uint8)
    refp = np.roll(cur, pitch - 2) ^ r.integers(0, 8, cur.size, dtype=np.uint8)
    lst = []
    cfgs = [(8, 3, 1), (8, 8, 0), (24, 24, 1), (16, 9, 0), (11, 4, 1), (3, 1, 0)]  # incl. the M8 / M6 / M4 full-pel areas of the bench presets
    k = 0
    for by in range(0, H, 64):
        for bx in range(0, W, 64):
            sa_w, sa_h, sub = cfgs[k % len(cfgs)]
            k += 1
            ox, oy = -(sa_w // 2) + (k % 5) - 2, -(sa_h // 2) + (k % 3) - 1
            lst.append(((pad + by) * pitch + pad + bx, (pad + by + oy) * pitch + pad + bx + ox, pitch, pitch, sa_w, sa_h, ox, oy, sub, 0, 0, 0, [0, 0]))
    items = np.array(lst, dtype=b200.FULLPEL_ITEM_DTYPE)
    d_cur, d_ref, d_items = _dev(torch, cur), _dev(torch, refp), _dev(torch, items)
    d_sad = torch.zeros((len(items), 85), dtype=torch.int32, device="cuda")
    d_mv = torch.zeros_like(d_sad)
    s = torch.cuda.current_stream().cuda_stream
    assert b200.lib.svt_b200_fullpel_search_batch_dev(d_cur.data_ptr(), d_ref.data_ptr(), d_items.data_ptr(), len(items), d_sad.data_ptr(),
                                                      d_mv.data_ptr(), s) == 0
    torch.cuda.synchronize()
    sad, mv = d_sad.cpu().numpy().view(np.uint32), d_mv.cpu().numpy().view(np.uint32)
    for i, it in enumerate(items):
        args = (cur, int(it["src_off"]), pitch, refp, int(it["ref_off"]), pitch, int(it["sa_w"]), int(it["sa_h"]), int(it["org_x"]), int(it["org_y"]),
                int(it["sub_sad"]))
        want = mh.ref_fullpel(oracle.ref, *args) if oracle.ref is not None else mh.port_fullpel(oracle.port, *args)
        assert np.array_equal(sad[i], want[0]), i
        assert np.array_equal(mv[i], want[1]), i


def test_hadamard_satd_batch_dev(b200, oracle):
    """fused Hadamard + sum |coeff| per item == svt_aom_hadamard_NxN_c followed by svt_aom_satd_c (TPL's use,
    src_ops_process.c); with and without the coefficient plane; extreme residuals included"""
    import torch
    r = rng(208)
    stride, rows = 160, 96
    res = r.integers(-255, 256, stride * rows).astype(np.int16)
    res[: stride * 32] = r.choice(np.array([-255, 255], np.int16), stride * 32)  # worst-case magnitudes
    lst, coff = [], 0
    for n in (4, 8, 16, 32):
        for (y, x) in [(0, 0), (32, 64), (64 - n, 128 - n), (40, 3)]:
            lst.append((y * stride + x, coff, stride, n))
            coff += n * n
    items = np.array(lst, dtype=b200.HADAMARD_ITEM_DTYPE)
    satd_c = oracle.ref.svt_aom_satd_c if oracle.ref is not None else None
    want_c, want_s = np.zeros(coff, np.int32), np.zeros(len(items), np.int32)
    for i, it in enumerate(items):
        n = int(it["size"])
        src = res[int(it["src_off"]):]
        if oracle.ref is not None:
            c = mh.hadamard_call(oracle.ref, "svt_aom_hadamard_%dx%d_c" % (n, n), src, stride, n)
            satd_c.restype = ct.c_int
            want_s[i] = satd_c(mh.P(c), n * n)
        else:
            c = mh.hadamard_call(oracle.port, "port_hadamard", src, stride, n)
            want_s[i] = int(np.abs(c.astype(np.int64)).sum())
        want_c[int(it["coeff_off"]):int(it["coeff_off"]) + n * n] = c
    d_res, d_items = _dev(torch, res), _dev(torch, items)
    s = torch.cuda.current_stream().cuda_stream
    for with_coeff in (True, False):
        d_coeff = torch.full((coff,), -7, dtype=torch.int32, device="cuda")
        d_satd = torch.full((len(items),), -7, dtype=torch.int32, device="cuda")
        rc = b200.lib.svt_b200_hadamard_satd_batch_dev(d_res.data_ptr(), d_items.data_ptr(), len(items), d_coeff.data_ptr() if with_coeff else None,
                                                       d_satd.data_ptr(), s)
        assert rc == 0
        torch.cuda.synchronize()
        assert np.array_equal(d_satd.cpu().numpy(), want_s), with_coeff
        if with_coeff:
            assert np.array_equal(d_coeff.cpu().numpy(), want_c)
    # an item with an unsupported size must be rejected, not overrun shared memory
    bad = items[:1].copy()
    bad["size"] = 24
    d_bad = _dev(torch, bad)
    d_satd = torch.zeros(1, dtype=torch.int32, device="cuda")
    rc = b200.lib.svt_b200_hadamard_satd_batch_dev(d_res.data_ptr(), d_bad.data_ptr(), 1, None, d_satd.data_ptr(), s)
    torch.cuda.synchronize()
    assert rc == 0 and int(d_satd[0]) == -1  # sentinel written for the invalid item


@pytest.mark.parametrize("bd", [8, 10, 12])
def test_sgr_units_dev(b200, oracle, golden, bd):
    """processing units of a padded device plane through svt_b200_sgr_units_dev == svt_av1_selfguided_restoration_c per unit"""
    import torch
    r = rng(209 + bd)
    W, H, pad = 200, 136, 8
    stride = W + 2 * pad
    mx = (1 << bd) - 1
    plane = r.integers(0, mx + 1, stride * (H + 2 * pad)).astype(np.uint8 if bd == 8 else np.uint16)
    plane[: stride * 40] = mx  # saturated band
    lst, foff = [], 0
    k = 0
    for y0 in range(0, H, 64):
        for x0 in range(0, W, 64):
            w, h = min(64, W - x0), min(64, H - y0)
            idx = (0, 3, 9, 10, 13, 14, 15, 5)[k % 8]
            k += 1
            lst.append(((pad + y0) * stride + pad + x0, foff, foff, stride, w, w, h, idx, 0))
            foff += w * h
    units = np.array(lst, dtype=b200.SGR_UNIT_DTYPE)
    d_plane, d_units = _dev(torch, plane), _dev(torch, units)
    d_f0 = torch.full((foff,), -12345, dtype=torch.int32, device="cuda")
    d_f1 = torch.full((foff,), -12345, dtype=torch.int32, device="cuda")
    s = torch.cuda.current_stream().cuda_stream
    assert b200.lib.svt_b200_sgr_units_dev(d_plane.data_ptr(), d_units.data_ptr(), len(units), d_f0.data_ptr(), d_f1.data_ptr(), bd, 64, 64, s) == 0
    torch.cuda.synchronize()
    f0, f1 = d_f0.cpu().numpy(), d_f1.cpu().numpy()
    for u in units:
        w, h, o = int(u["w"]), int(u["h"]), int(u["flt0_off"])
        want = rh.ref_selfguided(oracle.ref, plane, int(u["dgd_off"]), w, h, stride, int(u["params_idx"]), bd) if oracle.ref is not None else None
        prm = rh.SGR_PARAMS[int(u["params_idx"])]
        if prm[0]:  # r0 == 0: flt0 is not produced by the reference (left untouched)
            golden.check(f0[o:o + w * h], want and want[0], bd, int(u["params_idx"]), "flt0")
        if prm[1]:
            golden.check(f1[o:o + w * h], want and want[1], bd, int(u["params_idx"]), "flt1")
