"""GPU parity: T2 whole-picture open-loop ME (pyramid build, HME L0/L1/L2, centre, zero check,
85-PU full-pel search) vs the reference kernels driven by a numpy restatement of the reference's
driver arithmetic (tests/me_helpers.py: motion_estimation.c:820-1520)."""
import ctypes as ct

import numpy as np
import pytest

import me_helpers as mh
from helpers import rng

pytestmark = pytest.mark.gpu


def _content(r, w, h, shift):
    yy, xx = np.mgrid[0:h + 64, 0:w + 64]
    base = (np.sin(xx / 11.0) * 50 + np.cos(yy / 7.0) * 40 + ((xx // 24 + yy // 24) % 2) * 60 + 110)
    noise = r.normal(0, 6, base.shape)
    img = np.clip(base + noise, 0, 255).astype(np.uint8)
    return np.ascontiguousarray(img[32 + shift[1]:32 + shift[1] + h, 32 + shift[0]:32 + shift[0] + w])


def test_downsample_2d_t1(b200, oracle, golden):
    r = rng(120)
    if oracle.ref is not None:
        f = oracle.ref.svt_aom_downsample_2d_c; f.restype = None
    for (w, h, step) in [(64, 48, 2), (130, 70, 2), (64, 64, 4)]:
        src = r.integers(0, 256, (h, w + 6)).astype(np.uint8)
        ow, oh = w // step, h // step
        a = np.zeros((oh, ow + 3), np.uint8); b = a.copy()
        if oracle.ref is not None:
            f(mh.P(src), w + 6, w, h, mh.P(a), ow + 3, step)
        b200.lib.svt_b200_downsample_2d(mh.P(src), w + 6, w, h, mh.P(b), ow + 3, step)
        golden.check(b, a if oracle.ref is not None else None)


@pytest.mark.parametrize("sub,check0", [(0, 1), (1, 0)])
def test_me_picture_pipeline(b200, oracle, golden, sub, check0):
    import torch
    r = rng(121 + sub)
    W, H = 320, 200  # 5 x 4 b64s, last row 8 high, all edges exercised
    shapes = b200.me_plane_shapes(W, H)
    cur_full = _content(r, W, H, (0, 0))
    ref_fulls = [_content(r, W, H, (5, -3)), _content(r, W, H, (-19, 9))]
    params = [dict(hme_l0_sa_w=16, hme_l0_sa_h=8, hme_l1_sa_w=8, hme_l1_sa_h=3, hme_l2_sa_w=8, hme_l2_sa_h=3, me_sa_w=8, me_sa_h=3,
                   hme_sub_sad=sub, me_sub_sad=sub, check_zero_centre=check0),
              dict(hme_l0_sa_w=32, hme_l0_sa_h=12, hme_l1_sa_w=8, hme_l1_sa_h=3, hme_l2_sa_w=8, hme_l2_sa_h=3, me_sa_w=16, me_sa_h=5,
                   hme_sub_sad=sub, me_sub_sad=0, check_zero_centre=check0)]
    cur_np = mh.build_pyramid_np(cur_full, W, H, shapes)
    refs_np = [mh.build_pyramid_np(f, W, H, shapes) for f in ref_fulls]
    want = mh.ref_me_picture(oracle.ref, cur_np, refs_np, shapes, W, H, params) if oracle.ref is not None else [None] * 4

    def upload(full):
        planes = [torch.zeros((s[0], s[1]), dtype=torch.uint8, device="cuda") for s in shapes]
        pad = shapes[2][2]
        planes[2][pad:pad + H, pad:pad + W] = torch.from_numpy(full).cuda()
        # full-resolution padding is the caller's job (svt_aom_generate_padding on the input picture)
        planes[2].copy_(torch.from_numpy(mh.pad_np(planes[2].cpu().numpy(), pad, W, H)))
        d = b200.me_picture_desc(planes, W, H)
        assert b200.lib.svt_b200_build_hme_pyramid_dev(ct.byref(d), None) == 0
        return planes, d

    cur_t, cur_d = upload(cur_full)
    ref_t, ref_d = zip(*[upload(f) for f in ref_fulls])
    torch.cuda.synchronize()
    for lvl in range(3):  # the device pyramid equals the numpy one
        assert np.array_equal(cur_t[lvl].cpu().numpy(), cur_np[lvl]), lvl
    nb = ((W + 63) // 64) * ((H + 63) // 64)
    R = 2
    d_sad = torch.zeros((R, nb, 85), dtype=torch.int32, device="cuda"); d_mv = torch.zeros_like(d_sad)
    d_c = torch.zeros((R, nb, 2), dtype=torch.int16, device="cuda"); d_hs = torch.zeros((R, nb), dtype=torch.int64, device="cuda")
    refs_arr = (b200.MePicture * R)(*ref_d)
    prm_arr = (b200.MeParams * R)()
    for i, p in enumerate(params):
        for k, v in p.items():
            setattr(prm_arr[i], k, v)
    rc = b200.lib.svt_b200_me_picture_dev(ct.byref(cur_d), refs_arr, prm_arr, R, d_sad.data_ptr(), d_mv.data_ptr(), d_c.data_ptr(),
                                          d_hs.data_ptr(), None)
    assert rc == 0
    torch.cuda.synchronize()
    golden.check(d_c.cpu().numpy(), want[2])
    golden.check(d_hs.cpu().numpy().astype(np.uint64), want[3])
    golden.check(d_sad.cpu().numpy().astype(np.uint32), want[0])
    golden.check(d_mv.cpu().numpy().astype(np.uint32), want[1])
