"""GPU parity: the COMPLETE open-loop ME driver (svt_b200_me_b64_picture_dev) against the reference's OWN
svt_aom_motion_estimation_b64 (motion_estimation.c:3076) with a real MeContext whose controls come from the
reference's own svt_aom_sig_deriv_me (oracle/ref_me_b64.c) -- zz-SAD pruning, pre-HME, HME level 0/1/2, reference
pruning, search-area adjustment, the 8x8-variance probe, full-pel search, candidate construction, distortions and
global-motion flags.  The outputs compared are the encoder-visible ones (MeSbResults + the pcs distortion arrays)
plus the per-reference intermediate state (do_ref, search centres, zz SADs, best SAD/MV of every live reference)."""
import ctypes as ct

import numpy as np
import pytest

import me_helpers as mh
from helpers import rng
from oracle import support as sp

pytestmark = pytest.mark.gpu


def _sequence(r, w, h, n, pan=(3, 1), noise=4.0, still_rect=None):
    """n pictures of a panning synthetic scene (optionally with a static rectangle: early-exit / stationary paths)"""
    yy, xx = np.mgrid[0:h + 160, 0:w + 160]
    base = (np.sin(xx / 13.0) * 45 + np.cos(yy / 9.0) * 35 + ((xx // 20 + yy // 28) % 2) * 70 + ((xx // 7) % 3) * 9 + 100)
    out = []
    for t in range(n):
        ox, oy = 80 + pan[0] * (t - n // 2), 80 + pan[1] * (t - n // 2)
        img = base[oy:oy + h, ox:ox + w] + r.normal(0, noise, (h, w))
        if still_rect is not None:
            x0, y0, x1, y1 = still_rect
            img[y0:y1, x0:x1] = base[80 + y0:80 + y1, 80 + x0:80 + x1] + r.normal(0, 0.6, (y1 - y0, x1 - x0))
        out.append(np.clip(img, 0, 255).astype(np.uint8))
    return out


CASES = [
    # name, W, H, preset, n_ref, poc distances, temporal layer, is_ref, extra cfg, content
    ("m8_nonbase_2p2", 448, 272, 8, (2, 2), ((-1, -3, 0, 0), (1, 3, 0, 0)), 3, 0, {}, dict(pan=(3, 1), still_rect=(128, 64, 320, 192))),
    ("m8_base_3p2", 448, 272, 8, (3, 2), ((-4, -8, -16, 0), (-4, -8, 0, 0)), 0, 1, {}, dict(pan=(2, -1))),
    ("m6_nonbase_fast", 384, 208, 6, (2, 2), ((-2, -6, 0, 0), (2, 6, 0, 0)), 2, 1, {}, dict(pan=(9, 4), noise=7.0)),
    ("m4_mrp_off_gm", 320, 256, 4, (1, 1), ((-1, 0, 0, 0), (1, 0, 0, 0)), 4, 1, dict(max_l=(1, 1), gm_enabled=1), dict(pan=(6, 0))),
    ("m2_mvsa_zero_centre", 256, 192, 2, (2, 1), ((-2, -4, 0, 0), (2, 0, 0, 0)), 2, 1, dict(max_l=(4, 3), only_l_bwd=0), dict(pan=(13, 7), noise=9.0)),
    ("m8_p_single", 320, 192, 8, (1, 0), ((-1, 0, 0, 0), (0, 0, 0, 0)), 1, 1, dict(max_l=(1, 0)), dict(pan=(-4, 2))),
    ("m10_720p_geometry", 1280, 720, 10, (2, 2), ((-1, -2, 0, 0), (1, 2, 0, 0)), 3, 0, {}, dict(pan=(5, 2), still_rect=(256, 128, 900, 500))),
]


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_me_b64_matches_reference_driver(b200, oracle, golden, case):
    import torch
    name, W, H, preset, n_ref, dist, tl, is_ref, extra, content = case
    refc = oracle.ref
    if refc is not None:
        refc.ref_set_tier(0)
    r = rng(500 + len(name))
    shapes = b200.me_plane_shapes(W, H)
    n_pic = n_ref[0] + n_ref[1] + 1
    seq = _sequence(r, W, H, 2 * 4 + 1, **content)
    mid = len(seq) // 2
    # reference pictures: list 0 looks back, list 1 forward (or back again on a base-layer picture); the step follows the distance
    pick = lambda d: seq[int(np.clip(mid + np.sign(d) * min(abs(d), 4), 0, len(seq) - 1))]  # noqa: E731
    fulls = [pick(dist[0][i]) for i in range(n_ref[0])] + [pick(dist[1][i]) for i in range(n_ref[1])]
    cur_np = mh.build_pyramid_np(seq[mid], W, H, shapes)
    refs_np = [mh.build_pyramid_np(f, W, H, shapes) for f in fulls]
    cfg = sp.me_b64_cfg(preset=preset, n_ref=n_ref, poc_dist=dist, temporal_layer_index=tl, is_ref=is_ref, **extra)
    ctrl, want = sp.ref_me_b64_picture(refc, cur_np, refs_np, shapes, cfg) if refc is not None else (None, None)
    cd = golden.value(lambda: ctrl.as_dict())  # the controls the reference derived (svt_aom_sig_deriv_me)
    ref = (lambda k: want[k]) if want is not None else (lambda k: None)  # noqa: E731
    assert n_pic == len(fulls) + 1

    def upload(planes_np):
        planes = [torch.from_numpy(p).cuda() for p in planes_np]
        return planes, b200.me_picture_desc(planes, W, H)

    cur_t, cur_d = upload(cur_np)
    ref_t, ref_d = zip(*[upload(p) for p in refs_np])
    c = b200.MeControls.from_dict(cd)
    n_pu = b200.lib.svt_b200_me_b64_num_pus(ct.byref(c))
    nb = ((W + 63) // 64) * ((H + 63) // 64)
    R = len(fulls)
    dev = dict(total_me_candidate_index=torch.zeros((nb, n_pu), dtype=torch.uint8, device="cuda"),
               me_candidate_array=torch.zeros((nb, n_pu * cd["max_cand"]), dtype=torch.uint8, device="cuda"),
               me_mv_array=torch.zeros((nb, n_pu * cd["max_refs"]), dtype=torch.int32, device="cuda"),
               distortion=torch.zeros((nb, 6), dtype=torch.int32, device="cuda"), flags=torch.zeros((nb, 2), dtype=torch.uint8, device="cuda"),
               do_ref=torch.zeros((nb, 2, 4), dtype=torch.uint8, device="cuda"), hme_centre=torch.zeros((nb, 2, 4, 2), dtype=torch.int16, device="cuda"),
               zz_sad=torch.zeros((nb, 2, 4), dtype=torch.int32, device="cuda"), best_sad=torch.zeros((R, nb, 85), dtype=torch.int32, device="cuda"),
               best_mv=torch.zeros((R, nb, 85), dtype=torch.int32, device="cuda"))
    out = b200.MeB64Results()
    for k, v in dev.items():
        setattr(out, k, v.data_ptr())
    refs_arr = (b200.MePicture * R)(*ref_d)
    assert b200.lib.svt_b200_me_b64_picture_dev(ct.byref(cur_d), refs_arr, ct.byref(c), ct.byref(out), None) == 0
    torch.cuda.synchronize()
    got = {k: v.cpu().numpy() for k, v in dev.items()}
    # intermediate state first (a mismatch there explains everything after it)
    golden.check(got["zz_sad"].view(np.uint32), ref("zz_sad"), name)
    golden.check(got["hme_centre"], ref("hme_centre"), name)
    golden.check(got["do_ref"], ref("do_ref"), name)
    k = 0
    for li in range(2):
        for ri in range(n_ref[li]):
            live = got["do_ref"][:, li, ri].astype(bool)
            # references pruned after the full-pel search (me_prune_ref) still hold their search results in both; earlier-pruned ones are undefined
            golden.check(got["best_sad"][k].view(np.uint32)[live], want and want["best_sad"][:, li, ri][live], name, li, ri)
            golden.check(got["best_mv"][k].view(np.uint32)[live], want and want["best_mv"][:, li, ri][live], name, li, ri)
            k += 1
    # what the rest of the encoder consumes
    for key, dt in (("total_me_candidate_index", np.uint8), ("me_candidate_array", np.uint8), ("distortion", np.uint32), ("flags", np.uint8)):
        golden.check(got[key].view(dt), ref(key), name, key)
    golden.check(got["me_mv_array"].view(np.uint32), ref("me_mv_array"), name)
    # the case must exercise what it is there for
    if name == "m8_nonbase_2p2":
        assert (got["do_ref"][:, :, 1] == 0).any() and (got["zz_sad"].view(np.uint32)[:, 0, 0] < cd["me_early_exit_th"]).any()
    if name == "m4_mrp_off_gm":
        assert got["flags"][:, 1].any()
