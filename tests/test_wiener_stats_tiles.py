"""GPU parity of the 8-bit Wiener statistics at the edges of the tensor-core kernel's tiling: regions whose width
runs 1-3 pixels past a multiple of the 128-pixel tile rows, heights that are not a multiple of the tile height
(30 / 36 / 28 rows at WIN 7 / 5 / 3) or of the MMA row blocks (10 / 12 / 14 rows), a region smaller than one tile,
and a flat white picture large enough that every CTA passes the kernel's fold threshold (33025 pixels) and adds
tensor memory into its int64 partial more than once (raw products of 255 x 255 on every pixel, while dgd - avg = 0).
The threshold is conservative: each accumulator entry collects the products of about 1 / T of those pixels, so this
exercises the fold and drain path, not the s32 limit itself."""
import numpy as np
import pytest

import rest_helpers as rh
from helpers import rng

pytestmark = pytest.mark.gpu


def _want(oracle, win, dgd, src, hs, he, vs, ve, W):
    if oracle.ref is not None:
        return rh.ref_stats(oracle.ref, win, dgd, src, hs, he, vs, ve, W, W, 8)
    return rh.port_stats(oracle.port, win, dgd.astype(np.uint16), src.astype(np.uint16), hs, he, vs, ve, W, W, 8)


def _check(b200, oracle, win, dgd, src, hs, he, vs, ve, W, what):
    want = _want(oracle, win, dgd, src, hs, he, vs, ve, W)
    M = np.zeros(49, np.int64); H = np.zeros(2401, np.int64)
    b200.lib.svt_b200_av1_compute_stats(win, rh.P(dgd), rh.P(src), hs, he, vs, ve, W, W, rh.P(M), rh.P(H))
    assert np.array_equal(M[:win * win], want[0]), what
    assert np.array_equal(H[:win ** 4], want[1]), what


@pytest.mark.parametrize("win", [7, 5, 3])
def test_compute_stats_tile_edges_8bit(b200, oracle, win):
    r = rng(93)
    # (region width, region height): 1-3 columns past 128 / 256, heights off the tile and block grids, one region
    # below a tile, one exactly a tile
    shapes = [(129, 31), (130, 37), (131, 70), (257, 45), (259, 29), (256, 75), (20, 10), (128, 36)]
    for (w, h) in shapes:
        hs, vs = 5, 4
        W, Hh = w + 2 * hs + 3, h + 2 * vs + 2
        dgd = r.integers(0, 256, W * Hh).astype(np.uint8); src = r.integers(0, 256, W * Hh).astype(np.uint8)
        _check(b200, oracle, win, dgd, src, hs, hs + w, vs, vs + h, W, (win, w, h))


@pytest.mark.parametrize("win", [7, 5, 3])
def test_compute_stats_flat_white_fold_8bit(b200, oracle, win):
    W, Hh, hs, he, vs, ve = 1290, 1010, 3, 1283, 3, 1003  # 1280 x 1000: more than 33025 pixels per CTA at 32 CTAs
    dgd = np.full(W * Hh, 255, np.uint8); src = np.full(W * Hh, 255, np.uint8)
    _check(b200, oracle, win, dgd, src, hs, he, vs, ve, W, (win, "white"))
    if win == 7:
        r = rng(94)
        dgd = r.integers(0, 256, W * Hh).astype(np.uint8); src = r.integers(0, 256, W * Hh).astype(np.uint8)
        _check(b200, oracle, win, dgd, src, hs, he, vs, ve, W, (win, "random"))
