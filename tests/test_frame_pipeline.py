"""GPU parity at picture scale: one frame through the T2 pipeline (the path bench.py times) against
the reference arm -- the reference's own kernels driven by oracle/ref_driver.c -- bit for bit, at a
small size and at BASELINE's 1920x1080 (through the committed digests of tests/golden/frame_*.json where
oracle/_ref is not built)."""
import pytest

pytestmark = pytest.mark.gpu


# (width, height, bit_depth, preset): small cases + every BASELINE.json configuration (configs[1..4]) at full size
FRAME_CASES = [(384, 256, 8, 8), (384, 256, 10, 6), (448, 320, 10, 4), (1920, 1080, 8, 8), (1920, 1080, 10, 6), (3840, 2160, 8, 8),
               (3840, 2160, 10, 4)]


@pytest.mark.parametrize("case", FRAME_CASES, ids=lambda c: "%dx%d_b%d_m%d" % c)
def test_frame_pipeline_matches_reference(b200, case):
    """every output of the T2 frame pipeline == the reference's own kernels (8-bit: svt_av1_inv_txfm_add, svt_av1_compute_stats,
    svt_av1_wiener_convolve_add_src ...; 10-bit: svt_aom_inv_transform_recon with CONVERT_TO_BYTEPTR planes as in
    full_loop.c:1843-1846, svt_av1_highbd_quantize_fp_qm, svt_compute_cdef_dist_16bit, svt_av1_compute_stats_highbd,
    svt_av1_highbd_wiener_convolve_add_src as in restoration.c:933)"""
    import torch
    import bench
    from svt_av1_psy_b200.pipeline import FramePipeline
    from svt_av1_psy_b200.workload import FrameWorkload
    w, h, bd, m = case
    fp = FramePipeline(FrameWorkload(w, h, bit_depth=bd, preset=m), torch)
    bench.check_against_reference(fp, torch)
    # size-independent property: a second pass over the same inputs is idempotent
    a = fp.final.clone(), fp.qcoeff.clone(), fp.me["me_mv_array"].clone()
    fp.step()
    torch.cuda.synchronize()
    assert torch.equal(a[0], fp.final) and torch.equal(a[1], fp.qcoeff) and torch.equal(a[2], fp.me["me_mv_array"])


def test_cdef_apply_recomputes_directions_when_none_given(b200):
    """svt_b200_cdef_apply_frame_dev with d_dir = d_var = NULL finds the directions itself; the result
    must equal the apply that reuses the arrays of the search."""
    import ctypes as ct
    import torch
    from svt_av1_psy_b200 import dsp
    from svt_av1_psy_b200.pipeline import FramePipeline
    from svt_av1_psy_b200.workload import FrameWorkload
    fp = FramePipeline(FrameWorkload(384, 256), torch)
    fp.step()
    s = torch.cuda.current_stream().cuda_stream
    fp.stage_cdef(s)  # cdef_out without the border extension of the restoration stage
    torch.cuda.synchronize()
    want = fp.cdef_out.clone()
    f = fp.cdef_frame(fp.recon)
    fp.cdef_out.copy_(fp.recon)
    (oy, sy), (ocb, sc), (ocr, _) = fp.plane_views(fp.cdef_out, True)
    rc = dsp.lib.svt_b200_cdef_apply_frame_dev(ct.byref(f), fp.skip.data_ptr(), fp.fb_idx.data_ptr(), fp.app_y.data_ptr(),
                                               fp.app_uv.data_ptr(), None, None, oy, ocb, ocr, sy, sc, s)
    assert rc == 0
    torch.cuda.synchronize()
    assert torch.equal(want, fp.cdef_out)
    assert dsp.lib.svt_b200_cdef_apply_frame_dev(ct.byref(f), fp.skip.data_ptr(), fp.fb_idx.data_ptr(), fp.app_y.data_ptr(),
                                                 fp.app_uv.data_ptr(), fp.cdef_dir.data_ptr(), None, oy, ocb, ocr, sy, sc, s) == -4  # SVT_B200_ERR_BAD_ARG


def test_two_frames_in_flight_on_two_streams(b200):
    """bench.py keeps two independent frames in flight on two streams (CUDA-graph replays); every library
    scratch buffer is per stream, so the concurrent results must equal the one-at-a-time results."""
    import torch
    from svt_av1_psy_b200.pipeline import FramePipeline
    from svt_av1_psy_b200.workload import FrameWorkload
    fps = [FramePipeline(FrameWorkload(384, 256, seed=1234 + 7 * k), torch) for k in range(2)]
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    names = ("qcoeff", "eobs", "recon", "cdef_mse", "cdef_out", "M", "Hm", "final")
    me_names = ("total_me_candidate_index", "me_candidate_array", "me_mv_array", "distortion", "best_sad")
    want = []
    for fp, st in zip(fps, streams):  # one at a time (also warms up every lazily allocated scratch)
        with torch.cuda.stream(st):
            fp.load_inputs()
            fp.step()
        torch.cuda.synchronize()
        want.append([getattr(fp, n).clone() for n in names] + [fp.me[n].clone() for n in me_names])
    graphs = []
    for fp, st in zip(fps, streams):
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=st):
            fp.step()
        graphs.append(g)
    for rep in range(6):
        for fp in fps:
            for n in ("qcoeff", "eobs", "cdef_mse", "M", "Hm", "final"):
                getattr(fp, n).zero_()
            fp.me["me_mv_array"].zero_()
            fp.me["best_sad"].zero_()
        torch.cuda.synchronize()
        for g, st in zip(graphs, streams):
            with torch.cuda.stream(st):
                g.replay() if rep % 2 == 0 else None
        if rep % 2:  # eager launches, interleaved call by call
            for fp, st in zip(fps, streams):
                with torch.cuda.stream(st):
                    fp.step()
        torch.cuda.synchronize()
        for fp, w in zip(fps, want):
            for n, t in zip(names + me_names, w):
                assert torch.equal(getattr(fp, n) if n in names else fp.me[n], t), (rep, n)


@pytest.mark.parametrize("name", ["frame_384x256", "frame_640x360", "frame_384x256_b10_m6", "frame_640x360_b10_m4"])
def test_frame_matches_committed_golden_fixture(b200, name):
    """tests/golden/frame_WxH.json holds the SHA-256 of every output of the frame as computed by the reference's
    own C kernels (tools/make_golden.py, run where oracle/_ref is built).  Needs no oracle at run time."""
    import hashlib
    import json
    import os
    import numpy as np
    import torch
    from svt_av1_psy_b200.pipeline import FramePipeline
    from svt_av1_psy_b200.workload import FrameWorkload
    g = json.load(open(os.path.join(os.path.dirname(__file__), "golden", name + ".json")))
    fp = FramePipeline(FrameWorkload(g["width"], g["height"], seed=g["seed"], bit_depth=g.get("bit_depth", 8), preset=g.get("preset", 8)), torch)
    fp.load_inputs()
    fp.step()
    torch.cuda.synchronize()

    def digest(t):
        return hashlib.sha256(np.ascontiguousarray(t.cpu().numpy()).view(np.uint8).tobytes()).hexdigest()
    got = {k: fp.me[f] for k, f in b200.ME_OUTPUT_NAMES.items()}
    got.update({"qcoeff": fp.qcoeff, "dqcoeff": fp.dqcoeff, "eob": fp.eobs,
           "recon": fp.recon, "cdef_mse": fp.cdef_mse, "cdef_dir": fp.cdef_dir, "cdef_out": fp.cdef_out, "wiener_M": fp.M,
           "wiener_H": fp.Hm, "final": fp.final})
    bad = [k for k, t in got.items() if digest(t) != g["sha256"][k]]
    assert not bad, bad
    # the forward coefficients only exist on the 3-call transform chain
    s = torch.cuda.current_stream().cuda_stream
    fp.call_residual(s)
    fp.call_fwd_txfm(s)
    torch.cuda.synchronize()
    assert digest(fp.residual) == g["sha256"]["residual"]
    assert digest(fp.coeff) == g["sha256"]["coeff"]


def test_shutdown_then_init_again_leaves_no_stale_state():
    """svt_b200_shutdown() releases every module's scratch, side streams and cached attributes; a second svt_b200_init() in the
    same process must work from a clean slate (ADVICE r1: stale per-stream workspaces / skipped cudaFuncSetAttribute)"""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = r"""
import sys
sys.path.insert(0, %r)
import torch
import svt_av1_psy_b200 as pkg
from svt_av1_psy_b200.pipeline import FramePipeline
from svt_av1_psy_b200.workload import FrameWorkload
outs = []
for rnd in range(3):
    pkg.init(0)
    fp = FramePipeline(FrameWorkload(384, 256, bit_depth=8 if rnd != 1 else 10, preset=8 if rnd != 1 else 6), torch)
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        fp.step()          # the library's per-stream scratch is created outside the capture
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=st):
        fp.step()
    g.replay()
    torch.cuda.synchronize()
    outs.append((int(fp.final.to(torch.int64).sum()), int(fp.me["distortion"].to(torch.int64).sum()), int(fp.Hm.sum())))
    del g, fp
    torch.cuda.synchronize()
    pkg.shutdown()
assert outs[0] == outs[2], outs
print("REINIT_OK", outs)
""" % root
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "REINIT_OK" in r.stdout, (r.stdout[-500:], r.stderr[-2000:])
