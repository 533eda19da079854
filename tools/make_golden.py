#!/usr/bin/env python3
"""Generate tests/golden/frame_<W>x<H>.json: SHA-256 of every output of one synthetic frame computed by the
REFERENCE's own kernels (oracle/_ref, C tier, driven by oracle/ref_driver.c).  Run where `python __graft_entry__.py --oracle`
has built oracle/_ref (it needs the reference source tree); the fixtures are committed so that the GPU parity tests and
smoke() also work where oracle/_ref is absent.  One fixture per picture size of test_frame_pipeline.FRAME_CASES."""
import hashlib
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402

import oracle  # noqa: E402
from oracle.frame_ref import RefFrame, load_workload_module  # noqa: E402


def digest(a):
    return hashlib.sha256(np.ascontiguousarray(a).view(np.uint8).tobytes()).hexdigest()


def golden_for(width, height, seed=20260923, bit_depth=8, preset=8):
    ref = oracle.ref
    assert ref is not None, "oracle/_ref is not built"
    ref.ref_set_tier(0)
    wl = load_workload_module().FrameWorkload(width, height, seed=seed, bit_depth=bit_depth, preset=preset)
    fr = RefFrame(wl, ref)
    fr.step()
    outs = {k: fr.me[f] for k, f in load_workload_module().dsp.ME_OUTPUT_NAMES.items()}
    outs.update({"residual": fr.residual, "coeff": fr.coeff, "qcoeff": fr.q, "dqcoeff": fr.dq,
            "eob": fr.eobs, "recon": fr.recon, "cdef_mse": fr.mse, "cdef_dir": fr.dirs, "cdef_out": fr.cdef_out,
            "wiener_M": fr.M, "wiener_H": fr.Hm, "final": fr.final})
    return {"width": width, "height": height, "seed": seed, "bit_depth": bit_depth, "preset": preset, "reference_tier": "C (ref_set_tier(0))",
            "sha256": {k: digest(v) for k, v in outs.items()},
            "shape": {k: list(np.asarray(v).shape) for k, v in outs.items()}}


if __name__ == "__main__":
    for (w, h, bd, m) in ((384, 256, 8, 8), (640, 360, 8, 8), (384, 256, 10, 6), (640, 360, 10, 4), (448, 320, 10, 4), (1920, 1080, 8, 8),
                          (1920, 1080, 10, 6), (3840, 2160, 8, 8), (3840, 2160, 10, 4)):
        g = golden_for(w, h, bit_depth=bd, preset=m)
        path = os.path.join(ROOT, "tests", "golden", "frame_%dx%d%s.json" % (w, h, "" if (bd, m) == (8, 8) else "_b%d_m%d" % (bd, m)))
        json.dump(g, open(path, "w"), indent=1, sort_keys=True)
        print("wrote", path)
