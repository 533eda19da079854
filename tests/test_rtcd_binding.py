"""The drop-in boundary exercised from INSIDE the reference (SURVEY.md 8b, 8(c)(ii)).

oracle/_ref/libsvtav1_enc.so = the unmodified reference library sources (Codec, C_DEFAULT, Globals) + this repository's
integration shim (integration/svt_b200_rtcd.c, hooked at enc_handle.c:1445 by a -D on the compiler command line) + a
minimal API application (oracle/enc_app.c), linked against libsvtav1_b200.so.

  * svt_b200_install_rtcd() assigns every T1 entry point over the reference's own dispatch pointers;
  * with the pointers installed, the reference's own process-level loops (svt_cdef_filter_fb cdef.c:339,
    svt_av1_loop_restoration_filter_unit restoration.c:1067, svt_aom_inv_transform_recon8bit, svt_aom_copy_sb8_16 ...,
    driven by oracle/ref_driver.c) reproduce the C-tier golden fixtures;
  * the whole encoder (svt_av1_enc_init ... svt_av1_enc_get_packet; open-loop ME through svt_aom_motion_estimation_b64,
    mode decision, enc-dec, CDEF, restoration all calling through the pointers) produces a bitstream IDENTICAL to the
    "--asm c" encode of the same input.
"""
import hashlib
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ENC_LIB = os.path.join(ROOT, "oracle", "_ref", "libsvtav1_enc.so")

_ENCODE = r'''
import ctypes as ct, hashlib, json, os, sys, time
import numpy as np
sys.path.insert(0, %(root)r)
from oracle.frame_ref import load_workload_module
W = load_workload_module()
lib = ct.CDLL(%(lib)r)
lib.ref_encode.restype = ct.c_int64
lib.ref_encode.argtypes = [ct.c_void_p] + [ct.c_int] * 8 + [ct.c_void_p, ct.c_int64, ct.c_void_p]
w, h, n, bd, preset, crf, lp = %(w)d, %(h)d, %(n)d, %(bd)d, %(preset)d, %(crf)d, %(lp)d
seq = W.synth_sequence(w, h, n, seed=20260923, bit_depth=bd)
yuv = np.concatenate([np.concatenate([p.reshape(-1) for p in f]) for f in seq])
out = np.zeros(16 << 20, np.uint8)
npk = ct.c_int32(0)
t0 = time.time()
r = lib.ref_encode(yuv.ctypes.data, w, h, n, bd, preset, crf, lp, -1, out.ctypes.data, out.size, ct.byref(npk))
launches = 0
if os.environ.get("SVT_B200_DEVICE"):
    b = ct.CDLL(%(b200)r)
    b.svt_b200_launch_count.restype = ct.c_ulonglong
    launches = int(b.svt_b200_launch_count())
    lib.svt_b200_rtcd_count.restype = ct.c_int
print("RESULT " + json.dumps({"bytes": int(r), "packets": npk.value, "sha256": hashlib.sha256(out[:max(r, 0)].tobytes()).hexdigest(),
                              "seconds": round(time.time() - t0, 2), "launches": launches}))
'''


def _encode(b200_on, **kw):
    env = dict(os.environ)
    env.pop("SVT_B200_DEVICE", None)
    if b200_on:
        env["SVT_B200_DEVICE"] = "0"
    code = _ENCODE % dict(kw, root=ROOT, lib=ENC_LIB, b200=os.path.join(ROOT, "svt-av1-psy_b200", "libsvtav1_b200.so"))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, timeout=1500)
    assert r.returncode == 0, (r.stdout[-1500:], r.stderr[-3000:])
    line = [x for x in r.stdout.splitlines() if x.startswith("RESULT ")][-1]
    return json.loads(line[7:])


def _need_lib():
    if not os.path.exists(ENC_LIB):  # it is built from the reference source tree, which is not part of this repository
        pytest.skip("oracle/_ref/libsvtav1_enc.so is not built (`make -C oracle enc` needs the reference source tree)")


def test_install_rtcd_binds_the_reference_pointers(b200):
    """every T1 entry point lands on the reference's own global function pointers"""
    import ctypes as ct
    _need_lib()
    enc = ct.CDLL(ENC_LIB)
    enc.ref_set_tier.restype = ct.c_int
    enc.ref_set_tier(0)  # svt_aom_setup_*_rtcd_internal(0): everything = *_c
    before = ct.c_void_p.in_dll(enc, "svt_sad_loop_kernel").value
    assert enc.svt_b200_install_rtcd(0) == 0
    n = enc.svt_b200_rtcd_count()
    assert n >= 160, n
    lib = ct.CDLL(os.path.join(ROOT, "svt-av1-psy_b200", "libsvtav1_b200.so"))
    for ref_name, our in (("svt_sad_loop_kernel", "svt_b200_sad_loop_kernel"), ("svt_av1_fwd_txfm2d_16x16", "svt_b200_av1_fwd_txfm2d_16x16"),
                          ("svt_av1_inv_txfm2d_add_64x32", "svt_b200_av1_inv_txfm2d_add_64x32"), ("svt_av1_quantize_fp_qm", "svt_b200_av1_quantize_fp_qm"),
                          ("svt_cdef_filter_block", "svt_b200_cdef_filter_block"), ("svt_av1_compute_stats", "svt_b200_av1_compute_stats"),
                          ("svt_aom_sad64x64x4d", "svt_b200_aom_sad64x64x4d"), ("svt_handle_transform64x64", "svt_b200_handle_transform64x64")):
        assert ct.c_void_p.in_dll(enc, ref_name).value == ct.cast(getattr(lib, our), ct.c_void_p).value, ref_name
    assert ct.c_void_p.in_dll(enc, "svt_sad_loop_kernel").value != before


@pytest.mark.parametrize("name", ["frame_384x256", "frame_384x256_b10_m6"])
def test_reference_process_loops_with_b200_pointers_match_c_goldens(b200, name):
    """oracle/ref_driver.c's frame step = the reference's own loops around the dispatched pointers (svt_cdef_filter_fb,
    svt_aom_inv_transform_recon*, svt_aom_copy_sb8_16, svt_av1_compute_stats*, wiener convolve ...).  Run with the B200
    T1 functions installed, every output must hash to the committed C-tier fixture."""
    import ctypes as ct
    from oracle.frame_ref import RefFrame, load_workload_module
    _need_lib()
    g = json.load(open(os.path.join(ROOT, "tests", "golden", name + ".json")))
    enc = ct.CDLL(ENC_LIB)
    enc.ref_set_tier.restype = ct.c_int
    enc.ref_set_tier(0)
    assert enc.svt_b200_install_rtcd(0) == 0
    enc.ref_set_threads.restype = ct.c_int
    enc.ref_set_threads(8)  # the T1 calls are made concurrently from the pool's threads, like the encoder's workers do
    wl = load_workload_module().FrameWorkload(g["width"], g["height"], seed=g["seed"], bit_depth=g.get("bit_depth", 8), preset=g.get("preset", 8))
    l0 = b200.launch_count()
    fr = RefFrame(wl, enc)
    fr.step()
    assert b200.launch_count() - l0 > 1000  # the work really went through libsvtav1_b200.so
    outs = {k: fr.me[f] for k, f in b200.ME_OUTPUT_NAMES.items()}
    outs.update({"residual": fr.residual, "coeff": fr.coeff, "qcoeff": fr.q, "dqcoeff": fr.dq,
            "eob": fr.eobs, "recon": fr.recon, "cdef_mse": fr.mse, "cdef_dir": fr.dirs, "cdef_out": fr.cdef_out, "wiener_M": fr.M, "wiener_H": fr.Hm,
            "final": fr.final})
    # the residual kernel is not a B200 T1 pointer (it stays the reference's C function here): included because everything downstream reads it
    bad = [k for k, v in outs.items() if hashlib.sha256(np.ascontiguousarray(v).view(np.uint8).tobytes()).hexdigest() != g["sha256"][k]]
    assert not bad, bad
    enc.ref_set_tier(0)


def test_lr_filter_unit_with_b200_pointers(b200, refc):
    """svt_av1_loop_restoration_filter_unit (restoration.c:1067) -- stripes, saved boundary lines, Wiener and self-guided --
    with the B200 convolve / self-guided functions installed == the same call on the C tier"""
    import ctypes as ct
    from test_oracle_pins import _lr_case  # the fixture generator of the a13 oracle pins
    _need_lib()
    enc = ct.CDLL(ENC_LIB)
    enc.ref_set_tier.restype = ct.c_int
    for kind in ("wiener", "sgrproj"):
        res = []
        for lib_, install in ((refc, False), (enc, True)):
            lib_.ref_set_tier(0)
            if install:
                assert enc.svt_b200_install_rtcd(0) == 0
            res.append(_lr_case(lib_, kind))
        enc.ref_set_tier(0)
        assert len(res[0]) == len(res[1]) and all(np.array_equal(a, b) for a, b in zip(res[0], res[1])), kind


@pytest.mark.timeout(3000)
# the reference's own C path is not run-to-run deterministic at 10 bit with several worker threads (three `--asm c` encodes of
# the same input gave three bitstreams here); with one thread it is, so the 10-bit case pins lp = 1
@pytest.mark.parametrize("cfg", [dict(w=640, h=360, n=6, bd=8, preset=12, crf=35, lp=8), dict(w=640, h=360, n=4, bd=8, preset=8, crf=30, lp=8),
                                 dict(w=640, h=360, n=4, bd=10, preset=8, crf=30, lp=1)],
                         ids=["configs0_360p_8bit_M12", "360p_8bit_M8", "360p_10bit_M8_lp1"])
def test_encoder_bitstream_identical_to_c_path(cfg):
    """SURVEY.md 8(c)(ii): the encoder with the B200 tier installed writes the same bitstream as `--asm c`"""
    _need_lib()
    c = _encode(False, **cfg)
    g = _encode(True, **cfg)
    assert c["bytes"] > 0 and c["packets"] == cfg["n"], c
    assert g["launches"] > 10000, g  # the encode really ran on libsvtav1_b200.so
    assert (g["bytes"], g["packets"], g["sha256"]) == (c["bytes"], c["packets"], c["sha256"]), (c, g)
    print("encode %s: C %.1fs, B200 T1 pointers %.1fs, %d kernel launches" % (cfg, c["seconds"], g["seconds"], g["launches"]))
