"""Host-side mirror of the reference's process kernels for the hot path: a FramePipeline owns the
device-resident planes / work lists of one frame set and enqueues the T2 entry points of
libsvtav1_b200.so in the order the reference's ME -> EncDec(final pass) -> CDEF -> REST processes hand
work to the dispatched DSP functions (SURVEY.md 3.2-3.5).  torch is used for device memory, streams
and events only; every computation is a C-ABI call.
"""
import ctypes as ct

import numpy as np

from . import dsp
from .dsp import lib


def _t(torch, arr, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(arr))
    return t.cuda(non_blocking=False)


class _Arena:
    """one contiguous device buffer + its pinned host twin, carved into typed views at 256-byte aligned offsets: a frame's
    inputs (or fixed-size results) then cross PCIe in ONE copy instead of one per array"""

    def __init__(self, torch, specs, device):
        self.torch = torch
        off, self.slots = 0, {}
        for name, dtype, shape in specs:
            n = int(np.prod(shape)) * torch.empty(0, dtype=dtype).element_size()
            self.slots[name] = (off, n, dtype, tuple(shape))
            off = (off + n + 255) & ~255
        self.nbytes = off
        self.dev = torch.zeros(off, dtype=torch.uint8, device=device)
        self.host = torch.zeros(off, dtype=torch.uint8).pin_memory()

    def view(self, name, host=False):
        off, n, dtype, shape = self.slots[name]
        return (self.host if host else self.dev)[off:off + n].view(dtype).view(shape)


class FramePipeline:
    def __init__(self, wl, torch, device="cuda"):
        self.wl, self.torch = wl, torch
        self._side = self._forked = self._joined = None
        self._extents = None
        self.tx_counts = (ct.c_int * dsp.TXFM_CLASSES)(*wl.tx_class_counts)
        W, H = wl.width, wl.height
        T = torch
        self.bd, self.psz = wl.bit_depth, wl.pixel_bytes
        pix = T.uint8 if self.psz == 1 else T.int16  # torch has no uint16 arithmetic; the planes are only storage here
        # ---- ME: padded pyramids (current + references) -------------------------------------------
        self.cur_planes = [T.zeros((s[0], s[1]), dtype=T.uint8, device=device) for s in wl.me_shapes]
        self.ref_planes = [[T.zeros((s[0], s[1]), dtype=T.uint8, device=device) for s in wl.me_shapes] for _ in range(wl.n_refs)]
        pad = wl.me_shapes[2][2]
        self._full_pad = pad
        for r, ref in enumerate(wl.refs):
            self._upload_full(self.ref_planes[r], wl.me_luma(ref))
            d = dsp.me_picture_desc(self.ref_planes[r], W, H)
            assert lib.svt_b200_build_hme_pyramid_dev(ct.byref(d), None) == 0
        self.cur_desc = dsp.me_picture_desc(self.cur_planes, W, H)
        self.ref_descs = (dsp.MePicture * wl.n_refs)(*[dsp.me_picture_desc(p, W, H) for p in self.ref_planes])
        self.me_ctrl = dsp.MeControls.from_dict(wl.me_controls)   # the MeContext controls of the workload's ME picture
        assert lib.svt_b200_me_b64_num_pus(ct.byref(self.me_ctrl)) == wl.me_n_pu
        nb = ((W + 63) // 64) * ((H + 63) // 64)
        self.n_b64 = nb
        _, n_flat = wl.flat_offsets()
        _, n_pad = wl.padded_offsets()
        self.n_tx = len(wl.quant_items)
        # everything the host-side stages read back, in one arena (one device -> host copy per frame).  The restored picture is NOT
        # among it: it stays on the device as a reference picture (the host needs it only for recon output / PSNR)
        mc, mr, n_pu = wl.me_controls["max_cand"], wl.me_controls["max_refs"], wl.me_n_pu
        self._out = _Arena(T, [("me_mv_array", T.int32, (nb, n_pu * mr)), ("me_distortion", T.int32, (nb, 6)),
                               ("me_candidate_array", T.uint8, (nb, n_pu * mc)), ("me_total", T.uint8, (nb, n_pu)), ("me_flags", T.uint8, (nb, 2)),
                               ("eobs", T.int16, (self.n_tx,)),
                               ("level_offsets", T.int32, (self.n_tx + 2,)), ("mse", T.int64, (2, nb, len(wl.cdef_str_y))),
                               ("M", T.int64, (len(wl.stats_items), 49)), ("H", T.int64, (len(wl.stats_items), 2401))], device)
        # ... and what arrives from the host per frame (source picture + prediction): one host -> device copy
        self._in = _Arena(T, [("cur", pix, (n_flat,)), ("pred", pix, (n_pad,))], device)
        # ME results the host-side mode decision consumes (MeSbResults + the per-block distortions) ...
        self.me = {"total_me_candidate_index": self._out.view("me_total"), "me_candidate_array": self._out.view("me_candidate_array"),
                   "me_mv_array": self._out.view("me_mv_array"), "distortion": self._out.view("me_distortion"), "flags": self._out.view("me_flags"),
                   # ... and the per-reference search state, which stays on the device
                   "do_ref": T.zeros((nb, 2, 4), dtype=T.uint8, device=device), "hme_centre": T.zeros((nb, 2, 4, 2), dtype=T.int16, device=device),
                   "zz_sad": T.zeros((nb, 2, 4), dtype=T.int32, device=device),
                   "best_sad": T.zeros((wl.n_refs, nb, 85), dtype=T.int32, device=device), "best_mv": T.zeros((wl.n_refs, nb, 85), dtype=T.int32, device=device)}
        self.me_out = dsp.MeB64Results()
        for k, v in self.me.items():
            setattr(self.me_out, k, v.data_ptr())
        # ---- TX ---------------------------------------------------------------------------------------
        self.cur_flat = self._in.view("cur")                               # source picture Y|U|V
        self.residual = T.zeros(n_flat, dtype=T.int16, device=device)
        self.pred = self._in.view("pred")                                  # padded planes
        self.recon = T.zeros(n_pad, dtype=pix, device=device)
        self.cdef_out = T.zeros(n_pad, dtype=pix, device=device)
        self.final = T.zeros(n_pad, dtype=pix, device=device)
        self.coeff = T.zeros(wl.n_coeffs, dtype=T.int32, device=device)
        self.qcoeff = T.zeros_like(self.coeff)
        self.dqcoeff = T.zeros_like(self.coeff)
        self.eobs = self._out.view("eobs")
        self.fwd_items = _t(T, wl.fwd_items.view(np.uint8))
        self.inv_items = _t(T, wl.inv_items.view(np.uint8))
        self.quant_items = _t(T, wl.quant_items.view(np.uint8))
        self.trio_items = _t(T, wl.trio_items.view(np.uint8))
        self.scan = _t(T, wl.scan_table)
        self.iscan = _t(T, wl.iscan_table)
        self.qm = _t(T, wl.qm_table)
        # ---- CDEF -------------------------------------------------------------------------------------
        self.skip = _t(T, wl.skip8x8)
        self.str_y, self.str_uv = _t(T, wl.cdef_str_y), _t(T, wl.cdef_str_uv)
        self.cdef_mse = self._out.view("mse")
        self.cdef_dir = T.zeros((nb, 64), dtype=T.uint8, device=device)
        self.cdef_var = T.zeros((nb, 64), dtype=T.int32, device=device)
        self.fb_idx = _t(T, wl.cdef_fb_idx)
        self.app_y, self.app_uv = _t(T, wl.cdef_apply_y), _t(T, wl.cdef_apply_uv)
        # ---- REST -------------------------------------------------------------------------------------
        self.stats_items = _t(T, wl.stats_items.view(np.uint8))
        self.lr_units = [_t(T, u.view(np.uint8)) for u in wl.lr_units]
        self.lr_above = [T.zeros(2 * wl.lr_num_stripes(p) * wl.lr_boundary_stride(p), dtype=pix, device=device) for p in range(3)]
        self.lr_below = [T.zeros(2 * wl.lr_num_stripes(p) * wl.lr_boundary_stride(p), dtype=pix, device=device) for p in range(3)]
        self._lr_planes = None
        self.M = self._out.view("M")
        self.Hm = self._out.view("H")
        # ---- host staging for the end-to-end arm ------------------------------------------------------
        as_t = (lambda a: T.from_numpy(a)) if self.psz == 1 else (lambda a: T.from_numpy(a.view(np.int16)))
        self.h_cur = self._in.view("cur", host=True)
        self.h_pred = self._in.view("pred", host=True)
        self.h_cur.copy_(as_t(np.concatenate([p.reshape(-1) for p in wl.cur])))
        self.h_pred.copy_(as_t(self._pad_planes(wl.pred)))
        # 10-bit input: the 8-bit luma open-loop ME searches is made by the picture-input stage on the host
        self.h_luma8 = None if self.psz == 1 else T.from_numpy(np.ascontiguousarray(wl.me_luma(wl.cur))).pin_memory()
        # what the host-side stages consume: ME results, per-block eobs + the eob-bounded scan-order levels (entropy coder),
        # CDEF costs, Wiener statistics (the host solves the filters), the filtered picture
        self.level_bytes = 2 if self.bd == 8 else 4
        self.levels = T.zeros(wl.n_coeffs, dtype=T.int16 if self.level_bytes == 2 else T.int32, device=device)
        self.level_offsets = self._out.view("level_offsets")
        self.h_out = {k: self._out.view(k, host=True) for k in self._out.slots}
        self.h_levels = T.empty_like(self.levels, device="cpu").pin_memory()
        self._h_offs = self.h_out["level_offsets"].numpy()  # numpy view of the pinned buffer: cheap scalar reads on the host
        self._res_planes = None
        self.load_inputs()
        T.cuda.synchronize()

    # -- helpers ------------------------------------------------------------------------------------------
    def _pad_planes(self, planes):
        wl = self.wl
        off, n = wl.padded_offsets()
        buf = np.zeros(n, wl.pixel_dtype)
        for p in range(3):
            th, st = wl.padded_shape(p)
            w, h = wl.plane_dims[p]
            v = buf[off[p]:off[p] + th * st].reshape(th, st)
            v[:, :w + 2 * wl.PAD] = np.pad(planes[p], wl.PAD, mode="edge")
        return buf

    def _upload_full(self, planes, luma):
        pad, (H, W) = self._full_pad, luma.shape
        st = planes[2].shape[1]
        buf = np.zeros(planes[2].shape, np.uint8)
        buf[:, :W + 2 * pad] = np.pad(luma, pad, mode="edge")
        buf[:, W + 2 * pad:] = 0
        planes[2].copy_(self.torch.from_numpy(buf))

    def plane_views(self, flat, padded=True):
        """[(tensor_2d_interior_origin_ptr, stride)] for the three planes of a padded flat buffer"""
        wl = self.wl
        out = []
        off, _ = wl.padded_offsets() if padded else wl.flat_offsets()
        for p in range(3):
            if padded:
                th, st = wl.padded_shape(p)
                out.append((flat.data_ptr() + (off[p] + wl.PAD * st + wl.PAD) * self.psz, st))
            else:
                out.append((flat.data_ptr() + off[p] * self.psz, wl.plane_dims[p][0]))
        return out

    def load_inputs(self, stream=None):
        """host -> device copy of one frame's inputs (source picture + prediction: one transfer; a 10-bit picture also brings the
        8-bit luma the picture-input stage made for open-loop ME) on `stream` (a raw CUDA stream handle; default: torch's current)"""
        s = self.torch.cuda.current_stream().cuda_stream if stream is None else stream
        lib.svt_b200_copy_async(self._in.dev.data_ptr(), self._in.host.data_ptr(), self._in.nbytes, 0, s)
        if self.psz != 1:
            W, H, pad = self.wl.width, self.wl.height, self._full_pad
            p2 = self.cur_planes[2]
            lib.svt_b200_copy2d_async(p2.data_ptr() + pad * p2.stride(0) + pad, p2.stride(0), self.h_luma8.data_ptr(), W, W, H, 0, s)

    def read_outputs(self, stream=None):
        """device -> host, part 1: everything of fixed size in one transfer (includes the level offsets, whose last entries say how
        many levels follow)"""
        s = self.torch.cuda.current_stream().cuda_stream if stream is None else stream
        lib.svt_b200_copy_async(self._out.host.data_ptr(), self._out.dev.data_ptr(), self._out.nbytes, 1, s)

    def read_levels(self, stream=None):
        """part 2, once part 1 has arrived: exactly sum(eob) levels.  Returns the bytes copied."""
        s = self.torch.cuda.current_stream().cuda_stream if stream is None else stream
        total = int(self._h_offs[self.n_tx])
        assert int(self._h_offs[self.n_tx + 1]) == 0, "a quantised level did not fit the packed format"
        total = min(total, self.levels.numel())
        lib.svt_b200_copy_async(self.h_levels.data_ptr(), self.levels.data_ptr(), total * self.level_bytes, 1, s)
        return total * self.level_bytes

    @property
    def h2d_bytes(self):
        return (self.h_cur.numel() + self.h_pred.numel()) * self.psz + (0 if self.h_luma8 is None else self.h_luma8.numel())

    @property
    def d2h_fixed_bytes(self):
        return sum(n for (_, n, _, _) in self._out.slots.values())

    # -- the calls of one frame, in path order (each is one T2 entry point of include/svt_b200.h) -----------
    def call_me_pyramid(self, s):
        """the padded full-resolution luma of the ME pyramid (8-bit pictures: the source luma itself) + the two decimated levels"""
        W, H, pad = self.wl.width, self.wl.height, self._full_pad
        p2 = self.cur_planes[2]
        if self.psz == 1:
            lib.svt_b200_copy2d_async(p2.data_ptr() + pad * p2.stride(0) + pad, p2.stride(0), self.cur_flat.data_ptr(), W, W, H, 2, s)
        assert lib.svt_b200_extend_plane_dev(p2.data_ptr(), p2.stride(0), W, H, pad, pad, s) == 0
        assert lib.svt_b200_build_hme_pyramid_dev(ct.byref(self.cur_desc), s) == 0

    def call_me_search(self, s):
        """svt_aom_motion_estimation_b64 for every 64x64 block: pre-HME, HME, pruning, full-pel search, candidates, distortions"""
        rc = lib.svt_b200_me_b64_picture_dev(ct.byref(self.cur_desc), self.ref_descs, ct.byref(self.me_ctrl), ct.byref(self.me_out), s)
        assert rc == 0

    def call_txfm_trio(self, s):
        """residual (source - prediction) -> transform -> quantise -> inverse / reconstruction, one fused call"""
        rc = lib.svt_b200_residual_txfm_trio_batch_dev(self.cur_flat.data_ptr(), self.pred.data_ptr(), self.recon.data_ptr(), self.qcoeff.data_ptr(),
                                                       self.dqcoeff.data_ptr(), self.iscan.data_ptr(), self.qm.data_ptr(), self.trio_items.data_ptr(),
                                                       self.tx_counts, self.eobs.data_ptr(), self.psz, s)
        assert rc == 0

    def call_pack_levels(self, s):
        rc = lib.svt_b200_pack_levels_dev(self.qcoeff.data_ptr(), self.iscan.data_ptr(), self.trio_items.data_ptr(), self.eobs.data_ptr(), self.n_tx,
                                          self.level_offsets.data_ptr(), self.levels.data_ptr(), self.level_bytes, self.levels.numel(), s)
        assert rc == 0

    def call_residual(self, s):
        """svt_aom_residual_kernel over the three planes (the un-fused chain materialises the residual)"""
        wl = self.wl
        if self._res_planes is None:
            off, _ = wl.padded_offsets()
            soff, _ = wl.flat_offsets()
            self._res_planes = dsp.ResidualPlanes()
            for p in range(3):
                th, st = wl.padded_shape(p)
                w, h = wl.plane_dims[p]
                self._res_planes.p[p] = dsp.ResidualPlane(soff[p], off[p] + wl.PAD * st + wl.PAD, soff[p], w, st, w, w, h, 0)
        rc = lib.svt_b200_residual_planes_dev(self.cur_flat.data_ptr(), self.pred.data_ptr(), self.residual.data_ptr(), ct.byref(self._res_planes), 3,
                                              self.psz, s)
        assert rc == 0

    # the same three steps as separate calls (TPL / MD use them individually); results are identical
    def call_fwd_txfm(self, s):
        rc = lib.svt_b200_fwd_txfm_batch_dev(self.residual.data_ptr(), self.coeff.data_ptr(), self.fwd_items.data_ptr(), self.tx_counts, s)
        assert rc == 0

    def call_quant(self, s):
        rc = lib.svt_b200_quant_batch_dev(self.coeff.data_ptr(), self.qcoeff.data_ptr(), self.dqcoeff.data_ptr(), self.scan.data_ptr(), self.iscan.data_ptr(),
                                          self.qm.data_ptr(), self.quant_items.data_ptr(), len(self.wl.quant_items), self.eobs.data_ptr(), s)
        assert rc == 0

    def call_inv_txfm(self, s):
        rc = lib.svt_b200_inv_txfm_batch_dev(self.dqcoeff.data_ptr(), self.pred.data_ptr(), self.recon.data_ptr(), self.inv_items.data_ptr(),
                                             self.tx_counts, self.psz, s)
        assert rc == 0

    def cdef_frame(self, recon_flat):
        wl = self.wl
        f = dsp.CdefFrame()
        (f.recon_y, sy), (f.recon_cb, sc), (f.recon_cr, _) = self.plane_views(recon_flat, True)
        (f.src_y, ssy), (f.src_cb, ssc), (f.src_cr, _) = self.plane_views(self.cur_flat, False)
        f.recon_stride_y, f.recon_stride_c, f.src_stride_y, f.src_stride_c = sy, sc, ssy, ssc
        f.width, f.height, f.bit_depth, f.damping, f.subsampling_factor = wl.width, wl.height, self.bd, wl.cdef_damping, wl.cdef_subsampling
        return f

    def call_cdef_search(self, s):
        f = self.cdef_frame(self.recon)
        rc = lib.svt_b200_cdef_search_frame_dev(ct.byref(f), self.skip.data_ptr(), self.str_y.data_ptr(), self.str_uv.data_ptr(),
                                                len(self.wl.cdef_str_y), self.cdef_mse.data_ptr(), self.cdef_dir.data_ptr(),
                                                self.cdef_var.data_ptr(), s)
        assert rc == 0

    def call_cdef_apply(self, s):
        f = self.cdef_frame(self.recon)
        self.cdef_out.copy_(self.recon, non_blocking=True)  # svt_av1_cdef_frame filters in place
        (oy, sy), (ocb, sc), (ocr, _) = self.plane_views(self.cdef_out, True)
        rc = lib.svt_b200_cdef_apply_frame_dev(ct.byref(f), self.skip.data_ptr(), self.fb_idx.data_ptr(), self.app_y.data_ptr(),
                                               self.app_uv.data_ptr(), self.cdef_dir.data_ptr(), self.cdef_var.data_ptr(), oy, ocb, ocr, sy, sc, s)
        assert rc == 0

    def call_rest_extend(self, s):
        wl = self.wl
        if self._extents is None:  # svt_extend_frame: restoration reads beyond the picture edge
            off, _ = wl.padded_offsets()
            self._extents = (dsp.PlaneExtent * 3)()
            for p in range(3):
                th, st = wl.padded_shape(p)
                w, h = wl.plane_dims[p]
                self._extents[p] = dsp.PlaneExtent(self.cdef_out.data_ptr() + off[p] * self.psz, st, w, h, wl.PAD, wl.PAD, self.psz)
        assert lib.svt_b200_extend_planes_dev(self._extents, 3, s) == 0

    def call_wiener_stats(self, s):
        rc = lib.svt_b200_compute_stats_batch_dev(self.cdef_out.data_ptr(), self.cur_flat.data_ptr(), self.stats_items.data_ptr(),
                                                  len(self.wl.stats_items), self.bd, self.M.data_ptr(), self.Hm.data_ptr(), s)
        assert rc == 0

    def lr_planes(self):
        """SvtB200LrPlane x 3: deblocked = the reconstruction before CDEF, cdef = the CDEF output, dst = the restored picture"""
        if self._lr_planes is None:
            wl = self.wl
            self._lr_planes = (dsp.LrPlane * 3)()
            rec, cdf, fin = self.plane_views(self.recon, True), self.plane_views(self.cdef_out, True), self.plane_views(self.final, True)
            src = self.plane_views(self.cur_flat, False)
            for p in range(3):
                w, h = wl.plane_dims[p]
                ss = 1 if p else 0
                self._lr_planes[p] = dsp.LrPlane(rec[p][0], cdf[p][0], fin[p][0], src[p][0], self.lr_above[p].data_ptr(), self.lr_below[p].data_ptr(),
                                                 rec[p][1], cdf[p][1], fin[p][1], src[p][1], wl.lr_boundary_stride(p), w, h, ss, ss, wl.lr_unit_size[p],
                                                 1)  # frame_restoration_type = RESTORE_WIENER for every plane of this workload
            self._lr_unit_ptrs = (ct.c_void_p * 3)(*[u.data_ptr() for u in self.lr_units])
        return self._lr_planes

    def call_lr_boundaries(self, s):
        """svt_av1_loop_restoration_save_boundary_lines, both passes (deblocked lines from the reconstruction, CDEF lines from cdef_out)"""
        pl = self.lr_planes()
        assert lib.svt_b200_lr_save_boundary_lines_dev(pl, 3, 0, self.bd, s) == 0
        assert lib.svt_b200_lr_save_boundary_lines_dev(pl, 3, 1, self.bd, s) == 0

    def call_wiener_filter(self, s):
        """svt_av1_loop_restoration_filter_frame: every unit of the three planes, stripe by stripe with the saved boundary lines"""
        pl = self.lr_planes()
        assert lib.svt_b200_lr_filter_frame_dev(pl, 3, self._lr_unit_ptrs, 0, self.bd, s) == 0

    STAGES = ("me", "tx", "cdef", "rest")
    # (call, stage it belongs to, the kernels it launches)
    CALLS = (("me_pyramid", "me", "downsample_2d_kernel+pad_plane_kernel"),
             ("me_search", "me", "me_b64_hme_kernel + fullpel_search_kernel + me_b64_finish_kernel"),
             ("txfm_trio", "tx", "trio_txfm_kernel<4..64> (residual + forward transform + quantise + inverse transform fused)"),
             ("pack_levels", "tx", "eob_chunk_sum_kernel+eob_offsets_kernel+pack_levels_kernel"),
             ("cdef_search", "cdef", "cdef_dir_kernel+cdef_search_kernel"),
             ("cdef_apply", "cdef", "cdef_apply_kernel"),
             ("lr_boundaries", "rest", "lr_save_boundary_kernel x2"),
             ("rest_extend", "rest", "pad_plane_kernel"),
             ("wiener_stats", "rest", "stats_mma_kernel+stats_finalize_kernel (8-bit; 10-bit: stats_sum_kernel+stats_lag_*)"),
             ("wiener_filter", "rest", "lr_filter_kernel (striped restoration of the whole picture)"))

    def _stage(self, stage, s):
        for name, st, _ in self.CALLS:
            if st == stage:
                getattr(self, "call_" + name)(s)

    def stage_me(self, s):
        self._stage("me", s)

    def stage_tx(self, s):
        self._stage("tx", s)

    def stage_cdef(self, s):
        self._stage("cdef", s)

    def stage_rest(self, s):
        self._stage("rest", s)

    def step(self, events=None):
        """Enqueue one frame of hot-path work on torch's current stream.

        Motion estimation reads only source pictures; transform -> CDEF -> restoration reads only the
        residual/prediction of the block pass: the two chains share no data (in the encoder they are
        different pipeline stages working on different pictures at the same moment), so the step runs ME
        on a side stream, concurrently with the reconstruction chain, and joins at the end.
        With `events` (len(CALLS)+1 CUDA events, recorded before every call and after the last) the calls
        run strictly one after the other instead, so that each call can be timed on its own."""
        T = self.torch
        cur = T.cuda.current_stream()
        if events is not None:
            s = cur.cuda_stream
            for i, (name, _, _) in enumerate(self.CALLS):
                events[i].record()
                getattr(self, "call_" + name)(s)
            events[len(self.CALLS)].record()
            return
        if self._side is None:
            self._side, self._forked, self._joined = T.cuda.Stream(), T.cuda.Event(), T.cuda.Event()
        self._forked.record(cur)
        self._side.wait_event(self._forked)
        with T.cuda.stream(self._side):
            self._stage("me", self._side.cuda_stream)
            self._joined.record(self._side)
        for st in ("tx", "cdef", "rest"):
            self._stage(st, cur.cuda_stream)
        cur.wait_event(self._joined)
