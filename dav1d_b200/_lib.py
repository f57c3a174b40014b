"""ctypes binding of the C ABI in include/b200av1.h.

The product library is dav1d_b200/libb200av1.so (CUDA, sm_100a). There is no CPU
fallback: if it is missing it is built with nvcc, and if it cannot be built or loaded the
import fails loudly. (tests/emu builds a *test-only* host-emulated copy of the same ABI and
binds it through B200Lib(path) explicitly; the package itself never does.)
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libb200av1.so")


class ItxBlock(C.Structure):
    """struct B200ItxBlock (include/b200av1.h)"""
    _fields_ = [("dst_off", C.c_uint32), ("coef_off", C.c_uint32), ("eob", C.c_int16),
                ("txtp", C.c_uint8), ("plane", C.c_uint8)]


class RefGeom(C.Structure):
    """struct B200RefGeom: planes of a reference picture whose size differs from the frame's (scaled references)"""
    _fields_ = [("plane_off", C.c_uint32 * 3), ("stride", C.c_int32 * 3), ("w", C.c_int32 * 3), ("h", C.c_int32 * 3)]


class McFrame(C.Structure):
    """struct B200McFrame"""
    _fields_ = [("ref", C.c_void_p * 8), ("ref_plane_off", C.c_uint32 * 3), ("ref_stride", C.c_int32 * 3),
                ("ref_w", C.c_int32 * 3), ("ref_h", C.c_int32 * 3), ("dst", C.c_void_p),
                ("dst_stride", C.c_int32 * 3), ("tmp", C.c_void_p), ("mask", C.c_void_p), ("px_tmp", C.c_void_p),
                ("scaled_mask", C.c_uint32), ("pad_geom", C.c_uint32), ("ref_geom", RefGeom * 8)]


class McBlock(C.Structure):
    _fields_ = [("dst_off", C.c_uint32), ("src_x", C.c_int32), ("src_y", C.c_int32), ("w", C.c_uint8),
                ("h", C.c_uint8), ("mx", C.c_uint8), ("my", C.c_uint8), ("filter2d", C.c_uint8),
                ("op", C.c_uint8), ("plane", C.c_uint8), ("ref", C.c_uint8)]


class CompBlock(C.Structure):
    _fields_ = [("dst_off", C.c_uint32), ("tmp1_off", C.c_uint32), ("tmp2_off", C.c_uint32),
                ("mask_off", C.c_uint32), ("w", C.c_uint8), ("h", C.c_uint8), ("op", C.c_uint8),
                ("param", C.c_uint8), ("plane", C.c_uint8), ("pad", C.c_uint8 * 3)]


class BlendBlock(C.Structure):
    _fields_ = [("dst_off", C.c_uint32), ("tmp_off", C.c_uint32), ("mask_off", C.c_uint32),
                ("w", C.c_uint8), ("h", C.c_uint8), ("op", C.c_uint8), ("plane", C.c_uint8)]


class WarpBlock(C.Structure):
    _fields_ = [("dst_off", C.c_uint32), ("src_x", C.c_int32), ("src_y", C.c_int32), ("mx", C.c_int32),
                ("my", C.c_int32), ("abcd", C.c_int16 * 4), ("tmp_stride", C.c_uint16), ("op", C.c_uint8),
                ("plane", C.c_uint8), ("ref", C.c_uint8), ("pad", C.c_uint8)]


class FilterLUT(C.Structure):
    """Av1FilterLUT / B200FilterLUT"""
    _fields_ = [("e", C.c_uint8 * 64), ("i", C.c_uint8 * 64), ("sharp", C.c_uint64 * 2)]


class Av1Filter(C.Structure):
    """Av1Filter / B200Av1Filter (1348 bytes)"""
    _fields_ = [("filter_y", C.c_uint16 * 2 * 3 * 32 * 2), ("filter_uv", C.c_uint16 * 2 * 2 * 32 * 2),
                ("cdef_idx", C.c_int8 * 4), ("noskip_mask", C.c_uint16 * 2 * 16)]


class LfFrame(C.Structure):
    _fields_ = [("pic", C.c_void_p), ("plane_off", C.c_uint32 * 3), ("stride", C.c_int32 * 3),
                ("w4", C.c_int32), ("h4", C.c_int32), ("sb128w", C.c_int32), ("b4_stride", C.c_int32),
                ("ss_hor", C.c_int32), ("ss_ver", C.c_int32), ("sb128", C.c_int32), ("filter_y", C.c_int32),
                ("filter_uv", C.c_int32), ("mask", C.c_void_p), ("level", C.c_void_p), ("lut", FilterLUT)]


class CdefFrame(C.Structure):
    _fields_ = [("src", C.c_void_p), ("dst", C.c_void_p), ("plane_off", C.c_uint32 * 3), ("stride", C.c_int32 * 3),
                ("bw", C.c_int32), ("bh", C.c_int32), ("sb128w", C.c_int32), ("ss_hor", C.c_int32),
                ("ss_ver", C.c_int32), ("damping", C.c_int32), ("y_strength", C.c_int32 * 8),
                ("uv_strength", C.c_int32 * 8), ("mask", C.c_void_p)]


class LrFrame(C.Structure):
    _fields_ = [("cdef", C.c_void_p), ("dbl", C.c_void_p), ("dst", C.c_void_p), ("plane_off", C.c_uint32 * 3),
                ("stride", C.c_int32 * 3), ("w", C.c_int32), ("h", C.c_int32), ("ss_hor", C.c_int32),
                ("ss_ver", C.c_int32), ("sb128", C.c_int32), ("sr_sb128w", C.c_int32),
                ("unit_size_log2", C.c_int32 * 2), ("restore_planes", C.c_int32), ("lr_mask", C.c_void_p)]


class FilmGrainData(C.Structure):
    """Dav1dFilmGrainData / B200FilmGrainData (224 bytes)"""
    _fields_ = [("seed", C.c_uint), ("num_y_points", C.c_int), ("y_points", (C.c_uint8 * 2) * 14),
                ("chroma_scaling_from_luma", C.c_int), ("num_uv_points", C.c_int * 2),
                ("uv_points", ((C.c_uint8 * 2) * 10) * 2), ("scaling_shift", C.c_int), ("ar_coeff_lag", C.c_int),
                ("ar_coeffs_y", C.c_int8 * 24), ("ar_coeffs_uv", (C.c_int8 * 28) * 2), ("ar_coeff_shift", C.c_uint64),
                ("grain_scale_shift", C.c_int), ("uv_mult", C.c_int * 2), ("uv_luma_mult", C.c_int * 2),
                ("uv_offset", C.c_int * 2), ("overlap_flag", C.c_int), ("clip_to_restricted_range", C.c_int)]


class FgFrame(C.Structure):
    _fields_ = [("in_", C.c_void_p), ("out", C.c_void_p), ("plane_off", C.c_uint32 * 3), ("stride", C.c_int32 * 3),
                ("w", C.c_int32), ("h", C.c_int32), ("ss_hor", C.c_int32), ("ss_ver", C.c_int32), ("is_id", C.c_int32),
                ("data", FilmGrainData), ("scratch", C.c_void_p)]


class CompFusedBlock(C.Structure):
    _fields_ = [("dst_off", C.c_uint32), ("mask_off", C.c_uint32), ("src_x", C.c_int32 * 2), ("src_y", C.c_int32 * 2),
                ("w", C.c_uint8), ("h", C.c_uint8), ("mx", C.c_uint8 * 2), ("my", C.c_uint8 * 2), ("ref", C.c_uint8 * 2),
                ("filter2d", C.c_uint8), ("op", C.c_uint8), ("param", C.c_uint8), ("plane", C.c_uint8), ("pad", C.c_uint8 * 4)]


class McScaledBlock(C.Structure):
    _fields_ = [("dst_off", C.c_uint32), ("src_x", C.c_int32), ("src_y", C.c_int32), ("mx", C.c_uint16), ("my", C.c_uint16),
                ("dx", C.c_uint16), ("dy", C.c_uint16), ("w", C.c_uint8), ("h", C.c_uint8), ("filter2d", C.c_uint8),
                ("op", C.c_uint8), ("plane", C.c_uint8), ("ref", C.c_uint8), ("pad", C.c_uint8 * 2)]


class CoefBlock(C.Structure):
    _fields_ = [("dense_off", C.c_uint32), ("compact_off", C.c_uint32), ("eob", C.c_int16), ("tx", C.c_uint8), ("pad", C.c_uint8)]


class IntraTx(C.Structure):
    """struct B200IntraTx (40 bytes)"""
    _fields_ = [("dst_off", C.c_uint32), ("coef_off", C.c_uint32), ("luma_off", C.c_uint32), ("eob", C.c_int16),
                ("x4", C.c_uint16), ("y4", C.c_uint16), ("xend4", C.c_uint16), ("yend4", C.c_uint16),
                ("max_w", C.c_int16), ("max_h", C.c_int16), ("angle_flags", C.c_uint16), ("tx", C.c_uint8),
                ("txtp", C.c_uint8), ("mode", C.c_uint8), ("angle", C.c_int8), ("plane", C.c_uint8), ("flags", C.c_uint8),
                ("cfl_alpha", C.c_int8), ("cfl_w_pad", C.c_uint8), ("cfl_h_pad", C.c_uint8), ("pad", C.c_uint8 * 3)]


class IntraSb(C.Structure):
    _fields_ = [("first", C.c_uint32), ("count", C.c_uint32), ("sx", C.c_uint16), ("sy", C.c_uint16)]


class IntraFrame(C.Structure):
    _fields_ = [("pic", C.c_void_p), ("stride", C.c_int32 * 3), ("ss_hor", C.c_int32), ("ss_ver", C.c_int32),
                ("w4", C.c_int32 * 3), ("h4", C.c_int32 * 3), ("d_coef", C.c_void_p), ("zero_coefs", C.c_int32),
                ("grid", C.c_int32), ("scratch", C.c_void_p), ("plane_off", C.c_uint32 * 3), ("n_sb", C.c_int32),
                ("sb_w", C.c_int32), ("sb_h", C.c_int32), ("sb", C.c_void_p), ("mask", C.c_void_p), ("pal", C.c_void_p), ("done_init", C.c_void_p)]


class ResizeFrame(C.Structure):
    """struct B200ResizeFrame"""
    _fields_ = [("src", C.c_void_p), ("dst", C.c_void_p), ("src_plane_off", C.c_uint32 * 3), ("dst_plane_off", C.c_uint32 * 3),
                ("src_stride", C.c_int32 * 3), ("dst_stride", C.c_int32 * 3), ("src_w", C.c_int32 * 3), ("dst_w", C.c_int32 * 3),
                ("h", C.c_int32 * 3), ("dx", C.c_int32 * 3), ("mx0", C.c_int32 * 3), ("n_planes", C.c_int32), ("pad", C.c_int32)]


class FrameJob(C.Structure):
    """struct B200FrameJob"""
    _fields_ = [("bitdepth_max", C.c_int32), ("zero_coefs", C.c_int32), ("mc", McFrame),
                ("d_pred", C.c_void_p), ("n_pred", C.c_int32), ("pad0", C.c_int32),
                ("d_warp", C.c_void_p), ("n_warp", C.c_int32), ("pad1", C.c_int32),
                ("d_comp", C.c_void_p), ("n_comp", C.c_int32), ("pad2", C.c_int32),
                ("d_comp2", C.c_void_p), ("n_comp2", C.c_int32), ("pad2b", C.c_int32),
                ("d_blend", C.c_void_p), ("n_blend", C.c_int32), ("pad3", C.c_int32),
                ("d_itx", C.c_void_p * 19), ("n_itx", C.c_int32 * 19), ("pad4", C.c_int32),
                ("d_coef", C.c_void_p), ("itx_stride", C.c_int32 * 3),
                ("run_lf", C.c_int32), ("run_cdef", C.c_int32), ("run_lr", C.c_int32),
                ("lf", LfFrame), ("cdef", CdefFrame), ("lr", LrFrame),
                ("d_intra", C.c_void_p), ("n_intra", C.c_int32), ("pad6", C.c_int32), ("intra", IntraFrame),
                ("d_scaled", C.c_void_p), ("n_scaled", C.c_int32), ("pad7", C.c_int32),
                ("d_cfused", C.c_void_p), ("d_cfused2", C.c_void_p), ("n_cfused", C.c_int32), ("n_cfused2", C.c_int32),
                ("d_expand", C.c_void_p), ("n_expand", C.c_int32), ("pad8", C.c_int32), ("d_ccoef", C.c_void_p),
                ("coef_bytes", C.c_uint64),
                ("run_fg", C.c_int32), ("pad5", C.c_int32), ("fg", FgFrame),
                ("d_blend2", C.c_void_p), ("n_blend2", C.c_int32), ("pad9", C.c_int32),
                ("run_resize", C.c_int32), ("pad10", C.c_int32), ("resize", ResizeFrame * 2)]


class FrameBand(C.Structure):
    """struct B200FrameBand"""
    _fields_ = [("y0", C.c_int32), ("y1", C.c_int32), ("last", C.c_int32), ("pad", C.c_int32)] + \
               [(n, C.c_int32 * 2) for n in ("pred", "warp", "comp", "comp2", "blend", "blend2", "scaled", "cfused", "cfused2", "expand")] + \
               [("itx", (C.c_int32 * 2) * 19), ("intra", C.c_int32 * 2), ("edge_top", C.c_void_p), ("edge_bottom", C.c_void_p)]


class PutRange(C.Structure):
    """struct B200PutRange"""
    _fields_ = [("src", C.c_void_p), ("dst", C.c_void_p * 2), ("bytes", C.c_uint64)]


class PutFlag(C.Structure):
    """struct B200PutFlag"""
    _fields_ = [("flag", C.c_void_p), ("base", C.c_void_p), ("sub", C.c_int32), ("shift", C.c_int32), ("add", C.c_int32), ("pad", C.c_int32)]


class Xfer(C.Structure):
    _fields_ = [("host", C.c_void_p), ("dev", C.c_void_p), ("bytes", C.c_uint64)]


ITXFM_FN_8 = C.CFUNCTYPE(None, C.c_void_p, C.c_ssize_t, C.c_void_p, C.c_int)
ITXFM_FN_16 = C.CFUNCTYPE(None, C.c_void_p, C.c_ssize_t, C.c_void_p, C.c_int, C.c_int)

_SIGS = {
    "b200_version": (C.c_int, []),
    "b200_last_error": (C.c_char_p, []),
    "b200_launch_count": (C.c_uint64, []),
    "b200_set_pdl": (None, [C.c_int]),
    "b200_itx_dsp_init_8bpc": (None, [C.c_void_p, C.c_int]),
    "b200_itx_dsp_init_16bpc": (None, [C.c_void_p, C.c_int]),
    "b200_inv_txfm_add": (C.c_int, [C.c_void_p, C.c_ssize_t, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int]),
    "b200_itx_add_batch": (C.c_int, [C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                     C.POINTER(C.c_int32), C.c_int, C.c_void_p]),
    "b200_itx_add_frame": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "b200_itx_add_batch_host": (C.c_int, [C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_size_t,
                                          C.c_void_p, C.c_size_t, C.POINTER(C.c_int32), C.c_int]),
    # ---- mc
    "b200_mc_batch": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "b200_mc_comp_batch": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "b200_mc_blend_batch": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "b200_mc_warp_batch": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "b200_mc_comp_fused_batch": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "b200_mc_scaled_batch": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "b200_mc_put_scaled": (C.c_int, [C.c_void_p, C.c_ssize_t, C.c_void_p, C.c_ssize_t] + [C.c_int] * 8),
    "b200_mc_prep_scaled": (C.c_int, [C.c_void_p, C.c_void_p, C.c_ssize_t] + [C.c_int] * 8),
    "b200_mc_put": (C.c_int, [C.c_void_p, C.c_ssize_t, C.c_void_p, C.c_ssize_t] + [C.c_int] * 6),
    "b200_mc_prep": (C.c_int, [C.c_void_p, C.c_void_p, C.c_ssize_t] + [C.c_int] * 6),
    "b200_mc_comp": (C.c_int, [C.c_void_p, C.c_ssize_t, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
                               C.c_int, C.c_void_p, C.c_int]),
    "b200_mc_blend": (C.c_int, [C.c_void_p, C.c_ssize_t, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int]),
    "b200_mc_warp8x8": (C.c_int, [C.c_int, C.c_void_p, C.c_ssize_t, C.c_void_p, C.c_ssize_t, C.c_void_p,
                                  C.c_int, C.c_int, C.c_int]),
    "b200_mc_emu_edge": (C.c_int, [C.c_ssize_t] * 6 + [C.c_void_p, C.c_ssize_t, C.c_void_p, C.c_ssize_t, C.c_int]),
    "b200_mc_resize": (C.c_int, [C.c_void_p, C.c_ssize_t, C.c_void_p, C.c_ssize_t] + [C.c_int] * 6),
    "b200_resize_frame": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p]),
    "b200_mc_dsp_init_8bpc": (None, [C.c_void_p]),
    "b200_mc_dsp_init_16bpc": (None, [C.c_void_p]),
    # ---- loopfilter
    "b200_lf_frame": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p]),
    "b200_loop_filter_sb": (C.c_int, [C.c_int, C.c_int, C.c_void_p, C.c_ssize_t, C.c_void_p, C.c_void_p,
                                      C.c_ssize_t, C.c_void_p, C.c_int, C.c_int]),
    "b200_loop_filter_dsp_init_8bpc": (None, [C.c_void_p]),
    "b200_loop_filter_dsp_init_16bpc": (None, [C.c_void_p]),
    # ---- cdef
    "b200_cdef_frame": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p]),
    "b200_cdef_dir": (C.c_int, [C.c_void_p, C.c_ssize_t, C.c_void_p, C.c_int]),
    "b200_cdef_fb": (C.c_int, [C.c_void_p, C.c_ssize_t, C.c_void_p, C.c_void_p, C.c_void_p] + [C.c_int] * 8),
    "b200_cdef_dsp_init_8bpc": (None, [C.c_void_p]),
    "b200_cdef_dsp_init_16bpc": (None, [C.c_void_p]),
    # ---- looprestoration
    "b200_lr_frame": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p]),
    "b200_lr_filter": (C.c_int, [C.c_int, C.c_void_p, C.c_ssize_t, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                                 C.c_void_p, C.c_int, C.c_int]),
    "b200_loop_restoration_dsp_init_8bpc": (None, [C.c_void_p, C.c_int]),
    "b200_loop_restoration_dsp_init_16bpc": (None, [C.c_void_p, C.c_int]),
    "b200_coef_expand": (C.c_int, [C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    # ---- intra frame
    "b200_intra_scratch_bytes": (C.c_size_t, [C.c_void_p]),
    "b200_intra_frames": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "b200_frame_run_batch": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    "b200_intra_frame": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    # ---- filmgrain
    "b200_fg_apply_frame": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p]),
    "b200_fg_prep": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p]),
    "b200_fg_apply": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p]),
    "b200_fg_generate_grain": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int]),
    "b200_fgy_32x32xn": (C.c_int, [C.c_void_p, C.c_void_p, C.c_ssize_t, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p,
                                   C.c_int, C.c_int, C.c_int]),
    "b200_fguv_32x32xn": (C.c_int, [C.c_void_p, C.c_void_p, C.c_ssize_t, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p,
                                    C.c_int, C.c_int, C.c_void_p, C.c_ssize_t] + [C.c_int] * 5),
    "b200_film_grain_dsp_init_8bpc": (None, [C.c_void_p]),
    "b200_film_grain_dsp_init_16bpc": (None, [C.c_void_p]),
    # ---- memory / streams for C hosts
    "b200_dev_alloc": (C.c_void_p, [C.c_size_t]),
    "b200_dev_free": (None, [C.c_void_p]),
    "b200_host_alloc": (C.c_void_p, [C.c_size_t]),
    "b200_host_free": (None, [C.c_void_p]),
    "b200_stream_create": (C.c_void_p, []),
    "b200_stream_destroy": (None, [C.c_void_p]),
    "b200_dev_memset": (C.c_int, [C.c_void_p, C.c_int, C.c_size_t, C.c_void_p]),
    # ---- whole frame
    "b200_frame_run": (C.c_int, [C.c_void_p, C.c_void_p]),
    "b200_struct_size": (C.c_int, [C.c_int]),
    "b200_frame_run_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p]),
    "b200_frame_submit_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p]),
    "b200_frame_submit_host_batch": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p]),
    "b200_frame_wait": (C.c_int, [C.c_void_p]),
    # ---- band-sliced job + cross-GPU exchange
    "b200_frame_run_band": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "b200_frame_run_band_phase": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "b200_band_progress": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int]),
    "b200_ipc_export": (C.c_int, [C.c_void_p, C.c_void_p]),
    "b200_ipc_open": (C.c_void_p, [C.c_void_p]),
    "b200_ipc_close": (C.c_int, [C.c_void_p]),
    "b200_copy_async": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "b200_flag_signal": (C.c_int, [C.c_void_p, C.c_uint32, C.c_void_p]),
    "b200_flag_wait_geq": (C.c_int, [C.c_void_p, C.c_uint32, C.c_void_p]),
    "b200_put_rows": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "b200_flag_signal_rel": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    "b200_flag_wait_geq_rel": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    "b200_graph_begin": (C.c_int, [C.c_void_p]),
    "b200_graph_end": (C.c_void_p, [C.c_void_p]),
    "b200_graph_launch": (C.c_int, [C.c_void_p, C.c_void_p]),
    "b200_graph_destroy": (None, [C.c_void_p]),
    "b200_event_create": (C.c_void_p, []),
    "b200_event_destroy": (None, [C.c_void_p]),
    "b200_event_record": (C.c_int, [C.c_void_p, C.c_void_p]),
    "b200_stream_wait_event": (C.c_int, [C.c_void_p, C.c_void_p]),
    # ---- ipred
    "b200_ipred_batch": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "b200_ipred": (C.c_int, [C.c_int, C.c_void_p, C.c_ssize_t, C.c_void_p] + [C.c_int] * 6),
    "b200_cfl_ac": (C.c_int, [C.c_void_p, C.c_void_p, C.c_ssize_t] + [C.c_int] * 7),
    "b200_cfl_pred": (C.c_int, [C.c_int, C.c_void_p, C.c_ssize_t, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int]),
    "b200_pal_pred": (C.c_int, [C.c_void_p, C.c_ssize_t, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int]),
    "b200_intra_pred_dsp_init_8bpc": (None, [C.c_void_p]),
    "b200_intra_pred_dsp_init_16bpc": (None, [C.c_void_p]),
}


class B200Error(RuntimeError):
    pass


class B200Lib:
    """Thin typed wrapper; every symbol include/b200av1.h declares must resolve."""

    def __init__(self, path):
        if not os.path.exists(path):
            raise B200Error("b200av1 library not found: %s" % path)
        self.path = path
        self.dll = C.CDLL(path)
        for name, (res, args) in _SIGS.items():
            fn = getattr(self.dll, name)  # AttributeError if the symbol is missing
            fn.restype = res
            fn.argtypes = args
            setattr(self, name, fn)
        for i, cls in enumerate(ABI_STRUCTS):
            got = self.b200_struct_size(i)
            if got != C.sizeof(cls):
                raise B200Error("ABI mismatch: sizeof(%s) is %d in %s but %d in the Python binding"
                                % (cls.__name__, got, path, C.sizeof(cls)))

    def check(self, rc, what):
        if rc != 0:
            raise B200Error("%s failed (%d): %s" % (what, rc, self.b200_last_error().decode()))

    @staticmethod
    def symbols():
        return list(_SIGS)


ABI_STRUCTS = None   # filled below: index -> ctypes class, checked against b200_struct_size() on load

_lib = None


def get_lib():
    """Load (building first if needed) the CUDA library. Never falls back to anything else."""
    global _lib
    if _lib is None:
        if os.environ.get("B200AV1_LIB"):          # tuning aid: an alternative build of the same library
            _lib = B200Lib(os.environ["B200AV1_LIB"])
            return _lib
        if not os.path.exists(LIB_PATH):
            from . import build
            build.build()
        _lib = B200Lib(LIB_PATH)
    return _lib


class Av1Restoration(C.Structure):
    _fields_ = [("lr", C.c_uint8 * 108)]


ABI_STRUCTS = [McFrame, McBlock, CompBlock, BlendBlock, WarpBlock, ItxBlock, LfFrame, CdefFrame, LrFrame, FrameJob,
               Av1Filter, Av1Restoration, FgFrame, FilmGrainData, IntraTx, IntraFrame, McScaledBlock, CoefBlock, IntraSb, CompFusedBlock, FrameBand, ResizeFrame]
