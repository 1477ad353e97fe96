"""ctypes binding of libdca_b200.so (the C ABI declared in include/dca_b200.h).

There is NO fallback: if the shared library is missing the import of any compute entry point raises.
Build it with `python <package>/build.py` (or `__graft_entry__.build()`).
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libdca_b200.so")

_c_int = ctypes.c_int
_vp = ctypes.c_void_p
_f = ctypes.c_float
_ll = ctypes.c_longlong

# name -> argtypes (return type is int unless listed in _RESTYPES)
SIGNATURES = {
    "dca_version": [],
    "dca_plane_format": [],
    "dca_volume_gwc_concat": [_vp, _vp, _vp, _vp, _vp] + [_c_int] * 9 + [_vp],
    "dca_build_gwc_volume_f32": [_vp, _vp, _vp] + [_c_int] * 6 + [_vp],
    "dca_build_concat_volume_f32": [_vp, _vp, _vp] + [_c_int] * 5 + [_vp],
    "dca_conv3d_direct": [_c_int, _vp, _c_int, _vp, _vp, _vp, _vp, _vp, _c_int, _vp, _c_int, _c_int, _c_int]
                         + [_c_int] * 10 + [_vp],
    "dca_conv3d_cout1": [_vp, _c_int, _vp, _vp] + [_c_int] * 5 + [_vp],
    "dca_conv3d_tc": [_c_int, _vp, _c_int, _vp, _vp, _vp, _vp, _vp, _c_int, _vp, _c_int, _vp, _c_int, _vp, _c_int,
                      _c_int] + [_c_int] * 9 + [_vp],
    "dca_pack_weights_tc": [_vp, _c_int, _c_int, _c_int, _c_int, _vp, _c_int, _vp],
    "dca_pack_weights_tc_bytes": [_c_int] * 4,
    "dca_conv3d_tc_march": [_vp, _c_int, _vp, _vp, _vp, _vp, _vp, _c_int, _vp, _c_int] + [_c_int] * 5 + [_vp],
    "dca_pack_weights_tc_march": [_vp, _c_int, _vp, _c_int, _vp],
    "dca_pack_weights_tc_march_bytes": [_c_int] * 2,
    "dca_conv1_taps_tc": [_vp, _c_int, _vp, _vp] + [_c_int] * 5 + [_vp],
    "dca_conv3d_tc_taps27": [_vp, _c_int, _vp, _c_int, _vp, _vp, _vp, _vp, _c_int] + [_c_int] * 5 + [_vp],
    "dca_tap_gather_softmax_regress": [_vp, _vp, _vp] + [_c_int] * 4 + [_vp],
    "dca_tap_gather3d": [_vp, _vp] + [_c_int] * 4 + [_vp],
    "dca_conv2d_tc": [_vp, _c_int, _vp, _vp, _vp, _vp, _c_int, _c_int] + [_c_int] * 5 + [_vp],
    "dca_conv2d_tc_ex": [_vp, _c_int, _vp, _vp, _vp, _vp, _c_int, _vp, _c_int, _c_int] + [_c_int] * 6 + [_vp],
    "dca_conv2d_stem": [_vp, _vp, _vp, _vp, _vp, _c_int, _c_int] + [_c_int] * 4 + [_vp],
    "dca_conv2d_tc_cat": [_vp, _c_int, _vp, _c_int, _vp, _c_int, _c_int, _vp, _vp, _vp, _vp, _c_int, _c_int]
                         + [_c_int] * 4 + [_vp],
    "dca_planes_to_nchw_slice": [_vp, _c_int, _vp] + [_c_int] * 5 + [_ll, _vp],
    "dca_pack_weights_tc2d": [_vp, _c_int, _c_int, _vp, _c_int, _vp],
    "dca_pack_weights_tc2d_bytes": [_c_int] * 3,
    "dca_tc_set_halo": [_c_int],
    "dca_set_pdl": [_c_int],
    "dca_pdl_enabled": [],
    "dca_tc_set_deconv_pair": [_c_int],
    "dca_tc_set_march_n": [_c_int],
    "dca_tap_gather_set_groups": [_c_int],
    "dca_tc_set_up2_side_slots": [_c_int],
    "dca_volume_set_v2": [_c_int],
    "dca_attention_set_team": [_c_int],
    "dca_tc_set_tuning": [_c_int, _c_int],
    "dca_tc_set_trunc_comp": [_f],
    "dca_avgpool3d": [_vp, _vp] + [_c_int] * 6 + [_vp],
    "dca_avgpool3d_simple": [_vp, _vp] + [_c_int] * 6 + [_vp],
    "dca_pool_set_march": [_c_int],
    "dca_class_stats": [_vp, _vp, _vp, _vp, _vp] + [_c_int] * 4 + [_vp],
    "dca_disp_attention": [_vp, _vp, _vp, _vp, _vp, _c_int, _vp] + [_c_int] * 7 + [_vp],
    "dca_self_attention": [_vp, _vp, _vp, _vp] + [_c_int] * 6 + [_vp],
    "dca_regress_f32": [_vp, _vp] + [_c_int] * 4 + [_vp],
    "dca_up2_tc": [_c_int, _vp, _c_int, _vp, _c_int, _vp, _vp, _vp, _vp, _c_int, _vp, _c_int] + [_c_int] * 5 + [_vp],
    "dca_upsample_fuse": [_vp] * 6 + [_c_int] * 6 + [_vp],
    "dca_softmax_regress": [_vp, _vp] + [_c_int] * 4 + [_vp],
    "dca_convex_upsample": [_vp, _vp, _vp] + [_c_int] * 3 + [_vp],
    "dca_planes_from_ncdhw": [_vp, _vp] + [_c_int] * 7 + [_vp],
    "dca_planes_to_ncdhw": [_vp, _c_int, _vp] + [_c_int] * 6 + [_vp],
    "dca_pack_weights": [_vp, _c_int, _c_int, _c_int, _c_int, _vp, _c_int, _vp],
    "dca_conv3d_igemm": [_c_int, _vp, _c_int, _vp, _vp, _vp, _vp, _vp, _c_int, _vp, _c_int, _vp, _c_int, _vp, _c_int,
                         _c_int] + [_c_int] * 9 + [_vp],
    "dca_pool_conv": [_vp, _vp, _vp, _vp, _vp, _vp] + [_c_int] * 7 + [_vp],
    "dca_softmax_regress_upsample": [_vp, _vp, _vp, _vp] + [_c_int] * 4 + [_vp],
    "dca_halo_push_ctas": [],
    "dca_halo_set_timeout_ms": [_c_int],
    "dca_halo_push": [_vp, _ll, _ll, _ll, _c_int, _c_int, _vp, _vp, _vp, _vp, _vp],
    "dca_halo_exchange": [_vp, _ll, _ll, _ll, _c_int, _c_int, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, ctypes.c_ulonglong, _vp, _vp],
    "dca_halo_wait_unpack": [_vp, _ll, _ll, _ll, _c_int, _c_int, _vp, _vp, _vp, _vp, ctypes.c_ulonglong, _vp, _vp],
    "dca_adaptive_avgpool3d_rows": [_vp, _vp] + [_c_int] * 8 + [_vp],
    "dca_fold_bn": [_vp, _vp, _vp, _vp, _f, _vp, _vp, _c_int, _c_int, _vp],
    "dca_disparity_metrics": [_vp, _vp, _vp] + [_c_int] * 3 + [_f, _vp],
    "dca_class_confusion": [_vp, _vp, _vp] + [_c_int] * 4 + [_f, _vp],
    "dca_softmax_confidence_upsample": [_vp] * 6 + [_c_int] * 4 + [_vp],
    "dca_confidence_histograms": [_vp] * 5 + [_c_int] * 3 + [_f, _vp],
    "dca_lr_consistency": [_vp, _vp, _c_int, _vp, _vp, _vp] + [_c_int] * 3 + [_f, _vp],
    "dca_reproject": [_vp, _vp, _vp, _ll, _ll] + [_c_int] * 5 + [_vp, _vp, _f, _f, _f] + [_vp] * 6,
    "dca_depth_metrics": [_vp, _vp, _vp] + [_c_int] * 3 + [_f] * 5 + [_vp],
    "dca_rectify": [_vp, _vp, _c_int, _ll, _ll] + [_c_int] * 3 + [_vp] + [_c_int] * 2 + [_vp] * 3,
    "dca_standardise_frame": [_vp, _vp] + [_c_int] * 3 + [_vp, _vp] + [_c_int] * 6 + [_vp],
    "dca_wls_filter": [_vp, _vp, _vp, _ll, _ll] + [_c_int] * 3 + [_vp, _c_int, _ll, _ll, _vp, _f, _c_int, _f]
                      + [_vp] * 4,
    "dca_tsdf_integrate": [_vp] + [_c_int] * 4 + [_f] * 4 + [_c_int] * 6 + [_vp, _vp, _ll, _ll] + [_c_int] * 3
                          + [_vp, _c_int, _ll, _ll] + [_f] * 4 + [_c_int] * 2 + [_vp] + [_f] * 3 + [_vp],
    "dca_tsdf_count_surface": [_vp] + [_c_int] * 4 + [_f, _vp, _vp, _vp],
    "dca_tsdf_extract_surface": [_vp] + [_c_int] * 4 + [_f] * 5 + [_vp, _ll, _vp, _vp, _vp, _vp],
    "dca_tsdf_raycast": [_vp] + [_c_int] * 4 + [_f] * 10 + [_c_int] * 4 + [_vp, _f, _f] + [_vp, _ll] * 4 + [_vp],
    "dca_icp_track": [_vp, _vp, _ll, _c_int, _c_int] + [_f] * 4 + [_c_int] * 2 + [_f, _vp, _ll, _vp, _ll, _vp, _c_int]
                     + [_vp] * 3 + [_c_int] + [_vp] * 5,
}
_RESTYPES = {"dca_pack_weights_tc_bytes": ctypes.c_longlong, "dca_pack_weights_tc2d_bytes": ctypes.c_longlong,
             "dca_pack_weights_tc_march_bytes": ctypes.c_longlong}

ERRORS = {-1: "DCA_ERR_ARG (bad pointer/shape)", -2: "DCA_ERR_LAUNCH (CUDA launch failed)",
          -3: "DCA_ERR_UNSUPPORTED (shape outside what the kernels support)"}

_lib = None
LAUNCHES = 0   # kernels launched through this binding (bench.py reports it as gpu_launches)


class DcaError(RuntimeError):
    pass


def load():
    """Load the shared library (once) and declare every prototype.  Raises if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise DcaError(f"{LIB_PATH} not found: the CUDA extension is not built and there is no CPU fallback. "
                       f"Run `python {os.path.join(_HERE, 'build.py')}`.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, args in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if a declared symbol is not exported
        fn.argtypes = args
        fn.restype = _RESTYPES.get(name, ctypes.c_int)
    _lib = lib
    if os.environ.get("DCA_PDL", "1") == "0":       # diagnostics: plain stream order instead of programmatic dependent launch
        lib.dca_set_pdl(0)
    return lib


PROFILE = None   # set to a list to record (label, start_event, end_event) around every call (diagnostics)


def profile_summary():
    """Aggregate PROFILE records -> {label: (count, total_ms)} (synchronises)."""
    import torch
    torch.cuda.synchronize()
    agg = {}
    for label, a, b in PROFILE or []:
        n, tot = agg.get(label, (0, 0.0))
        agg[label] = (n + 1, tot + a.elapsed_time(b))
    return agg


def call(name, *args):
    """Invoke an entry point; non-zero status raises DcaError (the reference raises on its asserts)."""
    global LAUNCHES
    if PROFILE is not None:
        import torch
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        rc = getattr(load(), name)(*args)
        b.record()
        label = name
        if name in ("dca_conv3d_tc", "dca_conv3d_direct"):
            ints = [x for x in args if isinstance(x, int) and 0 < x < 4096]
            label = f"{name} mode={args[0]} dims={args[-10:-1] if name == 'dca_conv3d_tc' else args[-11:-1]}"
            if name == 'dca_conv3d_tc':
                label += (' +up' if args[9] else '') + (' +side' if args[11] else '')
        PROFILE.append((label, a, b))
        if rc != 0:
            raise DcaError(f"{name} failed: {ERRORS.get(rc, rc)}")
        return
    LAUNCHES += 8 if (name == "dca_conv3d_direct" and args[0] == 2) else 1
    rc = getattr(load(), name)(*args)
    if rc != 0:
        raise DcaError(f"{name} failed: {ERRORS.get(rc, rc)}")
