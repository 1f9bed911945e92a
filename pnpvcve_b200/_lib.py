"""ctypes binding of libpnpvcve.so (C ABI in include/pnp_vcve.h).

There is no CPU or PyTorch fallback: if the library is missing or the device is not sm_100 the
calls raise.  The library is built in-tree by ``pnpvcve_b200/build.py`` (``__graft_entry__.build``).
"""
import ctypes
import os

HERE = os.path.dirname(os.path.abspath(__file__))
#: PNP_LIB_PATH selects another BUILD of the same library (A/B timing of kernel revisions in tools/); it is
#: not a fallback -- whatever it names must export the same C ABI
LIB_PATH = os.environ.get("PNP_LIB_PATH") or os.path.join(HERE, "libpnpvcve.so")

PNP_CONV_BF16, PNP_CONV_LAST = 0, 1
PNP_ACT_NONE, PNP_ACT_LRELU, PNP_ACT_RELU = 0, 1, 2

#: every symbol include/pnp_vcve.h declares
EXPORTS = [
    "pnp_abi_version", "pnp_last_error", "pnp_device_check", "pnp_device_pairs", "pnp_set_pair_mode",
    "pnp_graph_begin", "pnp_graph_end", "pnp_graph_launch", "pnp_graph_destroy", "pnp_set_step", "pnp_fetch_pinned",
    "pnp_mv_warp", "pnp_mv_warp_dyn", "pnp_lr_im2col", "pnp_lr_im2col_dyn", "pnp_pack_conv3x3_rowstack",
    "pnp_pack_rows", "pnp_pack_aux", "pnp_pack_mix_blocks",
    "pnp_caa_heads", "pnp_mix_bias", "pnp_mv_rasterize", "pnp_conv3x3", "pnp_frame_quality", "pnp_frame_quality_u8",
    "pnp_unit_from_u8", "pnp_mv_rasterize_window",
]

_c = ctypes
_vp, _i, _i64 = _c.c_void_p, _c.c_int, _c.c_int64


class DynRef(_c.Structure):
    """struct pnp_dyn_ref"""
    _fields_ = [("table", _vp), ("step", _vp), ("node", _c.c_int32), ("stride", _c.c_int32)]


class ConvDesc(_c.Structure):
    """struct pnp_conv_desc"""
    _fields_ = [
        ("src", _vp), ("aux", _vp), ("idt", _vp), ("out", _vp), ("wpack", _vp),
        ("scale", _vp), ("bias", _vp),
        ("par", _vp), ("par_sn", _i64), ("par_sc", _i64), ("par_sy", _i64),
        ("lq", _vp), ("lq_sn", _i64), ("lq_sc", _i64), ("lq_sy", _i64),
        ("outf", _vp), ("of_sn", _i64), ("of_sc", _i64), ("of_sy", _i64),
        ("N", _c.c_int32), ("H", _c.c_int32), ("W", _c.c_int32),
        ("tap_n", _c.c_int32), ("aux_k16", _c.c_int32), ("act", _c.c_int32), ("mode", _c.c_int32),
        ("flip_y", _c.c_int32),
        ("out_spx", _i64), ("out_sy", _i64), ("out_sn", _i64),
        ("lq_up4", _c.c_int32), ("par_sparse", _c.c_int32), ("wpack_stable", _c.c_int32), ("per_image", _c.c_int32),
        ("img_off", _vp),
        ("dyn", DynRef),
        ("src_images", _c.c_int32), ("aux_images", _c.c_int32), ("idt_images", _c.c_int32), ("out_images", _c.c_int32),
        ("aux_channels", _c.c_int32), ("out_u8", _c.c_int32),
    ]


#: one 64-byte launch-table entry = 8 uint64 words: p[0..5], then (i[0] | i[1] << 32), (i[2] | i[3] << 32)
DYN_ENTRY_WORDS = 8


_PROTOS = {
    "pnp_abi_version": (_i, []),
    "pnp_last_error": (_c.c_char_p, []),
    "pnp_device_check": (_i, []),
    "pnp_device_pairs": (_i, []),
    "pnp_set_pair_mode": (_i, [_i]),
    "pnp_graph_begin": (_i, [_vp]),
    "pnp_graph_end": (_i, [_vp, _c.POINTER(_vp)]),
    "pnp_graph_launch": (_i, [_vp, _vp, _c.c_int32, _vp]),
    "pnp_graph_destroy": (_i, [_vp]),
    "pnp_set_step": (_i, [_vp, _c.c_int32, _vp]),
    "pnp_fetch_pinned": (_i, [_vp, _vp, _i64, _vp]),
    "pnp_mv_warp_dyn": (_i, [_c.POINTER(DynRef), _vp, _i, _i64, _i64, _i, _i, _i, _vp]),
    "pnp_lr_im2col_dyn": (_i, [_c.POINTER(DynRef), _i64, _i64, _i64, _i, _i, _i, _i, _vp]),
    "pnp_pack_mix_blocks": (_i, [_vp, _vp, _i, _i, _vp, _vp, _vp, _i64, _vp]),
    "pnp_mv_warp": (_i, [_vp, _vp, _vp, _i64, _i64, _vp, _i, _i, _i, _vp, _vp, _vp]),
    "pnp_lr_im2col": (_i, [_vp, _i64, _i64, _i64, _vp, _i, _i, _i, _i, _vp]),
    "pnp_pack_conv3x3_rowstack": (_i, [_vp, _i, _vp, _vp, _i, _i, _i, _i, _i, _vp, _i, _i, _vp]),
    "pnp_pack_rows": (_i, [_vp, _i, _i, _i64, _i64, _vp, _i, _vp]),
    "pnp_pack_aux": (_i, [_vp, _i, _i, _vp, _vp]),
    "pnp_caa_heads": (_i, [_vp, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _vp, _vp, _vp]),
    "pnp_mix_bias": (_i, [_vp, _i, _i, _vp, _vp, _i, _vp, _vp]),
    "pnp_mv_rasterize": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "pnp_mv_rasterize_window": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "pnp_conv3x3": (_i, [_c.POINTER(ConvDesc), _vp]),
    "pnp_frame_quality": (_i, [_vp, _i64, _i64, _i64, _vp, _i64, _i64, _i64, _i, _i, _i, _i, _vp, _vp, _vp]),
    "pnp_frame_quality_u8": (_i, [_vp, _i, _i64, _i64, _i64, _vp, _i, _i64, _i64, _i64, _i, _i, _i, _i, _vp, _vp, _vp]),
    "pnp_unit_from_u8": (_i, [_vp, _i64, _i64, _i64, _vp, _i64, _i64, _i64, _i, _i, _i, _vp]),
}

_lib = None


class PnpError(RuntimeError):
    pass


def load():
    """Load the shared library (once).  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        # not a fallback: the same sm_100a library, compiled on demand when nvcc is at hand
        try:
            from . import build as _build
            _build.build()
        except Exception:  # noqa: BLE001 - reported below
            pass
    if not os.path.isfile(LIB_PATH):
        raise PnpError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; "
            "g.build()'` (nvcc, sm_100a).  pnpvcve_b200 has no CPU / PyTorch fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in _PROTOS.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc, what=""):
    if rc != 0:
        msg = load().pnp_last_error().decode(errors="replace")
        raise PnpError(f"{what or 'libpnpvcve'} failed ({rc}): {msg}")


def require_device():
    """Raises unless the current CUDA device can run the kernels (sm_100)."""
    check(load().pnp_device_check(), "pnp_device_check")
