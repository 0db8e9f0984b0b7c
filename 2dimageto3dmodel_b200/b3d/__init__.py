"""ctypes binding of libb3d.so (the C ABI in include/b3d.h) for the drop-in Python modules.

No torch C++ extension, no CPU fallback: if the shared library is missing, or a tensor is not a
contiguous CUDA fp32 tensor, the call fails loudly.
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libb3d.so")

MODE_REFERENCE = 0
MODE_PAPER = 1
_MODES = {"R": MODE_REFERENCE, "reference": MODE_REFERENCE, "P": MODE_PAPER, "paper": MODE_PAPER,
          0: MODE_REFERENCE, 1: MODE_PAPER}


class B3DError(RuntimeError):
    pass


def _load():
    if not os.path.exists(LIB_PATH):
        raise B3DError(f"{LIB_PATH} is missing: build it with `make` (or __graft_entry__.build()). "
                       "There is no CPU fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    lib.b3d_last_error.restype = ctypes.c_char_p
    lib.b3d_last_variant.restype = ctypes.c_char_p
    lib.b3d_launch_count.restype = ctypes.c_uint64
    lib.b3d_pc_silhouette_workspace_bytes.restype = ctypes.c_size_t
    return lib


lib = _load()

_vp = ctypes.c_void_p
_i = ctypes.c_int
_f = ctypes.c_float
_sz = ctypes.c_size_t
_ll = ctypes.c_longlong


def _sig(name, *argtypes):
    fn = getattr(lib, name)
    fn.argtypes = list(argtypes)
    fn.restype = ctypes.c_int
    return fn


_sig("b3d_pc_bin_count", _i)
_sig("b3d_pc_tma_staging")
_sig("b3d_pc_stage_records")
_sig("b3d_pc_stream_plan", _vp, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp, _i)
_sig("b3d_inception_input", _vp, _i, _i, _i, _i, _i, _i, _i, _vp, _vp)
_sig("b3d_maxpool3x3s2_nhwc", _vp, _i, _i, _i, _i, _vp, _i, _vp)
_sig("b3d_mean_hw_nhwc", _vp, _i, _i, _i, _vp, _vp)
_sig("b3d_fid_accumulate", _vp, _i, _i, _vp, _vp, _vp)
_sig("b3d_pc_project", _vp, _vp, _i, _i, _i, _f, _f, _vp, _vp, _vp, _vp, _vp, _vp, _vp)
_sig("b3d_pc_silhouette_fwd_hosttaps", _vp, _vp, _vp, _i, _vp, _i, _i, _i, _i, _vp, _vp, _sz, _vp)
_sig("b3d_pc_silhouette_bwd_hosttaps", _vp, _vp, _vp, _i, _vp, _vp, _i, _i, _i, _i, _vp, _vp, _vp, _sz, _vp)
_sig("b3d_pc_silhouette_fwd", _vp, _vp, _vp, _i, _vp, _i, _i, _i, _i, _vp, _vp, _sz, _vp)
_sig("b3d_pc_silhouette_bwd", _vp, _vp, _vp, _i, _vp, _vp, _i, _i, _i, _i, _vp, _vp, _vp, _sz, _vp)
_sig("b3d_pc_project_bwd", _vp, _vp, _vp, _vp, _i, _i, _i, _f, _f, _vp, _vp, _vp)
_sig("b3d_pc_splat_grid", _vp, _i, _i, _i, _i, _vp, _vp)
_sig("b3d_mesh_face_setup", _vp, _vp, _vp, _i, _vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp)
_sig("b3d_mesh_render_fwd", _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp)
_sig("b3d_conv2d_tf32", _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i,
     _f, _i, _vp, _i, _vp, _i, _i, _vp, _vp)
_sig("b3d_conv2d_flat_tf32", _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _vp, _i, _i, _i, _f, _vp)
_sig("b3d_conv2d_wgrad_tf32", _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _vp)
_sig("b3d_conv2d_thin_fwd", _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _f, _vp)
_sig("b3d_conv2d_thin_wgrad", _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _vp)
_sig("b3d_vertex_pipeline_fwd", _vp, _ll, _ll, _ll, _ll, _i, _i, _vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp)
_sig("b3d_vertex_pipeline_bwd", _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp)
_sig("b3d_bank_forward", _vp, _vp, _i, _vp, _i, _vp, _i, _vp, _sz, _vp, _i, _vp)
_sig("b3d_bank_backward", _vp, _vp, _i, _vp, _i, _vp, _vp, _vp, _vp)
_sig("b3d_bank_up2_grad", _vp, _vp, _i, _i, _i, _vp)
_sig("b3d_pad_x_fwd", _vp, _vp, _ll, _i, _i, _i, _i, _vp)
_sig("b3d_pad_x_bwd", _vp, _vp, _ll, _i, _i, _i, _i, _vp)
_sig("b3d_stem_input_fwd", _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp)
_sig("b3d_stem_input_bwd", _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp)
_sig("b3d_leaky_bwd", _vp, _vp, _vp, _ll, _f, _vp)
_sig("b3d_fold_rows_fwd", _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp)
_sig("b3d_fold_rows_bwd", _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp)
_sig("b3d_wrap_x_inplace", _vp, _ll, _i, _i, _i, _i, _vp)
_sig("b3d_wrap_x_bwd_inplace", _vp, _ll, _i, _i, _i, _i, _vp)
_sig("b3d_pad_leaky_bias_bwd", _vp, _vp, _vp, _vp, _ll, _i, _i, _i, _i, _f, _vp)
_sig("b3d_vox_blur_axis", _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp)
_sig("b3d_vox_scale_clamp", _vp, _vp, _vp, _i, _i, _vp)
_sig("b3d_vox_scale_clamp_bwd", _vp, _vp, _vp, _vp, _vp, _i, _i, _vp)
_sig("b3d_vox_termination", _vp, _i, _i, _i, _vp, _vp, _vp)
_sig("b3d_vox_termination_bwd", _vp, _vp, _i, _i, _i, _vp, _vp)
_sig("b3d_vox_splat_sorted", _vp, _vp, _i, _i, _i, _i, _vp, _vp)
_sig("b3d_vox_clamp01", _vp, ctypes.c_longlong, _vp)
_sig("b3d_vox_gather", _vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp)
_sig("b3d_bn_stats", _vp, _ll, _i, _f, _vp, _vp, _vp, _vp)
_sig("b3d_cbn_act_fwd", _vp, _vp, _vp, _vp, _i, _i, _vp, _i, _i, _i, _i, _i, _i, _f, _i, _i, _vp)
_sig("b3d_cbn_act_bwd1", _vp, _vp, _vp, _vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _i, _i, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _f, _i, _i, _vp)
_sig("b3d_cbn_act_bwd2", _vp, _vp, _vp, _vp, _vp, _vp, _vp, _f, _i, _i, _i, _i, _vp)
_sig("b3d_bn_sums", _vp, _ll, _i, _vp, _vp)
_sig("b3d_cbn_prepare", _vp, _i, _i, _i, _vp, ctypes.c_double, _f, _f, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _vp)
_sig("b3d_cbn_bwd_reduce", _vp, _vp, _i, _vp, _vp, _i, _i, _vp)
_sig("b3d_cbn_prepare_sync", _vp, _vp, _i, _i, _vp, _vp, _vp, _i, _i, _i, _vp, ctypes.c_double, _f, _f, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
     _vp, _i, _i, _vp)
_sig("b3d_cbn_bwd_reduce_sync", _vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _i, _vp, _vp, _i, _i, _vp)
_sig("b3d_chamfer_nn", _vp, _vp, _i, _i, _i, _vp, _vp, _vp)
_sig("b3d_chamfer_bwd", _vp, _vp, _vp, _vp, _i, _i, _i, _vp, _vp, _vp)
_sig("b3d_flat_loss_fwd", _vp, _vp, _i, _i, _i, _vp, _vp)
_sig("b3d_face_normals_fwd", _vp, _vp, _i, _i, _i, _vp, _vp)
_sig("b3d_face_normals_bwd", _vp, _vp, _vp, _i, _i, _i, _vp, _vp)
_sig("b3d_flat_loss_bwd", _vp, _vp, _i, _i, _i, _vp, _vp, _vp)
_sig("b3d_rgba_mse_iou_fwd", _vp, _vp, _vp, _i, _i, _i, _vp, _vp, _vp)
_sig("b3d_rgba_mse_bwd", _vp, _vp, _vp, _i, _i, _i, _vp, _vp, _vp, _vp)
_sig("b3d_mesh_render_bwd", _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp)


def mode_id(mode):
    try:
        return _MODES[mode]
    except KeyError:
        raise B3DError(f"unknown semantics mode {mode!r} (use 'R' or 'P')") from None


def check(rc):
    if rc != 0:
        raise B3DError(f"libb3d error {rc}: {lib.b3d_last_error().decode()}")


def last_variant():
    """Kernel template instances launched by this thread's most recent convolution entry point (';'-joined)."""
    return lib.b3d_last_variant().decode()


def launch_count():
    return int(lib.b3d_launch_count())


def dev(t, name="tensor", dtype=torch.float32):
    """Validate a tensor for the C ABI and return it (contiguous CUDA tensor of `dtype`)."""
    if not isinstance(t, torch.Tensor):
        raise B3DError(f"{name}: expected a torch.Tensor")
    if not t.is_cuda:
        raise B3DError(f"{name}: libb3d runs on CUDA tensors only (got device {t.device}); "
                       "there is no CPU fallback")
    if t.dtype != dtype:
        raise B3DError(f"{name}: expected dtype {dtype}, got {t.dtype}")
    return t if t.is_contiguous() else t.contiguous()


def ptr(t):
    return _vp(t.data_ptr()) if t is not None else _vp(0)


def stream_ptr(t=None):
    return _vp(torch.cuda.current_stream(t.device if t is not None else None).cuda_stream)


def host_floats(values):
    arr = (ctypes.c_float * len(values))(*[float(v) for v in values])
    return arr


# ---------------------------------------------------------------------------------------------
# optional per-entry-point device timing (bench.py's kernel breakdown): CUDA events recorded on the
# launching stream around every libb3d call.  Off by default; enabling swaps the ctypes attributes.
# ---------------------------------------------------------------------------------------------
_prof_records = None
_prof_saved = {}


_PROF_SHAPES = bool(int(os.environ.get("B3D_PROF_SHAPES", "0")))


def prof_enable():
    global _prof_records
    if _prof_records is not None:
        return
    _prof_records = []
    for name in [n for n in dir(lib) if n.startswith("b3d_")] + list(_TIMED):
        fn = getattr(lib, name)
        if name in _prof_saved or not hasattr(fn, "argtypes") or name in ("b3d_last_error", "b3d_launch_count",
                                                                          "b3d_version", "b3d_last_variant"):
            continue
        _prof_saved[name] = fn

        def wrapper(*args, _fn=fn, _name=name):
            e0 = torch.cuda.Event(enable_timing=True)
            e1 = torch.cuda.Event(enable_timing=True)
            e0.record()
            rc = _fn(*args)
            e1.record()
            if _PROF_SHAPES and _name.startswith("b3d_conv2d"):        # B3D_PROF_SHAPES=1: one key per conv geometry
                _name = _name + ":" + ",".join(str(a) for a in args if isinstance(a, int))
            _prof_records.append((_name, e0, e1))
            return rc

        setattr(lib, name, wrapper)


def prof_disable():
    """-> {entry point: [ms, ...]} and restores the plain ctypes functions."""
    global _prof_records
    if _prof_records is None:
        return {}
    torch.cuda.synchronize()
    out = {}
    for name, e0, e1 in _prof_records:
        out.setdefault(name, []).append(e0.elapsed_time(e1))
    for name, fn in _prof_saved.items():
        setattr(lib, name, fn)
    _prof_saved.clear()
    _prof_records = None
    return out


_TIMED = ("b3d_pc_project", "b3d_pc_silhouette_fwd_hosttaps", "b3d_pc_silhouette_bwd_hosttaps", "b3d_pc_project_bwd",
          "b3d_pc_splat_grid", "b3d_mesh_face_setup", "b3d_mesh_render_fwd", "b3d_mesh_render_bwd", "b3d_face_normals_fwd", "b3d_face_normals_bwd", "b3d_flat_loss_fwd",
          "b3d_flat_loss_bwd", "b3d_rgba_mse_iou_fwd", "b3d_rgba_mse_bwd", "b3d_chamfer_nn", "b3d_chamfer_bwd", "b3d_conv2d_tf32", "b3d_conv2d_flat_tf32", "b3d_conv2d_wgrad_tf32", "b3d_conv2d_thin_fwd", "b3d_conv2d_thin_wgrad", "b3d_pad_x_fwd", "b3d_pad_x_bwd", "b3d_stem_input_fwd", "b3d_stem_input_bwd",
          "b3d_leaky_bwd", "b3d_bn_stats", "b3d_wrap_x_inplace", "b3d_wrap_x_bwd_inplace", "b3d_pad_leaky_bias_bwd", "b3d_fold_rows_fwd", "b3d_fold_rows_bwd", "b3d_cbn_act_fwd", "b3d_cbn_act_bwd1", "b3d_cbn_act_bwd2", "b3d_bn_sums", "b3d_cbn_prepare", "b3d_cbn_bwd_reduce",
          "b3d_bank_forward", "b3d_bank_backward", "b3d_vertex_pipeline_fwd", "b3d_vertex_pipeline_bwd")
