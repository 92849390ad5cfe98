"""ctypes binding of libngp_b200.so (declared in include/ngp_b200.h).

The library is the product: if it is missing or a call fails this module raises - there is no
CPU or PyTorch fallback for any op.
"""
import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libngp_b200.so")

NGP_F32, NGP_F16 = 0, 1
LAYOUT_LBC, LAYOUT_BLC = 0, 1

_u32, _f32, _i32, _u64, _vp = C.c_uint32, C.c_float, C.c_int, C.c_uint64, C.c_void_p

# name -> (restype, argtypes); mirrors include/ngp_b200.h one to one (tests check the export list).
SIGNATURES = {
    "ngp_version": (_i32, []),
    "ngp_error_string": (C.c_char_p, [_i32]),
    "ngp_device_info": (_i32, [C.c_char_p, _i32, C.POINTER(_i32), C.POINTER(_i32), C.POINTER(_i32)]),
    "ngp_grid_encode_forward": (_i32, [_vp, _vp, _vp, _vp, _u32, _u32, _u32, _u32, _f32, _u32, _vp, _u32, _i32, _i32, _i32, _vp]),
    "ngp_grid_encode_backward": (_i32, [_vp, _vp, _vp, _vp, _vp, _u32, _u32, _u32, _u32, _f32, _u32, _vp, _vp, _u32, _i32, _i32, _i32, _i32, _vp]),
    "ngp_grid_set_option": (_i32, [_i32, _i32]),
    "ngp_grid_red_count": (_i32, [C.POINTER(_u64), _i32]),
    "ngp_grid_level_params": (_i32, [_u32, _f32, _u32, _vp, _vp, _vp]),
    "ngp_near_far_from_aabb": (_i32, [_vp, _vp, _vp, _u32, _f32, _vp, _vp, _vp]),
    "ngp_sph_from_ray": (_i32, [_vp, _vp, _f32, _u32, _vp, _vp]),
    "ngp_morton3D": (_i32, [_vp, _u32, _vp, _vp]),
    "ngp_morton3D_invert": (_i32, [_vp, _u32, _vp, _vp]),
    "ngp_packbits": (_i32, [_vp, _u32, _f32, _vp, _vp]),
    "ngp_march_rays_train": (_i32, [_vp, _vp, _vp, _f32, _f32, _u32, _u32, _u32, _u32, _u32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _u64, _vp]),
    "ngp_march_rays_train_packed": (_i32, [_vp, _vp, _vp, _f32, _f32, _u32, _u32, _u32, _u32, _u32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "ngp_march_set_option": (_i32, [_i32, _i32]),
    "ngp_march_rays_train_workspace": (_u64, [_u32, _u32]),
    "ngp_composite_rays_train_forward": (_i32, [_vp, _vp, _vp, _vp, _u32, _u32, _f32, _vp, _vp, _vp, _vp]),
    "ngp_composite_rays_train_backward": (_i32, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _u32, _u32, _f32, _vp, _vp, _vp]),
    "ngp_march_rays": (_i32, [_u32, _u32, _vp, _vp, _vp, _vp, _f32, _f32, _u32, _u32, _u32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "ngp_composite_rays": (_i32, [_u32, _u32, _f32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "ngp_compact_alive": (_i32, [_vp, _u32, _vp, _vp, _vp, _u64, _vp]),
    "ngp_compact_alive_workspace": (_u64, [_u32]),
    "ngp_freq_encode_forward": (_i32, [_vp, _u32, _u32, _u32, _u32, _vp, _vp]),
    "ngp_freq_encode_backward": (_i32, [_vp, _vp, _u32, _u32, _u32, _u32, _vp, _vp]),
    "ngp_occupancy_cell_points": (_i32, [_u32, _f32, _f32, _vp, _vp, _vp]),
    "ngp_occupancy_cell_points_range": (_i32, [_u32, _f32, _f32, _vp, _u32, _u32, _vp, _vp]),
    "ngp_update_density_grid": (_i32, [_vp, _vp, _u32, _f32, _f32, _vp, _vp, _vp, _u64, _vp]),
    "ngp_bench_gather4": (_i32, [_vp, _u32, _vp, _u32, _u32, _u32, _vp]),
    "ngp_bench_red8": (_i32, [_vp, _u32, _u32, _u32, _u32, _vp]),
    "ngp_bench_red_width": (_i32, [_vp, _u32, _u32, _u32, _u32, _u32, _u32, _vp]),
    "ngp_field_forward": (_i32, [_vp, _u32, _vp, _vp, _vp, _u32, _u32, _f32, _u32, _u32, _i32, _f32, _vp, _vp, _vp, _vp, _vp, _vp,
                                 _u32, _u32, _vp, _vp, _vp, _vp, _vp, _vp]),
    "ngp_field_forward_quads": (_i32, [_vp, _u32, _vp, _vp, _vp, _vp, _u32, _u32, _f32, _u32, _u32, _i32, _f32, _vp, _vp, _vp, _vp, _vp,
                                       _vp, _u32, _u32, _vp, _vp, _vp, _vp, _vp, _vp]),
    "ngp_grid_quad_table": (_i32, [_vp, _vp, _u32, _u32, _f32, _u32, _u32, _i32, _vp, _vp]),
    "ngp_field_backward": (_i32, [_u32, _vp, _vp, _vp, _vp, _u32, _u32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                  _vp, _vp, _vp, _vp]),
    "ngp_grid_scatter_samples": (_i32, [_vp, _vp, _f32, _vp, _u32, _vp, _u32, _u32, _f32, _u32, _u32, _i32, _vp, _vp]),
    "ngp_grid_scatter_samples_split": (_i32, [_vp, _vp, _f32, _vp, _u32, _vp, _u32, _u32, _f32, _u32, _u32, _i32, _vp, _vp, _vp]),
    "ngp_grid_fold_odd": (_i32, [_vp, _vp, _u64, _vp]),
    "ngp_stamp": (_i32, [_vp, _vp]),
    "ngp_graph_launch": (_i32, [_vp, _vp]),
    "ngp_tc_selftest": (_i32, [_i32, _vp, _vp, _vp, _u32, _u32, _u32, _vp]),
    "ngp_field_set_option": (_i32, [_i32, _i32]),
    "ngp_bg_forward": (_i32, [_vp, _u32, _vp, _vp, _vp, _vp, _u32, _u32, _vp, _vp]),
    "ngp_bg_backward": (_i32, [_vp, _vp, _u32, _vp, _vp, _vp, _vp, _u32, _u32, _vp, _vp, _vp, _vp, _vp]),
    "ngp_check_finite": (_i32, [_vp, _u64, _vp, _vp]),
    "ngp_check_finite_fold": (_i32, [_vp, _u64, _vp, _vp, _u64, _vp, _vp]),
    "ngp_adam_step": (_i32, [_vp, _vp, _vp, _vp, _vp, _u64, _u32, C.POINTER(_u64), C.POINTER(_f32), _f32, _f32, _f32, _f32,
                             _f32, _f32, _f32, _f32, _u32, _i32, _vp, _vp, _vp]),
    "ngp_adam_step_dp": (_i32, [_vp, _vp, _vp, _vp, _vp, _u64, _u32, C.POINTER(_u64), C.POINTER(_f32), _f32, _f32, _f32, _f32,
                                _f32, _f32, _f32, _f32, _u32, _i32, _vp, _vp, _u32, _u32, C.POINTER(_u64), C.POINTER(_u64),
                                C.POINTER(_u64), C.POINTER(_u64), C.POINTER(_u64), _vp]),
    "ngp_dp_flags_bytes": (_u64, []),
    "ngp_dp_set_option": (_i32, [_i32, _i32]),
    "ngp_enable_peer_access": (_i32, [_i32]),
    "ngp_train_prologue": (_i32, [_vp, _vp, _vp, _u32, _f32, _vp, _vp, _vp, _u32, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "ngp_train_light": (_i32, [_vp, _vp, _i32, _vp, _vp]),
    "ngp_stencil_points": (_i32, [_vp, _u32, _vp, _f32, _f32, _i32, _vp, _vp, _vp]),
    "ngp_shade_forward": (_i32, [_vp, _vp, _u32, _u32, _vp, _f32, _i32, _vp, _vp, _vp]),
    "ngp_shade_backward": (_i32, [_vp, _vp, _u32, _u32, _vp, _f32, _i32, _vp, _vp, _vp, _vp, _vp]),
    "ngp_shade_forward_step": (_i32, [_vp, _vp, _u32, _vp, _vp, _f32, _i32, _vp, _vp, _vp]),
    "ngp_shade_backward_step": (_i32, [_vp, _vp, _u32, _vp, _vp, _u32, _vp, _vp, _f32, _i32, _vp, _vp, _f32, _vp, _vp, _vp, _vp,
                                       _vp]),
    "ngp_render_infer_workspace": (_u64, [_u32]),
    "ngp_render_infer_loop": (_i32, [_vp, _vp, _vp, _vp, _u32, _f32, _f32, _u32, _u32, _u32, _vp, _f32, _vp, _vp, _vp, _u32, _u32, _f32,
                                     _u32, _u32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _u32, _u32, _vp, _vp, _vp, _vp, _u64, _vp]),
    "ngp_render_infer_loop_quads": (_i32, [_vp, _vp, _vp, _vp, _u32, _f32, _f32, _u32, _u32, _u32, _vp, _f32, _vp, _vp, _vp, _vp, _u32, _u32,
                                           _f32, _u32, _u32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _u32, _u32, _vp, _vp, _vp, _vp, _u64, _vp]),
    "ngp_render_infer_state": (_i32, [_vp, C.POINTER(_i32), _vp]),
    "ngp_get_rays": (_i32, [_vp, _vp, _i32, _u32, _u32, _u32, _u32, _u32, _u32, _vp, _vp, _vp]),
    "ngp_train_prologue_rays": (_i32, [_vp, _vp, _i32, _u32, _u32, _u32, _u32, _u32, _u32, _vp, _vp, _vp, _f32, _vp, _vp, _vp, _u32,
                                       _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "ngp_train_ray_loss": (_i32, [_vp, _vp, _vp, _vp, _u32, _u32, _f32, _vp, _f32, _vp, _u32, _u32, _u32, _f32, _vp, _vp, _vp,
                                  _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "ngp_blend_background_forward": (_i32, [_vp, _vp, _vp, _vp, _i32, _vp, _vp, _u32, _vp, _vp, _vp, _vp]),
    "ngp_blend_background_backward": (_i32, [_vp, _vp, _vp, _i32, _u32, _vp, _vp, _vp]),
    "ngp_entropy_loss_forward": (_i32, [_vp, _u32, _f32, _vp, _vp]),
    "ngp_entropy_loss_backward": (_i32, [_vp, _u32, _f32, _vp, _vp, _i32, _vp]),
}

_lib = None


def load():
    """Load the CUDA library; raises ImportError (loudly) when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "libngp_b200.so is not built (expected at %s). Run `python __graft_entry__.py build` or "
            "`python single-stable-dreamfusion_b200/ngp_b200/build.py`; there is no fallback path." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the header and the library ever drift apart
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def error_string(code):
    return load().ngp_error_string(int(code)).decode()


def check(rc, what):
    if rc != 0:
        raise RuntimeError("%s failed: %s (code %d)" % (what, error_string(rc), rc))


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    return None if t is None else t.data_ptr()


def stream():
    return torch.cuda.current_stream().cuda_stream


def require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RuntimeError("expected a CUDA tensor (the B200 path has no CPU fallback)")


def require_contiguous(*tensors):
    for t in tensors:
        if t is not None and not t.is_contiguous():
            raise RuntimeError("expected a contiguous tensor")


# kernels launched per entry point (for bench.py's gpu_launches claim); everything else launches one
KERNELS_PER_CALL = {"ngp_march_rays_train": 3, "ngp_update_density_grid": 2, "ngp_compact_alive": 2}
DEBUG_SYNC = os.environ.get("NGP_DEBUG_SYNC", "0") not in ("", "0")   # synchronise + check for a CUDA fault after EVERY entry point
#                    (the reference never checks: faults surface at the next sync, SURVEY 8b; this pins them to the call)
LAUNCHES = 0       # running count of our kernels launched through this module
PROFILE = None     # optional {entry point name: [(start_event, end_event), ...]} filled while set (bench.py)
TRACE = None       # optional dict(buf=int64 device tensor, rows=[(name, stream id)]): every entry point called while it is
#                    set is bracketed by two ngp_stamp launches (%globaltimer) on its stream - capturable, so a graphed step
#                    replays its own timeline into `buf` (profiles/tools/timeline.py)


def call(name, device, *args):
    """Invoke an entry point with `device` current and the caller's current stream appended."""
    global LAUNCHES
    lib = load()
    with torch.cuda.device(device):
        prof = PROFILE.get(name) if PROFILE is not None else None
        if prof is not None:
            e0 = torch.cuda.Event(enable_timing=True)
            e1 = torch.cuda.Event(enable_timing=True)
            e0.record()
            rc = getattr(lib, name)(*args, stream())
            e1.record()
            prof.append((e0, e1))
        elif TRACE is not None and 2 * len(TRACE["rows"]) + 2 <= TRACE["buf"].numel():
            st = stream()
            i = len(TRACE["rows"])
            TRACE["rows"].append((name, st))
            base = TRACE["buf"].data_ptr()
            lib.ngp_stamp(base + 16 * i, st)
            rc = getattr(lib, name)(*args, st)
            lib.ngp_stamp(base + 16 * i + 8, st)
        else:
            rc = getattr(lib, name)(*args, stream())
    LAUNCHES += KERNELS_PER_CALL.get(name, 1)
    check(rc, name)
    if DEBUG_SYNC and not torch.cuda.is_current_stream_capturing():
        try:
            torch.cuda.synchronize(device)
        except RuntimeError as e:
            raise RuntimeError("%s: asynchronous CUDA fault: %s" % (name, e)) from e


def call_rc(name, device, *args, launches=1):
    """Like call(), but returns the status code instead of raising (for entry points with a documented fallback)."""
    global LAUNCHES
    lib = load()
    with torch.cuda.device(device):
        rc = getattr(lib, name)(*args, stream())
    if rc == 0:
        LAUNCHES += launches
    return rc


def dtype_code(dtype):
    if dtype == torch.float32:
        return NGP_F32
    if dtype == torch.float16:
        return NGP_F16
    raise RuntimeError("unsupported dtype %s (float32 / float16 only)" % dtype)
