"""ctypes binding of libflappy_b200.so (the C ABI of include/flappy_b200.h).

The library is built in-tree by ``build()`` (nvcc, sm_100a only).  There is no
CPU fallback: every product entry point raises if the library is missing or
the call fails.
"""
from __future__ import annotations

import ctypes as C
import glob
import os
import subprocess

_PKG = os.path.dirname(os.path.abspath(__file__))
_CSRC = os.path.join(_PKG, "csrc")
SO_PATH = os.path.join(_PKG, "libflappy_b200.so")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "-shared",
]


class FlappyError(RuntimeError):
    pass


def sources():
    return sorted(glob.glob(os.path.join(_CSRC, "*.cu")))


def needs_build() -> bool:
    if not os.path.exists(SO_PATH):
        return True
    t = os.path.getmtime(SO_PATH)
    deps = sources() + glob.glob(os.path.join(_CSRC, "*.cuh")) + glob.glob(os.path.join(_PKG, "..", "include", "*.h"))
    return any(os.path.getmtime(p) > t for p in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile every .cu under csrc/ for sm_100a (one nvcc per file, in parallel; objects under csrc/build/, rebuilt only
    when the source or a header is newer) and link them into libflappy_b200.so."""
    if not force and not needs_build():
        return SO_PATH
    from concurrent.futures import ThreadPoolExecutor
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    objdir = os.path.join(_CSRC, "build")
    os.makedirs(objdir, exist_ok=True)
    headers = glob.glob(os.path.join(_CSRC, "*.cuh")) + glob.glob(os.path.join(_PKG, "..", "include", "*.h"))
    hdr_t = max(os.path.getmtime(h) for h in headers)
    compile_flags = [f for f in NVCC_FLAGS if f != "-shared"]

    def one(src):
        obj = os.path.join(objdir, os.path.basename(src)[:-3] + ".o")
        if not force and os.path.exists(obj) and os.path.getmtime(obj) > max(os.path.getmtime(src), hdr_t):
            return obj, ""
        cmd = [nvcc] + compile_flags + (["-Xptxas", "-v"] if verbose else []) + ["-c", "-o", obj, src]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise FlappyError(f"nvcc failed on {os.path.basename(src)}:\n" + r.stdout + r.stderr)
        return obj, r.stderr

    with ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 1)) as ex:
        results = list(ex.map(one, sources()))
    if verbose:
        print("".join(log for _, log in results))
    r = subprocess.run([nvcc, "-shared", "-o", SO_PATH] + [o for o, _ in results] + ["-lcuda"], capture_output=True, text=True)
    if r.returncode != 0:
        raise FlappyError("link failed:\n" + r.stdout + r.stderr)
    return SO_PATH


_lib = None

_u8p, _i32p, _f32p, _vp = C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p


class StepSampling(C.Structure):
    """fb_step_sampling (include/flappy_b200.h): the minibatch draw that rides at the head of fb_qnet_step"""
    _fields_ = [("replay", C.c_void_p), ("ring_dev", C.c_void_p), ("act_dev", C.c_void_p), ("rew_dev", C.c_void_p), ("term_dev", C.c_void_p),
                ("t", C.c_longlong), ("batch", C.c_int), ("setsize", C.c_uint32), ("seed", C.c_uint64), ("idx_out_dev", C.c_void_p),
                ("frames_out_dev", C.c_void_p), ("act_out_dev", C.c_void_p), ("rew_out_dev", C.c_void_p), ("term_out_dev", C.c_void_p),
                ("env_out_dev", C.c_void_p), ("k_out_dev", C.c_void_p),
                ("prioritized", C.c_int), ("per_mode", C.c_int), ("beta", C.c_double), ("tree_idx_out_dev", C.c_void_p),
                ("is_weights_out_dev", C.c_void_p), ("prio_out_dev", C.c_void_p), ("is_weights_f32_out_dev", C.c_void_p),
                ("n_step", C.c_int), ("ret_out_dev", C.c_void_p), ("disc_out_dev", C.c_void_p)]


class QnetStepArgs(C.Structure):
    """fb_qnet_step_args (include/flappy_b200.h): one training step of the Q-network"""
    _fields_ = [("variant", C.c_int), ("loss_sum", C.c_int), ("batch", C.c_int), ("global_batch", C.c_int), ("gamma", C.c_double),
                ("params_dev", C.c_void_p), ("target_params_dev", C.c_void_p), ("sampling", C.c_void_p),
                ("frames_dev", C.c_void_p), ("sample_stride", C.c_longlong), ("chan_off_s", C.c_int32 * 4), ("chan_off_next", C.c_int32 * 4),
                ("actions_dev", C.c_void_p), ("rewards_dev", C.c_void_p), ("terminals_dev", C.c_void_p), ("is_weights_dev", C.c_void_p),
                ("grads_dev", C.c_void_p), ("loss_out_dev", C.c_void_p), ("abs_err_out_dev", C.c_void_p), ("q_target_out_dev", C.c_void_p),
                ("m_dev", C.c_void_p), ("v_dev", C.c_void_p), ("lr", C.c_float), ("beta1", C.c_float), ("beta2", C.c_float),
                ("eps", C.c_float), ("grad_scale", C.c_float), ("beta1_power", C.c_float), ("beta2_power", C.c_float)]


_SIGNATURES = {
    "fb_last_error": ([], C.c_char_p),
    "fb_version": ([], C.c_int),
    "fb_assets_load": ([C.c_char_p, C.c_size_t], C.c_int),
    "fb_resize_tables": ([_i32p], C.c_int),
    "fb_env_create": ([C.c_int, C.c_uint64, C.c_uint64, C.POINTER(C.c_void_p)], C.c_int),
    "fb_env_destroy": ([_vp], C.c_int),
    "fb_env_num_envs": ([_vp], C.c_int),
    "fb_env_set_gap_replay": ([_vp, _u8p, C.c_int], C.c_int),
    "fb_env_reset": ([_vp, _vp], C.c_int),
    "fb_env_step": ([_vp, C.c_int, _u8p, _u8p, C.c_int, C.c_int, _f32p, _u8p, _i32p, _vp], C.c_int),
    "fb_env_draw": ([_vp, _u8p, C.c_int, C.c_int, _vp], C.c_int),
    "fb_env_step_random": ([_vp, C.c_int, C.c_uint64, C.c_uint32, C.c_uint32, _u8p, _u8p, C.c_int, C.c_int,
                            _f32p, _u8p, _i32p, _vp], C.c_int),
    "fb_env_step_host": ([_vp, _u8p, _u8p, C.c_int, C.c_int, _f32p, _u8p, _i32p, _vp], C.c_int),
    "fb_env_step_host_submit": ([_vp, _u8p, _u8p, C.c_int, C.c_int, _f32p, _u8p, _i32p, _vp], C.c_int),
    "fb_env_step_host_wait": ([_vp], C.c_int),
    "fb_env_check": ([_vp, _vp], C.c_int),
    "fb_env_export_state": ([_vp, _i32p, _vp], C.c_int),
    "fb_env_import_state": ([_vp, _i32p, _vp], C.c_int),
    "fb_env_obs_exact": ([_vp, _u8p, _vp], C.c_int),
    "fb_render_full": ([_vp, C.c_int, C.c_int, _u8p, _vp], C.c_int),
    "fb_log_episodes": ([_u8p, _i32p, C.c_int, C.c_int, C.c_int, _i32p, _i32p, C.c_int, _vp], C.c_int),
    "fb_qnet_create": ([C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p)], C.c_int),
    "fb_qnet_create_c51": ([C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, C.c_double, C.POINTER(C.c_void_p)], C.c_int),
    "fb_qnet_forward_dist": ([_vp, _f32p, _u8p, C.c_longlong, _i32p, C.c_int, _f32p, _f32p, _vp], C.c_int),
    "fb_debug_c51_project": ([_vp, _f32p, _f32p, _u8p, _vp, _vp, C.c_double, C.c_int, _f32p, _vp], C.c_int),
    "fb_qnet_create_qr": ([C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, C.POINTER(C.c_void_p)], C.c_int),
    "fb_qnet_forward_quantiles": ([_vp, _f32p, _u8p, C.c_longlong, _i32p, C.c_int, _f32p, _f32p, _vp], C.c_int),
    "fb_debug_qr_loss": ([_vp, _f32p, _f32p, _u8p, _f32p, _u8p, _vp, _vp, C.c_double, C.c_int, _f32p, _f32p, _vp], C.c_int),
    "fb_qnet_destroy": ([_vp], C.c_int),
    "fb_qnet_set_precision": ([_vp, C.c_int], C.c_int),
    "fb_qnet_get_precision": ([_vp], C.c_int),
    "fb_qnet_invalidate": ([_vp], C.c_int),
    "fb_qnet_set_per_broadcast": ([_vp, C.c_int], C.c_int),
    "fb_debug_poison_packed": ([_vp, C.c_int, _vp], C.c_int),
    "fb_debug_write_probe": ([_vp, C.c_int, C.c_longlong, C.c_int, C.c_int, _vp], C.c_int),
    "fb_qnet_use_graphs": ([_vp, C.c_int], C.c_int),
    "fb_qnet_param_count": ([_vp], C.c_int),
    "fb_qnet_layout": ([_vp, _i32p], C.c_int),
    "fb_qnet_forward": ([_vp, _f32p, _u8p, C.c_longlong, _i32p, C.c_int, _f32p, _vp], C.c_int),
    "fb_qnet_act": ([_vp, _f32p, _u8p, C.c_longlong, _i32p, C.c_int, C.c_double, C.c_uint64, C.c_uint64, _vp, _f32p, _u8p, _vp], C.c_int),
    "fb_qnet_adam": ([_vp, _f32p, _f32p, _f32p, _f32p, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, _vp], C.c_int),
    "fb_qnet_step": ([_vp, _vp, _vp], C.c_int),
    "fb_qnet_sync_target": ([_vp, _f32p, _f32p, _vp], C.c_int),
    "fb_noisy_layout": ([_vp, _i32p], C.c_int),
    "fb_noisy_draw": ([_vp, C.c_uint64, C.c_int, C.c_uint64, _f32p, _vp], C.c_int),
    "fb_noisy_weights": ([_vp, _f32p, _f32p, _f32p, _f32p, _vp], C.c_int),
    "fb_qnet_noisy_adam": ([_vp, _f32p, _f32p, _f32p, _f32p, _f32p, _f32p, _f32p, _f32p, C.c_float, C.c_float, C.c_float, C.c_float,
                            C.c_float, _vp], C.c_int),
    "fb_debug_struct_layout": ([C.c_int, _i32p, C.c_int], C.c_int),
    "fb_debug_step_sampling_layout": ([_i32p, C.c_int], C.c_int),
    "fb_dist_debug_stamps": ([_vp, _vp], C.c_int),
    "fb_dist_create": ([C.c_int, C.c_int, C.c_longlong, C.POINTER(C.c_void_p)], C.c_int),
    "fb_dist_destroy": ([_vp], C.c_int),
    "fb_dist_handle_bytes": ([], C.c_int),
    "fb_dist_set_two_shot": ([_vp, C.c_int], C.c_int),
    "fb_dist_debug_mask": ([_vp, C.c_int], C.c_int),
    "fb_dist_handles": ([_vp, C.c_char_p], C.c_int),
    "fb_dist_connect": ([_vp, C.c_char_p], C.c_int),
    "fb_dist_connect_local": ([_vp, C.c_int, _vp], C.c_int),
    "fb_dist_grads": ([_vp, C.c_int, C.POINTER(C.c_void_p)], C.c_int),
    "fb_dist_parity": ([_vp], C.c_int),
    "fb_dist_advance": ([_vp], C.c_int),
    "fb_qnet_attach_exchange": ([_vp, _vp], C.c_int),
    "fb_dist_adam": ([_vp, _vp, _f32p, _f32p, _f32p, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float, _f32p, C.c_int, _vp], C.c_int),
    "fb_replay_create": ([C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p)], C.c_int),
    "fb_replay_destroy": ([_vp], C.c_int),
    "fb_replay_sample_uniform": ([_vp, C.c_longlong, C.c_int, C.c_uint32, C.c_uint64, _i32p, _vp], C.c_int),
    "fb_replay_gather": ([_vp, _u8p, _u8p, _f32p, _u8p, C.c_longlong, C.c_int, _i32p, C.c_int, _u8p, _u8p, _f32p, _u8p, _i32p, _i32p, _vp], C.c_int),
    "fb_per_store": ([_vp, C.c_longlong, C.c_int, _vp], C.c_int),
    "fb_per_sample": ([_vp, C.c_int, C.c_double, C.c_uint64, _i32p, _i32p, _vp, _vp, _f32p, _vp], C.c_int),
    "fb_per_update": ([_vp, _i32p, _f32p, _vp, C.c_int, C.c_int, _vp], C.c_int),
    "fb_per_tree_copy": ([_vp, _vp, C.c_int, _vp], C.c_int),
    "fb_per_aux_tree_copy": ([_vp, C.c_int, _vp, C.c_int, _vp], C.c_int),
    "fb_per_min_root": ([_vp, _vp, _vp], C.c_int),
    "fb_per_set_global_min": ([_vp, _vp], C.c_int),
    "fb_replay_rng_pos": ([_vp, _vp, C.c_int, _vp], C.c_int),
    "fb_debug_assets_load_host": ([C.c_char_p, C.c_size_t], C.c_int),
    "fb_debug_host_reset": ([_i32p, _u8p, C.c_int, C.c_uint64, C.c_uint64], C.c_int),
    "fb_debug_host_step": ([_i32p, C.c_int, _u8p, C.c_int, C.c_uint64, C.c_uint64, _f32p, _u8p, _i32p], C.c_int),
    "fb_debug_host_obs": ([_i32p, C.c_int, _u8p], C.c_int),
    "fb_debug_host_mixed": ([_i32p], C.c_int),
    "fb_debug_tc_mma_rate": ([C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _vp, _vp], C.c_int),
    "fb_debug_tc_kernel": ([_vp, C.c_int, C.c_int, C.c_int, _f32p, _vp], C.c_int),
    "fb_debug_tc_separate_kernels": ([_vp, C.c_int], C.c_int),
    "fb_debug_tc_slab": ([C.c_int, C.c_int, _vp, _vp, _f32p, _vp], C.c_int),
    "fb_debug_tc_gemm": ([C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _vp, _vp, _f32p, _vp, _vp], C.c_int),
}


def declared_symbols():
    return sorted(_SIGNATURES)


def lib():
    """The loaded library; builds it if the sources are newer.  Raises when it cannot be had."""
    global _lib
    if _lib is None:
        if needs_build():
            build()
        L = C.CDLL(SO_PATH)
        for name, (argtypes, restype) in _SIGNATURES.items():
            fn = getattr(L, name)            # AttributeError if the header and the library disagree
            fn.argtypes = argtypes
            fn.restype = restype
        _lib = L
    return _lib


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = lib().fb_last_error().decode("utf-8", "replace")
        if rc == -4:
            raise ValueError(msg or "Multiple input actions!")     # wrapped_flappy_bird.py:99-100
        raise FlappyError(f"{what} failed ({rc}): {msg}")


_assets_device = None


def ensure_assets(assets_dir: str | None = None, device_index: int = 0):
    """fb_assets_load once per process/device (flappy_bird_utils.load())."""
    global _assets_device
    key = (assets_dir, device_index)
    if _assets_device == key:
        return
    from .assets import load_blob
    blob = load_blob(assets_dir)
    check(lib().fb_assets_load(blob, len(blob)), "fb_assets_load")
    _assets_device = key
