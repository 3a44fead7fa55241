"""Builds (nvcc, sm_100a) and loads the C-ABI library declared in include/bitswap_b200.h.

There is deliberately no CPU fallback: if the shared library is missing or fails to
load, every product entry point raises."""
import ctypes
import glob
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
_CSRC = os.path.join(_HERE, "csrc")
SO_PATH = os.path.join(_HERE, "libbitswap_b200.so")
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC"]

_lib = None


def _nvcc():
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if c and (os.path.isabs(c) and os.path.exists(c) or not os.path.isabs(c)):
            return c
    return "nvcc"


def build(force=False, verbose=False):
    """Compile every csrc/*.cu into libbitswap_b200.so (in-tree, so it travels with gpurun)."""
    srcs = sorted(glob.glob(os.path.join(_CSRC, "*.cu")))
    deps = srcs + glob.glob(os.path.join(_CSRC, "*.cuh")) + [os.path.join(_HERE, "..", "include", "bitswap_b200.h")]
    if not force and os.path.exists(SO_PATH) and all(os.path.getmtime(SO_PATH) >= os.path.getmtime(d) for d in deps):
        return SO_PATH
    objdir = os.path.join(_HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    objs, procs = [], []
    for s in srcs:
        o = os.path.join(objdir, os.path.basename(s)[:-3] + ".o")
        objs.append(o)
        if force or not os.path.exists(o) or any(os.path.getmtime(o) < os.path.getmtime(d) for d in [s] + deps[len(srcs):]):
            cmd = [_nvcc()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", s, "-o", o]
            procs.append((s, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for s, p in procs:
        out, _ = p.communicate()
        if verbose and out:
            print(out)
        if p.returncode:
            raise RuntimeError(f"nvcc failed on {s}:\n{out}")
    link = [_nvcc(), "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", SO_PATH] + objs
    r = subprocess.run(link, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode:
        raise RuntimeError("link failed:\n" + r.stdout)
    return SO_PATH


class BswError(RuntimeError):
    pass


STATUS = {0: "BSW_OK", 1: "BSW_E_UNDERFLOW", 2: "BSW_E_OVERFLOW", 3: "BSW_E_BADTABLE", 4: "BSW_E_INVALID", 5: "BSW_E_CUDA"}


def check(rc):
    if rc != 0:
        msg = lib().bsw_last_error().decode()
        raise BswError(f"{STATUS.get(rc, rc)}: {msg}")


def lib():
    """The loaded library.  Raises if it has not been built (run __graft_entry__.build())."""
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            raise BswError(f"{SO_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(there is no CPU fallback)")
        L = ctypes.CDLL(SO_PATH)
        L.bsw_last_error.restype = ctypes.c_char_p
        L.bsw_streams_capacity.restype = ctypes.c_int64
        if hasattr(L, "bsw_logistic_scratch_bytes"):
            L.bsw_logistic_scratch_bytes.restype = ctypes.c_int64
        if hasattr(L, "bsw_codec_last_launches"):
            L.bsw_codec_last_launches.restype = ctypes.c_int64
        _set_argtypes(L)
        _lib = L
    return _lib


def _set_argtypes(L):
    P, I, L64, U64 = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_uint64
    PP = ctypes.POINTER(ctypes.c_void_p)
    sig = {
        "bsw_streams_create": [PP, I, L64],
        "bsw_streams_destroy": [P],
        "bsw_streams_count": [P],
        "bsw_streams_capacity": [P],
        "bsw_streams_import": [P, I, I, P, P, P],
        "bsw_streams_fill": [P, P, L64, U64],
        "bsw_streams_sizes": [P, P, P, P],
        "bsw_streams_export": [P, I, I, P, P],
        "bsw_streams_min_words": [P, P],
        "bsw_streams_rest_words": [P, P],
        "bsw_streams_device_ptrs": [P, PP, PP, PP, PP],
        "bsw_streams_pack": [P, I, I, P, P, P, P],
        "bsw_streams_unpack": [P, I, I, P, P, P, P],
        "bsw_streams_pack_trimmed": [P, I, I, P, P, P, P, P],
        "bsw_streams_unpack_trimmed": [P, I, I, P, P, P, P, P],
        "bsw_streams_total_words": [P, P, P],
        "bsw_ans_tables": [P, L64, I, I, I, P, P, P, P],
        "bsw_ans_push": [P, I, I, P, P, L64, L64, P, L64, I, I, P],
        "bsw_ans_pop": [P, I, I, P, P, L64, L64, P, L64, I, I, P],
        "bsw_logistic_pmfs": [P, L64, P, P, L64, L64, I, P, P],
        "bsw_logistic_tables": [P, L64, P, P, L64, L64, I, I, I, P, P, P],
        "bsw_logistic_push": [P, I, I, P, L64, P, L64, P, L64, P, L64, I, I, I, P],
        "bsw_logistic_pop": [P, I, I, P, L64, P, L64, P, L64, P, L64, I, I, I, P],
        "bsw_logistic_scratch_bytes": [I, L64, I, I],
        "bsw_set_rows_mode": [I],
        "bsw_bins_level_is_uniform": [P, I],
        "bsw_rows6_set_verify": [I],
        "bsw_rows6_set_lanes_per_row": [I],
        "bsw_set_conv_mode": [I],
        "bsw_rows6_verify_read": [P],
        "bsw_logistic_push_2p": [P, I, I, P, L64, P, L64, P, L64, P, L64, I, I, I, P, L64, P],
        "bsw_logistic_pop_2p": [P, I, I, P, L64, P, L64, P, L64, P, L64, I, I, I, P, L64, P],
        "bsw_bins_create": [PP, I, I, I, I, P, P],
        "bsw_bins_destroy": [P],
        "bsw_bins_device_ptrs": [P, I, PP, PP, PP],
        "bsw_gather_zcentres": [P, I, P, P, L64, P],
        "bsw_gather_xcentres": [P, P, L64, P],
        "bsw_model_create": [PP, P],
        "bsw_model_destroy": [P],
        "bsw_model_load_conv": [P, ctypes.c_char_p, P, P, P, I, I, I, I],
        "bsw_model_load_gen_std": [P, P],
        "bsw_model_finalize": [P],
        "bsw_vae_infer": [P, I, P, L64, P, P, P],
        "bsw_vae_generate": [P, I, P, L64, P, P, I, P],
        "bsw_codec_create": [PP, P, P, I],
        "bsw_codec_destroy": [P],
        "bsw_codec_encode": [P, P, I, I, P, I, P],
        "bsw_codec_decode": [P, P, I, I, P, I, P],
        "bsw_codec_encode_ext": [P, P, I, I, P, P, I, P],
        "bsw_codec_decode_ext": [P, P, I, I, P, P, I, P],
        "bsw_codec_last_launches": [P],
        "bsw_codec_profile": [P, I, P, P],
        "bsw_codec_set_two_phase": [P, I],
        "bsw_codec_set_dual_stream": [P, I],
        "bsw_discretize_reset": [P, I, P],
        "bsw_discretize_sample": [P, P, L64, P, ctypes.c_float, P, P, L64, I, P],
        "bsw_discretize_fold": [P, P, L64, I, P],
        "bsw_discretize_edges": [P, I, I, P, L64, P, L64, P],
        "bsw_selftest_cdf": [L64, U64, P, P],
        "bsw_selftest_cdf_apx": [L64, U64, P],
    }
    for name, args in sig.items():
        fn = getattr(L, name, None)
        if fn is not None:
            fn.argtypes = args


EXPORTS = ["bsw_last_error", "bsw_version", "bsw_has_tensor_cores", "bsw_measure_fp64_peak", "bsw_selftest_cdf", "bsw_selftest_cdf_apx", "bsw_streams_create", "bsw_streams_destroy", "bsw_streams_count",
           "bsw_streams_capacity", "bsw_streams_import", "bsw_streams_fill", "bsw_streams_sizes", "bsw_streams_min_words", "bsw_streams_rest_words", "bsw_streams_export",
           "bsw_streams_device_ptrs", "bsw_streams_pack", "bsw_streams_unpack", "bsw_streams_pack_trimmed", "bsw_streams_unpack_trimmed", "bsw_streams_total_words", "bsw_ans_tables", "bsw_ans_push", "bsw_ans_pop",
           "bsw_logistic_pmfs", "bsw_logistic_tables", "bsw_logistic_push", "bsw_logistic_pop", "bsw_logistic_scratch_bytes", "bsw_set_rows_mode", "bsw_bins_level_is_uniform", "bsw_rows6_set_verify", "bsw_rows6_verify_read", "bsw_rows6_set_lanes_per_row", "bsw_set_conv_mode", "bsw_logistic_push_2p",
           "bsw_logistic_pop_2p", "bsw_bins_create",
           "bsw_bins_destroy", "bsw_bins_device_ptrs", "bsw_gather_zcentres", "bsw_gather_xcentres",
           "bsw_model_create", "bsw_model_destroy", "bsw_model_load_conv", "bsw_model_load_gen_std",
           "bsw_model_finalize", "bsw_vae_infer", "bsw_vae_generate", "bsw_codec_create", "bsw_codec_destroy",
           "bsw_codec_encode", "bsw_codec_decode", "bsw_codec_encode_ext", "bsw_codec_decode_ext", "bsw_codec_last_launches", "bsw_codec_profile", "bsw_codec_set_two_phase", "bsw_codec_set_dual_stream",
           "bsw_discretize_reset", "bsw_discretize_sample", "bsw_discretize_fold", "bsw_discretize_edges"]


def device_index(device=None):
    """CUDA device ordinal of `device` (torch.device / "cuda:N" / int / None = the current device)."""
    import torch
    if device is None:
        return torch.cuda.current_device()
    if isinstance(device, int):
        return device
    d = torch.device(device)
    if d.type != "cuda":
        raise BswError(f"bitswap_b200 needs a CUDA device, got {device!r} (there is no CPU fallback)")
    return torch.cuda.current_device() if d.index is None else d.index


def on_device(index):
    """Context manager: every library object allocates and launches on the device it was created for, whatever the
    caller's current device is (the reference scripts pass device=f"cuda:{gpu}" without ever calling set_device)."""
    import torch
    return torch.cuda.device(index)


def cuda_stream_ptr():
    """torch's current CUDA stream as a void* for the `stream` argument of the C ABI."""
    import torch
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def measure_fp64_peak():
    """Peak float64 FMA lanes per second on the current device."""
    v = ctypes.c_double()
    check(lib().bsw_measure_fp64_peak(ctypes.byref(v)))
    return v.value


def has_tensor_core_path():
    return bool(lib().bsw_has_tensor_cores())
