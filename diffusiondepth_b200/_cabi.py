"""ctypes binding of libddengine.so (include/dd_engine.h).  There is no fallback: if the shared library
is missing or does not export the ABI, importing the engine raises."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None


class EngineError(RuntimeError):
    """Raised for any non-zero status coming back across the C ABI."""


class DDConfig(C.Structure):
    _fields_ = [("abi_version", C.c_int32), ("variant", C.c_int32), ("batch", C.c_int32),
                ("latent_h", C.c_int32), ("latent_w", C.c_int32), ("cond_h", C.c_int32),
                ("cond_w", C.c_int32), ("num_inference_steps", C.c_int32), ("device", C.c_int32),
                ("flags", C.c_int32)]


class DDProducerConfig(C.Structure):
    _fields_ = [("num_levels", C.c_int32), ("channels", C.c_int32 * 4), ("heights", C.c_int32 * 4),
                ("widths", C.c_int32 * 4), ("has_neck", C.c_int32)]


class DDBackboneConfig(C.Structure):
    _fields_ = [("kind", C.c_int32), ("embed_dims", C.c_int32), ("depths", C.c_int32 * 4),
                ("num_heads", C.c_int32 * 4), ("window", C.c_int32), ("height", C.c_int32), ("width", C.c_int32),
                ("mp_dims", C.c_int32 * 4), ("mp_paths", C.c_int32 * 4), ("mlp_ratio", C.c_int32)]


ABI_VERSION = 1
VARIANT_RES, VARIANT_SWIN = 0, 1
FLAG_CUDA_GRAPH, FLAG_SIMT_CONV, FLAG_CHECK_RANGE, FLAG_HALO_CONV, FLAG_SWAP_NARROW, FLAG_PAIR_WIDE = 1, 2, 4, 8, 16, 32
FLAG_STEP_DECODE, FLAG_FP8_CORR, FLAG_STOCHASTIC = 64, 128, 256
STATUS = {0: "DD_OK", 1: "DD_ERR_INVALID", 2: "DD_ERR_CUDA", 3: "DD_ERR_UNSUPPORTED", 4: "DD_ERR_RANGE"}

# name -> (restype, argtypes); every symbol include/dd_engine.h declares
SIGNATURES = {
    "dd_abi_version": (C.c_int, []),
    "dd_last_error": (C.c_char_p, []),
    "dd_create": (C.c_int, [C.POINTER(DDConfig), C.POINTER(C.c_void_p)]),
    "dd_destroy": (C.c_int, [C.c_void_p]),
    "dd_set_weight": (C.c_int, [C.c_void_p, C.c_char_p, C.c_void_p, C.POINTER(C.c_int64), C.c_int32]),
    "dd_finalize_weights": (C.c_int, [C.c_void_p, C.c_void_p]),
    "dd_set_schedule": (C.c_int, [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_double),
                                  C.POINTER(C.c_double), C.c_int32]),
    "dd_set_schedule_eta": (C.c_int, [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_double), C.POINTER(C.c_double),
                                      C.POINTER(C.c_double), C.c_int32]),
    "dd_workspace_bytes": (C.c_size_t, [C.c_void_p]),
    "dd_enable_producers": (C.c_int, [C.c_void_p, C.POINTER(DDProducerConfig)]),
    "dd_enable_backbone": (C.c_int, [C.c_void_p, C.POINTER(DDBackboneConfig)]),
    "dd_run_backbone": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p), C.c_void_p, C.c_size_t, C.c_void_p]),
    "dd_build_condition": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.c_void_p, C.c_void_p, C.c_size_t,
                                     C.c_void_p]),
    "dd_denoise_decode": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                    C.c_void_p, C.c_size_t, C.c_void_p]),
    "dd_denoise_decode_steps": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                          C.c_void_p, C.c_size_t, C.c_void_p]),
    "dd_denoise_decode_stochastic": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                               C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "dd_denoiser_forward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_int64), C.c_void_p,
                                      C.c_void_p, C.c_size_t, C.c_void_p]),
    "dd_decode": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "dd_encode": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]),
    "dd_last_launch_count": (C.c_int64, [C.c_void_p]),
    "dd_poll_status": (C.c_int, [C.c_void_p, C.c_void_p]),
    "dd_conv3x3": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                             C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_size_t, C.c_void_p]),
    "dd_conv3x3_workspace_bytes": (C.c_size_t, [C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32]),
    "dd_bench_gemm": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_float)]),
    "dd_bench_conv": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_float), C.c_void_p,
                                C.c_size_t, C.c_void_p]),
}


def lib_path() -> str:
    return os.environ.get("DD_ENGINE_LIB", os.path.join(_HERE, "libddengine.so"))


def load_library():
    """dlopen libddengine.so and type every entry point; raises EngineError if anything is missing."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = lib_path()
    if not os.path.exists(path):
        raise EngineError(
            f"{path} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc -gencode arch=compute_100a,code=sm_100a). There is no CPU/PyTorch fallback.")
    lib = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError as e:  # pragma: no cover
            raise EngineError(f"{path} does not export {name}") from e
        fn.restype, fn.argtypes = res, args
    if lib.dd_abi_version() != ABI_VERSION:
        raise EngineError(f"ABI mismatch: library {lib.dd_abi_version()} vs binding {ABI_VERSION}")
    _LIB = lib
    return lib


def check(status: int):
    if status != 0:
        msg = load_library().dd_last_error().decode("utf-8", "replace")
        raise EngineError(f"{STATUS.get(status, status)}: {msg}")
