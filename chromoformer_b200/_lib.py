"""ctypes binding of ``libchromo_b200.so`` (C ABI in ``include/chromoformer_b200.h``).

There is deliberately no fallback: if the shared library is missing or a call
fails, a :class:`ChromoLibError` is raised.  The only thing PyTorch provides
here is device memory and the current CUDA stream.
"""
import ctypes
import os
from ctypes import (POINTER, Structure, c_char_p, c_float, c_int32, c_int64, c_uint8, c_uint16,
                    c_void_p)

MAX_RES = 4
MAX_LAYERS = 8
F_TRAINING = 1
F_BF16 = 2
F_PACKED = 4
F_DENSE = 64
F_BWD_HEAD_REG = 16
F_BWD_REST = 32
F_FREQ_GRAD = 128

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libchromo_b200.so")


class ChromoLibError(RuntimeError):
    pass


class Config(Structure):
    """``chromo_config_t`` — mirrors configs/default.yaml of the reference."""
    _fields_ = [
        ("n_feats", c_int32), ("d_emb", c_int32), ("d_head", c_int32), ("n_out", c_int32),
        ("n_res", c_int32), ("i_max", c_int32),
        ("embed_layers", c_int32), ("embed_heads", c_int32), ("embed_d_model", c_int32), ("embed_d_ff", c_int32),
        ("pw_layers", c_int32), ("pw_heads", c_int32), ("pw_d_model", c_int32), ("pw_d_ff", c_int32),
        ("reg_layers", c_int32), ("reg_heads", c_int32), ("reg_d_model", c_int32), ("reg_d_ff", c_int32),
        ("n_bins", c_int32 * MAX_RES),
    ]


class Batch(Structure):
    """``chromo_batch_t`` — raw device pointers of one batch of genes."""
    _fields_ = [
        ("batch", c_int32),
        ("x_p", c_void_p * MAX_RES),
        ("x_pcre", c_void_p * MAX_RES),
        ("mask_p", c_void_p * MAX_RES),
        ("mask_p_stride", c_int64 * MAX_RES),
        ("mask_p_row_offset", c_int64 * MAX_RES),
        ("mask_pcre", c_void_p * MAX_RES),
        ("mask_pcre_stride", c_int64 * MAX_RES),
        ("mask_pcre_row_offset", c_int64 * MAX_RES),
        ("imask", c_void_p * MAX_RES),
        ("freq", c_void_p),
        ("pos_enc", c_void_p * MAX_RES),
    ]


class InputGrads(Structure):
    """``chromo_input_grads_t`` — where chromo_backward_inputs writes the feature gradients (NULL: not wanted) and,
    with ``F_FREQ_GRAD``, the interaction_freq gradient."""
    _fields_ = [
        ("x_p", c_void_p * MAX_RES),
        ("x_pcre", c_void_p * MAX_RES),
        ("freq", c_void_p),
    ]


class Region(Structure):
    """``chromo_region_t``"""
    _fields_ = [("offset", c_int64), ("length", c_int32), ("start", c_int32), ("width", c_int32),
                ("flip", c_int32)]


EXPORTS = {
    # name: (restype, argtypes)
    "chromo_abi_version": (c_int32, []),
    "chromo_last_error": (c_char_p, []),
    "chromo_param_total": (c_int64, [POINTER(Config)]),
    "chromo_param_active": (c_int64, [POINTER(Config)]),
    "chromo_param_count": (c_int32, [POINTER(Config)]),
    "chromo_param_info": (c_int64, [POINTER(Config), c_int32, c_char_p, c_int32, POINTER(c_int64)]),
    "chromo_workspace_floats": (c_int64, [POINTER(Config), c_int32, c_int32]),
    "chromo_forward": (c_int32, [POINTER(Config), c_void_p, POINTER(Batch), c_void_p, c_void_p, c_int64,
                                 c_int32, c_void_p]),
    "chromo_pcre_deletion_workspace_floats": (c_int64, [POINTER(Config), c_int32, c_int32]),
    "chromo_pcre_deletion": (c_int32, [POINTER(Config), c_void_p, POINTER(Batch), c_void_p, c_void_p, c_void_p, c_void_p,
                                       c_int64, c_int32, c_void_p]),
    "chromo_pcre_subsets_workspace_floats": (c_int64, [POINTER(Config), c_int32, c_int32, c_int32]),
    "chromo_pcre_subsets": (c_int32, [POINTER(Config), c_void_p, POINTER(Batch), c_void_p, c_void_p, c_int32, c_void_p,
                                      c_void_p, c_void_p, c_int64, c_int32, c_void_p]),
    "chromo_freq_edits_workspace_floats": (c_int64, [POINTER(Config), c_int32, c_int32, c_int32]),
    "chromo_freq_edits": (c_int32, [POINTER(Config), c_void_p, POINTER(Batch), c_void_p, c_void_p, c_int32, c_void_p,
                                    c_void_p, c_void_p, c_int64, c_int32, c_void_p]),
    "chromo_pcre_occlusion_workspace_floats": (c_int64, [POINTER(Config), c_int32, c_int32, c_int32]),
    "chromo_pcre_occlusion": (c_int32, [POINTER(Config), c_void_p, POINTER(Batch), c_int32, c_void_p, c_void_p, c_void_p,
                                        c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int32, c_void_p]),
    "chromo_regulation_layer": (c_int32, [POINTER(Config), c_void_p, c_int32, c_void_p, c_void_p, c_int64,
                                          POINTER(c_void_p), c_void_p, c_int32, c_void_p, c_int64, c_int32, c_void_p]),
    "chromo_linear": (c_int32, [c_void_p, c_void_p, c_void_p, c_void_p, c_int32, c_int32, c_int32, c_int32, c_int32,
                                c_int64, c_int64, c_int64, c_int64, c_int32, c_void_p]),
    "chromo_single_query_attention": (c_int32, [c_int32, c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                                c_float, c_void_p, c_void_p, c_int64, c_void_p]),
    "chromo_pack_linear_weight": (c_int32, [c_void_p, c_void_p, c_int32, c_int32, c_int32, c_int64, c_void_p]),
    "chromo_launch_counter": (c_int64, [c_int32]),
    "chromo_debug_trace": (c_int32, [c_void_p]),
    "chromo_backward": (c_int32, [POINTER(Config), c_void_p, POINTER(Batch), c_void_p, c_void_p, c_void_p,
                                  c_int64, c_int32, c_void_p]),
    "chromo_backward_inputs": (c_int32, [POINTER(Config), c_void_p, POINTER(Batch), c_void_p, c_void_p,
                                         POINTER(InputGrads), c_void_p, c_int64, c_int32, c_void_p]),
    "chromo_matmul": (c_int32, [c_void_p, c_int64, c_int32, c_void_p, c_int64, c_int32, c_void_p, c_int64, c_int32, c_int32,
                                c_int32, c_int32, c_int32, c_void_p]),
    "chromo_mse_loss": (c_int32, [c_void_p, c_void_p, c_int32, c_float, c_void_p, c_void_p, c_void_p]),
    "chromo_ce_loss": (c_int32, [c_void_p, c_void_p, c_int32, c_int32, c_float, c_void_p, c_void_p, c_void_p]),
    "chromo_clf_metrics": (c_int32, [c_void_p, c_void_p, c_int32, c_int32, c_void_p, c_void_p, c_void_p, c_void_p]),
    "chromo_reg_metrics": (c_int32, [c_void_p, c_void_p, c_int32, c_void_p, c_void_p]),
    "chromo_adamw": (c_int32, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_float, c_float, c_float,
                               c_float, c_float, c_int32, c_float, c_void_p]),
    "chromo_unpack_wire": (c_int32, [c_int32, POINTER(c_void_p), POINTER(c_void_p), POINTER(c_int64), c_int32,
                                     POINTER(c_void_p), POINTER(c_void_p), POINTER(c_int32), POINTER(c_int32), c_void_p]),
    "chromo_unpack_compact": (c_int32, [c_int32, POINTER(c_void_p), POINTER(c_void_p), POINTER(c_void_p), POINTER(c_int32),
                                        POINTER(c_void_p), POINTER(c_int32), POINTER(c_int32), c_int32, c_void_p]),
    "chromo_unpack_sparse": (c_int32, [c_int32, POINTER(c_void_p), POINTER(c_void_p), POINTER(c_void_p), POINTER(c_int32),
                                       POINTER(c_void_p), POINTER(c_int64), c_void_p]),
    "chromo_bin_regions": (c_int32, [c_void_p, c_void_p, c_int32, c_int32, c_int32, POINTER(c_int32),
                                     POINTER(c_int32), POINTER(c_void_p), c_void_p, c_void_p]),
}

_lib = None


def load():
    """Load the shared library once; raise loudly if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ChromoLibError(
            f"{LIB_PATH} not found - build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `make -C chromoformer_b200/csrc`. There is no CPU/PyTorch fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (restype, argtypes) in EXPORTS.items():
        fn = getattr(lib, name)      # AttributeError if the symbol is missing
        fn.restype = restype
        fn.argtypes = argtypes
    if lib.chromo_abi_version() != 1:
        raise ChromoLibError("libchromo_b200.so ABI version mismatch")
    _lib = lib
    return lib


def check(rc, what=""):
    if rc < 0:
        msg = load().chromo_last_error().decode()
        raise ChromoLibError(f"{what or 'libchromo_b200'} failed ({rc}): {msg}")
    return rc


def param_table(cfg):
    """{name: (offset, numel)} of the flat parameter buffer, straight from the library."""
    lib = load()
    n = check(lib.chromo_param_count(ctypes.byref(cfg)), "chromo_param_count")
    buf = ctypes.create_string_buffer(256)
    numel = c_int64()
    out = {}
    for i in range(n):
        off = check(lib.chromo_param_info(ctypes.byref(cfg), i, buf, 256, ctypes.byref(numel)), "chromo_param_info")
        out[buf.value.decode()] = (int(off), int(numel.value))
    return out
