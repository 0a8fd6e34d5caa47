"""ctypes loader for libvsrdec.so.  There is deliberately no fallback: if the CUDA extension is
missing the import of the product path fails loudly."""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

c_i32, c_i64, c_vp, c_f = ctypes.c_int32, ctypes.c_int64, ctypes.c_void_p, ctypes.c_float


class VsrError(RuntimeError):
    pass


class VsrDims(ctypes.Structure):
    _fields_ = [(n, c_i32) for n in ("seq_len", "vocab_size", "bos_idx", "det_feat_size",
                                      "input_encoding_size", "rnn_size", "att_size",
                                      "h2_first_lstm", "img_second_lstm")]


class VsrSortDims(ctypes.Structure):
    _fields_ = [(n, c_i32) for n in ("n_roles", "n_verbs", "d_model", "d_ff", "n_heads", "n_layers", "max_len", "add_fc")]


class VsrTrace(ctypes.Structure):
    _fields_ = [("step_out", c_vp), ("step_gate", c_vp), ("forced_beam", c_vp),
                ("forced_word", c_vp), ("forced_gate", c_vp)]


class VsrSampleParams(ctypes.Structure):
    _fields_ = [("seed", ctypes.c_uint64), ("n", c_i32), ("temperature", c_f), ("top_k", c_i32), ("top_p", c_f),
                ("use_verbs", c_i32), ("gt", c_i32)]


# every symbol include/vsrdec.h declares: name -> (restype, argtypes)
EXPORTED_SYMBOLS = {
    "vsr_last_error": (ctypes.c_char_p, []),
    "vsr_abi_version": (c_i32, []),
    "vsr_create": (ctypes.c_int, [ctypes.POINTER(VsrDims), ctypes.POINTER(c_vp), ctypes.POINTER(c_vp)]),
    "vsr_load_weights": (ctypes.c_int, [c_vp, ctypes.POINTER(c_vp), c_vp]),
    "vsr_destroy": (None, [c_vp]),
    "vsr_set_verb_table": (ctypes.c_int, [c_vp, ctypes.POINTER(c_i64), ctypes.POINTER(c_i32),
                                          ctypes.POINTER(c_i32), c_i32]),
    "vsr_prologue": (ctypes.c_int, [c_vp, c_vp, c_i64, c_i32, c_vp, c_i32, c_i32, c_i32, c_vp, c_i32, c_vp]),
    "vsr_prologue_indexed": (ctypes.c_int, [c_vp, c_vp, c_i64, c_i32, c_vp, c_i32, c_i32, c_i32, c_vp, c_i32, c_vp]),
    "vsr_prologue_ex": (ctypes.c_int, [c_vp, c_vp, c_i64, c_i32, c_vp, c_i32, c_i32, c_i32, c_i32, c_vp, c_i32, c_vp]),
    "vsr_prologue_indexed_ex": (ctypes.c_int, [c_vp, c_vp, c_i64, c_i32, c_vp, c_i32, c_i32, c_i32, c_i32, c_vp, c_i32,
                                               c_vp]),
    "vsr_step": (ctypes.c_int, [c_vp] + [c_vp] * 6 + [c_i32, c_i32] + [c_vp] * 6 + [c_vp]),
    "vsr_beam_search": (ctypes.c_int, [c_vp, c_i32, c_i32, ctypes.POINTER(c_i64), c_i32, c_i32,
                                       c_vp, c_vp, c_vp, c_vp, ctypes.POINTER(VsrTrace), c_vp]),
    "vsr_get_history": (ctypes.c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "vsr_forward_teacher": (ctypes.c_int, [c_vp, c_vp, c_i32, c_vp, c_vp, c_vp]),
    "vsr_greedy": (ctypes.c_int, [c_vp, c_vp, c_vp, c_vp]),
    "vsr_sample": (ctypes.c_int, [c_vp, ctypes.c_uint64, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "vsr_sample_ex": (ctypes.c_int, [c_vp, ctypes.POINTER(VsrSampleParams), c_vp, c_vp, c_vp, c_vp, c_vp]),
    "vsr_set_attention_capture": (ctypes.c_int, [c_vp, c_i32]),
    "vsr_get_attention": (ctypes.c_int, [c_vp, c_vp, c_vp, c_vp]),
    "vsr_set_no_repeat_ngram": (ctypes.c_int, [c_vp, c_i32]),
    "vsr_set_beam_diversity": (ctypes.c_int, [c_vp, c_i32, c_f]),
    "vsr_launch_count": (c_i64, [c_vp]),
    "vsr_gemm_kind": (ctypes.c_char_p, [c_vp]),
    "vsr_set_profiling": (ctypes.c_int, [c_vp, c_i32]),
    "vsr_get_phase_times": (ctypes.c_int, [c_vp, ctypes.POINTER(ctypes.c_char_p), ctypes.POINTER(c_f),
                                           ctypes.POINTER(c_i32), c_i32]),
    "vsr_get_step_times": (ctypes.c_int, [c_vp, ctypes.POINTER(c_f), c_i32]),
    "vsr_ssp_create": (ctypes.c_int, [ctypes.POINTER(c_vp), c_i32, c_i32, c_f, ctypes.POINTER(c_vp)]),
    "vsr_ssp_load_weights": (ctypes.c_int, [c_vp, ctypes.POINTER(c_vp), c_vp]),
    "vsr_ssp_destroy": (None, [c_vp]),
    "vsr_ssp_forward": (ctypes.c_int, [c_vp, c_vp, c_i32, c_vp, c_vp, c_vp]),
    "vsr_preorder_begin": (ctypes.c_int, [c_vp, c_vp, c_vp, c_i32, c_i32, c_i32, c_i32, c_i32, c_i32, ctypes.POINTER(c_vp),
                                          ctypes.POINTER(c_i32), ctypes.POINTER(c_i32), ctypes.POINTER(c_i32)]),
    "vsr_preorder_fill": (ctypes.c_int, [c_vp, c_vp, c_vp, c_i32, c_vp, c_vp]),
    "vsr_preorder_end": (ctypes.c_int, [c_vp, c_vp, c_i32, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "vsr_preorder_free": (None, [c_vp]),
    "vsr_sort_create": (ctypes.c_int, [ctypes.POINTER(VsrSortDims), ctypes.POINTER(c_vp), c_i32, ctypes.POINTER(c_vp)]),
    "vsr_sort_load_weights": (ctypes.c_int, [c_vp, ctypes.POINTER(c_vp), c_i32, c_vp]),
    "vsr_sort_destroy": (None, [c_vp]),
    "vsr_sort_generate": (ctypes.c_int, [c_vp, c_vp, c_vp, c_i32, c_i32, ctypes.POINTER(c_i32), c_vp, c_vp, c_vp, c_vp]),
}


def library_path() -> str:
    return os.environ.get("VSRDEC_LIB", os.path.join(_HERE, "libvsrdec.so"))


def load_library():
    """dlopen libvsrdec.so and bind every entry point of include/vsrdec.h."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = library_path()
    if not os.path.isfile(path):
        raise VsrError(f"{path} not found: build it with `make -C vsr-guided-cic_b200/csrc` "
                       f"(or `python -c 'import __graft_entry__ as g; g.build()'`). "
                       f"There is no CPU / PyTorch fallback for this path.")
    lib = ctypes.CDLL(path)
    for name, (res, args) in EXPORTED_SYMBOLS.items():
        fn = getattr(lib, name)     # AttributeError if the .so does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    if lib.vsr_abi_version() != 1:
        raise VsrError(f"{path}: ABI version {lib.vsr_abi_version()} != 1")
    _LIB = lib
    return lib


def check(lib, rc: int):
    if rc != 0:
        msg = lib.vsr_last_error()
        raise VsrError(f"libvsrdec error {rc}: {msg.decode() if msg else '?'}")
