"""ctypes binding of libzhilight_b200.so (the C-ABI in include/zhilight_b200.h).

The prototypes are parsed from the header so that the binding, the header and the library cannot
drift apart.  There is NO CPU fallback: if the shared library is missing, or a compute entry point
is called without a CUDA device, this raises.
"""
import ctypes
import os
import re

HERE = os.path.dirname(os.path.abspath(__file__))
HEADER = os.path.join(HERE, "..", "include", "zhilight_b200.h")
LIB_PATH = os.path.join(HERE, "libzhilight_b200.so")


class ZLError(RuntimeError):
    """Raised for every non-zero return code (mirrors BMEngineException -> RuntimeError in the reference,
    3rd/bmengine/bmengine/include/bmengine/core/exception.h:25-130)."""

    def __init__(self, code, msg):
        super().__init__("zhilight_b200 error %d: %s" % (code, msg))
        self.code = code


class LlamaConfig(ctypes.Structure):
    _fields_ = [
        ("num_layers", ctypes.c_int), ("dim_model", ctypes.c_int), ("num_heads", ctypes.c_int),
        ("num_kv_heads", ctypes.c_int), ("dim_head", ctypes.c_int), ("dim_ff", ctypes.c_int),
        ("vocab_size", ctypes.c_int),
        ("eps", ctypes.c_float), ("rope_theta", ctypes.c_float),
        ("rope_llama3_factor", ctypes.c_float), ("rope_low_freq_factor", ctypes.c_float),
        ("rope_high_freq_factor", ctypes.c_float), ("rope_orig_ctx", ctypes.c_float),
        ("quant_type", ctypes.c_int), ("group_size", ctypes.c_int), ("sym", ctypes.c_int),
        ("dtype", ctypes.c_int), ("max_batch", ctypes.c_int), ("max_seq", ctypes.c_int),
        ("tp_rank", ctypes.c_int), ("tp_size", ctypes.c_int),
        ("use_pdl", ctypes.c_int), ("use_graph", ctypes.c_int), ("tp_int8", ctypes.c_int), ("fuse", ctypes.c_int), ("prefill_chunk", ctypes.c_int),
        ("qkv_bias", ctypes.c_int),
    ]


class SampleParams(ctypes.Structure):
    """zl_sample_params_t"""
    _fields_ = [
        ("temperature", ctypes.c_float), ("top_p", ctypes.c_float), ("repetition_penalty", ctypes.c_float),
        ("presence_penalty", ctypes.c_float), ("top_k", ctypes.c_int), ("seed", ctypes.c_uint64),
    ]


class W4FusedArgs(ctypes.Structure):
    """zl_w4_fused_args_t"""
    _fields_ = [
        ("x", ctypes.c_void_p), ("ldx", ctypes.c_int), ("packed", ctypes.c_void_p), ("bias", ctypes.c_void_p),
        ("residual", ctypes.c_void_p), ("y", ctypes.c_void_p),
        ("M", ctypes.c_int), ("N", ctypes.c_int), ("K", ctypes.c_int), ("group_size", ctypes.c_int),
        ("epilogue", ctypes.c_int), ("pdl", ctypes.c_int),
        ("ln_weight", ctypes.c_void_p), ("eps", ctypes.c_float),
        ("cos", ctypes.c_void_p), ("sin", ctypes.c_void_p), ("q_out", ctypes.c_void_p),
        ("token_batch", ctypes.c_void_p), ("placement", ctypes.c_void_p), ("k_addrs", ctypes.c_void_p),
        ("v_addrs", ctypes.c_void_p),
        ("num_heads", ctypes.c_int), ("num_kv_heads", ctypes.c_int), ("dim_head", ctypes.c_int),
        ("prefetch_ptr", ctypes.c_void_p), ("prefetch_bytes", ctypes.c_size_t),
        ("variant", ctypes.c_int),
        ("tp_comm", ctypes.c_void_p), ("tp_mode", ctypes.c_int), ("tp_h_out", ctypes.c_void_p), ("tp_index", ctypes.c_int),
    ]


_SCALARS = {
    "int": ctypes.c_int, "float": ctypes.c_float, "double": ctypes.c_double, "size_t": ctypes.c_size_t,
    "uint64_t": ctypes.c_uint64, "uint32_t": ctypes.c_uint32, "int32_t": ctypes.c_int32,
    "long long": ctypes.c_longlong, "zl_stream_t": ctypes.c_void_p, "void": None, "unsigned": ctypes.c_uint,
}


def _ctype(decl):
    """Map a C parameter / return type string to a ctypes type."""
    t = decl.replace("const", " ").strip()
    t = re.sub(r"\s+", " ", t)
    if "*" in t:
        base = t.replace("*", "").strip()
        if base == "char" and t.count("*") == 1:
            return ctypes.c_char_p
        if base == "double" and t.count("*") == 1:
            return ctypes.POINTER(ctypes.c_double)
        if base == "int" and t.count("*") == 1:
            return ctypes.POINTER(ctypes.c_int)
        return ctypes.c_void_p
    return _SCALARS[t]


def parse_header(path=HEADER):
    """-> {name: (restype_str, [(type_str, arg_name), ...])} for every zl_* prototype."""
    src = open(path).read()
    src = re.sub(r"/\*.*?\*/", " ", src, flags=re.S)
    src = re.sub(r"//[^\n]*", " ", src)
    src = re.sub(r"typedef struct zl_llama_config \{.*?\} zl_llama_config_t;", " ", src, flags=re.S)
    src = re.sub(r"typedef struct zl_w4_fused_args \{.*?\} zl_w4_fused_args_t;", " ", src, flags=re.S)
    src = re.sub(r"typedef struct zl_sample_params \{.*?\} zl_sample_params_t;", " ", src, flags=re.S)
    protos = {}
    for m in re.finditer(r"([A-Za-z_][\w \*]*?)\b(zl_\w+)\s*\(([^;{}]*?)\)\s*;", src):
        ret, name, args = m.group(1).strip(), m.group(2), m.group(3).strip()
        if ret.startswith("typedef") or not ret:
            continue
        params = []
        if args and args != "void":
            for a in args.split(","):
                a = a.strip()
                mm = re.match(r"(.*?)(\w+)$", a)
                params.append((mm.group(1).strip(), mm.group(2)))
        protos[name] = (ret, params)
    return protos


_lib = None
_protos = None


def load():
    """Load the library (building nothing).  Raises if the .so is absent."""
    global _lib, _protos
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ZLError(-100, "libzhilight_b200.so not built (run `python -m zhilight_b200.build`); "
                            "there is no CPU fallback")
    lib = ctypes.CDLL(LIB_PATH)
    _protos = parse_header()
    for name, (ret, params) in _protos.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is missing
        fn.restype = ctypes.c_char_p if ret.replace("const", "").strip() == "char*" else _ctype(ret)
        fn.argtypes = [_ctype(t) for t, _ in params]
    _lib = lib
    return lib


def protos():
    load()
    return _protos


def last_error():
    s = load().zl_last_error()
    return s.decode() if s else ""


def check(rc):
    if rc != 0:
        raise ZLError(rc, last_error())


def call(name, *args):
    """Call an int-returning entry point and raise ZLError on failure."""
    check(getattr(load(), name)(*args))
