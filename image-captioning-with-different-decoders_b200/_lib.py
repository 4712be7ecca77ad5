"""ctypes binding of libicd_b200.so — the only way the Python modules reach the CUDA kernels.

The descriptor structs are generated from ``include/icd_b200.h`` itself (a tiny declaration parser), so the
Python side cannot drift from the C layout; ``icd_sizeof_*`` cross-checks the result at load time.
There is NO fallback: if the library is missing or does not load, importing any op raises.
"""
import ctypes
import os
import re

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
HEADER = os.path.join(_ROOT, "include", "icd_b200.h")
LIB_PATH = os.path.join(_HERE, "libicd_b200.so")

_SCALARS = {
    "int32_t": ctypes.c_int32, "int64_t": ctypes.c_int64, "float": ctypes.c_float,
    "int": ctypes.c_int, "uint64_t": ctypes.c_uint64, "uint8_t": ctypes.c_uint8,
}


def _strip_comments(text):
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return re.sub(r"//[^\n]*", "", text)


def _parse_header(path=HEADER):
    """-> (defines: dict, structs: dict name -> [(field, ctype)], functions: [names])"""
    raw = open(path).read()
    text = _strip_comments(raw)
    defines = {m.group(1): int(m.group(2)) for m in re.finditer(r"#define\s+(\w+)\s+(\d+)\s*$", text, flags=re.M)}
    structs = {}
    for m in re.finditer(r"typedef\s+struct\s*\{(.*?)\}\s*(\w+)\s*;", text, flags=re.S):
        body, name = m.group(1), m.group(2)
        fields = []
        for decl in body.split(";"):
            decl = " ".join(decl.split())
            if not decl:
                continue
            # split "const float *a, *b" / "int32_t B, T" / "const float* A" / "int32_t bt[N]"
            mm = re.match(r"^((?:const\s+)?\w+)\s*(.*)$", decl)
            base, rest = mm.group(1).replace("const ", "").strip(), mm.group(2)
            for d in rest.split(","):
                d = d.strip()
                ptr = d.count("*")
                d = d.replace("*", "").strip()
                arr = re.match(r"^(\w+)\[(\w+)\]$", d)
                if ptr:
                    fields.append((d, ctypes.c_void_p))
                elif arr:
                    n = arr.group(2)
                    n = int(n) if n.isdigit() else defines[n]
                    fields.append((arr.group(1), _SCALARS[base] * n))
                else:
                    fields.append((d, _SCALARS[base]))
        structs[name] = fields
    functions = re.findall(r"ICD_API\s+[\w\s\*]+?\b(icd_\w+)\s*\(", text)
    return defines, structs, functions


DEFINES, _STRUCT_FIELDS, FUNCTIONS = _parse_header()


def _make_struct(name):
    return type(name, (ctypes.Structure,), {"_fields_": _STRUCT_FIELDS[name]})


GemmDesc = _make_struct("icd_gemm_desc_t")
AttDesc = _make_struct("icd_att_desc_t")
BaseDesc = _make_struct("icd_base_desc_t")
BeamDesc = _make_struct("icd_beam_desc_t")
BaseBeamDesc = _make_struct("icd_base_beam_desc_t")
SampleDesc = _make_struct("icd_sample_desc_t")
BaseSampleDesc = _make_struct("icd_base_sample_desc_t")
AttIndex = _make_struct("icd_att_index_t")

PREC_FP32 = DEFINES["ICD_PREC_FP32"]
PREC_BF16 = DEFINES["ICD_PREC_BF16"]
PREC_FP32X3 = DEFINES["ICD_PREC_FP32X3"]
MAX_STEPS = DEFINES["ICD_MAX_STEPS"]

_lib = None


class IcdError(RuntimeError):
    pass


def lib():
    """Load (once) and return the ctypes handle; raise loudly if the CUDA library is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise IcdError(
            "libicd_b200.so not found at %s — build it with `python -c 'import __graft_entry__ as g; g.build()'`; "
            "there is no CPU / eager fallback for the decoder hot path" % LIB_PATH)
    L = ctypes.CDLL(LIB_PATH)
    L.icd_last_error_string.restype = ctypes.c_char_p
    L.icd_beam_search_ws_bytes.restype = ctypes.c_int64
    L.icd_baseline_beam_search_ws_bytes.restype = ctypes.c_int64
    L.icd_sample_captions_ws_bytes.restype = ctypes.c_int64
    L.icd_baseline_sample_captions_ws_bytes.restype = ctypes.c_int64
    L.icd_attention_proj_bwd_ws_floats.restype = ctypes.c_int64
    L.icd_launch_count.restype = ctypes.c_int64
    L.icd_gemm_ws_bytes.restype = ctypes.c_int64
    L.icd_gemm_bf16_splitk_ws_floats.restype = ctypes.c_int64
    L.icd_attention_decoder_ws_bytes.restype = ctypes.c_int64
    L.icd_attention_decoder_ws_bytes_indexed.restype = ctypes.c_int64
    L.icd_attention_proj_bwd_ws_floats_indexed.restype = ctypes.c_int64
    L.icd_baseline_decoder_ws_bytes.restype = ctypes.c_int64
    if L.icd_version() != DEFINES["ICD_B200_ABI_VERSION"]:
        raise IcdError("libicd_b200.so ABI %d != header ABI %d — rebuild" %
                       (L.icd_version(), DEFINES["ICD_B200_ABI_VERSION"]))
    for fn, st in (("icd_sizeof_att_desc", AttDesc), ("icd_sizeof_base_desc", BaseDesc),
                   ("icd_sizeof_beam_desc", BeamDesc), ("icd_sizeof_base_beam_desc", BaseBeamDesc),
                   ("icd_sizeof_sample_desc", SampleDesc), ("icd_sizeof_base_sample_desc", BaseSampleDesc),
                   ("icd_sizeof_att_index", AttIndex)):
        if getattr(L, fn)() != ctypes.sizeof(st):
            raise IcdError("%s: C says %d bytes, ctypes says %d" % (fn, getattr(L, fn)(), ctypes.sizeof(st)))
    _lib = L
    return L


def check(rc, what):
    if rc != 0:
        msg = lib().icd_last_error_string().decode("utf-8", "replace")
        raise IcdError("%s failed (rc=%d): %s" % (what, rc, msg))


def ptr(t):
    """Device pointer of a tensor (or None)."""
    if t is None:
        return None
    return ctypes.c_void_p(t.data_ptr())


def stream_ptr():
    import torch
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def fill(desc, **kw):
    """Set descriptor fields from python ints/floats/tensors; unknown names raise."""
    import torch
    names = {f[0] for f in desc._fields_}
    for k, v in kw.items():
        if k not in names:
            raise KeyError("descriptor has no field %r" % k)
        if isinstance(v, torch.Tensor):
            setattr(desc, k, v.data_ptr())
        elif v is None:
            setattr(desc, k, None)
        else:
            setattr(desc, k, v)
    return desc


def remember_versions(ctx, named):
    """Record the autograd version counters of the tensors a custom Function's backward will read through raw pointers
    ((name, tensor) pairs; None tensors skipped) — the stand-in for save_for_backward's in-place-modification check."""
    ctx._icd_versions = [(n, t, t._version) for n, t in named if hasattr(t, "_version")]


def check_versions(ctx, what):
    """Raise like autograd does when a tensor saved for backward was modified in place after the forward."""
    for n, t, v in getattr(ctx, "_icd_versions", ()):
        if t._version != v:
            raise RuntimeError("icd_b200: %s: '%s' needed for the backward was modified by an in-place operation after the forward "
                               "(is at version %d, expected %d); the backward reads it in place, like autograd's saved tensors"
                               % (what, n, t._version, v))
