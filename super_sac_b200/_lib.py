"""ctypes binding of libssac_b200.so (the C ABI declared in include/ssac_b200.h).

The header is the single source of truth: prototypes are parsed from it, so every declared symbol must be
exported by the library (checked at load time) and argument types always match the declaration.
There is no fallback of any kind: if the library is missing, or the device is not sm_100, importing callers
get an exception (BASELINE north_star: "no Triton, no multi-backend dispatch and no CPU fallback").
"""
import ctypes
import os
import re

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libssac_b200.so")
HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "ssac_b200.h")

_SCALARS = {
    "int": ctypes.c_int,
    "int32_t": ctypes.c_int32,
    "int64_t": ctypes.c_int64,
    "uint64_t": ctypes.c_uint64,
    "uint32_t": ctypes.c_uint32,
    "float": ctypes.c_float,
    "double": ctypes.c_double,
}


def parse_header(path=HEADER_PATH):
    """Returns {name: (restype, [argtypes], [argnames])} for every prototype in the header."""
    src = open(path).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    src = re.sub(r"//[^\n]*", "", src)
    src = re.sub(r"^\s*#.*$", "", src, flags=re.M)
    protos = {}
    for m in re.finditer(r"([A-Za-z_][\w\s\*]*?)\b(ssac_\w+)\s*\(([^;{}]*?)\)\s*;", src, flags=re.S):
        ret, name, args = m.group(1).strip(), m.group(2), m.group(3).strip()
        ret = ret.replace('extern "C"', "").strip()
        if "*" in ret:
            restype = ctypes.c_char_p if "char" in ret else ctypes.c_void_p
        else:
            restype = _SCALARS[ret.replace("const", "").strip()]
        argtypes, argnames = [], []
        if args and args != "void":
            for a in args.split(","):
                a = " ".join(a.split())
                pm = re.match(r"(.*?)(\w+)$", a)
                typ, nm = pm.group(1).strip(), pm.group(2)
                if "*" in typ:
                    argtypes.append(ctypes.c_void_p)
                else:
                    argtypes.append(_SCALARS[typ.replace("const", "").strip()])
                argnames.append(nm)
        protos[name] = (restype, argtypes, argnames)
    return protos


_NOT_STATUS = {"ssac_version", "ssac_default_mlp_impl", "ssac_get_overlap", "ssac_get_fused_forward", "ssac_get_pdl", "ssac_rows_supported"}  # int-returning entry points whose value is not a status code


class SsacError(RuntimeError):
    pass


class _Lib:
    def __init__(self):
        if not os.path.exists(LIB_PATH):
            raise SsacError(
                f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a). super_sac_b200 has no CPU or PyTorch fallback."
            )
        self.cdll = ctypes.CDLL(LIB_PATH)
        self.protos = parse_header()
        missing = []
        for name, (restype, argtypes, _) in self.protos.items():
            try:
                fn = getattr(self.cdll, name)
            except AttributeError:
                missing.append(name)
                continue
            fn.restype = restype
            fn.argtypes = argtypes
            if restype is ctypes.c_int and name not in _NOT_STATUS:
                setattr(self, name[len("ssac_"):], self._checked(fn, name))
            else:
                setattr(self, name[len("ssac_"):], fn)
        if missing:
            raise SsacError(f"libssac_b200.so does not export: {missing}")
        # debugging switches (results never depend on them)
        if os.environ.get("SSAC_NO_PDL"):
            self.cdll.ssac_set_pdl(0)
        if os.environ.get("SSAC_NO_OVERLAP"):
            self.cdll.ssac_set_overlap(0)
        if os.environ.get("SSAC_NO_ROWS"):
            self.cdll.ssac_set_rows_enabled(0)
        if os.environ.get("SSAC_NO_TMA"):
            self.cdll.ssac_set_tma_enabled(0)
        if os.environ.get("SSAC_CONV_HALO"):
            self.set_conv_halo(int(os.environ["SSAC_CONV_HALO"]))
        if os.environ.get("SSAC_NO_FUSED"):
            self.cdll.ssac_set_fused_forward(0)

    def _checked(self, fn, name):
        last_error = self.cdll.ssac_last_error
        last_error.restype = ctypes.c_char_p

        def call(*args):
            rc = fn(*args)
            if rc != 0:
                raise SsacError(f"{name} failed (code {rc}): {last_error().decode()}")

        call.__name__ = name
        call.raw = fn
        return call


_lib = None
_device_ok = set()


def lib():
    global _lib
    if _lib is None:
        _lib = _Lib()
    return _lib


def require_device(index):
    """Fail loudly unless CUDA device `index` is an sm_100 part."""
    if index not in _device_ok:
        lib().device_check(int(index))
        _device_ok.add(index)


_forced_stream = None


class on_stream:
    """Route every entry-point call inside the block to the raw stream ``ptr`` (cheaper than torch.cuda.stream(...) when
    the callee only needs the handle)."""

    def __init__(self, ptr):
        self.ptr = ptr

    def __enter__(self):
        global _forced_stream
        self.prev, _forced_stream = _forced_stream, self.ptr

    def __exit__(self, *a):
        global _forced_stream
        _forced_stream = self.prev


def stream_ptr():
    """Raw handle of torch's current CUDA stream on the current device (the private C accessor is an order of
    magnitude cheaper than building a torch.cuda.Stream object on every entry-point call)."""
    if _forced_stream is not None:
        return _forced_stream
    import torch

    try:
        return torch._C._cuda_getCurrentRawStream(torch.cuda.current_device())
    except AttributeError:
        return torch.cuda.current_stream().cuda_stream


def host_array(ctype, values):
    return (ctype * len(values))(*values)
