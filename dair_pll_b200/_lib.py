"""ctypes binding of ``libdair_pll_b200.so`` (C ABI: ``include/dair_pll_b200.h`` and its warm-start extensions
``include/dair_pll_b200_warm.h`` and ``include/dair_pll_b200_warm_body_tree.h``).

There is deliberately no fallback: if the CUDA library is missing or a call fails, the
caller gets an exception.  The library is built in-tree by ``dair_pll_b200.build``.
"""
import ctypes
import os
import re

from dair_pll_b200 import build as _build

_LIB = None
ABI_VERSION = 214        # DPLL_VERSION of include/dair_pll_b200.h this binding was written against
_INCLUDE = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'include')
HEADER = os.path.join(_INCLUDE, 'dair_pll_b200.h')
WARM_HEADER = os.path.join(_INCLUDE, 'dair_pll_b200_warm.h')
WARM_BODY_TREE_HEADER = os.path.join(_INCLUDE, 'dair_pll_b200_warm_body_tree.h')

_SCALARS = {'double': ctypes.c_double, 'float': ctypes.c_float, 'int': ctypes.c_int32, 'int32_t': ctypes.c_int32,
            'int64_t': ctypes.c_int64, 'uint32_t': ctypes.c_uint32, 'size_t': ctypes.c_size_t}


def _ctype(decl: str, where: str):
    """ctypes type of a C declaration (``const double* x``, ``void** comm_out``, ``size_t``): any single pointer is a
    ``c_void_p`` (the binding passes ``data_ptr()`` integers), ``void**`` a pointer to one.  Anything else (arrays,
    other scalar types, deeper pointers) raises."""
    stars = decl.count('*')
    base = decl.replace('*', ' ').replace('const', ' ').split()[0]
    if '[' not in decl:
        if stars == 1:
            return ctypes.c_void_p
        if stars == 2 and base == 'void':
            return ctypes.POINTER(ctypes.c_void_p)
        if stars == 0 and base in _SCALARS:
            return _SCALARS[base]
    raise TypeError(f'{where}: no ctypes mapping for C type {decl.strip()!r}')


def _signatures(path: str = HEADER) -> dict:
    """name -> (argtypes, restype) of every ``dpll_*`` prototype of the C header.  The argtypes are positional, so they
    are read from the header the library is compiled against instead of being restated here."""
    with open(path) as f:
        text = re.sub(r'/\*.*?\*/|//[^\n]*', ' ', f.read(), flags=re.S)
    text = re.sub(r'^\s*#[^\n]*', ' ', text, flags=re.M)
    out = {}
    for ret, name, params in re.findall(r'([\w\s*]+?)\b(dpll_\w+)\s*\(([^)]*)\)\s*;', text):
        params = [p for p in params.split(',') if p.strip() not in ('', 'void')]
        where = f'{name} in {path}'
        out[name] = ([_ctype(p, where) for p in params], _ctype(ret, where))
    return out


EXPORTS = _signatures()                      # the main header's entry points
WARM_EXPORTS = _signatures(WARM_HEADER)      # the warm-started elbow loss (its own header)
WARM_BODY_TREE_EXPORTS = _signatures(WARM_BODY_TREE_HEADER)      # the warm-started tree losses (their own header)


def lib_path() -> str:
    """In-tree library; DAIR_PLL_B200_LIB overrides it (A/B builds during kernel development)."""
    return os.environ.get('DAIR_PLL_B200_LIB', _build.LIB_PATH)


def load() -> ctypes.CDLL:
    """Load the CUDA library; raises if it has not been built (no CPU fallback exists)."""
    global _LIB
    if _LIB is None:
        path = lib_path()
        if not os.path.exists(path):
            raise RuntimeError(
                f'{path} not found: build it with `python -m dair_pll_b200.build` '
                '(nvcc, sm_100a). dair_pll_b200 has no CPU or PyTorch fallback.')
        if path == _build.LIB_PATH and _build.sources_present() and _build.is_stale():
            # argtypes are positional: a library older than its sources could take shifted pointers
            raise RuntimeError(f'{path} is older than csrc/ or include/: rebuild it with `python -m dair_pll_b200.build`')
        lib = ctypes.CDLL(path)
        for name, (argtypes, restype) in (*EXPORTS.items(), *WARM_EXPORTS.items(), *WARM_BODY_TREE_EXPORTS.items()):
            fn = getattr(lib, name)      # AttributeError if the symbol is missing
            fn.argtypes = argtypes
            fn.restype = restype
        version = lib.dpll_version()
        if version != ABI_VERSION:
            raise RuntimeError(f'{path} reports ABI version {version}, this binding expects {ABI_VERSION}: rebuild it')
        _LIB = lib
    return _LIB


def check(rc: int, what: str) -> None:
    if rc == 0:
        return
    if rc > 0:
        raise RuntimeError(f'{what}: CUDA error {rc}')
    if rc == -3:
        raise RuntimeError(f'{what}: a peer rank did not arrive at the gradient exchange (timeout)')
    raise RuntimeError(f'{what}: argument error {rc} (see include/dair_pll_b200.h)')
