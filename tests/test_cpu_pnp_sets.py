"""CPU-side checks of the multi-set PnP entry point (cp_pnp_ransac_sets): the host validation of ops.pnp_ransac's tuple
``flag`` and ``rng_index``, the library's own argument checks, and the ctypes signatures against the C header."""
import ctypes as C
import os
import re

import pytest
import torch

from helpers import REPO

torch.set_grad_enabled(False)

B, N = 4, 16


@pytest.fixture(scope="module")
def ops():
    from checkerpose_b200 import ops as o
    return o


def _args():
    packed = torch.zeros((B, 16 + 2 * N), dtype=torch.uint8)
    return packed, torch.zeros((1, N, 3)), torch.eye(3)


@pytest.mark.parametrize("flag, match", [
    ((), "empty"),
    ((1, 2, 4, 3), "at most 3"),
    ((1, 2, 1), "duplicate"),
    ((2, 4, 2), "duplicate"),
    ((0, 1), r"\[1, 7\]"),
    ((1, 8), r"\[1, 7\]"),
    ((-4,), r"\[1, 7\]"),
])
def test_flag_tuple_is_checked_on_the_host(ops, flag, match):
    packed, p3d, K = _args()
    with pytest.raises(RuntimeError, match=match):
        ops.pnp_ransac(packed, p3d, K, flag=flag)


@pytest.mark.parametrize("flag", [1, (1, 2, 4)])
@pytest.mark.parametrize("rng_index, match", [
    (torch.arange(B - 1, dtype=torch.int32), "shape"),
    (torch.arange(B + 1, dtype=torch.int32), "shape"),
    (torch.arange(B, dtype=torch.int32).view(2, 2), "shape"),
    (torch.arange(B, dtype=torch.int64), "int32"),
    (torch.arange(B, dtype=torch.float32), "int32"),
])
def test_rng_index_is_checked_on_the_host(ops, flag, rng_index, match):
    packed, p3d, K = _args()
    with pytest.raises(RuntimeError, match=match):
        ops.pnp_ransac(packed, p3d, K, flag=flag, rng_index=rng_index)


def test_valid_sets_reach_the_cuda_check(ops):
    """A well-formed tuple passes the host checks and stops at the refusal of CPU tensors (there is no CPU path)."""
    packed, p3d, K = _args()
    for flag in ((1,), (4, 1), (1, 2, 4), (7, 3, 5)):
        with pytest.raises(RuntimeError, match="CUDA"):
            ops.pnp_ransac(packed, p3d, K, flag=flag, rng_index=torch.arange(B, dtype=torch.int32))


def _call_sets(lib, masks, num_sets=None):
    arr = (C.c_int32 * max(1, len(masks)))(*masks)
    fake = C.c_void_p(256)        # never dereferenced: the arguments are refused before any CUDA call
    return lib.cp_pnp_ransac_sets(fake, None, fake, None, fake, 0, len(masks) if num_sets is None else num_sets, arr, None,
                                  2.0, 150, 0, fake, fake, None, B, N, 64, None)


def test_library_refuses_bad_flag_masks():
    from checkerpose_b200 import _lib
    for masks, num_sets, what in (((1, 2, 4, 3), None, b"1 to 3"), ((), 0, b"1 to 3"), ((1, 2, 1), None, b"both 1"),
                                  ((4, 4), None, b"both 4"), ((0, 1), None, b"[1,7]"), ((1, 8), None, b"[1,7]")):
        rc = _call_sets(_lib.lib, masks, num_sets)
        assert rc == -1, masks
        assert what in _lib.lib.cp_last_error_string(), (masks, _lib.lib.cp_last_error_string())
    fake = C.c_void_p(256)
    rc = _lib.lib.cp_pnp_ransac_sets(fake, None, fake, None, fake, 0, 2, None, None, 2.0, 150, 0, fake, fake, None, B, N, 64, None)
    assert rc == -1


# C parameter / return type -> the ctypes type _lib.SIGNATURES must give it
_SCALARS = {"int": C.c_int, "int32_t": C.c_int32, "int64_t": C.c_int64, "uint64_t": C.c_uint64, "size_t": C.c_size_t,
            "float": C.c_float, "double": C.c_double, "cp_stream_t": C.c_void_p}


def _prototypes():
    src = open(os.path.join(REPO, "include", "checkerpose_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    out = {}
    for ret, name, params in re.findall(r"\b((?:const\s+)?[a-z_0-9]+\s*\*?)\s*(cp_[a-z0-9_]+)\s*\(([^)]*)\)\s*;", src):
        params = [] if params.strip() in ("", "void") else [p.strip() for p in params.split(",")]
        out[name] = (ret.strip(), params)
    return out


def _matches(ctype, decl):
    decl = re.sub(r"\bconst\b", "", decl).strip()
    if "*" not in decl:
        base = decl.split()[0]
        return ctype is _SCALARS[base]
    if decl.split("*")[0].strip() == "char":
        return ctype is C.c_char_p
    # a pointer: an untyped address, or a typed pointer to the pointee (host arrays, parameter structs)
    return ctype is C.c_void_p or (hasattr(ctype, "_type_") and issubclass(ctype, C._Pointer))


@pytest.mark.parametrize("name", ["cp_pnp_ransac", "cp_pnp_ransac_sets"])
def test_pnp_argtypes_match_the_header(name):
    from checkerpose_b200 import _lib
    ret, params = _prototypes()[name]
    res, args = _lib.SIGNATURES[name]
    assert _matches(res, ret)
    assert len(args) == len(params), f"{name}: header {len(params)} parameters, ctypes {len(args)}"
    for i, (a, p) in enumerate(zip(args, params)):
        assert _matches(a, p), f"{name} parameter {i} `{p}`: ctypes {a}"
    fn = getattr(_lib.lib, name)
    assert fn.restype is res and list(fn.argtypes) == list(args)


def test_flag_masks_is_a_host_int32_array():
    from checkerpose_b200 import _lib
    _, params = _prototypes()["cp_pnp_ransac_sets"]
    i = next(k for k, p in enumerate(params) if p.endswith("flag_masks"))
    assert _lib.SIGNATURES["cp_pnp_ransac_sets"][1][i] is C.POINTER(C.c_int32)
