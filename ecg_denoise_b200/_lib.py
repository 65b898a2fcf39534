"""ctypes binding of libralenet_b200.so (the C ABI declared in include/ralenet_b200.h).

The argument structs are generated from the header itself, so the header is the single source of
truth for the ABI.  There is NO fallback: if the shared library is missing, or the device is not a
B200 (sm_100), every compute call raises.
"""
from __future__ import annotations

import ctypes
import os
import re
from typing import Dict

_HERE = os.path.dirname(os.path.abspath(__file__))
_ROOT = os.path.dirname(_HERE)
HEADER = os.path.join(_ROOT, "include", "ralenet_b200.h")
# RALENET_B200_LIB selects another build of the SAME library (A/B experiments on kernel variants); there is no
# alternative implementation behind it
LIB_PATH = os.environ.get("RALENET_B200_LIB") or os.path.join(_HERE, "libralenet_b200.so")

_SCALARS = {
    "int32_t": ctypes.c_int32, "int64_t": ctypes.c_int64, "uint64_t": ctypes.c_uint64,
    "float": ctypes.c_float,
}


def _parse_header(path: str):
    src = open(path).read()
    src = re.sub(r"/\*.*?\*/", " ", src, flags=re.S)
    src = re.sub(r"//[^\n]*", " ", src)
    consts: Dict[str, int] = {}
    for m in re.finditer(r"#define\s+(\w+)\s+(-?\d+)\s*$", src, flags=re.M):
        consts[m.group(1)] = int(m.group(2))
    for m in re.finditer(r"enum\s*\{(.*?)\}\s*;", src, flags=re.S):
        val = -1
        for item in m.group(1).split(","):
            item = item.strip()
            if not item:
                continue
            if "=" in item:
                name, v = [t.strip() for t in item.split("=")]
                val = int(v)
            else:
                name, val = item, val + 1
            consts[name] = val
    structs = {}
    for m in re.finditer(r"typedef\s+struct\s*\{(.*?)\}\s*(\w+)\s*;", src, flags=re.S):
        body, name = m.group(1), m.group(2)
        fields = []
        for stmt in body.split(";"):
            stmt = " ".join(stmt.split())
            if not stmt:
                continue
            stmt = stmt.replace("const ", "")
            mm = re.match(r"(\w+)\s*(\*?)\s*(.*)$", stmt)
            base, star, rest = mm.group(1), mm.group(2), mm.group(3)
            for decl in rest.split(","):
                decl = decl.strip()
                ptr = bool(star)
                if decl.startswith("*"):
                    ptr, decl = True, decl[1:].strip()
                dm = re.match(r"(\w+)((?:\[\w+\])*)$", decl)
                fname, dims = dm.group(1), re.findall(r"\[(\w+)\]", dm.group(2))
                if ptr or base == "void":
                    ctype = ctypes.c_void_p
                else:
                    ctype = _SCALARS[base]
                for d in reversed(dims):
                    ctype = ctype * (consts[d] if d in consts else int(d))
                fields.append((fname, ctype))
        structs[name] = type(name, (ctypes.Structure,), {"_fields_": fields})
    funcs = re.findall(r"^\s*(?:int|int32_t|uint64_t|int64_t|const char\*)\s+(ralenet_\w+)\s*\(", src, flags=re.M)
    return consts, structs, sorted(set(funcs))


CONSTS, STRUCTS, FUNCTIONS = _parse_header(HEADER)
globals().update(CONSTS)

_lib = None


class RalenetError(RuntimeError):
    pass


def load():
    """dlopen the library (once).  Raises RalenetError if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RalenetError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "or ./build.sh -- ecg_denoise_b200 has no CPU / PyTorch fallback path")
    lib = ctypes.CDLL(LIB_PATH)
    lib.ralenet_last_error.restype = ctypes.c_char_p
    lib.ralenet_abi_version.restype = ctypes.c_int
    lib.ralenet_net_workspace_bytes.restype = ctypes.c_uint64
    lib.ralenet_net_workspace_bytes.argtypes = [ctypes.c_int32] * 3
    lib.ralenet_net_workspace_bytes_ex.restype = ctypes.c_uint64
    lib.ralenet_net_workspace_bytes_ex.argtypes = [ctypes.c_int32] * 4
    lib.ralenet_launch_count.restype = ctypes.c_int64
    lib.ralenet_launch_count.argtypes = [ctypes.c_int32]
    lib.ralenet_check_device.argtypes = [ctypes.c_int]
    lib.ralenet_snr_mix.argtypes = [ctypes.c_void_p] * 4 + [ctypes.c_int32] * 2 + [ctypes.c_void_p]
    for name in ("ralenet_adam", "ralenet_adam_dev"):
        getattr(lib, name).argtypes = [ctypes.c_void_p] * 4 + [ctypes.c_int64] + [ctypes.c_float] * 4 + [
            ctypes.c_int32 if name == "ralenet_adam" else ctypes.c_void_p, ctypes.c_float, ctypes.c_void_p]
    P, I = ctypes.c_void_p, ctypes.c_int32
    lib.ralenet_linear_fwd.argtypes = [P, P, P, P, I, I, I, P]
    lib.ralenet_linear_bwd_data.argtypes = [P, P, P, I, I, I, P]
    lib.ralenet_pe_add.argtypes = [P, P, P, I, I, P]
    lib.ralenet_pconv1.argtypes = [P, P, P, I, I, I, I, P]
    lib.ralenet_pconv1_wgrad.argtypes = [P, P, P, I, I, I, P]
    lib.ralenet_wgrad.argtypes = [P, I, P, I, I, I, I, P, P, P]
    lib.ralenet_conv1d_slab_bytes.restype = ctypes.c_uint64
    lib.ralenet_conv1d_slab_bytes.argtypes = [I] * 4
    lib.ralenet_conv1d_bwd_det.argtypes = [P, P, ctypes.c_uint64, P]
    lib.ralenet_synth_windows.argtypes = [P, P, I, I, I, ctypes.c_uint64, P, I, P]
    lib.ralenet_comm_bytes.restype = ctypes.c_uint64
    lib.ralenet_comm_bytes.argtypes = [ctypes.c_uint64]
    lib.ralenet_comm_exchange.argtypes = [ctypes.c_void_p, ctypes.c_int32, ctypes.c_void_p, ctypes.c_int32,
                                          ctypes.c_void_p]
    lib.ralenet_comm_allreduce_adam.argtypes = [ctypes.c_void_p] * 4 + [ctypes.c_float] * 4 + [
        ctypes.c_void_p, ctypes.c_float, ctypes.c_int32, ctypes.c_void_p]
    if lib.ralenet_abi_version() != CONSTS["RL_ABI_VERSION"]:
        raise RalenetError("libralenet_b200.so ABI version does not match include/ralenet_b200.h; rebuild")
    _lib = lib
    return lib


_checked_devices = set()


def check(rc: int):
    if rc != 0:
        raise RalenetError(f"libralenet_b200 error {rc}: {load().ralenet_last_error().decode()}")


def deterministic_guard(what: str) -> None:
    """Behave like a PyTorch op without a deterministic implementation when `what` (a path of this package whose
    parameter gradients are accumulated with floating-point atomics) runs under torch.use_deterministic_algorithms(True):
    raise RuntimeError, or warn when the flag was set with warn_only=True.  Does nothing when the flag is off."""
    import torch
    if not torch.are_deterministic_algorithms_enabled():
        return
    msg = (f"{what} does not have a deterministic implementation, but you set "
           "'torch.use_deterministic_algorithms(True)'. The whole-network paths (ralenet and newrale modules, "
           "FusedTrainer and FineTuneTrainer on one GPU) are deterministic under that flag; see INTEGRATION.md "
           "section 4.")
    if torch.is_deterministic_algorithms_warn_only_enabled():
        import warnings
        warnings.warn(msg)
    else:
        raise RuntimeError(msg)


def check_device(index: int):
    if index not in _checked_devices:
        check(load().ralenet_check_device(int(index)))
        _checked_devices.add(index)


def call(fname: str, args: ctypes.Structure, stream: int):
    """invoke `int fname(const args*, void* stream)`."""
    check(getattr(load(), fname)(ctypes.byref(args), ctypes.c_void_p(stream)))


def set_attn_umma(mode: int) -> int:
    """select the forward kernels of the wide stages (C = 64, 128): 2 = tcgen05 tile kernels (attn_umma.cu),
    0 = one-window mma.sync kernels (attn.cu), 1 = tile kernels for single-wave launches only (default).
    Same function either way; returns the previous mode."""
    return int(load().ralenet_set_attn_umma(int(mode)))


def set_wgrad_umma(on: bool) -> bool:
    """weight-gradient GEMMs: True = tcgen05 kernels (wgrad_umma.cu, default), False = mma.sync kernels (wgrad.cu).
    Same function either way; returns the previous setting."""
    return bool(load().ralenet_set_wgrad_umma(1 if on else 0))


def launch_count(reset: bool = False) -> int:
    return int(load().ralenet_launch_count(1 if reset else 0))
