"""CPU reference for gsb_render_aux's (opacity, expected depth) planes: tests/aux_oracle.c over the oracle frame's own
attributes and sorted tile lists.  The C file is compiled on first use into a temporary directory (nothing is written to
the tree) with the oracle's flags and linked against oracle/liboracle.so for the shared-definition exp."""
from __future__ import annotations

import ctypes as C
import hashlib
import subprocess
import tempfile
from pathlib import Path

import numpy as np

import oracle as o

HERE = Path(__file__).resolve().parent
SRC = HERE / "aux_oracle.c"
ORACLE_DIR = Path(o.LIB_PATH).parent
_lib = None


def _load():
    global _lib
    if _lib is None:
        tag = hashlib.sha256(SRC.read_bytes()).hexdigest()[:16]
        out = Path(tempfile.gettempdir()) / f"gsb_aux_oracle_{tag}" / "libaux_oracle.so"
        if not out.exists():
            out.parent.mkdir(parents=True, exist_ok=True)
            tmp = out.with_suffix(".so.tmp")
            subprocess.run(["gcc", "-O2", "-std=c11", "-fPIC", "-ffp-contract=off", "-fno-fast-math", "-fopenmp", "-shared",
                            "-o", str(tmp), str(SRC), f"-L{ORACLE_DIR}", "-loracle", f"-Wl,-rpath,{ORACLE_DIR}", "-lm"],
                           check=True, capture_output=True)
            tmp.replace(out)
        _lib = C.CDLL(str(out))
        _lib.aux_blend.argtypes = [C.c_void_p] * 3 + [C.c_uint32] * 4 + [C.c_int, C.c_void_p, C.c_void_p]
        _lib.aux_blend.restype = None
    return _lib


def blend(attr, vals, ranges, width, height, rows=None, exp_mode=0):
    """(rgba (H, W, 4), aux (H, W, 2)); pixels outside tile rows `rows` stay zero."""
    at = np.ascontiguousarray(attr, o.ATTR_DTYPE)
    vv = np.ascontiguousarray(vals, np.uint32)
    rr = np.ascontiguousarray(ranges, np.uint32)
    rb, re = (0, o.ALL_ROWS) if rows is None else rows
    rgba = np.zeros((height, width, 4), np.float32)
    aux = np.zeros((height, width, 2), np.float32)
    _load().aux_blend(at.ctypes.data, vv.ctypes.data, rr.ctypes.data, width, height, rb, re, exp_mode, rgba.ctypes.data,
                      aux.ctypes.data)
    return rgba, aux


def render_frame(vtx, u, rows=None, exp_mode=1, probed=False):
    """oracle.render_frame (exp mode `exp_mode`) + "aux" and "rgba_aux" (this blend's colour); probed=True returns
    (frame, step-probe mask) like oracle.render_frame_probed."""
    o.set_exp_mode(exp_mode)
    try:
        if probed:
            f, mask = o.render_frame_probed(vtx, o.cov3d(vtx), u, rows)
        else:
            f, mask = o.render_frame(vtx, o.cov3d(vtx), u, rows), None
    finally:
        o.set_exp_mode(0)
    ou = o.Uniforms.from_buffer_copy(bytes(u))
    f["rgba_aux"], f["aux"] = blend(f["attr"], f["vals"], f["ranges"], ou.width, ou.height, rows, exp_mode)
    return (f, mask) if probed else f
