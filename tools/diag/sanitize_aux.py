"""Small gsb_render_aux frames for compute-sanitizer: C1 at gsb_set_tile_cull levels 0 and 2, both blend modes, float and
BGRA8 colour, device and (pageable, page-locked) host outputs, a band, timers on (direct launches) and off (graph replay)."""
import ctypes as C
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[2]
sys.path.insert(0, str(ROOT / "3dgs.cpp_b200" / "python"))
sys.path.insert(0, str(ROOT / "tests"))
import gs_b200 as g  # noqa: E402
import scenes  # noqa: E402

_, vtx, u = scenes.c1(n=4000)
c = g.Context(0)
c.upload(vtx)
ref = None
for level in (0, 2):
    c.set_tile_cull(level)
    for timers in (True, False):
        c.set_timers(timers)
        for mode in (g.MODE_EXACT, g.MODE_FAST):
            c.set_mode(mode)
            for fmt in (g.FORMAT_RGBA32F, g.FORMAT_BGRA8):
                img, aux = c.render_aux(u, fmt)
                if mode == g.MODE_EXACT and fmt == g.FORMAT_RGBA32F:
                    if ref is None:
                        ref = aux
                    assert np.array_equal(aux, ref), (level, timers)
        c.set_mode(g.MODE_EXACT)
        _, band = c.render_aux(u, rows=(5, 17))
        assert np.array_equal(band, ref[5 * 16:17 * 16])
p = C.c_void_p()
assert g.lib.gsb_host_alloc(C.byref(p), u.width * u.height * 8) == 0
img = np.zeros((u.height, u.width, 4), np.float32)
c._ck(g.lib.gsb_render_aux(c.h, C.byref(u), 0, g.ALL_ROWS, img.ctypes.data, 0, p, 0, g.MEM_HOST, g.FORMAT_RGBA32F, None))
pinned = np.frombuffer((C.c_char * (u.width * u.height * 8)).from_address(p.value), np.float32).reshape(u.height, u.width, 2)
assert np.array_equal(pinned, ref)
g.lib.gsb_host_free(p)
c.close()
print("sanitize aux target ok")
