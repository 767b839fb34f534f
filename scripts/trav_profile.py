"""Cycles per k_traverse phase, for the library named by RAYMOND_CUDA_LIB.  It needs the profiling build:
    python -c 'from raymond_b200 import build; build.build(defines=["RM_TRAV_PROFILE"], out="/tmp/trav_profile.so")'
    RAYMOND_CUDA_LIB=/tmp/trav_profile.so python scripts/trav_profile.py [spp]"""
import ctypes as C, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from raymond_b200 import api as A, fixtures as F
spp = int(sys.argv[1]) if len(sys.argv) > 1 else 16
sc = A.Scene.from_fixture(F.gold_dragon(F.dragon_standin()))
st = A.Settings(A.CameraSettings.from_fixture(F.camera(1920, 1080)), spp)
r = A.Renderer(sc, st, A.GpuOptions(seed=1))
r.render(0, spp); r.sync()
out = (C.c_ulonglong * 8)()
L = A.lib()
L.rm_debug_trav_profile(out)
s0 = r.stats()["device_ms"]
r.render(0, spp); r.sync()
L.rm_debug_trav_profile(out)
ms = r.stats()["device_ms"] - s0
v = list(out)
tot = sum(v[:7])
names = ["refill", "walk(A)", "pool set-up(B)", "finish(C)", "loop head", "stage-1 rounds(B)", "stage-2 rounds(B)"]
print(f"frame {ms:7.2f} ms | " + "  ".join(f"{n} {100*x/tot:5.1f}%" for n, x in zip(names, v[:7])) + f" | warps {v[7]}  cycles/warp {tot/max(v[7],1)/1e6:.2f}M")
