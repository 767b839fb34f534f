"""Per-kernel device time of one render (stage timing on), for the library named by RAYMOND_CUDA_LIB.
    python scripts/stage_times.py [spp] [f64|f32shade] [dragon|spheres|dof]"""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from raymond_b200 import api as A, fixtures as F
spp = int(sys.argv[1]) if len(sys.argv) > 1 else 32
prec = {"f64": 0, "f32shade": 1}[sys.argv[2] if len(sys.argv) > 2 else "f64"]
which = sys.argv[3] if len(sys.argv) > 3 else "dragon"
flags = A.FLAG_STAGE_TIMING
if which == "dragon":
    sc, cam = A.Scene.from_fixture(F.gold_dragon(F.dragon_standin())), F.camera(1920, 1080)
elif which == "spheres":
    sc, cam = A.Scene.from_fixture(F.reflective_spheres()), F.camera(1920, 1080)
else:
    sc, cam = A.Scene.from_fixture(F.reflective_spheres()), F.camera(1920, 1080, focal_length=2.5, aperture_radius=0.5)
st = A.Settings(A.CameraSettings.from_fixture(cam), spp)
r = A.Renderer(sc, st, A.GpuOptions(seed=1, flags=flags, precision=prec))
r.render(0, spp); r.sync()
s0 = r.stage_stats(); t0 = r.stats()["device_ms"]
r.render(0, spp); r.sync()
s1 = r.stage_stats(); t1 = r.stats()["device_ms"]
tot = {k: sum(b - a for a, b in zip(s0["ms"][k], s1["ms"][k])) for k in A.KERNEL_KINDS}
per = lambda k: [round(b - a, 2) for a, b in zip(s0["ms"][k], s1["ms"][k])][1:6]
ms = t1 - t0
print(f"{os.path.basename(os.environ.get('RAYMOND_CUDA_LIB', 'default'))} {which} {sys.argv[2] if len(sys.argv) > 2 else 'f64'}: total {ms:7.2f} ms = {1920*1080*spp/ms/1e3:7.1f} Msamples/s | " +
      "  ".join(f"{k} {v:6.2f}" for k, v in tot.items()) + f" | traverse {per('traverse')} shade {per('shade')} setup {per('setup')} bin {per('bin')}")
