"""Rate of the JPEG stripe path (B2V_FLAG_JPEG, quality 60, default stripes) at 4K, inputs resident in HBM, device-timed; desktop
content (damage in some stripes per picture) and noise (every stripe changes, worst-case entropy data).
B2V_LIB=<path> python tools/jpeg_rate.py   (run once per library; each process loads one build)"""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench                                     # noqa: E402
from selkies_b200 import _native as N            # noqa: E402
from tests import synth                          # noqa: E402

W, H = 3840, 2160
jpeg = dict(fps=60.0, flags=N.B2V_FLAG_JPEG, rc_mode=N.B2V_RC_CQP, crf=60, ring_slots=16)
out = {"lib": os.environ.get("B2V_LIB", "in-tree")}
for rep in range(2):
    out[f"desktop_{rep}"] = round(bench.resident_leg([synth.desktop(W, H, t) for t in range(16)], 256, 0, warm=32, **jpeg)["value"])
    out[f"noise_{rep}"] = round(bench.resident_leg([synth.noise(W, H, 100 + t) for t in range(4)], 96, 0, warm=16, **jpeg)["value"])
print(json.dumps(out))
