"""In-step numbers for the 4K headline workload with the library built as it is: pictures/s (inputs resident, no timing flags),
the CSC launch by CUDA-event pair and by the kernel's own %globaltimer stamps, and the per-stage event breakdown.
Run on the GPU box: python tools/instep.py [n_pictures]"""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from selkies_b200 import _native as N          # noqa: E402
from selkies_b200.session import Session        # noqa: E402
from tests import synth                         # noqa: E402

W, H, ND = 3840, 2160, 16
n = int(sys.argv[1]) if len(sys.argv) > 1 else 512
CONTENT = os.environ.get("B2V_CONTENT", "desktop")      # desktop (headline) | gradient (S4) | noise (S2)
frames = [{"desktop": synth.desktop, "gradient": synth.gradient}[CONTENT](W, H, t) if CONTENT != "noise" else synth.noise(W, H, 100 + t) for t in range(ND)]
out = {}


def run(flags, label):
    with Session(W, H, fps=60.0, rc_mode=N.B2V_RC_CBR, bitrate_kbps=20000, ring_slots=16, flags=flags, collect=False,
                 slice_rows=int(os.environ.get("B2V_SLICE_ROWS", "0"))) as s:
        for i, f in enumerate(frames):
            s.resident_upload(i, f)
        for k in range(64):
            s.submit_resident(k % ND)
        s.flush(); s.reset_stats()
        s.timer_start()
        for k in range(n):
            s.submit_resident(k % ND)
        ms = s.timer_stop()
        st = s.stats()
    out[label] = {"fps": n / (ms / 1000.0), "us_per_picture": ms * 1e3 / n}
    if st["n_csc"]:
        out[label]["csc_event_us"] = st["ms_csc"] / st["n_csc"] * 1e3
    if st["n_csc_device"]:
        out[label]["csc_device_us"] = st["ms_csc_device"] / st["n_csc_device"] * 1e3
    if st["n_inter"]:
        out[label].update({k + "_us": st["ms_" + k] / max(1, st["n_" + k]) * 1e3 for k in ("inter", "cavlc", "slice", "pack")})
        out[label]["span_us"] = st["ms_total_gpu"] / st["n_csc"] * 1e3


run(0, "plain")
run(N.B2V_FLAG_TIMING_CSC, "timing_csc")
run(N.B2V_FLAG_TIMING | N.B2V_FLAG_DEVICE_TIMER, "timing_all")
print(json.dumps(out))
