"""A dozen 4K CSC launches over distinct resident frames (CSC-only session) — the target of bench.py's live ncu traffic probe
and of the `ncu --set full` captures under profiles/.  CSC_SIZE=8k runs 7680x4320 instead."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from selkies_b200 import _native as N          # noqa: E402
from selkies_b200.session import Session        # noqa: E402
from tests import synth                         # noqa: E402

W, H = (7680, 4320) if os.environ.get("CSC_SIZE") == "8k" else (3840, 2160)
with Session(W, H, flags=N.B2V_FLAG_NO_ENCODE) as s:
    for i in range(4):
        s.resident_upload(i, synth.desktop(W, H, i))
    s.bench_csc_burst(4, 8)
