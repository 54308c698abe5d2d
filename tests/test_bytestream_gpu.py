"""GPU parity of the escape paths of both byte-stream back ends, on content chosen so that they are taken: H.264 emulation
prevention (00 00 03) and JPEG byte stuffing (FF 00), each in a unit longer than one 4096-byte round of the stuffing copy, so
the carry between rounds is used too."""
import numpy as np
import pytest

import oracle
from selkies_b200 import _native as N
from selkies_b200.session import Session
from tests import synth
from tests.test_encode_gpu import assert_same, encode_both

pytestmark = pytest.mark.gpu

COPY_ROUND = 256 * 16         # bytes one round of the stuffing copy moves (threads x bytes per thread)


def test_h264_emulation_prevention_bit_exact():
    w, h = 320, 192
    frames = [synth.noise(w, h, 3), synth.noise(w, h, 4)]
    got, ref, grec, rrec = encode_both(w, h, frames, qp=14, slice_rows=100)      # one slice per P picture
    assert_same(got, ref, grec, rrec)
    assert [g.is_key for g in got] == [True, False]
    for g in got:
        assert b"\x00\x00\x03" in g.data
    assert len(got[1].data) > COPY_ROUND       # the P picture is one slice


def test_jpeg_byte_stuffing_bit_exact():
    w, h, quality = 320, 192, 100
    f = synth.noise(w, h, 1)
    with Session(w, h, flags=N.B2V_FLAG_JPEG, rc_mode=N.B2V_RC_CQP, crf=quality, stripe_rows=1) as s:
        s.submit(f)
        s.flush()
        got = s.take_frames()
    assert len(got) == h // 16
    pairs = 0
    for k, g in enumerate(got):
        assert (g.y_start, g.height) == (16 * k, 16)
        assert g.data == oracle.jpeg_encode_bgra(np.ascontiguousarray(f[16 * k: 16 * k + 16]), quality), k
        scan = g.data[g.data.index(b"\xff\xda") + 14: -2]          # entropy-coded segment: after SOS, before EOI
        assert len(scan) > COPY_ROUND
        pairs += scan.count(b"\xff\x00")
    assert pairs > 0
