"""Session counters for the three output shapes (full-frame H.264, striped H.264, JPEG stripes), with and without the pixelflux
header: bytes and pictures delivered, key frames, kernel launches and device-to-host traffic, picture by picture."""
import pytest

from selkies_b200 import _native as N
from selkies_b200.session import Session
from tests import synth

pytestmark = pytest.mark.gpu

W, H = 1280, 720                 # 45 macroblock rows; every shape's access-unit buffer is larger than FIRST_CHUNK
FIRST_CHUNK = 256 << 10          # access-unit bytes copied to the host with the size word, whatever the picture's size
AU_HEADER = 64                   # the smallest offset of the first NAL in the access-unit buffer

SHAPES = {
    # name: session arguments, kernel launches per picture after the CSC
    "fullframe": (dict(rc_mode=N.B2V_RC_CQP, crf=24), 4),
    "striped": (dict(rc_mode=N.B2V_RC_CQP, crf=24, stripe_rows=8), 4),      # 5 bands of 8 rows and one of 5
    "jpeg": (dict(flags=N.B2V_FLAG_JPEG, rc_mode=N.B2V_RC_CQP, crf=60), 7),  # default stripes: 7 of 6 rows and one of 3
}
HEADERS = {"none": (N.B2V_HDR_NONE, 0), "pixelflux": (N.B2V_HDR_PIXELFLUX, 10)}

# colour bars with a moving square: access units far below FIRST_CHUNK, and only the bands the square crosses are delivered after
# the first picture.  The noise IDR at picture 3 needs a second copy for the tail of its access unit; the pictures around it change
# everywhere.
PICTURES = [("bars", 0), ("bars", 1), ("desktop", 2), ("noise", 3), ("bars", 4)]
IDR_AT = (0, 3)


@pytest.mark.parametrize("header", sorted(HEADERS))
@pytest.mark.parametrize("shape", sorted(SHAPES))
def test_session_counters(shape, header):
    kw, launches = SHAPES[shape]
    mode, hdr_len = HEADERS[header]
    if shape == "jpeg" and mode == N.B2V_HDR_PIXELFLUX:
        hdr_len = 4                                      # frame_id | y_start in front of each JFIF file
    small = tails = 0
    with Session(W, H, header_mode=mode, **kw) as s:
        prev = s.stats()
        for i, (kind, t) in enumerate(PICTURES):
            if i in IDR_AT and i > 0:
                s.request_idr()
            s.submit(getattr(synth, kind)(W, H, t))
            s.flush()
            got = s.take_frames()
            st = s.stats()
            d = {k: st[k] - prev[k] for k in ("frames_submitted", "frames_delivered", "key_frames", "bytes_out", "d2h_bytes", "kernel_launches")}
            prev = st
            assert got, f"picture {i}: nothing delivered"
            assert d["frames_submitted"] == d["frames_delivered"] == 1
            assert d["key_frames"] == (i in IDR_AT)
            assert all(g.is_key == (i in IDR_AT) and g.frame_id == i for g in got)
            assert d["kernel_launches"] == 1 + launches
            assert d["bytes_out"] == sum(len(g.data) for g in got)
            if shape == "fullframe":
                assert len(got) == 1 and (got[0].y_start, got[0].height) == (0, H)
            if mode == N.B2V_HDR_PIXELFLUX and shape != "jpeg":
                for g in got:
                    h = g.data[:10]
                    assert h[0] == 0x04 and h[1] == (i in IDR_AT) and int.from_bytes(h[2:4], "big") == i
                    assert [int.from_bytes(h[k:k + 2], "big") for k in (4, 6, 8)] == [g.y_start, W, g.height]
            payload = sum(len(g.data) - hdr_len for g in got)  # access-unit bytes delivered
            if payload < FIRST_CHUNK // 2:             # the access unit fits the first chunk: no tail fetch
                small += 1
                assert d["d2h_bytes"] == FIRST_CHUNK, f"picture {i}"
            elif shape == "fullframe":                   # the access unit is exactly what was delivered
                assert d["d2h_bytes"] == max(FIRST_CHUNK, AU_HEADER + payload), f"picture {i}"
            else:                                        # the access unit also holds the bands that were not delivered
                assert d["d2h_bytes"] >= max(FIRST_CHUNK, AU_HEADER + payload), f"picture {i}"
            tails += payload > FIRST_CHUNK
        total = s.stats()
    assert small >= 1 and tails >= 1, (small, tails)
    assert total["frames_delivered"] == total["frames_submitted"] == len(PICTURES)
    assert total["key_frames"] == len(IDR_AT)
