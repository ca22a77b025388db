"""Callers and data formats either side of the path (SURVEY.md 8f): host-side behaviour on CPU,
against the reference's outputs stored by tests/golden/make_reference_live.py; the filtering
itself is covered by the gpu tests."""
import io
import struct
import wave

import numpy as np
import pytest

import audiolazy_b200 as ab


def make_wav(bits, channels, values, rate=8000):
  buf = io.BytesIO()
  with wave.open(buf, "wb") as w:
    w.setnchannels(channels)
    w.setsampwidth(bits // 8)
    w.setframerate(rate)
    if bits == 8:
      raw = bytes((v + 128) & 0xff for v in values)
    elif bits == 16:
      raw = struct.pack("<%dh" % len(values), *values)
    elif bits == 24:
      raw = b"".join(struct.pack("<i", v)[:3] for v in values)
    else:
      raw = struct.pack("<%di" % len(values), *values)
    w.writeframes(raw)
  buf.seek(0)
  return buf


@pytest.mark.parametrize("bits", [8, 16, 24, 32])
def test_wavstream_decoding(bits):
  top = (1 << (bits - 1)) - 1
  values = [0, 1, -1, top, -top - 1, top // 3, -(top // 5), 7]
  ws = ab.WavStream(make_wav(bits, 2, values))
  assert (ws.rate, ws.channels, ws.bits) == (8000, 2, bits)
  got = list(ws)
  assert np.allclose(got, [v / float(1 << (bits - 1)) for v in values], rtol=0, atol=2.0 ** -(bits - 1) * 1e-3 + 1e-7)
  assert list(ab.WavStream(make_wav(bits, 1, values), keep=True)) == [v + (128 if bits == 8 else 0) for v in values]


def test_wavstream_matches_reference(live):
  values = [0, 100, -100, 32767, -32768, 12345]
  want = live["wavstream_16"]
  assert list(ab.WavStream(make_wav(16, 1, values))) == pytest.approx(want, rel=1e-7, abs=1e-9)


@pytest.mark.parametrize("bits", [8, 16, 24, 32])
def test_wavstream_matches_reference_every_width(live, bits):
  """Byte formats must be bit-exact: same floats (and same ints with keep=True) as the reference's WavStream."""
  top = 1 << (bits - 1)
  values = [0, 1, -1, top - 1, -top, top // 3, -(top // 7), 12345 % top, -(54321 % top)]
  for channels in (1, 2):
    vals = values if channels == 1 else values + values[::-1]
    want = live["wavstream_widths"][str(bits)][str(channels)]
    assert list(ab.WavStream(make_wav(bits, channels, vals))) == want["float"]
    assert list(ab.WavStream(make_wav(bits, channels, vals), keep=True)) == want["keep"]


def test_chunks():
  blocks = list(ab.chunks([.1, .2, .3, .4, .5], size=2))
  assert len(blocks) == 3 and all(len(b) == 8 for b in blocks)
  assert struct.unpack("2f", blocks[2]) == pytest.approx((.5, 0.0))
  assert struct.unpack("<3h", next(ab.chunks([1, 2, 3], size=3, dfmt="h", byte_order="<"))) == (1, 2, 3)
  assert len(next(ab.chunks(ab.zeros()))) == 2048 * 4              # default: 2048 float32 samples
  assert list(ab.chunks([])) == []


def test_chunks_match_reference(live):
  data = [0.5, -0.25, 1.0, 0.125, -1.0]
  assert list(ab.chunks(data, size=4)) == [bytes.fromhex(h) for h in live["chunks_f4"]]
  assert list(ab.chunks(data, size=2, dfmt="d", padval=9.)) == [bytes.fromhex(h) for h in live["chunks_d2_pad9"]]


def test_wav_batch(tmp_path):
  paths = []
  for i, n in enumerate([5, 3]):
    p = tmp_path / ("f%d.wav" % i)
    p.write_bytes(make_wav(16, 1, [1000 * (i + 1)] * n).getvalue())
    paths.append(str(p))
  batch, lengths, rates = ab.wav_batch(paths)
  assert batch.shape == (2, 5) and batch.dtype == np.float32 and lengths == [5, 3] and rates == [8000, 8000]
  assert batch[1].tolist() == pytest.approx([2000 / 32768.] * 3 + [0, 0])


def test_sources_and_maverage_designs():
  assert ab.impulse(4).take(10) == [1., 0., 0., 0.] and ab.impulse().take(3) == [1., 0., 0.]
  assert ab.zeros(3).take(9) == [0., 0., 0.] and ab.ones().take(2) == [1., 1.]
  w = ab.white_noise(100).take(200)
  assert len(w) == 100 and all(-1 <= v <= 1 for v in w)
  rec, fir = ab.maverage.recursive(4), ab.maverage.fir(4)
  assert rec.numlist == [.25, 0., 0., 0., -.25] and rec.denlist == [1, -1]
  assert fir.numlist == [.25] * 4 and fir.denlist == [1]
  assert list(ab.maverage.deque(2)([1., 3., 5.])) == [.5, 2., 4.]
  assert ab.accumulate_z.denlist == [1, -1]


def test_designs_match_reference(live):
  for size in (1, 3, 8):
    for name in ("recursive", "fir"):
      mine, theirs = ab.maverage[name](size), live["maverage"]["%s_%d" % (name, size)]
      assert [mine.numlist, mine.denlist] == theirs
  ks = ab.comb.tau(2 * np.pi / 0.05, 2e4).linearize()
  assert [ks.numlist, ks.denlist] == live["comb_tau_linearized"]
