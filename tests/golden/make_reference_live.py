#!/usr/bin/env python
"""Generate tests/golden/reference_live.json and reference_live_bank.npz by RUNNING THE REFERENCE.

    python tests/golden/make_reference_live.py PATH_TO_AUDIOLAZY_CHECKOUT

The reference (danilobellini/audiolazy, pure Python) is imported unmodified from the given
checkout; nothing of it is copied.  The files pin what tests/test_reference_live.py and the
``*_matches_reference`` tests of tests/test_callers_io.py compare with, on the same inputs
those tests build:

  * reference_live_bank.npz: the reference's gammatone outputs for every 7th channel of the
    64-channel bank on ``signal(123, 3000)``, as a SHA-256 of each float64 row (the tests check
    all 3000 samples bit for bit) plus the values at a fixed seeded sample of positions (so
    that a mismatch shows numbers, not only a digest);
  * reference_live.json: everything small -- scipy's lfilter grid through ZFilter, seeded
    random designs of seven builders, memory= / zero= seeding, WavStream decoding of every
    sample width, chunks() bytes, maverage / comb designs.
"""
import hashlib
import json
import os
import sys
import warnings

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
sys.path[:0] = [os.path.dirname(TESTS), TESTS]   # the package, and tests/ (make_wav is test_callers_io.py's)
BANK_SAMPLE = 64                                 # stored sample positions per bank row


def signal(seed, n):
  return np.random.default_rng(seed).uniform(-1, 1, n).astype(np.float32)


def run(filt, x, **kw):
  return np.array(list(filt(x.astype(np.float64).tolist(), **kw)), dtype=np.float64)


def sections_of(al, filt):
  if isinstance(filt, al.CascadeFilter):
    return [[list(map(float, f.numlist)), list(map(float, f.denlist))] for f in filt]
  return [[list(map(float, filt.numlist)), list(map(float, filt.denlist))]]


def row_digest(row):
  return hashlib.sha256(np.ascontiguousarray(row, dtype="<f8").tobytes()).hexdigest()


def main(ref):
  sys.path.insert(0, ref)
  sys.dont_write_bytecode = True
  warnings.simplefilter("ignore")
  import audiolazy as al
  import audiolazy_b200 as ab
  from test_callers_io import make_wav
  s, Hz = al.sHz(48000)

  # ---- test_oracle_vs_reference_all_64_channels
  x = signal(123, 3000)
  pos = np.sort(np.random.default_rng(0).choice(len(x), BANK_SAMPLE, replace=False))
  bank = {"channels": np.arange(0, 64, 7), "positions": pos}
  for name in ("slaney", "klapuri", "sampled"):
    freqs = ab.gammatone_bank(strategy=name).freqs
    rows = []
    for c in bank["channels"]:
      bw = al.gammatone_erb_constants(4)[0] * al.erb(freqs[c] * Hz, Hz)
      rows.append(run(al.gammatone[name](freqs[c] * Hz, bw), x))
    rows = np.stack(rows)
    bank[name + "_sha256"] = np.array([row_digest(r) for r in rows])
    bank[name + "_sample"] = rows[:, pos]
  np.savez_compressed(os.path.join(HERE, "reference_live_bank.npz"), **bank)

  live = {}
  # ---- test_lfilter_grid_like_reference_test
  grid = []
  for a in [[1.], [3.], [1., 3.], [15., -17.2], [-18., 9.8, 0., 14.3]]:
    for b in [[1.], [-1.], [1., 0., -1.], [1., 3.]]:
      for data in [list(range(5)), list(range(5, 0, -1)), [7, 22, -5], [8., 3., 15.]]:
        grid.append(run(al.ZFilter(b, a), np.asarray(data, dtype=np.float32)).tolist())
  live["lfilter_grid"] = grid

  # ---- test_random_designs_match_reference_bit_for_bit
  rng = np.random.default_rng(5)
  cases = []
  for _ in range(40):
    freq, bw, cutoff = rng.uniform(0.01, 3.0), rng.uniform(1e-3, 0.6), rng.uniform(0.01, 3.1)
    filts = [al.gammatone.slaney(freq, bw), al.gammatone.klapuri(freq, bw), al.gammatone.sampled(freq, bw),
             al.gammatone.sampled(freq, bw, phase=0.4, eta=5), al.lowpass.z(cutoff), al.highpass.pole(cutoff),
             al.resonator.z_exp(freq, bw)]
    rng.integers(1, 50)                         # the delays of a comb.tau pair the original live test also drew
    rng.integers(1, 50)
    cases.append({"params": [float(freq), float(bw), float(cutoff)], "sections": [sections_of(al, f) for f in filts]})
  live["random_designs"] = cases

  # ---- test_memory_semantics_vs_reference
  xm = signal(9, 50)
  live["memory_semantics"] = [run(al.ZFilter([0.3, 0.2, -0.4], [1.5, -0.2, 0.1, 0.05]), xm, memory=memory, zero=zero).tolist()
                              for memory, zero in [([0.1, 0.2, 0.3], 0.0), ([0.1], 0.25), ([0.1, 0.2, 0.3, 0.4, 0.5], -1.0),
                                                   (None, 0.5)]]

  # ---- test_callers_io: WavStream, chunks, maverage / comb designs
  live["wavstream_16"] = list(al.WavStream(make_wav(16, 1, [0, 100, -100, 32767, -32768, 12345])))
  widths = {}
  for bits in (8, 16, 24, 32):
    top = 1 << (bits - 1)
    values = [0, 1, -1, top - 1, -top, top // 3, -(top // 7), 12345 % top, -(54321 % top)]
    per = {}
    for channels in (1, 2):
      vals = values if channels == 1 else values + values[::-1]
      per[str(channels)] = {"float": list(al.WavStream(make_wav(bits, channels, vals))),
                            "keep": list(al.WavStream(make_wav(bits, channels, vals), keep=True))}
    widths[str(bits)] = per
  live["wavstream_widths"] = widths
  data = [0.5, -0.25, 1.0, 0.125, -1.0]
  live["chunks_f4"] = [blk.hex() for blk in al.chunks(data, size=4)]
  live["chunks_d2_pad9"] = [blk.hex() for blk in al.chunks(data, size=2, dfmt="d", padval=9.)]
  live["maverage"] = {"%s_%d" % (name, size): sections_of(al, al.maverage[name](size))[0]
                      for size in (1, 3, 8) for name in ("recursive", "fir")}
  live["comb_tau_linearized"] = sections_of(al, al.comb.tau(2 * np.pi / 0.05, 2e4).linearize())[0]

  with open(os.path.join(HERE, "reference_live.json"), "w") as fh:
    json.dump(live, fh, separators=(",", ":"))
  for f in ("reference_live.json", "reference_live_bank.npz"):
    print("wrote", os.path.join(HERE, f), os.path.getsize(os.path.join(HERE, f)), "bytes")


if __name__ == "__main__":
  if len(sys.argv) != 2:
    raise SystemExit(__doc__)
  main(os.path.abspath(sys.argv[1]))
