"""The oracle and the host-side designs against the reference on inputs beyond the golden fixtures
of make_golden.py: what the reference computed on these inputs is stored by
tests/golden/make_reference_live.py (reference_live.json, reference_live_bank.npz)."""
import hashlib

import numpy as np

import oracle
from conftest import signal


def sections(filt):
  import audiolazy_b200 as ab
  return [[list(map(float, f.numlist)), list(map(float, f.denlist))] for f in
          (filt if isinstance(filt, ab.CascadeFilter) else [filt])]


def test_oracle_vs_reference_all_64_channels(live_bank):
  import audiolazy_b200 as ab
  x = signal(123, 3000)
  pos = live_bank["positions"]
  for name in ("slaney", "klapuri", "sampled"):
    bank = ab.gammatone_bank(strategy=name)
    got = oracle.bank_apply(x, bank.sections())[0]
    for i, c in enumerate(live_bank["channels"]):
      assert np.array_equal(got[c][pos], live_bank[name + "_sample"][i]), (name, c)
      assert hashlib.sha256(np.ascontiguousarray(got[c], dtype="<f8").tobytes()).hexdigest() == \
          live_bank[name + "_sha256"][i], (name, c)


def test_lfilter_grid_like_reference_test(live):
  """reference tests/test_filters_extdep.py:41-47, through the oracle and the reference."""
  import audiolazy_b200 as ab
  from scipy.signal import lfilter
  want_grid = iter(live["lfilter_grid"])
  for a in [[1.], [3.], [1., 3.], [15., -17.2], [-18., 9.8, 0., 14.3]]:
    for b in [[1.], [-1.], [1., 0., -1.], [1., 3.]]:
      for data in [list(range(5)), list(range(5, 0, -1)), [7, 22, -5], [8., 3., 15.]]:
        x = np.asarray(data, dtype=np.float32)
        want = np.array(next(want_grid), dtype=np.float64)
        got = oracle.bank_apply(x, [[(b, a)]])[0, 0]
        assert np.array_equal(got, want)
        assert ab.almost_eq(got.tolist(), lfilter(b, a, data).tolist())


def test_random_designs_match_reference_bit_for_bit(live):
  """40 seeded (numpy default_rng(5)) parameter sets, seven builders each."""
  import audiolazy_b200 as ab
  assert len(live["random_designs"]) == 40
  for case in live["random_designs"]:
    freq, bw, cutoff = case["params"]
    mine = [ab.gammatone.slaney(freq, bw), ab.gammatone.klapuri(freq, bw), ab.gammatone.sampled(freq, bw),
            ab.gammatone.sampled(freq, bw, phase=0.4, eta=5), ab.lowpass.z(cutoff), ab.highpass.pole(cutoff),
            ab.resonator.z_exp(freq, bw)]
    assert len(mine) == len(case["sections"])
    for filt, want in zip(mine, case["sections"]):
      assert sections(filt) == want


def test_memory_semantics_vs_reference(live):
  x = signal(9, 50)
  b, a = [0.3, 0.2, -0.4], [1.5, -0.2, 0.1, 0.05]
  cases = [([0.1, 0.2, 0.3], 0.0), ([0.1], 0.25), ([0.1, 0.2, 0.3, 0.4, 0.5], -1.0), (None, 0.5)]
  assert len(cases) == len(live["memory_semantics"])
  for (memory, zero), want in zip(cases, live["memory_semantics"]):
    got = np.array(oracle.py_section(b, a, x.astype(np.float64).tolist(), memory=memory, zero=zero))
    assert np.array_equal(got, np.array(want, dtype=np.float64)), (memory, zero)
