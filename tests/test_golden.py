"""Committed golden vectors (tests/golden/*.npz, made by tests/golden/make_golden.py from oracle/_ref, i.e. with
the reference's own leaf classes) vs the strict restated oracle: bit-exact.  Also guards that the seeded case
generators still reproduce the input bytes the vectors were made from (numpy RNG stream stability): the files keep a
SHA-256 of those bytes rather than the bytes themselves."""
import os

import numpy as np
import pytest

import oracle_py as op
import reference_outputs as ro
from cases import CASES

GOLD = os.path.join(os.path.dirname(__file__), "golden")
NAMES = ["am_u8", "nfm_s16", "am_bw_f32", "s8_two_devices"]


def load(name):
    return np.load(os.path.join(GOLD, name + ".npz"))


@pytest.mark.parametrize("name", NAMES)
def test_case_inputs_reproduce(name):
    g = load(name)
    _, raws = CASES[name]()
    for d, r in enumerate(raws):
        assert ro.digest(r) == str(g[f"raw{d}_sha256"]), "seeded generator no longer reproduces the stored input"


@pytest.mark.parametrize("name", NAMES)
def test_restated_oracle_matches_golden(name):
    g = load(name)
    cfg, raws = CASES[name]()   # the stored input, as test_case_inputs_reproduce checks
    res, o = op.run_oracle(cfg, raws, "restated")
    for d, (wo, iq, ax) in enumerate(res):
        assert np.array_equal(wo.view(np.uint32), g[f"waveout{d}"].view(np.uint32))
        assert np.array_equal(iq.view(np.uint64), g[f"iq_out{d}"].view(np.uint64))
        assert np.array_equal(ax, g[f"axc{d}"])
        for c in range(wo.shape[0]):
            s = o.stats(d, c)
            assert [s.open_count, s.flappy_count, s.ctcss_count, s.no_ctcss_count, s.active_counter] == list(g[f"counts{d}"][c])
