"""Whole-path checks of the oracle itself: restated leaf classes vs the reference's own (bit-identical audio, against
their stored outputs: tests/reference_outputs.py), strict vs the reference's -ffast-math flags (spread must sit far inside
the 1e-4 parity gate, SURVEY.md §7.5), threaded == single-threaded, streaming pushes == one push, and basic signal sanity
(the 1 kHz AM tone comes out)."""
import numpy as np
import pytest

import oracle_py as op
import reference_outputs as ro
from airband_b200 import workloads as wl
from cases import CASES


def audio_close(a, b, tol=1e-4):
    return np.all(np.abs(a - b) <= tol * np.maximum(1.0, np.maximum(np.abs(a), np.abs(b))))


@pytest.mark.parametrize("name", list(CASES))
def test_signal_exercises_the_path(name):
    cfg, raws = CASES[name]()
    res, o = op.run_oracle(cfg, raws)
    opened = 0
    for d, (wo, iq, ax) in enumerate(res):
        assert wo.shape[1] > 0 and wo.shape[1] % cfg.wave_batch == 0
        assert np.all(np.abs(wo) <= 1.0)
        for c in range(wo.shape[0]):
            opened += o.stats(d, c).open_count
    assert opened >= 1, "squelch never opened: case does not exercise demodulation"


def pipeline_outputs(name, variant):
    """Per device: waveout, iq_out, axcindicate and every squelch statistic of every channel (as float64, exact)."""
    cfg, raws = CASES[name]()
    res, o = op.run_oracle(cfg, raws, variant)
    out = {}
    for d, (wo, iq, ax) in enumerate(res):
        out.update({f"waveout{d}": wo, f"iq_out{d}": iq, f"axc{d}": ax})
        out[f"stats{d}"] = np.array([[float(getattr(o.stats(d, c), f)) for f, _ in o.stats(d, c)._fields_] for c in range(wo.shape[0])])
    return out


def record_reference(out: dict) -> None:
    """What the original leaf classes compute for every case (tests/golden/make_golden.py)."""
    for name in CASES:
        ro.record(out, f"pipeline/{name}", pipeline_outputs(name, "ref"))


@pytest.mark.parametrize("name", list(CASES))
def test_restated_equals_reference_leaf(name):
    ro.check(f"pipeline/{name}", pipeline_outputs(name, "restated"))


@pytest.mark.parametrize("name", ["am_u8", "nfm_s16", "am_bw_f32"])
def test_fast_math_spread_is_inside_gate(name):
    cfg, raws = CASES[name]()
    ra, _ = op.run_oracle(cfg, raws, "restated")
    rb, _ = op.run_oracle(cfg, raws, "restated_fast")
    for (wa, ia, xa), (wb, ib, xb) in zip(ra, rb):
        assert np.array_equal(xa, xb)
        assert audio_close(wa, wb, 1e-4), float(np.abs(wa - wb).max())


def test_threads_and_streaming_equal_oneshot():
    cfg, raws = CASES["s8_two_devices"]()
    ra, _ = op.run_oracle(cfg, raws, n_threads=1)
    rb, _ = op.run_oracle(cfg, raws, n_threads=2)
    o = op.Oracle(cfg)
    rng = np.random.default_rng(0)
    pos = [0, 0]
    while any(pos[d] < raws[d].size for d in range(2)):
        for d in range(2):
            step = int(rng.integers(1, 200000)) * 2 * (1 if cfg.devices[d].bytes_per_sample else 1)
            o.push(d, raws[d][pos[d]:pos[d] + step])
            pos[d] += step
        o.run()
    rc = [o.fetch_all(d) for d in range(2)]
    for a, b, c in zip(ra, rb, rc):
        for x, y, z in zip(a, b, c):
            assert np.array_equal(x, y) and np.array_equal(x, z)


def test_am_tone_recovered():
    cfg = wl.cfg1()
    n = wl.samples_for_batches(cfg, 0, 6)
    raw = wl.synth_iq(cfg, 0, n, key_off_s=0.0)  # carrier always on, 60 % AM at 1 kHz
    (wo, _, ax), o = op.run_oracle(cfg, [raw])[0][0], None
    a = wo[0, 3000:6000].astype(np.float64)  # after the squelch has opened and AGC settled
    spec = np.abs(np.fft.rfft(a * np.hanning(a.size)))
    f = np.fft.rfftfreq(a.size, 1 / 8000.0)
    assert abs(f[np.argmax(spec[5:]) + 5] - 1000.0) < 10.0
    assert 0.2 < np.abs(a).max() < 0.8  # (wavein-agc)/(1.5 agc) with 60 % depth -> 0.4
    assert np.all(ax == ord('*'))
