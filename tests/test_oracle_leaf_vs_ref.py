"""Pins the restated leaf DSP (oracle/leaf_dsp.cpp) against the original project's own squelch.cpp / ctcss.cpp /
filters.cpp: identical inputs must give bit-identical traces.  What the original classes computed on these inputs is stored
in tests/golden/reference_leaf.npz (tests/reference_outputs.py; made by tests/golden/make_golden.py)."""
import numpy as np
import pytest

import oracle_py as op
import reference_outputs as ro

SQUELCH_MODES = ["auto", "manual", "snr0", "snr20"]
SQUELCH_SEEDS = [1, 2, 3]
NOTCH = [(8000, 100.0, 10.0), (16000, 100.0, 10.0), (8000, 123.0, 5.0), (16000, 254.1, 20.0)]
LOWPASS = [(8000, 2500.0), (16000, 2500.0), (16000, 6250.0), (8000, 1000.0)]
CTCSS_RATES = [8000, 16000]
CTCSS_TONES = [67.0, 100.0, 151.4, 254.1, 88.0]


def keyed_levels(n, seed, lo=0.05, hi=0.75, jitter=0.3):
    rng = np.random.default_rng(seed)
    x = np.empty(n, np.float32)
    i = 0
    on = False
    while i < n:
        seg = int(rng.integers(50, 3000))
        base = hi if on else lo
        x[i:i + seg] = base * (1.0 + jitter * rng.standard_normal(min(seg, n - i)))
        i += seg
        on = not on
    return np.abs(x).astype(np.float32)


def squelch_trace(mode, seed, variant):
    raw = keyed_levels(60000, seed)
    # a filtered stream that sometimes falls below the buffered pre-filter level (exercises the post-filter path)
    rng = np.random.default_rng(100 + seed)
    filt = (raw * rng.uniform(0.3, 1.2, raw.size)).astype(np.float32)
    audio = (0.2 * np.sin(2 * np.pi * 100.0 * np.arange(raw.size) / 8000.0)).astype(np.float32)
    s = op.SquelchHarness(variant)
    if mode == "manual":
        s.set_level(0.3)
    elif mode == "snr0":
        s.set_snr(0.0)
    elif mode == "snr20":
        s.set_snr(20.0)
    if seed == 2:
        s.set_ctcss(100.0, 8000.0)
    use_filt = filt if seed != 1 else None
    levels, flags = s.trace(raw, use_filt, audio)
    counts = np.array([s.open_count(), s.flappy_count(), s.ctcss_count(), s.no_ctcss_count()], np.int64)
    return {"levels": levels, "flags": flags, "counts": counts}


def notch(rate, freq, q, variant):
    x = np.random.default_rng(5).standard_normal(20000).astype(np.float32) * 0.3
    return {"out": op.notch_run(freq, rate, q, x, variant)}


def lowpass(rate, freq, variant):
    rng = np.random.default_rng(6)
    x = (rng.standard_normal(20000) + 1j * rng.standard_normal(20000)).astype(np.complex64)
    return {"out": op.lowpass_run(freq, rate, x, variant)}


def ctcss(rate, tone, variant):
    n = int(rate * 0.4) * 3 + 17
    rng = np.random.default_rng(7)
    x = (0.2 * np.sin(2 * np.pi * tone * np.arange(n) / rate) + 0.02 * rng.standard_normal(n)).astype(np.float32)
    res = {}
    for win in (int(rate * 0.05), int(rate * 0.4)):
        c = op.CtcssHarness(tone, rate, win, variant)
        seq = []
        for v in x:
            c.sample(float(v))
            seq.append((c.enough(), c.has_tone()))
        res[f"seq{win}"] = np.array(seq, np.uint8)
        res[f"counts{win}"] = np.array([c.L.abo_ctcss_found(c.c), c.L.abo_ctcss_not_found(c.c)], np.int64)
    return res


def record_reference(out: dict) -> None:
    """What the original classes compute for every case above (tests/golden/make_golden.py)."""
    for mode in SQUELCH_MODES:
        for seed in SQUELCH_SEEDS:
            ro.record(out, f"squelch/{mode}/{seed}", squelch_trace(mode, seed, "ref"))
    for rate, freq, q in NOTCH:
        ro.record(out, f"notch/{rate}/{freq}/{q}", notch(rate, freq, q, "ref"))
    for rate, freq in LOWPASS:
        ro.record(out, f"lowpass/{rate}/{freq}", lowpass(rate, freq, "ref"))
    for rate in CTCSS_RATES:
        for tone in CTCSS_TONES:
            ro.record(out, f"ctcss/{rate}/{tone}", ctcss(rate, tone, "ref"))


@pytest.mark.parametrize("mode", SQUELCH_MODES)
@pytest.mark.parametrize("seed", SQUELCH_SEEDS)
def test_squelch_trace_bit_identical(mode, seed):
    got = squelch_trace(mode, seed, "restated")
    ro.check(f"squelch/{mode}/{seed}", got)
    assert got["flags"].max() > 0, "trace never opened — test signal is not exercising the state machine"


@pytest.mark.parametrize("rate,freq,q", NOTCH)
def test_notch_bit_identical(rate, freq, q):
    got = notch(rate, freq, q, "restated")
    ro.check(f"notch/{rate}/{freq}/{q}", got)
    assert np.abs(got["out"]).max() > 0


@pytest.mark.parametrize("rate,freq", LOWPASS)
def test_lowpass_bit_identical(rate, freq):
    ro.check(f"lowpass/{rate}/{freq}", lowpass(rate, freq, "restated"))


@pytest.mark.parametrize("rate", CTCSS_RATES)
@pytest.mark.parametrize("tone", CTCSS_TONES)
def test_ctcss_bit_identical(rate, tone):
    ro.check(f"ctcss/{rate}/{tone}", ctcss(rate, tone, "restated"))
