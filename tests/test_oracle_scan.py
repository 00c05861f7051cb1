"""Scan mode of the oracle (reference: freqlist[] / freq_idx, src/rtl_airband.h:223-233,250-252; controller_thread
src/rtl_airband.cpp:101-139; fparms picked per batch, :498): every frequency-list entry owns its Squelch, filters,
AGC and counters, the channel keeps its waveform history."""
import numpy as np
import pytest

import oracle_py as op
import reference_outputs as ro
from airband_b200 import config as cm
from airband_b200 import workloads as wl


def _setup():
    sr, n, w, cf = 2560000, 1024, 16000, 120000000
    f0 = cf + 250000
    base = cm.make_channel(f0, cf, sr, n, w, modulation=cm.MOD_NFM, bandwidth=6000, squelch_dbfs=-35.0)
    freqs = [
        cm.make_channel(f0, cf, sr, n, w, modulation=cm.MOD_AM, bandwidth=6000, squelch_dbfs=-35.0),
        cm.make_channel(f0, cf, sr, n, w, modulation=cm.MOD_AM, bandwidth=6000, ampfactor=2.5, notch_hz=1000.0, squelch_snr_db=6.0),
        cm.make_channel(f0, cf, sr, n, w, modulation=cm.MOD_NFM, bandwidth=6000, squelch_dbfs=-35.0, ctcss_hz=100.0, ampfactor=1.5),
    ]
    base.synth_ctcss_hz = 100.0  # the synthetic FM signal carries the sub-tone entry 2 listens for
    cfg = cm.Config(fft_size=n, wave_rate=w, devices=[cm.Device(sample_rate=sr, sfmt=cm.SFMT_S16, centerfreq=cf, channels=[base])])
    return cfg, freqs


def _run(cfg, freqs, visits, raw, variant, nb=4, configure=True):
    o = op.Oracle(cfg, variant)
    if configure:
        o.scan_configure(0, 0, freqs)
    out, ax, stats, pos = [], [], [], 0
    for k, idx in enumerate(visits):
        need = wl.samples_for_batches(cfg, 0, nb * (k + 1)) * 2
        if configure:
            o.scan_select(0, 0, idx)
        o.push(0, raw[pos:need])
        pos = need
        assert o.run(nb) == nb
        w_, _, a_ = o.fetch_all(0)
        out.append(w_); ax.append(a_)
        s = o.stats(0, 0)
        stats.append((s.open_count, s.active_counter, s.ctcss_count + s.no_ctcss_count))
    o.close()
    return np.concatenate(out, 1), np.concatenate(ax, 0), stats


def single_entry_outputs(variant):
    cfg, freqs = _setup()
    raw = wl.synth_iq(cfg, 0, wl.samples_for_batches(cfg, 0, 12), key_on_s=1.2, key_off_s=0.2, amplitude=0.2)
    plain_cfg = cm.Config(fft_size=cfg.fft_size, wave_rate=cfg.wave_rate,
                          devices=[cm.Device(sample_rate=2560000, sfmt=cm.SFMT_S16, centerfreq=120000000, channels=[freqs[0]])])
    a, xa, _ = _run(plain_cfg, freqs, [0, 0, 0], raw, variant, configure=False)
    b, xb, _ = _run(cfg, [freqs[0]], [0, 0, 0], raw, variant)
    c, xc, _ = _run(cfg, freqs, [0, 0, 0], raw, variant)        # other entries exist but are never selected
    return {"plain": a, "plain_axc": xa, "single": b, "single_axc": xb, "unselected": c, "unselected_axc": xc}


@pytest.mark.parametrize("variant", ["restated", "ref"])
def test_single_entry_list_is_the_plain_channel(variant):
    # "ref": the restated runs must also equal, bit for bit, what the original leaf classes computed in them (stored)
    out = single_entry_outputs("restated")
    if variant == "ref":
        ro.check("scan_single_entry", out)
    a, xa, b, xb, c, xc = (out[k] for k in ("plain", "plain_axc", "single", "single_axc", "unselected", "unselected_axc"))
    assert np.array_equal(a.view(np.uint32), b.view(np.uint32)) and np.array_equal(xa, xb)
    assert np.array_equal(a.view(np.uint32), c.view(np.uint32)) and np.array_equal(xa, xc)


def test_entries_keep_their_own_state():
    cfg, freqs = _setup()
    visits = [0, 1, 2, 1, 0, 2, 2, 0]
    raw = wl.synth_iq(cfg, 0, wl.samples_for_batches(cfg, 0, 4 * len(visits)), key_on_s=1.2, key_off_s=0.2, amplitude=0.2)
    w_, ax, stats = _run(cfg, freqs, visits, raw, "restated")
    assert np.all(np.abs(w_) <= 2.5) and (ax != ord(' ')).any(), "no entry ever opened: the case does not exercise scan mode"
    # counters reported after each visit belong to the visited entry and never go backwards for that entry
    last = {}
    for idx, st in zip(visits, stats):
        if idx in last:
            assert all(x >= y for x, y in zip(st, last[idx])), (idx, st, last[idx])
        last[idx] = st
    assert last[2][2] > 0, "the NFM entry never evaluated a CTCSS window"
    assert last[0][2] == 0 and last[1][2] == 0, "CTCSS counters leaked into entries without a tone"
    # a different visiting order is a different result (the entries really differ)
    w2, _, _ = _run(cfg, freqs, [1] * len(visits), raw, "restated")
    assert not np.array_equal(w_, w2)


def scan_outputs(variant):
    cfg, freqs = _setup()
    visits = [0, 1, 2, 1, 0, 2, 2, 0]
    raw = wl.synth_iq(cfg, 0, wl.samples_for_batches(cfg, 0, 4 * len(visits)), key_on_s=1.2, key_off_s=0.2, amplitude=0.2)
    w_, ax, stats = _run(cfg, freqs, visits, raw, variant)
    return {"waveout": w_, "axc": ax, "stats": np.array(stats, np.int64)}


def record_reference(out: dict) -> None:
    """What the original leaf classes compute in scan mode (tests/golden/make_golden.py)."""
    ro.record(out, "scan", scan_outputs("ref"))
    ro.record(out, "scan_single_entry", single_entry_outputs("ref"))


def test_scan_restated_equals_reference_leaf():
    ro.check("scan", scan_outputs("restated"))
