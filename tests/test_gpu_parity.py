"""GPU parity tests proper (-m gpu): the CUDA path, driven through the C ABI, against the CPU oracle on the same
seeded inputs, and against the committed golden fixtures.
Gate (BASELINE.md §3): per audio sample |gpu - oracle| <= 1e-4 * max(1, |gpu|, |oracle|) — float32 path, tolerance
1e-4 as north_star states — plus identical squelch decisions (axcindicate per batch, open/flap/CTCSS counters)."""
import os

import numpy as np
import pytest

import oracle_py as op
import reference_outputs as ro
from airband_b200 import config as cm
from airband_b200 import lib
from airband_b200 import workloads as wl
from cases import CASES

pytestmark = pytest.mark.gpu
TOL = 1e-4


def gate(a, b, tol=TOL):
    a = np.asarray(a); b = np.asarray(b)
    err = np.abs(a - b) / np.maximum(1.0, np.maximum(np.abs(a), np.abs(b)))
    return float(err.max()) if err.size else 0.0


def compare(cfg, raws, gres, geng, ores, oorc, tol=TOL):
    for d in range(len(raws)):
        gw, gi, ga = gres[d]
        ow, oi, oa = ores[d]
        assert gw.shape == ow.shape, (gw.shape, ow.shape)
        assert np.array_equal(ga, oa), f"axcindicate differs on device {d}"
        assert gate(gw, ow) <= tol, f"audio dev {d}: {gate(gw, ow)}"
        assert gate(gi.real, oi.real) <= tol and gate(gi.imag, oi.imag) <= tol, f"iq_out dev {d}"
        for c in range(gw.shape[0]):
            gs, os_ = geng.stats(d, c), oorc.stats(d, c)
            for f in ("open_count", "flappy_count", "ctcss_count", "no_ctcss_count", "active_counter", "dm_phi", "bin"):
                assert getattr(gs, f) == getattr(os_, f), (d, c, f, getattr(gs, f), getattr(os_, f))
            for f in ("noise_level", "signal_level", "squelch_level", "agcavgfast"):
                a, b = getattr(gs, f), getattr(os_, f)
                assert abs(a - b) <= 1e-4 * max(1.0, abs(a), abs(b)), (d, c, f, a, b)


@pytest.mark.parametrize("fft_mode", [1, 2], ids=["full_fft", "pruned_fft"])
@pytest.mark.parametrize("name", list(CASES))
def test_case_matches_oracle(name, fft_mode):
    cfg, raws = CASES[name]()
    ores, oorc = op.run_oracle(cfg, raws)
    gres, geng = lib.demodulate_all(cfg, raws, fft_mode=fft_mode)
    compare(cfg, raws, gres, geng, ores, oorc)


@pytest.mark.parametrize("name", ["am_u8", "nfm_s16", "am_bw_f32", "s8_two_devices"])
def test_case_matches_golden_fixture(name):
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", name + ".npz"))
    cfg, raws = CASES[name]()
    for d, r in enumerate(raws):
        assert ro.digest(r) == str(g[f"raw{d}_sha256"]), "seeded generator no longer reproduces the stored input"
    gres, geng = lib.demodulate_all(cfg, raws)
    for d, (gw, gi, ga) in enumerate(gres):
        assert np.array_equal(ga, g[f"axc{d}"])
        assert gate(gw, g[f"waveout{d}"]) <= TOL
        assert gate(gi.real, g[f"iq_out{d}"].real) <= TOL and gate(gi.imag, g[f"iq_out{d}"].imag) <= TOL
        for c in range(gw.shape[0]):
            s = geng.stats(d, c)
            assert [s.open_count, s.flappy_count, s.ctcss_count, s.no_ctcss_count, s.active_counter] == list(g[f"counts{d}"][c])


@pytest.mark.parametrize("n", [256, 512, 1024, 2048, 4096, 8192])
@pytest.mark.parametrize("sfmt", [cm.SFMT_U8, cm.SFMT_S8, cm.SFMT_S16, cm.SFMT_F32])
def test_fft_stage_every_size_and_format(n, sfmt):
    """conversion + window + FFT of one frame, full spectrum, vs the oracle's fftin->fftout for the same bytes."""
    sr = 2560000
    cfg = cm.Config(fft_size=n, wave_rate=8000,
                    devices=[cm.Device(sample_rate=sr, sfmt=sfmt, centerfreq=0, channels=[cm.make_channel(100000, 0, sr, n, 8000)])])
    raw = wl.synth_iq(cfg, 0, n, key_off_s=0.0, seed=n + sfmt, amplitude=0.3, noise_sigma=0.05)
    o = op.Oracle(cfg)
    _, ospec = o.debug_frame(0, raw)
    e = lib.Engine(cfg)
    gspec = e.debug_frame(0, raw)
    scale = np.abs(ospec).max()
    assert scale > 1.0
    assert np.abs(gspec - ospec).max() / scale < 2e-6
    # and against float64 numpy on the oracle's own float32 input (independent of the oracle's FFT)
    fin, _ = o.debug_frame(0, raw)
    ref = np.fft.fft(fin.astype(np.complex128))
    assert np.abs(gspec - ref).max() / np.abs(ref).max() < 2e-6


@pytest.mark.parametrize("nbmax", [1, 2, 4])
def test_batches_per_run_do_not_change_results(nbmax):
    cfg, raws = CASES["s8_two_devices"](n_batches=4)
    ores, oorc = op.run_oracle(cfg, raws)
    gres, geng = lib.demodulate_all(cfg, raws, max_batches_per_run=nbmax)
    compare(cfg, raws, gres, geng, ores, oorc)


def test_streaming_pushes_of_odd_sizes():
    cfg, raws = CASES["am_u8"](n_batches=4)
    ores, oorc = op.run_oracle(cfg, raws)
    e = lib.Engine(cfg, max_batches_per_run=2, input_capacity_batches=3)
    rng = np.random.default_rng(3)
    pos, outs = 0, []
    r = raws[0]
    while pos < r.size or e.batches_available(0) > 0:
        if pos < r.size:
            step = 2 * int(rng.integers(1, 90000))
            e.push(0, r[pos:pos + step])
            pos += step
        e.run(-1)
        while True:
            got = e.fetch(0)
            if got is None:
                break
            outs.append(got)
    gw = np.concatenate([x[0] for x in outs], 1)
    assert gw.shape == ores[0][0].shape
    assert gate(gw, ores[0][0]) <= TOL
    assert np.array_equal(np.stack([x[2] for x in outs]), ores[0][2])


def _small(cfg, nb, fft_modes=(1, 2), **kw):
    raws = [wl.synth_iq(cfg, d, wl.samples_for_batches(cfg, d, nb), key_on_s=0.2, key_off_s=0.1, **kw) for d in range(len(cfg.devices))]
    ores, oorc = op.run_oracle(cfg, raws)
    for mode in fft_modes:  # 1 = full-spectrum kernel, 2 = output-pruned kernel
        gres, geng = lib.demodulate_all(cfg, raws, fft_mode=mode)
        compare(cfg, raws, gres, geng, ores, oorc)
        geng.close()


def test_cfg1_shape():
    _small(wl.cfg1(two_channels=True), 5)


def test_cfg2_shape_scaled_down():
    _small(wl.cfg2(n_devices=3, n_channels=8), 3)


@pytest.mark.parametrize("sfmt", [cm.SFMT_S16, cm.SFMT_F32])
def test_cfg3_shape_scaled_down(sfmt):
    _small(wl.cfg3(n_devices=1, n_channels=6, sfmt=sfmt, parity=True), 4)


def test_cfg5_shape_scaled_down():
    _small(wl.cfg5(n_devices=5, n_channels=8), 2)


@pytest.mark.parametrize("n", [256, 1024, 8192])
def test_other_fft_sizes_end_to_end(n):
    _small(wl.cfg2(n_devices=1, n_channels=4, fft_size=n), 2)


def test_many_channels_per_device():
    """49 channels on one device (config/big_mixer.conf has 49): exercises the pruned kernel's R1=16 path and its
    32-channel passes."""
    _small(wl.cfg2(n_devices=1, n_channels=49, fft_size=1024), 2)


@pytest.mark.parametrize("n,sfmt", [(4096, cm.SFMT_F32), (512, cm.SFMT_S8), (2048, cm.SFMT_S16)])
def test_pruned_equals_full_spectrum_bins(n, sfmt):
    """The two K1 kernels must agree on the extracted bins far inside the audio gate (same inputs, 2 batches)."""
    sr = 2560000
    chans = [cm.make_channel(o, 0, sr, n, 8000, squelch_dbfs=-30.0, rawfile=True) for o in (-600000, -25000, 12500, 333000, 910000)]
    cfg = cm.Config(fft_size=n, wave_rate=8000, devices=[cm.Device(sample_rate=sr, sfmt=sfmt, centerfreq=0, channels=chans)])
    raws = [wl.synth_iq(cfg, 0, wl.samples_for_batches(cfg, 0, 2), key_off_s=0.0, amplitude=0.1)]
    (fw, fi, fa), e1 = lib.demodulate_all(cfg, raws, fft_mode=1)[0][0], None
    (pw, pi, pa), e2 = lib.demodulate_all(cfg, raws, fft_mode=2)[0][0], None
    assert np.array_equal(fa, pa) and np.any(fa == ord('*'))
    scale = np.abs(fi).max()
    assert scale > 1.0 and np.abs(fi - pi).max() / scale < 3e-6
    assert gate(fw, pw) <= 1e-5


def test_mixer_matches_reference_sum():
    """cfg 4 shape: mixer m = sum over devices of channel m (reference src/mixer.cpp:133-140,189-214), mono and stereo."""
    cfg = wl.cfg4()
    nb = 3
    raws = [wl.synth_iq(cfg, d, wl.samples_for_batches(cfg, d, nb), key_on_s=0.2, key_off_s=0.1) for d in range(len(cfg.devices))]
    ores, _ = op.run_oracle(cfg, raws)
    e = lib.Engine(cfg, max_batches_per_run=2)
    mixers = [[(d, m, 1.0 + 0.25 * d, (-0.5 if (m == 1 and d == 0) else 0.0)) for d in range(len(cfg.devices))] for m in range(4)]
    e.configure_mixers(mixers)
    for d, r in enumerate(raws):
        e.push(d, r)
    got = {m: [] for m in range(4)}
    while e.run(-1) > 0:
        for d in range(len(raws)):
            while e.fetch(d) is not None:
                pass
        for m in range(4):
            while True:
                r = e.fetch_mixer(m)
                if r is None:
                    break
                got[m].append(r)
    B = cfg.wave_batch
    for m in range(4):
        assert len(got[m]) == nb
        for b in range(nb):
            left = np.zeros(B, np.float32); right = np.zeros(B, np.float32); sig = False
            for (d, c, amp, bal) in mixers[m]:
                wo, _, ax = ores[d]
                if ax[b, c] == ord(' '):
                    continue
                sig = True
                ampl, ampr = np.float32(min(1.0, 1.0 - bal)), np.float32(min(1.0, 1.0 + bal))
                x = wo[c, b * B:(b + 1) * B]
                left = (left + x * (np.float32(amp) * ampl)).astype(np.float32)
                right = (right + x * (np.float32(amp) * ampr)).astype(np.float32)
            gl, gr, gs = got[m][b]
            assert gs == sig
            assert gate(gl, left) <= TOL and gate(gr, right) <= TOL


def test_afc_follows_an_off_bin_carrier():
    """AFC (reference src/rtl_airband.cpp:180-251): carrier 3 bins above the configured one; the bin must move up on the
    squelch-open edge exactly as in the oracle, batch by batch."""
    sr, n, w, cf = 2560000, 512, 8000, 120000000
    ch = cm.make_channel(cf + 100000, cf, sr, n, w, squelch_dbfs=-40.0, afc=2)
    ch.offset_hz = 100000.0 + 3 * (sr / n)  # transmit 3 bins high
    cfg = cm.Config(fft_size=n, wave_rate=w, devices=[cm.Device(sample_rate=sr, sfmt=cm.SFMT_U8, centerfreq=cf, channels=[ch])])
    raws = [wl.synth_iq(cfg, 0, wl.samples_for_batches(cfg, 0, 5), key_on_s=0.25, key_off_s=0.15, amplitude=0.3)]
    ores, oorc = op.run_oracle(cfg, raws)
    gres, geng = lib.demodulate_all(cfg, raws, max_batches_per_run=1)
    assert np.any(ores[0][2] == ord('>')) or np.any(ores[0][2] == ord('<')), "oracle AFC never moved: case is not exercising AFC"
    compare(cfg, raws, gres, geng, ores, oorc)


def test_host_adapter_thread_function_matches_oracle():
    """demodulate_b200() (the reference's demod thread contract: input rings with wrap tail, locking, waveavail +
    Signal hand-shake) over the C ABI, fed like file_rx_thread() feeds it, vs the oracle on the same bytes.  The stream is
    longer than one ring (2.56 MB) so the ring wraps."""
    from airband_b200 import host
    cfg, _ = CASES["s8_two_devices"]()
    nb = 7
    raws = [wl.synth_iq(cfg, d, wl.samples_for_batches(cfg, d, nb), key_on_s=0.2, key_off_s=0.1) for d in range(2)]
    assert raws[1].nbytes > 2560000  # more than one ring (MIN_BUF_SIZE): the ring wraps
    ores, oorc = op.run_oracle(cfg, raws)
    hres = host.run_host_pipeline(cfg, raws)
    for d in range(2):
        gw, gi, ga, info = hres[d]
        ow, oi, oa = ores[d]
        assert gw.shape == ow.shape and np.array_equal(ga, oa)
        assert gate(gw, ow) <= TOL
        assert info["overflows"] == 0 and info["overruns"] == 0
        assert info["active"] == [int(np.sum(oa[:, c] != ord(' '))) for c in range(ow.shape[0])]


def test_bulk_fetch_equals_single_fetches():
    cfg, raws = CASES["am_u8"](n_batches=4)
    e1 = lib.Engine(cfg, max_batches_per_run=4)
    e2 = lib.Engine(cfg, max_batches_per_run=4)
    for e in (e1, e2):
        e.push(0, raws[0])
        assert e.run(-1) == 4
    singles = [e1.fetch(0) for _ in range(4)]
    C = len(cfg.devices[0].channels)
    wo = np.empty((4, C, cfg.wave_batch), np.float32)
    ax = np.empty((4, C), np.uint8)
    assert e2.fetch_many_into(0, 8, wo, ax) == 4 and e2.fetch(0) is None
    for b in range(4):
        assert np.array_equal(wo[b], singles[b][0]) and np.array_equal(ax[b], singles[b][2])


def test_error_codes():
    """Error behaviour of the C ABI mirrors the reference's engine branch: message + negative code, no exceptions cross."""
    cfg = wl.cfg1()
    bad = cm.Config(fft_size=300, wave_rate=8000, devices=cfg.devices)
    with pytest.raises(lib.AbgError) as ei:
        lib.Engine(bad)
    assert ei.value.code == -2 and "not supported" in str(ei.value)
    e = lib.Engine(cfg, max_batches_per_run=1, input_capacity_batches=1)
    with pytest.raises(lib.AbgError) as ei:
        e.push(5, np.zeros(16, np.uint8))
    assert ei.value.code == -5
    with pytest.raises(lib.AbgError) as ei:
        e.push(0, np.zeros(3, np.uint8))  # not a whole number of complex samples
    assert ei.value.code == -2
    big = np.zeros(2 * 320 * 1000 * 4, np.uint8)  # four batches into a one-batch buffer
    with pytest.raises(lib.AbgError) as ei:
        e.push(0, big)
    assert ei.value.code == -6
    assert e.fetch(0) is None and e.run(-1) == 0


def _scan_setup():
    """One scan device (one channel, rtl_airband.h:265 R_SCAN) with three freqlist[] entries that differ in everything a
    freq_t owns: manual-squelch AM, auto-squelch AM with another ampfactor and a notch, NFM with CTCSS."""
    sr, n, w, cf = 2560000, 1024, 16000, 120000000
    f0 = cf + 250000
    base = cm.make_channel(f0, cf, sr, n, w, modulation=cm.MOD_NFM, bandwidth=6000, squelch_dbfs=-35.0)   # needs_raw_iq as scan+NFM builds have
    freqs = [
        cm.make_channel(f0, cf, sr, n, w, modulation=cm.MOD_AM, bandwidth=6000, squelch_dbfs=-35.0),
        cm.make_channel(f0, cf, sr, n, w, modulation=cm.MOD_AM, bandwidth=6000, ampfactor=2.5, notch_hz=1000.0, squelch_snr_db=6.0),
        cm.make_channel(f0, cf, sr, n, w, modulation=cm.MOD_NFM, bandwidth=6000, squelch_dbfs=-35.0, ctcss_hz=100.0, ampfactor=1.5),
    ]
    base.synth_ctcss_hz = 100.0  # the synthetic FM signal carries the sub-tone entry 2 listens for
    cfg = cm.Config(fft_size=n, wave_rate=w, devices=[cm.Device(sample_rate=sr, sfmt=cm.SFMT_S16, centerfreq=cf, channels=[base])])
    return cfg, freqs


def test_scan_mode_frequency_list_matches_oracle():
    """controller_thread switches freq_idx between batches (rtl_airband.cpp:117-119,498); every entry keeps its own
    Squelch / filters / AGC / counters across visits."""
    cfg, freqs = _scan_setup()
    nb_per_visit, visits = 4, [0, 1, 2, 1, 0, 2, 2, 0]
    total = nb_per_visit * len(visits)
    raw = wl.synth_iq(cfg, 0, wl.samples_for_batches(cfg, 0, total), key_on_s=1.2, key_off_s=0.2, amplitude=0.2)
    hop = cfg.hop(0)
    B = cfg.wave_batch
    o = op.Oracle(cfg)
    e = lib.Engine(cfg, max_batches_per_run=nb_per_visit, input_capacity_batches=2 * nb_per_visit + 1)
    o.scan_configure(0, 0, freqs)
    e.scan_configure(0, 0, freqs)
    pos = 0
    for k, idx in enumerate(visits):
        need = wl.samples_for_batches(cfg, 0, nb_per_visit * (k + 1)) * 2    # items (I and Q) needed up to the end of this visit
        chunk = raw[pos:need]
        pos = need
        o.scan_select(0, 0, idx)
        e.scan_select(0, 0, idx)
        o.push(0, chunk)
        e.push(0, chunk)
        assert o.run(nb_per_visit) == nb_per_visit
        assert e.run(nb_per_visit) == nb_per_visit
        ow, oi, oa = o.fetch_all(0)
        outs = [e.fetch(0) for _ in range(nb_per_visit)]
        gw = np.concatenate([x[0] for x in outs], 1)
        ga = np.stack([x[2] for x in outs])
        assert gw.shape == ow.shape == (1, nb_per_visit * B)
        assert np.array_equal(ga, oa), (k, idx)
        assert gate(gw, ow) <= TOL, (k, idx, gate(gw, ow))
        gs, os_ = e.stats(0, 0), o.stats(0, 0)      # getters of the CURRENT entry
        for f in ("open_count", "flappy_count", "ctcss_count", "no_ctcss_count", "active_counter", "dm_phi"):
            assert getattr(gs, f) == getattr(os_, f), (k, idx, f, getattr(gs, f), getattr(os_, f))
        for f in ("noise_level", "signal_level", "squelch_level", "agcavgfast"):
            a, b = getattr(gs, f), getattr(os_, f)
            assert abs(a - b) <= 1e-4 * max(1.0, abs(a), abs(b)), (k, idx, f, a, b)
    # error behaviour
    with pytest.raises(lib.AbgError):
        e.scan_select(0, 0, 3)
    e.close()
    o.close()


def test_host_adapter_scan_channel_uses_the_selected_entry():
    """demodulate_b200() hands a channel's freqlist[] to the engine and follows channel_t.freq_idx (here fixed to entry 2
    before the thread starts, as controller_thread would have left it)."""
    from airband_b200 import host
    cfg, freqs = _scan_setup()
    nb = 6
    raw = wl.synth_iq(cfg, 0, wl.samples_for_batches(cfg, 0, nb), key_on_s=1.2, key_off_s=0.2, amplitude=0.2)
    o = op.Oracle(cfg)
    o.scan_configure(0, 0, freqs)
    o.scan_select(0, 0, 2)
    o.push(0, raw)
    assert o.run(-1) == nb
    ow, oi, oa = o.fetch_all(0)
    gw, gi, ga, info = host.run_host_pipeline(cfg, [raw], freqlists=[(0, 0, freqs, 2)])[0]
    assert gw.shape == ow.shape and np.array_equal(ga, oa)
    assert gate(gw, ow) <= TOL
    assert info["active"] == [int(np.sum(oa[:, 0] != ord(' ')))]


@pytest.mark.parametrize("speedup", [0.0, 4.0], ids=["lossless", "paced_4x_realtime"])
def test_pattern_input_plugin_through_the_adapter(speedup):
    """The "pattern" input plugin (host/input_pattern.cpp, shape of reference src/input-file.cpp) replays a block into the
    page-locked input rings; demodulate_b200() drains them.  Lossless mode must reproduce the oracle on block x repeat;
    the paced mode (a live SDR never waits) must do so too as long as nothing overflowed."""
    from airband_b200 import host
    cfg, _ = CASES["s8_two_devices"]()
    repeat = 3
    blocks = [wl.synth_iq(cfg, d, 3 * cfg.wave_batch * cfg.hop(d), key_on_s=0.2, key_off_s=0.1) for d in range(2)]
    raws = [np.tile(b, repeat) for b in blocks]
    ores, oorc = op.run_oracle(cfg, raws)
    hres = host.run_host_pipeline(cfg, blocks, pattern=(repeat, speedup))
    for d in range(2):
        gw, gi, ga, info = hres[d]
        ow, oi, oa = ores[d]
        assert info["overflows"] == 0 and info["overruns"] == 0, info
        assert gw.shape == ow.shape and ow.shape[1] >= 7 * cfg.wave_batch
        assert np.array_equal(ga, oa)
        assert gate(gw, ow) <= TOL


def test_full_size_cfg2_properties_and_sampled_oracle_parity():
    """BASELINE.json configs[1] at its FULL size (64 devices x 2.56 Msps U8, fft 2048, 8 AM channels, 4 batches per run),
    checked through properties that do not need the oracle on all 512 channels:
      * devices that receive identical bytes produce bit-identical audio and decisions, wherever they sit in the launch
        (tile / CTA / warp placement must not leak into results);
      * the output-pruned and the full-spectrum K1 agree within the audio gate, with identical squelch decisions;
      * one run of 4 batches == 4 runs of 1 batch, bit for bit;
    plus the oracle itself on a sample of the devices (one per distinct stream)."""
    import bench
    cfg, _ = bench.make_workload("cfg2")
    nb = 4
    raws = bench.synth_streams(cfg, nb, n_unique=4)
    D = len(cfg.devices)
    res, eng = lib.demodulate_all(cfg, raws, max_batches_per_run=nb, fft_mode=2)
    opened = 0
    for d in range(D):
        w, _, a = res[d]
        assert w.shape == (8, nb * cfg.wave_batch)
        w0, _, a0 = res[d % 4]
        assert np.array_equal(w.view(np.uint32), w0.view(np.uint32)) and np.array_equal(a, a0), f"device {d} differs from its twin {d % 4}"
        opened += int((a != ord(' ')).sum())
    assert opened > 0
    res_full, eng_full = lib.demodulate_all(cfg, raws, max_batches_per_run=nb, fft_mode=1)
    res_one, eng_one = lib.demodulate_all(cfg, raws, max_batches_per_run=1, fft_mode=2)
    for d in range(D):
        assert np.array_equal(res[d][2], res_full[d][2])
        assert gate(res[d][0], res_full[d][0]) <= TOL
        assert np.array_equal(res[d][0].view(np.uint32), res_one[d][0].view(np.uint32)) and np.array_equal(res[d][2], res_one[d][2])
    # the oracle on one device per distinct stream (channel plans are identical across devices)
    sub = cm.Config(fft_size=cfg.fft_size, wave_rate=cfg.wave_rate, devices=cfg.devices[:4])
    ores, oorc = op.run_oracle(sub, raws[:4])
    for d in range(4):
        ow, _, oa = ores[d]
        assert np.array_equal(res[d][2], oa)
        assert gate(res[d][0], ow) <= TOL
        for c in range(8):
            gs, os_ = eng.stats(d, c), oorc.stats(d, c)
            assert gs.open_count == os_.open_count and gs.active_counter == os_.active_counter
    for e in (eng, eng_full, eng_one):
        e.close()


@pytest.mark.parametrize("lpw", [2, 4, 32])
@pytest.mark.parametrize("name", ["am_u8", "nfm_s16", "am_bw_f32", "s8_two_devices", "uneven_devices"])
def test_channels_per_warp_variants_match_oracle(name, lpw, monkeypatch):
    """K2 is compiled for 1, 2, 4, 8, 16 and 32 channels per warp and the engine picks by channel count (more than 592
    channels -> several per warp), which the small cases never reach: force the wide variants.  `uneven_devices` feeds
    the two devices of one warp different numbers of batches, so some runs advance only one of them."""
    monkeypatch.setenv("ABG_K2_LPW", str(lpw))
    if name == "uneven_devices":
        cfg, _ = CASES["s8_two_devices"]()
        raws = [wl.synth_iq(cfg, i, wl.samples_for_batches(cfg, i, nb), key_on_s=0.1, key_off_s=0.05) for i, nb in enumerate((2, 5))]
    else:
        cfg, raws = CASES[name]()
    ores, oorc = op.run_oracle(cfg, raws)
    gres, geng = lib.demodulate_all(cfg, raws, max_batches_per_run=2)
    compare(cfg, raws, gres, geng, ores, oorc)
    geng.close()


def test_set_bin_moves_a_channel_between_runs():
    """abg_set_bin (what a retune does to dev->bins[] / base_bins[]): channel 0 is moved onto channel 1's bin after two
    batches and back after four; the oracle gets the same calls at the same batch boundaries."""
    cfg, _ = CASES["am_u8"]()
    nb_total = 6
    raw = wl.synth_iq(cfg, 0, wl.samples_for_batches(cfg, 0, nb_total), key_on_s=0.11, key_off_s=0.07, amplitude=0.2)
    b0, b1 = cfg.devices[0].channels[0].bin, cfg.devices[0].channels[1].bin
    o = op.Oracle(cfg)
    e = lib.Engine(cfg, max_batches_per_run=2, input_capacity_batches=5)
    pos = 0
    for k, new_bin in enumerate((None, b1, b0)):
        need = wl.samples_for_batches(cfg, 0, 2 * (k + 1)) * 2
        if new_bin is not None:
            o.set_bin(0, 0, new_bin)
            e.set_bin(0, 0, new_bin)
        o.push(0, raw[pos:need]); e.push(0, raw[pos:need])
        pos = need
        assert o.run(2) == 2 and e.run(2) == 2
        ow, _, oa = o.fetch_all(0)
        outs = [e.fetch(0) for _ in range(2)]
        gw = np.concatenate([x[0] for x in outs], 1)
        assert np.array_equal(np.stack([x[2] for x in outs]), oa), k
        assert gate(gw, ow) <= TOL, (k, gate(gw, ow))
        assert e.stats(0, 0).bin == o.stats(0, 0).bin == (new_bin if new_bin is not None else b0)
    e.close(); o.close()


@pytest.mark.parametrize("name,fill", [("am_u8", 127), ("am_u8", 0), ("am_bw_f32", 0.0), ("nfm_s16", 0)],
                         ids=["u8_midscale", "u8_rail", "f32_zeros", "s16_zeros"])
def test_constant_input_edge_cases(name, fill):
    """Silence and a railed ADC: every frame identical, exact zeros through sqrt / divisions / the squelch estimators
    (F32 and S16 zeros give |X| == 0 everywhere).  Outputs must stay finite and equal the oracle's."""
    cfg, raws = CASES[name]()
    raws = [np.full_like(r, fill) for r in raws]
    ores, oorc = op.run_oracle(cfg, raws)
    gres, geng = lib.demodulate_all(cfg, raws)
    for d in range(len(raws)):
        assert np.isfinite(gres[d][0]).all()
    compare(cfg, raws, gres, geng, ores, oorc)
    geng.close()
