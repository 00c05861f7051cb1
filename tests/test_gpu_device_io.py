"""GPU-resident I/O (-m gpu): IQ pushed from CUDA tensors (abg_push_device) and results kept in HBM
(ABG_RESULTS_DEVICE) and fetched into CUDA tensors on the caller's stream.  Every check compares against the host path
(abg_push + abg_fetch_batch) on the same configuration and bytes, bit for bit: the device path moves the same values and
must not change one."""
import ctypes as C

import numpy as np
import pytest

import oracle_py as op
from airband_b200 import config as cm
from airband_b200 import lib
from airband_b200 import workloads as wl
from cases import CASES
from test_gpu_parity import _scan_setup, compare

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


def _bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint8)


def _equal(a, b):
    return a.shape == b.shape and np.array_equal(_bits(a), _bits(b))


def _stats_bytes(e, cfg):
    out = []
    for d, dv in enumerate(cfg.devices):
        for c in range(len(dv.channels)):
            s = e.stats(d, c)
            out.append(C.string_at(C.addressof(s), C.sizeof(s)))
    return out


def _schedule(cfg, raws, step_b):
    """The chunks lib.demodulate_all pushes: (device, start, stop) per run, in push order."""
    B = cfg.wave_batch
    pos = [0] * len(raws)
    steps = []
    while any(pos[d] < r.size for d, r in enumerate(raws)):
        chunk = []
        for d, r in enumerate(raws):
            if pos[d] < r.size:
                hop_items = cfg.hop(d) * 2
                n = step_b * B * hop_items + (100 * hop_items + 2 * cfg.fft_size if pos[d] == 0 else 0)
                chunk.append((d, pos[d], min(pos[d] + n, r.size)))
                pos[d] += n
        steps.append(chunk)
    return steps


def _tensors(raws):
    return [torch.from_numpy(np.ascontiguousarray(r)).cuda() for r in raws]


class Collect:
    """Per device: lists of waveout [n, C, B], iq_out [n, C, B] (complex), axcindicate [n, C] batches."""

    def __init__(self, cfg):
        self.cfg = cfg
        self.out = [([], [], []) for _ in cfg.devices]

    def host(self, e):
        for d in range(len(self.cfg.devices)):
            while True:
                got = e.fetch(d)
                if got is None:
                    break
                for k in range(3):
                    self.out[d][k].append(got[k][None])

    def device(self, e):
        for d in range(len(self.cfg.devices)):
            wo, iq, ax = e.fetch_tensors(d, 64)
            for k, t in enumerate((wo, iq, ax)):
                self.out[d][k].append(t)

    def arrays(self):
        res = []
        for d, dv in enumerate(self.cfg.devices):
            parts = []
            for k in range(3):
                xs = [x.cpu().numpy() if torch.is_tensor(x) else x for x in self.out[d][k]]
                parts.append(np.concatenate(xs, 0) if xs else None)
            res.append(parts)
        return res

    def as_demodulate_all(self):
        """(waveout[C, n*B], iq_out[C, n*B], axc[n, C]) per device, the layout lib.demodulate_all returns."""
        res = []
        for wo, iq, ax in self.arrays():
            n, Cn, B = wo.shape
            res.append((wo.transpose(1, 0, 2).reshape(Cn, n * B), iq.transpose(1, 0, 2).reshape(Cn, n * B), ax))
        return res


def run_host(cfg, raws, nbmax=4, step_b=None, fft_mode=0, **kw):
    e = lib.Engine(cfg, max_batches_per_run=nbmax, fft_mode=fft_mode, **kw)
    col = Collect(cfg)
    for chunk in _schedule(cfg, raws, step_b or nbmax):
        for d, a, b in chunk:
            e.push(d, raws[d][a:b])
        e.run(-1)
        col.host(e)
    while e.run(-1) > 0:
        col.host(e)
    return col, e


def run_device(cfg, raws, nbmax=4, step_b=None, fft_mode=0, **kw):
    e = lib.Engine(cfg, max_batches_per_run=nbmax, fft_mode=fft_mode, **kw)
    e.results_on_device()
    ts = _tensors(raws)
    col = Collect(cfg)
    for chunk in _schedule(cfg, raws, step_b or nbmax):
        for d, a, b in chunk:
            e.push_tensor(d, ts[d][a:b])
        e.run(-1)
        col.device(e)
    while e.run(-1) > 0:
        col.device(e)
    torch.cuda.synchronize()
    return col, e


def assert_same(cfg, hcol, heng, dcol, deng):
    for d, (h, g) in enumerate(zip(hcol.arrays(), dcol.arrays())):
        for k, what in enumerate(("waveout", "iq_out", "axcindicate")):
            assert _equal(h[k], g[k]), f"device {d}: {what} differs between the host and the device path"
    assert _stats_bytes(heng, cfg) == _stats_bytes(deng, cfg)


@pytest.mark.parametrize("fft_mode", [0, 1, 2, 3])
@pytest.mark.parametrize("name", list(CASES))
def test_device_io_equals_host_path(name, fft_mode):
    cfg, raws = CASES[name]()
    hcol, heng = run_host(cfg, raws, fft_mode=fft_mode)
    dcol, deng = run_device(cfg, raws, fft_mode=fft_mode)
    assert_same(cfg, hcol, heng, dcol, deng)


def test_device_io_matches_oracle():
    cfg, raws = CASES["am_bw_f32"]()
    ores, oorc = op.run_oracle(cfg, raws)
    dcol, deng = run_device(cfg, raws)
    compare(cfg, raws, dcol.as_demodulate_all(), deng, ores, oorc)


def test_device_io_afc():
    """The AFC case of test_afc_follows_an_off_bin_carrier: one batch per run, bins moved by K2 between batches."""
    sr, n, w, cf = 2560000, 512, 8000, 120000000
    ch = cm.make_channel(cf + 100000, cf, sr, n, w, squelch_dbfs=-40.0, afc=2)
    ch.offset_hz = 100000.0 + 3 * (sr / n)
    cfg = cm.Config(fft_size=n, wave_rate=w, devices=[cm.Device(sample_rate=sr, sfmt=cm.SFMT_U8, centerfreq=cf, channels=[ch])])
    raws = [wl.synth_iq(cfg, 0, wl.samples_for_batches(cfg, 0, 5), key_on_s=0.25, key_off_s=0.15, amplitude=0.3)]
    hcol, heng = run_host(cfg, raws, nbmax=1)
    dcol, deng = run_device(cfg, raws, nbmax=1)
    ax = hcol.arrays()[0][2]
    assert np.any(ax == ord('>')) or np.any(ax == ord('<')), "AFC never moved: case is not exercising AFC"
    assert_same(cfg, hcol, heng, dcol, deng)


def test_device_io_host_fetch_in_device_mode():
    """abg_fetch_batch keeps working with the result slots in HBM (what the reference binding calls)."""
    cfg, raws = CASES["s8_two_devices"]()
    hcol, heng = run_host(cfg, raws)
    e = lib.Engine(cfg, max_batches_per_run=4)
    e.results_on_device()
    col = Collect(cfg)
    for chunk in _schedule(cfg, raws, 4):
        for d, a, b in chunk:
            e.push(d, raws[d][a:b])
        e.run(-1)
        col.host(e)
    while e.run(-1) > 0:
        col.host(e)
    assert_same(cfg, hcol, heng, col, e)


def test_device_io_scan_channel():
    cfg, freqs = _scan_setup()
    nb, visits = 2, [0, 2, 1, 2, 0]
    raw = wl.synth_iq(cfg, 0, wl.samples_for_batches(cfg, 0, nb * len(visits)), key_on_s=1.2, key_off_s=0.2, amplitude=0.2)
    t = torch.from_numpy(raw).cuda()
    engines = []
    for device in (False, True):
        e = lib.Engine(cfg, max_batches_per_run=nb, input_capacity_batches=2 * nb + 1)
        if device:
            e.results_on_device()
        e.scan_configure(0, 0, freqs)
        col = Collect(cfg)
        pos = 0
        for k, idx in enumerate(visits):
            need = wl.samples_for_batches(cfg, 0, nb * (k + 1)) * 2
            e.scan_select(0, 0, idx)
            if device:
                e.push_tensor(0, t[pos:need])
            else:
                e.push(0, raw[pos:need])
            pos = need
            assert e.run(nb) == nb
            if device:
                col.device(e)
            else:
                col.host(e)
        torch.cuda.synchronize()
        engines.append((col, e))
    assert_same(cfg, engines[0][0], engines[0][1], engines[1][0], engines[1][1])


def test_device_io_mixers():
    """cfg 4 shape: the mixer sums through fetch_mixer_tensors equal abg_fetch_mixer_batch's."""
    cfg = wl.cfg4()
    nb = 3
    raws = [wl.synth_iq(cfg, d, wl.samples_for_batches(cfg, d, nb), key_on_s=0.2, key_off_s=0.1) for d in range(len(cfg.devices))]
    mixers = [[(d, m, 1.0 + 0.25 * d, (-0.5 if (m == 1 and d == 0) else 0.0)) for d in range(len(cfg.devices))] for m in range(4)]
    h = lib.Engine(cfg, max_batches_per_run=2)
    g = lib.Engine(cfg, max_batches_per_run=2)
    h.configure_mixers(mixers)
    g.configure_mixers(mixers)  # before the switch: the mixer slots move to HBM with the rest
    g.results_on_device()
    ts = _tensors(raws)
    for d in range(len(raws)):
        h.push(d, raws[d])
        g.push_tensor(d, ts[d])
    hcol, gcol = Collect(cfg), Collect(cfg)
    hmix, glr, gsig = [], [], []
    while True:
        nh, ng = h.run(-1), g.run(-1)
        assert nh == ng
        if nh == 0:
            break
        hcol.host(h)
        gcol.device(g)
        while True:
            per = [h.fetch_mixer(m) for m in range(4)]
            if per[0] is None:
                break
            hmix.append(per)
        lr, sig = g.fetch_mixer_tensors(8)
        glr.append(lr)
        gsig.append(sig)
    torch.cuda.synchronize()
    assert_same(cfg, hcol, h, gcol, g)
    glr = torch.cat(glr).cpu().numpy()
    gsig = torch.cat(gsig).cpu().numpy()
    assert glr.shape == (nb, 4, 2, cfg.wave_batch) and len(hmix) == nb
    for b in range(nb):
        for m in range(4):
            left, right, sig = hmix[b][m]
            assert _equal(glr[b, m, 0], left) and _equal(glr[b, m, 1], right) and bool(gsig[b, m]) == sig
    assert gsig.any()


def test_streaming_odd_sized_mixed_pushes():
    """Odd-sized slices into a small ring (compaction runs), alternating abg_push and abg_push_device on one device."""
    cfg, raws = CASES["am_u8"](n_batches=6)
    r = raws[0]
    t = torch.from_numpy(r).cuda()
    rng = np.random.default_rng(7)
    cuts = [0]
    while cuts[-1] < r.size:
        cuts.append(min(r.size, cuts[-1] + 2 * int(rng.integers(1, 40000))))
    engines = []
    for mixed in (False, True):
        e = lib.Engine(cfg, max_batches_per_run=2, input_capacity_batches=3)
        if mixed:
            e.results_on_device()
        col = Collect(cfg)
        fetch = col.device if mixed else col.host
        for k in range(len(cuts) - 1):
            a, b = cuts[k], cuts[k + 1]
            if mixed and k % 2:
                e.push_tensor(0, t[a:b])
            else:
                e.push(0, r[a:b])
            e.run(-1)
            fetch(e)
        while e.run(-1) > 0:
            fetch(e)
        torch.cuda.synchronize()
        engines.append((col, e))
    assert len(cuts) > 8
    (hc, he), (dc, de) = engines
    assert hc.arrays()[0][0].shape[0] == 6
    assert_same(cfg, hc, he, dc, de)


def test_push_waits_for_the_producing_stream():
    """The input is written on a side stream behind a long sleep and pushed on that stream without a synchronise: the
    engine's copy must see the finished bytes."""
    cfg, raws = CASES["s8_two_devices"]()
    hcol, heng = run_host(cfg, raws)
    src = _tensors(raws)
    torch.cuda.synchronize()
    e = lib.Engine(cfg, max_batches_per_run=4)
    e.results_on_device()
    side = torch.cuda.Stream()
    col = Collect(cfg)
    with torch.cuda.stream(side):
        for chunk in _schedule(cfg, raws, 4):
            for d, a, b in chunk:
                buf = torch.empty(b - a, dtype=src[d].dtype, device="cuda")
                torch.cuda._sleep(20_000_000)
                buf.copy_(src[d][a:b])
                e.push_tensor(d, buf)
            e.run(-1)
            col.device(e)
    torch.cuda.synchronize()
    assert_same(cfg, hcol, heng, col, e)


def test_fetch_does_not_block_the_host():
    cfg, raws = CASES["s8_two_devices"](n_batches=6)
    hcol, heng = run_host(cfg, raws, nbmax=2, step_b=2)
    e = lib.Engine(cfg, max_batches_per_run=2)
    e.results_on_device()
    ts = _tensors(raws)
    stream = torch.cuda.current_stream()
    outs = []
    for k, chunk in enumerate(_schedule(cfg, raws, 2)):
        for d, a, b in chunk:
            e.push_tensor(d, ts[d][a:b])
        assert e.run(-1) == 2 * len(cfg.devices)
        if k == 0:  # the first fetch may load the gather kernel's module
            outs.append(e.fetch_all_tensors(2))
            continue
        torch.cuda._sleep(400_000_000)
        outs.append(e.fetch_all_tensors(2))
        assert not stream.query(), "fetch_all_tensors waited for the caller's stream"
    assert len(outs) == 3
    torch.cuda.synchronize()
    G = [len(d.channels) for d in cfg.devices]
    h = hcol.arrays()
    wo = torch.cat([o[0] for o in outs]).cpu().numpy()
    iq = torch.cat([o[1] for o in outs]).cpu().numpy()
    ax = torch.cat([o[2] for o in outs]).cpu().numpy()
    g0 = 0
    for d, Cn in enumerate(G):
        assert _equal(wo[:, g0:g0 + Cn], h[d][0]) and _equal(iq[:, g0:g0 + Cn], h[d][1]) and _equal(ax[:, g0:g0 + Cn], h[d][2])
        g0 += Cn


def test_fetches_three_runs_ahead_reuse_slots_in_stream_order():
    """Each gather is held back by a sleep on the caller's stream while later runs keep coming: the run that reuses a
    slot must wait for the slot's release event, not overwrite the batches still to be copied."""
    cfg, raws = CASES["am_u8"](n_batches=8)
    heng = lib.Engine(cfg, max_batches_per_run=1, input_capacity_batches=12)
    heng.push(0, raws[0])
    hcol = Collect(cfg)
    while heng.run(1) > 0:
        hcol.host(heng)
    e = lib.Engine(cfg, max_batches_per_run=1, input_capacity_batches=12)
    e.results_on_device()
    e.push_tensor(0, torch.from_numpy(raws[0]).cuda())
    outs = []
    while e.run(1) > 0:
        torch.cuda._sleep(50_000_000)
        outs.append(e.fetch_all_tensors(1))
    assert len(outs) == 8
    torch.cuda.synchronize()
    h = hcol.arrays()[0]
    for k, what in enumerate(("waveout", "iq_out", "axcindicate")):
        assert _equal(torch.cat([o[k] for o in outs]).cpu().numpy(), h[k]), what
    assert _stats_bytes(heng, cfg) == _stats_bytes(e, cfg)


def test_fetch_all_is_one_launch_for_512_devices():
    cfg = wl.cfg5(n_devices=512, n_channels=8)
    nb = 2
    uniq = [wl.synth_iq(cfg, u, wl.samples_for_batches(cfg, u, nb), key_on_s=0.05, key_off_s=0.05) for u in range(4)]
    tu = _tensors(uniq)
    engines = []
    for _ in range(2):
        e = lib.Engine(cfg, max_batches_per_run=nb)
        e.results_on_device()
        for d in range(len(cfg.devices)):
            e.push_tensor(d, tu[d % 4])
        assert e.run(nb) == nb * len(cfg.devices)
        engines.append(e)
    a, b = engines
    l0 = a.launch_count()
    wo, iq, ax = a.fetch_all_tensors(nb)
    assert a.launch_count() - l0 <= 1
    assert all(a.batches_ready(d) == 0 for d in range(len(cfg.devices)))
    per = [b.fetch_tensors(d, nb) for d in range(len(cfg.devices))]
    torch.cuda.synchronize()
    for k in range(3):
        assert _equal(torch.cat([p[k] for p in per], 1).cpu().numpy(), (wo, iq, ax)[k].cpu().numpy())


def test_device_io_errors():
    cfg, raws = CASES["s8_two_devices"]()
    ts = _tensors(raws)
    e = lib.Engine(cfg, max_batches_per_run=2, input_capacity_batches=3)
    e.results_on_device()

    def code(fn, *a):
        with pytest.raises(lib.AbgError) as ei:
            fn(*a)
        return ei.value.code

    host = np.ascontiguousarray(raws[0][:64])
    assert code(e.push_device_ptr, 0, host.ctypes.data, host.nbytes) == -2             # pageable host memory
    pinned = torch.from_numpy(host).pin_memory()
    assert code(e.push_device_ptr, 0, pinned.data_ptr(), host.nbytes) == -2            # page-locked host memory
    if torch.cuda.device_count() > 1:
        other = ts[0][:64].to("cuda:1")
        assert code(e.push_device_ptr, 0, other.data_ptr(), 64) == -2                   # another GPU
    assert code(e.push_device_ptr, 0, ts[0].data_ptr(), 3) == -2                       # not whole samples
    assert code(e.push_tensor, 0, ts[0].repeat(4)) == -6                                  # more than the ring holds
    with pytest.raises(TypeError):
        e.push_tensor(0, ts[1])                                                            # uint8 into the S8 device
    with pytest.raises(TypeError):
        e.push_tensor(0, ts[0].to(torch.int16))
    with pytest.raises(TypeError):
        e.push_tensor(0, raws[0])
    # uneven ready counts: only device 1 gets input
    e.push_tensor(1, ts[1][:wl.samples_for_batches(cfg, 1, 1) * 2])
    assert e.run(-1) == 1
    assert code(e.fetch_all_tensors, 1) == -2
    assert e.batches_ready(1) == 1 and e.batches_ready(0) == 0                           # nothing popped
    assert code(e.results_on_device) == -2                                                # after a run
    assert e.L.abg_set_result_location(e.h, lib.RESULTS_HOST) == -2
    # the engine is still usable: the rest of both streams gives what the host path gives
    h = lib.Engine(cfg, max_batches_per_run=2, input_capacity_batches=3)
    assert code(h.fetch_tensors, 0, 1) == -2                                             # device fetch in host mode
    h.push(1, raws[1][:wl.samples_for_batches(cfg, 1, 1) * 2])
    assert h.run(-1) == 1
    hw, hi, ha = h.fetch(1)
    gw, gi, ga = e.fetch_tensors(1, 4)
    torch.cuda.synchronize()
    assert _equal(gw[0].cpu().numpy(), hw) and _equal(ga[0].cpu().numpy(), ha)
    n0 = wl.samples_for_batches(cfg, 0, 1) * 2
    e.push_tensor(0, ts[0][:n0])
    h.push(0, raws[0][:n0])
    assert e.run(-1) == h.run(-1) == 1
    hw, hi, ha = h.fetch(0)
    gw, gi, ga = e.fetch_tensors(0, 4)
    torch.cuda.synchronize()
    assert _equal(gw[0].cpu().numpy(), hw) and _equal(gi[0].cpu().numpy(), hi) and _equal(ga[0].cpu().numpy(), ha)
