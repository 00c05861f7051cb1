#!/usr/bin/env python
"""bench.py — throughput of the multichannel demodulation hot path (BASELINE.json metric:
"IQ Msamples/s through FFT+demod at 1/2/4/8 B200; % HBM roofline; vs CPU ref").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload cfg2|cfg1|cfg3|cfg3f|cfg4|cfg5] [--impl reference]

A step = one pass of the hot path (K1 convert+window+DFT of the bins, K2 demodulation) over one batch of synthetic input:
`batches_per_step` WAVE_BATCHes (default 64 x 125 ms = 8 s of signal) of every device of the workload, executed as
batches_per_step / 4 engine runs of 4 batches.  Default workload at every N is BASELINE.json configs[1] per GPU: 64
devices x 2.56 Msps U8, fft_size 2048, 8 AM channels each ("cfg2"); devices shard by GPU with no data-path collective, so N
GPUs run N x 64 devices (scaling = "weak").

  value    device-timed (CUDA events on the engine's stream, max over ranks): IQ samples consumed / s, inputs resident in
           HBM (the resident stream, 168 MB per run, is larger than the 126 MB L2: every run re-reads HBM).
  e2e      same metric through the public C ABI with HOST buffers: abg_push (H2D from pinned memory) + abg_run +
           abg_fetch_batches (results written by the GPU into pinned host slots, then copied to the caller's arrays) inside
           the timed region, software-pipelined by one run like any streaming caller; `pcie_frac` = achieved H2D rate /
           the pinned-memory H2D rate measured on this box right before (the path is PCIe-bound).
  roofline K1 (the dominant HBM consumer): algorithmic bytes per launch / CUDA-event duration vs the measured HBM peak, the
           executed tensor-core work (int8 MACs) and, when a capture of this exact kernel source exists under profiles/,
           its DRAM traffic and issue-slot use.
  configs  short device-timed legs of the other BASELINE.json configs (cfg1, cfg3 S16 / F32 throughput variant, cfg4 with
           mixers, cfg5 one GPU's share), each with K1/K2 times, HBM fraction and a `parity_spot` (the CPU oracle on one
           device per distinct synthetic stream, same bytes, BASELINE.md gate).  At N > 1: cfg5 and the NCCL mixer
           all-reduce, timed like the headline.
  cpu_baseline  the CPU oracle built from the reference's own leaf classes (oracle/_ref) on this box's host cores over a
           bounded sample of the workload: one pinned thread per device (multiple_demod_threads mode) and the reference's
           default single-thread round-robin, plus the cfg1 point.
`--impl reference` times that CPU path alone (rank 0 only under torchrun) and prints the same line shape.
`--dump-outputs DIR` writes what the e2e leg's caller received in its last timed step (see dump_outputs); the inputs are
seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (os.path.join(ROOT, "rtlsdr-airband_b200", "py"), os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

METRIC = "iq_msamples_per_s_fft_demod"
UNIT = "Msamples/s"
NB_RUN = 4  # WAVE_BATCHes per engine run (abg_options.max_batches_per_run)


# ----------------------------------------------------------------------------------------------------------------------
# workloads
# ----------------------------------------------------------------------------------------------------------------------
def make_workload(name: str):
    from airband_b200 import config as cm
    from airband_b200 import workloads as wl
    if name == "cfg2":
        return wl.cfg2(n_devices=64, n_channels=8), "cfg2: 64 synthetic devices x 2.56 Msps U8, fft_size 2048, 8 AM channels each (BASELINE.json configs[1])"
    if name == "cfg1":
        return wl.cfg1(), "cfg1: 1 device, 2.56 Msps U8, fft_size 512, 1 AM channel (config/basic_multichannel.conf shape, BASELINE.json configs[0])"
    if name == "cfg3":
        return (wl.cfg3(n_devices=8, n_channels=32, sfmt=cm.SFMT_S16),
                "cfg3: 8 devices x 10 Msps S16, NFM build (WAVE_RATE 16000), fft_size 4096, 32 NFM channels with CTCSS+notch, squelch_snr_threshold 0 (BASELINE.json configs[2])")
    if name == "cfg3f":
        return (wl.cfg3(n_devices=8, n_channels=32, sfmt=cm.SFMT_F32),
                "cfg3 (F32 input): 8 devices x 10 Msps F32, NFM build (WAVE_RATE 16000), fft_size 4096, 32 NFM channels with CTCSS+notch, squelch_snr_threshold 0")
    if name == "cfg4":
        return wl.cfg4(), "cfg4: mixer path, 4 devices x 4 AM channels (2.56 Msps U8, fft_size 512) into 4 mixers spanning all devices (config/big_mixer.conf shape, BASELINE.json configs[3])"
    if name == "cfg5":
        return wl.cfg5(n_devices=512, n_channels=8), "cfg5 (one GPU's share of BASELINE.json configs[4]): 512 devices x 2.56 Msps U8, fft_size 512, 8 AM channels each"
    raise SystemExit(f"unknown workload {name}")


def synth_streams(cfg, n_batches: int, n_unique: int = 4):
    """Synthetic raw streams (SURVEY.md §8d): n_unique distinct seeded streams tiled over the devices."""
    from airband_b200 import workloads as wl
    uniq = []
    for u in range(min(n_unique, len(cfg.devices))):
        n = wl.samples_for_batches(cfg, u, n_batches)
        uniq.append(wl.synth_iq(cfg, u, n, key_on_s=0.30, key_off_s=0.12))
    return [uniq[d % len(uniq)] for d in range(len(cfg.devices))]


# ----------------------------------------------------------------------------------------------------------------------
# host: NUMA placement, CPU description, clocks
# ----------------------------------------------------------------------------------------------------------------------
def parse_cpulist(s: str):
    out = []
    for part in s.strip().split(","):
        if not part:
            continue
        if "-" in part:
            a, b = part.split("-")
            out.extend(range(int(a), int(b) + 1))
        else:
            out.append(int(part))
    return out


_ALL_CPUS = set(os.sched_getaffinity(0))  # what the process may use before any binding (restored for the CPU baseline leg)


def bind_to_gpu_numa(gpu_index: int) -> dict:
    """Run this process (and place the pinned buffers it allocates from now on: first touch) on the CPUs of the NUMA node
    the GPU hangs off.  H2D copies from the far socket cross UPI and cap the 8-GPU end-to-end rate."""
    info = {"bound": False}
    try:
        bdf = subprocess.run(["nvidia-smi", f"--id={gpu_index}", "--query-gpu=pci.bus_id", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=20).stdout.strip().lower()
        if bdf.startswith("00000000:"):
            bdf = bdf[4:]
        base = f"/sys/bus/pci/devices/{bdf}"
        cpus = parse_cpulist(open(base + "/local_cpulist").read())
        node = int(open(base + "/numa_node").read().strip())
        allowed = sorted(set(cpus) & set(os.sched_getaffinity(0)))
        if allowed:
            os.sched_setaffinity(0, allowed)
            info = {"bound": True, "gpu_pci": bdf, "numa_node": node, "cpus": open(base + "/local_cpulist").read().strip(), "n_cpus": len(allowed)}
    except Exception as ex:  # no sysfs / no nvidia-smi: run unbound and say so
        info = {"bound": False, "why": str(ex)[:120]}
    return info


def cpu_description() -> dict:
    model, phys = "unknown", set()
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                model = line.split(":", 1)[1].strip()
                break
    except Exception:
        pass
    firsts = []
    for c in sorted(os.sched_getaffinity(0)):
        try:
            sib = parse_cpulist(open(f"/sys/devices/system/cpu/cpu{c}/topology/thread_siblings_list").read())
        except Exception:
            sib = [c]
        if min(sib) not in phys:
            phys.add(min(sib))
            firsts.append(c)
    return {"model": model, "logical_cpus": len(os.sched_getaffinity(0)), "physical_cores": len(firsts), "one_cpu_per_core": firsts}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.idx}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def wait_first(self, timeout_s: float = 10.0):
        t0 = time.time()
        while self.proc and not self.rows and time.time() - t0 < timeout_s:
            time.sleep(0.01)

    def count_between(self, t0: float, t1: float) -> int:
        return sum(1 for (t, _) in self.rows if t0 <= t <= t1)

    def stop(self, windows=None):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.05)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for (ts, r) in self.rows:
            if windows is not None and not any(a <= ts <= b for (a, b) in windows):
                continue
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except ValueError:
                continue
            for k, nme in enumerate(names):
                if f[3 + k].lower().startswith("active"):
                    reasons.add(nme)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "power_w_max": float(max(pw)), "samples": len(sm),
                "reasons": sorted(reasons)}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return json.load(open(path)), "measured"
        except Exception:
            pass
    return {"hbm_gbs": 6650.0}, "fallback"


DUMP_BYTES = 48 << 20  # --dump-outputs: above this, a fixed seeded sample of the channels is written


def dump_outputs(dirname: str, runs) -> dict:
    """Write the engine runs of one step, runs = [(waveout[dev][NB_RUN, C, B], axcindicate[dev][NB_RUN, C]), ...] in time
    order, as dirname/waveout.npy float32 [batches, channels, B] and dirname/axcindicate.npy float32 [batches, channels]
    (the status characters' codes).  Channels are numbered across devices; all of them when they fit DUMP_BYTES, else a
    sample drawn with seed 0."""
    G, B = sum(w.shape[1] for w in runs[0][0]), runs[0][0][0].shape[2]
    nb = len(runs) * NB_RUN
    k = min(G, max(1, DUMP_BYTES // (nb * B * 4)))
    sel = np.arange(G) if k == G else np.sort(np.random.default_rng(0).choice(G, k, replace=False))
    wave = np.concatenate([np.concatenate(w, axis=1)[:, sel] for (w, _) in runs], axis=0)
    axc = np.concatenate([np.concatenate(a, axis=1)[:, sel] for (_, a) in runs], axis=0).astype(np.float32)
    os.makedirs(dirname, exist_ok=True)
    np.save(os.path.join(dirname, "waveout.npy"), wave)
    np.save(os.path.join(dirname, "axcindicate.npy"), axc)
    return {"dir": dirname, "waveout": list(wave.shape), "axcindicate": list(axc.shape),
            "channels": "all" if k == G else f"{k} of {G}, drawn with numpy default_rng(0)"}


def source_sha(*rel_paths) -> str:
    h = hashlib.sha256()
    for rp in rel_paths:
        try:
            h.update(open(os.path.join(ROOT, rp), "rb").read())
        except Exception:
            h.update(b"?")
    return h.hexdigest()[:16]


# ----------------------------------------------------------------------------------------------------------------------
# CPU arm (oracle): the reference's own leaf classes + the restated demodulate() loop on host cores
# ----------------------------------------------------------------------------------------------------------------------
def _cpu_time_config(cfg, variant, nthreads, pin, budget_s, steps, warmup):
    """Bounded sample: the first D devices of cfg, (warmup + steps) steps of `reps` x 4 batches.  Returns Msps over the timed
    steps, best single step, seconds, sample description."""
    import oracle_py as op
    D = len(cfg.devices)
    B, hop = cfg.wave_batch, cfg.hop(0)
    raws = synth_streams(cfg, NB_RUN)
    chunk_items = [NB_RUN * B * cfg.hop(d) * 2 for d in range(D)]
    prime_items = [(100 * cfg.hop(d) + cfg.fft_size) * 2 for d in range(D)]

    def fresh():
        o = op.Oracle(cfg, variant)
        o.set_discard(True)
        if pin:
            o.set_pin(pin)
        for d in range(D):
            o.push(d, raws[d][:prime_items[d]])
        return o

    o = fresh()
    for d in range(D):
        o.push(d, raws[d][prime_items[d]:prime_items[d] + chunk_items[d]])
    t0 = time.perf_counter()
    n0 = o.run(NB_RUN, nthreads)
    per_chunk = max(time.perf_counter() - t0, 1e-4)          # one pass of 4 batches over the sample devices
    assert n0 == D * NB_RUN
    total_steps = steps + warmup
    reps = max(1, min(256, int(budget_s / (per_chunk * total_steps))))
    done, dt, best = 0, 0.0, 0.0
    for step in range(total_steps):
        t_step, n_step = 0.0, 0
        for _ in range(reps):
            for d in range(D):
                o.push(d, raws[d][prime_items[d]:prime_items[d] + chunk_items[d]])
            t0 = time.perf_counter()
            n = o.run(NB_RUN, nthreads)
            t_step += time.perf_counter() - t0
            n_step += n
        if step >= warmup:
            done += n_step
            dt += t_step
            best = max(best, n_step * B * hop / t_step / 1e6)
    o.close()
    samples = done * B * hop
    return samples / dt / 1e6, best, dt, f"{D} devices x {NB_RUN * reps} batches/step x {steps} steps ({samples / 1e6:.1f} Msamples, {dt:.1f} s)"


def cpu_run(cfg, desc, steps: int, warmup: int, budget_s: float = 20.0, extras: bool = True):
    """Time the CPU path over bounded samples of the workload.  Returns (Msps, info dict, ms_per_step)."""
    import oracle_py as op
    variant = "ref_fast" if op.available("ref_fast") else "restated_fast"
    kind = "reference" if variant == "ref_fast" else "port"
    try:
        os.sched_setaffinity(0, _ALL_CPUS)  # the GPU arm binds itself to one NUMA node; the CPU arm gets every core of the box
    except Exception:
        pass
    cpu = cpu_description()
    cores = max(1, cpu["physical_cores"])
    D = min(len(cfg.devices), cores)
    sub = type(cfg)(fft_size=cfg.fft_size, wave_rate=cfg.wave_rate, fm_demod=cfg.fm_demod, devices=cfg.devices[:D])
    pin = cpu["one_cpu_per_core"][:D]
    msps, best, dt, sample = _cpu_time_config(sub, variant, D, pin, budget_s, steps, warmup)
    info = {"value": msps, "unit": UNIT, "cores": D, "kind": kind,
            "sample": f"{sample} of {len(cfg.devices)} configured devices; one thread per device (multiple_demod_threads mode, rtl_airband.cpp:1052), "
                      f"each pinned to its own physical core; oracle variant {variant} (-O3 -ffast-math, x86-64-v3); FFTW is not installable offline: "
                      f"own scalar radix-4 FP32 FFT, which understates FFTW's SIMD codelets by an unmeasured factor",
            "best_step_value": best, "cpu_model": cpu["model"], "physical_cores": cpu["physical_cores"], "logical_cpus": cpu["logical_cpus"]}
    try:
        sec = op.lib(variant).abo_fft_seconds(cfg.fft_size, 4000)
        info["fft"] = {"us_per_transform": sec * 1e6, "nominal_gflops": 5 * cfg.fft_size * math.log2(cfg.fft_size) / sec / 1e9,
                       "note": "the oracle's own FP32 FFT alone, one core, persistent plan; FFTW's AVX2 codelets reach roughly 20-30 GFLOP/s per core at "
                               "these sizes, so the FFT share of the CPU arm is within about 2x of what the reference would get from fftw3f"}
    except Exception:
        pass
    if extras:
        try:  # the reference's default: ONE demod thread round-robin over all devices (rtl_airband.cpp:1070-1086)
            os.sched_setaffinity(0, {pin[0]}) if pin else None
            rr, _, _, rr_sample = _cpu_time_config(sub, variant, 1, None, 4.0, 2, 1)
            info["single_thread_round_robin"] = {"value": rr, "unit": UNIT, "cores": 1, "sample": rr_sample}
            c1, _ = make_workload("cfg1")
            v1, _, _, s1 = _cpu_time_config(c1, variant, 1, None, 3.0, 2, 1)
            info["cfg1_point"] = {"value": v1, "unit": UNIT, "cores": 1, "sample": s1 + " (BASELINE.json configs[0], the reference's own CPU-runnable case)"}
        except Exception as ex:
            info["extras_error"] = str(ex)[:200]
        finally:
            try:
                os.sched_setaffinity(0, _ALL_CPUS)
            except Exception:
                pass
    return msps, info, dt / max(steps, 1) * 1e3


# ----------------------------------------------------------------------------------------------------------------------
# GPU legs
# ----------------------------------------------------------------------------------------------------------------------
def alg_bytes_per_run(cfg, nb):
    """SURVEY.md §8d: per frame hop*2*bytes_per_sample + 4*C (every input byte once, every |X| once)."""
    return float(sum((cfg.hop(d) * 2 * cfg.devices[d].bytes_per_sample + 4 * len(cfg.devices[d].channels)) * nb * cfg.wave_batch for d in range(len(cfg.devices))))


def parity_spot(cfg, raws, nb, n_unique=4, relaxed=False, mixers=None, fft_mode=0):
    """The CPU oracle on one device per distinct synthetic stream (same bytes, through the streaming C ABI), BASELINE.md gate."""
    import oracle_py as op
    import parity
    from airband_b200 import lib
    n = min(n_unique, len(cfg.devices))
    sub = type(cfg)(fft_size=cfg.fft_size, wave_rate=cfg.wave_rate, fm_demod=cfg.fm_demod, devices=cfg.devices[:n])
    sraws = raws[:n]
    ores, oorc = op.run_oracle(sub, sraws)
    out = {"devices_checked": n, "mode": "relaxed (SURVEY.md §7.3: transition indices and audio compared separately)" if relaxed else "strict"}
    if mixers is None:
        gres, geng = lib.demodulate_all(sub, sraws, max_batches_per_run=nb, fft_mode=fft_mode)
        per = [(parity.relaxed if relaxed else parity.strict)(gres[d], ores[d]) for d in range(n)]
        geng.close()
    else:
        # mixers spanning the checked devices: device audio AND the mixed sums vs the oracle-side sum (mixer.cpp:133-140,189-214)
        e = lib.Engine(sub, max_batches_per_run=nb, fft_mode=fft_mode)
        mix = [[(d, m, a, b) for (d, m, a, b) in mi if d < n] for mi in mixers]
        e.configure_mixers(mix)
        for d, r in enumerate(sraws):
            e.push(d, r)
        got_dev = [([], [], []) for _ in range(n)]
        got_mix = [[] for _ in mix]
        while e.run(-1) > 0:
            for d in range(n):
                while True:
                    g = e.fetch(d)
                    if g is None:
                        break
                    for k in range(3):
                        got_dev[d][k].append(g[k])
            for m in range(len(mix)):
                while True:
                    g = e.fetch_mixer(m)
                    if g is None:
                        break
                    got_mix[m].append(g)
        gres = [(np.concatenate(x[0], 1), np.concatenate(x[1], 1), np.stack(x[2], 0)) for x in got_dev]
        per = [parity.strict(gres[d], ores[d]) for d in range(n)]
        ref = parity.mixer_reference(sub, ores, mix, len(got_mix[0]))
        worst = 0.0
        flags_ok = True
        for m in range(len(mix)):
            for b, (gl, gr, gs) in enumerate(got_mix[m]):
                worst = max(worst, parity.gate(gl, ref[m][b][0]), parity.gate(gr, ref[m][b][1]))
                flags_ok &= (gs == ref[m][b][2])
        out["mixer_max_err"] = worst
        out["mixer_flags_equal"] = bool(flags_ok)
        per.append({"ok": bool(worst <= parity.TOL and flags_ok)})
        e.close()
    oorc.close()
    out["ok"] = bool(all(p.get("ok") for p in per))
    for k in ("max_err", "edges", "edges_unmatched", "audio_samples_compared", "audio_samples_outside_gate", "max_err_compared", "opened"):
        vals = [p[k] for p in per if k in p]
        if vals:
            out[k] = max(vals) if "err" in k else int(sum(vals))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="cfg2")
    ap.add_argument("--batches-per-step", type=int, default=64)
    ap.add_argument("--fft-mode", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the legs of the other BASELINE configs")
    ap.add_argument("--no-parity", action="store_true", help="skip the oracle parity spots of the legs")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the audio and squelch flags the e2e leg fetched in its last timed step "
                                                          "as DIR/*.npy (rank 0)")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 0)
    if args.steps < 1:
        raise SystemExit("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.no_e2e):
        raise SystemExit("--dump-outputs writes what the B200 arm's e2e leg computed: it cannot go with --impl reference or --no-e2e")
    if args.batches_per_step % NB_RUN:
        raise SystemExit(f"--batches-per-step must be a multiple of {NB_RUN}")
    runs_per_step = args.batches_per_step // NB_RUN

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    cfg, desc = make_workload(args.workload)
    D = len(cfg.devices)
    base_config = {"workload": desc, "devices_per_gpu": D, "batches_per_step": args.batches_per_step, "batches_per_engine_run": NB_RUN,
                   "wave_rate": cfg.wave_rate, "fft_mode": args.fft_mode,
                   "realtime_floor_msps_per_gpu": sum(dv.sample_rate for dv in cfg.devices) / 1e6}

    # ------------------------------------------------------------------------------------------ reference arm (CPU)
    if args.impl == "reference":
        if rank != 0:
            return
        msps, info, ms = cpu_run(cfg, desc, args.steps, args.warmup, extras=False)
        conf = dict(base_config)
        conf["note"] = "CPU reference arm: bounded sample of the same workload on host cores (see cpu_baseline.sample)"
        line = {"impl": "reference", "metric": METRIC, "value": msps, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic", "config": conf,
                "cpu_baseline": info, "e2e": {"value": msps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        print(json.dumps(line))
        return

    # ------------------------------------------------------------------------------------------ B200 arm
    numa = bind_to_gpu_numa(local_rank)   # before torch / CUDA allocate anything pinned
    import torch
    import torch.distributed as dist
    from airband_b200 import lib

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; this benchmark has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"  # NCCL prints its version banner on stdout: keep stdout to the one JSON line
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    stream = torch.cuda.Stream(device=local_rank)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def resident_engine(c, raws_c, fft_mode=args.fft_mode):
        e = lib.Engine(c, cuda_device=local_rank, max_batches_per_run=NB_RUN, input_capacity_batches=NB_RUN + 1, fft_mode=fft_mode)
        e.set_stream(stream.cuda_stream)
        for d in range(len(c.devices)):
            e.resident_load(d, raws_c[d])
        return e

    def time_resident(e, n_runs, warm_runs, after_run=None):
        """n_runs engine runs of NB_RUN batches, device-timed on the engine's stream, bracketed by barriers; max over ranks."""
        for _ in range(max(warm_runs, 1)):
            e.run_resident(NB_RUN)
            if after_run:
                after_run()
        barrier()
        l0 = e.launch_count()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        t0 = time.time()
        ev0.record(stream)
        for _ in range(n_runs):
            e.run_resident(NB_RUN)
            if after_run:
                after_run()
        e.join()  # main stream waits for the K2 stream: ev1 covers every kernel of every run
        ev1.record(stream)
        barrier()
        t1 = time.time()
        return max_over_ranks(ev0.elapsed_time(ev1)), e.launch_count() - l0, (t0, t1)

    def kernel_times(e, n=5):
        k1, k2 = [], []
        for _ in range(n):
            e.run_resident(NB_RUN)
            t = e.last_run_times()
            k1.append(t[0]); k2.append(t[1])
        return float(np.median(k1)), float(np.median(k2))

    B = cfg.wave_batch
    hop = [cfg.hop(d) for d in range(D)]
    raws = synth_streams(cfg, NB_RUN)
    samples_per_run = sum(NB_RUN * B * hop[d] for d in range(D))
    samples_per_step = samples_per_run * runs_per_step

    # ---- pinned-memory PCIe rates of this box (denominator of e2e.pcie_frac), measured before anything else runs ----
    pcie = None
    if not args.no_e2e:
        hbuf = torch.empty(256 << 20, dtype=torch.uint8).pin_memory()
        dbuf = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
        rates = {}
        half = 128 << 20
        s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
        for name, (dst, src) in {"h2d": (dbuf, hbuf), "d2h": (hbuf, dbuf)}.items():
            best = 0.0
            for rep in range(10):
                # one 256 MiB copy, and the same bytes as two concurrent 128 MiB copies on two streams (the engine keeps
                # several ring copies in flight): the denominator is the better of the two
                start, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
                torch.cuda.synchronize()
                start.record(s1)
                s2.wait_event(start)
                if rep % 2 == 0:
                    with torch.cuda.stream(s1):
                        dst.copy_(src, non_blocking=True)
                else:
                    with torch.cuda.stream(s1):
                        dst[:half].copy_(src[:half], non_blocking=True)
                    with torch.cuda.stream(s2):
                        dst[half:].copy_(src[half:], non_blocking=True)
                e1.record(s1)
                e2.record(s2)
                torch.cuda.synchronize()
                best = max(best, (256 << 20) / (max(start.elapsed_time(e1), start.elapsed_time(e2)) * 1e-3) / 1e9)
            rates[name] = best
        pcie = {"h2d_gbs": rates["h2d"], "d2h_gbs": rates["d2h"],
                "how": "256 MiB pinned <-> device, best of 10 (one copy / two concurrent 128 MiB copies on two streams), CUDA events"}
        del hbuf, dbuf

    # ---- value: device-timed, inputs resident in HBM ----
    eng = resident_engine(cfg, raws)
    resident_bytes = sum(eng.resident_bytes_needed(d) for d in range(D))
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        sampler.wait_first()
    elapsed_ms, launches, win = time_resident(eng, args.steps * runs_per_step, max(args.warmup, 3) * runs_per_step)
    clocks = None
    if rank == 0:
        windows = [win]
        note = None
        if sampler.count_between(*win) < 5:
            t_x0 = time.time()
            while sampler.proc and sampler.count_between(t_x0, time.time()) < 8 and time.time() - t_x0 < 3.0:
                for _ in range(50):
                    eng.run_resident(NB_RUN)
                eng.sync()
            windows.append((t_x0, time.time()))
            note = "timed region shorter than 5 sampling intervals: clocks also sampled over identical untimed runs right after it"
        clocks = sampler.stop(windows)
        if note:
            clocks["note"] = note
    k1_ms, k2_ms = kernel_times(eng)
    path = eng.fft_path(0)
    value = world * samples_per_step * args.steps / (elapsed_ms * 1e-3) / 1e6

    # ---- e2e: host buffers through the public API (push H2D + run + fetch D2H) ----
    e2e = None
    if not args.no_e2e:
        eng2 = lib.Engine(cfg, cuda_device=local_rank, max_batches_per_run=NB_RUN, input_capacity_batches=2 * NB_RUN + 1, fft_mode=args.fft_mode)
        step_items = [NB_RUN * B * hop[d] * 2 for d in range(D)]          # array items per engine run per device
        prime_items = [(100 * hop[d] + cfg.fft_size) * 2 for d in range(D)]
        pinned = [torch.from_numpy(np.ascontiguousarray(raws[d][:prime_items[d] + step_items[d]])).pin_memory() for d in range(D)]
        # the caller's arrays; with --dump-outputs every run of a step fetches into its own (written here, so that no page is
        # first touched inside the timed loop)
        keep = runs_per_step if args.dump_outputs else 1
        wo = [[np.full((NB_RUN, len(cfg.devices[d].channels), B), 0, np.float32) for d in range(D)] for _ in range(keep)]
        ax = [[np.full((NB_RUN, len(cfg.devices[d].channels)), 0, np.uint8) for d in range(D)] for _ in range(keep)]
        collected = [0]
        item = [cfg.devices[d].bytes_per_sample for d in range(D)]

        def submit(first: bool):
            for d in range(D):
                base = pinned[d].data_ptr()
                if first:
                    eng2.push_ptr(d, base, (prime_items[d] + step_items[d]) * item[d])
                else:  # replay the same 4 batches of host samples (skipping the priming part)
                    eng2.push_ptr(d, base + prime_items[d] * item[d], step_items[d] * item[d])
            n = eng2.run(NB_RUN)
            assert n == D * NB_RUN, (n, D * NB_RUN)

        def collect():
            k = collected[0] % keep
            for d in range(D):
                assert eng2.fetch_many_into(d, NB_RUN, wo[k][d], ax[k][d]) == NB_RUN
            collected[0] += 1

        submit(True)
        for _ in range(max(args.warmup, 1) * min(runs_per_step, 4)):
            submit(False)
            collect()
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps * runs_per_step):
            submit(False)   # run i+1 in flight ...
            collect()       # ... while run i's results are fetched (every run's input and output cross PCIe in here)
        eng2.sync()
        barrier()
        dt = max_over_ranks(time.perf_counter() - t0)
        collect()
        G = sum(len(dv.channels) for dv in cfg.devices)
        h2d_step = int(sum(step_items[d] * item[d] for d in range(D))) * runs_per_step
        e2e = {"value": world * samples_per_step * args.steps / dt / 1e6, "unit": UNIT, "h2d_bytes_per_step": h2d_step,
               "d2h_bytes_per_step": int(G * NB_RUN * B * 4 + NB_RUN * ((G + 31) // 32 * 32)) * runs_per_step,
               "timing": "wall clock around synchronised steps (includes host-side copies out of the pinned result slots)",
               "h2d_gbs_achieved": h2d_step * args.steps / dt / 1e9,
               "pcie": pcie, "pcie_frac": (h2d_step * args.steps / dt / 1e9) / pcie["h2d_gbs"] if pcie else None, "numa": numa}
        if pcie and e2e["pcie_frac"] > 1.0:
            e2e["pcie_note"] = "the streaming path moved bytes faster than the copy-rate probe: the probe understates this box's H2D rate"
        if args.dump_outputs and rank == 0:
            last = [(collected[0] - keep + i) % keep for i in range(keep)]  # the step's runs, oldest first
            e2e["dump_outputs"] = dump_outputs(args.dump_outputs, [(wo[k], ax[k]) for k in last])
        eng2.close()
        del pinned

    # ---- roofline of K1 ----
    peaks, peak_src = measured_peaks()
    N = cfg.fft_size
    frames_per_launch = D * NB_RUN * B
    alg_bytes = alg_bytes_per_run(cfg, NB_RUN)
    achieved = alg_bytes / (k1_ms * 1e-3) / 1e9
    kern = {1: "k1_fft_kernel (convert+window+full FFT+bin select, FP32)", 2: "k1_pruned_kernel (convert+window+output-pruned FFT, FP32)",
            3: "k1_tc_kernel (raw bytes x window*twiddle digits as an int8 GEMM on tcgen05, S32 accumulators in TMEM)"}[path]
    src_of = {1: "rtlsdr-airband_b200/csrc/k1_fft.cu", 2: "rtlsdr-airband_b200/csrc/k1_pruned.cu", 3: "rtlsdr-airband_b200/csrc/k1_tc.cu"}[path]
    sha = source_sha(src_of)
    traffic, issue = None, None
    tpath = os.path.join(ROOT, "profiles", "k1_captures.json")
    if os.path.exists(tpath):
        try:
            for cap in json.load(open(tpath)):
                if cap.get("workload") == args.workload and cap.get("fft_path") == path and cap.get("source_sha") == sha:
                    traffic = cap.get("dram_bytes_per_launch")
                    if cap.get("warp_instructions_per_launch"):
                        sm_mhz = (clocks or {}).get("sm_mhz") or 1965.0
                        issue = {"warp_instructions_per_launch": cap["warp_instructions_per_launch"],
                                 "issue_frac": cap["warp_instructions_per_launch"] / (148 * 4 * sm_mhz * 1e6 * k1_ms * 1e-3),
                                 "from": cap.get("file")}
        except Exception:
            pass
    roofline = {"bound": "hbm", "kernel": kern, "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": achieved / peaks["hbm_gbs"],
                "peak_source": peak_src + " (MEASURED_PEAKS.json hbm_gbs)" if peak_src == "measured" else "fallback 6650 GB/s",
                "traffic": traffic, "traffic_note": None if traffic else f"no ncu capture of this kernel source (sha {sha}) under profiles/k1_captures.json",
                "alg_bytes_per_launch": alg_bytes, "k1_ms": k1_ms, "k2_ms": k2_ms, "k1_share_of_kernel_time": k1_ms / max(k1_ms + k2_ms, 1e-12),
                "kernel_source_sha": sha, "issue": issue,
                "equivalent_fft_tflops": frames_per_launch * (5 * N * math.log2(N) + 2 * N) / (k1_ms * 1e-3) / 1e12,
                "equivalent_fft_note": "nominal 5*N*log2(N)+2N flop per frame of the full FFT the reference runs; NOT executed work"}
    # K2 (the per-channel state machine) is bound by instruction issue / dependent latency, not by bytes: report what it executed
    k2 = {"k2_ms": k2_ms, "bound": "sequential recurrences per channel: issue / dependent-latency bound (see DESIGN.md K2)",
          "samples_per_launch": int(sum(len(dv.channels) for dv in cfg.devices)) * NB_RUN * B}
    if os.path.exists(tpath):
        try:
            k2sha = source_sha("rtlsdr-airband_b200/csrc/k2_demod.cu")
            for cap in json.load(open(tpath)):
                if cap.get("workload") == args.workload and cap.get("fft_path") == "k2" and cap.get("source_sha") == k2sha and cap.get("warp_instructions_per_launch"):
                    sm_mhz = (clocks or {}).get("sm_mhz") or 1965.0
                    k2.update({"warp_instructions_per_launch": cap["warp_instructions_per_launch"],
                               "warp_instructions_per_sample": cap["warp_instructions_per_launch"] / k2["samples_per_launch"],
                               "issue_frac": cap["warp_instructions_per_launch"] / (148 * 4 * sm_mhz * 1e6 * k2_ms * 1e-3), "from": cap.get("file")})
        except Exception:
            pass
    roofline["k2"] = k2
    if path == 3:
        C = max(len(dv.channels) for dv in cfg.devices)
        nc = (4 * ((2 * C + 7) // 8 * 8) + 15) // 16 * 16
        macs = frames_per_launch * 2 * N * nc
        roofline["tensor"] = {"int8_macs_per_launch": macs, "achieved_tops": 2 * macs / (k1_ms * 1e-3) / 1e12,
                              "note": "executed tcgen05 kind::i8 work (frames x 2N bytes x columns); B200 int8 dense nominal 4500 TOPS"}

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": elapsed_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": dict(base_config, l2=(f"resident input {resident_bytes / 1e6:.0f} MB per engine run > 126 MB L2 (no flush needed)" if resident_bytes > 126e6
                                            else f"resident input {resident_bytes / 1e6:.0f} MB per engine run fits L2: value is L2-warm"),
                           k1_path=path),
            "clocks": clocks, "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline}
    eng.close()

    # ---- the other BASELINE configs ----
    if not args.no_configs:
        legs = {}
        leg_names = ["cfg1", "cfg3", "cfg3f", "cfg4", "cfg5"] if world == 1 else ["cfg5"]
        for name in leg_names:
            if name == args.workload:
                continue
            try:
                c, cdesc = make_workload(name)
                r = synth_streams(c, NB_RUN)
                e = resident_engine(c, r, fft_mode=0)
                mixers = None
                if name == "cfg4":
                    from airband_b200 import workloads as wl
                    mixers = [m[1] for m in wl.mixers_cfg4(c)]
                    e.configure_mixers(mixers)
                spr = sum(NB_RUN * c.wave_batch * c.hop(d) for d in range(len(c.devices)))
                ms_probe, _, _ = time_resident(e, 3, 3)
                n_runs = int(max(10, min(400, 0.4e3 / max(ms_probe / 3, 1e-3))))      # about 0.4 s of device time
                ms, nl, _ = time_resident(e, n_runs, 3)
                a1, a2 = kernel_times(e)
                ab = alg_bytes_per_run(c, NB_RUN)
                leg = {"workload": cdesc, "value": world * spr * n_runs / (ms * 1e-3) / 1e6, "unit": UNIT, "engine_runs_timed": n_runs,
                       "ms_per_engine_run": ms / n_runs, "k1_ms": a1, "k2_ms": a2, "k1_path": e.fft_path(0),
                       "hbm_frac": ab / (a1 * 1e-3) / 1e9 / peaks["hbm_gbs"], "alg_bytes_per_launch": ab, "gpu_launches": int(nl),
                       "realtime_floor_msps": sum(dv.sample_rate for dv in c.devices) / 1e6}
                # issue-slot use of the two kernels, when profiles/k1_captures.json holds ncu captures of these exact sources
                try:
                    sm_hz = ((clocks or {}).get("sm_mhz") or 1965.0) * 1e6
                    src_k1 = {1: "rtlsdr-airband_b200/csrc/k1_fft.cu", 2: "rtlsdr-airband_b200/csrc/k1_pruned.cu", 3: "rtlsdr-airband_b200/csrc/k1_tc.cu"}[leg["k1_path"]]
                    want = {leg["k1_path"]: ("k1", source_sha(src_k1), a1), "k2": ("k2", source_sha("rtlsdr-airband_b200/csrc/k2_demod.cu"), a2)}
                    for cap in (json.load(open(tpath)) if os.path.exists(tpath) else []):
                        w_ = want.get(cap.get("fft_path"))
                        if cap.get("workload") == name and w_ and cap.get("source_sha") == w_[1] and cap.get("warp_instructions_per_launch"):
                            leg[w_[0] + "_issue_frac"] = cap["warp_instructions_per_launch"] / (148 * 4 * sm_hz * w_[2] * 1e-3)
                            if w_[0] == "k1":
                                leg["k1_dram_traffic_over_alg_bytes"] = cap["dram_bytes_per_launch"] / ab
                except Exception:
                    pass
                e.close()
                if rank == 0 and world == 1 and not args.no_parity:
                    try:
                        leg["parity_spot"] = parity_spot(c, r, NB_RUN, relaxed=name in ("cfg3", "cfg3f"), mixers=mixers)
                    except Exception as ex:
                        leg["parity_spot"] = {"ok": False, "why": f"{type(ex).__name__}: {ex}"[:300]}
                legs[name] = leg
            except Exception as ex:
                legs[name] = {"error": f"{type(ex).__name__}: {ex}"[:300]}
        if world > 1:
            try:  # the one collective of the path: mixers whose inputs live on every rank (SURVEY.md §8e, mixer.cpp:189-214)
                from airband_b200 import shard
                from airband_b200 import workloads as wl
                c = wl.cfg4()
                r = synth_streams(c, NB_RUN)
                e = resident_engine(c, r, fft_mode=0)
                mixers = [m[1] for m in wl.mixers_cfg4(c)]
                e.configure_mixers(mixers)     # this rank's 4 devices feed all 4 mixers; the other ranks' partial sums arrive by NCCL
                sums, flags = shard.engine_mixer_tensors(e, len(mixers))

                def allreduce():
                    e.join()
                    with torch.cuda.stream(stream):
                        shard.allreduce_mixers(sums, flags)
                ms_plain, _, _ = time_resident(e, 50, 5)
                ms_coll, _, _ = time_resident(e, 50, 5, after_run=allreduce)
                legs["cfg4_mixer_allreduce"] = {"workload": f"cfg4 shape per rank (4 devices x 4 channels), 4 mixers spanning all {world} ranks, partial sums "
                                                            "all-reduced in place by NCCL after every engine run",
                                                "ms_per_engine_run_without_collective": ms_plain / 50, "ms_per_engine_run_with_collective": ms_coll / 50,
                                                "allreduce_bytes_per_run": int(sums.numel() * 4 + flags.numel() * 4), "world": world}
                e.close()
            except Exception as ex:
                legs["cfg4_mixer_allreduce"] = {"error": f"{type(ex).__name__}: {ex}"[:300]}
        line["configs"] = legs

    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            _, info, _ = cpu_run(cfg, desc, steps=3, warmup=1, budget_s=12.0)
            line["cpu_baseline"] = info
        except Exception as ex:  # the oracle is a checker; its absence must not hide the GPU number
            line["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "port", "sample": f"unavailable: {ex}"}
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
