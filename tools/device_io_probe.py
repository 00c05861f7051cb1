"""GPU-resident I/O against the two existing legs of bench.py, in one process on one GPU (needs a CUDA device):

  resident  abg_run_resident on the HBM-resident replay stream (bench.py's `value` leg), CUDA events on the engine's stream
  host      abg_push from pinned host memory + abg_run + abg_fetch_batches into host arrays (bench.py's `e2e` leg), wall
            clock around synchronised steps
  device    Engine.push_tensor from CUDA tensors + abg_run + Engine.fetch_all_tensors into preallocated CUDA tensors,
            CUDA events on the torch stream (every push waits on it and every fetch is ordered on it, so the events
            bracket the whole step); the host-side enqueue time of a step is reported beside it

plus the gather kernel alone (bytes it reads and writes over 7.7 TB/s, the HBM3e figure of one B200) and the D2D push
copy alone, and a bit-for-bit check of the device path against the host path on the same seeded inputs.

    python tools/device_io_probe.py [--configs cfg2,cfg5] [--runs 40] [--warmup 8] [--out FILE.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "rtlsdr-airband_b200", "py"), ROOT]

import numpy as np  # noqa: E402

HBM_TBS = 7.7
NB = 4  # batches per run, as bench.py's NB_RUN


def gpu_description():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = (x.strip() for x in q.split(","))
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as ex:  # the numbers are still reported, without the card's settings
        return {"error": str(ex)}


def median(xs):
    return float(np.median(np.asarray(xs, np.float64)))


def probe(name, runs, warmup):
    import torch
    import bench
    from airband_b200 import lib

    cfg, desc = bench.make_workload(name)
    D, B = len(cfg.devices), cfg.wave_batch
    G = sum(len(d.channels) for d in cfg.devices)
    hop = [cfg.hop(d) for d in range(D)]
    item = [cfg.devices[d].bytes_per_sample for d in range(D)]
    raws = bench.synth_streams(cfg, NB)
    samples_per_run = sum(NB * B * hop[d] for d in range(D))
    step_items = [NB * B * hop[d] * 2 for d in range(D)]
    prime_items = [(100 * hop[d] + cfg.fft_size) * 2 for d in range(D)]
    stream = torch.cuda.current_stream()
    out = {"config": desc, "samples_per_run": samples_per_run, "runs_timed": runs}

    # ---- resident ----
    e = lib.Engine(cfg, max_batches_per_run=NB, input_capacity_batches=NB + 1)
    e.set_stream(stream.cuda_stream)
    for d in range(D):
        e.resident_load(d, raws[d])
    for _ in range(warmup):
        e.run_resident(NB)
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    for _ in range(runs):
        e.run_resident(NB)
    e.join()
    ev1.record(stream)
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1) / runs
    out["resident"] = {"ms_per_run": ms, "gsamples_per_s": samples_per_run / ms / 1e6}
    e.close()

    # ---- host (pinned H2D in, pinned slots out) ----
    e = lib.Engine(cfg, max_batches_per_run=NB, input_capacity_batches=2 * NB + 1)
    pinned = [torch.from_numpy(np.ascontiguousarray(raws[d][:prime_items[d] + step_items[d]])).pin_memory() for d in range(D)]
    wo_h = [np.zeros((NB, len(cfg.devices[d].channels), B), np.float32) for d in range(D)]
    ax_h = [np.zeros((NB, len(cfg.devices[d].channels)), np.uint8) for d in range(D)]

    def h_submit(first):
        for d in range(D):
            base = pinned[d].data_ptr()
            if first:
                e.push_ptr(d, base, (prime_items[d] + step_items[d]) * item[d])
            else:
                e.push_ptr(d, base + prime_items[d] * item[d], step_items[d] * item[d])
        assert e.run(NB) == D * NB

    def h_collect():
        for d in range(D):
            assert e.fetch_many_into(d, NB, wo_h[d], ax_h[d]) == NB

    h_submit(True)
    for _ in range(warmup):
        h_submit(False)
        h_collect()
    e.sync()
    t0 = time.perf_counter()
    for _ in range(runs):
        h_submit(False)
        h_collect()
    e.sync()
    dt = (time.perf_counter() - t0) / runs
    h_collect()
    out["host"] = {"ms_per_run": dt * 1e3, "gsamples_per_s": samples_per_run / dt / 1e9, "timing": "wall clock, pipelined as bench.py's e2e leg"}
    e.close()
    del pinned

    # ---- device (CUDA tensors in and out) ----
    dev_in = [torch.from_numpy(np.ascontiguousarray(raws[d][:prime_items[d] + step_items[d]])).cuda() for d in range(D)]
    prime_t = [dev_in[d] for d in range(D)]
    step_t = [dev_in[d][prime_items[d]:] for d in range(D)]
    e = lib.Engine(cfg, max_batches_per_run=NB, input_capacity_batches=2 * NB + 1)
    e.results_on_device()
    outs = [(torch.empty((NB, G, B), dtype=torch.float32, device="cuda"), None, torch.empty((NB, G), dtype=torch.uint8, device="cuda"))
            for _ in range(2)]

    def d_step(first, k):
        for d in range(D):
            e.push_tensor(d, prime_t[d] if first else step_t[d])
        assert e.run(NB) == D * NB
        e.fetch_all_tensors(NB, out=outs[k % 2])

    d_step(True, 0)
    for k in range(warmup):
        d_step(False, k)
    torch.cuda.synchronize()
    ev0.record(stream)
    t0 = time.perf_counter()
    for k in range(runs):
        d_step(False, k)
    t_enq = (time.perf_counter() - t0) / runs
    ev1.record(stream)
    torch.cuda.synchronize()
    t_all = (time.perf_counter() - t0) / runs
    ms = ev0.elapsed_time(ev1) / runs
    out["device"] = {"ms_per_run": ms, "gsamples_per_s": samples_per_run / ms / 1e6,
                     "host_enqueue_ms_per_run": t_enq * 1e3, "wall_ms_per_run": t_all * 1e3,
                     "gsamples_per_s_wall": samples_per_run / t_all / 1e9}

    # ---- the gather kernel alone: one fetch_all of a finished run, events around it ----
    gms = []
    for k in range(10):
        for d in range(D):
            e.push_tensor(d, step_t[d])
        e.run(NB)
        torch.cuda.synchronize()
        torch.cuda._sleep(20_000_000)  # the GPU is busy while the host enqueues: the events time the device work only
        ev0.record(stream)
        l0 = e.launch_count()
        e.fetch_all_tensors(NB, out=outs[0])
        launches = e.launch_count() - l0
        ev1.record(stream)
        torch.cuda.synchronize()
        gms.append(ev0.elapsed_time(ev1))
    gbytes = 2 * (NB * G * B * 4 + NB * G)  # read the slot, write the caller's buffers (audio + squelch flags)
    g = median(gms)
    out["gather"] = {"ms": g, "bytes": gbytes, "tb_per_s": gbytes / g / 1e9, "frac_of_hbm_7_7_tbs": gbytes / g / 1e9 / HBM_TBS,
                     "launches_per_fetch_all": int(launches), "timing": "median of 10, CUDA events around one fetch_all_tensors enqueued behind a sleep"}

    # ---- the D2D push copy alone ----
    pms = []
    for k in range(10):
        torch.cuda.synchronize()
        torch.cuda._sleep(200_000_000)
        ev0.record(stream)
        for d in range(D):
            e.push_tensor(d, step_t[d])  # each push_tensor makes the stream wait for the engine's copy
        ev1.record(stream)
        torch.cuda.synchronize()
        pms.append(ev0.elapsed_time(ev1))
        e.run(NB)
        e.fetch_all_tensors(NB, out=outs[0])
    pbytes = sum(step_items[d] * item[d] for d in range(D))
    p = median(pms)
    out["push_copy"] = {"ms": p, "bytes": pbytes, "tb_per_s": 2 * pbytes / p / 1e9, "share_of_device_run": p / out["device"]["ms_per_run"],
                        "timing": "median of 10, CUDA events around one run's pushes enqueued behind a sleep (read + write bytes in tb_per_s)"}
    e.close()

    # ---- outputs: device path == host path on the same seeded inputs, three runs ----
    eh = lib.Engine(cfg, max_batches_per_run=NB, input_capacity_batches=2 * NB + 1)
    ed = lib.Engine(cfg, max_batches_per_run=NB, input_capacity_batches=2 * NB + 1)
    ed.results_on_device()
    same = True
    for r in range(3):
        for d in range(D):
            src = raws[d][:prime_items[d] + step_items[d]] if r == 0 else raws[d][prime_items[d]:prime_items[d] + step_items[d]]
            eh.push(d, src)
            ed.push_tensor(d, prime_t[d] if r == 0 else step_t[d])
        assert eh.run(NB) == ed.run(NB) == D * NB
        wo, iq, ax = ed.fetch_all_tensors(NB)
        wo, iq, ax = wo.cpu().numpy(), iq.cpu().numpy(), ax.cpu().numpy()
        g0 = 0
        for d in range(D):
            Cn = len(cfg.devices[d].channels)
            for b in range(NB):
                hw, hi, ha = eh.fetch(d)
                same &= np.array_equal(hw.view(np.uint32), wo[b, g0:g0 + Cn].view(np.uint32))
                same &= np.array_equal(hi.view(np.uint64), iq[b, g0:g0 + Cn].view(np.uint64))
                same &= np.array_equal(ha, ax[b, g0:g0 + Cn])
            g0 += Cn
    out["outputs_equal_host_path"] = bool(same)
    eh.close()
    ed.close()
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--configs", default="cfg2,cfg5")
    ap.add_argument("--runs", type=int, default=40)
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--out", help="also write the full result as indented JSON to this file")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("device_io_probe.py: no CUDA device")
    res = {"gpu": gpu_description(), "torch_device": torch.cuda.get_device_name(0), "results": {}}
    with torch.cuda.stream(torch.cuda.Stream()):  # a stream of its own, as bench.py's legs use
        for name in args.configs.split(","):
            res["results"][name] = probe(name, args.runs, args.warmup)
            print(json.dumps({name: res["results"][name]}), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res["gpu"]))


if __name__ == "__main__":
    main()
