#!/usr/bin/env python
"""Generates tests/golden/*.npz.  Needs oracle/_ref, which oracle/Makefile builds where the original project's sources
are present (REF=<their directory>):

    python tests/golden/make_golden.py

For every case in tests/cases.py listed in GOLDEN it stores a SHA-256 of the exact raw I/Q bytes fed in and the outputs of
oracle/_ref/libairband_ref.so — i.e. the reference's OWN squelch.cpp / ctcss.cpp / filters.cpp (compiled in place
from the original sources by oracle/Makefile) behind the restated demodulate() loop and the FP32 FFT stand-in.
(The reference's main translation unit cannot be built here: lame/shout/libconfig++/fftw3 are absent.)
reference_leaf.npz holds what the same classes compute in the cases of test_oracle_leaf_vs_ref.py, test_oracle_pipeline.py
and test_oracle_scan.py (see tests/reference_outputs.py)."""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
for p in (os.path.join(ROOT, "tests"), os.path.join(ROOT, "oracle"), os.path.join(ROOT, "rtlsdr-airband_b200", "py")):
    sys.path.insert(0, p)

import oracle_py as op  # noqa: E402
import reference_outputs as ro  # noqa: E402
import test_oracle_leaf_vs_ref  # noqa: E402
import test_oracle_pipeline  # noqa: E402
import test_oracle_scan  # noqa: E402
from cases import CASES  # noqa: E402

GOLDEN = ["am_u8", "nfm_s16", "am_bw_f32", "s8_two_devices"]


def main():
    assert op.available("ref"), "build oracle/_ref first (make -C oracle REF=<original sources>)"
    for name in GOLDEN:
        cfg, raws = CASES[name]()
        res, o = op.run_oracle(cfg, raws, "ref")
        out = {}
        for d, (wo, iq, ax) in enumerate(res):
            out[f"raw{d}_sha256"] = np.array(ro.digest(raws[d]))
            out[f"waveout{d}"] = wo
            out[f"iq_out{d}"] = iq
            out[f"axc{d}"] = ax
            st = []
            for c in range(wo.shape[0]):
                s = o.stats(d, c)
                st.append([s.open_count, s.flappy_count, s.ctcss_count, s.no_ctcss_count, s.active_counter])
            out[f"counts{d}"] = np.array(st, np.int64)
        path = os.path.join(HERE, name + ".npz")
        np.savez_compressed(path, **out)
        print(name, os.path.getsize(path), "bytes")
    out = {}
    for mod in (test_oracle_leaf_vs_ref, test_oracle_pipeline, test_oracle_scan):
        mod.record_reference(out)
    np.savez_compressed(ro.PATH, **out)
    print(os.path.basename(ro.PATH), os.path.getsize(ro.PATH), "bytes")


if __name__ == "__main__":
    main()
