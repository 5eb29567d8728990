"""Compact fresh ciphertexts (BFHECTS1) against full rows at STD128_OPT GINX: sizes, host encryption time, SetInput time for AES-128 on a
key-less evaluator, and device expansion against the host-to-device copy of the same full rows.

Every device time is the wall time of a call that ends in a device synchronise (set_input_ct / set_input_compact / expand_cts to the
device / Slab.upload all return after their rows are written).  Each is measured --reps times after one warm-up, and the median is
reported with the minimum and maximum.  Prints the GPU's name, power limit and max SM clock.

    python tools/compact_ct_times.py [--reps 9] [--host-bits 65536] [--rows 1048576]
"""
import argparse
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bfhe_loader  # noqa: E402


def gpu_info():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        return "unknown (%s)" % e


def timed(f):
    t = time.perf_counter()
    f()
    return time.perf_counter() - t


def med(f, reps):
    """(median, min, max) seconds of reps calls after one warm-up"""
    f()
    ts = [timed(f) for _ in range(reps)]
    return statistics.median(ts), min(ts), max(ts)


def fmt(t):
    return "median %.3f ms (min %.3f, max %.3f)" % tuple(1e3 * x for x in t)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=9)
    ap.add_argument("--host-bits", type=int, default=1 << 16)
    ap.add_argument("--rows", type=int, default=1 << 20)
    a = ap.parse_args()
    B = bfhe_loader.load_package()
    print("GPU:", gpu_info(), "| host CPUs:", os.cpu_count(), "| reps %d after one warm-up" % a.reps)
    gen = B.Context(B.STD128_OPT, B.GINX, -1)
    gen.keygen(1)
    gen.btkeygen(2)
    st = gen.stride
    print("STD128_OPT, ct_stride %d words" % st)
    for count in (256, 768, a.rows):
        full, comp = count * st * 4, gen.ct_compact_size(count)
        print("  %8d bits: full rows %11d B (%.0f B/bit), compact %9d B (%.2f B/bit), %.0fx smaller" %
              (count, full, full / count, comp, comp / count, full / comp))
    rng = np.random.default_rng(1)
    bits = rng.integers(0, 2, size=a.host_bits).astype(np.uint8)
    print("host encryption of %d bits: bfhe_encrypt %s; bfhe_encrypt_compact %s" %
          (bits.size, fmt(med(lambda: gen.encrypt(bits), a.reps)), fmt(med(lambda: gen.encrypt_compact(bits), a.reps))))

    ev = B.Context(B.STD128_OPT, B.GINX, 0)
    ev.import_keys(gen.export_keys(include_sk=False))
    c = B.Circuit(ev)
    c.load_npz(os.path.join(ROOT, "tests", "golden", "circuits", "AES-non-expanded.npz"))
    c.Reset()
    c.setEncrypted(True)
    aes = rng.integers(0, 2, size=sum(c.info()["input_bits"])).astype(np.uint8)
    blob = gen.encrypt_compact(aes)
    rows = gen.expand_cts(blob)
    t_ct = med(lambda: c.set_input_ct(rows), a.reps)
    t_cc = med(lambda: c.set_input_compact(blob), a.reps)
    t_clock = med(lambda: (c.set_input_compact(blob), c.clock_ct()), a.reps)
    print("AES-128 (%d input bits, key-less evaluator):" % aes.size)
    print("  set_input_ct from host rows (%d B): %s" % (rows.nbytes, fmt(t_ct)))
    print("  set_input_compact (%d B):           %s" % (blob.size, fmt(t_cc)))
    print("  set_input_compact + clock_ct:       %s" % fmt(t_clock))
    c.close()

    big = gen.encrypt_compact(rng.integers(0, 2, size=a.rows).astype(np.uint8), seed=3)
    host_rows = gen.expand_cts(big)
    slab = ev.slab(a.rows)
    try:
        t_exp = med(lambda: ev.expand_cts(big, out=slab), a.reps)
        assert np.array_equal(slab.download(0, 1024), host_rows[:1024])
        t_h2d = med(lambda: slab.upload(host_rows), a.reps)
    finally:
        slab.free()
    print("%d rows into device memory: expand_cts from the compact blob (%d B) %s; H2D copy of the full rows (%d B) %s" %
          (a.rows, big.size, fmt(t_exp), host_rows.nbytes, fmt(t_h2d)))


if __name__ == "__main__":
    main()
