"""Key blob sizes, host key-generation time and device import time, full (BFHEKEY1) vs compact (BFHEKEY2), at STD128_OPT GINX and AP.

Import time is the wall time of Context.import_keys from a blob in host memory, ending in a device synchronise: the first import of each
kind is a warm-up and is excluded, and the median of the next --reps is reported.  Prints the GPU's name, power limit and max SM clock.

    python tools/key_import_times.py [--reps 5] [--methods GINX,AP]
"""
import argparse
import os
import statistics
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--methods", default="GINX,AP")
    a = ap.parse_args()
    B = bfhe_loader.load_package()
    print("GPU:", gpu_info(), "| host CPUs:", os.cpu_count())
    for m in a.methods.split(","):
        M = getattr(B, m)
        gen = B.Context(B.STD128_OPT, M, -1)
        gen.keygen(1)
        t_full = timed(lambda: gen.btkeygen(2))
        full = gen.export_keys(include_sk=False)
        t_comp = timed(lambda: gen.btkeygen_compact(2))
        comp = gen.export_keys_compact(include_sk=False)
        del gen
        dev = B.Context(B.STD128_OPT, M, 0)
        res = {}
        for name, blob in (("full", full), ("compact", comp)):
            ts = []
            for _ in range(a.reps + 1):
                ts.append(timed(lambda: (dev.import_keys(blob), dev.sync())))
            res[name] = ts[1:]
        print("STD128_OPT %s: blob full %d B, compact %d B (%.2fx smaller)" % (m, full.size, comp.size, full.size / comp.size))
        print("  host keygen: btkeygen %.2f s, btkeygen_compact %.2f s" % (t_full, t_comp))
        for name in ("full", "compact"):
            ts = res[name]
            print("  import %-7s: median %.1f ms (min %.1f, max %.1f, %d reps after one warm-up)" %
                  (name, 1e3 * statistics.median(ts), 1e3 * min(ts), 1e3 * max(ts), len(ts)))
        del dev


if __name__ == "__main__":
    main()
