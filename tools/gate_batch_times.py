"""The reference's per-gate OpenMP scheduler over the shim (examples/tb_omp_gates.cpp) at several OMP_NUM_THREADS, against the
level-synchronous evaluator's own Clock on the same circuit and inputs.

For each circuit and thread count: wall time of the OpenMP run, bootstraps, blind-rotation launches and bootstraps per launch (how many
concurrent single-gate calls bfhe_eval_bingate_host combined into one wave on average), and whether the output ciphertexts equal
Clock's word for word.  The Clock time is the second of two clocks (the first captures the circuit's graph).  OMP_WAIT_POLICY=passive.
Prints the GPU's name, power limit and max SM clock first.  Needs build() (the example binary) and a GPU.

    python tools/gate_batch_times.py [--threads 1,16,64,148,296] [--circuits mult_32x32,AES-non-expanded] [--aes-one-thread]
                                     [--json out.jsonl]
"""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bfhe_loader  # noqa: E402


def gpu_info():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        return "unknown (%s)" % e


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--threads", default="1,16,64,148,296")
    ap.add_argument("--circuits", default="mult_32x32,AES-non-expanded")
    ap.add_argument("--aes-one-thread", action="store_true", help="also run AES at one thread (one wave latency per gate)")
    ap.add_argument("--json", help="append one JSON line per point to this file")
    a = ap.parse_args()
    B = bfhe_loader.load_package()
    exe = os.path.join(os.path.dirname(B.LIB_PATH), "examples", "tb_omp_gates")
    if not os.path.exists(exe):
        sys.exit("examples/tb_omp_gates is not built: run build() first")
    gpu = gpu_info()
    print("GPU:", gpu, "| host CPUs:", os.cpu_count())
    host = B.Context(B.STD128_OPT, B.GINX, -1)
    tmp = tempfile.mkdtemp(prefix="gate_batch_")
    print("%-18s %7s %10s %10s %10s %9s %10s %8s" % ("circuit", "threads", "omp_ms", "bootstraps", "br_launch", "boots/ln", "clock_ms", "ct_equal"))
    for name in a.circuits.split(","):
        path = os.path.join(tmp, name + ".out")
        c = B.Circuit(host)
        c.load_npz(os.path.join(ROOT, "tests", "golden", "circuits", name + ".npz"))
        c.write_out(path)
        c.close()
        for t in (int(x) for x in a.threads.split(",")):
            if t == 1 and name.startswith("AES") and not a.aes_one_thread:
                continue
            env = dict(os.environ, OMP_NUM_THREADS=str(t), OMP_WAIT_POLICY="passive")
            r = subprocess.run([exe, path, "-s", "STD128_OPT", "-m", "GINX"], capture_output=True, text=True, env=env)
            if r.returncode != 0:
                sys.exit("%s at %d threads failed (%d):\n%s%s" % (name, t, r.returncode, r.stdout[-2000:], r.stderr[-2000:]))
            kv = dict(re.findall(r"^(\w+) (\S+)$", r.stdout, flags=re.M))
            rec = dict(circuit=name, threads=t, omp_wall_ms=float(kv["omp_wall_ms"]), bootstraps=int(kv["bootstraps"]),
                       br_launches=int(kv["br_launches"]), bootstraps_per_launch=float(kv["bootstraps_per_launch"]),
                       clock_ms=float(kv["clock_ms"]), ct_equal=kv["ct_equal"] == "1", gpu=gpu)
            print("%-18s %7d %10.1f %10d %10d %9.2f %10.1f %8s" % (name, t, rec["omp_wall_ms"], rec["bootstraps"], rec["br_launches"],
                                                                 rec["bootstraps_per_launch"], rec["clock_ms"], rec["ct_equal"]), flush=True)
            if a.json:
                with open(a.json, "a") as f:
                    f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
