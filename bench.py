#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 gate-bootstrapping engine.

Metric (BASELINE.json): bootstrapped gates/sec, STD128_OPT GINX, on the synthetic wavefront of independent
NAND / AND / XOR gates (config 3: 1 048 576 gates, gate i has type i mod 3; the reference's composite XOR = 3 bootstraps,
src/gate.cpp:198-202), plus whole-circuit wall times (configs 4-5) with the CPU port's wall time beside them.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--gates G] [--impl reference] [--no-aux] [--dump-outputs DIR]

One process per GPU (torchrun for N > 1; torch.distributed is plumbing only: barrier + max-reduce of times).
A step = one pass of the hot path (bfhe_eval_bingate_batch: blind rotation + key switch) over one batch of G gates
per rank whose input ciphertexts are already resident in HBM.  By default the K timed steps together cover config 3's
1 048 576 gates per rank (G = 1 048 576 / K rounded up to whole launch waves).  `e2e` is the same step through
bfhe_eval_bingate_host with pinned HOST buffers (H2D of the inputs and D2H of the outputs inside the timed region).
"""
import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
import bfhe_loader  # noqa: E402

METRIC = "bootstrapped gates/sec (STD128_OPT GINX)"
UNIT = "bootstrapped gates/s"
CONFIG3_GATES = 1_048_576
# SURVEY 8(d): algorithmic work of one bootstrapped gate (STD128_OPT GINX): 45.25 M modular multiplications
# = 502 x [10 NTTs x 5120 butterflies + 36 N pointwise + 2 N scaling] + 3 NTT-equivalents; x3 IMAD-class instructions each
W_MODMUL = 45_250_000
W_IMAD = 3 * W_MODMUL
W_MODMUL_AP = 67_700_000  # SURVEY 8(a) row a11: ~973 active steps x 69 632
# algorithmic bytes per bootstrapped gate (DESIGN.md "roofline"): BK once per CTA tile of G gates + KSK row gather + I/O
BK_BYTES = 65_798_144
KS_ROW_BYTES = 1024 * 2 * 1024  # 2048 padded 1 KiB rows
IO_BYTES = 3 * 504 * 4
# dram__bytes_read.sum + dram__bytes_write.sum of ONE `ncu --set full` capture of the throughput kernel (see roofline.traffic_source)
STATIC_TRAFFIC = {"bytes": 74.46e6, "gates": 592, "source": "profiles/r2_blind_rotate_ncu_summary.md"}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--gates", type=int, default=0,
                    help="gates per rank per step (config 3 mix); 0 = 1 048 576 / steps, rounded up to whole waves of 4-gate CTAs")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-aux", action="store_true", help="skip the circuit wall-time / AP figures")
    ap.add_argument("--cpu-sample", type=int, default=0,
                    help="gates in the CPU baseline sample (0 = 4096 on >= 16 cores, scaled down on fewer; reference arm: 8 per core per step)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write rank 0's output ciphertexts of the last timed step (a fixed sample of rows) to DIR as .npy files")
    return ap.parse_args()


def make_workload(B, count, n_in):
    g = np.zeros(count, dtype=B.GATE_DTYPE)
    idx = np.arange(count)
    g["op"] = np.array([B.NAND, B.AND, B.XOR], dtype=np.uint32)[idx % 3]
    g["in0"] = (2 * idx) % n_in
    g["in1"] = (2 * idx + 1) % n_in
    g["out"] = n_in + idx
    boots = int(np.where(g["op"] == B.XOR, 3, 1).sum())
    return g, boots


def expected_bits(B, g, bits):
    a, b = bits[g["in0"]], bits[g["in1"]]
    return np.where(g["op"] == B.NAND, 1 - (a & b), np.where(g["op"] == B.AND, a & b, a ^ b))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (profiling recipe's clocks line)."""

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            if len(r) >= 9:
                for nm, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def oracle_with_keys(blob=None, seed_keys=(1, 2)):
    """The CPU oracle (oracle/bfhe_oracle.c: restatement of OpenFHE binfhe 1.0.x) -- used here ONLY for the cpu_baseline / reference legs
    and as the bit-exact checker of a sample of the GPU's outputs."""
    O = bfhe_loader.load_oracle()
    O.build()
    o = O.Oracle(O.STD128_OPT, O.GINX)
    if blob is not None:
        o.import_keys(blob)
    else:
        o.keygen(seed_keys[0])
    return O, o


def run_reference(args, rank):
    """--impl reference: the reference's CPU implementation of the path = the oracle port (OpenFHE itself cannot be
    built here: not vendored, no network), all host threads, same workload mix, bounded sample per step; one OpenMP task per
    ready gate of the wavefront, as the reference drives OpenFHE (src/circuit.cpp:698-710)."""
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    sample = args.cpu_sample or 8 * cores  # ~0.7 s per step on 16 cores; XOR gates are 3 serial bootstraps inside one task
    O, o = oracle_with_keys()
    n_in = 64
    bits = np.random.default_rng(42).integers(0, 2, n_in)
    slab = o.new_slab(n_in + sample)
    slab[:n_in] = o.encrypt(bits, seed=42)
    g, boots = make_workload(O, sample, n_in)
    times = []
    for it in range(args.warmup + args.steps):
        t = time.perf_counter()
        o.eval_gates(g, slab, nthreads=cores)
        dt = time.perf_counter() - t
        if it >= args.warmup:
            times.append(dt)
    ok = bool(np.array_equal(o.decrypt(slab[n_in:]), expected_bits(O, g, bits)))
    total = sum(times)
    val = boots * args.steps / total
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u32", "data": "synthetic",
            "config": {"workload": "synthetic independent NAND/AND/XOR gates, STD128_OPT GINX (config 3 mix), bounded sample per step",
                       "gates_per_step": sample, "bootstraps_per_step": boots, "xor": "composite, 3 bootstraps", "decrypt_ok": ok,
                       "arithmetic": "32-bit SIMD Shoup NTT inside a 64-bit port (oracle/bfhe_oracle.c) -- faster than OpenFHE's 64-bit path"},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port",
                             "sample": "%d gates (%d bootstraps) per step, one OpenMP task per gate, oracle/bfhe_oracle.c" % (sample, boots)},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the engine has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    B = bfhe_loader.load_package()
    ctx = B.Context(B.STD128_OPT, B.GINX, local)
    ctx.keygen(1)   # keys from seed 1 (config 3), replicated on every GPU; explicit seeds = reproducible benchmark keys, not secret ones
    ctx.btkeygen(2)
    stream = torch.cuda.Stream()  # every kernel of the engine is launched on this stream; the events below sit on it too
    torch.cuda.set_stream(stream)
    ctx.set_stream(stream.cuda_stream)

    # batch: a multiple of 3 (gate mix) x 4 (gates per CTA) x SM count, so every launch is whole waves; the K timed steps together
    # cover config 3's 1 048 576 gates per rank
    sms = torch.cuda.get_device_properties(local).multi_processor_count
    unit = 3 * 4 * sms
    count = args.gates or -(-CONFIG3_GATES // (args.steps * unit)) * unit
    n_in = 2 * count
    gates, boots = make_workload(B, count, n_in)
    bits = np.random.default_rng(42 + rank).integers(0, 2, n_in)
    st = ctx.stride
    host_in = torch.empty((n_in, st), dtype=torch.int32).pin_memory()
    host_in.numpy().view(np.uint32)[:] = ctx.encrypt(bits, seed=1000 + rank)
    host_out = torch.empty((count, st), dtype=torch.int32).pin_memory()
    slab = torch.zeros((n_in + count, st), dtype=torch.int32, device="cuda")
    slab[:n_in].copy_(host_in)
    torch.cuda.synchronize()
    slab_ptr = slab.data_ptr()

    # integer-pipe peak, measured live (the roofline denominator of this integer-bound path; SURVEY 8(d))
    imad_peak = max(ctx.microbench_int(0) for _ in range(3)) * 1e9

    # ---------------- device-resident throughput (value) ----------------
    for _ in range(args.warmup):
        ctx.eval_bingate_batch(slab_ptr, gates)
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ctx.profile_enable(True)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record(stream)
    for _ in range(args.steps):
        ctx.eval_bingate_batch(slab_ptr, gates)
    ev1.record(stream)
    barrier()
    dev_ms = max_over_ranks(ev0.elapsed_time(ev1))
    br_ms, br_n = ctx.profile_read(0)
    ks_ms, ks_n = ctx.profile_read(1)
    nt_ms, nt_n = ctx.profile_read(2)
    ctx.profile_enable(False)
    clocks = sampler.stop() if rank == 0 else None
    value = world * boots * args.steps / (dev_ms * 1e-3)

    # correctness of what was just timed: every output decrypts to the truth table
    out = slab[n_in:].cpu().numpy().view(np.uint32)
    ok = bool(np.array_equal(ctx.decrypt(out), expected_bits(B, gates, bits)))
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out, ctx.p.ct_words)

    # ---------------- end to end through the host-buffer API (e2e) ----------------
    hin, hout = host_in.numpy().view(np.uint32), host_out.numpy().view(np.uint32)
    ctx.eval_bingate_host(gates, hin, count, hout)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        ctx.eval_bingate_host(gates, hin, count, hout)
    torch.cuda.synchronize()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    barrier()
    e2e_val = world * boots * args.steps / e2e_s
    ok = ok and bool(np.array_equal(ctx.decrypt(hout), expected_bits(B, gates, bits)))
    ok = ok and bool(np.array_equal(hout, out))  # both paths: the same ciphertexts, bit for bit

    # ---------------- roofline of the dominant kernel (blind rotation) ----------------
    br_s_per_launch = br_ms * 1e-3 / max(br_n, 1)
    boots_per_launch = boots * args.steps / max(br_n, 1)
    achieved_imad = boots_per_launch * W_IMAD / br_s_per_launch
    tile = 4
    hbm_bytes_per_boot = BK_BYTES / tile + KS_ROW_BYTES + IO_BYTES
    roofline = {"bound": "int", "kernel": "blind_rotate_kernel<10,4,7,4,GINX>", "achieved": achieved_imad / 1e12,
                "peak": imad_peak / 1e12, "unit": "TIMAD/s", "frac": achieved_imad / imad_peak,
                "peak_source": "measured live: register-only IMAD microbenchmark (bfhe_microbench_int), %d SMs" % sms,
                "work_per_unit": "%d IMAD-class instr per bootstrapped gate (3 x 45.25M modular multiplications, SURVEY 8(d))" % W_IMAD,
                "kernel_ms_per_launch": 1e3 * br_s_per_launch, "kernel_share_of_step": br_ms / (br_ms + ks_ms + nt_ms),
                "gates_per_launch_avg": boots_per_launch,
                "step_ms_by_kernel": {"blind_rotate": br_ms / args.steps, "keyswitch": ks_ms / args.steps, "eval_not": nt_ms / args.steps},
                # NOT measured in this run: bytes of one `ncu --set full` capture of a 592-gate launch of this kernel (one wave of 148
                # four-gate CTAs).  The 65.8 MB key reaches DRAM once per launch and is served by L2 afterwards, so the traffic of a
                # longer launch grows only by the ciphertext I/O (6 KB per gate).
                "traffic": STATIC_TRAFFIC["bytes"], "traffic_source": "static: ncu capture of a %d-gate launch, %s; algorithmic bytes of that "
                "launch = %.1f MB (key once + I/O)" % (STATIC_TRAFFIC["gates"], STATIC_TRAFFIC["source"], (BK_BYTES + STATIC_TRAFFIC["gates"] * (IO_BYTES + 4112)) / 1e6),
                "hbm": {"achieved": boots_per_launch * hbm_bytes_per_boot / br_s_per_launch / 1e9, "peak": peak_hbm(),
                        "unit": "GB/s", "bytes_per_unit": hbm_bytes_per_boot,
                        "note": "key streaming is L2/HBM traffic shared by the %d gates of a CTA tile; the path is integer-bound" % tile}}
    roofline["hbm"]["frac"] = roofline["hbm"]["achieved"] / roofline["hbm"]["peak"]

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u32", "data": "synthetic",
            "config": {"workload": "BASELINE config 3: synthetic independent NAND/AND/XOR gates, STD128_OPT GINX; %d gates (%d bootstraps) "
                                   "per rank over the %d timed steps (stated size 1 048 576, rounded up to whole launch waves), "
                                   "%d gates/rank/step" % (count * args.steps, boots * args.steps, args.steps, count),
                       "gates_per_rank_per_step": count, "bootstraps_per_rank_per_step": boots, "gates_per_rank_timed": count * args.steps,
                       "xor": "composite, 3 bootstraps",
                       "gates_per_s": world * count * args.steps / (dev_ms * 1e-3),
                       "l2": "inputs (%d MB) + keys (330 MB) exceed the 126 MB L2" % (n_in * st * 4 // 2**20),
                       "parallelism": "replicated keys, gates sharded by rank, no data-path collective", "decrypt_ok": ok},
            "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": int(n_in * st * 4 + count * 32),
                    "d2h_bytes_per_step": int(count * st * 4)},
            "gpu_launches": int(br_n + ks_n + nt_n),
            "roofline": roofline, "clocks": clocks}
    if rank == 0 and world == 1:
        # CPU baseline = the oracle on the FIRST `sample` gates of this very workload (same keys, same input ciphertexts), one OpenMP task
        # per gate on all host cores -- which also makes it the bit-exact spot check of SURVEY 8(d) config 3 ("first 4 096 outputs")
        cores = os.cpu_count() or 1
        sample = args.cpu_sample or max(256, min(4096, 256 * cores))
        sample = min(sample, count)
        O, o = oracle_with_keys(ctx.export_keys())
        ref = o.new_slab(n_in + sample)
        ref[:2 * sample] = hin[:2 * sample]  # gate i reads rows 2i, 2i + 1
        g2 = gates[:sample].copy()
        g2["out"] = n_in + np.arange(sample)
        b2 = int(np.where(g2["op"] == B.XOR, 3, 1).sum())
        t = time.perf_counter()
        o.eval_gates(g2, ref, nthreads=cores)
        dt = time.perf_counter() - t
        w = ctx.p.ct_words
        exact = bool(np.array_equal(ref[n_in:n_in + sample, :w], out[:sample, :w]))
        line["cpu_baseline"] = {"value": b2 / dt, "unit": UNIT, "cores": cores, "kind": "port",
                                "sample": "first %d gates (%d bootstraps) of the same workload, same keys and inputs, one OpenMP task per gate, %.1f s"
                                          % (sample, b2, dt)}
        line["config"]["spot_check"] = {"gates": sample, "gpu_ciphertexts_bit_exact_vs_oracle": exact}
        ok = ok and exact
    if not args.no_aux:
        line["aux"] = aux_circuits(B, ctx, rank, world)
    if not ok:
        line["error"] = "outputs do not match (truth table / oracle spot check)"
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


DUMP_ROWS = 8192


def dump_outputs(d, out, words):
    """The output ciphertexts of the timed step, for comparing two builds output for output.  The whole set is ~400 MB at the default
    size, so a fixed seeded sample of at most DUMP_ROWS gates is written (8192 x 503 words x 8 B = 33 MB); float64 holds every 32-bit
    word exactly.  ciphertext_rows.npy holds the gate index of each sampled row."""
    n = out.shape[0]
    rows = np.arange(n) if n <= DUMP_ROWS else np.sort(np.random.default_rng(0).choice(n, size=DUMP_ROWS, replace=False))
    os.makedirs(d, exist_ok=True)
    np.save(os.path.join(d, "ciphertext_rows.npy"), rows.astype(np.float64))
    np.save(os.path.join(d, "ciphertexts.npy"), out[rows, :words].astype(np.float64))


def peak_hbm():
    try:
        return float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
    except Exception:
        return 6650.0  # fallback stated in B200_PROFILING.md


def level_blocks_digest(c, slab):
    """sha256 over the bootstrap-output rows of every level, in level order: independent of how the rows are padded for sharding"""
    h = hashlib.sha256()
    nl = c.plan_misc()["n_levels"]
    w = c.ctx.p.ct_words
    for L in range(nl):
        first, n = None, 0
        for r in range(max(1, c.world_size)):
            g, f, rpr = c.level_plan(L, r, c.world_size)
            first = f
            n += len(g) if rpr or c.world_size == 1 else (len(g) if r == 0 else 0)
        h.update(np.ascontiguousarray(slab[first:first + n, :w]).tobytes())
    return h.hexdigest()


def cpu_circuit_wall(B, name, vectors, every, cores):
    """The reference's `### Total time` (src/circuit.cpp:565-566) on the host CPU with the oracle port: the reference's ASAP waves, one
    OpenMP task per ready gate of a wave (src/circuit.cpp:698-710), waves in sequence.  every == 1: the whole circuit; every > 1: every
    `every`-th wave is executed and the total is extrapolated by bootstrap count (bootstrap time does not depend on the data)."""
    O = bfhe_loader.load_oracle()
    hctx = B.Context(B.STD128_OPT, B.GINX, device=-1)
    c = B.Circuit(hctx)
    c.load_npz(os.path.join(ROOT, "tests", "golden", "circuits", name + ".npz"))
    c.set_wave_capacity(0)  # ASAP = what the reference's manager produces
    misc = c.plan_misc()
    o = cpu_circuit_wall.oracle
    slab = o.new_slab(misc["total_rows"])
    rng = np.random.default_rng(5)
    fill = o.encrypt(rng.integers(0, 2, 64), seed=9)
    slab[:] = fill[np.arange(misc["total_rows"]) % 64]  # any valid ciphertexts: the timing does not depend on them
    done_boots, t_total, waves = 0, 0.0, 0
    total_boots = 0
    for L in range(misc["n_levels"]):
        g, _, _ = c.level_plan(L, 0, 1)
        total_boots += len(g)
        if L % every:
            continue
        t = time.perf_counter()
        if len(g):
            o.eval_gates(g, slab, nthreads=cores)
        t_total += time.perf_counter() - t
        done_boots += len(g)
        waves += 1
    c.close()
    est = t_total * total_boots / max(done_boots, 1)
    return {"cpu_wall_ms": 1e3 * est, "cpu_measured_ms": 1e3 * t_total, "cpu_waves_run": waves, "cpu_waves_total": misc["n_levels"],
            "cpu_bootstraps_run": done_boots, "cpu_bootstraps_total": total_boots, "extrapolated": every > 1}


def aux_circuits(B, ctx, rank, world):
    """Whole-circuit wall times (BASELINE configs 4-5): AES-128 and SHA-256 at every N (waves sharded over the ranks where that pays,
    ncclAllGather exchange), with `sharded_slab_equal` = every rank's wire ciphertexts equal those of an unsharded evaluation; at N = 1
    also MD5, the 32x32 multiplier and a comparator, the CPU port's wall time beside each, and the AP method's throughput."""
    import torch
    import torch.distributed as dist
    vectors = json.load(open(os.path.join(ROOT, "tests", "golden", "vectors.json")))
    res = {}
    cores = os.cpu_count() or 1
    # (name, key, repetitions -- the last one is reported; the first includes plan upload and graph capture --, CPU sampling stride)
    circuits = [("AES-non-expanded", "aes128", 2, 16), ("sha256", "sha256", 2 if world > 1 else 1, 100)]
    if world == 1:
        circuits += [("md5", "md5", 1, 50), ("mult_32x32", "mult32", 2, 1), ("comparator_32bit_signed_lt", "cmp32", 2, 1)]
    for name, key, reps, every in circuits:
        vec = vectors[name]["vectors"][1]
        c = B.Circuit(ctx)
        c.load_npz(os.path.join(ROOT, "tests", "golden", "circuits", name + ".npz"))
        if world > 1:
            uid = torch.from_numpy(B.nccl_unique_id() if rank == 0 else np.zeros(128, dtype=np.uint8)).cuda()
            dist.broadcast(uid, 0)
            c.set_sharding(rank, world, uid.cpu().numpy())
        for rep in range(reps):
            c.Reset()
            c.setEncrypted(True)
            c.SetInput(vec["inputs"], seed=7)
            if world > 1:
                dist.barrier()
            t = time.perf_counter()
            out = c.Clock()[0]
            wall = time.perf_counter() - t
            sch = c.schedule()
            res.update({key + "_wall_ms": 1e3 * wall, key + "_device_ms": c.stats()["device_ms"], key + "_kat_ok": out == vec["golden"],
                        key + "_bootstraps": c.info()["bootstraps"], key + "_levels": c.info()["levels"],
                        key + "_waves": sch["n_levels"] - 1, key + "_waves_sharded": sch["n_sharded"], key + "_wave_cap": sch["wave_cap"]})
        res["launch_cost_ms_probe"] = sch["cost_ms"]
        res["exchange"] = {0: "none (1 GPU)", 1: "ncclAllGather per sharded wave", 2: "key switch stores into every rank's slab (CUDA IPC + NVLink), flag per wave"}[c.exchange_mode()]
        if world > 1:  # every rank: same wire ciphertexts as an unsharded evaluation of the same schedule on this GPU
            mine = level_blocks_digest(c, c.download_slab())
            c1 = B.Circuit(ctx)
            c1.load_npz(os.path.join(ROOT, "tests", "golden", "circuits", name + ".npz"))
            c1.set_wave_capacity(sch["wave_cap"])
            c1.Reset()
            c1.setEncrypted(True)
            c1.SetInput(vec["inputs"], seed=7)
            out1 = c1.Clock()[0]
            same = (level_blocks_digest(c1, c1.download_slab()) == mine) and out1 == vec["golden"]
            c1.close()
            t = torch.tensor([1 if same else 0], device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
            res[key + "_sharded_slab_equal"] = bool(int(t.item()))
        c.close()
        if world == 1 and rank == 0:
            if not hasattr(cpu_circuit_wall, "oracle"):
                cpu_circuit_wall.oracle = oracle_with_keys(ctx.export_keys())[1]
            cpu = cpu_circuit_wall(B, name, vectors, every, cores)
            res.update({key + "_" + k: v for k, v in cpu.items()})
            res[key + "_cpu_kind"] = "port"
            res[key + "_cpu_cores"] = cores
            res[key + "_speedup_vs_cpu"] = cpu["cpu_wall_ms"] / res[key + "_wall_ms"]
    if world == 1:
        res["ap"] = ap_line(B, ctx.device)
    return res


def ap_line(B, device):
    """STD128_OPT with the AP (DM) method: bootstrapped gates/s on independent NAND gates and the integer roofline against SURVEY 8(a)
    row a11's 67.7 M modular multiplications per gate."""
    import torch
    ctx = B.Context(B.STD128_OPT, B.AP, device)
    ctx.keygen(1)
    ctx.btkeygen(2)
    sms = torch.cuda.get_device_properties(device).multi_processor_count
    count = 4 * sms * 8
    n_in = 256
    bits = np.random.default_rng(3).integers(0, 2, n_in)
    slab = ctx.slab(n_in + count)
    slab.upload(ctx.encrypt(bits, seed=11))
    idx = np.arange(count)
    g = np.zeros(count, dtype=B.GATE_DTYPE)
    g["op"], g["in0"], g["in1"], g["out"] = B.NAND, idx % n_in, (idx * 7 + 1) % n_in, n_in + idx
    ctx.eval_bingate_batch(slab, g)
    ctx.sync()
    imad_peak = max(ctx.microbench_int(0) for _ in range(3)) * 1e9
    reps = 3
    t = time.perf_counter()
    for _ in range(reps):
        ctx.eval_bingate_batch(slab, g)
    ctx.sync()
    dt = time.perf_counter() - t
    dec = ctx.decrypt(slab.download(n_in, count))
    ok = bool(np.array_equal(dec, 1 - (bits[g["in0"]] & bits[g["in1"]])))
    rate = reps * count / dt
    # one narrow wave (what a deep circuit's level costs with AP): the cost model's choice for 33 gates = the 4-CTA cluster form
    ctx.eval_bingate_batch(slab, g[:33])
    ctx.sync()
    ctx.profile_enable(True)
    ctx.eval_bingate_batch(slab, g[:33])
    ctx.sync()
    wave_br, _ = ctx.profile_read(0)
    wave_ks, _ = ctx.profile_read(1)
    ctx.profile_enable(False)
    slab.free()
    ctx.close()
    return {"metric": "bootstrapped gates/sec (STD128_OPT AP)", "value": rate, "gates_per_step": count, "decrypt_ok": ok,
            "wave_33_gates_ms": {"blind_rotate": wave_br, "key_switch": wave_ks},
            "roofline": {"bound": "int", "achieved": rate * 3 * W_MODMUL_AP / 1e12, "peak": imad_peak / 1e12, "unit": "TIMAD/s",
                         "frac": rate * 3 * W_MODMUL_AP / imad_peak, "work_per_unit": "3 x 67.7M modular multiplications per gate (SURVEY 8(a) a11)"}}


if __name__ == "__main__":
    main()
