"""Combining of concurrent bfhe_eval_bingate_host calls into shared GPU waves, and the host-side EvalNOT (bfhe_eval_not_host).

Threads that call EvalBinGate / Bootstrap / eval_bingate_host on one context at the same time (ctypes releases the GIL during the call)
are combined into one wave; every call must return exactly what it returns when made alone.  bfhe_dbg_hold_batches makes the combining
deterministic: while the hold is on, calls queue and nothing launches."""
import os
import re
import subprocess
import threading
import time

import numpy as np
import pytest

from conftest import shared_keys
from helpers import VECTORS, load_circuit

N_THREADS = 64


def _truth(op, a, b):
    g = op & 0xff
    a ^= (op >> 8) & 1
    b ^= (op >> 9) & 1
    return {0: a | b, 1: a & b, 2: 1 - (a | b), 3: 1 - (a & b), 4: a ^ b, 5: 1 - (a ^ b), 6: a ^ b, 7: 1 - (a ^ b), 8: a}[g]


def _run_threads(fns):
    """run every fn in a thread of its own, all released at once; returns (results, exceptions) in fn order"""
    res, exc = [None] * len(fns), [None] * len(fns)
    start = threading.Barrier(len(fns))

    def body(i):
        start.wait()
        try:
            res[i] = fns[i]()
        except Exception as e:  # noqa: BLE001 -- reported per call
            exc[i] = e
    ts = [threading.Thread(target=body, args=(i,)) for i in range(len(fns))]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    return res, exc


def _wait_queued(ctx, n, timeout=120.0):
    """with the hold on, wait until n calls have joined the queue (bfhe_dbg_hold_batches returns the queue length)"""
    t0 = time.time()
    while ctx.dbg_hold_batches(True) < n:
        assert time.time() - t0 < timeout, "only %d of %d calls queued" % (ctx.dbg_hold_batches(True), n)
        time.sleep(0.01)


# ------------------------------------------------------------------------------------------------------------------------------
# CPU: bfhe_eval_not_host
# ------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("ps", ["TOY", "STD128_OPT"])
def test_eval_not_host_matches_oracle(bfhe, orc, ps):
    ctx = bfhe.Context(getattr(bfhe, ps), bfhe.GINX, device=-1)  # host-only, no keys
    o = orc.Oracle(getattr(orc, ps), orc.GINX)
    rng = np.random.default_rng(5)
    q, w, st = ctx.p.q, ctx.p.ct_words, ctx.stride
    rows = rng.integers(0, q, size=(40, st), dtype=np.uint32)
    rows[:, w:] = rng.integers(1, 1 << 32, size=(40, st - w), dtype=np.uint64).astype(np.uint32)  # padding garbage
    rows[0, :w] = 0
    rows[1, :w] = q - 1
    out = ctx.eval_not_host(rows)
    assert not out[:, w:].any(), "padding words must be written as zero"
    for i in range(rows.shape[0]):
        clean = rows[i].copy()
        clean[w:] = 0
        assert np.array_equal(out[i, :w], o.eval_not(clean)[:w]), i
    assert np.array_equal(out[:, :w - 1], (q - rows[:, :w - 1].astype(np.int64)) % q)
    assert np.array_equal(out[:, w - 1], (q // 4 + q - rows[:, w - 1].astype(np.int64)) % q)
    assert np.array_equal(ctx.EvalNOT(rows[3]), out[3])
    assert np.array_equal(ctx.eval_not_host(out)[:, :w], rows[:, :w])  # an involution on the ciphertext words


def test_eval_not_host_rejects(bfhe):
    ctx = bfhe.Context(bfhe.STD128_OPT, bfhe.GINX, device=-1)
    q, n = ctx.p.q, ctx.p.n
    rows = np.zeros((5, ctx.stride), dtype=np.uint32)
    rows[3, n] = q  # b out of range
    rows[4, 0] = 0xffffffff
    with pytest.raises(bfhe.BfheError) as e:
        ctx.eval_not_host(rows)
    assert e.value.code == bfhe.ERR_FORMAT and "row 3 " in str(e.value)
    rows[3, n] = 0
    rows[2, ctx.p.n + 1] = 0xffffffff  # padding is not checked
    with pytest.raises(bfhe.BfheError) as e:
        ctx.eval_not_host(rows)
    assert e.value.code == bfhe.ERR_FORMAT and "row 4 " in str(e.value)
    out = np.full_like(rows, 7)
    L = ctx.L
    assert L.bfhe_eval_not_host(ctx.h, rows.ctypes.data, 4, out.ctypes.data) == 0
    assert L.bfhe_eval_not_host(ctx.h, None, 1, out.ctypes.data) == bfhe.ERR_ARG
    assert L.bfhe_eval_not_host(ctx.h, rows.ctypes.data, 1, None) == bfhe.ERR_ARG
    assert L.bfhe_eval_not_host(None, rows.ctypes.data, 1, out.ctypes.data) == bfhe.ERR_ARG


def test_omp_example_compiles(bfhe, tmp_path):
    """examples/tb_omp_gates.cpp builds against host/binfhecontext.h with OpenMP"""
    here = os.path.dirname(bfhe.LIB_PATH)
    exe = tmp_path / "tb_omp_gates"
    r = subprocess.run(["g++", "-O2", "-std=c++17", "-fopenmp", "-Wall", "-o", str(exe), os.path.join(here, "examples", "tb_omp_gates.cpp"),
                        "-L" + here, "-lbfhe_b200", "-Wl,-rpath," + here], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-3000:]
    assert exe.exists()


# ------------------------------------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------------------------------------
def _calls(bfhe, ctx, cts, bits, rng):
    """N_THREADS calls of every kind: (fn, truth), truth being the expected decryptions of the rows fn returns"""
    B = bfhe
    ops = [B.OR, B.AND, B.NOR, B.NAND, B.XOR_FAST, B.XNOR_FAST, B.XOR, B.XNOR]
    k = len(cts)
    calls = []
    for t in range(N_THREADS):
        i, j = (int(x) for x in rng.choice(k, 2, replace=False))
        kind = t % 4
        if kind == 0:  # EvalBinGate, NEG flags on some
            op = ops[t % len(ops)] | (B.NEG0 if t & 4 else 0) | (B.NEG1 if t & 8 else 0)
            calls.append((lambda op=op, i=i, j=j: ctx.EvalBinGate(op, cts[i], cts[j])[None], [_truth(op, bits[i], bits[j])]))
        elif kind == 1:  # Bootstrap
            calls.append((lambda i=i: ctx.Bootstrap(cts[i])[None], [bits[i]]))
        else:  # multi-gate eval_bingate_host; thread 2 makes one call much larger than the rest
            m = 300 if t == 2 else int(rng.integers(2, 7))
            sel = rng.integers(0, k, size=(m, 2))
            sel[sel[:, 0] == sel[:, 1], 1] = (sel[sel[:, 0] == sel[:, 1], 1] + 1) % k
            g = np.zeros(m, dtype=B.GATE_DTYPE)
            g["op"] = [ops[x] | (B.NEG0 if x & 1 else 0) | (B.NEG1 if x & 2 else 0) for x in rng.integers(0, 8, size=m)]
            g["op"][::5] = B.BOOTSTRAP
            g["in0"], g["in1"], g["out"] = sel[:, 0], sel[:, 1], k + np.arange(m)
            truth = [_truth(int(op), bits[a], bits[b]) for op, a, b in zip(g["op"], sel[:, 0], sel[:, 1])]
            calls.append((lambda g=g: ctx.eval_bingate_host(g, cts, len(g)), truth))
    return calls


@pytest.mark.gpu
@pytest.mark.parametrize("ps,method", [("STD128_OPT", "GINX"), ("STD128_OPT", "AP"), ("TOY", "GINX")])
def test_concurrent_calls_exact(bfhe, orc, ps, method):
    B = bfhe
    ctx = shared_keys(B, getattr(B, ps), getattr(B, method), 0)
    rng = np.random.default_rng(11)
    bits = rng.integers(0, 2, size=24).tolist()
    cts = ctx.encrypt(bits, seed=21)
    calls = _calls(B, ctx, cts, bits, rng)
    serial = [fn() for fn, _ in calls]  # one at a time, one thread
    conc, exc = _run_threads([fn for fn, _ in calls])
    assert not any(exc), [e for e in exc if e]
    for t, (a, b) in enumerate(zip(serial, conc)):
        assert np.array_equal(a, b), "call %d differs from the same call made alone" % t
    for t, ((_, truth), out) in enumerate(zip(calls, conc)):
        assert ctx.decrypt(out).tolist() == truth, t
    # a sample against the oracle: the large call and two single-gate calls
    o = orc.Oracle(getattr(orc, ps), getattr(orc, method))
    o.import_keys(ctx.export_keys())
    w = ctx.p.ct_words
    big = calls[2][0].__defaults__[0][:40]  # its gates read input rows only, so any prefix is a call of its own
    slab = o.new_slab(len(cts) + len(big))
    slab[:len(cts)] = cts
    o.eval_gates(big, slab)
    assert np.array_equal(conc[2][:len(big), :w], slab[len(cts):, :w])
    for t in (0, 1):
        dflt = calls[t][0].__defaults__
        if t == 0:
            op, i, j = dflt
            ref = o.eval_bingate(op & 0xff, cts[i] if not op & B.NEG0 else o.eval_not(cts[i]),
                                 cts[j] if not op & B.NEG1 else o.eval_not(cts[j]))
        else:
            ref = o.bootstrap(cts[dflt[0]])
        assert np.array_equal(conc[t][0, :w], ref[:w]), t


def _boot_calls(ctx, cts):
    return [lambda i=i: ctx.Bootstrap(cts[i % len(cts)]) for i in range(N_THREADS)]


@pytest.mark.gpu
def test_held_batch_is_one_launch(bfhe):
    B = bfhe
    ctx = shared_keys(B, B.STD128_OPT, B.GINX, 0)
    bits = [int(x) for x in np.random.default_rng(3).integers(0, 2, size=N_THREADS)]
    cts = ctx.encrypt(bits, seed=31)
    alone = [fn() for fn in _boot_calls(ctx, cts)]
    ctx.profile_read(0), ctx.profile_read(1)
    ctx.profile_enable(True)
    try:
        assert ctx.dbg_hold_batches(True) == 0
        res = [None] * N_THREADS
        fns = _boot_calls(ctx, cts)

        def body(i):
            res[i] = fns[i]()
        ts = [threading.Thread(target=body, args=(i,)) for i in range(N_THREADS)]
        for t in ts:
            t.start()
        _wait_queued(ctx, N_THREADS)
        assert all(r is None for r in res)  # nothing launched while held
        assert ctx.dbg_hold_batches(False) == N_THREADS
        for t in ts:
            t.join()
        assert ctx.profile_read(0)[1] == 1, "64 held single-bootstrap calls must run as one blind-rotation launch"
        assert ctx.profile_read(1)[1] == 1
        for i in range(N_THREADS):
            assert np.array_equal(res[i], alone[i]), i
        assert ctx.decrypt(np.stack(res)).tolist() == bits
        # a lone caller without the hold: one launch per call
        for i in range(3):
            assert np.array_equal(ctx.Bootstrap(cts[i]), alone[i])
        assert ctx.profile_read(0)[1] == 3 and ctx.profile_read(1)[1] == 3
    finally:
        ctx.dbg_hold_batches(False)
        ctx.profile_enable(False)


@pytest.mark.gpu
def test_bad_calls_fail_alone(bfhe):
    """aliased, out-of-range and unknown-op calls fail in their own threads, with their own codes and messages, and never reach the
    held batch; every other call of that batch succeeds exactly"""
    B = bfhe
    ctx = shared_keys(B, B.STD128_OPT, B.GINX, 0)
    bits = [int(x) for x in np.random.default_rng(4).integers(0, 2, size=8)]
    cts = ctx.encrypt(bits, seed=41)
    good = [lambda i=i: ctx.EvalBinGate(B.NAND, cts[i % 8], cts[(i + 1) % 8]) for i in range(N_THREADS - 3)]
    alone = [fn() for fn in good]
    bad = [
        (lambda: ctx.eval_bingate_host(np.array([(B.AND, 1, 1, 2)], dtype=B.GATE_DTYPE), cts[:2], 1), B.ERR_ALIAS, "independent ciphertexts"),
        (lambda: ctx.eval_bingate_host(np.array([(B.OR, 0, 1, 9)], dtype=B.GATE_DTYPE), cts[:2], 1), B.ERR_ARG, "out of range"),
        (lambda: ctx.eval_bingate_host(np.array([(9, 0, 1, 2)], dtype=B.GATE_DTYPE), cts[:2], 1), B.ERR_ARG, "unknown gate type"),
    ]
    res, errs = [None] * N_THREADS, [None] * 3

    def run_good(i):
        res[i] = good[i]()

    def run_bad(k):
        try:
            bad[k][0]()
        except B.BfheError as e:
            errs[k] = (e.code, str(e), ctx.L.bfhe_last_error().decode())
    try:
        ctx.dbg_hold_batches(True)
        ts = [threading.Thread(target=run_good, args=(i,)) for i in range(len(good))]
        tb = [threading.Thread(target=run_bad, args=(k,)) for k in range(3)]
        for t in ts + tb:
            t.start()
        for t in tb:  # they fail while the batch is still held
            t.join(timeout=120)
            assert not t.is_alive()
        _wait_queued(ctx, len(good))
        assert ctx.dbg_hold_batches(False) == len(good)
        for t in ts:
            t.join()
    finally:
        ctx.dbg_hold_batches(False)
    for k, (_, code, text) in enumerate(bad):
        assert errs[k] is not None, "bad call %d did not fail" % k
        assert errs[k][0] == code and text in errs[k][1] and text in errs[k][2], errs[k]
    for i in range(len(good)):
        assert np.array_equal(res[i], alone[i]), i
        assert ctx.decrypt(res[i][None]).tolist() == [1 - (bits[i % 8] & bits[(i + 1) % 8])]


@pytest.mark.gpu
def test_clock_interleaves_with_combined_gates(bfhe):
    B = bfhe
    ctx = shared_keys(B, B.STD128_OPT, B.GINX, 0)
    circ = load_circuit(B, ctx, "adder_32bit")
    v = VECTORS["adder_32bit"]["vectors"][0]
    bits = [int(x) for x in np.random.default_rng(6).integers(0, 2, size=16)]
    cts = ctx.encrypt(bits, seed=51)
    fns = [lambda i=i: [ctx.EvalBinGate(B.AND, cts[(i + r) % 16], cts[(i + r + 3) % 16]) for r in range(4)] for i in range(32)]
    alone = [fn() for fn in fns]
    clock_out = []

    def clock():
        circ.Reset()
        circ.setEncrypted(True)
        circ.SetInput(v["inputs"], seed=5)
        clock_out.append(circ.Clock()[0])
        return True
    res, exc = _run_threads(fns + [clock])
    assert not any(exc), [e for e in exc if e]
    assert clock_out == [v["golden"]]
    for i in range(32):
        for r in range(4):
            assert np.array_equal(res[i][r], alone[i][r])
            assert int(ctx.decrypt(res[i][r][None])[0]) == bits[(i + r) % 16] & bits[(i + r + 3) % 16]


def _golden(name, inp):
    a = sum(b << i for i, b in enumerate(inp[:32]))
    b = sum(x << i for i, x in enumerate(inp[32:64]))
    if name == "adder_32bit":
        return [((a + b) >> i) & 1 for i in range(33)]
    s = lambda x: x - (1 << 32) if x >> 31 else x  # noqa: E731
    return [int(s(a) < s(b))]


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["adder_32bit", "comparator_32bit_signed_lt"])
def test_omp_example(bfhe, tmp_path, name):
    """examples/tb_omp_gates.cpp: the reference's per-gate OpenMP scheduler over the shim, 64 threads"""
    ctx = shared_keys(bfhe, bfhe.STD128_OPT, bfhe.GINX, 0)
    p = tmp_path / (name + ".out")
    load_circuit(bfhe, ctx, name).write_out(p)
    exe = os.path.join(os.path.dirname(bfhe.LIB_PATH), "examples", "tb_omp_gates")
    assert os.path.exists(exe), "run build() first"
    env = dict(os.environ, OMP_NUM_THREADS="64", OMP_WAIT_POLICY="passive")
    r = subprocess.run([exe, str(p), "-s", "STD128_OPT", "-m", "GINX", "-i", "9"], capture_output=True, text=True, timeout=900, env=env)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    kv = dict(re.findall(r"^(\w+) (\S+)$", r.stdout, flags=re.M))
    assert kv["ct_equal"] == "1" and kv["decrypt_equal"] == "1"
    inp = [int(ch) for ch in kv["inputs"]]
    assert [int(ch) for ch in kv["outputs"]] == _golden(name, inp)
    assert int(kv["br_launches"]) < int(kv["bootstraps"]), kv


@pytest.mark.gpu
def test_eval_not_matches_device(bfhe):
    ctx = shared_keys(bfhe, bfhe.STD128_OPT, bfhe.GINX, 0)
    cts = ctx.encrypt([1, 0, 1, 1, 0], seed=61)
    s = ctx.slab(10)
    s.upload(cts)
    ctx.eval_not_batch(s, list(range(5)), list(range(5, 10)))
    dev = s.download(5, 5)
    s.free()
    assert np.array_equal(np.stack([ctx.EvalNOT(c) for c in cts]), dev)
    assert np.array_equal(ctx.eval_not_host(cts), dev)
    assert ctx.decrypt(dev).tolist() == [0, 1, 0, 0, 1]
