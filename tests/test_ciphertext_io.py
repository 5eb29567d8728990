"""Evaluation without the secret key: Circuit.set_input_ct / clock_ct (bfhe_circuit_set_input_ct / bfhe_circuit_clock_ct).

The "holder" is a context with every key (shared_keys); the "evaluator" is a context on the same device that imported
holder.export_keys(include_sk=False), so it can bootstrap but neither encrypt nor decrypt."""
import hashlib
import os
import subprocess

import numpy as np
import pytest

from conftest import shared_keys
from helpers import VECTORS, load_circuit, oracle_run_plan
from test_gpu_circuits import COUNTER, EXT_OUT

SHA256_IV = "6a09e667bb67ae853c6ef372a54ff53a510e527f9b05688c1f83d9ab5be0cd19"


def hex2bits(h):  # the fixtures' bit order (tests/golden/make_fixtures.py): last hex digit first, each nibble LSB first
    return [(int(ch, 16) >> b) & 1 for ch in reversed(h) for b in range(4)]


def sha256_blocks(msg):
    """FIPS 180-4 padding: the 512-bit blocks of msg as hex strings"""
    m = msg + b"\x80" + b"\x00" * ((55 - len(msg)) % 64) + (8 * len(msg)).to_bytes(8, "big")
    return [m[i:i + 64].hex() for i in range(0, len(m), 64)]


def ext_out_expected(a, b, d):  # the EXT_OUT netlist of test_gpu_circuits.py
    n3, n4 = 1 - (a & b), 1 - (b | d)
    r5 = 1 - (n3 ^ n4)
    r7 = 1 - ((r5 ^ a) ^ d)
    maj = int(a + b + d >= 2)
    return [n3, r5, r7, maj, 1 - maj, maj, 1 - maj, maj & r7]


_EVALUATORS = {}


def evaluator(bfhe, ps, m):
    """a context with the holder's evaluation keys and no secret key, one per (paramset, method)"""
    if (ps, m) not in _EVALUATORS:
        ctx = bfhe.Context(ps, m, 0)
        ctx.import_keys(shared_keys(bfhe, ps, m, 0).export_keys(include_sk=False))
        _EVALUATORS[(ps, m)] = ctx
    return _EVALUATORS[(ps, m)]


def _circuit(bfhe, ctx, name, tmp_path):
    if name == "ext_out":
        p = tmp_path / "ext.out"
        p.write_text(EXT_OUT)
        c = bfhe.Circuit(ctx)
        c.ReadFile(p)
    elif name == "counter":
        p = tmp_path / "counter.out"
        p.write_text(COUNTER)
        c = bfhe.Circuit(ctx)
        c.ReadFile(p)
    else:
        c = load_circuit(bfhe, ctx, name)
    c.Reset()
    c.setEncrypted(True)
    return c


def _code(excinfo):
    return excinfo.value.code


class _FakeDeviceArray:
    def __init__(self, shape, typestr="<u4", strides=None, ptr=0x7f0000000000):
        self.__cuda_array_interface__ = dict(shape=shape, typestr=typestr, strides=strides, data=(ptr, False), version=3)


# ---------------------------------------------------------------------------------------------------------------------
# CPU: argument and state checks come before the device check, so a host-only context answers them deterministically
# ---------------------------------------------------------------------------------------------------------------------
def test_cpu_modes_arguments_then_device(bfhe):
    ctx = bfhe.Context(bfhe.TOY, bfhe.GINX, -1)  # no keys at all: nothing here needs one
    c = load_circuit(bfhe, ctx, "adder_2bit")
    st = ctx.stride
    good = np.zeros((4, st), dtype=np.uint32)
    with pytest.raises(bfhe.BfheError) as e:  # encrypted mode off
        c.set_input_ct(good)
    assert _code(e) == bfhe.ERR_STATE
    c.setPlaintext(True)
    c.setEncrypted(True)
    with pytest.raises(bfhe.BfheError) as e:  # ciphertext inputs have no plaintext
        c.set_input_ct(good)
    assert _code(e) == bfhe.ERR_STATE
    c.Reset()
    c.setVerify(True)
    with pytest.raises(bfhe.BfheError) as e:
        c.set_input_ct(good)
    assert _code(e) == bfhe.ERR_STATE
    with pytest.raises(bfhe.BfheError) as e:
        c.clock_ct()
    assert _code(e) == bfhe.ERR_STATE
    c.Reset()
    c.setEncrypted(True)
    with pytest.raises(bfhe.BfheError) as e:  # adder_2bit has 2 + 2 input bits
        c.set_input_ct(np.zeros((3, st), dtype=np.uint32))
    assert _code(e) == bfhe.ERR_ARG
    with pytest.raises(bfhe.BfheError) as e:  # a good call needs the GPU: no CPU fallback
        c.set_input_ct(good)
    assert _code(e) == bfhe.ERR_CUDA
    with pytest.raises(bfhe.BfheError) as e:  # and leaves no input behind
        c.clock_ct()
    assert _code(e) == bfhe.ERR_STATE
    with pytest.raises(bfhe.BfheError) as e:
        c.set_input_ct(_FakeDeviceArray((3, st)))
    assert _code(e) == bfhe.ERR_ARG
    with pytest.raises(bfhe.BfheError) as e:
        c.set_input_ct(_FakeDeviceArray((4, st), typestr="<i4"))
    assert _code(e) == bfhe.ERR_CUDA


def test_cpu_python_buffer_checks(bfhe):
    ctx = bfhe.Context(bfhe.TOY, bfhe.GINX, -1)
    c = load_circuit(bfhe, ctx, "adder_2bit")
    c.setEncrypted(True)
    st = ctx.stride
    with pytest.raises(ValueError):
        c.set_input_ct(np.zeros((4, st + 1), dtype=np.uint32))
    with pytest.raises(TypeError):
        c.set_input_ct(np.zeros((4, st), dtype=np.int64))
    with pytest.raises(TypeError):
        c.set_input_ct([[0] * st] * 4)
    with pytest.raises(ValueError):
        c.set_input_ct(_FakeDeviceArray((4, st + 4)))
    with pytest.raises(TypeError):
        c.set_input_ct(_FakeDeviceArray((4, st), typestr="<f4"))
    with pytest.raises(TypeError):
        c.set_input_ct(_FakeDeviceArray((4, st), typestr="<u8"))
    with pytest.raises(ValueError):
        c.set_input_ct(_FakeDeviceArray((4, st), strides=(8 * st, 4)))
    with pytest.raises(ValueError):
        c.clock_ct(out=_FakeDeviceArray((3,)))


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", ["adder_2bit", "ext_out"])
@pytest.mark.parametrize("ps,m", [("STD128_OPT", "GINX"), ("TOY", "AP"), ("STD128_OPT", "AP")])
def test_bit_exact_against_both_references(bfhe, orc, tmp_path, ps, m, name):
    """Key-less set_input_ct + clock_ct equals the holder's SetInput(bits, seed) + clock_ct word for word, and every output row equals
    the oracle's slab row executing the evaluator's plan (through EvalNOT where the output reads its row negated)."""
    P, M = getattr(bfhe, ps), getattr(bfhe, m)
    holder, ev = shared_keys(bfhe, P, M, 0), evaluator(bfhe, P, M)
    if name == "adder_2bit":
        v = VECTORS["adder_2bit"]["vectors"][3]
        inputs, want = v["inputs"], v["golden"]
    else:
        inputs, want = [[1, 0, 1]], ext_out_expected(1, 0, 1)
    flat = np.concatenate([np.asarray(i, dtype=np.uint8) for i in inputs])
    seed = 61
    hc = _circuit(bfhe, holder, name, tmp_path)
    hc.SetInput(inputs, seed=seed)
    h_out = hc.clock_ct()
    ec = _circuit(bfhe, ev, name, tmp_path)
    fresh = holder.encrypt(flat, seed=seed)
    ec.set_input_ct(fresh)
    e_out = ec.clock_ct()
    w, st = ev.p.ct_words, ev.stride
    assert e_out.shape == (len(want), st)
    assert np.array_equal(e_out, h_out)
    assert not e_out[:, w:].any()
    assert holder.decrypt(e_out).tolist() == want
    o = orc.Oracle(getattr(orc, ps), getattr(orc, m))
    o.import_keys(holder.export_keys())
    _, ref = oracle_run_plan(ec, o, inputs, fresh=fresh)
    for b, r in enumerate(ec.plan_misc()["out_rows"]):
        row = ref[int(r) & 0x7fffffff]
        if int(r) >> 31:
            row = o.eval_not(row)
        assert np.array_equal(e_out[b, :w], row[:w]), b
    # the holder still decrypts with Clock() after a ciphertext SetInput
    hc.set_input_ct(fresh)
    assert hc.Clock()[0] == want


@pytest.mark.gpu
def test_keyless_evaluation_against_goldens(bfhe, tmp_path):
    P, M = bfhe.STD128_OPT, bfhe.GINX
    holder, ev = shared_keys(bfhe, P, M, 0), evaluator(bfhe, P, M)
    cases = [("adder_2bit", 0), ("adder_2bit", 1), ("comparator_32bit_signed_lt", 0), ("comparator_32bit_signed_lt", 1),
             ("mult_32x32", 0)]
    for t, (name, k) in enumerate(cases):
        v = VECTORS[name]["vectors"][k]
        c = _circuit(bfhe, ev, name, tmp_path)
        cts = holder.encrypt(np.concatenate(v["inputs"]), seed=200 + t)
        if t == 0:  # one input row through OpenFHE's JSON ciphertext format, imported by the evaluator
            p = str(tmp_path / "ct0.json")
            holder.export_openfhe_ct_json(cts[0], p)
            cts[0] = ev.import_openfhe_ct_json(p)
        c.set_input_ct(cts)
        assert holder.decrypt(c.clock_ct()).tolist() == v["golden"], (name, k)
    # without the secret key the outputs cannot be decrypted: Clock() refuses before launching anything
    v = VECTORS["adder_2bit"]["vectors"][2]
    c = _circuit(bfhe, ev, "adder_2bit", tmp_path)
    c.set_input_ct(holder.encrypt(np.concatenate(v["inputs"]), seed=9))
    with pytest.raises(bfhe.BfheError) as e:
        c.Clock()
    assert _code(e) == bfhe.ERR_STATE
    assert holder.decrypt(c.clock_ct()).tolist() == v["golden"]  # the input is still there
    with pytest.raises(bfhe.BfheError) as e:  # and SetInput on bits keeps needing the key
        c.SetInput(v["inputs"], seed=9)
    assert _code(e) == bfhe.ERR_STATE


@pytest.mark.gpu
def test_sha256_two_blocks_chained_on_device(bfhe, tmp_path):
    """The FIPS 448-bit message (two blocks) on the key-less evaluator: block 2's chaining value is block 1's clock_ct output,
    written into device memory and read from there by set_input_ct, never copied to the host."""
    P, M = bfhe.STD128_OPT, bfhe.GINX
    holder, ev = shared_keys(bfhe, P, M, 0), evaluator(bfhe, P, M)
    msg = b"abcdbcdecdefdefgefghfghighijhijkijkljklmklmnlmnomnopnopq"
    blocks = sha256_blocks(msg)
    assert len(blocks) == 2
    c = _circuit(bfhe, ev, "sha256", tmp_path)
    buf = ev.slab(512 + 256)  # input bus 1 (message block) | input bus 2 (chaining value)
    try:
        buf.upload(holder.encrypt(hex2bits(blocks[0]) + hex2bits(SHA256_IV), seed=301))
        c.set_input_ct(buf)
        c.clock_ct(out=buf.range(512, 256))
        buf.upload(holder.encrypt(hex2bits(blocks[1]), seed=302))
        c.set_input_ct(buf)
        digest = holder.decrypt(c.clock_ct()).tolist()
    finally:
        buf.free()
    assert digest == hex2bits(hashlib.sha256(msg).hexdigest())


@pytest.mark.gpu
def test_rejects_words_not_below_q(bfhe, tmp_path):
    import torch
    P, M = bfhe.TOY, bfhe.GINX
    holder, ev = shared_keys(bfhe, P, M, 0), evaluator(bfhe, P, M)
    n, q, st = ev.p.n, ev.p.q, ev.stride
    v = VECTORS["adder_2bit"]["vectors"][5]
    cts = holder.encrypt(np.concatenate(v["inputs"]), seed=17)
    bad = cts.copy()
    bad[3, n] = q               # b = q
    bad[1, 0] = 0xffffffff      # a_0 out of range: the lowest bad row is named
    c = _circuit(bfhe, ev, "adder_2bit", tmp_path)
    for src in ("host", "device"):
        arg = bad if src == "host" else torch.from_numpy(bad.view(np.int32)).cuda()
        torch.cuda.synchronize()
        with pytest.raises(bfhe.BfheError) as e:
            c.set_input_ct(arg)
        assert _code(e) == bfhe.ERR_FORMAT and "row 1 " in str(e.value), (src, str(e.value))
        with pytest.raises(bfhe.BfheError) as e:
            c.clock_ct()
        assert _code(e) == bfhe.ERR_STATE
        with pytest.raises(bfhe.BfheError) as e:
            c.Clock()
        assert _code(e) == bfhe.ERR_STATE
    one = cts.copy()
    one[2, n] = q
    with pytest.raises(bfhe.BfheError) as e:
        c.set_input_ct(one)
    assert _code(e) == bfhe.ERR_FORMAT and "row 2 " in str(e.value)
    # a following valid call works; padding words are ignored (and stored as zero)
    c.set_input_ct(cts)
    ref = c.clock_ct()
    assert holder.decrypt(ref).tolist() == v["golden"]
    noisy = cts.copy()
    noisy[:, n + 1:] = 0xdeadbeef
    dev = torch.from_numpy(noisy.view(np.int32)).cuda()
    out = torch.empty((ref.shape[0], st), dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()  # the evaluator reads on its own stream
    c.set_input_ct(dev)
    assert c.clock_ct(out=out) is out
    assert np.array_equal(out.cpu().numpy().view(np.uint32), ref)


@pytest.mark.gpu
@pytest.mark.parametrize("ps", ["TOY", "STD128_OPT"])
def test_dff_counter_keyless(bfhe, tmp_path, ps):
    """Flip-flops power up from the trivial encryption of 0 on the ciphertext path, also after a bit-path run left Encrypt(0) rows."""
    P, M = getattr(bfhe, ps), bfhe.GINX
    holder, ev = shared_keys(bfhe, P, M, 0), evaluator(bfhe, P, M)
    want = [[0, 0], [1, 0], [0, 1], [1, 1], [0, 0], [1, 0]]
    c = _circuit(bfhe, ev, "counter", tmp_path)
    c.set_input_ct(holder.encrypt([1], seed=5))
    assert [holder.decrypt(c.clock_ct()).tolist() for _ in range(6)] == want
    hc = _circuit(bfhe, holder, "counter", tmp_path)
    hc.SetInput([[1]], seed=5)
    assert hc.Clock()[0] == [0, 0] and hc.Clock()[0] == [1, 0]
    hc.Reset()
    hc.setEncrypted(True)
    hc.set_input_ct(holder.encrypt([1], seed=6))
    assert [holder.decrypt(hc.clock_ct()).tolist() for _ in range(6)] == want


@pytest.mark.gpu
def test_cpp_client_server(bfhe, tmp_path):
    """examples/tb_client_server.cpp: key holder and key-less evaluator through host/binfhecontext.h and host/circuit.h"""
    ctx = shared_keys(bfhe, bfhe.TOY, bfhe.GINX, 0)
    p = tmp_path / "adder_2bit.out"
    load_circuit(bfhe, ctx, "adder_2bit").write_out(p)
    exe = os.path.join(os.path.dirname(bfhe.LIB_PATH), "examples", "tb_client_server")
    assert os.path.exists(exe), "run build() first"
    r = subprocess.run([exe, str(p)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    assert "ALL PASSED" in r.stdout


def _sharded_worker(rank, world, port, q):
    import sys
    import torch
    import torch.distributed as dist
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, root)
    sys.path.insert(0, os.path.join(root, "tests"))
    import bfhe_loader
    from helpers import VECTORS, load_circuit
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world)
    B = bfhe_loader.load_package()
    ev = B.Context(B.STD128_OPT, B.GINX, rank)
    holder = None
    if rank == 0:  # the key holder lives on rank 0's host; the ranks receive the evaluation keys only
        holder = B.Context(B.STD128_OPT, B.GINX, -1)
        holder.keygen(41)
        holder.btkeygen(42)
        blob = torch.from_numpy(holder.export_keys(include_sk=False)).cuda()
        size = torch.tensor([blob.numel()], device="cuda")
    else:
        size = torch.tensor([0], device="cuda")
    dist.broadcast(size, 0)
    if rank != 0:
        blob = torch.empty(int(size), dtype=torch.uint8, device="cuda")
    dist.broadcast(blob, 0)
    ev.import_keys(blob.cpu().numpy())
    v = VECTORS["mult_32x32"]["vectors"][0]
    cts = holder.encrypt(np.concatenate(v["inputs"]), seed=43) if rank == 0 else None
    c = load_circuit(B, ev, "mult_32x32")
    uid = torch.from_numpy(B.nccl_unique_id() if rank == 0 else np.zeros(128, dtype=np.uint8)).cuda()
    dist.broadcast(uid, 0)
    c.set_sharding(rank, world, uid.cpu().numpy())
    c.Reset()
    c.setEncrypted(True)
    c.set_input_ct(cts)
    out = c.clock_ct()
    res = dict(digest=hashlib.sha256(out.tobytes()).hexdigest())
    if rank == 0:
        res["golden"] = holder.decrypt(out).tolist() == v["golden"]
        c1 = load_circuit(B, ev, "mult_32x32")  # unsharded on this GPU
        c1.Reset()
        c1.setEncrypted(True)
        c1.set_input_ct(cts)
        res["unsharded"] = hashlib.sha256(c1.clock_ct().tobytes()).hexdigest()
        c1.close()
        bad = cts.copy()
        bad[7, ev.p.n] = ev.p.q
    else:
        bad = None
    try:
        c.set_input_ct(bad)
        res["reject"] = 0
    except B.BfheError as e:
        res["reject"] = e.code
    c.set_input_ct(cts)  # still collective and usable afterwards
    res["again"] = hashlib.sha256(c.clock_ct().tobytes()).hexdigest()
    c.close()
    q.put((rank, res))
    dist.destroy_process_group()


@pytest.mark.gpu
def test_sharded_keyless_two_gpus():
    import torch
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two CUDA devices")
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_sharded_worker, args=(r, 2, 29640, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = dict(q.get(timeout=900) for _ in procs)
    for p in procs:
        p.join(timeout=60)
    r0, r1 = res[0], res[1]
    assert r0["golden"]
    assert r0["digest"] == r1["digest"] == r0["unsharded"] == r0["again"] == r1["again"]
    assert r0["reject"] == r1["reject"] == -4  # ERR_FORMAT on both ranks
