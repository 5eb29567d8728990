"""Compact fresh ciphertexts (include/bfhe.h "compact fresh ciphertexts"): encrypt_compact, the BFHECTS1 blob, expand_cts on the host
and on the device, and Circuit.set_input_compact on a key-less evaluator.

The masks are checked against the numpy ChaCha20 expansion of test_compact_keys (itself checked against RFC 8439), so the blob is
checked against the documented rule, not only against the library's own expander."""
import hashlib
import os
import subprocess

import numpy as np
import pytest

from conftest import shared_keys
from helpers import VECTORS, load_circuit
from test_ciphertext_io import _circuit, evaluator
from test_compact_keys import compact_keys, compact_sections, expand_rows

HDR = 64
SIGMA = 3.19


def pad8(x):
    return (x + 7) & ~7


def header(blob):
    """(magic, version, paramset, n, q, count, mask seed as 8 words)"""
    v = blob[8:24].view(np.uint32)
    return bytes(blob[:8]), int(v[0]), int(v[1]), int(v[2]), int(v[3]), int(blob[24:32].view(np.uint64)[0]), blob[32:64].view(np.uint32)


def bodies(blob, count):
    return blob[HDR:HDR + 2 * count].view(np.uint16)


_HOLDERS = {}


def holder(bfhe, ps):
    """a host-only context with a secret key and its sk as int64, one per parameter set"""
    if ps not in _HOLDERS:
        c = bfhe.Context(ps, bfhe.GINX, -1)
        c.keygen(71)
        c.btkeygen(72)
        sk = c.export_keys()[128:128 + 4 * c.p.n].view(np.int32).astype(np.int64)
        _HOLDERS[ps] = (c, sk)
    return _HOLDERS[ps]


class _DeviceView:
    def __init__(self, ptr, rows, stride):
        self.__cuda_array_interface__ = dict(shape=(rows, stride), typestr="<u4", strides=None, data=(ptr, False), version=3)


# ---------------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("ps", ["TOY", "STD128_OPT"])
def test_sizes(bfhe, ps):
    ctx = bfhe.Context(getattr(bfhe, ps), bfhe.GINX, -1)
    for count in (0, 1, 3, 4, 5, 256, 768, 1 << 20):
        assert ctx.ct_compact_size(count) == HDR + pad8(2 * count), count
    assert ctx.ct_compact_size(256) == 576


@pytest.mark.parametrize("ps", ["TOY", "STD128_OPT"])
def test_masks_bodies_and_decryption(bfhe, ps):
    ctx, _ = holder(bfhe, getattr(bfhe, ps))
    p = ctx.p
    rng = np.random.default_rng(3)
    for count in (0, 1, 37, 1000):
        bits = rng.integers(0, 256, size=count).astype(np.uint8)  # the message is bits % 4
        blob = ctx.encrypt_compact(bits, seed=5 + count)
        assert blob.dtype == np.uint8 and blob.size == HDR + pad8(2 * count)
        magic, ver, pset, n, q, cnt, seed = header(blob)
        assert (magic, ver, pset, n, q, cnt) == (b"BFHECTS1", 1, p.paramset, p.n, p.q, count)
        assert not blob[HDR + 2 * count:].any()
        rows = ctx.expand_cts(blob)
        assert rows.shape == (count, ctx.stride) and rows.dtype == np.uint32
        assert np.array_equal(rows[:, :p.n].astype(np.uint64), expand_rows(seed, np.arange(count, dtype=np.uint64), p.n, p.q))
        assert np.array_equal(rows[:, p.n], bodies(blob, count))
        assert not rows[:, p.n + 1:].any()
        assert ctx.decrypt(rows).tolist() == (bits % 4).tolist()
    # any context expands, without keys
    bare = bfhe.Context(getattr(bfhe, ps), bfhe.AP, -1)
    assert np.array_equal(bare.expand_cts(blob), rows)
    out = np.full((count + 2, ctx.stride), 7, dtype=np.uint32)
    assert bare.expand_cts(blob, out=out) is out
    assert np.array_equal(out[:count], rows) and (out[count:] == 7).all()


def test_noise_distribution(bfhe):
    ctx, sk = holder(bfhe, bfhe.TOY)
    p = ctx.p
    count = 100_000
    bits = np.random.default_rng(4).integers(0, 4, size=count).astype(np.uint8)
    rows = ctx.expand_cts(ctx.encrypt_compact(bits, seed=9)).astype(np.int64)
    phase = (rows[:, p.n] - rows[:, :p.n] @ sk - bits.astype(np.int64) * (p.q // 4)) % p.q
    e = np.where(phase >= p.q // 2, phase - p.q, phase)
    assert np.abs(e).max() <= 8 * SIGMA
    assert abs(e.std(ddof=1) - SIGMA) < 0.1 * SIGMA, e.std(ddof=1)
    assert abs(e.mean()) < 0.05


def test_mask_seeds(bfhe):
    gen, kblob = compact_keys(bfhe, bfhe.TOY, bfhe.GINX)  # keygen(21), btkeygen_compact(22)
    bits = [1, 0, 1, 1, 0]
    a, b = gen.encrypt_compact(bits, seed=22), gen.encrypt_compact(bits, seed=22)
    assert np.array_equal(a, b)
    c = gen.encrypt_compact(bits, seed=23)
    assert not np.array_equal(header(a)[6], header(c)[6])
    r0, r1 = gen.encrypt_compact(bits), gen.encrypt_compact(bits)
    assert not np.array_equal(header(r0)[6], header(r1)[6])
    assert gen.decrypt(gen.expand_cts(r0)).tolist() == bits
    key_seed = compact_sections(gen.p, kblob)[1]
    for blob in (a, c, r0, r1):
        assert not np.array_equal(header(blob)[6], key_seed)
    # the mask seed is not the only difference from bfhe_encrypt: the rows differ from Encrypt's under the same seed
    assert not np.array_equal(gen.expand_cts(a), gen.encrypt(bits, seed=22))


def _rejects(bfhe, ctx, blob, what):
    out = np.full((8, ctx.stride), 0xAB, dtype=np.uint32)
    with pytest.raises(bfhe.BfheError) as e:
        ctx.expand_cts(blob, out=out)
    assert e.value.code == bfhe.ERR_FORMAT and what in str(e.value), (what, str(e.value))
    assert (out == 0xAB).all()


def test_rejections(bfhe):
    ctx, _ = holder(bfhe, bfhe.STD128_OPT)
    blob = ctx.encrypt_compact([1, 0, 1, 1, 0], seed=3)  # 10 body bytes, 6 padding bytes
    assert blob.size == HDR + 16
    bad = blob.copy()
    bad[0] ^= 1
    _rejects(bfhe, ctx, bad, "magic")
    bad = blob.copy()
    bad[8] = 2
    _rejects(bfhe, ctx, bad, "version 2")
    toy, _ = holder(bfhe, bfhe.TOY)
    _rejects(bfhe, ctx, toy.encrypt_compact([1, 0, 1, 1, 0], seed=3), "do not match")
    for cut in (blob[:-1], blob[:-8], np.concatenate([blob, np.zeros(1, np.uint8)]), np.concatenate([blob, np.zeros(8, np.uint8)])):
        _rejects(bfhe, ctx, cut, "length")
    _rejects(bfhe, ctx, blob[:HDR - 1], "header")
    bad = blob.copy()
    bad[HDR + 2 * 3:HDR + 2 * 4].view(np.uint16)[0] = ctx.p.q
    _rejects(bfhe, ctx, bad, "body 3 = %d" % ctx.p.q)
    bad = blob.copy()
    bad[-1] = 1
    _rejects(bfhe, ctx, bad, "padding")
    with pytest.raises(bfhe.BfheError) as e:  # too few destination rows
        ctx.expand_cts(blob, out=np.zeros((4, ctx.stride), np.uint32))
    assert e.value.code == bfhe.ERR_ARG


def test_state_and_device_errors(bfhe):
    from test_ciphertext_io import _FakeDeviceArray
    bare = bfhe.Context(bfhe.TOY, bfhe.GINX, -1)
    with pytest.raises(bfhe.BfheError) as e:
        bare.encrypt_compact([1, 0])
    assert e.value.code == bfhe.ERR_STATE
    ctx, _ = holder(bfhe, bfhe.TOY)
    public = bfhe.Context(bfhe.TOY, bfhe.GINX, -1)
    public.import_keys(ctx.export_keys(include_sk=False))
    with pytest.raises(bfhe.BfheError) as e:
        public.encrypt_compact([1, 0])
    assert e.value.code == bfhe.ERR_STATE
    blob = ctx.encrypt_compact([1, 0, 1], seed=2)
    with pytest.raises(bfhe.BfheError) as e:
        bare.expand_cts(blob, out=_FakeDeviceArray((3, bare.stride)))
    assert e.value.code == bfhe.ERR_CUDA


def test_circuit_checks_before_the_device(bfhe):
    """On a host-only context: modes, then the count and the blob's checks, all before the device is needed."""
    ctx, _ = holder(bfhe, bfhe.TOY)
    c = load_circuit(bfhe, ctx, "adder_2bit")  # 2 + 2 input bits
    good = ctx.encrypt_compact([1, 0, 0, 1], seed=4)
    with pytest.raises(bfhe.BfheError) as e:  # encrypted mode off
        c.set_input_compact(good)
    assert e.value.code == bfhe.ERR_STATE
    c.setEncrypted(True)
    with pytest.raises(bfhe.BfheError) as e:
        c.set_input_compact(ctx.encrypt_compact([1, 0, 0], seed=4))
    assert e.value.code == bfhe.ERR_ARG
    bad = good.copy()
    bad[HDR:HDR + 2].view(np.uint16)[0] = ctx.p.q
    with pytest.raises(bfhe.BfheError) as e:
        c.set_input_compact(bad)
    assert e.value.code == bfhe.ERR_FORMAT and "body 0" in str(e.value)
    with pytest.raises(bfhe.BfheError) as e:
        c.set_input_compact(None)
    assert e.value.code == bfhe.ERR_ARG
    with pytest.raises(bfhe.BfheError) as e:  # a good blob needs the GPU
        c.set_input_compact(good)
    assert e.value.code == bfhe.ERR_CUDA


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("ps", ["TOY", "STD128_OPT"])
def test_device_expansion_equals_host(bfhe, ps):
    import torch
    h, _ = holder(bfhe, getattr(bfhe, ps))
    dev = bfhe.Context(getattr(bfhe, ps), bfhe.GINX, 0)  # no keys: expansion needs none
    st = dev.stride
    rng = np.random.default_rng(6)
    for count in (1, 3, 257, 100_003):
        blob = h.encrypt_compact(rng.integers(0, 2, size=count), seed=count)
        want = h.expand_cts(blob)
        slab = dev.slab(count + 1)
        try:
            canary = rng.integers(0, 1 << 32, size=(1, st), dtype=np.uint64).astype(np.uint32)
            slab.upload(canary, first_row=count)
            assert dev.expand_cts(blob, out=slab.range(0, count)) is not None
            got = slab.download()
        finally:
            slab.free()
        assert np.array_equal(got[:count], want), (ps, count)
        assert np.array_equal(got[count:], canary), (ps, count)
    t = torch.zeros((4 * st + 4,), dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()
    blob = h.encrypt_compact([1, 0, 1], seed=1)
    with pytest.raises(bfhe.BfheError) as e:
        dev.expand_cts(blob, out=_DeviceView(t.data_ptr() + 4, 3, st))
    assert e.value.code == bfhe.ERR_ARG and "aligned" in str(e.value)
    dev.expand_cts(blob, out=_DeviceView(t.data_ptr() + 16, 3, st))
    assert np.array_equal(t.cpu().numpy().view(np.uint32)[4:4 + 3 * st].reshape(3, st), h.expand_cts(blob))
    with pytest.raises(bfhe.BfheError) as e:  # host memory is not device memory
        dev.expand_cts(blob, out=_DeviceView(np.zeros((3, st), np.uint32).ctypes.data, 3, st))
    assert e.value.code == bfhe.ERR_ARG


@pytest.mark.gpu
@pytest.mark.parametrize("ps,m,name", [("TOY", "GINX", "adder_2bit"), ("TOY", "AP", "adder_2bit"),
                                       ("STD128_OPT", "GINX", "AES-non-expanded")])
def test_keyless_compact_equals_full_rows(bfhe, tmp_path, ps, m, name):
    """set_input_compact(blob) + clock_ct equals set_input_ct(expand_cts(blob)) + clock_ct word for word, on an evaluator without
    the secret key; the holder decrypts the known answer."""
    P, M = getattr(bfhe, ps), getattr(bfhe, m)
    hold, ev = shared_keys(bfhe, P, M, 0), evaluator(bfhe, P, M)
    v = VECTORS[name]["vectors"][1 if name == "adder_2bit" else 0]
    blob = hold.encrypt_compact(np.concatenate(v["inputs"]), seed=81)
    c = _circuit(bfhe, ev, name, tmp_path)
    c.set_input_compact(blob)
    out_c = c.clock_ct()
    c.Reset()
    c.setEncrypted(True)
    c.set_input_ct(ev.expand_cts(blob))
    out_f = c.clock_ct()
    assert np.array_equal(out_c, out_f)
    assert hold.decrypt(out_c).tolist() == v["golden"]
    c.close()


@pytest.mark.gpu
def test_dff_counter_from_compact_input(bfhe, tmp_path):
    P, M = bfhe.TOY, bfhe.GINX
    hold, ev = shared_keys(bfhe, P, M, 0), evaluator(bfhe, P, M)
    c = _circuit(bfhe, ev, "counter", tmp_path)
    c.set_input_compact(hold.encrypt_compact([1], seed=5))
    assert [hold.decrypt(c.clock_ct()).tolist() for _ in range(6)] == [[0, 0], [1, 0], [0, 1], [1, 1], [0, 0], [1, 0]]


@pytest.mark.gpu
def test_bad_blob_leaves_no_input(bfhe, tmp_path):
    P, M = bfhe.TOY, bfhe.GINX
    hold, ev = shared_keys(bfhe, P, M, 0), evaluator(bfhe, P, M)
    v = VECTORS["adder_2bit"]["vectors"][2]
    blob = hold.encrypt_compact(np.concatenate(v["inputs"]), seed=12)
    c = _circuit(bfhe, ev, "adder_2bit", tmp_path)
    c.set_input_compact(blob)
    assert hold.decrypt(c.clock_ct()).tolist() == v["golden"]
    c.Reset()
    c.setEncrypted(True)
    c.set_input_compact(blob)
    bad = blob.copy()
    bad[HDR + 2:HDR + 4].view(np.uint16)[0] = 0xffff
    with pytest.raises(bfhe.BfheError) as e:
        c.set_input_compact(bad)
    assert e.value.code == bfhe.ERR_FORMAT and "body 1" in str(e.value)
    with pytest.raises(bfhe.BfheError) as e:
        c.clock_ct()
    assert e.value.code == bfhe.ERR_STATE
    with pytest.raises(bfhe.BfheError) as e:
        c.set_input_compact(hold.encrypt_compact([1, 0, 1], seed=12))
    assert e.value.code == bfhe.ERR_ARG
    c.set_input_compact(blob)
    assert hold.decrypt(c.clock_ct()).tolist() == v["golden"]
    c.close()


@pytest.mark.gpu
@pytest.mark.parametrize("ps,m", [("STD128_OPT", "GINX"), ("TOY", "AP")])
def test_cpp_client_server_compact(bfhe, tmp_path, ps, m):
    """examples/tb_client_server.cpp -c: one compact blob per test through EncryptCompact / SetInputCompact"""
    ctx = shared_keys(bfhe, bfhe.TOY, bfhe.GINX, 0)
    p = tmp_path / "adder_2bit.out"
    load_circuit(bfhe, ctx, "adder_2bit").write_out(p)
    exe = os.path.join(os.path.dirname(bfhe.LIB_PATH), "examples", "tb_client_server")
    assert os.path.exists(exe), "run build() first"
    r = subprocess.run([exe, str(p), "-s", ps, "-m", m, "-n", "2", "-c"], capture_output=True, text=True, timeout=900)
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
    hold = None
    if rank == 0:
        hold = B.Context(B.STD128_OPT, B.GINX, -1)
        hold.keygen(45)
        hold.btkeygen(46)
        blob = torch.from_numpy(hold.export_keys(include_sk=False)).cuda()
        size = torch.tensor([blob.numel()], device="cuda")
    else:
        size = torch.tensor([0], device="cuda")
    dist.broadcast(size, 0)
    if rank != 0:
        blob = torch.empty(int(size), dtype=torch.uint8, device="cuda")
    dist.broadcast(blob, 0)
    ev.import_keys(blob.cpu().numpy())
    v = VECTORS["mult_32x32"]["vectors"][0]
    cblob = hold.encrypt_compact(np.concatenate(v["inputs"]), seed=47) if rank == 0 else None
    c = load_circuit(B, ev, "mult_32x32")
    uid = torch.from_numpy(B.nccl_unique_id() if rank == 0 else np.zeros(128, dtype=np.uint8)).cuda()
    dist.broadcast(uid, 0)
    c.set_sharding(rank, world, uid.cpu().numpy())
    c.Reset()
    c.setEncrypted(True)
    c.set_input_compact(cblob)
    out = c.clock_ct()
    res = dict(digest=hashlib.sha256(out.tobytes()).hexdigest())
    if rank == 0:
        res["golden"] = hold.decrypt(out).tolist() == v["golden"]
        c1 = load_circuit(B, ev, "mult_32x32")  # unsharded, from the full rows
        c1.Reset()
        c1.setEncrypted(True)
        c1.set_input_ct(ev.expand_cts(cblob))
        res["unsharded"] = hashlib.sha256(c1.clock_ct().tobytes()).hexdigest()
        c1.close()
    for name in ("format", "count"):
        bad = None
        if rank == 0 and name == "format":
            bad = cblob.copy()
            bad[HDR + 14] = 0xff
        elif rank == 0:
            bad = hold.encrypt_compact([1, 0, 1], seed=48)
        try:
            c.set_input_compact(bad)
            res[name] = 0
        except B.BfheError as e:
            res[name] = e.code
        try:
            c.clock_ct()
            res[name + "_clock"] = 0
        except B.BfheError as e:
            res[name + "_clock"] = e.code
    c.set_input_compact(cblob)  # still collective and usable afterwards
    res["again"] = hashlib.sha256(c.clock_ct().tobytes()).hexdigest()
    c.close()
    q.put((rank, res))
    dist.destroy_process_group()


@pytest.mark.gpu
def test_sharded_compact_two_gpus():
    import torch
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two CUDA devices")
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_sharded_worker, args=(r, 2, 29650, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = dict(q.get(timeout=900) for _ in procs)
    for p in procs:
        p.join(timeout=60)
    r0, r1 = res[0], res[1]
    assert r0["golden"]
    assert r0["digest"] == r1["digest"] == r0["unsharded"] == r0["again"] == r1["again"]
    assert r0["format"] == r1["format"] == -4  # ERR_FORMAT on both ranks
    assert r0["count"] == r1["count"] == -1    # ERR_ARG on both ranks
    assert r0["format_clock"] == r1["format_clock"] == r0["count_clock"] == r1["count_clock"] == -2
