"""The STD128_OPT GINX throughput kernel reads its own copy of the bootstrapping key, with the top gadget digit folded into the other rows.
That copy is derived state: replacing the key on a context (a new btkeygen, or import_keys of another context's blob) must rebuild it,
or the throughput form would go on bootstrapping with the old key.  Every evaluation is compared bit for bit with an oracle built from
the key the context holds at that moment."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _gates(bfhe, n_in, count):
    rng = np.random.default_rng(5)
    ops = [bfhe.NAND, bfhe.AND | bfhe.NEG1, bfhe.XOR_FAST, bfhe.BOOTSTRAP, bfhe.OR | bfhe.NEG0, bfhe.XNOR]
    g = np.zeros(count, dtype=bfhe.GATE_DTYPE)
    for i in range(count):
        a, b = rng.choice(n_in, size=2, replace=False)
        g[i] = (ops[i % len(ops)], a, b, n_in + i)
    return g


def _check_throughput_form(bfhe, orc, ctx, enc_seed):
    """Evaluate on the four-gates-per-CTA form and compare with an oracle holding the context's current keys."""
    o = orc.Oracle(orc.STD128_OPT, orc.GINX)
    o.import_keys(ctx.export_keys())
    n_in, count = 8, 9  # two full CTAs and a ragged third
    bits = np.random.default_rng(enc_seed).integers(0, 2, size=n_in)
    cts = ctx.encrypt(bits, seed=enc_seed)
    gates = _gates(bfhe, n_in, count)
    ctx.dbg_set_gates_per_cta(4)
    try:
        out = ctx.eval_bingate_host(gates, cts, count)
    finally:
        ctx.dbg_set_gates_per_cta(0)
    ref = o.new_slab(n_in + count)
    ref[:n_in] = cts
    o.eval_gates(gates, ref)
    w = ctx.p.ct_words
    assert np.array_equal(out[:, :w], ref[n_in:, :w])
    return out[:, :w]


def test_folded_key_follows_key_replacement(bfhe, orc):
    ctx = bfhe.Context(bfhe.STD128_OPT, bfhe.GINX, 0)
    ctx.keygen(seed=31)
    ctx.btkeygen(seed=32)
    first = _check_throughput_form(bfhe, orc, ctx, enc_seed=41)

    ctx.btkeygen(seed=33)  # same secret key, new bootstrapping key
    second = _check_throughput_form(bfhe, orc, ctx, enc_seed=41)
    assert not np.array_equal(first, second)  # the same inputs really went through another key

    other = bfhe.Context(bfhe.STD128_OPT, bfhe.GINX, 0)
    other.keygen(seed=51)
    other.btkeygen(seed=52)
    ctx.import_keys(other.export_keys())
    _check_throughput_form(bfhe, orc, ctx, enc_seed=42)
