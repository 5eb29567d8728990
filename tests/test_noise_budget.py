"""Noise budget: keys, accumulators and gate outputs decrypted with the secret keys and checked against the definition of the scheme.

The parity tests compare the GPU with the CPU oracle, which is given the product's own keys, and the circuit tests decrypt output bits.
Neither looks at the noise: keys without noise, a Gaussian of the wrong width, or an accumulator coefficient off by a large amount that
sample extraction never reads would pass both.  Everything here is computed from the definitions in plain numpy, without the oracle:

- keys (CPU): s and z are uniform ternary; every KSK row and every RGSW row of the BK decrypts to its documented message plus noise that
  follows the discrete Gaussian of hostmath.hpp::GaussTable (sigma = 3.19, tail cut at 12 sigma);
- accumulators (GPU, every kernel form): every coefficient of b - a*z equals the rotated test vector plus noise inside a hard bound, and
  the noise variance matches the blind-rotation variance derived below;
- gate outputs (GPU): every phase b - <a, s> lies within a hard bound of bit * q/4, with the mean and variance of the output budget, and
  every kernel form gives the same words.

Blind-rotation variance (sigma_BR^2), per gate.  An external product acc [] RGSW(mu) is sum_l d_l * row_l over the 2 dG rows, d_l the
signed base-B_g digits of acc's two components; its phase is mu * acc plus sum_l d_l * e_l, e_l the row noise.  Each output coefficient
sums every coefficient of every digit polynomial against an independent noise coefficient, so the added variance is
sigma^2 * sum_l sum_j d_l[j]^2.  While acc is uniform mod Q this is V_u = sigma^2 * N * 2 * sum_l E[d_l^2], with E[d_l^2] the exact
second moment of digit l over all residues mod Q (the top digit's range is narrower than B_g, so it is computed per digit row).  The
first step that changes acc starts from the trivial (0, TV): a-digits are zero and the b-digits are those of the test vector's +-Q8
entries, V_TV = sigma^2 * sum_j sum_l d_l(TV_j)^2, exactly per gate.
- GINX: acc += (X^m - 1)(acc [] RGSW(s_i = 1)) + (X^-m - 1)(acc [] RGSW(s_i = -1)), m = ((q - a_i) mod q) * 2N/q.  Multiplying a noise
  polynomial by X^m - 1 multiplies its coefficient variance by 2, by 4 for m = N (X^N - 1 = -2) and by 0 for m = 0; two products per
  step.  The old noise is carried (rotated), so sigma_BR^2 = sum_i 2 c(m_i) V_i.
- AP: acc <- acc [] RGSW(X^{s_i d B_r^k}) for every nonzero digit d of (q - a_i) mod q; zero digits are skipped, so sigma_BR^2 is V per
  applied step (V_TV for the first one).
- The signed-digit decomposition wraps for the residues whose top digit would be B_g/2 (TOY only: about 0.1 % of them, see
  test_oracle.py::test_signed_digit_decompose); the recomposition is then off by delta = -B_g^dG mod Q.  The product carries
  mu * (delta_b - delta_a * z), variance E[delta^2] (1 + |z|^2) per product with a message, times the same c(m) for GINX.  Every moment is
  computed exactly by enumerating all residues mod Q; the test vector's digits never wrap (asserted).

Output budget, per gate.  Sample extraction and ModSwitch Q -> qKS add the rounding error r_b - sum_k r_k z_k, KeySwitch subtracts
N * dKS key rows, one per (i, k), picked by digit k of the extracted mask a_i, and ModSwitch qKS -> q adds r_b - sum_i r_i s_i:
  V_out = (q/qKS)^2 [ (qKS/Q)^2 sigma_BR^2 + V_r(Q, qKS) (1 + |z|^2) + V_KS ] + V_r(qKS, q) (1 + |s|^2)
  mean  = 2 Q8 q/Q - q/4 (bit 1; 0 for bit 0) + (q/qKS) (m_r(Q, qKS) (1 - sum z) - m_KS) + m_r(qKS, q) (1 - sum s)
m_r and V_r are the exact mean and variance of the round-half-up error floor(v T / F + 1/2) - v T / F for v uniform mod F (1/32 and
43/512 - 1/1024 for 16 residues: half-up rounding is biased).  Over random keys m_KS = 0 and V_KS = N dKS sigma^2.  For the one key a
test uses, each row's noise is a fixed number, so m_KS and V_KS are the mean and spread of the selected rows' realized noise over the
digit distribution: at STD128_OPT m_KS / 16 varies by about 0.8 q-units from key to key, far more than the standard error of the mean
over 2^16 gates (0.04), so the budget uses the realized values.

Tolerances: fixed seeds make every check deterministic.  Means within 6 standard errors; variances within 6 standard errors of the
estimate, sqrt(2 / M) relative for M Gaussian samples (key noise: the exact fourth moment of the pmf); chi-square tests fail below
p = 1e-6.  Hard bounds: 8 sigma of the predicted noise (a Gaussian exceeds it with probability 1.2e-15 per sample); key noise: the
sampler's own cut, 12 sigma.

Run with -s to see the measured and predicted numbers (DESIGN.md section 2 records them)."""
import functools
import math
from fractions import Fraction

import numpy as np
import pytest
from scipy import stats

from conftest import shared_keys

SIGMA = 3.19
TAIL = int(math.ceil(12 * SIGMA))  # GaussTable's cut: |e| <= 39
HDR = 128  # sizeof(KeyBlobHeader)
P_MIN = 1e-6  # chi-square: a correct sampler fails with this probability per test
Z_SE = 6.0  # standard errors allowed for a mean or a variance
HARD = 8.0  # hard bound in predicted sigmas


def pad8(x):
    return (x + 7) & ~7


# ---- exact references -----------------------------------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def gauss_pmf():
    """support and pmf of GaussTable(3.19): P(x = k) proportional to exp(-k^2 / 2 sigma^2) for |k| <= ceil(12 sigma).  The table stores
    the CDF as floor(2^64 P) and draws a 64-bit uniform, which moves each probability by at most 2^-64: far below any test here."""
    k = np.arange(-TAIL, TAIL + 1)
    w = np.array([math.exp(-(int(v) * int(v)) / (2 * SIGMA * SIGMA)) for v in k])
    return k, w / w.sum()


def gauss_moments():
    k, p = gauss_pmf()
    return float((p * k**2).sum()), float((p * k**4).sum())


GAUSS_VAR = gauss_moments()[0]


def centre(x, m):
    """x mod m as a signed value in [-m/2, m/2)"""
    x = np.asarray(x, dtype=np.int64) % m
    return np.where(x >= (m + 1) // 2, x - m, x)


def negacyclic_matrix(z):
    """Z with (a @ Z)[k] = sum_j a_j z_{k-j} (sign -1 when k < j): the product a*z in Z[X]/(X^N + 1)"""
    N = z.size
    j, k = np.meshgrid(np.arange(N), np.arange(N), indexing="ij")
    return (z[(k - j) % N] * np.where(k >= j, 1, -1)).astype(np.float64)


def negacyclic_mul(a, z):
    """a*z for a batch of polynomials a (..., N), z ternary.  Every a_j < 2^27 and |z_j| <= 1, so every partial sum is an integer below
    N * 2^27 <= 2^37 < 2^53 and the float64 product is exact in any summation order."""
    a = np.asarray(a)
    assert a.size == 0 or (a.min() >= 0 and a.max() < 1 << 27)
    assert np.isin(z, (-1, 0, 1)).all() and z.size <= 1 << 10
    N = z.size
    r = a.reshape(-1, N).astype(np.float64) @ negacyclic_matrix(z)
    return np.rint(r).astype(np.int64).reshape(a.shape)


def monomial_mul(poly, e, N):
    """X^e * poly in Z[X]/(X^N + 1), e taken mod 2N; poly (..., N), e scalar or per leading row"""
    poly = np.asarray(poly, dtype=np.int64)
    ext = np.concatenate([poly, -poly], axis=-1)
    e = np.asarray(e, dtype=np.int64)
    idx = (np.arange(N) - e[..., None]) % (2 * N)
    return np.take_along_axis(ext, np.broadcast_to(idx, poly.shape), axis=-1)


def signed_digits(t, Q, log_b, dG):
    """OpenFHE's SignedDigitDecompose of residues t mod Q: centre (t < Q >> 1 stays positive), then dG signed remainders in
    [-B/2, B/2), each followed by an exact division.  Returns (digits (dG, ...), the part left above the top digit)."""
    B = 1 << log_b
    d = np.asarray(t, dtype=np.int64)
    d = np.where(d < Q >> 1, d, d - Q)
    out = []
    for _ in range(dG):
        r = ((d + B // 2) & (B - 1)) - B // 2
        out.append(r)
        d = (d - r) >> log_b
    return np.stack(out), d


def digit_moments_brute(Q, log_b, dG):
    """exact E[d_l^2] per digit row, E[delta^2] (delta = recomposition error, centred mod Q) and the wrap rate, over all Q residues"""
    dig, rest = signed_digits(np.arange(Q), Q, log_b, dG)
    delta = centre(-rest * (1 << (log_b * dG)), Q)
    return (dig.astype(np.float64) ** 2).mean(axis=1), float((delta.astype(np.float64) ** 2).mean()), float(np.mean(rest != 0))


@functools.lru_cache(maxsize=None)
def digit_moments(Q, log_b, dG):
    """digit_moments_brute without enumerating Q values: the centred residues are the integers of [(Q >> 1) - Q, (Q >> 1) - 1], each
    once; digit 0 splits d = B d_1 + r_0, so every d_1 strictly inside the range takes each r_0 of [-B/2, B/2) once, and only the two
    end rows are partial.  The remaining digits run on the values d_1 with those multiplicities."""
    B = 1 << log_b
    lo, hi = (Q >> 1) - Q, (Q >> 1) - 1
    d1 = np.arange((lo + B // 2) >> log_b, ((hi + B // 2) >> log_b) + 1, dtype=np.int64)
    r = np.arange(-(B // 2), B // 2, dtype=np.int64)
    w = np.full(d1.size, B, dtype=np.int64)
    sq0 = float(d1.size - 2) * float((r**2).sum())
    for end in (0, d1.size - 1):
        d = d1[end] * B + r
        inside = (d >= lo) & (d <= hi)
        w[end] = int(inside.sum())
        sq0 += float((r[inside] ** 2).sum())
    assert w.sum() == Q
    dig, rest = signed_digits(d1 % Q, Q, log_b, dG - 1)
    wf = w.astype(np.float64)
    sq = np.concatenate([[sq0], ((dig.astype(np.float64) ** 2) * wf).sum(axis=1)]) / Q
    delta = centre(-rest * (1 << (log_b * dG)), Q).astype(np.float64)
    return sq, float((delta**2 * wf).sum() / Q), float(wf[rest != 0].sum() / Q)


def round_moments(F, T):
    """exact mean and variance of r = floor(v T / F + 1/2) - v T / F for v uniform mod F (the (2vT + F) / (2F) rounding).  v T mod F is
    uniform over the multiples of g = gcd(T, F), so r = [2w >= F'] - w / F' for w uniform in [0, F'), F' = F / g."""
    Fp = F // math.gcd(T, F)
    h = (Fp + 1) // 2  # first w with 2w >= F'

    def s2(m):
        return m * (m + 1) * (2 * m + 1) // 6

    mean = Fraction(Fp - h, Fp) - Fraction(Fp - 1, 2 * Fp)
    e2 = Fraction(s2(h - 1) + s2(Fp - h), Fp ** 3)
    return float(mean), float(e2 - mean * mean)


# ---- key blob ---------------------------------------------------------------------------------------------------------------------------
def parse_keys(p, blob):
    """BFHEKEY1 (include/bfhe.h): s (n,), BK (rgsw, 2 dG rows, 2 columns, N), KSK (N, baseKS, dKS, n + 1)"""
    assert bytes(blob[:8]) == b"BFHEKEY1"
    o = HDR
    s = blob[o:o + 4 * p.n].view(np.int32).astype(np.int64)
    o += pad8(4 * p.n)
    per = 2 * p.dG * 2 * p.N
    n_rgsw = p.n * 2 if p.method == 1 else p.n * (p.baseR - 1) * p.dR
    bk = blob[o:o + 4 * n_rgsw * per].view(np.uint32).reshape(n_rgsw, 2 * p.dG, 2, p.N)
    o += pad8(4 * n_rgsw * per)
    dt = np.uint16 if p.qKS <= 1 << 16 else np.uint32
    cnt = p.N * p.baseKS * p.dKS * (p.n + 1)
    ksk = blob[o:o + np.dtype(dt).itemsize * cnt].view(dt).reshape(p.N, p.baseKS, p.dKS, p.n + 1)
    return s, bk, ksk


def ksk_weights(p):
    """digit weight j * baseKS^k mod qKS of every KSK row, (baseKS, dKS)"""
    j = np.arange(p.baseKS, dtype=np.int64)[:, None]
    k = np.array([pow(p.baseKS, kk, p.qKS) for kk in range(p.dKS)], dtype=np.int64)[None, :]
    return j * k % p.qKS


def ksk_phases(p, s, ksk):
    """b - <a, s> mod qKS for every KSK row, (N, baseKS, dKS); partial sums below n * qKS < 2^53: exact in float64"""
    rows = ksk.reshape(-1, p.n + 1)
    out = np.empty(rows.shape[0], dtype=np.int64)
    sf = s.astype(np.float64)
    for lo in range(0, rows.shape[0], 1 << 15):
        blk = rows[lo:lo + (1 << 15)]
        dot = np.rint(blk[:, :p.n].astype(np.float64) @ sf).astype(np.int64)
        out[lo:lo + blk.shape[0]] = (blk[:, p.n].astype(np.int64) - dot) % p.qKS
    return out.reshape(p.N, p.baseKS, p.dKS)


def recover_z(p, s, ksk):
    """z from the KSK: each KSK row is an encryption of z_i * j * baseKS^k under s.  The row whose weight w keeps 0, w and -w furthest
    apart mod qKS decides z_i (at TOY, qKS = Q and baseKS = 25, so it is a k = 5 row); then every row must agree with it: its phase minus
    z_i * w is inside the sampler's tail cut.  Returns (z, KSK noise (N, baseKS, dKS))."""
    w = ksk_weights(p)
    sep = np.minimum(np.abs(centre(w, p.qKS)), np.abs(centre(2 * w, p.qKS)))
    j, k = np.unravel_index(int(np.argmax(sep)), w.shape)
    assert sep[j, k] > 2 * TAIL
    ph = ksk_phases(p, s, ksk)
    cand = np.array([-1, 0, 1])
    dist = np.abs(centre(ph[:, j, k][:, None] - cand[None, :] * w[j, k], p.qKS))
    z = cand[np.argmin(dist, axis=1)]
    noise = centre(ph - z[:, None, None] * w[None], p.qKS)
    bad = np.argwhere(np.abs(noise) > TAIL)
    assert bad.size == 0, "KSK rows (i, j, k) disagree with the recovered z: %s" % bad[:5].tolist()
    return z, noise


def bk_messages(p, s, idx):
    """(mu, monomial exponent e in [0, 2N)) of the RGSWs idx: GINX RGSW(s_i == 1), RGSW(s_i == -1); AP X^{(s_i j B_r^k mod q) 2N/q}"""
    idx = np.asarray(idx, dtype=np.int64)
    if p.method == 1:
        i, which = idx // 2, idx % 2
        mu = np.where(which == 0, s[i] == 1, s[i] == -1).astype(np.int64)
        return mu, np.zeros_like(idx)
    k = idx % p.dR
    j = (idx // p.dR) % (p.baseR - 1) + 1
    i = idx // (p.dR * (p.baseR - 1))
    m = s[i] * j * np.array([p.baseR ** kk for kk in range(p.dR)], dtype=np.int64)[k]
    return np.ones_like(idx), (m % p.q) * (2 * p.N // p.q)


def bk_noise(p, s, z, bk, idx):
    """decrypt rows of the RGSWs idx with z.  Row 2l carries -mu g^l X^e z (message in the mask, or in the body of compact keys), row
    2l + 1 carries mu g^l X^e (in the body).  Returns the noise, (len(idx), 2 dG, N)."""
    N, Q = p.N, int(p.Q)
    mu, e = bk_messages(p, s, idx)
    rows = bk[idx].astype(np.int64)  # (R, 2dG, 2, N)
    phase = (rows[:, :, 1] - negacyclic_mul(rows[:, :, 0], z)) % Q
    unit = np.zeros((len(idx), N), dtype=np.int64)
    unit[:, 0] = 1
    xe = monomial_mul(unit, e, N) * mu[:, None]  # mu X^e
    xez = monomial_mul(np.broadcast_to(z, (len(idx), N)), e, N) * mu[:, None]  # mu X^e z
    msg = np.empty_like(phase)
    for l in range(p.dG):
        g = pow(p.baseG, l, Q)
        msg[:, 2 * l] = -g * xez
        msg[:, 2 * l + 1] = g * xe
    return centre(phase - msg, Q)


def assert_gaussian(noise, what):
    """noise ~ GaussTable(3.19): tail cut, chi-square of the histogram against the exact pmf, mean and variance within 6 standard errors
    (the variance's from the pmf's fourth moment: se = sqrt((m4 - var^2) / M))"""
    x = np.asarray(noise, dtype=np.int64).ravel()
    M = x.size
    var, m4 = gauss_moments()
    assert np.abs(x).max() <= TAIL, "%s: |noise| %d beyond the 12 sigma cut" % (what, np.abs(x).max())
    k, pmf = gauss_pmf()
    obs = np.bincount(x + TAIL, minlength=k.size).astype(np.float64)
    exp = M * pmf
    keep = exp >= 5  # the central bins; the rest pooled into one
    o = np.append(obs[keep], obs[~keep].sum())
    e = np.append(exp[keep], exp[~keep].sum())
    if e[-1] < 5:
        o, e = o[:-1], e[:-1]
        o[0] += obs[~keep].sum()  # negligible mass: fold it into the first bin rather than drop it
    chi = float(((o - e) ** 2 / e).sum())
    pv = stats.chi2.sf(chi, o.size - 1)
    mean, v = float(x.mean()), float((x.astype(np.float64) ** 2).mean())
    assert pv > P_MIN, "%s: histogram against the discrete Gaussian: chi2 %.1f, p %.2g" % (what, chi, pv)
    assert abs(mean) <= Z_SE * math.sqrt(var / M), "%s: mean %.4f" % (what, mean)
    assert abs(v - var) <= Z_SE * math.sqrt((m4 - var * var) / M), "%s: variance %.4f, exact %.4f" % (what, v, var)
    return v


def check_keys(p, blob, rgsw_idx=None):
    """every check of a key blob; rgsw_idx: the RGSWs to decrypt (all when None).  Returns a report for the pooled tests."""
    s, bk, ksk = parse_keys(p, blob)
    assert np.isin(s, (-1, 0, 1)).all()
    z, kn = recover_z(p, s, ksk)
    idx = np.arange(bk.shape[0]) if rgsw_idx is None else np.asarray(rgsw_idx)
    bn = np.concatenate([bk_noise(p, s, z, bk, idx[lo:lo + 256]).ravel() for lo in range(0, idx.size, 256)])
    v_k = assert_gaussian(kn, "KSK")
    assert np.abs(bn).max() <= TAIL, "BK: message missing or misplaced (|phase - message| up to %d)" % np.abs(bn).max()
    v_b = assert_gaussian(bn, "BK")
    return {"s": s, "z": z, "ksk_var": v_k, "bk_var": v_b, "ksk_m": kn.size, "bk_m": bn.size}


# ---- keys (CPU) -------------------------------------------------------------------------------------------------------------------------
KEY_SETS = [(ps, m, compact) for ps in ("TOY", "STD128_OPT") for m in ("GINX", "AP") for compact in (False, True)]
AP_STD_SAMPLE = 300  # RGSWs of the 31 124 in the 2.3 GB STD128_OPT AP key
_KEY_REPORTS = {}


def host_keys(bfhe, ps, m, compact):
    """the BFHEKEY1 blob of a host-only context, keys from btkeygen or btkeygen_compact with a seed per key set"""
    i = KEY_SETS.index((ps, m, compact))
    ctx = bfhe.Context(getattr(bfhe, ps), getattr(bfhe, m), -1)
    ctx.keygen(seed=900 + i)
    (ctx.btkeygen_compact if compact else ctx.btkeygen)(seed=950 + i)
    blob = ctx.export_keys(include_sk=True)
    p = ctx.p
    ctx.close()
    return p, blob


def key_report(bfhe, ps, m, compact):
    k = (ps, m, compact)
    if k not in _KEY_REPORTS:
        p, blob = host_keys(bfhe, ps, m, compact)
        sample = None
        if (ps, m) == ("STD128_OPT", "AP"):
            n_rgsw = p.n * (p.baseR - 1) * p.dR
            sample = np.sort(np.random.default_rng(4242).choice(n_rgsw, AP_STD_SAMPLE, replace=False))
        _KEY_REPORTS[k] = check_keys(p, blob, sample)
        del blob
    return _KEY_REPORTS[k]


@pytest.mark.parametrize("ps,m,compact", KEY_SETS)
def test_key_noise(bfhe, ps, m, compact):
    """KSK and BK of one key set: every row decrypts to its documented message, the noise follows the discrete Gaussian (histogram,
    mean, variance, tail cut).  Every RGSW is decrypted except for the STD128_OPT AP key, of which a fixed sample of 300 is."""
    r = key_report(bfhe, ps, m, compact)
    print("\n[keys] %s %s %s: KSK sigma %.4f (%d samples), BK sigma %.4f (%d samples), exact %.4f"
          % (ps, m, "compact" if compact else "full", math.sqrt(r["ksk_var"]), r["ksk_m"], math.sqrt(r["bk_var"]), r["bk_m"],
             math.sqrt(GAUSS_VAR)))


def test_secrets_are_uniform_ternary(bfhe):
    """s and z of all eight key sets (eight keygen seeds) pooled: the frequencies of -1, 0, 1 pass a chi-square test against 1/3 each"""
    for what in ("s", "z"):
        v = np.concatenate([key_report(bfhe, *k)[what] for k in KEY_SETS])
        assert np.isin(v, (-1, 0, 1)).all()
        obs = np.array([(v == c).sum() for c in (-1, 0, 1)])
        pv = stats.chisquare(obs).pvalue
        assert pv > P_MIN, "%s frequencies %s (p %.2g)" % (what, obs.tolist(), pv)


def test_negacyclic_product_helper():
    """the float64 product equals a Python-int schoolbook product"""
    rng = np.random.default_rng(5)
    N = 1024
    a = rng.integers(0, 1 << 27, size=N)
    a[:4] = (1 << 27) - 1
    z = rng.integers(-1, 2, size=N)
    ref = [0] * N
    al, zl = [int(x) for x in a], [int(x) for x in z]
    for i in range(N):
        for j in range(N):
            if i + j < N:
                ref[i + j] += al[i] * zl[j]
            else:
                ref[i + j - N] -= al[i] * zl[j]
    assert negacyclic_mul(a[None], z)[0].tolist() == ref
    with pytest.raises(AssertionError):
        negacyclic_mul(np.array([[1 << 27] + [0] * (N - 1)]), z)


def test_reference_moments():
    """the exact moments used by the budgets: rounding of 16 residues (STD128_OPT qKS -> q) and of Q residues (half-up is unbiased
    for odd F), and the digit wrap: none for STD128_OPT, about 0.1 % of residues for TOY"""
    assert round_moments(1 << 14, 1 << 10) == (1 / 32, 344 / 4096 - 1 / 1024)
    mean, var = round_moments(134215681, 1 << 14)
    assert mean == 0 and abs(var - 1 / 12) < 1e-12
    assert round_moments(134215681, 134215681) == (0.0, 0.0)
    for Q, log_b, dG in ((12289, 3, 5), (7681, 4, 3), (3329, 2, 6), (40961, 5, 3)):  # with and without wraps
        fast, brute = digit_moments(Q, log_b, dG), digit_moments_brute(Q, log_b, dG)
        assert np.allclose(fast[0], brute[0], rtol=1e-12) and math.isclose(fast[1], brute[1], rel_tol=1e-12)
        assert math.isclose(fast[2], brute[2], rel_tol=1e-12)
    _, _, wrap_std = digit_moments(134215681, 7, 4)
    _, _, wrap_toy = digit_moments(134215681, 9, 3)
    assert wrap_std == 0 and 0.0005 < wrap_toy < 0.003


# ---- gates: definitions -------------------------------------------------------------------------------------------------------------------
def ops12(bfhe):
    return [bfhe.OR, bfhe.AND, bfhe.NOR, bfhe.NAND, bfhe.XOR_FAST, bfhe.XNOR_FAST, bfhe.XOR, bfhe.XNOR, bfhe.BOOTSTRAP,
            bfhe.AND | bfhe.NEG0, bfhe.AND | bfhe.NEG1, bfhe.XOR | bfhe.NEG0]


def single_ops(bfhe):
    """the 12-op list with the composite XOR / XNOR, which the accumulator hook refuses, replaced by the single-bootstrap gates they
    consist of (OR(AND(a, !b), AND(!a, b))): AND | NEG1 and OR are already in the list, so they become XOR_FAST and XNOR_FAST with fused
    NOTs"""
    return [bfhe.OR, bfhe.AND, bfhe.NOR, bfhe.NAND, bfhe.XOR_FAST, bfhe.XNOR_FAST, bfhe.XOR_FAST | bfhe.NEG0,
            bfhe.XNOR_FAST | bfhe.NEG1, bfhe.BOOTSTRAP, bfhe.AND | bfhe.NEG0, bfhe.AND | bfhe.NEG1, bfhe.OR | bfhe.NEG0 | bfhe.NEG1]


def truth(bfhe, op, a, b):
    a = a ^ (1 if op & bfhe.NEG0 else 0)
    b = b ^ (1 if op & bfhe.NEG1 else 0)
    g = op & 0xff
    return {bfhe.OR: a | b, bfhe.AND: a & b, bfhe.NOR: 1 - (a | b), bfhe.NAND: 1 - (a & b), bfhe.XOR_FAST: a ^ b,
            bfhe.XNOR_FAST: 1 - (a ^ b), bfhe.XOR: a ^ b, bfhe.XNOR: 1 - (a ^ b), bfhe.BOOTSTRAP: a}[g]


def gate_const(bfhe, q, g):
    """RingGSWCryptoParams' gate constants; Bootstrap uses AND's"""
    return {bfhe.OR: 5 * q // 8, bfhe.AND: 7 * q // 8, bfhe.NOR: q // 8, bfhe.NAND: 3 * q // 8, bfhe.XOR_FAST: 5 * q // 8,
            bfhe.XNOR_FAST: q // 8, bfhe.BOOTSTRAP: 7 * q // 8}[g]


def eval_not(p, c):
    c = c.copy()
    c[:, :p.n] = (p.q - c[:, :p.n]) % p.q
    c[:, p.n] = (p.q // 4 + p.q - c[:, p.n]) % p.q
    return c


def prepare(bfhe, p, ops, c0, c1):
    """EvalBinGate's LWE step: the fused NOTs, then x + y, 2(x - y) for XOR_FAST / XNOR_FAST, and Bootstrap's (a, b + q/4); (G, n + 1)"""
    q, n = p.q, p.n
    c0 = np.asarray(c0, dtype=np.int64)[:, :n + 1]
    c1 = np.asarray(c1, dtype=np.int64)[:, :n + 1]
    neg0 = (ops & bfhe.NEG0) != 0
    neg1 = (ops & bfhe.NEG1) != 0
    x = np.where(neg0[:, None], eval_not(p, c0), c0)
    y = np.where(neg1[:, None], eval_not(p, c1), c1)
    g = ops & 0xff
    fast = (g == bfhe.XOR_FAST) | (g == bfhe.XNOR_FAST)
    out = np.where(fast[:, None], 2 * (x - y), x + y) % q
    boot = g == bfhe.BOOTSTRAP
    out[boot, :n] = x[boot, :n]
    out[boot, n] = (x[boot, n] + q // 4) % q
    return out


def expected_acc(bfhe, p, ops, prep, s):
    """the accumulator's message b - a*z without noise, (G, N), signed.  Test vector of blind_rotate_kernel's init: coefficient
    j * 2N/q (j < q/2) is -Q8 when (b - j - q1) mod q < q/2 and Q8 otherwise, Q8 = Q/8 + 1, q1 the gate constant; the blind rotation
    multiplies it by X^{(2N/q) sum_i ((q - a_i) mod q) s_i}.  Also returns the bit the test vector gives at coefficient 0."""
    N, q, Q = p.N, p.q, int(p.Q)
    f = 2 * N // q
    Q8 = Q // 8 + 1
    q1 = np.array([gate_const(bfhe, q, int(g)) for g in ops & 0xff], dtype=np.int64)
    j = np.arange(q // 2)
    t = (prep[:, p.n][:, None] - j[None, :]) % q
    zero = (t - q1[:, None]) % q < q // 2
    tv = np.zeros((len(ops), N), dtype=np.int64)
    tv[:, j * f] = np.where(zero, -Q8, Q8)
    aneg = (q - prep[:, :p.n]) % q
    rot = f * ((aneg * s[None, :]).sum(axis=1) % q)
    msg = monomial_mul(tv, rot, N)
    return msg, (msg[:, 0] > 0).astype(np.int64), tv


def br_variance(p, prep, s, z, tv):
    """sigma_BR^2 per gate (module docstring), from its prepared mask and test vector"""
    N, q, Q = p.N, p.q, int(p.Q)
    log_b = int(p.baseG).bit_length() - 1
    ed2, edelta2, _ = digit_moments(Q, log_b, p.dG)
    v_u = GAUSS_VAR * N * 2 * ed2.sum()
    w = edelta2 * (1 + float((z * z).sum()))
    dig, rest = signed_digits(tv % Q, Q, log_b, p.dG)
    assert not rest.any()  # the test vector's digits recompose exactly
    v_tv = GAUSS_VAR * (dig.astype(np.float64) ** 2).sum(axis=(0, 2))
    aneg = (q - prep[:, :p.n]) % q
    if p.method == 1:
        m = aneg * (2 * N // q) % (2 * N)
        c = np.where(m == 0, 0.0, np.where(m == N, 4.0, 2.0))
        applied = c > 0
        first = applied & (np.cumsum(applied, axis=1) == 1)
        var = np.where(first, 2 * c * v_tv[:, None], 2 * c * v_u + c * (s[None, :] != 0) * w)
    else:
        dg = np.stack([(aneg // p.baseR ** k) % p.baseR for k in range(p.dR)], axis=2).reshape(len(prep), -1)  # step i * dR + k
        applied = dg != 0
        first = applied & (np.cumsum(applied, axis=1) == 1)
        var = np.where(first, v_tv[:, None], np.where(applied, v_u + w, 0.0))
    return var.sum(axis=1)


def acc_errors(p, acc, msg, z):
    """b - a*z - message, centred mod Q, (G, N)"""
    Q = int(p.Q)
    acc = np.asarray(acc, dtype=np.int64)
    return centre(acc[:, 1] - negacyclic_mul(acc[:, 0], z) - msg, Q)


def check_accumulators(p, err, var_br, what):
    """every coefficient within 8 predicted sigmas; the sum of squares within 6 standard errors of its prediction
    (se^2 = sum_g N * 2 sigma_g^4 for independent Gaussian coefficients)"""
    N = p.N
    sig = np.sqrt(var_br)
    worst = np.abs(err) / sig[:, None]
    g, k = np.unravel_index(int(np.argmax(worst)), worst.shape)
    assert worst[g, k] <= HARD, "%s: gate %d coefficient %d off by %d = %.1f sigma_BR" % (what, g, k, err[g, k], worst[g, k])
    ss = float((err.astype(np.float64) ** 2).sum())
    pred = float(N * var_br.sum())
    se = math.sqrt(float(N * 2 * (var_br**2).sum()))
    ratio = ss / pred
    assert abs(ss - pred) <= Z_SE * se, "%s: sum of squared errors %.6g, predicted %.6g (ratio %.5f, 6 se = %.5f)" % (
        what, ss, pred, ratio, Z_SE * se / pred)
    return ratio, float(worst.max())


def gate_inputs(bfhe, ctx, count, n_in, seed):
    rng = np.random.default_rng(seed)
    bits = rng.integers(0, 2, size=n_in)
    cts = ctx.encrypt(bits, seed=seed)
    g = np.zeros(count, dtype=bfhe.GATE_DTYPE)
    a = rng.integers(0, n_in, size=count)
    b = (a + rng.integers(1, n_in, size=count)) % n_in  # never a == b (EvalBinGate refuses aliased operands)
    return bits, cts, g, a, b


# ---- the reference model holds for the oracle (CPU) --------------------------------------------------------------------------------------
def test_accumulator_model_on_oracle(bfhe, orc):
    """the accumulator checker and sigma_BR^2 on the CPU oracle's blind rotation, TOY GINX and AP, 120 gates of every single-bootstrap
    op: the reference model is the oracle's definition too, independently of the GPU"""
    for m in ("GINX", "AP"):
        ctx = bfhe.Context(bfhe.TOY, getattr(bfhe, m), -1)
        ctx.keygen(seed=31)
        ctx.btkeygen(seed=32)
        p = ctx.p
        blob = ctx.export_keys(include_sk=True)
        s, _, ksk = parse_keys(p, blob)
        z, _ = recover_z(p, s, ksk)
        o = orc.Oracle(orc.TOY, getattr(orc, m))
        o.import_keys(blob)
        ops_l = single_ops(bfhe)
        G = 120
        bits, cts, gates, a, b = gate_inputs(bfhe, ctx, G, 16, 77)
        ops = np.array([ops_l[i % len(ops_l)] for i in range(G)], dtype=np.int64)
        prep = prepare(bfhe, p, ops, cts[a], cts[b])
        acc = np.stack([o.blind_rotate(int(ops[i]) & 0xff, o.prep(int(ops[i]), cts[a[i]], cts[b[i]])).reshape(2, p.N)
                        for i in range(G)])
        assert np.array_equal(np.stack([o.prep(int(ops[i]), cts[a[i]], cts[b[i]])[:p.n + 1] for i in range(G)]), prep)
        msg, bit, tv = expected_acc(bfhe, p, ops, prep, s)
        assert bit.tolist() == [truth(bfhe, int(ops[i]), int(bits[a[i]]), int(bits[b[i]])) for i in range(G)]
        err = acc_errors(p, acc, msg, z)
        check_accumulators(p, err, br_variance(p, prep, s, z, tv), "oracle TOY " + m)
        ctx.close()


# ---- accumulators (GPU) ------------------------------------------------------------------------------------------------------------------
_GPU_KEYS = {}


def gpu_keys(bfhe, ps, m):
    """the shared device key set with s and z taken from its BFHEKEY1 export"""
    ctx = shared_keys(bfhe, getattr(bfhe, ps), getattr(bfhe, m), 0)
    if (ps, m) not in _GPU_KEYS:
        blob = ctx.export_keys(include_sk=True)
        s, _, ksk = parse_keys(ctx.p, blob)
        z, kn = recover_z(ctx.p, s, ksk)
        _GPU_KEYS[(ps, m)] = (s.copy(), z, ks_noise_moments(ctx.p, kn))
        del blob
    return (ctx,) + _GPU_KEYS[(ps, m)]


ACC_FORMS = ([("STD128_OPT", "GINX", g) for g in (1, 2, 4, 8, 32, 128)] + [("STD128_OPT", "AP", g) for g in (1, 2, 4, 8, 128)]
             + [(ps, m, g) for ps, m in (("TOY", "GINX"), ("TOY", "AP")) for g in (1, 2, 4, 8)])
ACC_GATES = 1024


def run_accumulators(bfhe, ps, m, gpc):
    ctx, s, z, _ = gpu_keys(bfhe, ps, m)
    p = ctx.p
    ops_l = single_ops(bfhe)
    n_in = 64
    bits, cts, gates, a, b = gate_inputs(bfhe, ctx, ACC_GATES, n_in, 1000 + gpc)
    ops = np.array([ops_l[i % len(ops_l)] for i in range(ACC_GATES)], dtype=np.int64)
    gates["op"], gates["in0"], gates["in1"], gates["out"] = ops, a, b, n_in + np.arange(ACC_GATES)
    slab = ctx.slab(n_in + ACC_GATES)
    slab.upload(cts)
    ctx.dbg_set_gates_per_cta(gpc)
    try:
        acc = ctx.dbg_blind_rotate(slab, gates)
    finally:
        ctx.dbg_set_gates_per_cta(0)
        slab.free()
    prep = prepare(bfhe, p, ops, cts[a], cts[b])
    msg, bit, tv = expected_acc(bfhe, p, ops, prep, s)
    assert bit.tolist() == [truth(bfhe, int(ops[i]), int(bits[a[i]]), int(bits[b[i]])) for i in range(ACC_GATES)]
    return p, acc, msg, br_variance(p, prep, s, z, tv), z


@pytest.mark.gpu
@pytest.mark.parametrize("ps,m,gpc", ACC_FORMS)
def test_accumulator_noise(bfhe, ps, m, gpc):
    """1 024 blind rotations of the single-bootstrap ops on fresh inputs, one kernel form: every coefficient of every accumulator is
    the rotated test vector plus noise within 8 sigma_BR, and the noise variance is sigma_BR^2"""
    p, acc, msg, var_br, z = run_accumulators(bfhe, ps, m, gpc)
    ratio, worst = check_accumulators(p, acc_errors(p, acc, msg, z), var_br, "%s %s form %d" % (ps, m, gpc))
    print("\n[acc] %s %s form %d: sigma_BR predicted %.1f, measured/predicted variance %.4f (6 se %.4f), largest |error| %.2f sigma_BR"
          % (ps, m, gpc, math.sqrt(var_br.mean()), ratio, Z_SE * math.sqrt(2 * (var_br**2).sum() / p.N) / var_br.sum(), worst))


# ---- gate outputs (GPU) ------------------------------------------------------------------------------------------------------------------
OUT_CONFIGS = [("STD128_OPT", "GINX", 1 << 16, (1, 2, 4, 8, 32, 128)), ("STD128_OPT", "AP", 1 << 14, (1, 2, 4, 8, 128)),
               ("TOY", "GINX", 1 << 14, (1, 2, 4, 8)), ("TOY", "AP", 1 << 14, (1, 2, 4, 8))]


def ks_digit_probs(p):
    """P(digit k of v = j) for v uniform mod qKS, (baseKS, dKS), by exact counting (uniform when qKS = baseKS^dKS)"""
    F, B = int(p.qKS), int(p.baseKS)
    P = np.empty((B, p.dKS))
    for k in range(p.dKS):
        bk, cyc = B**k, B ** (k + 1)
        rem = F % cyc
        P[:, k] = [(F // cyc) * bk + min(max(rem - j * bk, 0), bk) for j in range(B)]
    return P / F


def ks_noise_moments(p, ksk_noise):
    """mean and variance of the key switch's noise sum_{i,k} e[i, j_ik, k] for this key: each row's noise is a fixed value of the key,
    so the output sees its average over the digit j (not zero) and its spread around that average.  Over many keys these average to
    0 and N dKS sigma^2."""
    P = ks_digit_probs(p)[None]
    e = ksk_noise.astype(np.float64)
    mean = (P * e).sum(axis=1)
    return float(mean.sum()), float(((P * e**2).sum(axis=1) - mean**2).sum())


def output_budget(p, s, z, ks, var_br):
    """(mean for bit 0, mean for bit 1, variance) of the output phase error, per gate (module docstring); ks = ks_noise_moments"""
    q, Q, qKS = p.q, int(p.Q), int(p.qKS)
    m1, v1 = round_moments(Q, qKS)
    m2, v2 = round_moments(qKS, q)
    var = ((q / qKS) ** 2 * ((qKS / Q) ** 2 * var_br + v1 * (1 + float((z * z).sum())) + ks[1])
           + v2 * (1 + float((s * s).sum())))
    base = (q / qKS) * (m1 * (1 - float(z.sum())) - ks[0]) + m2 * (1 - float(s.sum()))
    return base, base + 2 * (Q // 8 + 1) * q / Q - q / 4, var


def output_errors(p, s, out, bit):
    """b - <a, s> - bit q/4, centred mod q"""
    out = np.asarray(out, dtype=np.int64)
    dot = np.rint(out[:, :p.n].astype(np.float64) @ s.astype(np.float64)).astype(np.int64)
    return centre(out[:, p.n] - dot - bit * (p.q // 4), p.q)


def check_outputs(p, err, mean, var, what):
    """no decryption failure; every |error - mean| within 8 predicted sigmas; mean and variance within 6 standard errors"""
    M = err.size
    assert np.abs(err).max() < p.q // 8, "%s: %d decryption failures" % (what, int((np.abs(err) >= p.q // 8).sum()))
    dev = err - mean
    sig = np.sqrt(var)
    worst = float((np.abs(dev) / sig).max())
    assert worst <= HARD, "%s: an output error of %.1f sigma" % (what, worst)
    pm, pv = float(dev.mean()), float((dev**2).mean())
    assert abs(pm) <= Z_SE * math.sqrt(var.mean() / M), "%s: mean error %.4f off the budget's mean" % (what, pm)
    se = math.sqrt(2 * (var**2).sum()) / M
    assert abs(pv - var.mean()) <= Z_SE * se, "%s: variance %.3f, predicted %.3f (6 se %.3f)" % (what, pv, var.mean(), Z_SE * se)
    return float(err.mean()), float(mean.mean()), pv, float(var.mean()), worst


@pytest.mark.gpu
@pytest.mark.parametrize("ps,m,count,forms", OUT_CONFIGS)
def test_output_noise_and_forms(bfhe, ps, m, count, forms):
    """the 12-op list on fresh inputs through eval_bingate_host with the cost model's choice: every output decrypts, every phase is
    within 8 sigma_out of bit q/4, mean and variance match the output budget.  The same batch forced through every kernel form gives
    the same words, all of them (race and determinism check at full batch size)."""
    ctx, s, z, ks = gpu_keys(bfhe, ps, m)
    p = ctx.p
    ops_l = ops12(bfhe)
    n_in = 4096
    bits, cts, gates, a, b = gate_inputs(bfhe, ctx, count, n_in, 2000 + count)
    ops = np.array([ops_l[i % len(ops_l)] for i in range(count)], dtype=np.int64)
    gates["op"], gates["in0"], gates["in1"], gates["out"] = ops, a, b, n_in + np.arange(count)
    out = ctx.eval_bingate_host(gates, cts, count)
    bit = np.array([truth(bfhe, int(ops[i]), int(bits[a[i]]), int(bits[b[i]])) for i in range(count)])
    # sigma_BR^2 of the last bootstrap: exact from the prepared input; the composite XOR / XNOR end in an OR of two bootstrapped
    # ciphertexts whose masks are uniform, so they take the mean over uniform masks (the mean of the single gates' OR rows is close
    # to it; both enter the output variance scaled by (q/Q)^2)
    g = ops & 0xff
    single = (g != bfhe.XOR) & (g != bfhe.XNOR)
    prep = prepare(bfhe, p, ops[single], cts[a[single]], cts[b[single]])
    _, _, tv = expected_acc(bfhe, p, ops[single], prep, s)
    var_br = np.empty(count)
    var_br[single] = br_variance(p, prep, s, z, tv)
    var_br[~single] = var_br[single & (g == bfhe.OR)].mean()
    m0, m1, var = output_budget(p, s, z, ks, var_br)
    mean = np.where(bit == 1, m1, m0)
    err = output_errors(p, s, out, bit)
    got_m, pred_m, got_v, pred_v, worst = check_outputs(p, err, mean, var, "%s %s" % (ps, m))
    z_fail = (p.q / 8) / math.sqrt(got_v)  # failure probability the measured sigma implies
    print("\n[out] %s %s, %d gates: mean %.3f (predicted %.3f), sigma_out %.3f (predicted %.3f), largest |error - mean| %.2f sigma "
          "(bound %.0f), q/8 = %.1f sigma_out -> failure probability per gate %.2g"
          % (ps, m, count, got_m, pred_m, math.sqrt(got_v), math.sqrt(pred_v), worst, HARD, z_fail, math.erfc(z_fail / math.sqrt(2))))
    for form in forms:
        ctx.dbg_set_gates_per_cta(form)
        try:
            o2 = ctx.eval_bingate_host(gates, cts, count)
        finally:
            ctx.dbg_set_gates_per_cta(0)
        diff = np.flatnonzero((o2[:, :p.ct_words] != out[:, :p.ct_words]).any(axis=1))
        assert diff.size == 0, "form %d: %d of %d gates differ from the cost model's launch, first %s" % (
            form, diff.size, count, diff[:8].tolist())


# ---- the checkers have teeth (CPU) -------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def toy_blob(bfhe):
    ctx = bfhe.Context(bfhe.TOY, bfhe.GINX, -1)
    ctx.keygen(seed=61)
    ctx.btkeygen(seed=62)
    p, blob = ctx.p, ctx.export_keys(include_sk=True)
    ctx.close()
    return p, blob


def test_checker_accepts_clean_toy_keys(toy_blob):
    p, blob = toy_blob
    check_keys(p, blob.copy())


def test_checker_catches_noiseless_bk(toy_blob):
    """BK bodies re-encrypted with zero noise: every row still decrypts to its message, the noise test fails"""
    p, blob = toy_blob
    blob = blob.copy()
    s, bk, ksk = parse_keys(p, blob)
    z, _ = recover_z(p, s, ksk)
    idx = np.arange(bk.shape[0])
    noise = bk_noise(p, s, z, bk, idx)
    bk[:, :, 1] = (bk[:, :, 1].astype(np.int64) - noise) % int(p.Q)
    assert not bk_noise(p, s, z, bk, idx).any()
    with pytest.raises(AssertionError, match="BK"):
        check_keys(p, blob)


def test_checker_catches_flipped_z(toy_blob):
    """every KSK row of one z_i re-encrypted for another value: the KSK alone is consistent, the BK no longer decrypts under it"""
    p, blob = toy_blob
    blob = blob.copy()
    s, bk, ksk = parse_keys(p, blob)
    z, _ = recover_z(p, s, ksk)
    i = 5
    dz = (1 if z[i] == 0 else -2 * int(z[i]))
    w = ksk_weights(p)
    ksk[i, :, :, p.n] = ((ksk[i, :, :, p.n].astype(np.int64) + dz * w) % p.qKS).astype(ksk.dtype)
    assert recover_z(p, s, ksk)[0][i] == z[i] + dz
    with pytest.raises(AssertionError, match="BK"):
        check_keys(p, blob)


def _toy_accumulators(bfhe, orc, toy_blob, G=48):
    """oracle accumulators of the toy key: a stand-in for a downloaded accumulator, host data only"""
    p, blob = toy_blob
    s, _, ksk = parse_keys(p, blob)
    z, _ = recover_z(p, s, ksk)
    ctx = bfhe.Context(bfhe.TOY, bfhe.GINX, -1)
    ctx.import_keys(blob)
    o = orc.Oracle(orc.TOY, orc.GINX)
    o.import_keys(blob)
    ops_l = single_ops(bfhe)
    bits, cts, _, a, b = gate_inputs(bfhe, ctx, G, 16, 5)
    ops = np.array([ops_l[i % len(ops_l)] for i in range(G)], dtype=np.int64)
    acc = np.stack([o.blind_rotate(int(ops[i]) & 0xff, o.prep(int(ops[i]), cts[a[i]], cts[b[i]])).reshape(2, p.N) for i in range(G)])
    prep = prepare(bfhe, p, ops, cts[a], cts[b])
    msg, _, tv = expected_acc(bfhe, p, ops, prep, s)
    ctx.close()
    return p, acc.astype(np.int64), msg, br_variance(p, prep, s, z, tv), z


def test_checker_catches_accumulator_changes(bfhe, orc, toy_blob):
    """a downloaded accumulator with one coefficient changed, and one rotated by a single position, must fail.  No oracle-free check
    can see a change of 1 in one coefficient -- it is a legitimate noise value -- so the smallest change tested is the one the hard
    bound resolves, one unit past 8 sigma_BR of that gate; bit-level agreement is what the oracle parity tests pin."""
    p, acc, msg, var_br, z = _toy_accumulators(bfhe, orc, toy_blob)
    err = acc_errors(p, acc, msg, z)
    check_accumulators(p, err, var_br, "clean")
    Q = int(p.Q)
    g, k = 7, 100
    bad = acc.copy()
    bad[g, 1, k] = (bad[g, 1, k] + int(HARD * math.sqrt(var_br[g])) - err[g, k] + 1) % Q
    with pytest.raises(AssertionError, match="coefficient"):
        check_accumulators(p, acc_errors(p, bad, msg, z), var_br, "changed")
    rot = acc.copy()
    rot[g] = monomial_mul(acc[g], 1, p.N) % Q  # X * acc: the message moves by one coefficient
    with pytest.raises(AssertionError, match="coefficient"):
        check_accumulators(p, acc_errors(p, rot, msg, z), var_br, "rotated")


def test_checker_catches_output_offset(bfhe, toy_blob):
    """fresh encryptions stand in for outputs with a known budget (variance sigma^2, mean 0); a constant 1 added to every phase must
    fail the mean test, and the clean set must pass"""
    p, blob = toy_blob
    s = parse_keys(p, blob)[0]
    ctx = bfhe.Context(bfhe.TOY, bfhe.GINX, -1)
    ctx.import_keys(blob)
    rng = np.random.default_rng(8)
    bit = rng.integers(0, 2, size=1 << 14)
    cts = ctx.encrypt(bit, seed=3)
    ctx.close()
    mean, var = np.zeros(bit.size), np.full(bit.size, GAUSS_VAR)
    check_outputs(p, output_errors(p, s, cts, bit), mean, var, "fresh")
    cts[:, p.n] = (cts[:, p.n] + 1) % p.q
    with pytest.raises(AssertionError, match="mean"):
        check_outputs(p, output_errors(p, s, cts, bit), mean, var, "offset")
