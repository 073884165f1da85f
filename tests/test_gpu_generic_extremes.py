"""The generic ring kernels (ring_generic.cu: every degree 32..1024 and every NTT-friendly prime q < 2^31) at the edges of
their arithmetic, against an exact numpy reference.

Random data sits far from the limits the one-polynomial-per-warp kernels rely on: Shoup products below 2q < 2^32, the
inverse butterfly's u + q - v, the offset pos_off (a multiple of q just above 2^31) that lifts signed coefficients, the
64-bit Barrett product.  Those limits matter only at the top of the 31-bit range, so every operation here runs at the
smallest, the largest 16-bit, the first 32-bit (65537) and the largest 31-bit modulus of each degree, with inputs at
+-q//2, at the limits of the element type and with NTT slots all at q - 1.  Batches larger than two trips of each
kernel's persistent grid (plus a ragged tail) are built by tiling a few reference-checked items in scrambled order, with
output buffers pre-filled with a sentinel, so an item a grid-stride loop skips or computes twice shows.

The reference splits operands into 16-bit limbs so that no sum can round or overflow: negacyclic products are direct
convolutions (np.convolve) on int64, whose terms stay below 2^47 and sums of at most 1024 terms below 2^57; NTT slots are
products with the evaluation matrix V[j, p] = psi^(j (2 bitrev(p) + 1)), both sides split, so terms stay below 2^32 and
sums below 2^43, exact in float64.  test_reference_matches_the_oracle checks both
against the Python-integer restatement of lattice_algebra and needs no GPU."""
import functools
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gpu = pytest.mark.gpu
GW = 4                      # warps (items in flight) per block of the generic kernels, ring_generic.cu


def _is_prime(n):
    """Deterministic Miller-Rabin (these bases decide every n < 3.4 * 10^14)."""
    if n < 2:
        return False
    for p in (2, 3, 5, 7, 11, 13, 17):
        if n % p == 0:
            return n == p
    e, s = n - 1, 0
    while e % 2 == 0:
        e, s = e // 2, s + 1
    for a in (2, 3, 5, 7, 11, 13, 17):
        x = pow(a, e, n)
        if x in (1, n - 1):
            continue
        for _ in range(s - 1):
            x = x * x % n
            if x == n - 1:
                break
        else:
            return False
    return True


def _moduli(d):
    """The smallest prime q = 1 mod 2d, the largest below 2^16 (d != 256: the shipped geometry has its own kernels),
    65537 (the first modulus with 32-bit elements) and the largest below 2^31."""
    m = 2 * d
    smallest = next(q for q in range(m + 1, 1 << 31, m) if _is_prime(q))
    narrow_top = next(q for q in range((65535 // m) * m + 1, 0, -m) if _is_prime(q))
    top = next(q for q in range(((1 << 31) - 1) // m * m + 1, 0, -m) if _is_prime(q))
    return [smallest] + ([narrow_top] if d != 256 else []) + [65537, top]


DEGREES = (32, 64, 256, 512, 1024)
CASES = [(d, q) for d in DEGREES for q in _moduli(d)]
CASES_L = [(d, q, l) for d, q in CASES for l in (1, 3)] + [(d, q, 64) for d, q in CASES if d >= 512]
CASES_13 = [c for c in CASES_L if c[2] != 64]
ORACLE_CASES = [(32, 193), (64, 257), (32, 65537), (256, 2147483137)]


def _ids(case):
    return '-'.join(f'{k}{v}' for k, v in zip('dql', case))


def _bitrev(x, bits):
    return int(format(x, f'0{bits}b')[::-1], 2) if bits else 0


def _least_root(q, d):
    """The least element of order exactly 2d (the reference's rou): the minimum over the odd powers of any one of them."""
    h = 2
    while True:
        r = pow(h, (q - 1) // (2 * d), q)
        if pow(r, d, q) == q - 1:
            return min(pow(r, k, q) for k in range(1, 2 * d, 2))
        h += 1


def _matmul_mod(a, m, q):
    """(a @ m) mod q exactly for entries in [0, q), q < 2^31, inner dimension <= 2048: both operands split into 16-bit
    limbs, so every partial product is below 2^32 and every sum below 2^43 - exact in the float64 products."""
    a = np.asarray(a, dtype=np.int64)
    al, ah = (a & 0xFFFF).astype(np.float64), (a >> 16).astype(np.float64)
    ml, mh = (m & 0xFFFF).astype(np.float64), (m >> 16).astype(np.float64)
    part = lambda x, y: (x @ y).astype(np.int64) % q
    return (part(al, ml) + (part(al, mh) + part(ah, ml)) * 65536 % q + part(ah, mh) * (1 << 32) % q) % q


class Ref(object):
    """Exact statement of the ring operations of Z_q[X]/(X^d + 1) on numpy int64."""

    def __init__(self, d, q):
        self.d, self.q, self.half = d, q, q // 2
        self.psi = _least_root(q, d)
        pw = [1]
        for _ in range(2 * d - 1):
            pw.append(pw[-1] * self.psi % q)
        self.pw = np.array(pw, dtype=np.int64)                  # psi^e, e in [0, 2d)
        logd = d.bit_length() - 1
        self.odd = np.array([2 * _bitrev(p, logd) + 1 for p in range(d)], dtype=np.int64)
        j = np.arange(d, dtype=np.int64)
        self.V = self.pw[(j[:, None] * self.odd[None, :]) % (2 * d)]          # slot p = a(psi^odd[p])

    def centred(self, x):
        x = np.asarray(x, dtype=np.int64) % self.q
        return np.where(x > self.half, x - self.q, x)

    def slots(self, a):
        a = np.asarray(a, dtype=np.int64)
        return _matmul_mod(a.reshape(-1, self.d) % self.q, self.V, self.q).reshape(a.shape)

    def slots_of_pairs(self, pairs):
        """NTT slots of sparse polynomials given as (index, coefficient) pairs [..., wt, 2]."""
        pairs = np.asarray(pairs, dtype=np.int64)
        idx, co = pairs[..., 0] % self.d, pairs[..., 1] % self.q
        terms = self.pw[(idx[..., None] * self.odd) % (2 * self.d)] * co[..., None] % self.q
        return terms.sum(axis=-2) % self.q

    def repr2d(self, a):
        """lattice_algebra's ntt_representation: a(psi^k) for k in [0, 2d), centred."""
        j = np.arange(self.d, dtype=np.int64)
        w = self.pw[(j[:, None] * np.arange(2 * self.d)[None, :]) % (2 * self.d)]
        return self.centred(_matmul_mod(np.asarray(a, dtype=np.int64) % self.q, w, self.q))

    def mul(self, a, b):
        """Negacyclic product of two coefficient vectors, residues in [0, q)."""
        a, b = np.asarray(a, dtype=np.int64) % self.q, np.asarray(b, dtype=np.int64) % self.q
        full = (np.convolve(a, b & 0xFFFF) % self.q + (np.convolve(a, b >> 16) % self.q) * 65536) % self.q
        res = full[:self.d].copy()
        res[:self.d - 1] -= full[self.d:]
        return res % self.q

    def dot(self, u, v):
        """sum_i u[i] * v[i] over the vector index, residues."""
        acc = np.zeros(self.d, dtype=np.int64)
        for a, b in zip(u, v):
            acc = (acc + self.mul(a, b)) % self.q
        return acc


@functools.lru_cache(maxsize=6)
def _ref(d, q):
    return Ref(d, q)


def _dense(pairs, d):
    out = np.zeros(pairs.shape[:-2] + (d,), dtype=np.int64)
    flat, p = out.reshape(-1, d), np.asarray(pairs, dtype=np.int64).reshape(-1, pairs.shape[-2], 2)
    for i in range(p.shape[0]):
        flat[i, p[i, :, 0] % d] = p[i, :, 1]
    return out


def _limits(ct):
    info = np.iinfo(ct)
    return int(info.min), int(info.max)


def _patterns(rng, shape, m):
    """Arrays whose every entry has magnitude m: all +m, all -m, alternating, random signs."""
    alt = np.where(np.arange(shape[-1]) % 2 == 0, m, -m)
    return [np.full(shape, m, dtype=np.int64), np.full(shape, -m, dtype=np.int64),
            np.broadcast_to(alt, shape).astype(np.int64), rng.choice(np.array([-m, m], dtype=np.int64), shape)]


def _type_limits(rng, shape, ct):
    lo, hi = _limits(ct)
    alt = np.where(np.arange(shape[-1]) % 2 == 0, hi, lo)
    return [np.full(shape, hi, dtype=np.int64), np.full(shape, lo, dtype=np.int64),
            np.broadcast_to(alt, shape).astype(np.int64), rng.choice(np.array([lo, hi], dtype=np.int64), shape)]


def _need_gpu():
    import torch
    if not torch.cuda.is_available():
        pytest.skip('needs a CUDA device')


@pytest.fixture(scope='module')
def engines():
    """One context per (d, q, l) for the whole module (creating one builds its tables on the host)."""
    _need_gpu()
    from lattice_cryptography_b200 import Engine
    cache = {}

    def get(d, q, l):
        if (d, q, l) not in cache:
            cache[(d, q, l)] = Engine(128, q, d, l)
        return cache[(d, q, l)]
    yield get
    for e in cache.values():
        e.close()


def _np(x):
    """numpy copy of an engine output (torch device tensors included)."""
    if isinstance(x, np.ndarray):
        return x
    import torch
    via = {torch.uint16: (torch.int16, np.uint16), torch.uint32: (torch.int32, np.uint32)}.get(x.dtype)
    if via:
        return x.view(via[0]).cpu().numpy().view(via[1])
    return x.cpu().numpy()


class _Sentinel(object):
    """Engine outputs as device buffers pre-filled with 0xA5 bytes, so an element no kernel writes keeps a value that
    differs from the reference instead of whatever the memory pool held."""

    def __init__(self, eng):
        import torch
        self.eng, self.orig = eng, eng._out
        tdt = {np.int16: torch.int16, np.uint16: torch.uint16, np.uint8: torch.uint8, np.int32: torch.int32,
               np.uint32: torch.uint32, np.int64: torch.int64}

        def out(shape, dtype, device):
            t = torch.empty(shape, dtype=tdt[dtype], device=f'cuda:{eng.device}')
            t.view(-1).view(torch.uint8).fill_(0xA5)
            return t
        eng._out = out

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.eng._out = self.orig


# ------------------------------------------------------------------------------------------------ the reference itself
@pytest.mark.parametrize('d,q', ORACLE_CASES, ids=list(map(_ids, ORACLE_CASES)))
def test_reference_matches_the_oracle(d, q):
    """Products, slots and the 2d-point representation of the numpy reference against oracle/lattice_algebra (Python
    integers), at small degrees and at the top 31-bit prime; no GPU."""
    import lattice_algebra as ola
    ref = Ref(d, q)
    lp = ola.LatticeParameters(modulus=q, degree=d, length=1)
    assert ref.psi == lp.rou
    rng = np.random.default_rng(q)
    half = q // 2
    rows = _patterns(rng, (d,), half) + [rng.integers(-half, half + 1, d)]
    poly = lambda a: ola.Polynomial(lp, {i: int(v) for i, v in enumerate(a) if v}, False)
    for a, b in zip(rows, rows[1:] + rows[:1]):
        want = np.zeros(d, dtype=np.int64)
        for i, v in poly(a).__mul__(poly(b)).get_coef_rep()[0].items():
            want[i] = v
        assert np.array_equal(ref.centred(ref.mul(a, b)), want)
        rep = [int(x) for x in poly(a).ntt_representation]
        assert ref.repr2d(a[None])[0].tolist() == rep
        assert np.array_equal(ref.centred(ref.slots(a[None])[0]), np.array(rep)[ref.odd])
        # the slot transform is a ring map: the product's slots are the products of the slots
        assert np.array_equal(ref.slots(ref.mul(a, b)[None])[0], ref.slots(a[None])[0] * ref.slots(b[None])[0] % q)
    pairs = np.array([[[3, -half], [d - 1, half], [0, 1]]])
    assert np.array_equal(ref.slots_of_pairs(pairs), ref.slots(_dense(pairs, d)))


# ------------------------------------------------------------------------------------------------ transforms and products
@gpu
@pytest.mark.parametrize('d,q', CASES, ids=list(map(_ids, CASES)))
def test_transforms_and_products_at_extremes(engines, d, q):
    e, ref = engines(d, q, 1), _ref(d, q)
    assert e.root_of_unity == ref.psi
    rng = np.random.default_rng(d * 7 + q)
    half, ct = q // 2, e.ct
    a = np.stack(_patterns(rng, (d,), half) + _type_limits(rng, (d,), ct) + [rng.integers(-half, half + 1, d)])
    a_ct = np.ascontiguousarray(a.astype(ct))
    fa = e.ntt_fwd(a_ct).astype(np.int64)
    assert np.array_equal(fa, ref.slots(a)), 'ntt_fwd'
    assert np.array_equal(e.ntt_reference_repr(a_ct).astype(np.int64), ref.repr2d(a)), 'ntt_reference_repr'
    # every pair of rows
    i, j = np.meshgrid(np.arange(len(a)), np.arange(len(a)), indexing='ij')
    i, j = i.ravel(), j.ravel()
    got = e.poly_mul(np.ascontiguousarray(a_ct[i]), np.ascontiguousarray(a_ct[j])).astype(np.int64)
    for k in range(len(i)):
        assert np.array_equal(got[k], ref.centred(ref.mul(a[i[k]], a[j[k]]))), ('poly_mul', i[k], j[k])
    add = e.vec_add(np.ascontiguousarray(a_ct[i]), np.ascontiguousarray(a_ct[j])).astype(np.int64)
    sub = e.vec_sub(np.ascontiguousarray(a_ct[i]), np.ascontiguousarray(a_ct[j])).astype(np.int64)
    assert np.array_equal(add, ref.centred(a[i] + a[j])), 'vec_add'
    assert np.array_equal(sub, ref.centred(a[i] - a[j])), 'vec_sub'
    # NTT-form inputs: all q - 1, alternating 0 / q - 1, random choices of the two, uniform
    s = np.stack([np.full(d, q - 1), np.where(np.arange(d) % 2 == 0, q - 1, 0), rng.choice(np.array([0, q - 1]), d),
                  rng.integers(0, q, d)]).astype(np.int64)
    c = e.ntt_inv(np.ascontiguousarray(s.astype(e.nt))).astype(np.int64)
    assert np.abs(c).max() <= half, 'ntt_inv output not centred'
    assert np.array_equal(ref.slots(c), s), 'ntt_inv'


# ------------------------------------------------------------------------------------------------ keygen, sign, verify
@gpu
@pytest.mark.parametrize('d,q,l', CASES_L, ids=list(map(_ids, CASES_L)))
def test_keygen_product_at_extreme_public_row(engines, d, q, l):
    """vk = key_ch * sk with key_ch at +-q//2 and signing keys sampled with sk_bd = q//2 at full weight."""
    from lattice_cryptography_b200 import make_scheme
    e, ref = engines(d, q, l), _ref(d, q)
    rng = np.random.default_rng(11 * l + q + d)
    half = q // 2
    sch = make_scheme(sk_bd=half, sk_wt=d, ch_bd=1, ch_wt=1)
    nseed = 2 if l == 64 else 3
    for kp, key_ch in enumerate(_patterns(rng, (l, d), half)[::(2 if l == 64 else 1)]):
        e.set_key_ch(np.ascontiguousarray(key_ch.astype(e.ct)))
        seeds = [''.join(rng.choice(['0', '1'], 128)) for _ in range(nseed)]
        sk_coef, sk_ntt, vk_ntt, vk_coef = (x.astype(np.int64) for x in e.lm_keygen(sch, seeds))
        assert np.abs(sk_coef).max() <= half and np.count_nonzero(sk_coef) == sk_coef.size
        for i in range(nseed):
            for side in (0, 1):
                assert np.array_equal(vk_coef[i, side], ref.centred(ref.dot(key_ch, sk_coef[i, side]))), (kp, i, side)
        assert np.array_equal(vk_ntt, ref.slots(vk_coef)), kp
        assert np.array_equal(sk_ntt, ref.slots(sk_coef)), kp


@gpu
@pytest.mark.parametrize('d,q,l', CASES_13, ids=list(map(_ids, CASES_13)))
def test_sign_at_extreme_key_slots(engines, d, q, l):
    """sig = sk_left * c + sk_right with the key slots all at q - 1 (and mixed, and uniform), challenges of full weight
    with coefficients +-1 and up to +-q//2."""
    from lattice_cryptography_b200 import make_scheme
    e, ref = engines(d, q, l), _ref(d, q)
    rng = np.random.default_rng(7 * l + q + d)
    sk = np.stack([np.full((2, l, d), q - 1), rng.choice(np.array([0, q - 1]), (2, l, d)),
                   rng.integers(0, q, (2, l, d))]).astype(np.int64)
    n = len(sk)
    for ch_bd in (1, q // 2):
        sch = make_scheme(sk_bd=1, sk_wt=d, ch_bd=ch_bd, ch_wt=d)
        msgs = [bytes(rng.integers(0, 256, 40 + i, dtype=np.uint8)) for i in range(n)]
        pairs = e.challenge(sch, msgs)
        sig = e.lm_sign(sch, np.ascontiguousarray(sk.astype(e.nt)), msgs).astype(np.int64)
        assert np.abs(sig).max() <= q // 2
        cs = ref.slots(_dense(pairs, d))
        want = (cs[:, None, :] * sk[:, 0] + sk[:, 1]) % q
        assert np.array_equal(ref.slots(sig), want), ch_bd


def _verify_case(e, ref, rng, key_ch, sig, sch, msgs):
    """NTT-form keys for which key_ch * sig == vk_left * c + vk_right holds: vk_left slots all q - 1 for item 0, uniform
    for the others, vk_right solved from the equation."""
    q, d, n = ref.q, ref.d, len(sig)
    pairs = _np(e.challenge(sch, msgs))
    vkl = rng.integers(0, q, (n, d)).astype(np.int64)
    vkl[0] = q - 1
    lhs = (ref.slots(key_ch)[None] * ref.slots(sig) % q).sum(axis=1) % q
    vkr = (lhs - vkl * ref.slots(_dense(pairs, d))) % q
    return np.ascontiguousarray(np.stack([vkl, vkr], axis=1).astype(e.nt))


@gpu
@pytest.mark.parametrize('d,q,l', CASES_13, ids=list(map(_ids, CASES_13)))
def test_verify_holds_at_extreme_magnitudes(engines, d, q, l):
    """The equation holds for every item, so the verdict is 1 only if every residue is right; one tampered key slot or
    signature coefficient, a bound one below the largest magnitude or a weight one below the largest weight flips it."""
    from lattice_cryptography_b200 import make_scheme
    e, ref = engines(d, q, l), _ref(d, q)
    rng = np.random.default_rng(1000 * l + q + d)
    half = q // 2
    lo, hi = _limits(e.ct)
    sch = make_scheme(sk_bd=1, sk_wt=d, ch_bd=1, ch_wt=min(d, 20))
    for key_ch in _patterns(rng, (l, d), half)[::3]:
        e.set_key_ch(np.ascontiguousarray(key_ch.astype(e.ct)))
        for m in (half, hi):
            sig = np.stack(_patterns(rng, (l, d), m) + [np.full((l, d), lo)])          # the last one: beyond every bound
            n = len(sig)
            msgs = [bytes(rng.integers(0, 256, 30 + i, dtype=np.uint8)) for i in range(n)]
            vk = _verify_case(e, ref, rng, key_ch, sig, sch, msgs)
            s = np.ascontiguousarray(sig.astype(e.ct))
            ok = [1] * (n - 1) + [0]
            assert e.lm_verify(sch, vk, msgs, s, m, d).tolist() == ok, m
            assert e.lm_verify(sch, vk, msgs, s, m - 1, d).tolist() == [0] * n, m
            assert e.lm_verify(sch, vk, msgs, s, m, d - 1).tolist() == [0] * n, m
            bad = vk.copy()
            bad[:, 1, d - 1] = (bad[:, 1, d - 1].astype(np.int64) + 1) % q
            assert e.lm_verify(sch, bad, msgs, s, m, d).tolist() == [0] * n, m
            flip = s.copy()
            flip[:, l - 1, d // 2] = -flip[:, l - 1, d // 2]                           # same magnitude, wrong sign
            assert e.lm_verify(sch, vk, msgs, flip, m, d).tolist() == [0] * n, m
    # weight: w non-zero coefficients per polynomial passes wt = w and fails wt = w - 1
    w = d // 2 + 1
    sig = np.zeros((2, l, d), dtype=np.int64)
    for i in range(2):
        for j in range(l):
            sig[i, j, rng.choice(d, w, replace=False)] = rng.choice(np.array([-half, half]), w)
    msgs = [b'weight 0', b'weight 1']
    vk = _verify_case(e, ref, rng, key_ch, sig, sch, msgs)
    s = np.ascontiguousarray(sig.astype(e.ct))
    assert e.lm_verify(sch, vk, msgs, s, half, w).tolist() == [1, 1]
    assert e.lm_verify(sch, vk, msgs, s, half, w - 1).tolist() == [0, 0]


# ------------------------------------------------------------------------------------------------ BKLM aggregation
def _agg_schemes(d):
    from lattice_cryptography_b200 import make_scheme
    return [make_scheme(sk_bd=1, sk_wt=d, ch_bd=1, ch_wt=min(d, 20)),                        # signed monomials
            make_scheme(sk_bd=1, sk_wt=d, ch_bd=1, ch_wt=min(d, 20), ag_bd=1000, ag_wt=d)]    # dense polynomials


@gpu
@pytest.mark.parametrize('d,q,l', CASES_L, ids=list(map(_ids, CASES_L)))
def test_aggregation_at_extremes(engines, d, q, l):
    """aggregate = sum_i sig_i ** ag_i with signatures at +-q//2, aggregate_verify's right-hand side with key slots at
    q - 1, for monomial and dense (ag_wt = d) coefficients; then aggverify_finish at each of its limits."""
    e, ref = engines(d, q, l), _ref(d, q)
    rng = np.random.default_rng(3 * l + q + d)
    half = q // 2
    key_ch = _patterns(rng, (l, d), half)[0]
    e.set_key_ch(np.ascontiguousarray(key_ch.astype(e.ct)))
    sig = np.stack(_patterns(rng, (l, d), half)[:(2 if l == 64 else 4)])
    n = len(sig)
    kcs = ref.slots(key_ch)
    for sch in _agg_schemes(d):
        agmsg = bytes(rng.integers(0, 256, 300, dtype=np.uint8))
        coefs = e.agg_coefs(sch, agmsg, 0, n)
        ags = ref.slots_of_pairs(coefs)
        want = (ref.slots(sig) * ags[:, None, :] % q).sum(axis=0) % q
        ag_sig = e.aggregate_finish(e.aggregate_partial(sch, np.ascontiguousarray(sig.astype(e.ct)), coefs))
        assert np.abs(ag_sig.astype(np.int64)).max() <= half
        assert np.array_equal(ref.slots(ag_sig), want), sch.ag_wt
        # aggregate_verify's right-hand side
        vk = rng.integers(0, q, (n, 2, d)).astype(np.int64)
        vk[0] = q - 1
        msgs = [bytes(rng.integers(0, 256, 20 + i, dtype=np.uint8)) for i in range(n)]
        cs = ref.slots(_dense(e.challenge(sch, msgs), d))
        rhs = ((vk[:, 0] * cs % q + vk[:, 1]) % q * ags % q).sum(axis=0) % q
        got = e.aggverify_partial(sch, np.ascontiguousarray(vk.astype(e.nt)), msgs, coefs).astype(np.int64) % q
        assert np.array_equal(got, rhs), sch.ag_wt
    # aggverify_finish: partial := key_ch * ag_sig, so only the limits decide
    a = ag_sig.astype(np.int64)
    part = np.ascontiguousarray(((kcs * ref.slots(a) % q).sum(axis=0) % q).astype(e.pt))
    bd, wt = int(np.abs(a).max()), int(max(np.count_nonzero(r) for r in a))
    fin = lambda s, total, cap, b, w: e.aggverify_finish(part, np.ascontiguousarray(s.astype(e.ct)), total, cap, b, w)
    assert fin(a, n, n, bd, wt) is True
    assert fin(a, n, n - 1, bd, wt) is False
    assert fin(a, n, n, bd - 1, wt) is False
    assert fin(a, n, n, bd, wt - 1) is False
    assert fin(a, 0, n, bd, wt) is False
    tam = a.copy()
    tam[l - 1, 0] = -tam[l - 1, 0] if tam[l - 1, 0] else 1
    assert fin(tam, n, n, bd, wt) is False
    zero = np.zeros((l, d), dtype=np.int64)
    assert e.aggverify_finish(np.zeros(d, dtype=e.pt), np.ascontiguousarray(zero.astype(e.ct)), n, n, bd, wt) is False


# ------------------------------------------------------------------------------------------------ multi-trip batches
MULTI = [(32, 2147483137), (64, 64513), (1024, 2147473409)]


def _tiling(rng, k, n):
    """n source indices in [0, k), scrambled, every source present."""
    src = np.concatenate([np.arange(k), rng.integers(0, k, n - k)])
    rng.shuffle(src)
    return src


@gpu
@pytest.mark.parametrize('d,q', MULTI, ids=list(map(_ids, MULTI)))
def test_multi_trip_batches(engines, d, q):
    """More than two trips of every persistent grid plus a ragged tail: each output against the reference of its source
    item, every verdict exactly, every aggregation sum over all items."""
    import torch
    from lattice_cryptography_b200 import make_scheme
    l, k = 2, 16
    e, ref = engines(d, q, l), _ref(d, q)
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    n = 2 * 8 * GW * sms + 37               # g_grid caps a launch at 8 * num_sms blocks of GW items
    rng = np.random.default_rng(d + q)
    half = q // 2
    key_ch = rng.integers(-half, half + 1, (l, d))
    e.set_key_ch(np.ascontiguousarray(key_ch.astype(e.ct)))
    src = _tiling(rng, k, n)
    tile = lambda x: np.ascontiguousarray(x[src])
    with _Sentinel(e):
        run = lambda f, *args: _np(f(*args)).astype(np.int64)
        # transforms and products
        a = rng.integers(-half, half + 1, (k, d))
        a[0], a[1] = half, -half
        b = rng.integers(-half, half + 1, (k, d))
        assert np.array_equal(run(e.ntt_fwd, tile(a.astype(e.ct))), ref.slots(a)[src]), 'ntt_fwd'
        want = np.stack([ref.centred(ref.mul(a[i], b[i])) for i in range(k)])
        assert np.array_equal(run(e.poly_mul, tile(a.astype(e.ct)), tile(b.astype(e.ct))), want[src]), 'poly_mul'
        # keygen: the k distinct keys come from a one-trip call checked against the reference
        sch = make_scheme(sk_bd=half, sk_wt=d, ch_bd=1, ch_wt=min(d, 16))
        seeds = [format(int(x), '0128b') for x in rng.integers(0, 2 ** 62, k)]
        one = [_np(x).astype(np.int64) for x in e.lm_keygen(sch, seeds)]
        sk_coef, sk_ntt, vk_ntt, vk_coef = one
        for i in range(k):
            assert np.array_equal(vk_coef[i, 0], ref.centred(ref.dot(key_ch, sk_coef[i, 0]))), i
        assert np.array_equal(vk_ntt, ref.slots(vk_coef)) and np.array_equal(sk_ntt, ref.slots(sk_coef))
        big = [_np(x).astype(np.int64) for x in e.lm_keygen(sch, [seeds[i] for i in src])]
        for got, want in zip(big, one):
            assert np.array_equal(got, want[src]), 'keygen'
        # sign
        sk = rng.integers(0, q, (k, 2, l, d))
        sk[0] = q - 1
        msgs = [b'multi-trip %d' % i for i in range(k)]
        tmsgs = [msgs[i] for i in src]
        cs = ref.slots(_dense(_np(e.challenge(sch, msgs)), d))
        want = (cs[:, None, :] * sk[:, 0] + sk[:, 1]) % q
        sig = run(e.lm_sign, sch, tile(sk.astype(e.nt)), tmsgs)
        assert np.abs(sig).max() <= half
        assert np.array_equal(ref.slots(sig), want[src]), 'sign'
        # verify at weight d - 1: 12 valid items, then a tampered key slot, a sign-flipped coefficient, a coefficient
        # above the bound and a polynomial of weight d (all with the equation holding otherwise)
        vs = rng.choice(np.array([-half, half]), (k, l, d))
        vs[:, :, 0] = 0
        vs[15, 1, 0] = half
        vk = _verify_case(e, ref, rng, key_ch, vs, sch, msgs)
        vk[12, 1, 0] = (int(vk[12, 1, 0]) + 1) % q
        vs[13, 0, 5] = -vs[13, 0, 5]
        vs[14, 1, d - 1] = half + 1
        expect = np.array([1] * 12 + [0] * 4, dtype=np.int64)
        assert np.array_equal(run(e.lm_verify, sch, vk, msgs, np.ascontiguousarray(vs.astype(e.ct)), half, d - 1), expect)
        got = run(e.lm_verify, sch, tile(vk), tmsgs, tile(vs.astype(e.ct)), half, d - 1)
        assert np.array_equal(got, expect[src]), 'verify'
        # aggregation partial sums over all n items: signed monomials and sparse polynomials
        vsig = rng.choice(np.array([-half, half]), (k, l, d))
        vkk = rng.integers(0, q, (k, 2, d))
        vkk[0] = q - 1
        ts = (vkk[:, 0] * cs % q + vkk[:, 1]) % q
        sig_slots = ref.slots(vsig)
        for agsch in (make_scheme(ch_bd=1, ch_wt=min(d, 16)), make_scheme(ch_bd=1, ch_wt=min(d, 16), ag_bd=3, ag_wt=3)):
            coefs = _np(e.agg_coefs(agsch, b'multi-trip aggregate', 0, n))
            ags = ref.slots_of_pairs(coefs)
            per_src = np.zeros((k, d), dtype=np.int64)
            np.add.at(per_src, src, ags)
            per_src %= q
            part = _np(e.aggregate_partial(agsch, tile(vsig.astype(e.ct)), coefs))
            ag_sig = run(e.aggregate_finish, np.ascontiguousarray(part))
            assert np.array_equal(ref.slots(ag_sig), (sig_slots * per_src[:, None, :] % q).sum(axis=0) % q), \
                ('aggregate', agsch.ag_wt)
            vpart = run(e.aggverify_partial, agsch, tile(vkk.astype(e.nt)), tmsgs, coefs) % q
            assert np.array_equal(vpart, (ts * per_src % q).sum(axis=0) % q), ('aggverify_partial', agsch.ag_wt)


# ------------------------------------------------------------------------------------------------ checked build
@gpu
def test_generic_extremes_pass_on_the_checked_build():
    """A representative subset (multi-trip batches, l = 64 at d = 1024) on liblcb200_checked.so, whose device-side
    asserts trap out-of-range accesses."""
    _need_gpu()
    from lattice_cryptography_b200 import _ffi
    if _ffi.load().lcb_build_is_checked():
        pytest.skip('already running on the checked build')
    lib = os.path.join(ROOT, 'lattice_cryptography_b200', 'liblcb200_checked.so')
    if not os.path.exists(lib):
        subprocess.run(['make', '-C', os.path.join(ROOT, 'lattice_cryptography_b200', 'csrc'), '-j4', 'CHECKED=1'], check=True,
                       capture_output=True)
    env = dict(os.environ, LCB200_LIB=lib)
    r = subprocess.run([sys.executable, '-m', 'pytest', 'tests/test_gpu_generic_extremes.py', '-q', '-x', '-m', 'gpu', '-k',
                        'd32-q2147483137 or (aggregation and d1024-q2147473409-l64)', '-p', 'no:cacheprovider'],
                       env=env, capture_output=True, text=True, timeout=1500, cwd=ROOT)
    tail = r.stdout[-2500:] + r.stderr[-1500:]
    assert r.returncode == 0, tail
    assert ' passed' in r.stdout and 'failed' not in r.stdout, tail
