"""The tensor-core verify (ring.cu, k_verify_tc) at worst-case magnitudes, at every 16-bit modulus range and vector length
it can meet, and through each caller that reaches it (run with -m gpu).

k_verify_tc decides every int16-row verify batch of at least one 128-verify tile per SM (TC_MIN items, from the device's
SM count).  The cases here send at least TC_MIN items: the smallest NTT prime, the shipped ones, the largest with the lazy
limb reduction (32257), the smallest without it (36353), the two smallest that need the subtraction (45569, 51713) and the
largest (64513); vectors of 1, 3, 13 and 64 polynomials
(4, 12, 52 and 256 K chunks through three shared-memory stages); key_ch at +-q//2; signature rows at +-32767, +-q//2 and
-32768, random over [-32767, 32767], and built from the coefficient pairs whose limb inputs are least reduced by the
Barrett step (at q >= 45569 beyond 2^16 without the subtraction); every vk_left slot at q - 1; challenge weights 1, 20, 50
and 256.  The equation is built to HOLD (vk_right, or the
adaptor statement, is solved for it with schoolbook negacyclic products on int64), so one wrong residue anywhere flips a
verdict.  A few base items are solved once per (q, l, key_ch) and tiled on the device to the batch size.  Verdicts are
compared with the statement of the rules and with k_verify, which takes every slice of fewer than TC_MIN items.
Callers: lm_verify, lm_verify with adaptor statements (extra_rhs), and batched BKLM aggregate-verify (rhs_only, with the
bound min(avf_bd, 32768): at 32768 every int16 passes)."""
import hashlib
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
D = 256
BR8 = np.array([int(format(p, '08b')[::-1], 2) for p in range(D)], np.int64)


def _tc_min():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count * 128


# ---------------------------------------------------------------- the reference
def negacyclic_mul(a, b, q):
    full = np.convolve(a.astype(np.int64), b.astype(np.int64))
    res = full[:D].copy()
    res[:D - 1] -= full[D:]
    return res % q


def centred(x, q):
    x = np.asarray(x, dtype=np.int64) % q
    return np.where(x > (q - 1) // 2, x - q, x)


def dense_challenge(pairs):
    c = np.zeros(D, dtype=np.int64)
    for idx, s in pairs:
        c[int(idx)] = int(s)
    return c


def _alt(m, l):
    return np.broadcast_to(np.where(np.arange(D) % 2 == 0, m, -m), (l, D)).astype(np.int64)


def _key_ch_patterns(q, l):
    half = q // 2
    return [('all_plus', np.full((l, D), half, np.int64)), ('all_minus', np.full((l, D), -half, np.int64)),
            ('alternating', _alt(half, l))]


def _target(q, key_ch, sig, pairs):
    """key_ch . sig + c + 1 (mod q, centred): with vk_left = -1 (every NTT slot q - 1) the equation
    key_ch . sig == vk_left c + vk_right + st holds when vk_right + st equals this minus the constant polynomial 1."""
    acc = dense_challenge(pairs)
    acc[0] += 1
    for j in range(key_ch.shape[0]):
        acc = acc + negacyclic_mul(key_ch[j], sig[j], q)
    return centred(acc, q)


def _solved_keys(e, q, key_ch, sigs, pairs):
    """vk [n, 2, D]: vk_left slots all q - 1 (the polynomial -1), vk_right solved so that the equation holds."""
    one = np.eye(1, D, dtype=np.int64)[0]                 # the constant polynomial 1
    vkr = np.stack([centred(_target(q, key_ch, s, p) - one, q) for s, p in zip(sigs, pairs)])
    vk = np.empty((len(sigs), 2, D), np.uint16)
    vk[:, 0] = q - 1
    vk[:, 1] = e.ntt_fwd(np.ascontiguousarray(vkr.astype(np.int16)))
    return vk


def _tile(base, idx_d):
    """base[idx] on the device (uint16 rows are gathered as int16 and viewed back)."""
    import torch
    base = np.ascontiguousarray(base)
    if base.dtype == np.uint16:
        return torch.from_numpy(base.view(np.int16)).cuda()[idx_d].contiguous().view(torch.uint16)
    return torch.from_numpy(base).cuda()[idx_d].contiguous()


def _set_u16(t, item, slot, v):
    import torch
    t.view(torch.int16)[item, slot] = int(np.uint16(v).view(np.int16))


def _verify(e, sch, vk, msgs, sig, bd, wt, st=None):
    import torch
    torch.cuda.synchronize()
    return e.lm_verify(sch, vk, msgs, sig, bd, wt, st_ntt=st, device=True).cpu().numpy()


def _k_verify(e, sch, vk, msgs, sig, bd, wt, st=None):
    """The verdicts of k_verify: slices of fewer than TC_MIN items never reach k_verify_tc."""
    step = _tc_min() // 2
    return np.concatenate([_verify(e, sch, vk[i:i + step], msgs[i:i + step], sig[i:i + step], bd, wt,
                                   None if st is None else st[i:i + step]) for i in range(0, len(msgs), step)])


def _batch_sizes():
    m = _tc_min()
    return [m + 1, 2 * m + 77]             # last tile with 1 and with 77 live items; some SMs take one tile more


def _index(n, nb, last):
    import torch
    idx = np.arange(n) % nb
    idx[-1] = last                          # the last item (in a partial tile) is one that passes
    return torch.from_numpy(idx).cuda(), idx


def _worst_pair_rows(q, l, rng):
    """l rows built from the coefficient pairs (a_lo = coefficient j, a_hi = coefficient j + 128) whose limb inputs
    hi z + lo + kz (biased halves hi = a_hi + 32768, lo = a_lo + 32768, z either square root of -1) have the largest
    Barrett results before any subtraction (barrett_lazy), out of 2^20 random pairs in [-32767, 32767].  From q = 45569
    up these results reach 2^16: without the subtraction k_verify_tc takes for q > 32768 a limb would lose a bit.
    -> rows [l, D], the smallest such result used"""
    psi = next(g for g in range(2, q) if pow(g, 256, q) == q - 1)
    z0 = pow(psi, 128, q)
    a = rng.integers(-32767, 32768, (1 << 20, 2))
    lo, hi = (a[:, 0] + 32768).astype(np.uint64), (a[:, 1] + 32768).astype(np.uint64)
    barrett = np.uint64(((1 << 32) - 1) // q)
    worst = np.zeros(len(a), np.uint64)
    for z in (z0, q - z0):
        b15 = 32768 % q
        x = hi * np.uint64(z) + lo + np.uint64((2 * q - b15 - b15 * z % q) % q)
        worst = np.maximum(worst, x - np.uint64(q) * ((x * barrett) >> np.uint64(32)))
    pick = np.argsort(worst)[::-1][:128 * l].reshape(l, 128)
    return np.concatenate([a[pick, 0], a[pick, 1]], axis=1), int(worst[pick].min())


# ---------------------------------------------------------------- lm_verify at the extremes
# 45569 and 51713: the smallest moduli where the limbs need k_verify_tc's subtraction (tests/test_verify_tc_limbs_cpu.py)
CASES = [(7681, 1, 1), (7681, 3, 256), (11777, 13, 20), (11777, 64, 1), (32257, 3, 20), (32257, 64, 256),
         (36353, 1, 256), (36353, 13, 1), (39937, 3, 50), (39937, 13, 256), (45569, 13, 50), (51713, 3, 20),
         (64513, 1, 20), (64513, 64, 1)]


@pytest.mark.parametrize('q,l,ch_wt', CASES, ids=[f'q{q}-l{l}-w{w}' for q, l, w in CASES])
def test_verify_holds_at_extremes(q, l, ch_wt):
    from lattice_cryptography_b200 import Engine, make_scheme
    half = q // 2
    sch = make_scheme(sk_bd=1, sk_wt=D, ch_bd=1, ch_wt=ch_wt)
    e = Engine(128, q, D, l)
    try:
        rng = np.random.default_rng(q * 100 + l)
        low = _alt(32767, l).copy()
        low[l - 1] = -32768                               # -32768 in the last row: its bound flag is set in the last chunk
        sigs = np.stack([low, np.full((l, D), 32767), np.full((l, D), -32767), _alt(32767, l),
                         rng.choice(np.array([-32767, 32767]), (l, D)), np.full((l, D), half), np.full((l, D), -half),
                         _alt(half, l), rng.integers(-32767, 32768, (l, D))]).astype(np.int64)
        worst_rows, worst = _worst_pair_rows(q, l, rng)
        assert (worst >= 1 << 16) == (q >= 45569)
        sigs = np.concatenate([sigs, worst_rows[None]])
        mag = np.abs(sigs).max(axis=(1, 2))
        nb = len(sigs)
        for kname, key_ch in _key_ch_patterns(q, l):
            e.set_key_ch(np.ascontiguousarray(key_ch.astype(np.int16)))
            msgs = [f'tc extremes q{q} l{l} {kname} item {i}'.encode() for i in range(nb)]
            vk = _solved_keys(e, q, key_ch, sigs, e.challenge(sch, msgs))
            for n in _batch_sizes():
                idx_d, idx = _index(n, nb, 1)
                sig_d, vk_d = _tile(sigs.astype(np.int16), idx_d), _tile(vk, idx_d)
                m_all = [msgs[i] for i in idx]
                for bd in (32767, 32766, half, half - 1):
                    want = (mag[idx] <= bd).astype(np.uint8)
                    got = _verify(e, sch, vk_d, m_all, sig_d, bd, D)
                    assert np.array_equal(got, want), (kname, n, bd, np.flatnonzero(got != want)[:8])
                assert np.array_equal(_k_verify(e, sch, vk_d, m_all, sig_d, 32767, D), (mag[idx] <= 32767).astype(np.uint8))
                # one coefficient of the last item, in the last chunk, one step towards zero
                sig_d[n - 1, l - 1, D - 1] -= 1
                want = (mag[idx] <= 32767).astype(np.uint8)
                want[n - 1] = 0
                assert np.array_equal(_verify(e, sch, vk_d, m_all, sig_d, 32767, D), want), (kname, n)
                del sig_d, vk_d
    finally:
        e.close()


# ---------------------------------------------------------------- adaptor verify: three terms in the right-hand side
@pytest.mark.parametrize('q,l', [(11777, 13), (39937, 23), (64513, 3)])
def test_adaptor_statements_at_extremes(q, l):
    """lm_verify(..., st_ntt): vk and statement slots at q - 1.  Half the items have both key halves all q - 1 and a
    solved statement, the other half vk_left and the statement all q - 1 and a solved vk_right."""
    from lattice_cryptography_b200 import Engine, make_scheme
    half = q // 2
    sch = make_scheme(sk_bd=1, sk_wt=D, ch_bd=1, ch_wt=20 if q != 39937 else 50)
    e = Engine(128 if q != 39937 else 256, q, D, l)
    try:
        key_ch = _alt(half, l)
        e.set_key_ch(np.ascontiguousarray(key_ch.astype(np.int16)))
        rng = np.random.default_rng(q + l)
        sig4 = [np.full((l, D), 32767), np.full((l, D), -half), _alt(32767, l), rng.choice(np.array([-32767, 32767]), (l, D))]
        sigs = np.stack(sig4 + sig4).astype(np.int64)
        nb = len(sigs)
        msgs = [f'adaptor extremes q{q} item {i}'.encode() for i in range(nb)]
        pairs = e.challenge(sch, msgs)
        t_ntt = e.ntt_fwd(np.ascontiguousarray(np.stack([_target(q, key_ch, s, p) for s, p in zip(sigs, pairs)]).astype(np.int16)))
        vk = np.full((nb, 2, D), q - 1, np.uint16)
        st = np.full((nb, D), q - 1, np.uint16)
        st[:4] = t_ntt[:4]                  # vk all q - 1, statement solved
        vk[4:, 1] = t_ntt[4:]               # vk_left and statement all q - 1, vk_right solved
        n = _tc_min() + 77
        idx_d, idx = _index(n, nb, 5)
        sig_d, vk_d, st_d = _tile(sigs.astype(np.int16), idx_d), _tile(vk, idx_d), _tile(st, idx_d)
        m_all = [msgs[i] for i in idx]
        assert _verify(e, sch, vk_d, m_all, sig_d, 32767, D, st_d).all()
        assert np.array_equal(_k_verify(e, sch, vk_d, m_all, sig_d, 32767, D, st_d), np.ones(n, np.uint8))
        assert not _verify(e, sch, vk_d, m_all, sig_d, 32767, D).any()        # the statement term is not optional
        for item in (n - 1, n // 3):
            keep = int(st[idx[item], 77])
            _set_u16(st_d, item, 77, (keep + 1) % q)
            want = np.ones(n, np.uint8)
            want[item] = 0
            assert np.array_equal(_verify(e, sch, vk_d, m_all, sig_d, 32767, D, st_d), want), item
            _set_u16(st_d, item, 77, keep)
    finally:
        e.close()


# ---------------------------------------------------------------- weight at the limit (CHECK_WT)
def _positions(rng, k, hh=None):
    """k distinct coefficient positions; with hh, only those of converter half hh (coefficient j of a row belongs to
    pair m = j mod 128, quarter m // 32 and half (m mod 32) // 16)."""
    pool = np.arange(D) if hh is None else np.flatnonzero((np.arange(D) % 32) // 16 == hh)
    return rng.choice(pool, k, replace=False)


@pytest.mark.parametrize('q,l', [(11777, 1), (64513, 64)])
@pytest.mark.parametrize('wt', [1, 37, 255])
def test_weight_at_the_limit(q, l, wt):
    """Rows with exactly wt non-zeros pass; wt + 1 in one row fails, whether that row is the first or the last, and
    when each converter half of the row holds at most wt of them (only the pairwise sum exceeds wt).  Every item's
    vk_right is solved, so the weight alone decides: with the bound wt + 1 every item passes."""
    from lattice_cryptography_b200 import Engine, make_scheme
    sch = make_scheme(sk_bd=1, sk_wt=D, ch_bd=1, ch_wt=20)
    e = Engine(128, q, D, l)
    try:
        rng = np.random.default_rng(wt * 7 + l)
        key_ch = rng.choice(np.array([-(q // 2), q // 2]), (l, D))
        e.set_key_ch(np.ascontiguousarray(key_ch.astype(np.int16)))

        def row(k, hh=None):
            r = np.zeros(D, np.int64)
            if hh is None:
                r[_positions(rng, k)] = rng.choice(np.array([-32767, 32767]), k)
            else:
                k0 = (k + 1) // 2
                r[_positions(rng, k0, 0)] = 32767
                r[_positions(rng, k - k0, 1)] = -32767
            return r

        def item(heavy_row=None, split=False):
            s = np.stack([row(wt) for _ in range(l)])
            if heavy_row is not None:
                s[heavy_row] = row(wt + 1, 0 if split else None)
            return s

        sigs = [item(), item(l - 1), item(0), item(l - 1, split=True), item(0, split=True), item()]
        one_more = sigs[5].copy()                       # item 5 with one more non-zero in its last row
        one_more[l - 1, int(np.flatnonzero(one_more[l - 1] == 0)[0])] = 1
        sigs = np.stack(sigs + [one_more])
        want_base = ((sigs != 0).sum(axis=2).max(axis=1) <= wt).astype(np.uint8)
        assert want_base.tolist() == [1, 0, 0, 0, 0, 1, 0]
        nb = len(sigs)
        msgs = [f'weight q{q} l{l} wt{wt} item {i}'.encode() for i in range(nb)]
        vk = _solved_keys(e, q, key_ch, sigs, e.challenge(sch, msgs))
        n = _tc_min() + 77
        for last in (5, 6):                             # the last item (partial tile) at the limit, then one past it
            idx_d, idx = _index(n, nb, last)
            sig_d, vk_d = _tile(sigs.astype(np.int16), idx_d), _tile(vk, idx_d)
            m_all = [msgs[i] for i in idx]
            got = _verify(e, sch, vk_d, m_all, sig_d, 32767, wt)
            assert got[-1] == want_base[last]
            assert np.array_equal(got, want_base[idx])
            assert np.array_equal(_k_verify(e, sch, vk_d, m_all, sig_d, 32767, wt), want_base[idx])
            assert _verify(e, sch, vk_d, m_all, sig_d, 32767, wt + 1).all()
            del sig_d, vk_d
    finally:
        e.close()


# ---------------------------------------------------------------- batched BKLM aggregate-verify
def _coefs(msgs):
    """(k, s) of the single item of each group: hash of b'AG_SALT' + b'0' + the group's aggregation message."""
    ks, ss = [], []
    for m in msgs:
        dg = hashlib.shake_256(b'AG_SALT' + b'0' + m).digest(2)
        ks.append(dg[0])
        ss.append(1 if dg[1] & 0x80 else -1)
    return np.array(ks, np.int64), np.array(ss, np.int64)


def _mono_ntt(q, k, s, inverse=False):
    """NTT images [n, D] of s X^k (or of s X^-k): slot p evaluates at psi^(2 bitrev8(p) + 1), psi the least primitive
    512-th root of unity."""
    psi = next(g for g in range(2, q) if pow(g, 256, q) == q - 1)
    pw = np.array([pow(psi, t, q) for t in range(512)], np.int64)
    e = (2 * BR8 + 1)[None, :] * k[:, None] * (-1 if inverse else 1)
    return (s[:, None] * pw[e % 512]) % q


def _rules(z, bd, wt):
    z = z.astype(np.int64)
    mx = np.abs(z).max(axis=(1, 2))
    rw = (z != 0).sum(axis=2).max(axis=1)
    return ((mx >= 1) & (mx <= bd) & (rw <= wt)).astype(np.uint8)


@pytest.mark.parametrize('secpar', [128, 256])
def test_bklm_batch_verify_at_extremes(secpar):
    """At least TC_MIN aggregates of one signature each: aggregates at +-32767, one with a -32768 coefficient and one with
    a row of -32768, keys solved so that every equation holds; avf_bd = 32767 rejects exactly the -32768 aggregates, 32768
    and 40000 accept every aggregate."""
    from lattice_cryptography_b200 import Engine, make_scheme
    q, l, ch_wt = (11777, 13, 20) if secpar == 128 else (39937, 23, 50)
    sch = make_scheme(sk_bd=1, sk_wt=D, ch_bd=1, ch_wt=ch_wt)
    e = Engine(secpar, q, D, l)
    try:
        rng = np.random.default_rng(secpar + 5)
        key_ch = rng.integers(-(q // 2), q // 2 + 1, (l, D))
        e.set_key_ch(np.ascontiguousarray(key_ch.astype(np.int16)))
        one = _alt(32767, l).copy()
        one[l - 1, D - 1] = -32768
        row = _alt(32767, l).copy()
        row[0] = -32768
        zs = np.stack([np.full((l, D), 32767), np.full((l, D), -32767), _alt(32767, l),
                       rng.choice(np.array([-32767, 32767]), (l, D)), one, row]).astype(np.int16)
        nb = len(zs)
        msgs = [f'bklm tc extremes {secpar} group {g}'.encode() for g in range(nb)]
        chm = [f'bklm tc extremes {secpar} item {g}'.encode() for g in range(nb)]
        ks, ss = _coefs(msgs)
        key_hat = e.ntt_fwd(np.ascontiguousarray(key_ch.astype(np.int16))).astype(np.int64)
        y = (key_hat[None] * e.ntt_fwd(zs).astype(np.int64)).sum(axis=1) % q
        pairs = e.challenge(sch, chm)
        c_hat = e.ntt_fwd(np.ascontiguousarray(np.stack([dense_challenge(p) for p in pairs]).astype(np.int16))).astype(np.int64)
        vk = np.empty((nb, 2, D), np.int64)
        vk[:, 0] = q - 1
        vk[:, 1] = (y * _mono_ntt(q, ks, ss, inverse=True) - (q - 1) * c_hat) % q
        assert np.array_equal((vk[:, 0] * c_hat + vk[:, 1]) % q * _mono_ntt(q, ks, ss) % q, y)
        vk = vk.astype(np.uint16)
        n = _batch_sizes()[0 if secpar == 128 else 1]
        idx = np.arange(n) % nb
        idx[-1] = 0
        off = np.arange(n + 1, dtype=np.int64)
        vk_all, zs_all = np.ascontiguousarray(vk[idx]), np.ascontiguousarray(zs[idx])
        m_all, c_all = [msgs[i] for i in idx], [chm[i] for i in idx]
        for bd in (32767, 32768, 40000):
            want = _rules(zs, bd, D)
            assert want.tolist() == ([1, 1, 1, 1, 0, 0] if bd == 32767 else [1] * nb)
            single = [e.aggverify_finish(e.aggverify_partial(sch, vk[g:g + 1], chm[g:g + 1], e.agg_coefs(sch, msgs[g], 0, 1)),
                                         np.ascontiguousarray(zs[g]), 1, 1, bd, D) for g in range(nb)]
            assert np.array_equal(np.array(single, np.uint8), want), bd
            got = e.aggregate_verify_batch(sch, off, vk_all, c_all, m_all, zs_all, 1, bd, D)
            assert np.array_equal(got, want[idx]), (bd, np.flatnonzero(got != want[idx])[:8])
        zs_all[n - 1, l - 1, D - 1] = 32766
        want = _rules(zs, 32768, D)[idx]
        want[n - 1] = 0
        assert np.array_equal(e.aggregate_verify_batch(sch, off, vk_all, c_all, m_all, zs_all, 1, 32768, D), want)
    finally:
        e.close()


# ---------------------------------------------------------------- the checked build
def test_extremes_pass_on_the_checked_build():
    from lattice_cryptography_b200 import _ffi
    if _ffi.load().lcb_build_is_checked():
        pytest.skip('already running on the checked build')
    lib = os.path.join(ROOT, 'lattice_cryptography_b200', 'liblcb200_checked.so')
    if not os.path.exists(lib):
        subprocess.run(['make', '-C', os.path.join(ROOT, 'lattice_cryptography_b200', 'csrc'), '-j4', 'CHECKED=1'], check=True,
                       capture_output=True)
    env = dict(os.environ, LCB200_LIB=lib)
    r = subprocess.run([sys.executable, '-m', 'pytest', 'tests/test_gpu_verify_tc_extremes.py', '-q', '-x', '-m', 'gpu', '-k',
                        'q7681-l3 or (bklm_batch_verify_at_extremes and 128)', '-p', 'no:cacheprovider'],
                       env=env, capture_output=True, text=True, timeout=1500, cwd=ROOT)
    tail = r.stdout[-2500:] + r.stderr[-1500:]
    assert r.returncode == 0, tail
    assert '2 passed' in r.stdout and 'failed' not in r.stdout, tail
