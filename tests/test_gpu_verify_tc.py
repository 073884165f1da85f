"""The tensor-core verify (ring.cu, k_verify_tc) at its tile edges (run with -m gpu): batches that are not multiples of the
128-verify tile or of the grid, key_ch re-set between calls (the context rebuilds its key_ch matrices), every tampering
kind of bench.py, and the bound and weight checks one step either side of the limit, on full-range int16 rows.  Batches
below one tile per SM (n = 1, 127) take k_verify, the others k_verify_tc; SMS is the B200's SM count."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

D = 256
Q, L, SK_BD, CH_WT, VF_BD = 11777, 13, 45, 20, 945
SMS = 148
TC_MIN = SMS * 128                  # the smallest batch k_verify_tc takes


def negacyclic_mul(a, b, q):
    full = np.convolve(a.astype(np.int64), b.astype(np.int64))
    res = full[:D].copy()
    res[:D - 1] -= full[D:]
    return res % q


def centred(x, q):
    x = np.asarray(x, dtype=np.int64) % q
    return np.where(x > (q - 1) // 2, x - q, x)


def engine(seed):
    from lattice_cryptography_b200 import Engine, make_scheme
    e = Engine(128, Q, D, L)
    rng = np.random.default_rng(seed)
    key_ch = rng.integers(-(Q // 2), Q // 2 + 1, (L, D)).astype(np.int16)
    e.set_key_ch(np.ascontiguousarray(key_ch))
    return e, make_scheme(sk_bd=SK_BD, sk_wt=D, ch_bd=1, ch_wt=CH_WT), key_ch


def signed_batch(e, sch, n, tag):
    seeds = [f'{tag}-seed-{i}' for i in range(n)]
    msgs = [f'{tag} message {i} '.encode() + bytes([48 + (i & 1)]) for i in range(n)]
    _, sk_ntt, vk_ntt, _ = e.lm_keygen(sch, seeds, want_sk_coef=False, want_vk_coef=False)
    return vk_ntt, msgs, e.lm_sign(sch, sk_ntt, msgs)


@pytest.mark.parametrize('n', [1, 127, TC_MIN, TC_MIN + 5, 2 * TC_MIN + 77])
def test_batches_with_every_tampering_kind(n):
    e, sch, _ = engine(n)
    try:
        vk, msgs, sig = signed_batch(e, sch, n, 'b')
        sig = sig.copy()
        expect = np.ones(n, np.uint8)
        for i in range(0, n, 64):
            kind = (i // 64) % 3
            if kind == 0:
                sig[i, i % L, (3 * i) % D] += 1
            elif kind == 1:
                sig[i, (i + 1) % L, (7 * i) % D] = VF_BD + 1
            else:
                msgs[i] = msgs[i][:-1] + bytes([msgs[i][-1] ^ 1])
            expect[i] = 0
        assert np.array_equal(e.lm_verify(sch, vk, msgs, sig, VF_BD, D), expect)
        if n > 1:                                           # the last row of a partial tile, alone and tampered
            sig[n - 1, L - 1, D - 1] ^= 1
            expect[n - 1] = 0
            assert np.array_equal(e.lm_verify(sch, vk, msgs, sig, VF_BD, D), expect)
    finally:
        e.close()


def test_key_ch_reset_between_calls():
    e, sch, key_a = engine(1)
    try:
        n = TC_MIN + 300
        vk_a, msgs_a, sig_a = signed_batch(e, sch, n, 'a')
        assert e.lm_verify(sch, vk_a, msgs_a, sig_a, VF_BD, D).all()
        key_b = np.ascontiguousarray(np.roll(key_a, 1, axis=1))
        e.set_key_ch(key_b)
        assert not e.lm_verify(sch, vk_a, msgs_a, sig_a, VF_BD, D).any()
        vk_b, msgs_b, sig_b = signed_batch(e, sch, n, 'b')
        assert e.lm_verify(sch, vk_b, msgs_b, sig_b, VF_BD, D).all()
        e.set_key_ch(np.ascontiguousarray(key_a))
        assert e.lm_verify(sch, vk_a, msgs_a, sig_a, VF_BD, D).all()
        assert not e.lm_verify(sch, vk_b, msgs_b, sig_b, VF_BD, D).any()
    finally:
        e.close()


def witness_case(e, key_ch, rows):
    """(witnesses, statements) for the given rows, each repeated so that the batch reaches k_verify_tc"""
    st = np.empty((len(rows), D), np.int64)
    for i, w in enumerate(rows):
        acc = np.zeros(D, np.int64)
        for k in range(L):
            acc = (acc + negacyclic_mul(key_ch[k], w[k], Q)) % Q
        st[i] = centred(acc, Q)
    reps = -(-(TC_MIN + 3) // len(rows))
    wit = np.ascontiguousarray(np.tile(np.stack(rows).astype(np.int16), (reps, 1, 1)))
    return wit, np.ascontiguousarray(np.tile(e.ntt_fwd(np.ascontiguousarray(st.astype(np.int16))), (reps, 1)))


@pytest.mark.parametrize('mag', [1, VF_BD, 32767])
def test_bound_at_the_limit_and_one_past(mag):
    e, _, key_ch = engine(mag)
    try:
        rng = np.random.default_rng(mag)
        rows = []
        for sign in (1, -1):
            w = rng.integers(-mag, mag + 1, (L, D))
            w[rng.integers(L), rng.integers(D)] = sign * mag
            rows.append(w)
        rows.append(np.full((L, D), -mag))
        rows.append(np.where(np.arange(D) % 2 == 0, mag, -mag)[None, :].repeat(L, axis=0))
        wit, st = witness_case(e, key_ch, rows)
        n = len(wit)
        assert e.witness_verify(wit, st, mag, D).all()
        assert not e.witness_verify(wit, st, mag - 1, D).any()
        st_bad = st.copy()
        st_bad[n - 1, 200] = (int(st_bad[n - 1, 200]) + 1) % Q
        want = np.ones(n, np.uint8)
        want[n - 1] = 0
        assert np.array_equal(e.witness_verify(wit, st_bad, mag, D), want)
    finally:
        e.close()


def test_int16_limits_and_weight():
    e, _, key_ch = engine(5)
    try:
        rng = np.random.default_rng(5)
        full = rng.integers(-32768, 32768, (L, D))
        full[0, 0], full[1, 1] = -32768, 32767
        sparse = np.zeros((L, D), np.int64)
        for k in range(L):                                   # exactly 40 non-zero coefficients in every row
            sparse[k, rng.choice(D, 40, replace=False)] = rng.choice(np.array([-32767, 32767, 5]), 40)
        wit, st = witness_case(e, key_ch, [full, sparse])
        # every row passes a bound of 32767 but the one holding -32768; the sparse rows pass a weight of 40, not 39
        got = e.witness_verify(wit, st, 32767, D)
        assert np.array_equal(got, np.arange(len(wit)) % 2)
        assert np.array_equal(e.witness_verify(wit, st, 32767, 40), np.arange(len(wit)) % 2)
        assert not e.witness_verify(wit, st, 32767, 39).any()
    finally:
        e.close()
