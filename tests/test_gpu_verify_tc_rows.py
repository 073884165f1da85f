"""The tensor-core verify (ring.cu, k_verify_tc) at tile and grid edges and on caller views (run with -m gpu): last tiles
with a few live items, grids where some SMs take one tile more than others, caller device views that start at a non-zero
item, a caller view that is not 16-byte aligned, and secpar 256 (l = 23, q > 32768: limbs reduced below q) either side of
the one-tile-per-SM threshold and on full-range int16 rows.  Every verdict is compared with the construction rule and,
where k_verify_tc ran, with k_verify, which takes any slice below one tile per SM; SMS is the B200's SM count."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

D = 256
SMS = 148
TC_MIN = SMS * 128                  # the smallest batch k_verify_tc takes
PARAMS = {128: dict(q=11777, l=13, sk_bd=45, ch_wt=20, vf_bd=945), 256: dict(q=39937, l=23, sk_bd=65, ch_wt=50, vf_bd=3315)}


def engine(secpar):
    from lattice_cryptography_b200 import Engine, make_scheme
    p = PARAMS[secpar]
    e = Engine(secpar, p['q'], D, p['l'])
    rng = np.random.default_rng(secpar)
    key_ch = rng.integers(-(p['q'] // 2), p['q'] // 2 + 1, (p['l'], D)).astype(np.int16)
    e.set_key_ch(np.ascontiguousarray(key_ch))
    return e, make_scheme(sk_bd=p['sk_bd'], sk_wt=D, ch_bd=1, ch_wt=p['ch_wt']), p


def tampered_batch(e, sch, p, n, tag):
    """n signed triples; every 61st item and the last three are tampered (a coefficient off by one, one past the bound,
    or a flipped message bit, in turn).  -> vk, msgs, sig, expected verdicts"""
    seeds = [f'{tag}-seed-{i}' for i in range(n)]
    msgs = [f'{tag} message {i} '.encode() + bytes([48 + (i & 1)]) for i in range(n)]
    _, sk_ntt, vk, _ = e.lm_keygen(sch, seeds, want_sk_coef=False, want_vk_coef=False)
    sig = e.lm_sign(sch, sk_ntt, msgs).copy()
    expect = np.ones(n, np.uint8)
    l = p['l']
    for k, i in enumerate(sorted(set(range(0, n, 61)) | {n - 3, n - 2, n - 1})):
        if i < 0:
            continue
        kind = k % 3
        if kind == 0:
            sig[i, (5 * i) % l, (3 * i) % D] += 1
        elif kind == 1:
            sig[i, (i + 1) % l, (7 * i) % D] = p['vf_bd'] + 1
        else:
            msgs[i] = msgs[i][:-1] + bytes([msgs[i][-1] ^ 1])
        expect[i] = 0
    return vk, msgs, sig, expect


def k_verify_reference(e, sch, p, vk, msgs, sig):
    """The verdicts of k_verify: slices of fewer than TC_MIN items never reach k_verify_tc"""
    n, step = len(msgs), TC_MIN // 2
    return np.concatenate([e.lm_verify(sch, vk[i:i + step], msgs[i:i + step], sig[i:i + step], p['vf_bd'], D)
                           for i in range(0, n, step)])


@pytest.mark.parametrize('n', [
    TC_MIN + 1,                     # 149 tiles: the last holds one live item, one SM takes two tiles
    TC_MIN + 74 * 128 + 3,          # half the SMs take two tiles, the last tile has 3 live items
    3 * TC_MIN - 125,               # every SM three tiles but one, the last tile has 3 live items
])
def test_tile_edges_match_k_verify(n):
    e, sch, p = engine(128)
    try:
        vk, msgs, sig, expect = tampered_batch(e, sch, p, n, f'edge{n}')
        got = e.lm_verify(sch, vk, msgs, sig, p['vf_bd'], D)
        assert np.array_equal(got, expect)
        assert np.array_equal(got, k_verify_reference(e, sch, p, vk, msgs, sig))
    finally:
        e.close()


@pytest.mark.parametrize('first', [1, 77, 130])
def test_device_view_at_an_item_offset(first):
    import torch
    e, sch, p = engine(128)
    try:
        n = TC_MIN + 200
        vk, msgs, sig, expect = tampered_batch(e, sch, p, first + n, f'off{first}')
        d_sig, d_vk = torch.from_numpy(sig).cuda(), torch.from_numpy(vk).cuda()
        got = e.lm_verify(sch, d_vk[first:], msgs[first:], d_sig[first:], p['vf_bd'], D, device=True)
        assert np.array_equal(got.cpu().numpy(), expect[first:])
    finally:
        e.close()


def test_misaligned_device_view_is_refused():
    """A caller device buffer of signatures that is 4- but not 16-byte aligned is refused before any kernel runs (the row
    copies and k_verify's 16-byte loads both need the alignment); the context stays usable."""
    import torch
    from lattice_cryptography_b200 import LcbError
    e, sch, p = engine(128)
    try:
        n = TC_MIN + 9
        vk, msgs, sig, expect = tampered_batch(e, sch, p, n, 'mis')
        raw = torch.zeros(sig.nbytes + 16, dtype=torch.uint8, device='cuda')
        view = raw[4:4 + sig.nbytes]
        view.copy_(torch.from_numpy(sig.reshape(-1).view(np.uint8)).cuda())
        assert view.data_ptr() % 16 == 4
        with pytest.raises(LcbError):
            e.lm_verify(sch, vk, msgs, view.view(torch.int16).view(sig.shape), p['vf_bd'], D)
        assert np.array_equal(e.lm_verify(sch, vk, msgs, sig, p['vf_bd'], D), expect)
    finally:
        e.close()


@pytest.mark.parametrize('n', [TC_MIN - 1, TC_MIN, TC_MIN + 77])
def test_secpar_256_either_side_of_the_threshold(n):
    e, sch, p = engine(256)
    try:
        vk, msgs, sig, expect = tampered_batch(e, sch, p, n, f's256n{n}')
        got = e.lm_verify(sch, vk, msgs, sig, p['vf_bd'], D)
        assert np.array_equal(got, expect)
        if n >= TC_MIN:
            assert np.array_equal(got, k_verify_reference(e, sch, p, vk, msgs, sig))
    finally:
        e.close()


def test_secpar_256_full_int16_rows():
    """Witness rows anywhere in [-32767, 32767] at q = 39937: the limbs of the largest products, through k_verify_tc"""
    e, _, p = engine(256)
    try:
        q, l = p['q'], p['l']
        rng = np.random.default_rng(256)
        key_ch = rng.integers(-(q // 2), q // 2 + 1, (l, D))
        e.set_key_ch(np.ascontiguousarray(key_ch.astype(np.int16)))
        rows = [rng.integers(-32767, 32768, (l, D)), np.full((l, D), 32767), np.full((l, D), -32767),
                np.where(np.arange(D) % 2 == 0, 32767, -32767)[None, :].repeat(l, axis=0)]
        st = []
        for w in rows:
            acc = np.zeros(2 * D - 1, np.int64)
            for k in range(l):
                acc += np.convolve(key_ch[k].astype(np.int64), w[k].astype(np.int64))
            res = acc[:D].copy()
            res[:D - 1] -= acc[D:]
            st.append((res + q // 2) % q - q // 2)
        st_ntt = e.ntt_fwd(np.ascontiguousarray(np.stack(st).astype(np.int16)))
        reps = -(-(TC_MIN + 5) // len(rows))
        wit = np.ascontiguousarray(np.tile(np.stack(rows).astype(np.int16), (reps, 1, 1)))
        st_all = np.ascontiguousarray(np.tile(st_ntt, (reps, 1)))
        n = len(wit)
        assert e.witness_verify(wit, st_all, 32767, D).all()
        st_all[n - 2, 17] = (int(st_all[n - 2, 17]) + 1) % q
        want = np.ones(n, np.uint8)
        want[n - 2] = 0
        assert np.array_equal(e.witness_verify(wit, st_all, 32767, D), want)
    finally:
        e.close()
