"""Batches of independent BKLM aggregates (lcb_bklm_aggregate_batch / lcb_bklm_aggregate_verify_batch and the drop-in
aggregate_batch / aggregate_verify_batch): every group must come out exactly as the single-aggregate path makes it, and
the aggregates must also match a statement that does not use the engine (hashlib coefficients, numpy rotations)."""
import hashlib
import os
import subprocess
import sys
from secrets import randbits

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SECPAR, Q, L, D, SK_BD, CH_WT = 128, 11777, 13, 256, 45, 20
VF_BD = SK_BD * (1 + CH_WT)


def _sign_pool(eng, sch, n, tag):
    seeds = [bin((0x9E3779B97F4A7C15 * (i + 7)) % (1 << eng.secpar))[2:].zfill(eng.secpar) for i in range(n)]
    chm = [f'<key {tag} {i}>, ' + format(i * 2654435761 % (1 << 32), '032b') for i in range(n)]
    _, sk_ntt, vk_ntt, _ = eng.lm_keygen(sch, seeds, want_sk_coef=False, want_vk_coef=False)
    return vk_ntt, chm, eng.lm_sign(sch, sk_ntt, chm)


def _messages(n_agg, seed, lens=None):
    rng = np.random.default_rng(seed)
    if lens is None:
        lens = rng.integers(0, 300, n_agg)
    return [bytes(rng.integers(32, 127, int(m), dtype=np.uint8)) for m in lens]


def _single_aggregate(eng, sch, sigs, off, msgs):
    out = []
    for g in range(len(msgs)):
        a, b = int(off[g]), int(off[g + 1])
        ag = eng.agg_coefs(sch, msgs[g], 0, b - a)
        out.append(eng.aggregate_finish(eng.aggregate_partial(sch, np.ascontiguousarray(sigs[a:b]), ag)))
    return np.stack(out)


def _single_verify(eng, sch, vk, chm, off, msgs, ag_sig, cap, bd, wt):
    out = []
    for g in range(len(msgs)):
        a, b = int(off[g]), int(off[g + 1])
        ag = eng.agg_coefs(sch, msgs[g], 0, b - a)
        part = eng.aggverify_partial(sch, np.ascontiguousarray(vk[a:b]), chm[a:b], ag)
        out.append(eng.aggverify_finish(part, np.ascontiguousarray(ag_sig[g]), b - a, cap, bd, wt))
    return np.array(out, dtype=np.uint8)


def _offsets(sizes):
    return np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)


@pytest.fixture(scope='module')
def world():
    from lattice_cryptography_b200 import Engine, make_scheme
    eng = Engine(SECPAR, Q, D, L)
    sch = make_scheme(sk_bd=SK_BD, sk_wt=D, ch_bd=1, ch_wt=CH_WT)
    key_ch, _ = eng.hash2polyvec('KEY_CH_SEED', ['bklm batch'], Q // 2, D, L)
    eng.set_key_ch(np.ascontiguousarray(key_ch[0]))
    vk, chm, sigs = _sign_pool(eng, sch, 8000, 'w')
    yield dict(eng=eng, sch=sch, key_ch=np.ascontiguousarray(key_ch[0]), vk=vk, chm=chm, sigs=sigs)
    eng.close()


def _edge_batch(lead):
    """Group sizes whose local index crosses 9 -> 10, 99 -> 100 and 999 -> 1000, messages whose first sponge input
    salt + str(j) + agmsg is 135, 136 or 137 bytes long, and a run of groups of 3 after a leading group of `lead`, so that
    every range boundary of the segmented kernels lies strictly inside a group in two of the three variants."""
    sizes = [lead, 1, 2, 3, 17, 255, 1100] + [3] * 400 + [1, 2, 64, 5]
    lens = [127, 128, 129] + [8 + (7 * g) % 400 for g in range(len(sizes) - 3)]
    return sizes, _messages(len(sizes), lead, lens)


@pytest.mark.parametrize('lead', [1, 2, 3])
def test_edge_batch_equals_single_path(world, lead):
    eng, sch, sigs, vk, chm = world['eng'], world['sch'], world['sigs'], world['vk'], world['chm']
    sizes, msgs = _edge_batch(lead)
    off = _offsets(sizes)
    n = int(off[-1])
    got = eng.aggregate_batch(sch, off, np.ascontiguousarray(sigs[:n]), msgs)
    want = _single_aggregate(eng, sch, sigs, off, msgs)
    assert np.array_equal(got, want)
    bd, cap = Q // 2, 1 << 20
    v = eng.aggregate_verify_batch(sch, off, np.ascontiguousarray(vk[:n]), chm[:n], msgs, got, cap, bd, D)
    assert v.tolist() == [1] * len(sizes)
    assert np.array_equal(v, _single_verify(eng, sch, vk, chm, off, msgs, got, cap, bd, D))


def test_batch_matches_hashlib_and_numpy(world):
    eng, sch, sigs = world['eng'], world['sch'], world['sigs']
    rng = np.random.default_rng(5)
    sizes = rng.integers(1, 6, 2400)
    off = _offsets(sizes)
    n = int(off[-1])
    msgs = _messages(len(sizes), 6)
    got = eng.aggregate_batch(sch, off, np.ascontiguousarray(sigs[:n]), msgs).astype(np.int64)
    ks, ss = np.zeros(n, np.int64), np.zeros(n, np.int64)
    for g, m in enumerate(msgs):
        for j in range(int(sizes[g])):
            dg = hashlib.shake_256(b'AG_SALT' + str(j).encode() + m).digest(2)
            ks[off[g] + j], ss[off[g] + j] = dg[0], (1 if dg[1] & 0x80 else -1)
    p = np.arange(D)
    want = np.zeros((len(sizes), L, D), np.int64)
    for a in range(0, n, 1024):
        b = min(a + 1024, n)
        k = ks[a:b, None]
        src = (p[None, :] - k) & (D - 1)
        sign = np.where(p[None, :] < k, -1, 1) * ss[a:b, None]
        rot = np.take_along_axis(sigs[a:b].astype(np.int64), np.broadcast_to(src[:, None, :], (b - a, L, D)), axis=2)
        np.add.at(want, np.searchsorted(off, np.arange(a, b), side='right') - 1, rot * sign[:, None, :])
    want %= Q
    want = np.where(want > Q // 2, want - Q, want)
    assert np.array_equal(got, want)


def _crafted(world, zs, msgs):
    """One-signature groups whose aggregate is the chosen vector z: vk_left = 0 and vk_right = (key_ch . z) * a^-1 for
    the group's coefficient a = s X^k, so that key_ch . z == (vk_left c + vk_right) a holds exactly."""
    eng, sch, key_ch = world['eng'], world['sch'], world['key_ch']
    vks = []
    for z, m in zip(zs, msgs):
        y = eng.poly_mul(key_ch, z).astype(np.int64).sum(axis=0) % Q
        k, s = (int(x) for x in eng.agg_coefs(sch, m, 0, 1)[0, 0])
        inv = np.zeros(D, np.int16)
        if k == 0:
            inv[0] = s
        else:
            inv[D - k] = -s
        yc = np.where(y > Q // 2, y - Q, y).astype(np.int16)
        right = eng.poly_mul(yc[None], inv[None])[0]
        vks.append(np.stack([np.zeros(D, np.uint16), eng.ntt_fwd(right[None])[0]]))
    return np.ascontiguousarray(np.stack(vks))


def test_verdicts_reject_each_tamper_alone(world):
    eng, sch, sigs, vk, chm = world['eng'], world['sch'], world['sigs'], world['vk'], world['chm']
    sizes = [2, 3, 1, 2, 2, 2, 3, 2, 2]
    off = _offsets(sizes)
    n = int(off[-1])
    msgs = _messages(len(sizes), 11)
    vk_s, chm_s = np.ascontiguousarray(vk[:n]), list(chm[:n])
    ag = eng.aggregate_batch(sch, off, np.ascontiguousarray(sigs[:n]), msgs)
    bd, cap = Q // 2, 3
    args = (sch, off, vk_s, chm_s, msgs)
    assert eng.aggregate_verify_batch(*args, ag, cap, bd, D).tolist() == [1] * len(sizes)
    cases = []
    t = ag.copy(); t[[0, 3]] = t[[3, 0]]; cases.append((t, chm_s, msgs, {0, 3}))                       # swapped aggregates
    c2 = list(chm_s); c2[int(off[1]) + 1] += '0'; cases.append((ag, c2, msgs, {1}))                     # a signed message
    t = ag.copy(); t[2] = 0; cases.append((t, chm_s, msgs, {2}))                                        # all-zero aggregate
    t = ag.copy(); t[4, 5, 9] = bd + 1; cases.append((t, chm_s, msgs, {4}))                             # above avf_bd
    m2 = list(msgs); m2[5] = m2[5] + b'x'; cases.append((ag, chm_s, m2, {5}))                           # aggregation message
    for t, c, m, bad in cases:
        v = eng.aggregate_verify_batch(sch, off, vk_s, c, m, t, cap, bd, D)
        assert v.tolist() == [0 if g in bad else 1 for g in range(len(sizes))], bad
        assert np.array_equal(v, _single_verify(eng, sch, vk_s, c, off, m, t, cap, bd, D))
    # above ag_cap, and an empty group
    big = _offsets([2, 4, 0, 1])
    nb = int(big[-1])
    mb = _messages(4, 12)
    agb = eng.aggregate_batch(sch, _offsets([2, 4, 1]), np.ascontiguousarray(sigs[:nb]), [mb[0], mb[1], mb[3]])
    agb = np.ascontiguousarray(agb[[0, 1, 0, 2]])
    v = eng.aggregate_verify_batch(sch, big, np.ascontiguousarray(vk[:nb]), chm[:nb], mb, agb, cap, bd, D)
    assert v.tolist() == [1, 0, 0, 1]
    assert np.array_equal(v, _single_verify(eng, sch, vk, chm, big, mb, agb, cap, bd, D))
    # row weight above avf_wt and coefficient at the bound, on crafted low-weight aggregates
    rng = np.random.default_rng(13)
    zs = []
    for w, top in ((10, 7), (11, 7), (10, 8), (10, 7)):
        z = np.zeros((L, D), np.int16)
        for i in range(L):
            pos = rng.choice(D, w, replace=False)
            z[i, pos] = rng.choice(np.array([-1, 1], np.int16), w)
        z[3, int(np.flatnonzero(z[3])[0])] = top
        zs.append(z)
    zs = np.ascontiguousarray(np.stack(zs))
    mz = _messages(4, 14)
    vkz = _crafted(world, zs, mz)
    chz = [f'crafted {g}' for g in range(4)]
    v = eng.aggregate_verify_batch(sch, _offsets([1] * 4), vkz, chz, mz, zs, cap, 7, 10)
    assert v.tolist() == [1, 0, 0, 1]
    assert np.array_equal(v, _single_verify(eng, sch, vkz, chz, _offsets([1] * 4), mz, zs, cap, 7, 10))


def test_device_buffers_and_empty_batches(world):
    import torch
    from lattice_cryptography_b200 import _ffi, ragged
    eng, sch, sigs, vk, chm = world['eng'], world['sch'], world['sigs'], world['vk'], world['chm']
    sizes = [1, 5, 2, 40, 3]
    off = _offsets(sizes)
    n = int(off[-1])
    msgs = _messages(len(sizes), 21)
    host = eng.aggregate_batch(sch, off, np.ascontiguousarray(sigs[:n]), msgs)
    dev = lambda x: torch.from_numpy(np.array(x)).cuda()
    mblob, moff = ragged(msgs)
    cblob, coff = ragged(chm[:n])
    d_off, d_sig, d_mb, d_mo, d_vk, d_cb, d_co = (dev(x) for x in (off, sigs[:n], mblob, moff, vk[:n], cblob, coff))
    torch.cuda.synchronize()                  # the engine runs on its own stream: inputs first, outputs after eng.synchronize()
    got = eng.aggregate_batch(sch, d_off, d_sig, (d_mb, d_mo), device=True)
    eng.synchronize()
    assert np.array_equal(got.cpu().numpy(), host)
    vh = eng.aggregate_verify_batch(sch, off, np.ascontiguousarray(vk[:n]), chm[:n], msgs, host, 1 << 20, Q // 2, D)
    vd = eng.aggregate_verify_batch(sch, d_off, d_vk, (d_cb, d_co), (d_mb, d_mo), got, 1 << 20, Q // 2, D, device=True)
    eng.synchronize()
    assert vh.tolist() == [1] * len(sizes) and np.array_equal(vd.cpu().numpy(), vh)
    z = np.zeros(1, np.int64)
    lib = _ffi.load()
    from ctypes import byref, c_void_p
    assert lib.lcb_bklm_aggregate_batch(eng._ctx, byref(sch), c_void_p(z.ctypes.data), 0, None, None,
                                        c_void_p(z.ctypes.data), None) == _ffi.LCB_OK
    assert lib.lcb_bklm_aggregate_verify_batch(eng._ctx, byref(sch), c_void_p(z.ctypes.data), 0, None, None,
                                               c_void_p(z.ctypes.data), None, c_void_p(z.ctypes.data), None, 2, 1, 1,
                                               None) == _ffi.LCB_OK
    assert eng.aggregate_batch(sch, z, np.zeros((0, L, D), np.int16), []).shape == (0, L, D)


def test_invalid_host_offsets(world):
    from lattice_cryptography_b200 import LcbError, _ffi
    eng, sch, sigs, vk, chm = world['eng'], world['sch'], world['sigs'], world['vk'], world['chm']
    s = np.ascontiguousarray(sigs[:6])
    for off in ([0, 4, 2, 6], [1, 3, 6], [0, 3, 3, 6]):                # non-monotone, not at 0, an empty group
        with pytest.raises(LcbError) as e:
            eng.aggregate_batch(sch, np.array(off, np.int64), s, _messages(len(off) - 1, 3))
        assert e.value.status == _ffi.LCB_ERR_INVALID, off
    ag = np.zeros((3, L, D), np.int16)
    for off in ([0, 4, 2, 6], [1, 3, 6, 6]):
        with pytest.raises(LcbError) as e:
            eng.aggregate_verify_batch(sch, np.array(off, np.int64), np.ascontiguousarray(vk[:6]), chm[:6],
                                       _messages(len(off) - 1, 3), ag[:len(off) - 1], 2, Q // 2, D)
        assert e.value.status == _ffi.LCB_ERR_INVALID, off


def test_partial_sums_at_the_largest_16_bit_prime():
    """One group of 2^14 signatures next to 10,000 groups of two at q = 64513: centred coefficients up to 32,256 in
    magnitude, the case in which the int32 partial sums come closest to their bound."""
    from lattice_cryptography_b200 import Engine, make_scheme
    q, l = 64513, 2
    eng = Engine(SECPAR, q, D, l)
    try:
        sch = make_scheme(sk_bd=q // 2, sk_wt=D, ch_bd=1, ch_wt=CH_WT)
        key_ch, _ = eng.hash2polyvec('KEY_CH_SEED', ['bklm batch extremes'], q // 2, D, l)
        eng.set_key_ch(np.ascontiguousarray(key_ch[0]))
        sizes = [1 << 14] + [2] * 10000
        off = _offsets(sizes)
        vk, chm, sigs = _sign_pool(eng, sch, int(off[-1]), 'x')
        assert int(np.abs(sigs.astype(np.int64)).max()) > 32000
        msgs = _messages(len(sizes), 31)
        got = eng.aggregate_batch(sch, off, sigs, msgs)
        assert np.array_equal(got, _single_aggregate(eng, sch, sigs, off, msgs))
        v = eng.aggregate_verify_batch(sch, off, vk, chm, msgs, got, 1 << 20, q // 2, D)
        assert v.tolist() == [1] * len(sizes)
        sub = _offsets([1 << 14, 2, 2])
        assert np.array_equal(v[:3], _single_verify(eng, sch, vk, chm, sub, msgs[:3], got[:3], 1 << 20, q // 2, D))
    finally:
        eng.close()


@pytest.mark.parametrize('secpar,q,d,l,ag_wt,ag_bd', [(128, 12289, 512, 2, 1, 1), (128, Q, D, L, 2, 1)])
def test_other_parameter_sets_equal_single_path(secpar, q, d, l, ag_wt, ag_bd):
    from lattice_cryptography_b200 import Engine, make_scheme
    eng = Engine(secpar, q, d, l)
    try:
        sk_bd, ch_wt = (2, 5) if d != D else (SK_BD, CH_WT)
        sch = make_scheme(sk_bd=sk_bd, sk_wt=d, ch_bd=1, ch_wt=ch_wt, ag_bd=ag_bd, ag_wt=ag_wt)
        key_ch, _ = eng.hash2polyvec('KEY_CH_SEED', ['bklm batch generic'], q // 2, d, l)
        eng.set_key_ch(np.ascontiguousarray(key_ch[0]))
        sizes = [1, 3, 2, 12, 1]
        off = _offsets(sizes)
        vk, chm, sigs = _sign_pool(eng, sch, int(off[-1]), 'g')
        msgs = _messages(len(sizes), 41)
        got = eng.aggregate_batch(sch, off, sigs, msgs)
        assert np.array_equal(got, _single_aggregate(eng, sch, sigs, off, msgs))
        bd, cap = q // 2, 64
        v = eng.aggregate_verify_batch(sch, off, vk, chm, msgs, got, cap, bd, d)
        assert v.tolist() == [1] * len(sizes)
        t = got.copy()
        t[2, 0, 1] += 1
        v2 = eng.aggregate_verify_batch(sch, off, vk, chm, msgs, t, cap, bd, d)
        assert v2.tolist() == [1, 1, 0, 1, 1]
        assert np.array_equal(v2, _single_verify(eng, sch, vk, chm, off, msgs, t, cap, bd, d))
    finally:
        eng.close()


@pytest.mark.parametrize('mode', ['reference', 'tree'])
def test_dropin_batch_equals_per_group_calls(mode):
    from lattice_cryptography_b200 import bklm_one_time_agg_sigs as bk
    from lattice_cryptography_b200.lm_one_time_sigs import keygen, sign
    pp = bk.set_aggregation_mode(bk.make_setup_parameters(SECPAR), mode)
    keys = keygen(pp=pp, num_keys_to_gen=12)
    msgs = [bin(randbits(32))[2:].zfill(32) for _ in keys]
    sigs = [sign(pp=pp, otk=k, msg=m) for k, m in zip(keys, msgs)]
    vks = [k[2] for k in keys]
    cuts = [(0, 2), (2, 3), (3, 5), (5, 7), (7, 10), (10, 12)]
    gk, gm, gs = ([x[a:b] for a, b in cuts] for x in (vks, msgs, sigs))
    gk, gm, gs = gk[:4] + gk[5:], gm[:4] + gm[5:], gs[:4] + gs[5:]      # every group within ag_cap = 2
    ags = bk.aggregate_batch(pp, gk, gm, gs)
    for g in range(len(gk)):
        assert np.array_equal(ags[g].coef, bk.aggregate(pp, gk[g], gm[g], gs[g]).coef)
    ags[2].coef[0, 0] += 1                                            # a tampered aggregate
    vk_over, m_over = vks[7:10], msgs[7:10]                            # three signatures: above ag_cap
    from lattice_cryptography_b200.lattice_algebra import PolynomialVector
    short = PolynomialVector(pp['scheme_parameters'].lp, const_time_flag=False, _coef=ags[0].coef[:3])     # ill-formed
    otv = gk + [vk_over, gk[0], gk[0]]
    otm = gm + [m_over, gm[0], gm[0][:1]]                             # the last: length mismatch
    oag = ags + [ags[0], short, ags[0]]
    want = [bk.aggregate_verify(pp, k, m, a) for k, m, a in zip(otv, otm, oag)]
    assert want == [True, True, False, True, True, False, False, False]
    assert bk.aggregate_verify_batch(pp, otv, otm, oag) == want
    bad = [gm[0][0][:-1] + '2', gm[0][1]]
    with pytest.raises(ValueError, match='bitstrings'):
        bk.aggregate(pp, gk[0], bad, gs[0])
    with pytest.raises(ValueError, match='bitstrings'):
        bk.aggregate_batch(pp, [gk[1], gk[0]], [gm[1], bad], [gs[1], gs[0]])
    with pytest.raises(ValueError, match='bitstrings'):
        bk.aggregate_verify_batch(pp, [gk[0]], [bad], [ags[0]])


# ---- the checked build and guard bands (tests/test_gpu_checked.py does the same for the other entry points) ----
def test_batch_outputs_stay_inside_their_buffers(world):
    import torch
    eng, sch, sigs, vk, chm = world['eng'], world['sch'], world['sigs'], world['vk'], world['chm']
    pad = 4096
    for sizes in ([1], [3, 1, 2], [17, 1, 2, 5]):
        off = _offsets(sizes)
        n = int(off[-1])
        msgs = _messages(len(sizes), len(sizes))
        raw_a = torch.full((2 * pad + len(sizes) * L * D * 2,), 0xA5, dtype=torch.uint8, device='cuda')
        raw_v = torch.full((2 * pad + len(sizes),), 0xA5, dtype=torch.uint8, device='cuda')
        ag = raw_a[pad:pad + len(sizes) * L * D * 2].view(torch.int16).view(len(sizes), L, D)
        ver = raw_v[pad:pad + len(sizes)]
        dev = lambda x: torch.from_numpy(np.array(x)).cuda()
        from lattice_cryptography_b200 import ragged
        mb, mo = ragged(msgs)
        cb, co = ragged(chm[:n])
        d_off, d_sig, d_mb, d_mo, d_vk, d_cb, d_co = (dev(x) for x in (off, sigs[:n], mb, mo, vk[:n], cb, co))
        torch.cuda.synchronize()              # bands and inputs are written on torch's stream, the engine has its own
        eng._ck(eng._lib.lcb_bklm_aggregate_batch(eng._ctx, _byref(sch), _p(d_off), len(sizes), _p(d_sig), _p(d_mb),
                                                  _p(d_mo), _p(ag)))
        eng._ck(eng._lib.lcb_bklm_aggregate_verify_batch(eng._ctx, _byref(sch), _p(d_off), len(sizes), _p(d_vk), _p(d_cb),
                                                         _p(d_co), _p(d_mb), _p(d_mo), _p(ag), 1 << 20, Q // 2, D, _p(ver)))
        eng.synchronize()
        assert ver.cpu().tolist() == [1] * len(sizes)
        for raw, body in ((raw_a, len(sizes) * L * D * 2), (raw_v, len(sizes))):
            assert bool((raw[:pad] == 0xA5).all().item()) and bool((raw[pad + body:] == 0xA5).all().item()), sizes


def _p(t):
    from ctypes import c_void_p
    return c_void_p(t.data_ptr())


def _byref(s):
    from ctypes import byref
    return byref(s)


def test_edge_cases_pass_on_the_checked_build():
    from lattice_cryptography_b200 import _ffi
    if _ffi.load().lcb_build_is_checked():
        pytest.skip('already running on the checked build')
    lib = os.path.join(ROOT, 'lattice_cryptography_b200', 'liblcb200_checked.so')
    if not os.path.exists(lib):
        subprocess.run(['make', '-C', os.path.join(ROOT, 'lattice_cryptography_b200', 'csrc'), '-j4', 'CHECKED=1'], check=True,
                       capture_output=True)
    env = dict(os.environ, LCB200_LIB=lib)
    r = subprocess.run([sys.executable, '-m', 'pytest', 'tests/test_gpu_bklm_batch.py', '-q', '-x', '-m', 'gpu', '-k',
                        'edge_batch or device_buffers or other_parameter or stay_inside', '-p', 'no:cacheprovider'],
                       env=env, capture_output=True, text=True, timeout=1500, cwd=ROOT)
    tail = r.stdout[-2500:] + r.stderr[-1500:]
    assert r.returncode == 0, tail
    assert ' passed' in r.stdout and 'failed' not in r.stdout, tail
