"""Batched BKLM aggregate / aggregate-verify, unpacked and on the packed wire format, against a reference that does not
run on the engine, at worst-case magnitudes and at every verdict boundary.

The reference: aggregation coefficients from hashlib (k = byte 0 of shake_256(ag_salt || str(j) || agmsg_g), sign = top
bit of byte 1), aggregates as numpy negacyclic rotations summed in int64, packing by oracle/wire.py, NTT images of
monomials from the least primitive 512-th root of unity (slot p of s X^k is s psi^((2 bitrev8(p) + 1) k)), and verdicts
as a numpy statement of the rules (1 <= max|coef| <= avf_bd, row weights <= avf_wt, 1 <= count <= ag_cap, equation).
Inputs are built so that the equation holds exactly (the last item's vk_right is solved for it), so that each rule
decides on its own.  ntt_fwd / poly_mul only build inputs; other tests pin them against the oracle.

LCB_SEG_RANGES caps the ranges per polynomial of the segmented kernels: it lets a few hundred MB reach ranges of more
than 2^16 rows (the in-register reduction of k_agg_partial_seg) and long half-warp ranges of k_aggv_partial_seg."""
import hashlib
import os
import subprocess
import sys

import numpy as np
import pytest

import wire as owire

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
D = 256
AGG_DEPTH = 4                                   # rows in flight per warp of k_agg_partial_seg (ring.cu)
BR8 = np.array([int(format(p, '08b')[::-1], 2) for p in range(D)], np.int64)


# ---------------------------------------------------------------- the reference
def _offsets(sizes):
    return np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)


def _messages(n, seed):
    rng = np.random.default_rng(seed)
    return [bytes(rng.integers(32, 127, int(m), dtype=np.uint8)) for m in rng.integers(0, 300, n)]


def _coefs(sizes, msgs):
    """(k, s) of every item: item j of group g hashes b'AG_SALT' + str(j) + msgs[g]."""
    ks, ss = [], []
    for size, m in zip(sizes, msgs):
        for j in range(int(size)):
            dg = hashlib.shake_256(b'AG_SALT' + str(j).encode() + m).digest(2)
            ks.append(dg[0])
            ss.append(1 if dg[1] & 0x80 else -1)
    return np.array(ks, np.int64), np.array(ss, np.int64)


def _centre(x, q):
    x = np.asarray(x, np.int64) % q
    return np.where(x > q // 2, x - q, x)


def _unrotate(t, k, s):
    """s X^(-k) t for each item (t [n, l, D] or [l, D], k / s [n]): s X^k times the result is t."""
    p = np.arange(D)
    src = (p[None, :] + k[:, None]) % D
    sign = np.where(p[None, :] + k[:, None] >= D, -1, 1) * s[:, None]
    t = np.broadcast_to(t, (len(k),) + t.shape[-2:])
    return np.take_along_axis(t, np.broadcast_to(src[:, None, :], t.shape), axis=2) * sign[:, None, :]


def _aggregate(sigs, off, ks, ss, q):
    """sum over the items of group g of s X^k sig, in int64, reduced mod q and centred."""
    n, l = sigs.shape[0], sigs.shape[1]
    want = np.zeros((len(off) - 1, l, D), np.int64)
    grp = np.searchsorted(off, np.arange(n), side='right') - 1
    p = np.arange(D)
    for a in range(0, n, 2048):
        b = min(a + 2048, n)
        k = ks[a:b, None]
        src = (p[None, :] - k) & (D - 1)
        sign = np.where(p[None, :] < k, -1, 1) * ss[a:b, None]
        rot = np.take_along_axis(sigs[a:b].astype(np.int64), np.broadcast_to(src[:, None, :], (b - a, l, D)), axis=2)
        np.add.at(want, grp[a:b], rot * sign[:, None, :])
    return _centre(want, q)


def _psi_powers(q):
    """psi^t mod q for t = 0 .. 511, psi the least primitive 512-th root of unity."""
    psi = next(g for g in range(2, q) if pow(g, 256, q) == q - 1)
    return np.array([pow(psi, t, q) for t in range(512)], np.int64)


def _mono_ntt(pw, k, s, q, inverse=False):
    """NTT images [n, D] of s X^k (or of its inverse s X^-k)."""
    e = (2 * BR8 + 1)[None, :] * k[:, None] * (-1 if inverse else 1)
    return (s[:, None] * pw[e % 512]) % q


def _rules(z, counts, cap, bd, wt):
    z = z.astype(np.int64)
    mx = np.abs(z).max(axis=(1, 2))
    rw = (z != 0).sum(axis=2).max(axis=1)
    return ((mx >= 1) & (mx <= bd) & (rw <= wt) & (counts >= 1) & (counts <= cap)).astype(np.uint8)


def _patterns(rng, shape, v):
    alt = np.where(np.arange(shape[-1]) % 2 == 0, v, -v)
    return [('all_plus', np.full(shape, v, np.int64)), ('all_minus', np.full(shape, -v, np.int64)),
            ('alternating', np.broadcast_to(alt, shape).astype(np.int64)),
            ('random_signs', rng.choice(np.array([-v, v], np.int64), shape))]


def _engine(secpar, q, l, ch_wt=20):
    from lattice_cryptography_b200 import Engine, make_scheme
    return Engine(secpar, q, D, l), make_scheme(sk_bd=1, sk_wt=D, ch_bd=1, ch_wt=ch_wt)


def _misaligned(x):
    """A device copy of x that is 4-byte but not 16-byte aligned."""
    import torch
    flat = torch.from_numpy(np.ascontiguousarray(x).reshape(-1)).cuda()
    raw = torch.zeros(flat.numel() + 16, dtype=torch.uint8, device='cuda')
    view = raw[4:4 + flat.numel()]
    view.copy_(flat)
    torch.cuda.synchronize()
    assert view.data_ptr() % 16 == 4
    return view.view(*x.shape)


# ---------------------------------------------------------------- A1: worst-case aggregate growth
def _coherent(rng, q, l, v, counts, extra=()):
    """Groups whose items all add exactly the same target T (sig = s^-1 X^-k T): the aggregate is count T mod q.
    `extra` appends groups of arbitrary rows (list of [count, l, D] arrays)."""
    groups = []
    for (name, t), c in zip(_patterns(rng, (l, D), v), counts):
        groups.append((t, c))
    sizes = [c for _, c in groups] + [len(x) for x in extra]
    msgs = _messages(len(sizes), int(rng.integers(1 << 30)))
    ks, ss = _coefs(sizes, msgs)
    off = _offsets(sizes)
    sigs = np.empty((int(off[-1]), l, D), np.int64)
    for g, (t, c) in enumerate(groups):
        sigs[off[g]:off[g + 1]] = _unrotate(t, ks[off[g]:off[g + 1]], ss[off[g]:off[g + 1]])
    for g, x in enumerate(extra, start=len(groups)):
        sigs[off[g]:off[g + 1]] = x
    closed = np.stack([_centre(c * t, q) for t, c in groups]) if groups else None
    return off, msgs, ks, ss, sigs.astype(np.int16), closed


def _end_rows(rng, l, lo, hi):
    """Rows at both ends of a packed width: all lo, all hi, alternating, and random choices of the two."""
    alt = np.where(np.arange(D) % 2 == 0, lo, hi)
    return [np.full((3, l, D), lo), np.full((2, l, D), hi), np.broadcast_to(alt, (5, l, D)).copy(),
            rng.choice(np.array([lo, hi]), (17, l, D))]


@pytest.mark.parametrize('l', [1, 13, 64])
@pytest.mark.parametrize('q', [7681, 11777, 39937, 64513])
def test_worst_case_growth(q, l):
    """Every item of a group adds the same target T (+-v everywhere, alternating, random signs; v = q//2, 32767 and the
    extremes of the packed widths), so the sums grow like count * T; the all-minus group of 2^16 / l items spreads over
    hundreds of warp ranges, so its partial sum is far below -2^20 (the x + off argument of k_agg_finish_pack).  Checked
    on aggregate_batch, on the fused packed route (11 / 13 bits, biases whose decoded values reach both ends of the
    width) and on the unpack-first route (12 bits; 13 bits from a 4-byte aligned device buffer)."""
    eng, sch = _engine(128, q, l)
    rng = np.random.default_rng(q * 100 + l)
    big = (1 << 16) // l
    counts = [3, big, 255, 1000 // l + 2]            # all_plus, all_minus, alternating, random_signs
    try:
        for v in (q // 2, 32767):
            off, msgs, ks, ss, sigs, closed = _coherent(rng, q, l, v, counts)
            want = _aggregate(sigs, off, ks, ss, q)
            assert np.array_equal(want, closed)
            assert np.array_equal(eng.aggregate_batch(sch, off, sigs, msgs), want), v
        # packed: (bits, bias, route); the coherent magnitude is the largest +-m the width holds
        for sb, sbias, route in ((11, 1023, 'fused'), (13, 4095, 'fused'), (13, 32767, 'fused'), (12, 2047, 'first'),
                                 (13, 4096, 'device')):
            lo, hi = -sbias, (1 << sb) - 1 - sbias
            m = min(sbias, hi)
            off, msgs, ks, ss, sigs, closed = _coherent(rng, q, l, m, counts if m > 0 else [], _end_rows(rng, l, lo, hi))
            want = _aggregate(sigs, off, ks, ss, q)
            if closed is not None:
                assert np.array_equal(want[:len(closed)], closed)
            sigp, ok = eng.pack(sigs, sb, sbias, want_range=True)
            assert ok.all() and sigs.min() == lo and sigs.max() == hi
            for ab, abias in ((16, 32767), (12, 2047)):
                want_p, want_ok = owire.pack(want.astype(np.int16), ab, abias)
                if route == 'device':
                    got = eng.aggregate_packed_batch(sch, off, _misaligned(sigp), sb, sbias, msgs, ab, abias, device=True,
                                                     want_range=True)
                    eng.synchronize()
                    got = tuple(x.cpu().numpy() for x in got)
                else:
                    got = eng.aggregate_packed_batch(sch, off, sigp, sb, sbias, msgs, ab, abias, want_range=True)
                assert np.array_equal(got[0], want_p) and np.array_equal(got[1], want_ok), (sb, sbias, route, ab)
    finally:
        eng.close()


# ---------------------------------------------------------------- A2: ranges longer than 2^16 rows
def test_long_segment_ranges(monkeypatch):
    """q = 64513, l = 1, every row of a group adding +-q//2 to every slot: with LCB_SEG_RANGES=8 (one chunk) each warp
    walks 2^16 + 2^12 rows, whose coherent sum (2.25e9) exceeds int32 unless k_agg_partial_seg reduces in registers
    every 2^15 rows.  Then group boundaries 2^15 - 1, 2^15, 2^15 + 1 rows into a range, at every position mod AGG_DEPTH,
    at range starts and ends, and runs of one-row groups; the bytes must not depend on the range count."""
    q, l = 64513, 1
    eng, sch = _engine(128, q, l)
    rng = np.random.default_rng(64513)
    r = (1 << 16) + (1 << 12)                    # rows per range at 8 ranges
    try:
        def build(sizes):
            sizes = np.array(sizes, np.int64)
            assert int(sizes.sum()) == 8 * r
            msgs = _messages(len(sizes), int(sizes[0]))
            ks, ss = _coefs(sizes, msgs)
            off = _offsets(sizes)
            ts = rng.choice(np.array([-(q // 2), q // 2], np.int64), (len(sizes), l, D))
            ts[0] = q // 2
            sigs = np.empty((int(off[-1]), l, D), np.int16)
            for g in range(len(sizes)):
                sigs[off[g]:off[g + 1]] = _unrotate(ts[g], ks[off[g]:off[g + 1]], ss[off[g]:off[g + 1]])
            return off, msgs, sigs, _centre(sizes[:, None, None] * ts, q)

        monkeypatch.setenv('LCB_SEG_RANGES', '8')
        off, msgs, sigs, want = build([8 * r])
        assert np.array_equal(eng.aggregate_batch(sch, off, sigs, msgs), want)
        # the construction itself, on a sample of the rows: each adds q//2 to every slot
        sub = np.arange(0, 8 * r, 4099)
        ks, ss = _coefs([8 * r], msgs)
        rot = _aggregate(sigs[sub], np.array([0, len(sub)]), ks[sub], ss[sub], q)
        assert np.array_equal(rot[0], np.full((l, D), _centre(len(sub) * (q // 2), q)))
        del sigs
        cuts = [0, (1 << 15) - 1, r + (1 << 15), 2 * r + (1 << 15) + 1, 3 * r + (1 << 15) + 2, 4 * r, 4 * r + 1, 4 * r + 2,
                4 * r + 3, 4 * r + 4, 4 * r + 9, 5 * r - 1, 5 * r, 6 * r + 5, 6 * r + 6, 6 * r + 11, 7 * r + 100, 8 * r]
        assert {c % r % AGG_DEPTH for c in cuts[1:-1]} == set(range(AGG_DEPTH))
        off, msgs, sigs, want = build(np.diff(cuts))
        for knob in ('8', '64', None):
            if knob is None:
                monkeypatch.delenv('LCB_SEG_RANGES')
            else:
                monkeypatch.setenv('LCB_SEG_RANGES', knob)
            assert np.array_equal(eng.aggregate_batch(sch, off, sigs, msgs), want), knob
    finally:
        eng.close()


# ---------------------------------------------------------------- A3: each verdict rule on its own
def _verify_world(secpar):
    q, l, kb, ab, avf_bd, ch_wt = (11777, 13, 14, 12, 1890, 20) if secpar == 128 else (39937, 23, 16, 14, 6630, 50)
    eng, sch = _engine(secpar, q, l, ch_wt)
    rng = np.random.default_rng(secpar)
    key_ch = rng.integers(-(q // 2), q // 2 + 1, (l, D)).astype(np.int16)
    eng.set_key_ch(key_ch)
    return dict(eng=eng, sch=sch, q=q, l=l, kb=kb, ab=ab, avf_bd=avf_bd, pw=_psi_powers(q),
                key_hat=eng.ntt_fwd(key_ch).astype(np.int64))


def _challenge_ntt(w, chm):
    pairs = w['eng'].challenge(w['sch'], chm)
    dense = np.zeros((len(chm), D), np.int16)
    for i in range(len(chm)):
        dense[i, pairs[i, :, 0].astype(np.int64)] = pairs[i, :, 1]
    return w['eng'].ntt_fwd(dense).astype(np.int64)


def _solve_keys(w, sizes, msgs, zs, rng, zero_keys=()):
    """Keys such that key_ch . z_g == sum_i (vk_left_i c_i + vk_right_i) a_i holds in NTT form for every group: random
    slots for every item but the last of a group, whose vk_right is solved (vk_left = vk_right = 0 for the groups in
    zero_keys)."""
    q, eng = w['q'], w['eng']
    off = _offsets(sizes)
    n = int(off[-1])
    chm = [f'edge item {i} {rng.integers(1 << 30)}' for i in range(n)]
    ks, ss = _coefs(sizes, msgs)
    a_hat = _mono_ntt(w['pw'], ks, ss, q)
    c_hat = _challenge_ntt(w, chm) if n else np.zeros((0, D), np.int64)
    vk = rng.integers(0, q, (n, 2, D)).astype(np.int64)
    y = (w['key_hat'][None] * eng.ntt_fwd(np.ascontiguousarray(zs)).astype(np.int64)).sum(axis=1) % q
    for g in range(len(sizes)):
        a, b = int(off[g]), int(off[g + 1])
        if a == b:
            continue
        if g in zero_keys:
            vk[a:b] = 0
        rest = ((vk[a:b - 1, 0] * c_hat[a:b - 1] + vk[a:b - 1, 1]) % q * a_hat[a:b - 1]).sum(axis=0)
        inv = _mono_ntt(w['pw'], ks[b - 1:b], ss[b - 1:b], q, inverse=True)[0]
        vk[b - 1, 1] = ((y[g] - rest) % q * inv - vk[b - 1, 0] * c_hat[b - 1]) % q
        got = ((vk[a:b, 0] * c_hat[a:b] + vk[a:b, 1]) % q * a_hat[a:b]).sum(axis=0) % q
        assert np.array_equal(got, y[g])
    return off, chm, vk.astype(np.uint16)


def _single(w, off, vk, chm, msgs, zs, cap, bd, wt):
    eng, sch = w['eng'], w['sch']
    out = []
    for g in range(len(msgs)):
        a, b = int(off[g]), int(off[g + 1])
        ag = eng.agg_coefs(sch, msgs[g], 0, b - a)
        part = eng.aggverify_partial(sch, np.ascontiguousarray(vk[a:b]), chm[a:b], ag)
        out.append(eng.aggverify_finish(part, np.ascontiguousarray(zs[g]), b - a, cap, bd, wt))
    return np.array(out, np.uint8)


def _check_verdicts(w, sizes, zs, cap, bd, wt, rng, zero_keys=(), want=None):
    """Every route == the rules; packed routes only for the groups whose aggregate the width represents."""
    eng, sch, kb, ab = w['eng'], w['sch'], w['kb'], w['ab']
    sizes = np.array(sizes, np.int64)
    zs = np.ascontiguousarray(zs.astype(np.int16))
    msgs = _messages(len(sizes), int(rng.integers(1 << 30)))
    off, chm, vk = _solve_keys(w, sizes, msgs, zs, rng, zero_keys)
    rule = _rules(zs, sizes, cap, bd, wt)
    if want is not None:
        assert rule.tolist() == want
    got = eng.aggregate_verify_batch(sch, off, vk, chm, msgs, zs, cap, bd, wt)
    assert got.tolist() == rule.tolist(), 'batch'
    assert _single(w, off, vk, chm, msgs, zs, cap, bd, wt).tolist() == rule.tolist(), 'single'
    vkp, _ = owire.pack(vk, kb, 0)
    compared = 0
    for bits in (ab, 16):                         # the fused route, then the unpack-first route
        for bias in (w['avf_bd'], 0, 32767):
            agp, ok = owire.pack(zs, bits, bias)
            rep = ok.all(axis=1).astype(bool)
            v = eng.aggregate_verify_packed_batch(sch, off, vkp, kb, chm, msgs, agp, bits, bias, cap, bd, wt)
            assert v[rep].tolist() == rule[rep].tolist(), (bits, bias)
            compared += int(rep.sum())
    assert compared >= len(sizes)
    return rule


def _spike(w, rng, value, row, slot, nonneg):
    """An aggregate of small background coefficients (0 / 1, or -1 / 0 / 1) with one coefficient set to value."""
    z = rng.choice(np.array([0, 1] if nonneg else [-1, 0, 1]), (w['l'], D))
    z[row, slot] = value
    return z


@pytest.fixture(scope='module', params=[128, 256])
def vworld(request):
    w = _verify_world(request.param)
    yield w
    w['eng'].close()


def test_verdict_rules_each_decide_alone(vworld):
    w = vworld
    rng = np.random.default_rng(w['q'])
    l, bd, cap, wt = w['l'], w['avf_bd'], 2, D
    # bound: |coef| == avf_bd passes, avf_bd + 1 fails; both signs, first / last slot of the first / last row
    zs, sizes, want = [], [], []
    for value in (bd, bd + 1):
        for sign in (1, -1):
            for row in (0, l - 1):
                for slot in (0, D - 1):
                    zs.append(_spike(w, rng, sign * value, row, slot, sign > 0))
                    sizes.append(1 + (slot & 1))
                    want.append(int(value == bd))
    _check_verdicts(w, sizes, np.stack(zs), cap, bd, wt, rng, want=want)
    # weight: a row of weight exactly avf_wt passes, avf_wt + 1 fails (k_verify<true, ...>)
    for awt in (1, 10, 255):
        zs, want = [], []
        for extra, row in ((0, 0), (1, 0), (0, l - 1), (1, l - 1)):
            z = np.zeros((l, D), np.int64)
            for i in range(l):
                wi = awt + extra if i == row else int(rng.integers(1, awt + 1))
                z[i, rng.choice(D, wi, replace=False)] = rng.choice(np.array([-1, 1]), wi)
            zs.append(z)
            want.append(1 - extra)
        _check_verdicts(w, [1, 2, 2, 1], np.stack(zs), cap, bd, awt, rng, want=want)
    # zero aggregate: the equation and the bounds hold with keys all zero, only the lower limit rejects it; its twin
    # has a single non-zero coefficient in the last field of the last row
    zs = np.zeros((6, l, D), np.int64)
    zs[1, l - 1, D - 1], zs[3, l - 1, D - 1], zs[4, l - 1, D - 1] = 1, -bd, bd
    _check_verdicts(w, [1, 1, 2, 2, 1, 2], zs, cap, bd, wt, rng, zero_keys={0, 2, 5}, want=[0, 1, 0, 1, 1, 0])
    # count: ag_cap passes, ag_cap + 1 fails
    for c in (2, 3):
        zs = np.stack([_spike(w, rng, 5, 1, 7, False) for _ in range(4)])
        _check_verdicts(w, [c - 1, c, c + 1, c], zs, c, bd, wt, rng, want=[1, 1, 0, 1])
    # empty groups (zero aggregate): first, in the middle, last, and in runs
    sizes = [0, 2, 0, 0, 1, 0, 2, 0, 0, 0]
    zs = np.stack([np.zeros((l, D), np.int64) if s == 0 else _spike(w, rng, 3, 0, 0, False) for s in sizes])
    _check_verdicts(w, sizes, zs, cap, bd, wt, rng, want=[int(s > 0) for s in sizes])


def test_bound_clamp_at_int16_minimum(vworld):
    """A -32768 coefficient: avf_bd = 32767 rejects it, avf_bd >= 32768 accepts it (k_verify gets min(avf_bd, 32768))."""
    w = vworld
    rng = np.random.default_rng(7)
    zs = np.stack([_spike(w, rng, -32768, r, s, False) for r, s in ((0, 0), (w['l'] - 1, D - 1))])
    for bd, ok in ((32767, 0), (32768, 1), (40000, 1)):
        _check_verdicts(w, [1, 2], zs, 2, bd, D, rng, want=[ok, ok])


# ---------------------------------------------------------------- A4: aggregate-verify sums at extreme key slots
@pytest.mark.parametrize('q,secpar,l', [(11777, 128, 13), (39937, 256, 23), (64513, 128, 2)])
@pytest.mark.parametrize('knob', [None, '1', '5'])
def test_extreme_key_slots(q, secpar, l, knob, monkeypatch):
    """Groups of 1 .. 2^16 items whose key slots are all q - 1, all 0, mixed, or all 2^bits - 1 (>= q on 16-bit keys):
    a slot v acts as v mod q.  Most items have vk_left = 0 and share the group's vk_right pattern (their share of the
    right-hand side depends only on the (k, s) histogram); 200 items per large group carry extreme vk_left slots.  The
    equation holds (1), then fails after one slot changes by one (0), on the uint16, fused 14- / 16-bit and
    unpack-first routes; LCB_SEG_RANGES = 1 puts the whole batch in one half-warp range."""
    if knob is not None:
        monkeypatch.setenv('LCB_SEG_RANGES', knob)
    big = 1 << 16 if knob is None else 1 << 13
    eng, sch = _engine(secpar, q, l, 20 if secpar == 128 else 50)
    rng = np.random.default_rng(q + l)
    pw = _psi_powers(q)
    try:
        key_ch = rng.integers(-(q // 2), q // 2 + 1, (l, D)).astype(np.int16)
        eng.set_key_ch(key_ch)
        key_hat = eng.ntt_fwd(key_ch).astype(np.int64)
        sizes = np.array([1, 2, 3, 300, big, 17, 1000, 2], np.int64)
        off = _offsets(sizes)
        n = int(off[-1])
        msgs = _messages(len(sizes), q)
        ks, ss = _coefs(sizes, msgs)
        chm = [f'x{i}' for i in range(n)]
        zs = rng.choice(np.array([-3, -1, 1, 2]), (len(sizes), l, D)).astype(np.int16)
        y = (key_hat[None] * eng.ntt_fwd(zs).astype(np.int64)).sum(axis=1) % q
        grp = np.searchsorted(off, np.arange(n), side='right') - 1
        last = off[1:] - 1
        body = np.ones(n, bool)
        body[last] = False
        hist = np.zeros((len(sizes), D), np.int64)                     # sum of s per rotation k over the body items
        np.add.at(hist, (grp[body], ks[body]), ss[body])
        a_body = (hist @ pw[((2 * BR8 + 1)[None, :] * np.arange(D)[:, None]) % 512]) % q
        inv = _mono_ntt(pw, ks[last], ss[last], q, inverse=True)
        # (key bits, device): 16 / 14 bits from host memory take the fused route; 16 bits from a 4-byte aligned device
        # buffer and 15 bits take the unpack-first route
        routes = [(16, False), (16, True)] + [(kb, False) for kb in (14, 15) if q < (1 << kb)]
        for kb, device in routes:
            ab = 14 if kb != 14 else 12
            abias = (1 << (ab - 1)) - 1
            top = (1 << kb) - 1
            rights = np.stack([(np.full(D, q - 1), np.zeros(D, np.int64), rng.choice(np.array([0, q - 1]), D),
                                np.full(D, top))[g % 4] for g in range(len(sizes))])
            vk = np.zeros((n, 2, D), np.int64)
            vk[:, 1] = rights[grp]
            ext = np.concatenate([np.arange(a, min(b - 1, a + 200)) for a, b in zip(off[:-1], off[1:])]).astype(np.int64)
            vk[ext, 0] = np.stack([np.full(D, q - 1), np.full(D, top), rng.choice(np.array([0, q - 1, top]), D)])[ext % 3]
            pairs = eng.challenge(sch, [chm[i] for i in ext])
            dense = np.zeros((len(ext), D), np.int16)
            for j in range(len(ext)):
                dense[j, pairs[j, :, 0].astype(np.int64)] = pairs[j, :, 1]
            c_hat = eng.ntt_fwd(dense).astype(np.int64)
            # right-hand side of every item but the last: (vk_left c + vk_right) a with slots taken mod q
            rhs = a_body * (rights % q) % q
            np.add.at(rhs, grp[ext], (vk[ext, 0] % q) * c_hat % q * _mono_ntt(pw, ks[ext], ss[ext], q) % q)
            sol = (y - rhs) % q * inv % q
            up = (sol + q <= top) & (rng.random(sol.shape) < 0.5)          # v + q acts as v where the width has room
            vk[last, 0] = 0
            vk[last, 1] = np.where(up, sol + q, sol)
            vk = vk.astype(np.uint16)
            assert int(vk.max()) == top
            agp = owire.pack(zs, ab, abias)[0]
            # one slot changed by one in four groups: a body vk_right, an extreme vk_left, the solved slot, a pair's first
            bad = vk.copy()
            for i, half, p in ((int(off[3]) + 5, 1, 9), (int(off[4]) + 1, 0, 200), (int(last[6]), 1, 255), (int(off[1]), 1, 0)):
                bad[i, half, p] = bad[i, half, p] - 1 if bad[i, half, p] > 0 else 1
            for keys, want in ((vk, [1] * len(sizes)), (bad, [0 if g in (1, 3, 4, 6) else 1 for g in range(len(sizes))])):
                kp = eng.pack(keys, kb, 0)
                got = eng.aggregate_verify_packed_batch(sch, off, _misaligned(kp) if device else kp, kb, chm, msgs, agp, ab,
                                                        abias, 1 << 20, q // 2, D, device=device)
                if device:
                    eng.synchronize()
                    got = got.cpu().numpy()
                assert got.tolist() == want, (kb, device)
                if kb == 16:
                    assert eng.aggregate_verify_batch(sch, off, keys, chm, msgs, zs, 1 << 20, q // 2, D).tolist() == want
    finally:
        eng.close()


# ---------------------------------------------------------------- A5: the checked build
def test_edges_pass_on_the_checked_build():
    from lattice_cryptography_b200 import _ffi
    if _ffi.load().lcb_build_is_checked():
        pytest.skip('already running on the checked build')
    lib = os.path.join(ROOT, 'lattice_cryptography_b200', 'liblcb200_checked.so')
    if not os.path.exists(lib):
        subprocess.run(['make', '-C', os.path.join(ROOT, 'lattice_cryptography_b200', 'csrc'), '-j4', 'CHECKED=1'], check=True,
                       capture_output=True)
    env = dict(os.environ, LCB200_LIB=lib)
    r = subprocess.run([sys.executable, '-m', 'pytest', 'tests/test_gpu_bklm_edges.py', '-q', '-x', '-m', 'gpu', '-k',
                        '(worst_case_growth and 11777-13) or verdict_rules or (extreme_key_slots and 5-64513)',
                        '-p', 'no:cacheprovider'],
                       env=env, capture_output=True, text=True, timeout=1500, cwd=ROOT)
    tail = r.stdout[-2500:] + r.stderr[-1500:]
    assert r.returncode == 0, tail
    assert ' passed' in r.stdout and 'failed' not in r.stdout, tail
