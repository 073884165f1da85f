"""BKLM batch aggregate / aggregate-verify on the packed wire format (lcb_bklm_aggregate_packed_batch,
lcb_bklm_aggregate_verify_packed_batch, wire.aggregate_batch_packed / aggregate_verify_batch_packed).  Every result must
equal, bit for bit, unpack -> the unpacked batch call -> pack, for honest inputs, tampered ones and arbitrary bytes, on the
fused route (kernels read and write the packed rows) and on the unpack-first route alike."""
import os
import subprocess
import sys
from secrets import randbits

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
D = 256


def _offsets(sizes):
    return np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)


def _messages(n_agg, seed, lens=None):
    rng = np.random.default_rng(seed)
    if lens is None:
        lens = rng.integers(0, 300, n_agg)
    return [bytes(rng.integers(32, 127, int(m), dtype=np.uint8)) for m in lens]


@pytest.fixture(scope='module', params=[128, 256])
def world(request):
    from lattice_cryptography_b200 import bklm_one_time_agg_sigs as bk
    from lattice_cryptography_b200 import wire
    from lattice_cryptography_b200.lm_one_time_sigs import _ctx
    secpar = request.param
    pp = bk.make_setup_parameters(secpar)
    eng, sch = _ctx(pp)
    n = 2700
    seeds = [bin((0x9E3779B97F4A7C15 * (i + 11)) % (1 << secpar))[2:].zfill(secpar) for i in range(n)]
    chm = [f'<packed key {i}>, ' + format(i * 2654435761 % (1 << 32), '032b') for i in range(n)]
    _, sk_ntt, vk, _ = eng.lm_keygen(sch, seeds, want_sk_coef=False, want_vk_coef=False)
    sigs = eng.lm_sign(sch, sk_ntt, chm)
    w = dict(pp=pp, eng=eng, sch=sch, vk=vk, chm=chm, sigs=sigs, l=int(sigs.shape[1]), q=pp['scheme_parameters'].lp.modulus,
             sb=wire.sig_bits(pp), kb=wire.key_bits(pp), ab=wire.sig_bits(pp, 'avf_bd'), vf_bd=pp['vf_bd'], avf_bd=pp['avf_bd'],
             avf_wt=pp['avf_wt'], cap=pp['ag_cap'])
    assert (w['sb'], w['kb'], w['ab']) == ((11, 14, 12) if secpar == 128 else (13, 16, 14))
    w['sigp'] = eng.pack(sigs, w['sb'], w['vf_bd'])
    w['vkp'] = eng.pack(vk, w['kb'], 0)
    return w


def _ref_aggregate(w, off, sigp, msgs, sb, sbias, ab, abias, sch=None):
    eng = w['eng']
    ag = eng.aggregate_batch(sch or w['sch'], off, eng.unpack(sigp, sb, sbias), msgs)
    return eng.pack(ag, ab, abias, want_range=True)


def _ref_verify(w, off, vkp, kb, chm, msgs, agp, ab, abias, cap=None, sch=None):
    eng = w['eng']
    vk = eng.unpack(vkp, kb, 0, dtype=np.uint16)
    return eng.aggregate_verify_batch(sch or w['sch'], off, vk, chm, msgs, eng.unpack(agp, ab, abias),
                                      w['cap'] if cap is None else cap, w['avf_bd'], w['avf_wt'])


def _aggregate(w, off, sigp, msgs, sb=None, sbias=None, ab=None, abias=None, sch=None, **kw):
    pick = lambda x, default: default if x is None else x
    return w['eng'].aggregate_packed_batch(sch or w['sch'], off, sigp, pick(sb, w['sb']), pick(sbias, w['vf_bd']), msgs,
                                           pick(ab, w['ab']), pick(abias, w['avf_bd']), want_range=True, **kw)


def _verify(w, off, vkp, chm, msgs, agp, kb=None, ab=None, abias=None, cap=None, sch=None, **kw):
    pick = lambda x, default: default if x is None else x
    return w['eng'].aggregate_verify_packed_batch(sch or w['sch'], off, vkp, pick(kb, w['kb']), chm, msgs, agp, pick(ab, w['ab']),
                                                  pick(abias, w['avf_bd']), pick(cap, w['cap']), w['avf_bd'], w['avf_wt'], **kw)


def _check_both(w, off, msgs, cap=None):
    """aggregate + verify of the pool's first agg_off[-1] items against the unpacked calls; returns (agp, ok, verdict)."""
    n = int(off[-1])
    sigp, vkp, chm = np.ascontiguousarray(w['sigp'][:n]), np.ascontiguousarray(w['vkp'][:n]), w['chm'][:n]
    agp, ok = _aggregate(w, off, sigp, msgs)
    want_p, want_ok = _ref_aggregate(w, off, sigp, msgs, w['sb'], w['vf_bd'], w['ab'], w['avf_bd'])
    assert np.array_equal(agp, want_p) and np.array_equal(ok, want_ok)
    v = _verify(w, off, vkp, chm, msgs, agp, cap=cap)
    assert np.array_equal(v, _ref_verify(w, off, vkp, w['kb'], chm, msgs, agp, w['ab'], w['avf_bd'], cap=cap))
    return agp, ok, v


@pytest.mark.parametrize('lead', [1, 2, 3])
def test_edge_batch_equals_unpacked_calls(world, lead):
    """Group sizes whose local index crosses 9/99/999, 135/136/137-byte first sponge inputs, range boundaries of the
    segmented kernels inside groups (the groups of tests/test_gpu_bklm_batch.py::_edge_batch)."""
    sizes = [lead, 1, 2, 3, 17, 255, 1100] + [3] * 400 + [1, 2, 64, 5]
    lens = [127, 128, 129] + [8 + (7 * g) % 400 for g in range(len(sizes) - 3)]
    off = _offsets(sizes)
    _, ok, v = _check_both(world, off, _messages(len(sizes), lead, lens), cap=1 << 20)
    small = [g for g, s in enumerate(sizes) if s <= 2]
    assert ok[small].all() and v[small].all()


def test_tampers_flip_only_their_own_group(world):
    w = world
    eng, l, q, bd = w['eng'], w['l'], w['q'], w['avf_bd']
    sizes = [2, 1, 2, 2, 2, 2, 2, 2, 2]
    off = _offsets(sizes)
    n = int(off[-1])
    msgs = _messages(len(sizes), 11)
    vkp, chm = np.ascontiguousarray(w['vkp'][:n]), list(w['chm'][:n])
    agp, ok = _aggregate(w, off, np.ascontiguousarray(w['sigp'][:n]), msgs)
    assert ok.all()
    assert _verify(w, off, vkp, chm, msgs, agp).tolist() == [1] * len(sizes)
    ag = eng.unpack(agp, w['ab'], bd)
    pk = lambda a: eng.pack(np.ascontiguousarray(a), w['ab'], bd)
    cases = []
    t = ag.copy(); t[0, 1, 2] += 1; t[8, 0, 255] -= 1; cases.append((pk(t), vkp, chm, msgs, {0, 8}))     # +-1
    t = ag.copy(); t[1, 5, 9] = bd + 1; t[2, l - 1, 0] = bd + 2; cases.append((pk(t), vkp, chm, msgs, {1, 2}))   # above avf_bd
    t = ag.copy(); t[3] = 0; cases.append((pk(t), vkp, chm, msgs, {3}))                                  # all-bias fields
    c2 = list(chm); c2[int(off[4]) + 1] += '0'; cases.append((agp, vkp, c2, msgs, {4}))                  # challenge message
    m2 = list(msgs); m2[5] = m2[5] + b'x'; cases.append((agp, vkp, chm, m2, {5}))                        # aggregation message
    vk = eng.unpack(vkp, w['kb'], 0, dtype=np.uint16)
    vk[int(off[6]), 1, 77] = (int(vk[int(off[6]), 1, 77]) + 1) % q
    cases.append((agp, eng.pack(vk, w['kb'], 0), chm, msgs, {6}))                                        # one key slot
    for a, k, c, m, bad in cases:
        v = _verify(w, off, k, c, m, a)
        assert v.tolist() == [0 if g in bad else 1 for g in range(len(sizes))], bad
        assert np.array_equal(v, _ref_verify(w, off, k, w['kb'], c, m, a, w['ab'], bd)), bad
    # above ag_cap and an empty group
    big = _offsets([2, 3, 0, 1])
    nb = int(big[-1])
    mb = _messages(4, 12)
    agb, _ = _aggregate(w, _offsets([2, 3, 1]), np.ascontiguousarray(w['sigp'][:nb]), [mb[0], mb[1], mb[3]])
    agb = np.ascontiguousarray(agb[[0, 1, 0, 2]])
    kb_, cb = np.ascontiguousarray(w['vkp'][:nb]), w['chm'][:nb]
    v = _verify(w, big, kb_, cb, mb, agb)
    assert v.tolist() == [1, 0, 0, 1]
    assert np.array_equal(v, _ref_verify(w, big, kb_, w['kb'], cb, mb, agb, w['ab'], bd))


def test_out_of_range_aggregates(world):
    """Aggregates of 16 and 64 signatures leave the 12 / 14-bit range: in_range is 0 exactly where lcb_pack_batch says
    so and where a numpy range test of the unpacked aggregate says so, and the bytes are still equal."""
    w = world
    sizes = [16] * 12 + [64] * 4 + [1, 2]
    off = _offsets(sizes)
    msgs = _messages(len(sizes), 17)
    agp, ok, _ = _check_both(w, off, msgs)
    ag = w['eng'].aggregate_batch(w['sch'], off, np.ascontiguousarray(w['sigs'][:int(off[-1])]), msgs)
    field = ag.astype(np.int64) + w['avf_bd']
    want_ok = ((field >= 0) & (field < (1 << w['ab']))).all(axis=2)
    assert np.array_equal(ok.astype(bool), want_ok)
    assert not want_ok[12:16].all() and want_ok[16:].all()


def _misaligned(x):
    """A device copy of x that is 4-byte but not 16-byte aligned."""
    import torch
    flat = torch.from_numpy(np.ascontiguousarray(x).reshape(-1)).cuda()
    raw = torch.zeros(flat.numel() + 16, dtype=torch.uint8, device='cuda')
    view = raw[4:4 + flat.numel()]
    view.copy_(flat)
    assert view.data_ptr() % 16 == 4
    return view.view(*x.shape)


def test_random_bytes_fused_and_unpack_first_agree(world):
    import torch
    w = world
    eng, l = w['eng'], w['l']
    rng = np.random.default_rng(23)
    sizes = [1, 2] * 20
    off = _offsets(sizes)
    n = int(off[-1])
    msgs = _messages(len(sizes), 29)
    chm = w['chm'][:n]
    sigp = np.ascontiguousarray(w['sigp'][:n]).copy()
    sigp[1::2] = rng.integers(0, 256, sigp[1::2].shape, dtype=np.uint8)           # every other signature: random bytes
    for sbias, abias in ((w['vf_bd'], w['avf_bd']), (0, 32767), (1234, 77)):
        want = _ref_aggregate(w, off, sigp, msgs, w['sb'], sbias, w['ab'], abias)
        fused = _aggregate(w, off, sigp, msgs, sbias=sbias, abias=abias)
        torch.cuda.synchronize()
        first = _aggregate(w, off, _misaligned(sigp), msgs, sbias=sbias, abias=abias, device=True)
        eng.synchronize()
        for got in (fused, tuple(x.cpu().numpy() for x in first)):
            assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]), (sbias, abias)
    # non-shipped widths: signatures at 12 bits, aggregates at 13 and 16
    for sb, ab in ((12, 13), (12, 16)):
        s12 = rng.integers(0, 256, (n, l, 32 * sb), dtype=np.uint8)
        got = _aggregate(w, off, s12, msgs, sb=sb, sbias=2000, ab=ab, abias=3000)
        want = _ref_aggregate(w, off, s12, msgs, sb, 2000, ab, 3000)
        assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]), (sb, ab)
    # verify: honest groups next to groups with random aggregate rows and a group with random key bytes
    agp, _ = _aggregate(w, off, np.ascontiguousarray(w['sigp'][:n]), msgs)
    agp = agp.copy()
    agp[[1, 4]] = rng.integers(0, 256, agp[[1, 4]].shape, dtype=np.uint8)
    vkp = np.ascontiguousarray(w['vkp'][:n]).copy()
    vkp[int(off[6])] = rng.integers(0, 256, vkp[0].shape, dtype=np.uint8)
    for abias in (w['avf_bd'], 0, 32767):
        want = _ref_verify(w, off, vkp, w['kb'], chm, msgs, agp, w['ab'], abias)
        fused = _verify(w, off, vkp, chm, msgs, agp, abias=abias)
        torch.cuda.synchronize()
        first = _verify(w, off, _misaligned(vkp), chm, msgs, _misaligned(agp), abias=abias, device=True)
        eng.synchronize()
        assert np.array_equal(fused, want) and np.array_equal(first.cpu().numpy(), want), abias
        if abias == w['avf_bd']:
            assert want.tolist() == [0 if g in (1, 4, 6) else 1 for g in range(len(sizes))]
    # keys at 15 bits, aggregates at 13 and 16 bits: the unpack-first route
    vk = eng.unpack(vkp, w['kb'], 0, dtype=np.uint16)
    ag = eng.unpack(agp, w['ab'], w['avf_bd'])
    for kb, ab in ((15, 13), (15, 16), (w['kb'], 16)):
        k = eng.pack(vk, kb, 0)
        a = eng.pack(ag, ab, w['avf_bd'])
        got = _verify(w, off, k, chm, msgs, a, kb=kb, ab=ab)
        assert np.array_equal(got, _ref_verify(w, off, k, kb, chm, msgs, a, ab, w['avf_bd'])), (kb, ab)
        if kb >= w['kb'] and ab >= w['ab']:          # wide enough for every honest key slot and aggregate coefficient
            assert got.tolist() == [0 if g in (1, 4, 6) else 1 for g in range(len(sizes))]


def test_device_buffers_and_group_loop(world):
    import torch
    from lattice_cryptography_b200.lm_one_time_sigs import _ctx
    w = world
    eng = w['eng']
    sizes = [1, 5, 2, 40, 3]
    off = _offsets(sizes)
    n = int(off[-1])
    msgs = _messages(len(sizes), 21)
    sigp, vkp, chm = np.ascontiguousarray(w['sigp'][:n]), np.ascontiguousarray(w['vkp'][:n]), w['chm'][:n]
    host = _aggregate(w, off, sigp, msgs)
    dev = lambda x: torch.from_numpy(np.array(x)).cuda()
    d_off, d_sigp, d_vkp = dev(off), dev(sigp), dev(vkp)
    torch.cuda.synchronize()
    got = _aggregate(w, d_off, d_sigp, msgs, device=True)
    eng.synchronize()
    assert np.array_equal(got[0].cpu().numpy(), host[0]) and np.array_equal(got[1].cpu().numpy(), host[1])
    vh = _verify(w, off, vkp, chm, msgs, host[0], cap=1 << 20)
    vd = _verify(w, d_off, d_vkp, chm, msgs, got[0], cap=1 << 20, device=True)
    eng.synchronize()
    assert np.array_equal(vd.cpu().numpy(), vh)
    assert vh[[0, 2]].all()
    # ag_wt = 2 on the shipped geometry: the per-group loop, after unpacking
    _, sch2 = _ctx(dict(w['pp'], ag_wt=2))
    a2 = _aggregate(w, off, sigp, msgs, sch=sch2)
    want = _ref_aggregate(w, off, sigp, msgs, w['sb'], w['vf_bd'], w['ab'], w['avf_bd'], sch=sch2)
    assert np.array_equal(a2[0], want[0]) and np.array_equal(a2[1], want[1])
    assert not np.array_equal(a2[0], host[0])
    v2 = _verify(w, off, vkp, chm, msgs, a2[0], cap=1 << 20, sch=sch2)
    assert np.array_equal(v2, _ref_verify(w, off, vkp, w['kb'], chm, msgs, a2[0], w['ab'], w['avf_bd'], cap=1 << 20, sch=sch2))


def test_argument_errors(world):
    import torch
    from lattice_cryptography_b200 import Engine, LcbError, _ffi
    w = world
    eng, sch, l = w['eng'], w['sch'], w['l']
    off = _offsets([2, 1])
    msgs = _messages(2, 3)
    sigp, vkp, chm = np.ascontiguousarray(w['sigp'][:3]), np.ascontiguousarray(w['vkp'][:3]), w['chm'][:3]
    agp, _ = _aggregate(w, off, sigp, msgs)

    def invalid(fn):
        with pytest.raises(LcbError) as e:
            fn()
        assert e.value.status == _ffi.LCB_ERR_INVALID

    for bits in (0, 17):
        invalid(lambda: _aggregate(w, off, np.zeros((3, l, 32 * bits), np.uint8), msgs, sb=bits))
        invalid(lambda: _aggregate(w, off, sigp, msgs, ab=bits))
        invalid(lambda: _verify(w, off, np.zeros((3, 2, 32 * bits), np.uint8), chm, msgs, agp, kb=bits))
        invalid(lambda: _verify(w, off, vkp, chm, msgs, np.zeros((2, l, 32 * bits), np.uint8), ab=bits))
    for bias in (-1, 32768):
        invalid(lambda: _aggregate(w, off, sigp, msgs, sbias=bias))
        invalid(lambda: _aggregate(w, off, sigp, msgs, abias=bias))
        invalid(lambda: _verify(w, off, vkp, chm, msgs, agp, abias=bias))
    raw = torch.zeros(sigp.size + 16, dtype=torch.uint8, device='cuda')
    odd = raw[1:1 + sigp.size].view(*sigp.shape)
    invalid(lambda: _aggregate(w, off, odd, msgs))
    rawa = torch.zeros(agp.size + 16, dtype=torch.uint8, device='cuda')
    invalid(lambda: _verify(w, off, vkp, chm, msgs, rawa[2:2 + agp.size].view(*agp.shape)))
    invalid(lambda: _aggregate(w, np.array([0, 2, 2, 3], np.int64), sigp, _messages(3, 4)))     # an empty group
    lib = _ffi.load()
    from ctypes import byref, c_void_p
    z = np.zeros(1, np.int64)
    assert lib.lcb_bklm_aggregate_packed_batch(eng._ctx, byref(sch), c_void_p(z.ctypes.data), 0, None, 11, 0, None,
                                               c_void_p(z.ctypes.data), 12, 0, None, None) == _ffi.LCB_OK
    assert lib.lcb_bklm_aggregate_verify_packed_batch(eng._ctx, byref(sch), c_void_p(z.ctypes.data), 0, None, 14, None,
                                                      c_void_p(z.ctypes.data), None, c_void_p(z.ctypes.data), None, 12, 0,
                                                      2, 1, 1, None) == _ffi.LCB_OK
    gen = Engine(128, 12289, 512, 2)
    try:
        gsch = _ffi.LcbScheme()
        gsch.ag_bd = gsch.ag_wt = gsch.ch_bd = gsch.ch_wt = gsch.sk_bd = gsch.sk_wt = 1
        with pytest.raises(LcbError) as e:
            gen.aggregate_packed_batch(gsch, off, np.zeros((3, 2, 512 * 11 // 8), np.uint8), 11, 0, msgs, 12, 0)
        assert e.value.status == _ffi.LCB_ERR_INVALID and 'd == 256' in str(e.value)
        with pytest.raises(LcbError) as e:
            gen.aggregate_verify_packed_batch(gsch, off, np.zeros((3, 2, 512 * 14 // 8), np.uint8), 14, chm, msgs,
                                              np.zeros((2, 2, 512 * 12 // 8), np.uint8), 12, 0, 2, 1, 1)
        assert e.value.status == _ffi.LCB_ERR_INVALID and 'd == 256' in str(e.value)
    finally:
        gen.close()


@pytest.mark.parametrize('mode', ['reference', 'tree'])
def test_wire_layer_equals_dropin_batch(mode):
    from lattice_cryptography_b200 import bklm_one_time_agg_sigs as bk
    from lattice_cryptography_b200 import wire
    from lattice_cryptography_b200.lm_one_time_sigs import keygen, sign
    pp = bk.set_aggregation_mode(bk.make_setup_parameters(128), mode)
    keys = keygen(pp=pp, num_keys_to_gen=11)
    msgs = [bin(randbits(32))[2:].zfill(32) for _ in keys]
    sigs = [sign(pp=pp, otk=k, msg=m) for k, m in zip(keys, msgs)]
    vks = [k[2] for k in keys]
    cuts = [(0, 2), (2, 3), (3, 5), (5, 7), (7, 9), (9, 11)]
    gk, gm, gs = ([x[a:b] for a, b in cuts] for x in (vks, msgs, sigs))
    ags = bk.aggregate_batch(pp, gk, gm, gs)
    rows, vrows, chm, agmsgs, counts = [], [], [], [], []
    for keys_g, msgs_g, sigs_g in zip(gk, gm, gs):
        srt_keys, srt_msgs, srt_sigs = bk.prepare_aggregate(otvks=keys_g, msgs=msgs_g, sigs=sigs_g)
        rows.extend(s.coef for s in srt_sigs)
        vrows.extend(np.stack([k[0].ntt, k[1].ntt]) for k in srt_keys)
        chm.extend(bk.challenge_messages(srt_keys, srt_msgs))
        agmsgs.append(str(list(zip(srt_keys, srt_msgs))))
        counts.append(len(srt_sigs))
    off = _offsets(counts)
    sigp, ok = wire.pack_signatures(pp, np.ascontiguousarray(np.stack(rows)))
    assert ok.all()
    vkp = wire.pack_keys(pp, np.ascontiguousarray(np.stack(vrows)))
    agp, in_range = wire.aggregate_batch_packed(pp, off, sigp, agmsgs)
    want, want_ok = wire.pack_signatures(pp, np.ascontiguousarray(np.stack([a.coef for a in ags])), bound_key='avf_bd')
    assert np.array_equal(agp, want) and np.array_equal(in_range, want_ok) and in_range.all()
    v = wire.aggregate_verify_batch_packed(pp, off, vkp, chm, agmsgs, agp)
    assert v.tolist() == [1] * len(cuts)
    t = [a for a in ags]
    from lattice_cryptography_b200.lattice_algebra import PolynomialVector
    bad = ags[3].coef.copy()
    bad[0, 0] += 1
    t[3] = PolynomialVector(pp['scheme_parameters'].lp, const_time_flag=False, _coef=bad)
    tp, _ = wire.pack_signatures(pp, np.ascontiguousarray(np.stack([a.coef for a in t])), bound_key='avf_bd')
    v = wire.aggregate_verify_batch_packed(pp, off, vkp, chm, agmsgs, tp)
    assert [bool(x) for x in v] == bk.aggregate_verify_batch(pp, gk, gm, t) == [g != 3 for g in range(len(cuts))]


def test_small_batch_all_routes(world):
    """A small case of the three checks above (the checked build runs it)."""
    w = world
    sizes = [1, 2, 3, 17, 2, 16, 1]
    off = _offsets(sizes)
    agp, ok, v = _check_both(w, off, _messages(len(sizes), 7))
    assert v.tolist() == [1, 1, 0, 0, 1, 0, 1] and ok[[0, 1, 4, 6]].all()
    ag = w['eng'].unpack(agp, w['ab'], w['avf_bd'])
    ag[4, 0, 3] += 1
    t = w['eng'].pack(ag, w['ab'], w['avf_bd'])
    n = int(off[-1])
    v2 = _verify(w, off, np.ascontiguousarray(w['vkp'][:n]), w['chm'][:n], _messages(len(sizes), 7), t)
    assert v2.tolist() == [1, 1, 0, 0, 0, 0, 1]


def test_packed_batches_pass_on_the_checked_build():
    from lattice_cryptography_b200 import _ffi
    if _ffi.load().lcb_build_is_checked():
        pytest.skip('already running on the checked build')
    lib = os.path.join(ROOT, 'lattice_cryptography_b200', 'liblcb200_checked.so')
    if not os.path.exists(lib):
        subprocess.run(['make', '-C', os.path.join(ROOT, 'lattice_cryptography_b200', 'csrc'), '-j4', 'CHECKED=1'], check=True,
                       capture_output=True)
    env = dict(os.environ, LCB200_LIB=lib)
    r = subprocess.run([sys.executable, '-m', 'pytest', 'tests/test_gpu_bklm_packed.py', '-q', '-x', '-m', 'gpu', '-k',
                        'small_batch_all_routes', '-p', 'no:cacheprovider'],
                       env=env, capture_output=True, text=True, timeout=1500, cwd=ROOT)
    tail = r.stdout[-2500:] + r.stderr[-1500:]
    assert r.returncode == 0, tail
    assert '2 passed' in r.stdout and 'failed' not in r.stdout, tail
