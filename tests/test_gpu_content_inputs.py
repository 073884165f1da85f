"""Content-mode hash inputs built on the GPU (include/lcb200.h: lcb_content_str_batch, lcb_challenge_inputs_batch,
lcb_aggregation_inputs_batch; wire.content_strs / challenge_inputs / aggregation_inputs), compared byte for byte with
repr() and the challenge / aggregation strings of the drop-in objects in content mode, with hashlib over the C oracle's
key coefficients and over unpack -> ntt_inv of random bytes, and run end to end on packed records only."""
import hashlib
from ctypes import c_void_p

import numpy as np
import pytest

from test_gpu_parity import D, SHIPPED, engines, scheme   # noqa: F401  (fixture re-export)

pytestmark = pytest.mark.gpu
NAMES = {'vk': 'OneTimeVerificationKey', 'st': 'OneTimePublicStatement'}
KEY_BITS = {128: 14, 256: 16}


@pytest.fixture
def content_mode():
    from lattice_cryptography_b200.one_time_keys import set_content_str
    set_content_str(True)
    try:
        yield
    finally:
        set_content_str(False)


def _ref_str(kind, secpar, rows) -> str:
    """repr() in content mode of a key / statement with these centred int16 coefficient rows (one_time_keys._content_digest)."""
    h = hashlib.shake_256(NAMES[kind].encode() + secpar.to_bytes(2, 'little') +
                          np.ascontiguousarray(rows, dtype=np.int16).astype('<i2').tobytes())
    return f'<{NAMES[kind]} {h.hexdigest(16)}>'


def _strs(arr):
    return [bytes(r).decode() for r in np.asarray(arr)]


def _seed_objs(pp, n, seed):
    from lattice_cryptography_b200.one_time_keys import SecretSeed
    sp = pp['scheme_parameters']
    rng = np.random.default_rng(seed)
    return [SecretSeed(''.join(rng.choice(['0', '1'], sp.secpar)), sp.secpar, sp.lp) for _ in range(n)]


def _misaligned(x):
    """A device copy of x that is 4-byte but not 16-byte aligned."""
    import torch
    flat = torch.from_numpy(np.ascontiguousarray(x).reshape(-1).view(np.uint8)).cuda()
    raw = torch.zeros(flat.numel() + 16, dtype=torch.uint8, device='cuda')
    view = raw[4:4 + flat.numel()]
    view.copy_(flat)
    assert view.data_ptr() % 16 == 4
    torch.cuda.synchronize()                 # the engine reads it on its own stream
    return view.view(*x.shape)


def _dev(x):
    """A device copy of x, complete before an engine call reads it on the engine's stream."""
    import torch
    t = torch.from_numpy(np.ascontiguousarray(x)).cuda()
    torch.cuda.synchronize()
    return t


def _bitmsgs(rng, n, lens=(0, 1, 31, 32, 77, 135, 136, 137, 200, 271, 272, 300)):
    return [''.join(rng.choice(['0', '1'], int(lens[i % len(lens)]))) for i in range(n)]


# ------------------------------------------------------------------------------------------- 1. vs the drop-in objects
@pytest.mark.parametrize('n', [1, 7, 2049])
@pytest.mark.parametrize('secpar', [128, 256])
def test_content_strs_equal_dropin_repr(content_mode, secpar, n):
    from lattice_cryptography_b200 import adaptor_sigs as ad
    from lattice_cryptography_b200 import lm_one_time_sigs as lm
    from lattice_cryptography_b200 import wire
    pp = lm.make_setup_parameters(secpar)
    e = wire._engine(pp)
    seeds = _seed_objs(pp, n, 11 * secpar + n)
    keys = lm.keygen(pp, n, seeds=seeds, multiprocessing=False)
    want = [repr(k[2]) for k in keys]
    assert all(len(w) == 57 for w in want)
    _, vkp = wire.keygen_batch_packed(pp, seeds)
    assert _strs(wire.content_strs(pp, vkp)) == want
    # plain uint16 NTT arrays as 16 bits, packed 16-bit rows, device buffers (16- and 4-byte aligned)
    vk_ntt = lm.keygen_batch(pp, seeds, want_coef=False)['vk_ntt']
    assert _strs(e.content_str('vk', vk_ntt, 16)) == want
    assert _strs(e.content_str('vk', e.pack(vk_ntt, 16, 0), 16)) == want
    got = e.content_str('vk', _dev(vkp), KEY_BITS[secpar], device=True)
    e.synchronize()                          # every buffer on the device: the call is asynchronous
    assert _strs(got.cpu().numpy()) == want
    assert _strs(e.content_str('vk', _misaligned(vkp), KEY_BITS[secpar])) == want
    # statements
    app = ad.make_setup_parameters(secpar)
    wseeds = _seed_objs(app, n, 13 * secpar + n)
    sts = [w[2] for w in ad.witgen(app, n, seeds=wseeds)]
    want_st = [repr(s) for s in sts]
    _, stp = wire.witgen_batch_packed(app, wseeds)
    assert _strs(wire.content_strs(app, stp, 'st')) == want_st
    assert _strs(e.content_str('st', _misaligned(stp), KEY_BITS[secpar])) == want_st


# ------------------------------------------------------------------------------------------- 2. vs independent references
@pytest.mark.parametrize('secpar', [128, 256])
def test_content_strs_of_c_oracle_keys(engines, golden, secpar):
    import c_oracle
    arrays, _ = golden
    e = engines[secpar]
    s = SHIPPED[secpar]
    p = c_oracle.params(secpar, s['q'], s['l'], s['sk_bd'], s['ch_wt'])
    key_ch = np.ascontiguousarray(arrays[f's{secpar}_key_ch'])
    rng = np.random.default_rng(5 + secpar)
    seeds = [''.join(rng.choice(['0', '1'], secpar)) for _ in range(6)]
    _, _, vkp = e.lm_keygen_packed(scheme(secpar), seeds, 8, s['sk_bd'], KEY_BITS[secpar], want_sk=False)
    got = _strs(e.content_str('vk', vkp, KEY_BITS[secpar]))
    for i, seed in enumerate(seeds):
        _, _, vkl, vkr = c_oracle.lm_keygen(p, key_ch, seed.encode())
        assert got[i] == _ref_str('vk', secpar, np.stack([vkl, vkr]))


@pytest.mark.parametrize('bits', [1, 7, 14, 16])
@pytest.mark.parametrize('secpar', [128, 256])
def test_content_strs_of_random_bytes(engines, secpar, bits):
    """Any packed bytes, slots >= q included: hashlib over unpack -> ntt_inv."""
    e = engines[secpar]
    rng = np.random.default_rng(bits * secpar)
    n = 300
    for kind, lead in (('vk', (n, 2)), ('st', (n,))):
        packed = rng.integers(0, 256, lead + (32 * bits,), dtype=np.uint8)
        packed[0] = 0xFF                                            # every slot at 2^bits - 1
        coef = e.ntt_inv(e.unpack(packed, bits, 0, dtype=np.uint16))
        got = _strs(e.content_str(kind, packed, bits))
        assert got == [_ref_str(kind, secpar, coef[i]) for i in range(n)]


def test_content_strs_across_chunks(engines):
    """More items than one internal chunk (four sampler waves): every chunk boundary lands on the right row."""
    e = engines[128]
    import torch
    n = 4 * torch.cuda.get_device_properties(0).multi_processor_count * 5 * 128 + 129
    rng = np.random.default_rng(3)
    packed = rng.integers(0, 256, (n, 32 * 14), dtype=np.uint8)
    got = e.content_str('st', packed, 14)
    coef = e.ntt_inv(e.unpack(packed, 14, 0, dtype=np.uint16))
    for i in list(range(0, n, 9973)) + [n - 129, n - 128, n - 1]:
        assert bytes(got[i]).decode() == _ref_str('st', 128, coef[i])


# ------------------------------------------------------------------------------------------- 3. challenge inputs
@pytest.mark.parametrize('secpar', [128, 256])
def test_challenge_inputs_equal_dropin(content_mode, secpar):
    from lattice_cryptography_b200 import adaptor_sigs as ad
    from lattice_cryptography_b200 import lm_one_time_sigs as lm
    from lattice_cryptography_b200 import ragged, wire
    pp = ad.make_setup_parameters(secpar)
    e = wire._engine(pp)
    n = 301
    seeds = _seed_objs(pp, n, secpar)
    keys = lm.keygen(pp, n, seeds=seeds, multiprocessing=False)
    wits = ad.witgen(pp, n, seeds=seeds)
    rng = np.random.default_rng(secpar)
    msgs = [''.join(rng.choice(['0', '1'], i)) for i in range(n)]           # lengths 0 .. 300
    msgs[5] = 'ünïcødé ✓ ' * 7                                               # UTF-8 bytes
    vks, sts = [k[2] for k in keys], [w[2] for w in wits]
    _, vkp = wire.keygen_batch_packed(pp, seeds)
    _, stp = wire.witgen_batch_packed(pp, seeds)
    for st_packed, want in ((None, lm.challenge_messages(vks, msgs)), (stp, ad.challenge_messages(sts, vks, msgs))):
        want_blob, want_off = ragged(want)
        blob, off = wire.challenge_inputs(pp, vkp, msgs, st_packed=st_packed)
        assert np.array_equal(off, want_off) and bytes(blob) == bytes(want_blob)
        dblob, doff = wire.challenge_inputs(pp, _dev(vkp), ragged(msgs), device=True,
                                            st_packed=None if st_packed is None else _dev(st_packed))
        e.synchronize()
        assert np.array_equal(doff.cpu().numpy(), want_off) and bytes(dblob.cpu().numpy()) == bytes(want_blob)


def test_challenge_inputs_offsets_not_starting_at_zero(engines):
    """msg_off[0] > 0 through the C ABI, host and device message buffers."""
    from lattice_cryptography_b200 import _ffi
    e = engines[128]
    rng = np.random.default_rng(8)
    n = 50
    vk = rng.integers(33, 127, (n, 57), dtype=np.uint8)
    st = rng.integers(33, 127, (n, 57), dtype=np.uint8)
    lens = rng.integers(0, 300, n)
    off = (1000 + np.concatenate([[0], np.cumsum(lens)])).astype(np.int64)
    msg = rng.integers(0, 256, int(off[-1]) + 10, dtype=np.uint8)
    for with_st in (False, True):
        want, woff = [], [0]
        for i in range(n):
            item = (bytes(st[i]) + b', ' if with_st else b'') + bytes(vk[i]) + b', ' + bytes(msg[off[i]:off[i + 1]])
            want.append(item)
            woff.append(woff[-1] + len(item))
        total = woff[-1]
        assert total == int(off[-1] - off[0]) + n * (118 if with_st else 59)
        for dev in (False, True):
            put = _dev if dev else (lambda x: x)
            m, o, v, s = put(msg), put(off), put(vk), put(st)
            out = np.zeros(total, np.uint8)
            out_off = np.zeros(n + 1, np.int64)
            ptr = lambda x: c_void_p(x.data_ptr() if dev else x.ctypes.data)   # noqa: E731
            assert e._lib.lcb_challenge_inputs_batch(e._ctx, ptr(s) if with_st else None, ptr(v), ptr(m), ptr(o), n,
                                                     c_void_p(out.ctypes.data), c_void_p(out_off.ctypes.data)) == _ffi.LCB_OK
            assert out_off.tolist() == woff and bytes(out) == b''.join(want)


# ------------------------------------------------------------------------------------------- 4. aggregation inputs
def _groups(pp, sizes, seed, dup=None):
    from lattice_cryptography_b200 import lm_one_time_sigs as lm
    from lattice_cryptography_b200 import wire
    total = sum(sizes)
    seeds = _seed_objs(pp, total, seed)
    if dup is not None:
        seeds[dup[1]] = seeds[dup[0]]                                # the same key twice in one group
    keys = lm.keygen(pp, total, seeds=seeds, multiprocessing=False)
    _, vkp = wire.keygen_batch_packed(pp, seeds)
    rng = np.random.default_rng(seed)
    msgs = _bitmsgs(rng, total)
    if dup is not None:
        msgs[dup[1]] = msgs[dup[0]][::-1] + '1'
    off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    return keys, vkp, msgs, off


@pytest.mark.parametrize('secpar', [128, 256])
def test_aggregation_inputs_equal_dropin(content_mode, secpar):
    from lattice_cryptography_b200 import bklm_one_time_agg_sigs as bk
    from lattice_cryptography_b200 import ragged, wire
    pp = bk.make_setup_parameters(secpar)
    sizes = [0, 1, 2, 3, 1000, 0, 2, 4]
    keys, vkp, msgs, off = _groups(pp, sizes, secpar, dup=(1 + 2 + 3 + 1000 + 2 + 1, 1 + 2 + 3 + 1000 + 2 + 3))
    vks = [k[2] for k in keys]
    order, chmsgs, agmsgs = wire.aggregation_inputs(pp, off, vkp, msgs)
    want_order, want_ag, want_ch = [], [], []
    for g in range(len(sizes)):
        a, b = int(off[g]), int(off[g + 1])
        srt_keys, srt_msgs = bk.prepare_make_agg_coefs(vks[a:b], msgs[a:b])
        idx = sorted(range(a, b), key=lambda i: str(vks[i]))                # stable, as prepare_make_agg_coefs sorts
        assert [vks[i] for i in idx] == srt_keys
        want_order.extend(idx)
        want_ag.append(str(list(zip(srt_keys, srt_msgs))))
        want_ch.extend(bk.challenge_messages(srt_keys, srt_msgs))
    assert order.tolist() == want_order and agmsgs == want_ag
    assert agmsgs[0] == '[]'
    wb, wo = ragged(want_ch)
    assert np.array_equal(chmsgs[1], wo) and bytes(chmsgs[0]) == bytes(wb)
    dup = [i for i in order[off[7]:off[8]] if i in (1009, 1011)]              # one key twice: input order kept
    assert dup == [1009, 1011] and repr(vks[1009]) == repr(vks[1011])
    # the engine call alone, device buffers
    e = wire._engine(pp)
    vk_str = wire.content_strs(pp, vkp)[order]
    blob, aoff = e.aggregation_inputs(_dev(off), _dev(vk_str), ragged([msgs[i] for i in order]), device=True)
    e.synchronize()
    assert _strs_ragged(blob.cpu().numpy(), aoff.cpu().numpy()) == want_ag


def _strs_ragged(blob, off):
    return [bytes(blob[off[i]:off[i + 1]]).decode() for i in range(len(off) - 1)]


def test_aggregation_inputs_rejects_non_bitstrings(content_mode):
    from lattice_cryptography_b200 import bklm_one_time_agg_sigs as bk
    from lattice_cryptography_b200 import wire
    pp = bk.make_setup_parameters(128)
    _, vkp, msgs, off = _groups(pp, [2], 1)
    with pytest.raises(ValueError, match='Input messages must be bitstrings.'):
        wire.aggregation_inputs(pp, off, vkp, [msgs[0], 'hello'])


# ------------------------------------------------------------------------------------------- 5. end to end on packed records
@pytest.mark.parametrize('secpar', [128, 256])
def test_packed_lm_and_adaptor_end_to_end(content_mode, secpar):
    from lattice_cryptography_b200 import adaptor_sigs as ad
    from lattice_cryptography_b200 import lm_one_time_sigs as lm
    from lattice_cryptography_b200 import one_time_keys, wire
    from lattice_cryptography_b200.lattice_algebra import PolynomialVector
    pp = ad.make_setup_parameters(secpar)
    n = 40
    seeds = _seed_objs(pp, n, 3 * secpar)
    rng = np.random.default_rng(secpar)
    msgs = _bitmsgs(rng, n)
    skp, vkp = wire.keygen_batch_packed(pp, seeds)
    chm = wire.challenge_inputs(pp, vkp, msgs)
    sigp, ok = wire.sign_batch_packed_sk(pp, skp, chm)
    assert ok.all()
    keys = lm.keygen(pp, n, seeds=seeds, multiprocessing=False)
    want = np.stack([lm.sign(pp, k, m).coef for k, m in zip(keys, msgs)])
    assert np.array_equal(sigp, wire.pack_signatures(pp, want)[0])
    assert wire.verify_batch_packed(pp, vkp, chm, sigp).all()
    flipped = list(msgs)
    flipped[3] = ('1' if flipped[3][:1] == '0' else '0') + flipped[3][1:] if flipped[3] else '0'
    v = wire.verify_batch_packed(pp, vkp, wire.challenge_inputs(pp, vkp, flipped), sigp)
    assert v.tolist() == [i != 3 for i in range(n)]
    one_time_keys.set_content_str(False)                                      # reference-mode signature of the same key
    ref = wire.pack_signatures(pp, np.stack([lm.sign(pp, keys[0], msgs[0]).coef]))[0]
    one_time_keys.set_content_str(True)
    assert not wire.verify_batch_packed(pp, vkp[:1], wire.challenge_inputs(pp, vkp[:1], msgs[:1]), ref).any()
    # adaptor: presign -> preverify -> adapt -> verify, against the drop-in objects
    witp, stp = wire.witgen_batch_packed(pp, seeds)
    wits = ad.witgen(pp, n, seeds=seeds)
    achm = wire.challenge_inputs(pp, vkp, msgs, st_packed=stp)
    presig, ok = wire.presign_batch_packed_sk(pp, skp, achm)
    assert ok.all()
    want_pre = np.stack([ad.presign(pp, k, m, w[2]).coef for k, m, w in zip(keys, msgs, wits)])
    assert np.array_equal(presig, wire.pack_signatures(pp, want_pre, bound_key='pvf_bd')[0])
    assert wire.preverify_batch_packed(pp, vkp, achm, presig).all()
    asig, ok = wire.adapt_batch_packed_wit(pp, presig, witp)
    assert ok.all()
    dropin = [ad.adapt(PolynomialVector(pp['scheme_parameters'].lp, const_time_flag=False, _coef=want_pre[i]), wits[i][1])
              for i in range(n)]
    assert all(ad.verify(pp, k[2], m, w[2], s) for k, m, w, s in zip(keys, msgs, wits, dropin))
    assert np.array_equal(asig, wire.pack_signatures(pp, np.stack([d.coef for d in dropin]))[0])
    assert wire.adaptor_verify_batch_packed(pp, vkp, achm, stp, asig).all()


def test_packed_bklm_end_to_end(content_mode):
    from lattice_cryptography_b200 import bklm_one_time_agg_sigs as bk
    from lattice_cryptography_b200 import lm_one_time_sigs as lm
    from lattice_cryptography_b200 import wire
    pp = bk.set_aggregation_capacity(bk.make_setup_parameters(128), 2)
    n_agg = 2000
    sizes = [1 + (g % 2) for g in range(n_agg)]
    total = sum(sizes)
    seeds = _seed_objs(pp, total, 77)
    rng = np.random.default_rng(77)
    msgs = _bitmsgs(rng, total, lens=(32, 0, 100, 150))
    off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    skp, vkp = wire.keygen_batch_packed(pp, seeds)
    sigp, ok = wire.sign_batch_packed_sk(pp, skp, wire.challenge_inputs(pp, vkp, msgs))
    assert ok.all()
    order, chm, agmsgs = wire.aggregation_inputs(pp, off, vkp, msgs)
    agp, in_range = wire.aggregate_batch_packed(pp, off, np.ascontiguousarray(sigp[order]), agmsgs)
    assert in_range.all()
    # the drop-in batch on objects
    keys = lm.keygen(pp, total, seeds=seeds, multiprocessing=False)
    sigs = [lm.sign(pp, k, m) for k, m in zip(keys, msgs)]
    cut = [(int(off[g]), int(off[g + 1])) for g in range(n_agg)]
    gk, gm, gs = ([x[a:b] for a, b in cut] for x in ([k[2] for k in keys], msgs, sigs))
    ags = bk.aggregate_batch(pp, gk, gm, gs)
    want = wire.pack_signatures(pp, np.stack([a.coef for a in ags]), bound_key='avf_bd')[0]
    assert np.array_equal(agp, want)
    v = wire.aggregate_verify_batch_packed(pp, off, np.ascontiguousarray(vkp[order]), chm, agmsgs, agp)
    assert v.all() and [bool(x) for x in v] == bk.aggregate_verify_batch(pp, gk, gm, ags)
    bad = agp.copy()
    bad[5, 0, 0] ^= 1
    v = wire.aggregate_verify_batch_packed(pp, off, np.ascontiguousarray(vkp[order]), chm, agmsgs, bad)
    assert v.tolist() == [g != 5 for g in range(n_agg)]


# ------------------------------------------------------------------------------------------- 6. errors
def test_argument_errors(engines):
    from lattice_cryptography_b200 import Engine, _ffi
    e = engines[128]
    lib, ctx = e._lib, e._ctx
    buf = np.zeros(4096 + 8, np.uint8)
    out = np.zeros(57 * 4, np.uint8)
    p = lambda x, k=0: c_void_p(x.ctypes.data + k)   # noqa: E731
    import torch
    dev = torch.zeros(4096 + 8, dtype=torch.uint8, device='cuda')
    odd = c_void_p(dev.data_ptr() + 2)                                         # a device buffer that is not 4-byte aligned
    for kind, bits, ptr in ((2, 14, p(buf)), (-1, 14, p(buf)), (0, 0, p(buf)), (0, 17, p(buf)), (1, 14, odd)):
        assert lib.lcb_content_str_batch(ctx, kind, ptr, bits, 2, p(out)) == _ffi.LCB_ERR_INVALID
    assert lib.lcb_content_str_batch(ctx, 0, p(buf), 14, 0, p(out)) == _ffi.LCB_OK
    off = np.zeros(3, np.int64)
    o2 = np.zeros(3, np.int64)
    assert lib.lcb_challenge_inputs_batch(ctx, None, None, p(buf), p(off), 2, p(out), p(o2)) == _ffi.LCB_ERR_INVALID
    assert lib.lcb_challenge_inputs_batch(ctx, None, p(buf), p(buf), p(off), 0, p(out), p(o2)) == _ffi.LCB_OK
    assert lib.lcb_aggregation_inputs_batch(ctx, p(off), 0, p(buf), p(buf), p(off), p(out), p(o2)) == _ffi.LCB_OK
    with pytest.raises(ValueError):
        e.content_str('sk', buf[:4 * 448].reshape(4, 448), 14)
    with pytest.raises(ValueError):
        e.content_str('st', buf[:4 * 448].reshape(4, 448), 13)
    for args in ((128, 12289, 512, 2), (128, 65537, 256, 2)):                # d = 512, q >= 2^16
        g = Engine(*args)
        try:
            st = lib.lcb_content_str_batch(g._ctx, 0, p(buf), 14, 1, p(out))
            assert st == _ffi.LCB_ERR_INVALID
            assert b'd == 256' in lib.lcb_last_error(g._ctx)
        finally:
            g.close()


def test_content_inputs_pass_on_the_checked_build():
    """A small case of every call on the checked build (device-side asserts on every new global access)."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    code = r'''
import numpy as np, hashlib
from lattice_cryptography_b200 import Engine, ragged
e = Engine(128, 11777, 256, 13)
assert e._lib.lcb_build_is_checked() == 1
rng = np.random.default_rng(1)
packed = rng.integers(0, 256, (130, 2, 448), dtype=np.uint8)
s = e.content_str('vk', packed, 14)
coef = e.ntt_inv(e.unpack(packed, 14, 0, dtype=np.uint16))
h = hashlib.shake_256(b'OneTimeVerificationKey' + (128).to_bytes(2, 'little') + coef[129].astype('<i2').tobytes())
assert bytes(s[129]).decode() == '<OneTimeVerificationKey ' + h.hexdigest(16) + '>'
msgs = ['0' * (i % 140) for i in range(130)]
blob, off = e.challenge_inputs(s, msgs, st_str=s)
assert bytes(blob[off[7]:off[8]]) == bytes(s[7]) + b', ' + bytes(s[7]) + b', ' + b'0' * 7
agg = np.array([0, 0, 1, 3, 130], np.int64)
blob, off = e.aggregation_inputs(agg, s, msgs)
assert bytes(blob[off[0]:off[1]]) == b'[]' and int(off[-1]) == blob.shape[0]
e.synchronize()
print('ok')
'''
    env = dict(os.environ, LCB200_LIB=os.path.join(root, 'lattice_cryptography_b200', 'liblcb200_checked.so'))
    r = subprocess.run([sys.executable, '-c', code], cwd=root, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and 'ok' in r.stdout, r.stdout + r.stderr
