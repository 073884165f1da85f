"""Keys on the packed wire format (include/lcb200.h: lcb_lm_keygen_packed_batch, lcb_lm_sign_packed_sk_batch), compared
byte for byte with the composition each call is defined as (keygen -> pack; unpack -> ntt_fwd -> lm_sign_packed), on the
fused route (7- / 8-bit keys, 11- / 13-bit signatures, k_sign_sk) and on the composed one, and with an independent numpy
statement of the signature: the challenge pairs, oracle/wire.py's decoder and the signed negacyclic rotations summed in
int64."""
import os
import subprocess
import sys
from ctypes import byref, c_void_p

import numpy as np
import pytest

from test_gpu_parity import D, SHIPPED, engines, scheme   # noqa: F401  (fixture re-export)

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# signing-key bits, signature bits, key bits, pvf_bd (presignatures; LM vf_bd), vf_bd (adaptor signatures)
WIDTHS = {128: (7, 11, 14, 945, 946), 256: (8, 13, 16, 3315, 3316)}


def _seeds(secpar, n, seed):
    rng = np.random.default_rng(seed)
    return [''.join(rng.choice(['0', '1'], secpar)) for _ in range(n)]


def _msgs(n, seed):
    rng = np.random.default_rng(seed)
    return [bytes(rng.integers(1, 256, int(rng.integers(0, 120)), dtype=np.uint8)) for _ in range(n)]


def _misaligned(x):
    """A device copy of x that is 4-byte but not 16-byte aligned."""
    import torch
    flat = torch.from_numpy(np.ascontiguousarray(x).reshape(-1).view(np.uint8)).cuda()
    raw = torch.zeros(flat.numel() + 16, dtype=torch.uint8, device='cuda')
    view = raw[4:4 + flat.numel()]
    view.copy_(flat)
    assert view.data_ptr() % 16 == 4
    return view.view(*x.shape)


def _composed(e, sch, skp, skb, skbias, msgs, sb, sbias):
    sk_ntt = e.ntt_fwd(e.unpack(skp, skb, skbias))
    return e.lm_sign_packed(sch, sk_ntt, msgs, sb, sbias, want_range=True)


def _numpy_sign(e, sch, skp, skb, skbias, msgs, q):
    """sk_left ** c + sk_right from the challenge pairs and oracle/wire.py's decoder, in int64, centred mod q."""
    import wire as owire
    pairs = e.challenge(sch, msgs).astype(np.int64)
    x = owire.unpack(skp, skb, skbias).astype(np.int64)             # [n, 2, l, 256]
    n, _, l, _ = x.shape
    acc = x[:, 1].copy()
    for i in range(n):
        for idx, s in pairs[i]:
            rolled = np.roll(x[i, 0], idx, axis=-1)
            rolled[:, :idx] *= -1
            acc[i] += s * rolled
    return ((acc + q // 2) % q - q // 2).astype(np.int16)


# ------------------------------------------------------------------------------------------- keygen
@pytest.mark.parametrize('n', [1, 7, 2049])
@pytest.mark.parametrize('secpar', [128, 256])
def test_keygen_packed_equals_keygen_then_pack(engines, secpar, n):
    e = engines[secpar]
    sch = scheme(secpar)
    skb, _, kb, _, _ = WIDTHS[secpar]
    sk_bd = SHIPPED[secpar]['sk_bd']
    seeds = _seeds(secpar, n, secpar + n)
    sk_coef, _, vk_ntt, _ = e.lm_keygen(sch, seeds, want_sk_ntt=False, want_vk_coef=False)
    want_sk, want_ok = e.pack(sk_coef, skb, sk_bd, want_range=True)
    want_vk = e.pack(vk_ntt, kb, 0)
    assert want_ok.all()
    sk, ok, vk = e.lm_keygen_packed(sch, seeds, skb, sk_bd, kb, want_sk_range=True)
    assert np.array_equal(sk, want_sk) and np.array_equal(ok, want_ok) and np.array_equal(vk, want_vk)
    # each output NULL in turn
    sk, ok, vk = e.lm_keygen_packed(sch, seeds, skb, sk_bd, kb, want_vk=False)
    assert np.array_equal(sk, want_sk) and ok is None and vk is None
    sk, ok, vk = e.lm_keygen_packed(sch, seeds, skb, sk_bd, kb, want_sk=False)
    assert sk is None and np.array_equal(vk, want_vk)
    # a batch over several internal chunks
    if n > 1:
        os.environ['LCB_KEYGEN_CHUNK'] = '3'
        try:
            sk, ok, vk = e.lm_keygen_packed(sch, seeds, skb, sk_bd, kb, want_sk_range=True)
        finally:
            os.environ.pop('LCB_KEYGEN_CHUNK')
        assert np.array_equal(sk, want_sk) and np.array_equal(ok, want_ok) and np.array_equal(vk, want_vk)


@pytest.mark.parametrize('secpar', [128, 256])
def test_keygen_packed_other_widths_and_device_buffers(engines, secpar):
    import torch
    from lattice_cryptography_b200 import ragged
    e = engines[secpar]
    sch = scheme(secpar)
    skb, _, kb, _, _ = WIDTHS[secpar]
    n = 300
    seeds = _seeds(secpar, n, 5 * secpar)
    sk_coef, _, vk_ntt, _ = e.lm_keygen(sch, seeds, want_sk_ntt=False, want_vk_coef=False)
    for sbits, sbias, vbits in ((6, 0, 15), (9, 300, 16), (16, 32767, 14), (skb, 0, kb)):
        want_sk, want_ok = e.pack(sk_coef, sbits, sbias, want_range=True)
        sk, ok, vk = e.lm_keygen_packed(sch, seeds, sbits, sbias, vbits, want_sk_range=True)
        assert np.array_equal(sk, want_sk) and np.array_equal(ok, want_ok) and np.array_equal(vk, e.pack(vk_ntt, vbits, 0))
        if (sbits, sbias) == (6, 0):                # negative coefficients do not fit without a bias
            assert not ok.all()
        elif sbias > 0:
            assert ok.all()
    blob, off = ragged(seeds)
    d_blob, d_off = (torch.from_numpy(np.array(x)).cuda() for x in (blob, off))
    torch.cuda.synchronize()
    sk, ok, vk = e.lm_keygen_packed(sch, (d_blob, d_off), skb, SHIPPED[secpar]['sk_bd'], kb, want_sk_range=True, device=True)
    e.synchronize()
    want_sk, want_ok = e.pack(sk_coef, skb, SHIPPED[secpar]['sk_bd'], want_range=True)
    assert np.array_equal(sk.cpu().numpy(), want_sk) and np.array_equal(ok.cpu().numpy(), want_ok)
    assert np.array_equal(vk.cpu().numpy(), e.pack(vk_ntt, kb, 0))


@pytest.mark.parametrize('secpar', [128, 256])
def test_keygen_packed_golden(engines, golden, secpar):
    """The golden seeds' packed keys unpack to the golden signing keys and, through ntt_inv, to the golden vk."""
    from lattice_cryptography_b200 import lm_one_time_sigs as lm
    from lattice_cryptography_b200 import wire
    from lattice_cryptography_b200.lattice_algebra import PolynomialVector
    from lattice_cryptography_b200.one_time_keys import SchemeParameters
    arrays, meta = golden
    m = meta['cases'][str(secpar)]
    pp = lm.make_setup_parameters(secpar)
    sp = pp['scheme_parameters']
    key_ch = PolynomialVector(sp.lp, const_time_flag=False, _coef=np.ascontiguousarray(arrays[f's{secpar}_key_ch']))
    pp['scheme_parameters'] = SchemeParameters(secpar=sp.secpar, lp=sp.lp, distribution=sp.distribution, key_ch=key_ch)
    skb = WIDTHS[secpar][0]
    assert wire.signing_key_bits(pp) == skb
    seeds = [c['seed'] for c in m['lm']]
    skp, vkp = wire.keygen_batch_packed(pp, seeds)
    assert skp.shape == (len(seeds), 2, m['l'], 32 * skb)
    sk = wire.unpack_signing_keys(pp, skp)
    vk = wire._engine(pp).ntt_inv(wire.unpack_keys(pp, vkp))
    for j in range(len(seeds)):
        assert np.array_equal(sk[j, 0], arrays[f's{secpar}_lm{j}_skL']) and np.array_equal(sk[j, 1], arrays[f's{secpar}_lm{j}_skR'])
        assert np.array_equal(vk[j, 0], arrays[f's{secpar}_lm{j}_vkL']) and np.array_equal(vk[j, 1], arrays[f's{secpar}_lm{j}_vkR'])
    # random_seed_batch output is accepted as it is by keygen_batch
    blob_off = lm.random_seed_batch(pp, 5, secret=bytes(range(32)))
    skp2, vkp2 = wire.keygen_batch_packed(pp, blob_off)
    keys = lm.keygen_batch(pp, blob_off)
    assert np.array_equal(skp2, wire.pack_signing_keys(pp, keys['sk_coef'])[0])
    assert np.array_equal(vkp2, wire.pack_keys(pp, keys['vk_ntt']))


# ------------------------------------------------------------------------------------------- sign
@pytest.mark.parametrize('n', [1, 7, 8, 9, 2049, 6151])
@pytest.mark.parametrize('secpar', [128, 256])
def test_sign_packed_sk_equals_composition(engines, secpar, n):
    """Genuine keys, and about a third of the items with uniformly random key bytes, under every sk bias and sig bias."""
    e = engines[secpar]
    sch = scheme(secpar)
    skb, sb, _, pvf_bd, vf_bd = WIDTHS[secpar]
    sk_bd = SHIPPED[secpar]['sk_bd']
    seeds = _seeds(secpar, n, 3 * secpar + n)
    msgs = _msgs(n, n)
    skp, _, _ = e.lm_keygen_packed(sch, seeds, skb, sk_bd, 14, want_vk=False)
    rng = np.random.default_rng(n)
    rnd = rng.random(n) < 0.3
    skp[rnd] = rng.integers(0, 256, (int(rnd.sum()),) + skp.shape[1:], dtype=np.uint8)
    for skbias in (sk_bd, 0, 32767):
        for sbias in (vf_bd, pvf_bd, 0, 32767):
            want, want_ok = _composed(e, sch, skp, skb, skbias, msgs, sb, sbias)
            got, ok = e.lm_sign_packed_sk(sch, skp, skb, skbias, msgs, sb, sbias, want_range=True)
            assert np.array_equal(got, want) and np.array_equal(ok, want_ok), (skbias, sbias)
            if skbias == sk_bd and sbias in (vf_bd, pvf_bd):
                assert ok[~rnd].all()
    want, _ = _composed(e, sch, skp, skb, sk_bd, msgs, sb, vf_bd)
    assert np.array_equal(e.lm_sign_packed_sk(sch, skp, skb, sk_bd, msgs, sb, vf_bd), want)     # in_range = NULL


@pytest.mark.parametrize('secpar', [128, 256])
def test_sign_packed_sk_composed_routes(engines, secpar):
    """Widths the kernel does not read or write, and 4-byte aligned caller device buffers: unpack -> ntt_fwd -> sign."""
    import torch
    from lattice_cryptography_b200 import _ffi, ragged
    e = engines[secpar]
    sch = scheme(secpar)
    skb, sb, _, pvf_bd, _ = WIDTHS[secpar]
    sk_bd = SHIPPED[secpar]['sk_bd']
    l = SHIPPED[secpar]['l']
    n = 777
    seeds = _seeds(secpar, n, 11 * secpar)
    msgs = _msgs(n, 12)
    sk_coef, _, _, _ = e.lm_keygen(sch, seeds, want_sk_ntt=False, want_vk_ntt=False, want_vk_coef=False)
    rng = np.random.default_rng(3)
    for kbits, kbias, sbits, sbias in ((9, 300, sb, pvf_bd), (16, 0, sb, 0), (16, 32767, sb, 32767), (skb, sk_bd, 12, pvf_bd),
                                       (skb, 0, 12, 32767)):
        skp = e.pack(sk_coef, kbits, kbias)
        skp[::7] = rng.integers(0, 256, skp[::7].shape, dtype=np.uint8)
        want, want_ok = _composed(e, sch, skp, kbits, kbias, msgs, sbits, sbias)
        got, ok = e.lm_sign_packed_sk(sch, skp, kbits, kbias, msgs, sbits, sbias, want_range=True)
        assert np.array_equal(got, want) and np.array_equal(ok, want_ok), (kbits, kbias, sbits, sbias)
    # 4-byte aligned device buffers for the keys, then for the signatures, at the shipped widths
    skp = e.pack(sk_coef, skb, sk_bd)
    skp[::5] = rng.integers(0, 256, skp[::5].shape, dtype=np.uint8)
    want, want_ok = _composed(e, sch, skp, skb, sk_bd, msgs, sb, pvf_bd)
    blob, off = ragged(msgs)
    d_blob, d_off = (torch.from_numpy(np.array(x)).cuda() for x in (blob, off))
    lib = _ffi.load()
    for mis_key in (True, False):
        d_sk = _misaligned(skp) if mis_key else torch.from_numpy(skp).cuda()
        out = torch.zeros(want.size, dtype=torch.uint8, device='cuda') if mis_key else _misaligned(np.zeros(want.shape, np.uint8))
        rng_d = torch.zeros(n * l, dtype=torch.uint8, device='cuda')
        torch.cuda.synchronize()
        assert lib.lcb_lm_sign_packed_sk_batch(e._ctx, byref(sch), c_void_p(d_sk.data_ptr()), skb, sk_bd,
                                               c_void_p(d_blob.data_ptr()), c_void_p(d_off.data_ptr()), n, sb, pvf_bd,
                                               c_void_p(out.data_ptr()), c_void_p(rng_d.data_ptr())) == _ffi.LCB_OK
        e.synchronize()
        assert np.array_equal(out.cpu().numpy().reshape(want.shape), want), mis_key
        assert np.array_equal(rng_d.cpu().numpy().reshape(n, l), want_ok), mis_key
    # aligned device buffers: the fused route, asynchronous
    got, ok = e.lm_sign_packed_sk(sch, torch.from_numpy(skp).cuda(), skb, sk_bd, (d_blob, d_off), sb, pvf_bd, device=True,
                                  want_range=True)
    e.synchronize()
    assert np.array_equal(got.cpu().numpy(), want) and np.array_equal(ok.cpu().numpy(), want_ok)


# ------------------------------------------------------------------------------------------- independent reference
@pytest.mark.parametrize('secpar', [128, 256])
def test_sign_packed_sk_independent_reference(engines, secpar):
    """A few hundred items against numpy, worst-case rows (every field 0 or 2^bits - 1 under biases 0 and 32767), and a
    subsample against the C oracle's lm_sign."""
    import c_oracle
    import wire as owire
    e = engines[secpar]
    sch = scheme(secpar)
    skb, sb, _, pvf_bd, vf_bd = WIDTHS[secpar]
    p = SHIPPED[secpar]
    q, l, sk_bd = p['q'], p['l'], p['sk_bd']
    n = 300
    seeds = _seeds(secpar, n, 17 * secpar)
    msgs = _msgs(n, 19)
    skp, _, _ = e.lm_keygen_packed(sch, seeds, skb, sk_bd, 14, want_vk=False)
    rng = np.random.default_rng(23)
    skp[100:200] = rng.integers(0, 256, skp[100:200].shape, dtype=np.uint8)
    top = (1 << skb) - 1
    fields = np.zeros((n, 2, l, D), np.int64)
    fields[200:225] = top                                    # every field at its maximum
    fields[225:235, 0] = top                                 # left at the maximum, right 0
    fields[235:245, 1] = top
    fields[245:250, 0, :, ::2] = top                         # alternating extremes
    ext = owire.pack(fields[200:250].astype(np.uint16), skb, 0)[0]   # bias 0 packs the fields as they are
    skp[200:250] = ext
    # 250..299: all fields 0
    skp[250:] = 0
    for skbias in (sk_bd, 0, 32767):
        want = _numpy_sign(e, sch, skp, skb, skbias, msgs, q)
        for sbias in (vf_bd, 0, 32767):
            got, ok = e.lm_sign_packed_sk(sch, skp, skb, skbias, msgs, sb, sbias, want_range=True)
            wpk, wok = owire.pack(want, sb, sbias)
            assert np.array_equal(got, wpk) and np.array_equal(ok, wok), (skbias, sbias)
    # genuine keys against the C oracle
    cp = c_oracle.params(secpar, q, l, sk_bd, p['ch_wt'])
    skc = owire.unpack(skp[:12], skb, sk_bd)
    got = owire.unpack(e.lm_sign_packed_sk(sch, skp[:12], skb, sk_bd, msgs[:12], sb, vf_bd), sb, vf_bd)
    for j in range(12):
        assert np.array_equal(got[j], c_oracle.lm_sign(cp, skc[j, 0], skc[j, 1], msgs[j])), j


@pytest.mark.parametrize('ch_bd, ch_wt', [(1, 256), (1, 3), (2, 20), (32767, 100)])
def test_sign_packed_sk_other_challenges(engines, ch_bd, ch_wt):
    """Schemes the shipped tables do not use: the widest monomial challenge (ch_wt = d, the fused kernel's 16-bit lane sums
    at their largest), a narrow one, and non-monomial challenges, up to ch_wt * ch_bd far beyond the int32 range of an
    exact 16-bit-coefficient accumulation (these take the composed route)."""
    from lattice_cryptography_b200 import make_scheme
    import wire as owire
    e = engines[128]
    q, l = SHIPPED[128]['q'], SHIPPED[128]['l']
    sch = make_scheme(sk_bd=127, sk_wt=256, ch_bd=ch_bd, ch_wt=ch_wt)
    n = 40
    rng = np.random.default_rng(ch_wt)
    skp = rng.integers(0, 256, (n, 2, l, 256), dtype=np.uint8)
    skp[:8] = 255
    msgs = _msgs(n, ch_bd)
    for skbias in (0, 127, 32767):
        want = _numpy_sign(e, sch, skp, 8, skbias, msgs, q)
        for sb, sbias in ((11, 0), (13, 4000), (16, 32767)):
            got, ok = e.lm_sign_packed_sk(sch, skp, 8, skbias, msgs, sb, sbias, want_range=True)
            wpk, wok = owire.pack(want, sb, sbias)
            assert np.array_equal(got, wpk) and np.array_equal(ok, wok), (skbias, sb, sbias)


# ------------------------------------------------------------------------------------------- round trips through `wire`
@pytest.mark.parametrize('secpar', [128, 256])
def test_packed_lifecycle_round_trips(engines, secpar):
    from lattice_cryptography_b200 import adaptor_sigs as ad
    from lattice_cryptography_b200 import lm_one_time_sigs as lm
    from lattice_cryptography_b200 import wire
    n = 64
    pp = wire.setup_parameters_from_seed(lm.make_setup_parameters, secpar, 'packed keys')
    skp, vkp = wire.keygen_batch_packed(pp, [bin(5 * i + 2)[2:].zfill(secpar) for i in range(n)])
    chm = [f'<vk {i}>, message {i}' for i in range(n)]
    sig, ok = wire.sign_batch_packed_sk(pp, skp, chm)
    assert ok.all()
    assert wire.verify_batch_packed(pp, vkp, chm, sig).tolist() == [1] * n
    bad = sig.copy()
    bad[5, 3, 17] ^= 0x10
    assert wire.verify_batch_packed(pp, vkp, chm, bad).tolist() == [1] * 5 + [0] + [1] * (n - 6)
    skb = skp.copy()
    skb[9, 0, 2, 40] ^= 0x01                                  # one byte of one signing key
    sig2, _ = wire.sign_batch_packed_sk(pp, skb, chm)
    assert wire.verify_batch_packed(pp, vkp, chm, sig2).tolist() == [1] * 9 + [0] + [1] * (n - 10)
    vkb = vkp.copy()
    vkb[11, 1, 3] ^= 0x04                                     # one byte of one verification key
    assert wire.verify_batch_packed(pp, vkb, chm, sig).tolist() == [1] * 11 + [0] + [1] * (n - 12)
    # the adaptor chain
    app = wire.setup_parameters_from_seed(ad.make_setup_parameters, secpar, 'packed keys adaptor')
    askp, avkp = wire.keygen_batch_packed(app, [bin(7 * i + 3)[2:].zfill(secpar) for i in range(n)])
    wits = ad.witgen_batch(app, [bin(11 * i + 5)[2:].zfill(secpar) for i in range(n)])
    stp = wire.pack_keys(app, wits['st_ntt'])
    presig, ok = wire.presign_batch_packed_sk(app, askp, chm)
    assert ok.all()
    assert wire.preverify_batch_packed(app, avkp, chm, presig).tolist() == [1] * n
    asig, ok = wire.adapt_batch_packed(app, presig, wits['wit_coef'])
    assert ok.all()
    assert wire.adaptor_verify_batch_packed(app, avkp, chm, stp, asig).tolist() == [1] * n
    assert np.array_equal(wire.extract_batch_packed(app, presig, asig), wits['wit_coef'])


# ------------------------------------------------------------------------------------------- argument errors
def test_argument_errors(engines):
    import torch
    from lattice_cryptography_b200 import Engine, LcbError, _ffi, ragged
    e = engines[128]
    sch = scheme(128)
    seeds = _seeds(128, 3, 1)
    msgs = _msgs(3, 1)
    skp, _, _ = e.lm_keygen_packed(sch, seeds, 7, 45, 14, want_vk=False)

    def invalid(fn):
        with pytest.raises(LcbError) as x:
            fn()
        assert x.value.status == _ffi.LCB_ERR_INVALID

    for bits in (0, 17):
        invalid(lambda: e.lm_keygen_packed(sch, seeds, bits, 0, 14))
        invalid(lambda: e.lm_keygen_packed(sch, seeds, 7, 45, bits))
        invalid(lambda: e.lm_sign_packed_sk(sch, np.zeros((3, 2, 13, 32 * bits), np.uint8), bits, 0, msgs, 11, 945))
        invalid(lambda: e.lm_sign_packed_sk(sch, skp, 7, 45, msgs, bits, 0))
    for bias in (-1, 32768):
        invalid(lambda: e.lm_keygen_packed(sch, seeds, 7, bias, 14))
        invalid(lambda: e.lm_sign_packed_sk(sch, skp, 7, bias, msgs, 11, 945))
        invalid(lambda: e.lm_sign_packed_sk(sch, skp, 7, 45, msgs, 11, bias))
    invalid(lambda: e.lm_keygen_packed(sch, seeds, 7, 45, 14, want_sk=False, want_vk=False))
    # packed buffers that are only 2-byte aligned
    half = lambda x: torch.zeros(x.size + 16, dtype=torch.uint8, device='cuda')[2:2 + x.size].view(*x.shape)
    torch.cuda.synchronize()
    invalid(lambda: e.lm_sign_packed_sk(sch, half(skp), 7, 45, msgs, 11, 945))
    lib = _ffi.load()
    blob, off = ragged(msgs)
    P = lambda a: c_void_p(a.ctypes.data)
    out = half(np.zeros((3, 13, 352), np.uint8))
    torch.cuda.synchronize()
    assert lib.lcb_lm_sign_packed_sk_batch(e._ctx, byref(sch), P(skp), 7, 45, P(blob), P(off), 3, 11, 945,
                                           c_void_p(out.data_ptr()), None) == _ffi.LCB_ERR_INVALID
    assert lib.lcb_lm_keygen_packed_batch(e._ctx, byref(sch), P(blob), P(off), 3, 7, 45, c_void_p(out.data_ptr()), None, 14,
                                          None) == _ffi.LCB_ERR_INVALID
    z, zo = np.zeros(16, np.uint8), np.zeros(4, np.int64)
    assert lib.lcb_lm_sign_packed_sk_batch(e._ctx, byref(sch), P(z), 7, 45, P(z), P(zo), (1 << 30) + 1, 11, 945, P(z),
                                           None) == _ffi.LCB_ERR_INVALID
    assert b'2^30' in lib.lcb_last_error(e._ctx)
    assert lib.lcb_lm_sign_packed_sk_batch(e._ctx, byref(sch), P(z), 7, 45, None, P(zo), 0, 11, 945, P(z), None) == _ffi.LCB_OK
    # generic (d = 512) and wide (q >= 2^16) contexts
    gsch = _ffi.LcbScheme()
    gsch.ch_bd = gsch.ch_wt = gsch.sk_bd = gsch.sk_wt = 1
    for q, d in ((12289, 512), (65537, 256)):
        g = Engine(128, q, d, 2)
        try:
            g.set_key_ch(np.zeros((2, d), np.int32 if q >= 65536 else np.int16))
            for fn in (lambda: g.lm_keygen_packed(gsch, ['0' * 128], 7, 45, 14),
                       lambda: g.lm_sign_packed_sk(gsch, np.zeros((1, 2, 2, d * 7 // 8), np.uint8), 7, 45, [b'x'], 11, 945)):
                with pytest.raises(LcbError) as x:
                    fn()
                assert x.value.status == _ffi.LCB_ERR_INVALID and 'd == 256' in str(x.value)
        finally:
            g.close()


# ------------------------------------------------------------------------------------------- checked build
def test_small_cases(engines):
    """A small case of both calls on both routes (the checked build runs it)."""
    e = engines[256]
    sch = scheme(256)
    seeds, msgs = _seeds(256, 37, 4), _msgs(37, 4)
    sk_coef, _, vk_ntt, _ = e.lm_keygen(sch, seeds, want_sk_ntt=False, want_vk_coef=False)
    skp, _, vkp = e.lm_keygen_packed(sch, seeds, 8, 65, 16)
    assert np.array_equal(skp, e.pack(sk_coef, 8, 65)) and np.array_equal(vkp, e.pack(vk_ntt, 16, 0))
    for kbits, sbits in ((8, 13), (8, 12), (9, 13)):
        k = e.pack(sk_coef, kbits, 65)
        want, want_ok = _composed(e, sch, k, kbits, 65, msgs, sbits, 3315)
        got, ok = e.lm_sign_packed_sk(sch, k, kbits, 65, msgs, sbits, 3315, want_range=True)
        assert np.array_equal(got, want) and np.array_equal(ok, want_ok)
        assert ok.all() == (sbits == 13)             # 12 bits cannot hold +-vf_bd = +-3315


def test_packed_keys_pass_on_the_checked_build():
    from lattice_cryptography_b200 import _ffi
    if _ffi.load().lcb_build_is_checked():
        pytest.skip('already running on the checked build')
    lib = os.path.join(ROOT, 'lattice_cryptography_b200', 'liblcb200_checked.so')
    if not os.path.exists(lib):
        subprocess.run(['make', '-C', os.path.join(ROOT, 'lattice_cryptography_b200', 'csrc'), '-j4', 'CHECKED=1'], check=True,
                       capture_output=True)
    env = dict(os.environ, LCB200_LIB=lib)
    r = subprocess.run([sys.executable, '-m', 'pytest', 'tests/test_gpu_packed_keys.py', '-q', '-x', '-m', 'gpu', '-k',
                        'small_cases or (sign_packed_sk_equals_composition and 2049)', '-p', 'no:cacheprovider'],
                       env=env, capture_output=True, text=True, timeout=1500, cwd=ROOT)
    tail = r.stdout[-2500:] + r.stderr[-1500:]
    assert r.returncode == 0, tail
    assert '3 passed' in r.stdout and 'failed' not in r.stdout, tail
