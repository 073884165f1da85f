"""Signing and the adaptor protocol on the packed wire format (include/lcb200.h: lcb_lm_sign_packed_batch,
lcb_adaptor_verify_packed_batch, lcb_adaptor_adapt_packed_batch, lcb_adaptor_extract_packed_batch), compared bit for
bit with the composition each call is defined as: sign -> pack, unpack -> verify(st_ntt), unpack -> add -> pack,
unpack -> sub.  Both routes of each fused call run: the shipped widths from 16-byte aligned buffers (the kernels
read and write the packed rows) and everything else (unpacked or packed in engine scratch)."""
import os
import subprocess
import sys
from ctypes import byref, c_void_p

import numpy as np
import pytest

from test_gpu_parity import D, SHIPPED, engines, scheme   # noqa: F401  (fixture re-export)

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# signature bits, key bits, pvf_bd (presignatures; LM vf_bd), vf_bd (adaptor signatures)
WIDTHS = {128: (11, 14, 945, 946), 256: (13, 16, 3315, 3316)}


def _items(e, sch, secpar, n, seed):
    rng = np.random.default_rng(seed)
    seeds = [''.join(rng.choice(['0', '1'], secpar)) for _ in range(n)]
    msgs = [bytes(rng.integers(1, 256, int(rng.integers(0, 120)), dtype=np.uint8)) for _ in range(n)]
    _, sk_ntt, vk_ntt, _ = e.lm_keygen(sch, seeds, want_sk_coef=False, want_vk_coef=False)
    return sk_ntt, vk_ntt, msgs


def _misaligned(x):
    """A device copy of x that is 4-byte but not 16-byte aligned."""
    import torch
    flat = torch.from_numpy(np.ascontiguousarray(x).reshape(-1).view(np.uint8)).cuda()
    raw = torch.zeros(flat.numel() + 16, dtype=torch.uint8, device='cuda')
    view = raw[4:4 + flat.numel()]
    view.copy_(flat)
    assert view.data_ptr() % 16 == 4
    return view.view(*x.shape) if x.dtype == np.uint8 else view


# ------------------------------------------------------------------------------------------- sign
@pytest.mark.parametrize('n', [1, 7, 8, 9, 2049, 6151])
@pytest.mark.parametrize('secpar', [128, 256])
def test_sign_packed_equals_sign_then_pack(engines, secpar, n):
    """n = 6151 is more than one persistent grid of k_sign (148 SMs x 4 blocks x 8 half-warps); about a third of the
    items sign with uniformly random sk_ntt slots (values >= q included), whose rows are out of range."""
    e = engines[secpar]
    sch = scheme(secpar)
    sb, _, pvf_bd, vf_bd = WIDTHS[secpar]
    sk, _, msgs = _items(e, sch, secpar, n, secpar + n)
    rng = np.random.default_rng(n)
    rnd = rng.random(n) < 0.3
    sk[rnd] = rng.integers(0, 1 << 16, (int(rnd.sum()), 2, SHIPPED[secpar]['l'], D), dtype=np.uint16)
    sig = e.lm_sign(sch, sk, msgs)
    for bias in (pvf_bd, vf_bd, 0, 32767):     # the shipped biases, then both ends of the bias range
        want, want_ok = e.pack(sig, sb, bias, want_range=True)
        got, ok = e.lm_sign_packed(sch, sk, msgs, sb, bias, want_range=True)
        assert np.array_equal(got, want) and np.array_equal(ok, want_ok), bias
        if bias in (pvf_bd, vf_bd):             # genuine keys fit the shipped packings
            assert ok[~rnd].all() and (not rnd.any() or not ok[rnd].all())
        assert np.array_equal(e.lm_sign_packed(sch, sk, msgs, sb, bias), want)          # in_range = NULL


@pytest.mark.parametrize('secpar', [128, 256])
def test_sign_packed_device_buffers_and_composed_route(engines, secpar):
    import torch
    from lattice_cryptography_b200 import _ffi, ragged
    e = engines[secpar]
    sch = scheme(secpar)
    sb, _, pvf_bd, _ = WIDTHS[secpar]
    l = SHIPPED[secpar]['l']
    n = 777
    sk, _, msgs = _items(e, sch, secpar, n, 7 * secpar)
    rng = np.random.default_rng(3)
    sk[::5] = rng.integers(0, 1 << 16, sk[::5].shape, dtype=np.uint16)
    sig = e.lm_sign(sch, sk, msgs)
    blob, off = ragged(msgs)
    d_sk, d_blob, d_off = (torch.from_numpy(np.array(x)).cuda() for x in (sk, blob, off))
    torch.cuda.synchronize()
    got, ok = e.lm_sign_packed(sch, d_sk, (d_blob, d_off), sb, pvf_bd, device=True, want_range=True)
    e.synchronize()
    want, want_ok = e.pack(sig, sb, pvf_bd, want_range=True)
    assert np.array_equal(got.cpu().numpy(), want) and np.array_equal(ok.cpu().numpy(), want_ok)
    assert not want_ok.all() and want_ok.any()
    # widths the kernel does not write: sign into scratch, then pack
    for bits, bias in ((12, pvf_bd), (16, 0), (16, 32767), (sb + 1, 0)):
        want, want_ok = e.pack(sig, bits, bias, want_range=True)
        got, ok = e.lm_sign_packed(sch, sk, msgs, bits, bias, want_range=True)
        assert np.array_equal(got, want) and np.array_equal(ok, want_ok), (bits, bias)
    # a 4-byte aligned caller device buffer at a shipped width: the composed route
    want, want_ok = e.pack(sig, sb, pvf_bd, want_range=True)
    out = _misaligned(np.zeros(want.shape, np.uint8))
    rng_d = torch.zeros(n * l, dtype=torch.uint8, device='cuda')
    torch.cuda.synchronize()
    lib = _ffi.load()
    assert lib.lcb_lm_sign_packed_batch(e._ctx, byref(sch), c_void_p(d_sk.data_ptr()), c_void_p(d_blob.data_ptr()),
                                        c_void_p(d_off.data_ptr()), n, sb, pvf_bd, c_void_p(out.data_ptr()),
                                        c_void_p(rng_d.data_ptr())) == _ffi.LCB_OK
    e.synchronize()
    assert np.array_equal(out.cpu().numpy(), want) and np.array_equal(rng_d.cpu().numpy().reshape(n, l), want_ok)


# ------------------------------------------------------------------------------------------- adaptor verify
def _adaptor_world(e, sch, secpar, n, seed):
    sk, vk, msgs = _items(e, sch, secpar, n, seed)
    rng = np.random.default_rng(seed + 1)
    wit, st_ntt, _ = e.witgen(sch, [''.join(rng.choice(['0', '1'], secpar)) for _ in range(n)], want_st_coef=False)
    presig = e.lm_sign(sch, sk, msgs)
    return vk, msgs, e.vec_add(presig, wit), st_ntt


def _ref_verify(e, sch, vkp, kb, msgs, sigp, sb, sbias, stp, stb, bd, wt):
    vk = e.unpack(vkp, kb, 0, dtype=np.uint16)
    sig = e.unpack(sigp, sb, sbias)
    st = e.unpack(stp, stb, 0, dtype=np.uint16)
    return e.lm_verify(sch, vk, msgs, sig, bd, wt, st_ntt=st)


@pytest.mark.parametrize('secpar', [128, 256])
def test_adaptor_verify_packed_equals_unpack_then_verify(engines, secpar):
    import torch
    e = engines[secpar]
    sch = scheme(secpar)
    sb, kb, _, vf_bd = WIDTHS[secpar]
    q, l = SHIPPED[secpar]['q'], SHIPPED[secpar]['l']
    n = 600
    vk, msgs, sig, st = _adaptor_world(e, sch, secpar, n, 11 * secpar)
    rng = np.random.default_rng(secpar)
    sig, st, msgs = sig.copy(), st.copy(), list(msgs)
    kind = np.arange(n) % 6                 # 0 genuine, 1 statement slot + 1, 2 coefficient + 1, 3 message byte,
    for i in range(n):                      # 4 a coefficient at vf_bd, 5 a coefficient at vf_bd + 1
        a, b = int(rng.integers(0, l)), int(rng.integers(0, D))
        if kind[i] == 1:
            st[i, b] = (int(st[i, b]) + 1) % q
        elif kind[i] == 2:
            sig[i, a, b] += 1
        elif kind[i] == 3:
            msgs[i] = msgs[i] + b'\x01' if not msgs[i] else bytes([msgs[i][0] ^ 1]) + msgs[i][1:]
        elif kind[i] == 4:
            sig[i, a, b] = vf_bd * int(rng.choice([-1, 1]))
        elif kind[i] == 5:                  # -(vf_bd + 1) has no field under bias vf_bd; + (vf_bd + 1) has one
            sig[i, a, b] = vf_bd + 1
    want = e.lm_verify(sch, vk, msgs, sig, vf_bd, 256, st_ntt=st)
    assert want[kind == 0].all() and not want[(kind == 1) | (kind == 2) | (kind == 3) | (kind == 5)].any()
    vkp, stp = e.pack(vk, kb, 0), e.pack(st, kb, 0)
    sigp, ok = e.pack(sig, sb, vf_bd, want_range=True)
    assert ok.all()
    got = e.adaptor_verify_packed(sch, vkp, kb, msgs, sigp, sb, vf_bd, stp, kb, vf_bd, 256)
    assert np.array_equal(got, want)
    # device buffers (fused) and 4-byte aligned device buffers (composed)
    d = [torch.from_numpy(x).cuda() for x in (vkp, sigp, stp)]
    torch.cuda.synchronize()
    got = e.adaptor_verify_packed(sch, d[0], kb, msgs, d[1], sb, vf_bd, d[2], kb, vf_bd, 256, device=True)
    e.synchronize()
    assert np.array_equal(got.cpu().numpy(), want)
    m = [_misaligned(x) for x in (vkp, sigp, stp)]
    torch.cuda.synchronize()
    got = e.adaptor_verify_packed(sch, m[0], kb, msgs, m[1], sb, vf_bd, m[2], kb, vf_bd, 256, device=True)
    e.synchronize()
    assert np.array_equal(got.cpu().numpy(), want)
    # wt < d: the weight-checking instantiations, against the composition
    for wt in (200, 255):
        w2 = e.lm_verify(sch, vk, msgs, sig, vf_bd, wt, st_ntt=st)
        assert np.array_equal(e.adaptor_verify_packed(sch, vkp, kb, msgs, sigp, sb, vf_bd, stp, kb, vf_bd, wt), w2), wt
    # statements and keys at other widths (st_bits != vk_bits and non-shipped widths): the composed route
    for k2, s2 in ((kb, kb + 1 if kb < 16 else 15), (15, 15), (16, 16)):
        if (k2, s2) == (kb, kb):
            continue
        vk2, st2 = e.pack(vk, k2, 0), e.pack(st, s2, 0)
        got = e.adaptor_verify_packed(sch, vk2, k2, msgs, sigp, sb, vf_bd, st2, s2, vf_bd, 256)
        assert np.array_equal(got, _ref_verify(e, sch, vk2, k2, msgs, sigp, sb, vf_bd, st2, s2, vf_bd, 256)), (k2, s2)
        if min(k2, s2) >= kb:                   # wide enough for every slot < q
            assert np.array_equal(got, want), (k2, s2)
    # statement slots >= q (only the 16-bit packing holds them at secpar 256; 14 bits hold up to 16383 > 11777)
    st_hi = st.copy()
    rows = np.arange(0, n, 7)
    st_hi[rows, 5] = np.uint16((1 << kb) - 1 - (rows % 3))
    stp_hi = e.pack(st_hi, kb, 0)
    want_hi = _ref_verify(e, sch, vkp, kb, msgs, sigp, sb, vf_bd, stp_hi, kb, vf_bd, 256)
    assert np.array_equal(e.adaptor_verify_packed(sch, vkp, kb, msgs, sigp, sb, vf_bd, stp_hi, kb, vf_bd, 256), want_hi)
    ms = _misaligned(stp_hi)
    torch.cuda.synchronize()
    got = e.adaptor_verify_packed(sch, vkp, kb, msgs, sigp, sb, vf_bd, ms, kb, vf_bd, 256)
    assert np.array_equal(got, want_hi)


@pytest.mark.parametrize('secpar', [128, 256])
def test_adaptor_verify_packed_random_bytes(engines, secpar):
    import torch
    e = engines[secpar]
    sch = scheme(secpar)
    sb, kb, _, vf_bd = WIDTHS[secpar]
    n = 513
    vk, msgs, sig, st = _adaptor_world(e, sch, secpar, n, 5 * secpar)
    rng = np.random.default_rng(77)
    vkp, stp = e.pack(vk, kb, 0), e.pack(st, kb, 0)
    sigp = e.pack(sig, sb, vf_bd)
    # random key bytes, statement bytes and signature bytes, each in its own set of items
    vkp[0::3] = rng.integers(0, 256, vkp[0::3].shape, dtype=np.uint8)
    stp[1::3] = rng.integers(0, 256, stp[1::3].shape, dtype=np.uint8)
    sigp[2::5] = rng.integers(0, 256, sigp[2::5].shape, dtype=np.uint8)
    for bias in (vf_bd, 0, 32767):
        want = _ref_verify(e, sch, vkp, kb, msgs, sigp, sb, bias, stp, kb, vf_bd, 256)
        assert np.array_equal(e.adaptor_verify_packed(sch, vkp, kb, msgs, sigp, sb, bias, stp, kb, vf_bd, 256), want), bias
        m = [_misaligned(x) for x in (vkp, sigp, stp)]
        torch.cuda.synchronize()
        got = e.adaptor_verify_packed(sch, m[0], kb, msgs, m[1], sb, bias, m[2], kb, vf_bd, 256, device=True)
        e.synchronize()
        assert np.array_equal(got.cpu().numpy(), want), bias
    honest = np.setdiff1d(np.arange(n), np.concatenate([np.arange(0, n, 3), np.arange(1, n, 3), np.arange(2, n, 5)]))
    assert _ref_verify(e, sch, vkp, kb, msgs, sigp, sb, vf_bd, stp, kb, vf_bd, 256)[honest].all()


def test_adaptor_verify_packed_host_pipeline(engines):
    """Host-resident packed signatures cross PCIe in 2^18-item chunks: more than one chunk, ragged tail, tampers in
    every chunk - verdicts equal the all-device call and the int16 composition."""
    import torch
    from lattice_cryptography_b200 import ragged
    e = engines[128]
    sch = scheme(128)
    sb, kb, _, vf_bd = WIDTHS[128]
    n0 = 1024
    vk, msgs, sig, st = _adaptor_world(e, sch, 128, n0, 99)
    sig = sig.copy()
    sig[3::17, 0, 9] += 1
    want0 = e.lm_verify(sch, vk, msgs, sig, vf_bd, 256, st_ntt=st)
    reps = ((1 << 18) + 4099 + n0 - 1) // n0
    n = (1 << 18) + 4099
    vkp = np.ascontiguousarray(np.tile(e.pack(vk, kb, 0), (reps, 1, 1))[:n])
    stp = np.ascontiguousarray(np.tile(e.pack(st, kb, 0), (reps, 1))[:n])
    sigp = np.ascontiguousarray(np.tile(e.pack(sig, sb, vf_bd), (reps, 1, 1))[:n])
    blob, off = ragged((msgs * reps)[:n])
    want = np.tile(want0, reps)[:n]
    got = e.adaptor_verify_packed(sch, vkp, kb, (blob, off), sigp, sb, vf_bd, stp, kb, vf_bd, 256)
    assert np.array_equal(got, want)
    d = [torch.from_numpy(np.array(x)).cuda() for x in (vkp, sigp, stp, blob, off)]
    torch.cuda.synchronize()
    got = e.adaptor_verify_packed(sch, d[0], kb, (d[3], d[4]), d[1], sb, vf_bd, d[2], kb, vf_bd, 256, device=True)
    e.synchronize()
    assert np.array_equal(got.cpu().numpy(), want)


# ------------------------------------------------------------------------------------------- adapt / extract
@pytest.mark.parametrize('bits', [1, 2, 11, 12, 13, 16])
def test_adapt_extract_packed_equal_composition(engines, bits):
    e = engines[128]
    q = SHIPPED[128]['q']
    rng = np.random.default_rng(bits)
    npoly = 2049
    wit = rng.integers(-(q // 2), q // 2 + 1, (npoly, D)).astype(np.int16)
    for bias in (0, 946, 32767):
        pre = rng.integers(0, 256, (npoly, 32 * bits), dtype=np.uint8)
        sig = rng.integers(0, 256, (npoly, 32 * bits), dtype=np.uint8)
        want, want_ok = e.pack(e.vec_add(e.unpack(pre, bits, bias), wit), bits, bias, want_range=True)
        got, ok = e.adapt_packed(pre, bits, bias, wit, bits, bias, want_range=True)
        assert np.array_equal(got, want) and np.array_equal(ok, want_ok), bias
        assert np.array_equal(e.adapt_packed(pre, bits, bias, wit, bits, bias), want)
        want = e.vec_sub(e.unpack(sig, bits, bias), e.unpack(pre, bits, bias))
        assert np.array_equal(e.extract_packed(sig, bits, bias, pre, bits, bias), want), bias
    # mixed widths (presignature and signature at different widths and biases), as the shipped packings are
    pre = rng.integers(0, 256, (npoly, 32 * bits), dtype=np.uint8)
    want = e.pack(e.vec_add(e.unpack(pre, bits, 0), wit), 13, 3316)
    assert np.array_equal(e.adapt_packed(pre, bits, 0, wit, 13, 3316), want)
    sig = rng.integers(0, 256, (npoly, 32 * 13), dtype=np.uint8)
    want = e.vec_sub(e.unpack(sig, 13, 3316), e.unpack(pre, bits, 0))
    assert np.array_equal(e.extract_packed(sig, 13, 3316, pre, bits, 0), want)


def test_adapt_extract_packed_device_buffers(engines):
    import torch
    e = engines[256]
    rng = np.random.default_rng(9)
    l = SHIPPED[256]['l']
    wit = rng.integers(-1, 2, (40, l, D)).astype(np.int16)
    pre = rng.integers(0, 256, (40, l, 32 * 13), dtype=np.uint8)
    want, want_ok = e.adapt_packed(pre, 13, 3315, wit, 13, 3316, want_range=True)
    d_pre, d_wit = torch.from_numpy(pre).cuda(), torch.from_numpy(wit).cuda()
    torch.cuda.synchronize()
    got, ok = e.adapt_packed(d_pre, 13, 3315, d_wit, 13, 3316, device=True, want_range=True)
    e.synchronize()
    assert np.array_equal(got.cpu().numpy(), want) and np.array_equal(ok.cpu().numpy(), want_ok)
    m_pre = _misaligned(pre)
    torch.cuda.synchronize()
    ext = e.extract_packed(_misaligned(want), 13, 3316, m_pre, 13, 3315, device=True)
    e.synchronize()
    assert np.array_equal(ext.cpu().numpy(), e.extract_packed(want, 13, 3316, pre, 13, 3315))


# ------------------------------------------------------------------------------------------- the protocol through `wire`
@pytest.mark.parametrize('secpar', [128, 256])
def test_wire_protocol_equals_golden_adaptor(golden, secpar):
    """witgen -> pack_keys(st) -> presign -> preverify -> adapt -> verify -> extract -> witness_verify on packed records,
    verdict for verdict and coefficient for coefficient the golden adaptor case."""
    from lattice_cryptography_b200 import adaptor_sigs as ad
    from lattice_cryptography_b200 import wire
    from lattice_cryptography_b200.lattice_algebra import PolynomialVector
    from lattice_cryptography_b200.one_time_keys import SchemeParameters
    arrays, meta = golden
    m = meta['cases'][str(secpar)]
    cases = m['adaptor']
    pp = ad.make_setup_parameters(secpar)
    sp = pp['scheme_parameters']
    key_ch = PolynomialVector(sp.lp, const_time_flag=False, _coef=np.ascontiguousarray(arrays[f's{secpar}_key_ch']))
    pp['scheme_parameters'] = SchemeParameters(secpar=sp.secpar, lp=sp.lp, distribution=sp.distribution, key_ch=key_ch)
    for k, v in m['adaptor_params'].items():
        assert pp[k] == v, k
    sb, kb, pvf_bd, vf_bd = WIDTHS[secpar]
    assert (wire.sig_bits(pp, 'pvf_bd'), wire.sig_bits(pp), wire.key_bits(pp)) == (sb, sb, kb)
    keys = ad.keygen_batch(pp, [m['lm'][c['key_index']]['seed'] for c in cases])
    wits = ad.witgen_batch(pp, [c['wit_seed'] for c in cases])
    chmsgs = [c['chmsg'] for c in cases]
    eng = wire._engine(pp)
    stp = wire.pack_keys(pp, wits['st_ntt'])
    vkp = wire.pack_keys(pp, keys['vk_ntt'])
    presig_p, ok = wire.presign_batch_packed(pp, keys['sk_ntt'], chmsgs)
    assert ok.all()
    gold = lambda name: np.ascontiguousarray(np.stack([arrays[f's{secpar}_ad{j}_{name}'] for j in range(len(cases))]))
    assert np.array_equal(presig_p, eng.pack(gold('presig'), sb, pvf_bd))
    assert wire.preverify_batch_packed(pp, vkp, chmsgs, presig_p).tolist() == [int(c['preverify']) for c in cases]
    sig_p, ok = wire.adapt_batch_packed(pp, presig_p, wits['wit_coef'])
    assert ok.all() and np.array_equal(sig_p, eng.pack(gold('sig'), sb, vf_bd))
    assert wire.adaptor_verify_batch_packed(pp, vkp, chmsgs, stp, sig_p).tolist() == [int(c['verify']) for c in cases]
    ext = wire.extract_batch_packed(pp, presig_p, sig_p)
    assert np.array_equal(ext, gold('ext'))
    assert ad.witness_verify_batch(pp, ext, wits['st_ntt']).tolist() == [int(c['witness_verify']) for c in cases]
    # a tampered statement, signature or message fails adaptor verify for its own item only
    st2 = wits['st_ntt'].copy()
    st2[1, 0] = (int(st2[1, 0]) + 1) % sp.lp.modulus
    v = wire.adaptor_verify_batch_packed(pp, vkp, chmsgs, wire.pack_keys(pp, st2), sig_p)
    assert v.tolist() == [int(cases[0]['verify']), 0]
    # LM signing through wire equals sign_batch -> pack_signatures
    from lattice_cryptography_b200 import lm_one_time_sigs as lm
    lpp = wire.setup_parameters_from_seed(lm.make_setup_parameters, secpar, 'wire sign')
    lkeys = lm.keygen_batch(lpp, [bin(3 * i + 1)[2:].zfill(secpar) for i in range(9)])
    chm = [f'<vk {i}>, message {i}' for i in range(9)]
    got, ok = wire.sign_batch_packed(lpp, lkeys['sk_ntt'], chm)
    want, want_ok = wire.pack_signatures(lpp, lm.sign_batch(lpp, lkeys['sk_ntt'], chm))
    assert np.array_equal(got, want) and np.array_equal(ok, want_ok) and ok.all()
    assert wire.verify_batch_packed(lpp, wire.pack_keys(lpp, lkeys['vk_ntt']), chm, got).tolist() == [1] * 9


# ------------------------------------------------------------------------------------------- argument errors
def test_argument_errors(engines):
    import torch
    from lattice_cryptography_b200 import Engine, LcbError, _ffi
    e = engines[128]
    sch = scheme(128)
    l = SHIPPED[128]['l']
    sk, vk, msgs = _items(e, sch, 128, 3, 1)
    vkp = e.pack(vk, 14, 0)
    stp = e.pack(np.zeros((3, D), np.uint16), 14, 0)
    sigp = e.lm_sign_packed(sch, sk, msgs, 11, 945)
    wit = np.zeros((3, l, D), np.int16)

    def invalid(fn):
        with pytest.raises(LcbError) as x:
            fn()
        assert x.value.status == _ffi.LCB_ERR_INVALID

    for bits in (0, 17):
        invalid(lambda: e.lm_sign_packed(sch, sk, msgs, bits, 0))
        invalid(lambda: e.adaptor_verify_packed(sch, vkp, 14, msgs, np.zeros((3, l, 32 * bits), np.uint8), bits, 0, stp, 14,
                                                946, 256))
        invalid(lambda: e.adaptor_verify_packed(sch, vkp, 14, msgs, sigp, 11, 945, np.zeros((3, 32 * bits), np.uint8), bits,
                                                946, 256))
        invalid(lambda: e.adapt_packed(sigp, 11, 945, wit, bits, 0))
        invalid(lambda: e.extract_packed(np.zeros((3, l, 32 * bits), np.uint8), bits, 0, sigp, 11, 945))
    for bias in (-1, 32768):
        invalid(lambda: e.lm_sign_packed(sch, sk, msgs, 11, bias))
        invalid(lambda: e.adaptor_verify_packed(sch, vkp, 14, msgs, sigp, 11, bias, stp, 14, 946, 256))
        invalid(lambda: e.adapt_packed(sigp, 11, bias, wit, 11, 945))
        invalid(lambda: e.adapt_packed(sigp, 11, 945, wit, 11, bias))
        invalid(lambda: e.extract_packed(sigp, 11, bias, sigp, 11, 945))
    # packed buffers that are not 4-byte aligned
    odd = lambda x: torch.zeros(x.size + 16, dtype=torch.uint8, device='cuda')[1:1 + x.size].view(*x.shape)
    torch.cuda.synchronize()
    invalid(lambda: e.adaptor_verify_packed(sch, vkp, 14, msgs, odd(sigp), 11, 945, stp, 14, 946, 256))
    invalid(lambda: e.adaptor_verify_packed(sch, vkp, 14, msgs, sigp, 11, 945, odd(stp), 14, 946, 256))
    invalid(lambda: e.adapt_packed(odd(sigp), 11, 945, wit, 11, 946))
    invalid(lambda: e.extract_packed(sigp, 11, 946, odd(sigp), 11, 945))
    lib = _ffi.load()
    d_sk = torch.from_numpy(sk).cuda()
    from lattice_cryptography_b200 import ragged
    blob, off = ragged(msgs)
    out = odd(sigp)
    torch.cuda.synchronize()
    assert lib.lcb_lm_sign_packed_batch(e._ctx, byref(sch), c_void_p(d_sk.data_ptr()), c_void_p(blob.ctypes.data),
                                        c_void_p(off.ctypes.data), 3, 11, 945, c_void_p(out.data_ptr()), None) == _ffi.LCB_ERR_INVALID
    # st_packed = NULL, and more than 2^30 items
    z = np.zeros(16, np.uint8)
    zo = np.zeros(4, np.int64)
    P = lambda a: c_void_p(a.ctypes.data)
    assert lib.lcb_adaptor_verify_packed_batch(e._ctx, byref(sch), P(vkp), 14, P(blob), P(off), P(sigp), 11, 945, None, 14, 3,
                                               946, 256, P(z)) == _ffi.LCB_ERR_INVALID
    assert lib.lcb_adaptor_verify_packed_batch(e._ctx, byref(sch), P(z), 14, P(z), P(zo), P(z), 11, 945, P(z), 14,
                                               (1 << 30) + 1, 946, 256, P(z)) == _ffi.LCB_ERR_INVALID
    assert b'2^30' in lib.lcb_last_error(e._ctx)
    # n = 0 is a no-op
    assert lib.lcb_lm_sign_packed_batch(e._ctx, byref(sch), P(z), None, P(zo), 0, 11, 945, P(z), None) == _ffi.LCB_OK
    assert lib.lcb_adaptor_adapt_packed_batch(e._ctx, P(z), 11, 945, P(z), 0, 11, 946, P(z), None) == _ffi.LCB_OK
    # generic contexts
    gen = Engine(128, 12289, 512, 2)
    try:
        gsch = _ffi.LcbScheme()
        gsch.ch_bd = gsch.ch_wt = gsch.sk_bd = gsch.sk_wt = 1
        gen.set_key_ch(np.zeros((2, 512), np.int16))
        checks = [
            lambda: gen.lm_sign_packed(gsch, np.zeros((1, 2, 2, 512), np.uint16), [b'x'], 11, 945),
            lambda: gen.adaptor_verify_packed(gsch, np.zeros((1, 2, 512 * 14 // 8), np.uint8), 14, [b'x'],
                                              np.zeros((1, 2, 512 * 11 // 8), np.uint8), 11, 945,
                                              np.zeros((1, 512 * 14 // 8), np.uint8), 14, 946, 256),
            lambda: gen.adapt_packed(np.zeros((1, 512 * 11 // 8), np.uint8), 11, 945, np.zeros((1, 512), np.int16), 11, 946),
            lambda: gen.extract_packed(np.zeros((1, 512 * 11 // 8), np.uint8), 11, 946, np.zeros((1, 512 * 11 // 8), np.uint8),
                                       11, 945)]
        for fn in checks:
            with pytest.raises(LcbError) as x:
                fn()
            assert x.value.status == _ffi.LCB_ERR_INVALID and 'd == 256' in str(x.value)
    finally:
        gen.close()


# ------------------------------------------------------------------------------------------- checked build
def test_small_cases(engines):
    """A small case of each call on both routes (the checked build runs it)."""
    import torch
    e = engines[128]
    sch = scheme(128)
    sk, vk, msgs = _items(e, sch, 128, 37, 4)
    sig = e.lm_sign(sch, sk, msgs)
    for bits in (11, 12):
        assert np.array_equal(e.lm_sign_packed(sch, sk, msgs, bits, 945), e.pack(sig, bits, 945))
    rng = np.random.default_rng(2)
    st = rng.integers(0, 11777, (37, D), dtype=np.uint16)
    want = e.lm_verify(sch, vk, msgs, sig, 945, 256, st_ntt=st)
    vkp, stp, sigp = e.pack(vk, 14, 0), e.pack(st, 14, 0), e.pack(sig, 11, 945)
    assert np.array_equal(e.adaptor_verify_packed(sch, vkp, 14, msgs, sigp, 11, 945, stp, 14, 945, 256), want)
    m = [_misaligned(x) for x in (vkp, sigp, stp)]
    torch.cuda.synchronize()
    got = e.adaptor_verify_packed(sch, m[0], 14, msgs, m[1], 11, 945, m[2], 14, 945, 256, device=True)
    e.synchronize()
    assert np.array_equal(got.cpu().numpy(), want)
    wit = rng.integers(-1, 2, sig.shape).astype(np.int16)
    ap = e.adapt_packed(sigp, 11, 945, wit, 11, 946)
    assert np.array_equal(ap, e.pack(e.vec_add(sig, wit), 11, 946))
    assert np.array_equal(e.extract_packed(ap, 11, 946, sigp, 11, 945), wit)


def test_packed_sign_adaptor_pass_on_the_checked_build():
    from lattice_cryptography_b200 import _ffi
    if _ffi.load().lcb_build_is_checked():
        pytest.skip('already running on the checked build')
    lib = os.path.join(ROOT, 'lattice_cryptography_b200', 'liblcb200_checked.so')
    if not os.path.exists(lib):
        subprocess.run(['make', '-C', os.path.join(ROOT, 'lattice_cryptography_b200', 'csrc'), '-j4', 'CHECKED=1'], check=True,
                       capture_output=True)
    env = dict(os.environ, LCB200_LIB=lib)
    r = subprocess.run([sys.executable, '-m', 'pytest', 'tests/test_gpu_sign_adaptor_packed.py', '-q', '-x', '-m', 'gpu', '-k',
                        'small_cases or (sign_packed_equals_sign_then_pack and 2049)', '-p', 'no:cacheprovider'],
                       env=env, capture_output=True, text=True, timeout=1500, cwd=ROOT)
    tail = r.stdout[-2500:] + r.stderr[-1500:]
    assert r.returncode == 0, tail
    assert '3 passed' in r.stdout and 'failed' not in r.stdout, tail
