"""Adaptor witnesses on the packed wire format (include/lcb200.h: lcb_adaptor_witgen_packed_batch,
lcb_adaptor_witness_verify_packed_batch, lcb_adaptor_adapt_packed_wit_batch, lcb_adaptor_extract_packed_wit_batch), compared
byte for byte with the composition each call is defined as (witgen -> pack; unpack -> witness_verify; unpack -> vec_add /
vec_sub -> pack), on the fused routes (k_verify reading packed witness and statement rows, k_addsub_packed) and on the
composed one, and with the golden witnesses packed by the independent oracle/wire.py."""
import os
import subprocess
import sys
from ctypes import byref, c_void_p

import numpy as np
import pytest

from test_gpu_parity import D, SHIPPED, engines, scheme   # noqa: F401  (fixture re-export)

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# presig bits, sig bits, key (statement) bits, pvf_bd, vf_bd, ext_wit_bd, ext_wit_wt, extracted-witness bits
ADP = {128: (11, 11, 14, 945, 946, 1891, 256, 12), 256: (13, 13, 16, 3315, 3316, 6631, 256, 14)}
WIT_BITS, WIT_BD, WIT_WT = 2, 1, 20
CHUNK = {128: (1 << 20) // 13, 256: (1 << 20) // 23}       # witnesses per internal chunk of the packed calls


def _seeds(secpar, n, seed):
    rng = np.random.default_rng(seed)
    return [''.join(rng.choice(['0', '1'], secpar)) for _ in range(n)]


def _misaligned(x):
    """A device copy of x that is 4-byte but not 16-byte aligned."""
    import torch
    flat = torch.from_numpy(np.ascontiguousarray(x).reshape(-1).view(np.uint8)).cuda()
    raw = torch.zeros(flat.numel() + 16, dtype=torch.uint8, device='cuda')
    view = raw[4:4 + flat.numel()]
    view.copy_(flat)
    assert view.data_ptr() % 16 == 4
    return view.view(*x.shape)


def _wv_composed(e, witp, wb, wbias, stp, sb, bd, wt):
    return e.witness_verify(e.unpack(witp, wb, wbias), e.unpack(stp, sb, 0, dtype=np.uint16), bd, wt)


def _addsub_composed(e, a, ab, abias, b, bb, bbias, sub, ob, obias):
    x, y = e.unpack(a, ab, abias), e.unpack(b, bb, bbias)
    return e.pack(e.vec_sub(x, y) if sub else e.vec_add(x, y), ob, obias, want_range=True)


def _pairs(e, secpar, n, seed):
    """n genuine (witness int16, statement uint16 NTT form) pairs."""
    wit, st, _ = e.witgen(scheme(secpar), _seeds(secpar, n, seed), want_st_coef=False)
    return wit, st


# ------------------------------------------------------------------------------------------- witgen
@pytest.mark.parametrize('n', [1, 7, 2049, 'chunk'])
@pytest.mark.parametrize('secpar', [128, 256])
def test_witgen_packed_equals_witgen_then_pack(engines, secpar, n):
    e = engines[secpar]
    sch = scheme(secpar)
    kb = ADP[secpar][2]
    n = CHUNK[secpar] + 3 if n == 'chunk' else n
    seeds = _seeds(secpar, n, secpar + n)
    wit, st = e.witgen(sch, seeds, want_st_coef=False)[:2]
    want_w, want_ok = e.pack(wit, WIT_BITS, WIT_BD, want_range=True)
    want_st = e.pack(st, kb, 0)
    assert want_ok.all()
    w, ok, s = e.witgen_packed(sch, seeds, WIT_BITS, WIT_BD, kb, want_wit_range=True)
    assert np.array_equal(w, want_w) and np.array_equal(ok, want_ok) and np.array_equal(s, want_st)
    # each output NULL in turn
    w, ok, s = e.witgen_packed(sch, seeds, WIT_BITS, WIT_BD, kb, want_st=False)
    assert np.array_equal(w, want_w) and ok is None and s is None
    w, ok, s = e.witgen_packed(sch, seeds, WIT_BITS, WIT_BD, kb, want_wit=False)
    assert w is None and ok is None and np.array_equal(s, want_st)


@pytest.mark.parametrize('secpar', [128, 256])
def test_witgen_packed_other_widths_and_device_buffers(engines, secpar):
    import torch
    from lattice_cryptography_b200 import ragged
    e = engines[secpar]
    sch = scheme(secpar)
    kb = ADP[secpar][2]
    n = 300
    seeds = _seeds(secpar, n, 5 * secpar)
    wit, st = e.witgen(sch, seeds, want_st_coef=False)[:2]
    for wbits, wbias, sbits in ((1, 0, 15), (12, 1891, 16), (16, 32767, 14)):
        want_w, want_ok = e.pack(wit, wbits, wbias, want_range=True)
        w, ok, s = e.witgen_packed(sch, seeds, wbits, wbias, sbits, want_wit_range=True)
        assert np.array_equal(w, want_w) and np.array_equal(ok, want_ok) and np.array_equal(s, e.pack(st, sbits, 0))
        assert ok.all() == ((wbits, wbias) != (1, 0))      # -1 does not fit one bit without a bias
    blob, off = ragged(seeds)
    d_blob, d_off = (torch.from_numpy(np.array(x)).cuda() for x in (blob, off))
    torch.cuda.synchronize()
    w, ok, s = e.witgen_packed(sch, (d_blob, d_off), WIT_BITS, WIT_BD, kb, want_wit_range=True, device=True)
    e.synchronize()
    want_w, want_ok = e.pack(wit, WIT_BITS, WIT_BD, want_range=True)
    assert np.array_equal(w.cpu().numpy(), want_w) and np.array_equal(ok.cpu().numpy(), want_ok)
    assert np.array_equal(s.cpu().numpy(), e.pack(st, kb, 0))


@pytest.mark.parametrize('secpar', [128, 256])
def test_witgen_packed_golden(engines, golden, secpar):
    """The golden seeds' packed witnesses and statements equal the golden witnesses and statements (through ntt_fwd) packed
    by oracle/wire.py."""
    import wire as owire
    arrays, meta = golden
    cases = meta['cases'][str(secpar)]['adaptor']
    e = engines[secpar]
    kb = ADP[secpar][2]
    seeds = [c['wit_seed'] for c in cases]
    w, ok, s = e.witgen_packed(scheme(secpar), seeds, WIT_BITS, WIT_BD, kb, want_wit_range=True)
    for j in range(len(seeds)):
        want_w, want_ok = owire.pack(arrays[f's{secpar}_ad{j}_wit'], WIT_BITS, WIT_BD)
        st_ntt = e.ntt_fwd(np.ascontiguousarray(arrays[f's{secpar}_ad{j}_st'][None]))[0]
        want_s, _ = owire.pack(st_ntt, kb, 0)
        assert np.array_equal(w[j], want_w) and np.array_equal(ok[j], want_ok) and np.array_equal(s[j], want_s), j


# ------------------------------------------------------------------------------------------- witness verify
def _wv_inputs(e, secpar, n, wb, wbias, sb, seed):
    """Packed witnesses / statements at (wb, wbias, sb): genuine pairs, one flipped byte, uniformly random bytes,
    coefficients at +-ext_wit_bd and one past it (where the width holds them), statement slots >= q."""
    q, ext = SHIPPED[secpar]['q'], ADP[secpar][5]
    wit, st = _pairs(e, secpar, n, seed)
    rng = np.random.default_rng(seed)
    wit[n // 3: n // 3 + 6, 0, :3] = [ext, -ext, 0]          # at the bound
    wit[n // 3 + 6: n // 3 + 12, 1, 5] = ext + 1             # one past it
    wit[n // 3 + 12: n // 3 + 18, 2, 7] = -ext - 1
    st[n // 2: n // 2 + 6, 3] = q + np.arange(6)             # slots >= q
    witp, _ = e.pack(wit, wb, wbias, want_range=True)
    stp = e.pack(st, sb, 0)
    witp[1, 0, 5] ^= 0x04                                    # one flipped byte
    stp[2, 9] ^= 0x01
    r = rng.random(n) < 0.2
    witp[r] = rng.integers(0, 256, (int(r.sum()),) + witp.shape[1:], dtype=np.uint8)
    r2 = rng.random(n) < 0.1
    stp[r2] = rng.integers(0, 256, (int(r2.sum()),) + stp.shape[1:], dtype=np.uint8)
    return witp, stp


@pytest.mark.parametrize('secpar', [128, 256])
def test_witness_verify_packed_fused_routes(engines, secpar):
    e = engines[secpar]
    kb, ext, ext_wt, xb = ADP[secpar][2], ADP[secpar][5], ADP[secpar][6], ADP[secpar][7]
    n = 6151                                                 # more than one persistent grid of k_verify
    for wb, wbias in ((WIT_BITS, WIT_BD), (xb, ext)):
        witp, stp = _wv_inputs(e, secpar, n, wb, wbias, kb, wb + secpar)
        for bd, wt in ((ext, ext_wt), (ext, WIT_WT), (WIT_BD, WIT_WT)):
            want = _wv_composed(e, witp, wb, wbias, stp, kb, bd, wt)
            got = e.witness_verify_packed(witp, wb, wbias, stp, kb, bd, wt)
            assert np.array_equal(got, want), (wb, bd, wt)
        assert 0 < want.sum() < n
    # genuine pairs: all 1; one flipped byte: only that item goes to 0
    wit, st = _pairs(e, secpar, 64, 9)
    witp, _ = e.pack(wit, WIT_BITS, WIT_BD, want_range=True)
    stp = e.pack(st, kb, 0)
    assert e.witness_verify_packed(witp, WIT_BITS, WIT_BD, stp, kb, ext, ext_wt).tolist() == [1] * 64
    witp[17, 4, 9] ^= 0x02
    assert e.witness_verify_packed(witp, WIT_BITS, WIT_BD, stp, kb, ext, ext_wt).tolist() == [1] * 17 + [0] + [1] * 46


@pytest.mark.parametrize('secpar', [128, 256])
def test_witness_verify_packed_composed_routes(engines, secpar):
    """Other widths, statements not at the key width and a 4-byte aligned caller device buffer: unpack -> witness_verify."""
    import torch
    from lattice_cryptography_b200 import _ffi
    e = engines[secpar]
    kb, ext, ext_wt, xb = ADP[secpar][2], ADP[secpar][5], ADP[secpar][6], ADP[secpar][7]
    other_st = 16 if kb == 14 else 15
    n = 777
    for wb, wbias, sb in ((3, 1, 16), (16, 32767, kb), (16, 0, kb), (WIT_BITS, WIT_BD, other_st), (xb, ext, other_st),
                          (13, ext, kb)):
        witp, stp = _wv_inputs(e, secpar, n, wb, wbias, sb, wb * sb)
        want = _wv_composed(e, witp, wb, wbias, stp, sb, ext, ext_wt)
        assert np.array_equal(e.witness_verify_packed(witp, wb, wbias, stp, sb, ext, ext_wt), want), (wb, wbias, sb)
    lib = _ffi.load()
    for wb, wbias in ((WIT_BITS, WIT_BD), (xb, ext)):
        witp, stp = _wv_inputs(e, secpar, n, wb, wbias, kb, 3 * wb)
        want = _wv_composed(e, witp, wb, wbias, stp, kb, ext, ext_wt)
        for mis_wit in (True, False):
            d_w = _misaligned(witp) if mis_wit else torch.from_numpy(witp).cuda()
            d_s = torch.from_numpy(stp).cuda() if mis_wit else _misaligned(stp)
            out = torch.zeros(n, dtype=torch.uint8, device='cuda')
            torch.cuda.synchronize()
            assert lib.lcb_adaptor_witness_verify_packed_batch(e._ctx, c_void_p(d_w.data_ptr()), wb, wbias,
                                                               c_void_p(d_s.data_ptr()), kb, n, ext, ext_wt,
                                                               c_void_p(out.data_ptr())) == _ffi.LCB_OK
            e.synchronize()
            assert np.array_equal(out.cpu().numpy(), want), (wb, mis_wit)
        # aligned device buffers: the fused route, asynchronous
        got = e.witness_verify_packed(torch.from_numpy(witp).cuda(), wb, wbias, torch.from_numpy(stp).cuda(), kb, ext,
                                      ext_wt, device=True)
        e.synchronize()
        assert np.array_equal(got.cpu().numpy(), want)


# ------------------------------------------------------------------------------------------- adapt / extract
WIDTHS = (1, 2, 11, 12, 13, 14, 16)


@pytest.mark.parametrize('secpar', [128, 256])
def test_adapt_extract_packed_wit_random_bytes(engines, secpar):
    """Uniformly random bytes at every width of WIDTHS and biases 0 / 32767 on each operand and on the output (a 16-bit
    field with bias 0 wraps to a negative int16, as unpack + vec_add do)."""
    e = engines[secpar]
    rng = np.random.default_rng(secpar)
    npoly = 1031
    k = len(WIDTHS)
    combos = [(WIDTHS[i], bias, WIDTHS[(i + 3) % k], 32767 - bias, WIDTHS[(i + 5) % k], b2)
              for i in range(k) for bias in (0, 32767) for b2 in (0, 32767)]
    combos += [(w, bias, w, bias, w, bias) for w in WIDTHS for bias in (0, 32767)]
    for ab, abias, bb, bbias, ob, obias in combos:
        a = rng.integers(0, 256, (npoly, 32 * ab), dtype=np.uint8)
        b = rng.integers(0, 256, (npoly, 32 * bb), dtype=np.uint8)
        want, want_ok = _addsub_composed(e, a, ab, abias, b, bb, bbias, 0, ob, obias)
        got, ok = e.adapt_packed_wit(a, ab, abias, b, bb, bbias, ob, obias, want_range=True)
        assert np.array_equal(got, want) and np.array_equal(ok, want_ok), ('adapt', ab, abias, bb, bbias, ob, obias)
        want, want_ok = _addsub_composed(e, a, ab, abias, b, bb, bbias, 1, ob, obias)
        got, ok = e.extract_packed_wit(a, ab, abias, b, bb, bbias, ob, obias, want_range=True)
        assert np.array_equal(got, want) and np.array_equal(ok, want_ok), ('extract', ab, abias, bb, bbias, ob, obias)
    # in_range = NULL
    assert np.array_equal(e.adapt_packed_wit(a, ab, abias, b, bb, bbias, ob, obias),
                          _addsub_composed(e, a, ab, abias, b, bb, bbias, 0, ob, obias)[0])


@pytest.mark.parametrize('secpar', [128, 256])
def test_adapt_extract_packed_wit_genuine(engines, secpar):
    """adapt_packed_wit(presig, pack(wit)) equals adapt_packed(presig, wit); extraction returns the witgen_packed bytes at 2
    bits and pack(wit, ext width, ext_wit_bd) at the extracted width, every in_range 1; device buffers."""
    import torch
    e = engines[secpar]
    sch = scheme(secpar)
    pb, sb, kb, pvf, vf, ext, _, xb = ADP[secpar]
    n = 500
    seeds = _seeds(secpar, n, 77)
    sk_coef, sk_ntt, _, _ = e.lm_keygen(sch, _seeds(secpar, n, 78), want_vk_ntt=False, want_vk_coef=False)
    chm = [f'<st {i}>, <vk {i}>, msg {i}' for i in range(n)]
    presig, pok = e.lm_sign_packed(sch, sk_ntt, chm, pb, pvf, want_range=True)
    assert pok.all()
    wit = e.witgen(sch, seeds, want_st_ntt=False, want_st_coef=False)[0]
    witp, _, _ = e.witgen_packed(sch, seeds, WIT_BITS, WIT_BD, kb, want_st=False)
    sig, ok = e.adapt_packed_wit(presig, pb, pvf, witp, WIT_BITS, WIT_BD, sb, vf, want_range=True)
    want, want_ok = e.adapt_packed(presig, pb, pvf, wit, sb, vf, want_range=True)
    assert np.array_equal(sig, want) and np.array_equal(ok, want_ok) and ok.all()
    w2, ok2 = e.extract_packed_wit(sig, sb, vf, presig, pb, pvf, WIT_BITS, WIT_BD, want_range=True)
    assert np.array_equal(w2, witp) and ok2.all()
    wx, okx = e.extract_packed_wit(sig, sb, vf, presig, pb, pvf, xb, ext, want_range=True)
    assert np.array_equal(wx, e.pack(wit, xb, ext)) and okx.all()
    d = lambda x: torch.from_numpy(x).cuda()
    g, gok = e.adapt_packed_wit(d(presig), pb, pvf, d(witp), WIT_BITS, WIT_BD, sb, vf, device=True, want_range=True)
    gw, gwok = e.extract_packed_wit(g, sb, vf, d(presig), pb, pvf, WIT_BITS, WIT_BD, device=True, want_range=True)
    e.synchronize()
    assert np.array_equal(g.cpu().numpy(), sig) and gok.cpu().numpy().all()
    assert np.array_equal(gw.cpu().numpy(), witp) and gwok.cpu().numpy().all()


# ------------------------------------------------------------------------------------------- round trip through `wire`
@pytest.mark.parametrize('secpar', [128, 256])
def test_packed_witness_lifecycle_round_trips(secpar):
    from lattice_cryptography_b200 import adaptor_sigs as ad
    from lattice_cryptography_b200 import wire
    n = 64
    app = wire.setup_parameters_from_seed(ad.make_setup_parameters, secpar, 'packed witnesses')
    assert wire.sig_bits(app, 'wit_bd') == WIT_BITS and wire.sig_bits(app, 'ext_wit_bd') == ADP[secpar][7]
    witp, stp = wire.witgen_batch_packed(app, [bin(11 * i + 5)[2:].zfill(secpar) for i in range(n)])
    skp, vkp = wire.keygen_batch_packed(app, [bin(7 * i + 3)[2:].zfill(secpar) for i in range(n)])
    chm = [f'<st {i}>, <vk {i}>, message {i}' for i in range(n)]
    presig, ok = wire.presign_batch_packed_sk(app, skp, chm)
    assert ok.all()
    assert wire.preverify_batch_packed(app, vkp, chm, presig).tolist() == [1] * n
    sig, ok = wire.adapt_batch_packed_wit(app, presig, witp)
    assert ok.all()
    assert wire.adaptor_verify_batch_packed(app, vkp, chm, stp, sig).tolist() == [1] * n
    ext, ok = wire.extract_batch_packed_wit(app, presig, sig)
    assert ok.all()
    assert np.array_equal(wire.unpack_witnesses(app, ext, bound_key='ext_wit_bd'), wire.unpack_witnesses(app, witp))
    assert wire.witness_verify_batch_packed(app, ext, stp, bound_key='ext_wit_bd').tolist() == [1] * n
    assert wire.witness_verify_batch_packed(app, witp, stp).tolist() == [1] * n
    ext2, ok2 = wire.extract_batch_packed_wit(app, presig, sig, bound_key='wit_bd')
    assert np.array_equal(ext2, witp) and ok2.all()
    assert np.array_equal(wire.pack_witnesses(app, wire.unpack_witnesses(app, witp))[0], witp)
    # one tampered witness byte changes exactly its own item downstream
    bad = witp.copy()
    bad[13, 2, 7] ^= 0x01
    sig2, _ = wire.adapt_batch_packed_wit(app, presig, bad)
    assert wire.adaptor_verify_batch_packed(app, vkp, chm, stp, sig2).tolist() == [1] * 13 + [0] + [1] * (n - 14)
    ext3, _ = wire.extract_batch_packed_wit(app, presig, sig2)
    assert wire.witness_verify_batch_packed(app, ext3, stp, bound_key='ext_wit_bd').tolist() == [1] * 13 + [0] + [1] * (n - 14)


# ------------------------------------------------------------------------------------------- argument errors
def test_argument_errors(engines):
    import torch
    from lattice_cryptography_b200 import Engine, LcbError, _ffi
    e = engines[128]
    sch = scheme(128)
    seeds = _seeds(128, 3, 1)
    witp, _, stp = e.witgen_packed(sch, seeds, 2, 1, 14)
    pre = np.zeros((3, 13, 352), np.uint8)

    def status(fn, want=_ffi.LCB_ERR_INVALID):
        with pytest.raises(LcbError) as x:
            fn()
        assert x.value.status == want
        return str(x.value)

    for bits in (0, 17):
        status(lambda: e.witgen_packed(sch, seeds, bits, 1, 14))
        status(lambda: e.witgen_packed(sch, seeds, 2, 1, bits))
        status(lambda: e.witness_verify_packed(np.zeros((3, 13, 32 * bits), np.uint8), bits, 0, stp, 14, 1891, 256))
        status(lambda: e.witness_verify_packed(witp, 2, 1, np.zeros((3, 32 * bits), np.uint8), bits, 1891, 256))
        status(lambda: e.adapt_packed_wit(pre, 11, 945, witp, 2, 1, bits, 946))
        status(lambda: e.extract_packed_wit(pre, 11, 946, pre, 11, 945, bits, 1))
    for bias in (-1, 32768):
        status(lambda: e.witgen_packed(sch, seeds, 2, bias, 14))
        status(lambda: e.witness_verify_packed(witp, 2, bias, stp, 14, 1891, 256))
        status(lambda: e.adapt_packed_wit(pre, 11, bias, witp, 2, 1, 11, 946))
        status(lambda: e.adapt_packed_wit(pre, 11, 945, witp, 2, bias, 11, 946))
        status(lambda: e.adapt_packed_wit(pre, 11, 945, witp, 2, 1, 11, bias))
        status(lambda: e.extract_packed_wit(pre, 11, 946, pre, 11, 945, 2, bias))
    status(lambda: e.witgen_packed(sch, seeds, 2, 1, 14, want_wit=False, want_st=False))
    # packed buffers that are only 2-byte aligned
    half = lambda x: torch.zeros(x.size + 16, dtype=torch.uint8, device='cuda')[2:2 + x.size].view(*x.shape)
    torch.cuda.synchronize()
    status(lambda: e.witness_verify_packed(half(witp), 2, 1, stp, 14, 1891, 256))
    status(lambda: e.witness_verify_packed(witp, 2, 1, half(stp), 14, 1891, 256))
    status(lambda: e.adapt_packed_wit(pre, 11, 945, half(witp), 2, 1, 11, 946))
    status(lambda: e.extract_packed_wit(half(pre), 11, 946, pre, 11, 945, 2, 1))
    lib = _ffi.load()
    from lattice_cryptography_b200 import ragged
    blob, off = ragged(seeds)
    P = lambda a: c_void_p(a.ctypes.data)
    out = half(np.zeros((3, 13, 352), np.uint8))
    torch.cuda.synchronize()
    assert lib.lcb_adaptor_witgen_packed_batch(e._ctx, byref(sch), P(blob), P(off), 3, 2, 1, c_void_p(out.data_ptr()), None,
                                               14, None) == _ffi.LCB_ERR_INVALID
    assert lib.lcb_adaptor_adapt_packed_wit_batch(e._ctx, P(pre), 11, 945, P(witp), 2, 1, 39, 11, 946,
                                                  c_void_p(out.data_ptr()), None) == _ffi.LCB_ERR_INVALID
    z = np.zeros(16, np.uint8)
    assert lib.lcb_adaptor_witness_verify_packed_batch(e._ctx, P(z), 2, 1, P(z), 14, (1 << 30) + 1, 1891, 256,
                                                       P(z)) == _ffi.LCB_ERR_INVALID
    assert b'2^30' in lib.lcb_last_error(e._ctx)
    # n = 0
    assert lib.lcb_adaptor_witness_verify_packed_batch(e._ctx, P(z), 2, 1, P(z), 14, 0, 1891, 256, P(z)) == _ffi.LCB_OK
    assert lib.lcb_adaptor_witgen_packed_batch(e._ctx, byref(sch), None, P(np.zeros(1, np.int64)), 0, 2, 1, P(z), None, 14,
                                               None) == _ffi.LCB_OK
    assert lib.lcb_adaptor_adapt_packed_wit_batch(e._ctx, P(z), 11, 945, P(z), 2, 1, 0, 11, 946, P(z), None) == _ffi.LCB_OK
    assert lib.lcb_adaptor_extract_packed_wit_batch(e._ctx, P(z), 11, 946, P(z), 11, 945, 0, 2, 1, P(z), None) == _ffi.LCB_OK
    # a context without key_ch
    g = Engine(128, SHIPPED[128]['q'], D, SHIPPED[128]['l'])
    try:
        status(lambda: g.witgen_packed(sch, seeds, 2, 1, 14), _ffi.LCB_ERR_NO_KEY_CH)
        status(lambda: g.witness_verify_packed(witp, 2, 1, stp, 14, 1891, 256), _ffi.LCB_ERR_NO_KEY_CH)
    finally:
        g.close()
    # generic (d = 512) and wide (q >= 2^16) contexts
    gsch = _ffi.LcbScheme()
    gsch.ch_bd = gsch.ch_wt = gsch.sk_bd = gsch.sk_wt = gsch.wit_bd = gsch.wit_wt = 1
    for q, d in ((12289, 512), (65537, 256)):
        g = Engine(128, q, d, 2)
        try:
            g.set_key_ch(np.zeros((2, d), np.int32 if q >= 65536 else np.int16))
            row = lambda bits: np.zeros((1, 2, d * bits // 8), np.uint8)
            for fn in (lambda: g.witgen_packed(gsch, ['0' * 128], 2, 1, 14),
                       lambda: g.witness_verify_packed(row(2), 2, 1, np.zeros((1, d * 14 // 8), np.uint8), 14, 1, 1),
                       lambda: g.adapt_packed_wit(row(11), 11, 945, row(2), 2, 1, 11, 946),
                       lambda: g.extract_packed_wit(row(11), 11, 946, row(11), 11, 945, 2, 1)):
                assert 'd == 256' in status(fn)
        finally:
            g.close()


# ------------------------------------------------------------------------------------------- checked build
def test_small_cases(engines):
    """A small case of all four calls on both routes (the checked build runs it)."""
    e = engines[128]
    sch = scheme(128)
    n = 37
    seeds = _seeds(128, n, 4)
    wit, st = e.witgen(sch, seeds, want_st_coef=False)[:2]
    w, ok, s = e.witgen_packed(sch, seeds, 2, 1, 14, want_wit_range=True)
    assert np.array_equal(w, e.pack(wit, 2, 1)) and ok.all() and np.array_equal(s, e.pack(st, 14, 0))
    for wb, wbias, sb in ((2, 1, 14), (12, 1891, 14), (3, 1, 16)):
        witp, stp = e.pack(wit, wb, wbias), e.pack(st, sb, 0)
        witp[5] ^= 0x10
        want = _wv_composed(e, witp, wb, wbias, stp, sb, 1891, 256)
        assert np.array_equal(e.witness_verify_packed(witp, wb, wbias, stp, sb, 1891, 256), want)
        assert want.tolist() == [1] * 5 + [0] + [1] * (n - 6)
    rng = np.random.default_rng(5)
    a = rng.integers(0, 256, (n, 13, 32 * 11), dtype=np.uint8)
    for ob, obias in ((11, 946), (2, 1)):
        want, want_ok = _addsub_composed(e, a, 11, 945, w, 2, 1, 0, ob, obias)
        got, gok = e.adapt_packed_wit(a, 11, 945, w, 2, 1, ob, obias, want_range=True)
        assert np.array_equal(got, want) and np.array_equal(gok, want_ok)
        want, want_ok = _addsub_composed(e, a, 11, 946, a, 11, 945, 1, ob, obias)
        got, gok = e.extract_packed_wit(a, 11, 946, a, 11, 945, ob, obias, want_range=True)
        assert np.array_equal(got, want) and np.array_equal(gok, want_ok)


def test_packed_witnesses_pass_on_the_checked_build():
    from lattice_cryptography_b200 import _ffi
    if _ffi.load().lcb_build_is_checked():
        pytest.skip('already running on the checked build')
    lib = os.path.join(ROOT, 'lattice_cryptography_b200', 'liblcb200_checked.so')
    if not os.path.exists(lib):
        subprocess.run(['make', '-C', os.path.join(ROOT, 'lattice_cryptography_b200', 'csrc'), '-j4', 'CHECKED=1'], check=True,
                       capture_output=True)
    env = dict(os.environ, LCB200_LIB=lib)
    r = subprocess.run([sys.executable, '-m', 'pytest', 'tests/test_gpu_packed_witness.py', '-q', '-x', '-m', 'gpu', '-k',
                        'small_cases', '-p', 'no:cacheprovider'], env=env, capture_output=True, text=True, timeout=1500, cwd=ROOT)
    tail = r.stdout[-2500:] + r.stderr[-1500:]
    assert r.returncode == 0, tail
    assert '1 passed' in r.stdout and 'failed' not in r.stdout, tail
