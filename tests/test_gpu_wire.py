"""GPU parity of the packed wire format (include/lcb200.h: lcb_pack_batch / lcb_unpack_batch /
lcb_lm_verify_packed_batch; SURVEY.md 8(f)2) against oracle/wire.py, and of the public-seed key_ch
(8(f)3) against the restated hash2polynomialvector.  Bit-exact."""
import numpy as np
import pytest

from test_gpu_parity import D, SHIPPED, engines, scheme   # noqa: F401  (fixture re-export)

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize('bits,bias', [(1, 0), (2, 1), (5, 7), (8, 128), (11, 945), (13, 3315), (14, 0), (15, 9), (16, 0),
                                       (16, 32768)])
@pytest.mark.parametrize('npoly', [1, 7, 8, 9, 2049])
def test_pack_unpack_vs_oracle(engines, bits, bias, npoly):
    import wire as owire
    e = engines[128]
    rng = np.random.default_rng(bits * 1000 + npoly)
    lo, hi = -bias, (1 << bits) - bias                                   # representable range of x
    x = rng.integers(lo, hi, size=(npoly, D)).astype(np.int64)
    vals = (x & 0xFFFF).astype(np.uint16)
    # a few polynomials carry one value just outside the range
    bad_rows = rng.choice(npoly, size=min(npoly, 3), replace=False) if bits < 16 else np.zeros(0, dtype=np.int64)
    for r in bad_rows:
        vals[r, int(rng.integers(0, D))] = np.uint16((hi + int(rng.integers(0, 5))) & 0xFFFF)
    want, want_ok = owire.pack(vals, bits, bias)
    got, got_ok = e.pack(vals, bits, bias, want_range=True)
    assert got.shape == (npoly, 32 * bits) and np.array_equal(got, want)
    assert np.array_equal(got_ok, want_ok) and int(want_ok.sum()) == npoly - len(set(bad_rows.tolist()))
    back = e.unpack(got, bits, bias, dtype=np.uint16)
    assert np.array_equal(back, owire.unpack(want, bits, bias, np.uint16))
    good = want_ok.astype(bool)
    assert np.array_equal(back[good], vals[good])
    # signed view of the same call
    assert np.array_equal(e.unpack(got, bits, bias, dtype=np.int16).view(np.uint16), back)


def test_pack_device_buffers_and_errors(engines):
    import torch
    from lattice_cryptography_b200 import LcbError
    import wire as owire
    e = engines[256]
    rng = np.random.default_rng(5)
    sig = rng.integers(-3315, 3316, size=(33, 23, D)).astype(np.int16)
    dsig = torch.from_numpy(sig).cuda()
    packed = e.pack(dsig, 13, 3315, device=True)
    e.synchronize()
    assert packed.is_cuda and tuple(packed.shape) == (33, 23, 416)
    assert np.array_equal(packed.cpu().numpy(), owire.pack(sig, 13, 3315)[0])
    back = e.unpack(packed, 13, 3315, device=True)
    e.synchronize()
    assert np.array_equal(back.cpu().numpy(), sig)
    assert e.pack(np.zeros((0, D), np.int16), 11, 945).shape == (0, 352)
    for bits in (0, 17):
        with pytest.raises(LcbError):
            e.pack(np.zeros((1, D), np.int16), bits, 0)
    with pytest.raises(LcbError):
        e.unpack(np.zeros((1, 32), np.uint8), 1, 70000)


@pytest.mark.parametrize('secpar', [128, 256])
def test_verify_packed_equals_verify(engines, golden, secpar):
    """Verdicts from packed records == verdicts from the int16 / uint16 arrays, over good and tampered
    triples; coefficients at the bound +1..+2 are representable in the packing and must still be rejected."""
    from lattice_cryptography_b200 import ragged
    arrays, meta = golden
    e = engines[secpar]
    sch = scheme(secpar)
    s = SHIPPED[secpar]
    m = meta['cases'][str(secpar)]
    vf_bd, vf_wt = m['vf_bd'], m['vf_wt']
    sbits = int(np.ceil(np.log2(2 * vf_bd + 1)))
    kbits = int(np.ceil(np.log2(s['q'])))
    assert (sbits, kbits) == ((11, 14) if secpar == 128 else (13, 16))
    n = 700
    rng = np.random.default_rng(secpar)
    seeds = [''.join(rng.choice(['0', '1'], secpar)) for _ in range(n)]
    chmsgs = [bytes(rng.integers(1, 256, int(rng.integers(0, 300)), dtype=np.uint8)) for _ in range(n)]
    _, sk_ntt, vk_ntt, _ = e.lm_keygen(sch, seeds)
    sig = e.lm_sign(sch, sk_ntt, chmsgs)
    bad = sig.copy()
    msgs2 = list(chmsgs)
    for i in range(n):
        kind = int(rng.integers(0, 8))
        a, b = int(rng.integers(0, s['l'])), int(rng.integers(0, D))
        if kind == 0:
            bad[i, a, b] += int(rng.choice([-1, 1]))
        elif kind == 1:
            bad[i, a, b] = vf_bd + int(rng.integers(1, 3))
        elif kind == 2:
            msgs2[i] = chmsgs[i] + b'!'
    want = e.lm_verify(sch, vk_ntt, ragged(msgs2), bad, vf_bd, vf_wt)
    # the shipped widths are expanded inside k_verify; a wider packing takes the unpack-first route
    for sb, kb in ((sbits, kbits), (sbits + 1, min(16, kbits + 1))):
        sig_p, ok = e.pack(bad, sb, vf_bd, want_range=True)
        assert ok.all()
        vk_p = e.pack(vk_ntt, kb, 0)
        got = e.lm_verify_packed(sch, vk_p, kb, ragged(msgs2), sig_p, sb, vf_bd, vf_bd, vf_wt)
        assert np.array_equal(got, want) and 0.5 < want.mean() < 0.9
        assert sig_p.nbytes * 16 == bad.nbytes * sb
    # a bias other than vf_bd (still covering the coefficient range) must give the same verdicts
    sig_p = e.pack(bad, sbits + 1, vf_bd + 7)
    vk_p = e.pack(vk_ntt, kbits, 0)
    assert np.array_equal(e.lm_verify_packed(sch, vk_p, kbits, ragged(msgs2), sig_p, sbits + 1, vf_bd + 7, vf_bd, vf_wt), want)


def test_wire_module_and_seeded_key_ch(golden):
    """The Python layer: pack/unpack through pp, packed verify, and key_ch from a public seed equal to the
    oracle's hash2polynomialvector with the reference's distribution parameters (one_time_keys.py:284-290)."""
    import lattice_algebra as ola                     # oracle restatement (tests only)
    from lattice_cryptography_b200 import lm_one_time_sigs as lm
    from lattice_cryptography_b200 import wire
    from lattice_cryptography_b200.one_time_keys import bits_per_coefficient, bits_per_index_set
    pp = wire.setup_parameters_from_seed(lm.make_setup_parameters, 128, 'a public string')
    lp = pp['scheme_parameters'].lp
    olp = ola.LatticeParameters(modulus=lp.modulus, degree=lp.degree, length=lp.length)
    want = ola.hash2polynomialvector(
        secpar=128, lp=olp, distribution=ola.UNIFORM_INFINITY_WEIGHT, dist_pars={'bd': lp.modulus // 2, 'wt': lp.degree},
        salt=wire.KEY_CH_SALT, msg='a public string', num_coefs=lp.degree,
        bti=bits_per_index_set(secpar=128, degree=lp.degree, wt=lp.degree),
        btd=bits_per_coefficient(secpar=128, bd=lp.modulus // 2), const_time_flag=False)
    got = pp['scheme_parameters'].key_ch.get_coef_rep()
    assert [g[0] for g in got] == [w[0] for w in want.get_coef_rep()]
    # same seed -> same row; different seed -> different row
    again = wire.key_ch_from_seed(lp, 128, 'a public string')
    other = wire.key_ch_from_seed(lp, 128, 'another public string')
    assert again == pp['scheme_parameters'].key_ch and other != again
    seeds = [bin(7 * i + 1)[2:].zfill(128) for i in range(9)]
    keys = lm.keygen_batch(pp, seeds)
    chm = [f'<vk {i}>, message {i}' for i in range(9)]
    sigs = lm.sign_batch(pp, keys['sk_ntt'], chm)
    packed, ok = wire.pack_signatures(pp, sigs)
    assert ok.all() and packed.shape == (9, 13, 352)
    assert np.array_equal(wire.unpack_signatures(pp, packed), sigs)
    vkp = wire.pack_keys(pp, keys['vk_ntt'])
    assert vkp.shape == (9, 2, 448) and np.array_equal(wire.unpack_keys(pp, vkp), keys['vk_ntt'])
    assert wire.verify_batch_packed(pp, vkp, chm, packed).tolist() == [1] * 9
    chm[4] += '?'
    assert wire.verify_batch_packed(pp, vkp, chm, packed).tolist() == [1, 1, 1, 1, 0, 1, 1, 1, 1]
    # unseeded batch path: fresh seeds as (blob, offsets) give the same keys as their bitstrings
    blob, off = lm.random_seed_batch(pp, 5)
    fresh = lm.keygen_batch(pp, (blob, off))
    again = lm.keygen_batch(pp, [bytes(r).decode() for r in blob.reshape(5, 128)])
    assert np.array_equal(fresh['sk_coef'], again['sk_coef']) and np.array_equal(fresh['vk_ntt'], again['vk_ntt'])
    assert lm.verify_batch(pp, fresh['vk_ntt'], chm[:5], lm.sign_batch(pp, fresh['sk_ntt'], chm[:5])).tolist() == [1] * 5


def test_host_buffers_pipeline_over_several_chunks(engines):
    """Host-resident signatures are copied and verified in 2^17-triple chunks on a second stream
    (api.cu, Staging::pipe_chunk): more than one chunk, ragged tail, tampered triples in every chunk -
    verdicts must equal the all-device path, for the int16 and the packed entry points."""
    import torch
    from lattice_cryptography_b200 import ragged
    e = engines[128]
    sch = scheme(128)
    n = (1 << 17) + 4099
    rng = np.random.default_rng(17)
    seeds = (rng.integers(0, 2, (n, 128), dtype=np.uint8) + 48).astype(np.uint8)
    seed_off = np.arange(n + 1, dtype=np.int64) * 128
    msgs = rng.integers(33, 127, (n, 40), dtype=np.uint8)
    msg_off = np.arange(n + 1, dtype=np.int64) * 40
    d_seeds = (torch.from_numpy(seeds).cuda().view(-1), torch.from_numpy(seed_off).cuda())
    d_msgs = (torch.from_numpy(msgs).cuda().view(-1), torch.from_numpy(msg_off).cuda())
    _, sk_ntt, vk_ntt, _ = e.lm_keygen(sch, d_seeds, want_sk_coef=False, want_vk_coef=False, device=True)
    sig = e.lm_sign(sch, sk_ntt, d_msgs, device=True)
    e.synchronize()                      # the engine runs on its own stream, torch on another
    del sk_ntt
    bad = torch.arange(5, n, 997, device='cuda')
    sig.view(torch.int16)[bad, bad % 13, (5 * bad) % D] += 1
    torch.cuda.synchronize()
    want = e.lm_verify(sch, vk_ntt, d_msgs, sig, 945, 256, device=True)
    e.synchronize()
    want = want.cpu().numpy()
    assert want.sum() == n - len(bad) and not want[bad.cpu().numpy()].any()
    h_sig, h_vk = sig.cpu().numpy(), vk_ntt.cpu().numpy()
    h_msgs = (msgs.reshape(-1), msg_off)
    assert np.array_equal(e.lm_verify(sch, h_vk, h_msgs, h_sig, 945, 256), want)
    sig_p, vk_p = e.pack(sig, 11, 945, device=True), e.pack(vk_ntt, 14, 0, device=True)
    e.synchronize()
    sig_p, vk_p = sig_p.cpu().numpy(), vk_p.cpu().numpy()
    assert np.array_equal(e.lm_verify_packed(sch, vk_p, 14, h_msgs, sig_p, 11, 945, 945, 256), want)


@pytest.mark.parametrize('secpar', [128, 256])
def test_verify_packed_weight_below_d(engines, secpar):
    """vf_wt < 256 selects the weight-checking k_verify<true, 11, 14> / <true, 13, 0> on the fused packed route.  The
    signatures are built so that the equation holds (vk_right := key_ch * sig - vk_left * c), with one row of weight exactly
    wt or wt + 1: the verdicts must equal the numpy rule max|sig| <= bd and every row weight <= wt."""
    from lattice_cryptography_b200 import Engine
    s = SHIPPED[secpar]
    q, l = s['q'], s['l']
    sch = scheme(secpar)
    rng = np.random.default_rng(secpar + 1)
    e = Engine(secpar, q, D, l)
    try:
        key_ch = rng.integers(-(q // 2), q // 2 + 1, (l, D)).astype(np.int16)
        e.set_key_ch(key_ch)
        sb, kb, bd = (11, 14, 945) if secpar == 128 else (13, 16, 3315)
        for wt in (1, 10, 255):
            sigs, want = [], []
            for extra in (0, 1, 0, 1):
                row = int(rng.integers(0, l))
                z = np.zeros((l, D), np.int16)
                for i in range(l):
                    wi = wt + extra if i == row else int(rng.integers(1, wt + 1))
                    z[i, rng.choice(D, wi, replace=False)] = rng.choice(np.array([-bd, -1, 1, bd], np.int16), wi)
                sigs.append(z)
                want.append(1 - extra)
            sig = np.ascontiguousarray(np.stack(sigs))
            n = len(sigs)
            msgs = [f'weight {wt} {i}'.encode() for i in range(n)]
            pairs = e.challenge(sch, msgs)
            c = np.zeros((n, D), np.int16)
            for i in range(n):
                c[i, pairs[i, :, 0].astype(np.int64)] = pairs[i, :, 1]
            lhs = sum(e.poly_mul(np.ascontiguousarray(np.broadcast_to(key_ch[j], (n, D))), np.ascontiguousarray(sig[:, j]))
                      .astype(np.int64) for j in range(l))
            vkl = rng.integers(-(q // 2), q // 2 + 1, (n, D)).astype(np.int16)
            vkr = (lhs - e.poly_mul(vkl, c).astype(np.int64)) % q
            vkr = np.where(vkr > q // 2, vkr - q, vkr).astype(np.int16)
            vk = np.ascontiguousarray(np.stack([e.ntt_fwd(vkl), e.ntt_fwd(vkr)], axis=1))
            rule = [int((np.abs(x.astype(np.int64)).max() <= bd) and (x != 0).sum(axis=1).max() <= wt) for x in sigs]
            assert rule == want
            assert e.lm_verify(sch, vk, msgs, sig, bd, wt).tolist() == want, wt
            got = e.lm_verify_packed(sch, e.pack(vk, kb, 0), kb, msgs, e.pack(sig, sb, bd), sb, bd, bd, wt)
            assert got.tolist() == want, wt
    finally:
        e.close()
