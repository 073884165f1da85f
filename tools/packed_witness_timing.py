"""Packed adaptor witnesses (lcb_adaptor_witgen_packed_batch, lcb_adaptor_witness_verify_packed_batch,
lcb_adaptor_adapt_packed_wit_batch, lcb_adaptor_extract_packed_wit_batch) against the calls they replace, on a B200 with the
shipped adaptor parameters at secpar 128 and 256.

  adapt / extract, device-resident, 2^20 adaptor signatures: adapt_packed_wit (k_addsub_packed), adapt_packed with int16
        witnesses (k_unpack -> k_vec_addsub -> k_pack) and unpacked vec_add; the same three arms for extract
  adapt and witness verify from pinned host memory, 2^18 items: time (host clock around calls that end synchronised) and
        bytes over the host link
  witness verify, device-resident, 2^20: the fused route (k_verify reading 2-bit witnesses and packed statements), the
        composed route (a 4-byte aligned witness buffer: k_unpack -> k_verify) and int16 witness_verify
  witgen, device-resident, 2^20: witgen_packed against witgen + two packs

Device arms are alternated rep by rep and timed with CUDA events (median); per-kernel times come from lcb_profile_read.
Every timed output is checked: packed arms equal the packed unpacked arm, extraction returns the generated witnesses, every
verdict and in_range flag is 1.

  python tools/packed_witness_timing.py [reps] [output file]
"""
import os
import subprocess
import sys
import time
from ctypes import c_void_p

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from lattice_cryptography_b200 import Engine, _ffi, make_scheme
from lattice_cryptography_b200 import adaptor_sigs as ad
from lattice_cryptography_b200 import wire

REPS = int(sys.argv[1]) if len(sys.argv) > 1 else 5
OUT = open(sys.argv[2], 'w') if len(sys.argv) > 2 else sys.stdout
N_DEV = 1 << 20
N_HOST = 1 << 18


def say(s=''):
    print(s, file=OUT, flush=True)


smi = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                     capture_output=True, text=True).stdout.strip().splitlines()
say(f'card: {torch.cuda.get_device_name(0)}; nvidia-smi name, power limit, max SM clock: {smi[0] if smi else "n/a"}')
say(f'device times are the median of {REPS} alternated reps (CUDA events); inputs far beyond the 126 MB L2')

P = lambda t: c_void_p(t.data_ptr())


def misaligned(t):
    """a copy of t whose data pointer is 4-byte but not 16-byte aligned (forces the composed route)"""
    raw = torch.empty(t.numel() * t.element_size() + 16, dtype=torch.uint8, device=t.device)
    v = raw[4:4 + t.numel() * t.element_size()]
    v.copy_(t.reshape(-1).view(torch.uint8))
    return v.view(t.dtype).view(*t.shape)


def timed_alternating(arms):
    for fn in arms.values():
        fn()
    ms = {k: [] for k in arms}
    for _ in range(REPS):
        for k, fn in arms.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            b.synchronize()
            ms[k].append(a.elapsed_time(b))
    return {k: float(np.median(v)) for k, v in ms.items()}


def kernels(eng, fn, names):
    eng.profile(True)
    eng.profile_reset()
    fn()
    torch.cuda.synchronize()
    out = {k: eng.profile_read(k) for k in names}
    eng.profile(False)
    return ', '.join(f'{k} {ms:.3f} ms' + (f' ({n}x)' if n > 1 else '') for k, (ms, n) in out.items() if n)


def host_alternating(arms):
    for fn in arms.values():
        fn()
    ts = {k: [] for k in arms}
    for _ in range(REPS):
        for k, fn in arms.items():
            t0 = time.perf_counter()
            fn()
            ts[k].append(time.perf_counter() - t0)
    return {k: 1e3 * float(np.median(v)) for k, v in ts.items()}


def report(eng, title, arms, names):
    ms = timed_alternating(arms)
    say(title)
    for k, fn in arms.items():
        say(f'  {k:30s} {ms[k]:8.3f} ms   [{kernels(eng, fn, names)}]')


def run(secpar):
    pp = ad.make_setup_parameters(secpar)
    lp = pp['scheme_parameters'].lp
    q, l = lp.modulus, lp.length
    pb, sb, kb = wire.sig_bits(pp, 'pvf_bd'), wire.sig_bits(pp), wire.key_bits(pp)
    wb, xb = wire.sig_bits(pp, 'wit_bd'), wire.sig_bits(pp, 'ext_wit_bd')
    pvf, vf, wbd, ext, ext_wt = pp['pvf_bd'], pp['vf_bd'], pp['wit_bd'], pp['ext_wit_bd'], pp['ext_wit_wt']
    eng = Engine(secpar, q, 256, l)
    eng.use_torch_stream()
    lib = _ffi.load()
    sch = make_scheme(sk_bd=pp['sk_bd'], sk_wt=pp['sk_wt'], ch_bd=pp['ch_bd'], ch_wt=pp['ch_wt'], wit_bd=wbd,
                      wit_wt=pp['wit_wt'])
    key_ch, _ = eng.hash2polyvec('KEY_CH_SEED', ['packed witness timing'], q // 2, 256, l)
    eng.set_key_ch(np.ascontiguousarray(key_ch[0]))
    n = N_DEV
    seeds = eng.expand_seeds(bytes(range(32)), n, device=True)
    wit, st, _ = eng.witgen(sch, seeds, want_st_coef=False, device=True)
    witp, wok = eng.pack(wit, wb, wbd, device=True, want_range=True)
    stp = eng.pack(st, kb, 0, device=True)
    g = torch.Generator(device='cuda').manual_seed(secpar)
    pre = torch.randint(-pvf, pvf + 1, (n, l, 256), dtype=torch.int16, device='cuda', generator=g)
    prep = eng.pack(pre, pb, pvf, device=True)
    torch.cuda.synchronize()
    assert bool(wok.all())
    say(f'\nsecpar {secpar}: q = {q}, l = {l}; witnesses {wb} bits (bias wit_bd = {wbd}), extracted {xb} bits (bias '
        f'ext_wit_bd = {ext}), presignatures {pb} / adaptor signatures {sb} bits, statements {kb} bits')
    say(f'bytes per witness: int16 {l * 512}, packed {l * 32 * wb} ({xb}-bit: {l * 32 * xb}); per statement packed {32 * kb}')

    # ---- adapt / extract, device-resident
    sig_w, sok = eng.adapt_packed_wit(prep, pb, pvf, witp, wb, wbd, sb, vf, device=True, want_range=True)
    sig_i = eng.adapt_packed(prep, pb, pvf, wit, sb, vf, device=True)
    sig_c = eng.vec_add(pre, wit, device=True)
    torch.cuda.synchronize()
    assert torch.equal(sig_w, sig_i) and torch.equal(sig_w, eng.pack(sig_c, sb, vf, device=True)) and bool(sok.all())
    del sig_i
    report(eng, f'adapt, device-resident, {n} adaptor signatures:', {
        'adapt_packed_wit (packed wit)': lambda: eng.adapt_packed_wit(prep, pb, pvf, witp, wb, wbd, sb, vf, device=True,
                                                                      want_range=True),
        'adapt_packed (int16 wit)': lambda: eng.adapt_packed(prep, pb, pvf, wit, sb, vf, device=True, want_range=True),
        'vec_add (unpacked)': lambda: eng.vec_add(pre, wit, device=True),
    }, ['unpack', 'vec_addsub', 'pack'])
    ew, eok = eng.extract_packed_wit(sig_w, sb, vf, prep, pb, pvf, wb, wbd, device=True, want_range=True)
    ex, exok = eng.extract_packed_wit(sig_w, sb, vf, prep, pb, pvf, xb, ext, device=True, want_range=True)
    ei = eng.extract_packed(sig_w, sb, vf, prep, pb, pvf, device=True)
    torch.cuda.synchronize()
    assert torch.equal(ew, witp) and torch.equal(ei, wit) and torch.equal(ex, eng.pack(wit, xb, ext, device=True))
    assert bool(eok.all()) and bool(exok.all())
    del ew, ex, ei
    report(eng, f'extract, device-resident, {n} adaptor signatures:', {
        f'extract_packed_wit ({wb}-bit wit)': lambda: eng.extract_packed_wit(sig_w, sb, vf, prep, pb, pvf, wb, wbd, device=True,
                                                                          want_range=True),
        f'extract_packed_wit ({xb}-bit wit)': lambda: eng.extract_packed_wit(sig_w, sb, vf, prep, pb, pvf, xb, ext, device=True,
                                                                           want_range=True),
        'extract_packed (int16 wit)': lambda: eng.extract_packed(sig_w, sb, vf, prep, pb, pvf, device=True),
        'vec_sub (unpacked)': lambda: eng.vec_sub(sig_c, pre, device=True),
    }, ['unpack', 'vec_addsub', 'pack'])
    del sig_c, pre

    # ---- witness verify, device-resident
    witp_m = misaligned(witp)
    v_c = torch.zeros(n, dtype=torch.uint8, device='cuda')

    def composed():
        assert lib.lcb_adaptor_witness_verify_packed_batch(eng._ctx, P(witp_m), wb, wbd, P(stp), kb, n, ext, ext_wt,
                                                           P(v_c)) == 0
    v_f = eng.witness_verify_packed(witp, wb, wbd, stp, kb, ext, ext_wt, device=True)
    v_i = eng.witness_verify(wit, st, ext, ext_wt, device=True)
    composed()
    torch.cuda.synchronize()
    assert bool(v_f.all()) and bool(v_i.all()) and bool(v_c.all())
    report(eng, f'witness verify, device-resident, {n} pairs (bound ext_wit_bd, weight ext_wit_wt):', {
        'witness_verify_packed fused': lambda: eng.witness_verify_packed(witp, wb, wbd, stp, kb, ext, ext_wt, device=True),
        'witness_verify_packed composed': composed,
        'witness_verify (int16)': lambda: eng.witness_verify(wit, st, ext, ext_wt, device=True),
    }, ['unpack', 'verify'])
    del witp_m, v_c

    # ---- from pinned host memory
    m = N_HOST

    def pinned(t):
        h = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
        h.copy_(t)
        return h
    h_pre, h_wit, h_witp, h_st, h_stp = (pinned(t[:m]) for t in (prep, wit, witp, st, stp))
    h_s1 = torch.empty((m, l, 32 * sb), dtype=torch.uint8, pin_memory=True)
    h_s2 = torch.empty((m, l, 32 * sb), dtype=torch.uint8, pin_memory=True)
    h_r = torch.empty((m, l), dtype=torch.uint8, pin_memory=True)
    h_v1 = torch.empty(m, dtype=torch.uint8, pin_memory=True)
    h_v2 = torch.empty(m, dtype=torch.uint8, pin_memory=True)
    assert all(t.is_pinned() for t in (h_pre, h_wit, h_witp, h_st, h_stp, h_s1, h_s2, h_r, h_v1, h_v2))
    mp = m * l

    def a_int16():
        assert lib.lcb_adaptor_adapt_packed_batch(eng._ctx, P(h_pre), pb, pvf, P(h_wit), mp, sb, vf, P(h_s1), P(h_r)) == 0

    def a_packed():
        assert lib.lcb_adaptor_adapt_packed_wit_batch(eng._ctx, P(h_pre), pb, pvf, P(h_witp), wb, wbd, mp, sb, vf, P(h_s2),
                                                      P(h_r)) == 0

    def v_int16():
        assert lib.lcb_adaptor_witness_verify_batch(eng._ctx, P(h_wit), P(h_st), m, ext, ext_wt, P(h_v1)) == 0

    def v_packed():
        assert lib.lcb_adaptor_witness_verify_packed_batch(eng._ctx, P(h_witp), wb, wbd, P(h_stp), kb, m, ext, ext_wt,
                                                           P(h_v2)) == 0
    hm = host_alternating({'a16': a_int16, 'apk': a_packed, 'v16': v_int16, 'vpk': v_packed})
    assert torch.equal(h_s1, h_s2) and torch.equal(h_s2, sig_w[:m].cpu()) and bool(h_r.all())
    assert bool(h_v1.all()) and bool(h_v2.all())
    pre_b, sig_b = mp * 32 * pb, mp * 32 * sb + mp
    b_a16, b_apk = pre_b + mp * 512 + sig_b, pre_b + mp * 32 * wb + sig_b
    b_v16, b_vpk = m * (l * 512 + 512 + 1), m * (l * 32 * wb + 32 * kb + 1)
    say(f'from pinned host memory, {m} items (host clock, calls end synchronised):')
    say(f'  adapt_packed (int16 wit)       {hm["a16"]:8.3f} ms   bytes over the host link {b_a16 / 1e9:.3f} GB')
    say(f'  adapt_packed_wit (packed wit)  {hm["apk"]:8.3f} ms   bytes over the host link {b_apk / 1e9:.3f} GB '
        f'({100 * (1 - b_apk / b_a16):.0f} % fewer; time {100 * (1 - hm["apk"] / hm["a16"]):.0f} % less)')
    say(f'  witness_verify (int16)         {hm["v16"]:8.3f} ms   bytes over the host link {b_v16 / 1e9:.3f} GB')
    say(f'  witness_verify_packed          {hm["vpk"]:8.3f} ms   bytes over the host link {b_vpk / 1e9:.3f} GB '
        f'({100 * (1 - b_vpk / b_v16):.0f} % fewer; time {100 * (1 - hm["vpk"] / hm["v16"]):.0f} % less)')
    del h_pre, h_wit, h_witp, h_st, h_stp, h_s1, h_s2, sig_w, prep

    # ---- witgen, device-resident
    del wit, st
    torch.cuda.synchronize()

    def witgen_then_pack():
        w, s, _ = eng.witgen(sch, seeds, want_st_coef=False, device=True)
        return eng.pack(w, wb, wbd, device=True), eng.pack(s, kb, 0, device=True)
    a_w, a_s = witgen_then_pack()
    b_w, _, b_s = eng.witgen_packed(sch, seeds, wb, wbd, kb, device=True)
    torch.cuda.synchronize()
    assert torch.equal(a_w, b_w) and torch.equal(a_s, b_s) and torch.equal(b_w, witp) and torch.equal(b_s, stp)
    del a_w, a_s, b_w, b_s
    report(eng, f'witgen, device-resident, {n} witnesses:', {
        'witgen + 2 x pack': witgen_then_pack,
        'witgen_packed': lambda: eng.witgen_packed(sch, seeds, wb, wbd, kb, device=True),
    }, ['sampler', 'matvec', 'pack'])
    eng.close()
    torch.cuda.empty_cache()


for secpar in (128, 256):
    run(secpar)
