"""Signing and adaptor verification on the packed wire format (lcb_lm_sign_packed_batch, lcb_adaptor_verify_packed_batch)
against the int16 calls they replace, on a B200 with the shipped parameters at secpar 128 and 256.

  sign, device-resident, 2^20 signatures: lm_sign alone, lm_sign + pack, lm_sign_packed (fused: k_sign writes the packed
        rows) and lm_sign_packed into a 4-byte aligned buffer (the composed route: k_sign into scratch, then k_pack);
        alternated rep by rep, CUDA events; k_sign time of each arm from lcb_profile_read
  sign, pinned host memory, 2^18 signatures: lm_sign + pack (three PCIe crossings of the int16 signature) against
        lm_sign_packed, host clock around calls that end synchronised
  adaptor verify, device-resident, 2^20 items: fused packed, composed route (4-byte aligned buffers) and the unpacked
        lm_verify with st_ntt

Every timed output is checked: packed signatures equal pack(lm_sign), in_range flags are 1, every verdict is 1.

  python tools/sign_packed_timing.py [reps] [output file]
"""
import os
import subprocess
import sys
import time
from ctypes import byref, c_void_p

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
    for _ in range(max(3, REPS // 2)):
        for k, fn in arms.items():
            t0 = time.perf_counter()
            fn()
            ts[k].append(time.perf_counter() - t0)
    return {k: 1e3 * float(np.median(v)) for k, v in ts.items()}


def run(secpar):
    pp = ad.make_setup_parameters(secpar)
    lp = pp['scheme_parameters'].lp
    q, l = lp.modulus, lp.length
    sb, kb = wire.sig_bits(pp), wire.key_bits(pp)
    pvf_bd, vf_bd, vf_wt = pp['pvf_bd'], pp['vf_bd'], pp['vf_wt']
    eng = Engine(secpar, q, 256, l)
    eng.use_torch_stream()
    lib = _ffi.load()
    sch = make_scheme(sk_bd=pp['sk_bd'], sk_wt=pp['sk_wt'], ch_bd=pp['ch_bd'], ch_wt=pp['ch_wt'], wit_bd=pp['wit_bd'],
                      wit_wt=pp['wit_wt'])
    key_ch, _ = eng.hash2polyvec('KEY_CH_SEED', ['sign packed timing'], q // 2, 256, l)
    eng.set_key_ch(np.ascontiguousarray(key_ch[0]))
    n = N_DEV
    seeds = eng.expand_seeds(bytes(range(32)), n, device=True)
    _, sk, vk, _ = eng.lm_keygen(sch, seeds, want_sk_coef=False, want_vk_coef=False, device=True)
    wit, st, _ = eng.witgen(sch, eng.expand_seeds(bytes(range(1, 33)), n, device=True), want_st_coef=False, device=True)
    cm = torch.randint(32, 127, (n * 96,), dtype=torch.uint8, device='cuda')
    co = torch.arange(0, n * 96 + 1, 96, dtype=torch.int64, device='cuda')
    msgs = (cm, co)
    torch.cuda.synchronize()
    say(f'\nsecpar {secpar}: q = {q}, l = {l}; presignatures {sb} bits (bias pvf_bd = {pvf_bd}), keys and statements {kb} bits')
    say(f'bytes per signature: int16 {l * 512}, packed {l * 32 * sb}')

    # ---- sign, device-resident
    sig = eng.lm_sign(sch, sk, msgs, device=True)
    want = eng.pack(sig, sb, pvf_bd, device=True)
    out_m = misaligned(torch.zeros_like(want))
    rng_m = torch.zeros((n, l), dtype=torch.uint8, device='cuda')

    def composed():
        assert lib.lcb_lm_sign_packed_batch(eng._ctx, byref(sch), P(sk), P(cm), P(co), n, sb, pvf_bd, P(out_m),
                                            P(rng_m)) == 0
    arms = {
        'lm_sign (int16)': lambda: eng.lm_sign(sch, sk, msgs, device=True),
        'lm_sign + pack': lambda: eng.pack(eng.lm_sign(sch, sk, msgs, device=True), sb, pvf_bd, device=True, want_range=True),
        'lm_sign_packed fused': lambda: eng.lm_sign_packed(sch, sk, msgs, sb, pvf_bd, device=True, want_range=True),
        'lm_sign_packed composed': composed,
    }
    got, ok = eng.lm_sign_packed(sch, sk, msgs, sb, pvf_bd, device=True, want_range=True)
    composed()
    torch.cuda.synchronize()
    assert torch.equal(got, want) and bool(ok.all()) and torch.equal(out_m, want) and bool(rng_m.all())
    ms = timed_alternating(arms)
    say(f'sign, device-resident, {n} signatures:')
    for k, fn in arms.items():
        say(f'  {k:26s} {ms[k]:8.3f} ms   [{kernels(eng, fn, ["sampler", "sign", "pack"])}]')
    del got, ok

    # ---- sign from pinned host memory
    m = N_HOST
    h_sk = torch.empty((m, 2, l, 256), dtype=torch.int16, pin_memory=True)
    h_sk.copy_(sk[:m].view(torch.int16))
    h_cm, h_co = cm[:m * 96].cpu().pin_memory(), co[:m + 1].cpu().pin_memory()
    h_sig = torch.empty((m, l, 256), dtype=torch.int16, pin_memory=True)
    h_p1 = torch.empty((m, l, 32 * sb), dtype=torch.uint8, pin_memory=True)
    h_p2 = torch.empty((m, l, 32 * sb), dtype=torch.uint8, pin_memory=True)     # empty_like would not pin it
    h_r = torch.empty((m, l), dtype=torch.uint8, pin_memory=True)
    assert all(t.is_pinned() for t in (h_sk, h_cm, h_co, h_sig, h_p1, h_p2, h_r)), 'both arms must use pinned buffers'

    def sign_then_pack():
        assert lib.lcb_lm_sign_batch(eng._ctx, byref(sch), P(h_sk), P(h_cm), P(h_co), m, P(h_sig)) == 0
        assert lib.lcb_pack_batch(eng._ctx, P(h_sig), m * l, sb, pvf_bd, P(h_p1), P(h_r)) == 0

    def sign_packed():
        assert lib.lcb_lm_sign_packed_batch(eng._ctx, byref(sch), P(h_sk), P(h_cm), P(h_co), m, sb, pvf_bd, P(h_p2),
                                            P(h_r)) == 0
    hm = host_alternating({'lm_sign + pack': sign_then_pack, 'lm_sign_packed': sign_packed})
    assert torch.equal(h_p1, h_p2) and torch.equal(h_p2, want[:m].cpu())
    say(f'sign from pinned host memory, {m} signatures (host clock, calls end synchronised):')
    say(f'  lm_sign + pack             {hm["lm_sign + pack"]:8.3f} ms   PCIe bytes {m * l * (2 * 512 + 32 * sb) / 1e9:.2f} GB '
        f'(+ keys {m * 2 * l * 512 / 1e9:.2f} GB)')
    say(f'  lm_sign_packed             {hm["lm_sign_packed"]:8.3f} ms   PCIe bytes {m * l * 32 * sb / 1e9:.2f} GB '
        f'(+ keys {m * 2 * l * 512 / 1e9:.2f} GB)')
    del h_sk, h_sig, h_p1, h_p2, sig, want, out_m, rng_m

    # ---- adaptor verify, device-resident
    presig = eng.lm_sign(sch, sk, msgs, device=True)
    asig = eng.vec_add(presig, wit, device=True)
    del presig, sk
    vkp, stp = eng.pack(vk, kb, 0, device=True), eng.pack(st, kb, 0, device=True)
    sigp = eng.pack(asig, sb, vf_bd, device=True)
    mv, ms_, mt = misaligned(vkp), misaligned(sigp), misaligned(stp)
    torch.cuda.synchronize()
    arms = {
        'packed fused': lambda: eng.adaptor_verify_packed(sch, vkp, kb, msgs, sigp, sb, vf_bd, stp, kb, vf_bd, vf_wt, device=True),
        'packed composed': lambda: eng.adaptor_verify_packed(sch, mv, kb, msgs, ms_, sb, vf_bd, mt, kb, vf_bd, vf_wt, device=True),
        'unpacked lm_verify(st)': lambda: eng.lm_verify(sch, vk, msgs, asig, vf_bd, vf_wt, st_ntt=st, device=True),
    }
    for k, fn in arms.items():
        v = fn()
        torch.cuda.synchronize()
        assert bool(v.all()), k
    ms = timed_alternating(arms)
    say(f'adaptor verify, device-resident, {n} items:')
    for k, fn in arms.items():
        say(f'  {k:26s} {ms[k]:8.3f} ms   [{kernels(eng, fn, ["sampler", "unpack", "verify"])}]')
    eng.close()
    torch.cuda.empty_cache()


for secpar in (128, 256):
    run(secpar)
