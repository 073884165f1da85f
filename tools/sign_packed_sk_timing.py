"""Packed keys (lcb_lm_keygen_packed_batch, lcb_lm_sign_packed_sk_batch) against the calls they replace, on a B200 with the
shipped parameters at secpar 128 and 256.

  sign, device-resident, 2^20 signatures: lm_sign_packed from uint16 NTT-form keys (k_sign with the packed epilogue),
        lm_sign_packed_sk on the fused route (k_sign_sk: rotations of the packed coefficient-form rows) and on the composed
        route (a 4-byte aligned key buffer: k_unpack -> k_ntt_fwd -> k_sign); alternated rep by rep, CUDA events; per-kernel
        times from lcb_profile_read
  sign, pinned host memory, 2^18 signatures: lm_sign_packed (NTT-form keys cross the host link) against lm_sign_packed_sk
        (packed keys), host clock around calls that end synchronised, and the bytes each moves
  keygen, device-resident, 2^20 keys: lm_keygen_packed against lm_keygen (sk_coef, vk_ntt) + two packs

Every timed output is checked: the packed signatures of all arms are equal, in_range flags are 1, packed keys equal
pack(keygen).

  python tools/sign_packed_sk_timing.py [reps] [output file]
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
from lattice_cryptography_b200 import lm_one_time_sigs as lm
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


def run(secpar):
    pp = lm.make_setup_parameters(secpar)
    lp = pp['scheme_parameters'].lp
    q, l = lp.modulus, lp.length
    sb, kb, skb = wire.sig_bits(pp), wire.key_bits(pp), wire.signing_key_bits(pp)
    vf_bd, sk_bd = pp['vf_bd'], pp['sk_bd']
    eng = Engine(secpar, q, 256, l)
    eng.use_torch_stream()
    lib = _ffi.load()
    sch = make_scheme(sk_bd=sk_bd, sk_wt=pp['sk_wt'], ch_bd=pp['ch_bd'], ch_wt=pp['ch_wt'])
    key_ch, _ = eng.hash2polyvec('KEY_CH_SEED', ['sign packed sk timing'], q // 2, 256, l)
    eng.set_key_ch(np.ascontiguousarray(key_ch[0]))
    n = N_DEV
    seeds = eng.expand_seeds(bytes(range(32)), n, device=True)
    sk_coef, sk_ntt, vk_ntt, _ = eng.lm_keygen(sch, seeds, want_vk_coef=False, device=True)
    skp = eng.pack(sk_coef, skb, sk_bd, device=True)
    del sk_coef
    cm = torch.randint(32, 127, (n * 96,), dtype=torch.uint8, device='cuda')
    co = torch.arange(0, n * 96 + 1, 96, dtype=torch.int64, device='cuda')
    msgs = (cm, co)
    torch.cuda.synchronize()
    say(f'\nsecpar {secpar}: q = {q}, l = {l}, ch_wt = {pp["ch_wt"]}; signing keys {skb} bits (bias sk_bd = {sk_bd}), '
        f'signatures {sb} bits (bias vf_bd = {vf_bd})')
    say(f'bytes per signing key: uint16 NTT form {2 * l * 512}, packed coefficient form {2 * l * 32 * skb}; '
        f'per signature (packed) {l * 32 * sb}')

    # ---- sign, device-resident
    want, want_ok = eng.lm_sign_packed(sch, sk_ntt, msgs, sb, vf_bd, device=True, want_range=True)
    skp_m = misaligned(skp)
    out_c = torch.zeros_like(want)
    rng_c = torch.zeros((n, l), dtype=torch.uint8, device='cuda')

    def composed():
        assert lib.lcb_lm_sign_packed_sk_batch(eng._ctx, byref(sch), P(skp_m), skb, sk_bd, P(cm), P(co), n, sb, vf_bd, P(out_c),
                                               P(rng_c)) == 0
    arms = {
        'lm_sign_packed (NTT keys)': lambda: eng.lm_sign_packed(sch, sk_ntt, msgs, sb, vf_bd, device=True, want_range=True),
        'sign_packed_sk fused': lambda: eng.lm_sign_packed_sk(sch, skp, skb, sk_bd, msgs, sb, vf_bd, device=True, want_range=True),
        'sign_packed_sk composed': composed,
    }
    got, ok = eng.lm_sign_packed_sk(sch, skp, skb, sk_bd, msgs, sb, vf_bd, device=True, want_range=True)
    composed()
    torch.cuda.synchronize()
    assert torch.equal(got, want) and torch.equal(out_c, want) and bool(want_ok.all()) and bool(ok.all()) and bool(rng_c.all())
    ms = timed_alternating(arms)
    say(f'sign, device-resident, {n} signatures:')
    for k, fn in arms.items():
        say(f'  {k:28s} {ms[k]:8.3f} ms   [{kernels(eng, fn, ["sampler", "unpack", "ntt_fwd", "sign", "pack"])}]')
    del got, ok, out_c, rng_c, skp_m

    # ---- sign from pinned host memory
    m = N_HOST
    h_ntt = torch.empty((m, 2, l, 256), dtype=torch.int16, pin_memory=True)
    h_ntt.copy_(sk_ntt[:m].view(torch.int16))
    h_skp = torch.empty((m, 2, l, 32 * skb), dtype=torch.uint8, pin_memory=True)
    h_skp.copy_(skp[:m])
    h_cm, h_co = cm[:m * 96].cpu().pin_memory(), co[:m + 1].cpu().pin_memory()
    h_p1 = torch.empty((m, l, 32 * sb), dtype=torch.uint8, pin_memory=True)
    h_p2 = torch.empty((m, l, 32 * sb), dtype=torch.uint8, pin_memory=True)
    h_r = torch.empty((m, l), dtype=torch.uint8, pin_memory=True)
    assert all(t.is_pinned() for t in (h_ntt, h_skp, h_cm, h_co, h_p1, h_p2, h_r)), 'both arms must use pinned buffers'

    def from_ntt():
        assert lib.lcb_lm_sign_packed_batch(eng._ctx, byref(sch), P(h_ntt), P(h_cm), P(h_co), m, sb, vf_bd, P(h_p1), P(h_r)) == 0

    def from_packed():
        assert lib.lcb_lm_sign_packed_sk_batch(eng._ctx, byref(sch), P(h_skp), skb, sk_bd, P(h_cm), P(h_co), m, sb, vf_bd,
                                               P(h_p2), P(h_r)) == 0
    hm = host_alternating({'ntt': from_ntt, 'packed': from_packed})
    assert torch.equal(h_p1, h_p2) and torch.equal(h_p2, want[:m].cpu()) and bool(h_r.all())
    msg_b, sig_b = m * (96 + 8), m * l * 32 * sb
    b_ntt, b_pk = m * 2 * l * 512 + msg_b + sig_b, m * 2 * l * 32 * skb + msg_b + sig_b
    say(f'sign from pinned host memory, {m} signatures (host clock, calls end synchronised):')
    say(f'  lm_sign_packed (NTT keys)    {hm["ntt"]:8.3f} ms   bytes over the host link {b_ntt / 1e9:.2f} GB')
    say(f'  sign_packed_sk               {hm["packed"]:8.3f} ms   bytes over the host link {b_pk / 1e9:.2f} GB '
        f'({100 * (1 - b_pk / b_ntt):.0f} % fewer; time {100 * (1 - hm["packed"] / hm["ntt"]):.0f} % less)')
    del h_ntt, h_skp, h_p1, h_p2, want, want_ok, sk_ntt, skp

    # ---- keygen, device-resident
    vk_want = eng.pack(vk_ntt, kb, 0, device=True)
    del vk_ntt
    torch.cuda.synchronize()

    def keygen_then_pack():
        skc, _, vkn, _ = eng.lm_keygen(sch, seeds, want_sk_ntt=False, want_vk_coef=False, device=True)
        return eng.pack(skc, skb, sk_bd, device=True), eng.pack(vkn, kb, 0, device=True)
    a_sk, a_vk = keygen_then_pack()
    b_sk, _, b_vk = eng.lm_keygen_packed(sch, seeds, skb, sk_bd, kb, device=True)
    torch.cuda.synchronize()
    assert torch.equal(a_sk, b_sk) and torch.equal(a_vk, b_vk) and torch.equal(b_vk, vk_want)
    del a_sk, a_vk, b_sk, b_vk
    arms = {'lm_keygen + 2 x pack': keygen_then_pack,
            'lm_keygen_packed': lambda: eng.lm_keygen_packed(sch, seeds, skb, sk_bd, kb, device=True)}
    ms = timed_alternating(arms)
    say(f'keygen, device-resident, {n} keys:')
    for k, fn in arms.items():
        say(f'  {k:28s} {ms[k]:8.3f} ms   [{kernels(eng, fn, ["sampler", "matvec", "pack"])}]')
    eng.close()
    torch.cuda.empty_cache()


for secpar in (128, 256):
    run(secpar)
