"""Batched BKLM aggregate / aggregate-verify on the packed wire format (lcb_bklm_aggregate_packed_batch,
lcb_bklm_aggregate_verify_packed_batch) against the unpacked batch calls on a B200: 2^18 aggregates of 2 signatures at
secpar 128 and at secpar 256 with the shipped parameters (inputs of 1.8 to 6 GB, far beyond the 126 MB L2).

  device-resident: unpacked call, packed call (fused route) and packed call from 4-byte aligned buffers (the
                   unpack-first route), alternated rep by rep, CUDA events; per-kernel times from lcb_profile_read
  host-resident:   pinned host inputs, both calls end to end (host clock around a call that ends synchronised), with
                   the bytes each moves over PCIe

Every timed output is checked: the packed aggregates equal lcb_pack_batch of the unpacked ones, every verdict is 1.

  python tools/bklm_packed_timing.py [reps] [output file]
"""
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from lattice_cryptography_b200 import Engine, make_scheme, ragged
from lattice_cryptography_b200 import bklm_one_time_agg_sigs as bk
from lattice_cryptography_b200 import wire

REPS = int(sys.argv[1]) if len(sys.argv) > 1 else 5
OUT = open(sys.argv[2], 'w') if len(sys.argv) > 2 else sys.stdout
N_AGG = 1 << 18
AGG_K = ['group_ids', 'agg_coefs_seg', 'unpack', 'agg_partial_seg', 'agg_finish', 'agg_finish_pack', 'pack']
VER_K = ['sampler', 'group_ids', 'agg_coefs_seg', 'unpack', 'aggv_partial_seg', 'aggv_residues', 'verify', 'aggv_limits']


def say(s=''):
    print(s, file=OUT, flush=True)


smi = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                     capture_output=True, text=True).stdout.strip().splitlines()
say(f'card: {torch.cuda.get_device_name(0)}; nvidia-smi name, power limit, max SM clock: {smi[0] if smi else "n/a"}')
say(f'{N_AGG} aggregates of 2 signatures per call; device times are the median of {REPS} alternated reps')


def misaligned(t):
    """a copy of t whose data pointer is 4-byte but not 16-byte aligned (forces the unpack-first route)"""
    raw = torch.empty(t.numel() * t.element_size() + 16, dtype=torch.uint8, device=t.device)
    v = raw[4:4 + t.numel() * t.element_size()]
    v.copy_(t.reshape(-1).view(torch.uint8))
    return v.view(t.dtype).view(*t.shape)


def kernels(eng, fn, names):
    eng.profile(True)
    eng.profile_reset()
    fn()
    torch.cuda.synchronize()
    out = {k: eng.profile_read(k) for k in names}
    eng.profile(False)
    return ', '.join(f'{k} {ms:.3f} ms' + (f' ({n}x)' if n > 1 else '') for k, (ms, n) in out.items() if n)


def timed_alternating(arms):
    """{name: fn}: every rep runs each arm once, in turn, between CUDA events; median ms per arm"""
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


def host_ms(fn):
    fn()
    ts = []
    for _ in range(max(3, REPS // 2)):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return 1e3 * float(np.median(ts))


def run(secpar):
    pp = bk.make_setup_parameters(secpar)
    lp = pp['scheme_parameters'].lp
    q, l = lp.modulus, lp.length
    sb, kb, ab = wire.sig_bits(pp), wire.key_bits(pp), wire.sig_bits(pp, 'avf_bd')
    vf_bd, avf_bd, avf_wt = pp['vf_bd'], pp['avf_bd'], pp['avf_wt']
    eng = Engine(secpar, q, 256, l)
    eng.use_torch_stream()
    sch = make_scheme(sk_bd=pp['sk_bd'], sk_wt=pp['sk_wt'], ch_bd=pp['ch_bd'], ch_wt=pp['ch_wt'])
    key_ch, _ = eng.hash2polyvec('KEY_CH_SEED', ['bklm packed timing'], q // 2, 256, l)
    eng.set_key_ch(np.ascontiguousarray(key_ch[0]))
    total = 2 * N_AGG
    seeds = eng.expand_seeds(bytes(range(32)), total, device=True)
    _, sk_ntt, vk, _ = eng.lm_keygen(sch, seeds, want_sk_coef=False, want_vk_coef=False, device=True)
    chm = [f'<lattice_cryptography.one_time_keys.OneTimeVerificationKey object at 0x7f{16 * i:010x}>, '
           + format((i * 2654435761) % (1 << 32), '032b') for i in range(total)]
    cb_h, co_h = ragged(chm)
    cb, co = torch.from_numpy(cb_h.copy()).cuda(), torch.from_numpy(co_h).cuda()
    sigs = eng.lm_sign(sch, sk_ntt, (cb, co), device=True)
    del sk_ntt, seeds
    off_h = np.arange(0, total + 1, 2, dtype=np.int64)
    rng = np.random.default_rng(secpar)
    mb_h = rng.integers(32, 127, 248 * N_AGG, dtype=np.uint8)
    mo_h = np.arange(0, 248 * N_AGG + 1, 248, dtype=np.int64)
    off, mb, mo = (torch.from_numpy(x).cuda() for x in (off_h, mb_h, mo_h))
    sigp = eng.pack(sigs, sb, vf_bd, device=True)
    vkp = eng.pack(vk, kb, 0, device=True)
    torch.cuda.synchronize()
    say(f'\nsecpar {secpar}: q = {q}, l = {l}; signatures {sb} bits, keys {kb} bits, aggregates {ab} bits (avf_bd {avf_bd})')

    # ---- device-resident
    agg_u = lambda: eng.aggregate_batch(sch, off, sigs, (mb, mo), device=True)
    agg_p = lambda s=sigp: eng.aggregate_packed_batch(sch, off, s, sb, vf_bd, (mb, mo), ab, avf_bd, device=True, want_range=True)
    ag = agg_u()
    agp, ok = agg_p()
    want_p, want_ok = eng.pack(ag, ab, avf_bd, device=True, want_range=True)
    assert torch.equal(agp, want_p) and torch.equal(ok, want_ok) and bool(ok.all().item())
    sigp_m = misaligned(sigp)
    agp_m, vkp_m = misaligned(agp), misaligned(vkp)
    ver_u = lambda: eng.aggregate_verify_batch(sch, off, vk, (cb, co), (mb, mo), ag, 1 << 30, avf_bd, avf_wt, device=True)
    ver_p = lambda k=vkp, a=agp: eng.aggregate_verify_packed_batch(sch, off, k, kb, (cb, co), (mb, mo), a, ab, avf_bd, 1 << 30,
                                                                  avf_bd, avf_wt, device=True)
    t = timed_alternating({'agg unpacked': agg_u, 'agg packed fused': agg_p, 'agg packed unpack-first': lambda: agg_p(sigp_m),
                           'verify unpacked': ver_u, 'verify packed fused': ver_p,
                           'verify packed unpack-first': lambda: ver_p(vkp_m, agp_m)})
    r_u, r_p, r_m = agg_u(), agg_p(), agg_p(sigp_m)
    v_u, v_p, v_m = ver_u(), ver_p(), ver_p(vkp_m, agp_m)
    torch.cuda.synchronize()
    assert torch.equal(r_p[0], eng.pack(r_u, ab, avf_bd, device=True)) and torch.equal(r_m[0], r_p[0]) and torch.equal(r_m[1], r_p[1])
    assert bool(v_u.all().item()) and torch.equal(v_u, v_p) and torch.equal(v_u, v_m)
    say('device-resident (outputs checked: packed aggregates == pack(unpacked aggregates), all verdicts 1 on every route)')
    for k, ms in t.items():
        say(f'  {k:28s} {ms:8.3f} ms = {N_AGG / ms / 1e3:7.2f} M aggregates/s')
    say('  kernels, aggregate unpacked:         ' + kernels(eng, agg_u, AGG_K))
    say('  kernels, aggregate packed fused:     ' + kernels(eng, agg_p, AGG_K))
    say('  kernels, aggregate packed unpack-1st: ' + kernels(eng, lambda: agg_p(sigp_m), AGG_K))
    say('  kernels, verify unpacked:            ' + kernels(eng, ver_u, VER_K))
    say('  kernels, verify packed fused:        ' + kernels(eng, ver_p, VER_K))
    say('  kernels, verify packed unpack-1st:   ' + kernels(eng, lambda: ver_p(vkp_m, agp_m), VER_K))
    del sigp_m, agp_m, vkp_m, r_u, r_p, r_m

    # ---- host-resident, pinned inputs
    pin = lambda x: x.cpu().pin_memory().numpy()
    sigs_h, sigp_h, vk_h, vkp_h, ag_h, agp_h = (pin(x) for x in (sigs, sigp, vk, vkp, ag, agp))
    del sigs, sigp, vk, vkp
    torch.cuda.empty_cache()
    mmsgs = (mb_h, mo_h)
    cmsgs = (cb_h, co_h)
    h = {}
    h['aggregate unpacked'] = host_ms(lambda: eng.aggregate_batch(sch, off_h, sigs_h, mmsgs))
    h['aggregate packed'] = host_ms(lambda: eng.aggregate_packed_batch(sch, off_h, sigp_h, sb, vf_bd, mmsgs, ab, avf_bd,
                                                                         want_range=True))
    h['verify unpacked'] = host_ms(lambda: eng.aggregate_verify_batch(sch, off_h, vk_h, cmsgs, mmsgs, ag_h, 1 << 30, avf_bd, avf_wt))
    h['verify packed'] = host_ms(lambda: eng.aggregate_verify_packed_batch(sch, off_h, vkp_h, kb, cmsgs, mmsgs, agp_h, ab, avf_bd,
                                                                            1 << 30, avf_bd, avf_wt))
    hu = eng.aggregate_batch(sch, off_h, sigs_h, mmsgs)
    hp, hok = eng.aggregate_packed_batch(sch, off_h, sigp_h, sb, vf_bd, mmsgs, ab, avf_bd, want_range=True)
    assert np.array_equal(hp, eng.pack(hu, ab, avf_bd)) and hok.all()
    vh_u = eng.aggregate_verify_batch(sch, off_h, vk_h, cmsgs, mmsgs, ag_h, 1 << 30, avf_bd, avf_wt)
    vh_p = eng.aggregate_verify_packed_batch(sch, off_h, vkp_h, kb, cmsgs, mmsgs, agp_h, ab, avf_bd, 1 << 30, avf_bd, avf_wt)
    assert vh_u.all() and np.array_equal(vh_u, vh_p)
    common = mb_h.nbytes + mo_h.nbytes + off_h.nbytes
    nbytes = {'aggregate unpacked': sigs_h.nbytes + ag_h.nbytes + common,
              'aggregate packed': sigp_h.nbytes + agp_h.nbytes + hok.nbytes + common,
              'verify unpacked': vk_h.nbytes + ag_h.nbytes + cb_h.nbytes + co_h.nbytes + N_AGG + common,
              'verify packed': vkp_h.nbytes + agp_h.nbytes + cb_h.nbytes + co_h.nbytes + N_AGG + common}
    say('host-resident (pinned inputs; outputs land in pageable arrays the engine allocates; outputs checked as above)')
    for k, ms in h.items():
        say(f'  {k:20s} {ms:8.2f} ms = {N_AGG / ms / 1e3:6.2f} M aggregates/s; {nbytes[k] / 1e9:.3f} GB over PCIe '
            f'({nbytes[k] / ms / 1e6:.1f} GB/s)')
    for op in ('aggregate', 'verify'):
        u, p = f'{op} unpacked', f'{op} packed'
        say(f'  {op}: packed moves {100 * (1 - nbytes[p] / nbytes[u]):.1f} % fewer bytes and takes '
            f'{100 * (1 - h[p] / h[u]):.1f} % less time')
    eng.close()


for sp in (128, 256):
    run(sp)
    torch.cuda.empty_cache()
