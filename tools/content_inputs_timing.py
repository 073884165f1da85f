"""Content-mode hash inputs on the GPU (lcb_content_str_batch, lcb_challenge_inputs_batch) against the host route they
replace, on a B200 with the shipped LM parameters at secpar 128 and 256.

  k_content_str, device-resident, 2^20 packed keys and 2^20 packed statements: kernel time (lcb_profile_read, CUDA
        events) and its rate in Keccak permutations per second (8 per key, 4 per statement) against the 4.28 Gperm/s
        Keccak roofline of tools/keccak_bench2.cu; the unpack and ntt_inv launches of the same call beside it
  packed verification of 2^20 device-resident triples from raw 32-bit messages: content strings + challenge inputs +
        lm_verify_packed, against lm_verify_packed with the challenge messages already built (the input-building share)
  the host route, 2^16 keys: unpack -> ntt_inv on the GPU -> copy to the host -> hashlib + string format per key ->
        upload of the finished challenge messages; a host figure, per key

Device arms are alternated rep by rep and timed with CUDA events (median).  Every timed output is checked: the GPU strings
of a subsample equal hashlib over the inverse transform, the host route's strings equal the GPU's, every verdict is 1.

  python tools/content_inputs_timing.py [reps] [output file]
"""
import hashlib
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from lattice_cryptography_b200 import lm_one_time_sigs as lm
from lattice_cryptography_b200 import wire

REPS = int(sys.argv[1]) if len(sys.argv) > 1 else 5
OUT = open(sys.argv[2], 'w') if len(sys.argv) > 2 else sys.stdout
N = 1 << 20
N_HOST = 1 << 16
ROOFLINE = 4.28e9
NAMES = {'vk': 'OneTimeVerificationKey', 'st': 'OneTimePublicStatement'}


def say(s=''):
    print(s, file=OUT, flush=True)


smi = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                     capture_output=True, text=True).stdout.strip().splitlines()
say(f'card: {torch.cuda.get_device_name(0)}; nvidia-smi name, power limit, max SM clock: {smi[0] if smi else "n/a"}')
say(f'device times are the median of {REPS} alternated reps (CUDA events); inputs far beyond the 126 MB L2')


def timed_alternating(arms):
    for fn in arms.values():
        fn()
    torch.cuda.synchronize()
    ts = {k: [] for k in arms}
    for _ in range(REPS):
        for k, fn in arms.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            b.synchronize()
            ts[k].append(a.elapsed_time(b))
    return {k: float(np.median(v)) for k, v in ts.items()}


def ref_str(kind, secpar, rows):
    h = hashlib.shake_256(NAMES[kind].encode() + secpar.to_bytes(2, 'little') + rows.astype('<i2').tobytes())
    return f'<{NAMES[kind]} {h.hexdigest(16)}>'


def kernel_ms(e, fn, names):
    e.profile(True)
    e.profile_reset()
    for _ in range(REPS):
        fn()
    e.synchronize()
    out = {k: e.profile_read(k)[0] / REPS for k in names}
    e.profile(False)
    return out


for secpar in (128, 256):
    pp = lm.make_setup_parameters(secpar)
    e, sch = lm._ctx(pp)
    e.use_torch_stream()
    kb = wire.key_bits(pp)
    say()
    say(f'=== secpar {secpar}: keys and statements packed at {kb} bits')
    rng = np.random.default_rng(secpar)
    gen = torch.Generator(device='cuda').manual_seed(secpar)
    # ---- k_content_str on 2^20 keys / statements (random packed bytes: the kernel's work does not depend on them)
    for kind, lead, perms in (('vk', (N, 2), 8), ('st', (N,), 4)):
        packed = torch.randint(0, 256, lead + (32 * kb,), dtype=torch.uint8, device='cuda', generator=gen)
        out = e.content_str(kind, packed, kb, device=True)
        coef = e.ntt_inv(e.unpack(packed[:64].cpu().numpy(), kb, 0, dtype=np.uint16))
        got = out[:64].cpu().numpy()
        assert all(bytes(got[i]).decode() == ref_str(kind, secpar, coef[i]) for i in range(64))
        ms = kernel_ms(e, lambda: e.content_str(kind, packed, kb, device=True), ('content_str', 'unpack', 'ntt_inv'))
        t = timed_alternating({'call': lambda: e.content_str(kind, packed, kb, device=True)})['call']
        rate = perms * N / (ms['content_str'] * 1e-3)
        say(f'{kind}: 2^20 items, {perms} permutations each: k_content_str {ms["content_str"]:.3f} ms = {rate / 1e9:.2f} Gperm/s '
            f'= {rate / ROOFLINE:.2f} of the 4.28 Gperm/s Keccak roofline; k_unpack {ms["unpack"]:.3f} ms, k_ntt_inv '
            f'{ms["ntt_inv"]:.3f} ms; whole call {t:.3f} ms ({N / t / 1e3:.1f} M strings/s)')
        del packed, out
    # ---- packed verification of 2^20 triples from raw messages
    seeds = e.expand_seeds(bytes(range(32)), N, device=True)
    skp, _, vkp = e.lm_keygen_packed(sch, seeds, wire.signing_key_bits(pp), pp['sk_bd'], kb, device=True)
    mlen = 32
    mblob = torch.randint(48, 50, (N * mlen,), dtype=torch.uint8, device='cuda', generator=gen)
    moff = torch.arange(N + 1, dtype=torch.int64, device='cuda') * mlen
    vk_str = e.content_str('vk', vkp, kb, device=True)
    chm = e.challenge_inputs(vk_str, (mblob, moff), device=True)
    sigp = e.lm_sign_packed_sk(sch, skp, wire.signing_key_bits(pp), pp['sk_bd'], chm, wire.sig_bits(pp), pp['vf_bd'],
                               device=True)
    del skp
    verdict = torch.empty(N, dtype=torch.uint8, device='cuda')

    def from_raw():
        s = e.content_str('vk', vkp, kb, device=True)
        c = e.challenge_inputs(s, (mblob, moff), device=True)
        e.lm_verify_packed(sch, vkp, kb, c, sigp, wire.sig_bits(pp), pp['vf_bd'], pp['vf_bd'], pp['vf_wt'], out=verdict)

    def prebuilt():
        e.lm_verify_packed(sch, vkp, kb, chm, sigp, wire.sig_bits(pp), pp['vf_bd'], pp['vf_bd'], pp['vf_wt'], out=verdict)

    t = timed_alternating({'from_raw': from_raw, 'prebuilt': prebuilt})
    from_raw()
    assert bool(verdict.all())
    ms = kernel_ms(e, from_raw, ('content_str', 'challenge_inputs'))
    say(f'packed verify of 2^20 triples, {mlen}-bit messages: from raw messages {t["from_raw"]:.3f} ms '
        f'({N / t["from_raw"] / 1e3:.2f} M verifies/s), with prebuilt chmsgs {t["prebuilt"]:.3f} ms '
        f'({N / t["prebuilt"] / 1e3:.2f} M verifies/s); input building {t["from_raw"] - t["prebuilt"]:.3f} ms = '
        f'{(t["from_raw"] - t["prebuilt"]) / t["from_raw"]:.0%} of the step (k_content_str {ms["content_str"]:.3f} ms, '
        f'k_challenge_inputs {ms["challenge_inputs"]:.3f} ms)')
    # ---- the host route it replaces, 2^16 keys
    vh = vkp[:N_HOST]
    mh = [bytes(r).decode() for r in mblob[:N_HOST * mlen].view(N_HOST, mlen).cpu().numpy()]
    torch.cuda.synchronize()
    times = []
    for _ in range(max(1, REPS // 2)):
        t0 = time.perf_counter()
        coef = e.ntt_inv(e.unpack(vh, kb, 0, dtype=np.uint16, device=True), device=True).cpu().numpy()
        strs = [ref_str('vk', secpar, coef[i]) + ', ' + mh[i] for i in range(N_HOST)]
        from lattice_cryptography_b200 import ragged
        b, o = ragged(strs)
        up = (torch.from_numpy(b).cuda(), torch.from_numpy(o).cuda())
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
    th = float(np.median(times))
    gb, go = e.challenge_inputs(e.content_str('vk', vh, kb, device=True), (mblob[:N_HOST * mlen].contiguous(),
                                                                             moff[:N_HOST + 1].contiguous()), device=True)
    assert torch.equal(gb, up[0]) and torch.equal(go, up[1])
    say(f'host route, 2^16 keys (unpack -> ntt_inv -> copy back -> hashlib + format per key -> upload): {th * 1e3:.1f} ms = '
        f'{th / N_HOST * 1e6:.2f} us per key (host figure: one CPU thread of the GPU machine); the GPU route makes the same '
        f'bytes')
    del vkp, sigp, mblob, moff, chm, vk_str, verdict
    torch.cuda.empty_cache()
say()
say('lane form: one thread per sponge (k_content_str); the two-lanes-per-sponge form was not built or measured')
