"""Batched BKLM aggregate / aggregate-verify (lcb_bklm_aggregate_batch, lcb_bklm_aggregate_verify_batch) on a B200,
secpar 128 with the shipped parameters, device-resident inputs far beyond the 126 MB L2, CUDA events around warm calls:

  (a) 2^18 aggregates of 2 signatures (the reference's ag_cap)   (b) 2^14 aggregates of 16
  (c) a mixed batch of sizes 1 .. 64                              (d) one aggregate of 2^16, against the single path

For each: aggregates/s and signatures/s of both calls and the per-kernel times from lcb_profile_read (a separate,
profiled pass).  Then the per-aggregate loop over the single-aggregate entry points on 4,096 aggregates of (a), and the
drop-in aggregate_verify_batch on 4,096 object-level aggregates (host-side string work included).  Every timed batch
is checked to verify (all verdicts 1).

  python tools/bklm_batch_timing.py [reps]
"""
import os
import subprocess
import sys
import time
from ctypes import byref, c_void_p

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from lattice_cryptography_b200 import Engine, _ffi, make_scheme, ragged

REPS = int(sys.argv[1]) if len(sys.argv) > 1 else 5
Q, L, D, CH_WT, SK_BD = 11777, 13, 256, 20, 45
POOL = 1 << 19
BATCH_KERNELS = ['sampler', 'group_ids', 'agg_coefs_seg', 'agg_partial_seg', 'agg_finish', 'aggv_partial_seg',
                 'aggv_residues', 'verify', 'aggv_limits']

smi = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                     capture_output=True, text=True).stdout.strip().splitlines()
print(f'card: {torch.cuda.get_device_name(0)}; nvidia-smi name, power limit, max SM clock: {smi[0] if smi else "n/a"}')

eng = Engine(128, Q, D, L)
eng.use_torch_stream()
sch = make_scheme(sk_bd=SK_BD, sk_wt=D, ch_bd=1, ch_wt=CH_WT)
key_ch, _ = eng.hash2polyvec('KEY_CH_SEED', ['bklm batch timing'], Q // 2, D, L)
eng.set_key_ch(np.ascontiguousarray(key_ch[0]))
seeds = eng.expand_seeds(bytes(range(32)), POOL, device=True)
_, sk_ntt, vk, _ = eng.lm_keygen(sch, seeds, want_sk_coef=False, want_vk_coef=False, device=True)
chm = [f'<lattice_cryptography.one_time_keys.OneTimeVerificationKey object at 0x7f{16 * i:010x}>, '
       + format((i * 2654435761) % (1 << 32), '032b') for i in range(POOL)]
cblob, coff = ragged(chm)
cblob, coff = torch.from_numpy(cblob.copy()).cuda(), torch.from_numpy(coff).cuda()
sigs = eng.lm_sign(sch, sk_ntt, (cblob, coff), device=True)
del sk_ntt
torch.cuda.synchronize()
AVF_BD, AVF_WT = Q // 2, D


def workload(sizes, seed):
    """device (agg_off, agmsg blob, agmsg offsets) for groups of the given sizes: each aggregation message is
    str(list(zip(keys, msgs))) of its group (122 bytes per entry + separators), as the drop-in builds it."""
    off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    lens = 124 * np.asarray(sizes, np.int64)
    rng = np.random.default_rng(seed)
    mblob = rng.integers(32, 127, int(lens.sum()), dtype=np.uint8)
    moff = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    return [torch.from_numpy(x).cuda() for x in (off, mblob, moff)]


def events_ms(fn):
    for _ in range(2):
        fn()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(REPS):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / REPS


def kernels(fn):
    eng.profile(True)
    eng.profile_reset()
    fn()
    torch.cuda.synchronize()
    out = {k: eng.profile_read(k) for k in BATCH_KERNELS}
    eng.profile(False)
    return ', '.join(f'{k} {ms:.3f} ms' + (f' ({n}x)' if n > 1 else '') for k, (ms, n) in out.items() if n)


def run(name, sizes, seed):
    sizes = np.asarray(sizes, np.int64)
    n_agg, total = len(sizes), int(sizes.sum())
    off, mblob, moff = workload(sizes, seed)
    cb = cblob[:int(coff[total].item())]
    co = coff[:total + 1]
    s, v = sigs[:total], vk[:total]
    ag = eng.aggregate_batch(sch, off, s, (mblob, moff), device=True)
    verdict = eng.aggregate_verify_batch(sch, off, v, (cb, co), (mblob, moff), ag, 1 << 30, AVF_BD, AVF_WT, device=True)
    assert bool(verdict.all().item()), f'{name}: an honest aggregate did not verify'
    t_agg = events_ms(lambda: eng.aggregate_batch(sch, off, s, (mblob, moff), device=True))
    t_ver = events_ms(lambda: eng.aggregate_verify_batch(sch, off, v, (cb, co), (mblob, moff), ag, 1 << 30, AVF_BD, AVF_WT,
                                                         device=True))
    print(f'\n({name}) {n_agg} aggregates, {total} signatures, sizes {int(sizes.min())}..{int(sizes.max())}')
    for what, t in (('aggregate_batch', t_agg), ('aggregate_verify_batch', t_ver)):
        print(f'  {what}: {t:.3f} ms = {n_agg / t / 1e3:.3f} M aggregates/s, {total / t / 1e3:.3f} M signatures/s')
    print('  kernels, aggregate_batch:        ' + kernels(lambda: eng.aggregate_batch(sch, off, s, (mblob, moff), device=True)))
    print('  kernels, aggregate_verify_batch: ' + kernels(lambda: eng.aggregate_verify_batch(
        sch, off, v, (cb, co), (mblob, moff), ag, 1 << 30, AVF_BD, AVF_WT, device=True)))
    return off, mblob, moff, ag


off_a, mblob_a, moff_a, ag_a = run('a', [2] * (1 << 18), 1)
run('b', [16] * (1 << 14), 2)
mixed = np.random.default_rng(3).integers(1, 65, 16000)
run('c', mixed[:np.searchsorted(np.cumsum(mixed), POOL, side='right')], 3)
off_d, mblob_d, moff_d, ag_d = run('d', [1 << 16], 4)

# (d) against the single-aggregate path (k_agg_coefs_il + k_agg_partial / k_aggv_partial + finish)
lib = _ffi.load()
P = lambda t: c_void_p(t.data_ptr())
part = torch.empty(L * D, dtype=torch.int32, device='cuda')
vpart = torch.empty(D, dtype=torch.int32, device='cuda')
out1 = torch.empty(L * D, dtype=torch.int16, device='cuda')
ver1 = torch.empty(1, dtype=torch.uint8, device='cuda')
n16 = 1 << 16
msg_d = mblob_d


def single(first, count, msg, sig_rows, vk_rows, ch_blob, ch_off, ag_sig):
    eng._ck(lib.lcb_bklm_aggregate_partial(eng._ctx, byref(sch), P(sig_rows), None, P(msg), int(msg.shape[0]), 0, count, P(part)))
    eng._ck(lib.lcb_bklm_aggregate_finish(eng._ctx, P(part), P(out1)))
    eng._ck(lib.lcb_bklm_aggverify_partial(eng._ctx, byref(sch), P(vk_rows), P(ch_blob), P(ch_off), None, P(msg),
                                           int(msg.shape[0]), 0, count, P(vpart)))
    eng._ck(lib.lcb_bklm_aggverify_finish(eng._ctx, P(vpart), P(ag_sig), count, 1 << 30, AVF_BD, AVF_WT, P(ver1)))


cb16 = cblob[:int(coff[n16].item())]
t_single = events_ms(lambda: single(0, n16, msg_d, sigs, vk, cb16, coff[:n16 + 1], ag_d[0]))
assert int(ver1.item()) == 1 and torch.equal(out1.view(L, D), ag_d[0])
print(f'\n(d) single-aggregate path, aggregate + aggregate_verify of the same 2^16 group: {t_single:.3f} ms '
      f'(k_agg_coefs_il: two lanes per sponge; the batch path above uses one thread per sponge)')
print('  kernels: ' + kernels(lambda: single(0, n16, msg_d, sigs, vk, cb16, coff[:n16 + 1], ag_d[0]))
      + ', ' + ', '.join(f'{k} {eng.profile_read(k)[0]:.3f} ms' for k in ('agg_coefs', 'agg_partial', 'aggv_partial')))

# the per-aggregate loop over the single-aggregate entry points: 4,096 aggregates of (a), device buffers
N_LOOP = 4096
off_h = off_a.cpu().numpy()
moff_h = moff_a.cpu().numpy()
coff_h = coff.cpu().numpy()
groups = []
for g in range(N_LOOP):
    a, b = int(off_h[g]), int(off_h[g + 1])
    ch_off = torch.from_numpy(coff_h[a:b + 1] - coff_h[a]).cuda()
    groups.append((a, b - a, mblob_a[int(moff_h[g]):int(moff_h[g + 1])], sigs[a:b], vk[a:b],
                   cblob[int(coff_h[a]):int(coff_h[b])], ch_off, ag_a[g]))
for gr in groups[:8]:
    single(*gr)
torch.cuda.synchronize()
l0 = eng.launch_count
t0 = time.perf_counter()
for gr in groups:
    single(*gr)
torch.cuda.synchronize()
dt = time.perf_counter() - t0
per_launch = (eng.launch_count - l0) / N_LOOP
print(f'\nper-aggregate loop, {N_LOOP} aggregates of 2 (aggregate + aggregate_verify each, host clock to a device sync): '
      f'{dt * 1e3:.1f} ms = {N_LOOP / dt / 1e3:.2f} k aggregates/s, {per_launch:.1f} launches per aggregate')
off4 = off_a[:N_LOOP + 1]
n4 = 2 * N_LOOP
cb4, co4 = cblob[:int(coff_h[n4])], coff[:n4 + 1]
m4 = mblob_a[:int(moff_h[N_LOOP])]
mo4 = moff_a[:N_LOOP + 1]
t_b4 = events_ms(lambda: (eng.aggregate_batch(sch, off4, sigs[:n4], (m4, mo4), device=True),
                          eng.aggregate_verify_batch(sch, off4, vk[:n4], (cb4, co4), (m4, mo4), ag_a[:N_LOOP], 1 << 30,
                                                     AVF_BD, AVF_WT, device=True)))
print(f'the same {N_LOOP} aggregates through the two batch calls: {t_b4:.3f} ms = {N_LOOP / t_b4 / 1e3:.2f} M aggregates/s')

# the drop-in aggregate_verify_batch on 4,096 object-level aggregates of 2
from lattice_cryptography_b200 import bklm_one_time_agg_sigs as bk
from lattice_cryptography_b200.lm_one_time_sigs import keygen, sign
pp = bk.make_setup_parameters(128)
keys = keygen(pp=pp, num_keys_to_gen=2 * N_LOOP)
msgs = [format((7 * i + 3) % (1 << 32), '032b') for i in range(2 * N_LOOP)]
osigs = [sign(pp=pp, otk=k, msg=m) for k, m in zip(keys, msgs)]
gk = [[keys[2 * g][2], keys[2 * g + 1][2]] for g in range(N_LOOP)]
gm = [msgs[2 * g:2 * g + 2] for g in range(N_LOOP)]
gs = [osigs[2 * g:2 * g + 2] for g in range(N_LOOP)]
ags = bk.aggregate_batch(pp, gk, gm, gs)
assert all(bk.aggregate_verify_batch(pp, gk, gm, ags))
engine_s = []
dropin_ctx = bk._ctx


def timed_ctx(pp_):
    """the drop-in's engine, with its one aggregate_verify_batch call timed (host inputs: the call ends synchronised)"""
    e, s_ = dropin_ctx(pp_)

    class Timed(object):
        def __getattr__(self, name):
            return getattr(e, name)

        def aggregate_verify_batch(self, *a, **k):
            t0_ = time.perf_counter()
            r = e.aggregate_verify_batch(*a, **k)
            engine_s.append(time.perf_counter() - t0_)
            return r
    return Timed(), s_


bk._ctx = timed_ctx
times = []
for _ in range(3):
    t0 = time.perf_counter()
    bk.aggregate_verify_batch(pp, gk, gm, ags)
    times.append(time.perf_counter() - t0)
k = int(np.argmin(times))
dt, de = times[k], engine_s[k]
print(f'\ndrop-in aggregate_verify_batch, {N_LOOP} object-level aggregates of 2: {dt * 1e3:.1f} ms = '
      f'{N_LOOP / dt / 1e3:.2f} k aggregates/s; the engine call inside it (host buffers staged, one synchronisation) '
      f'{de * 1e3:.1f} ms, so the host-side work (sorting, str(list(zip(...))), challenge strings, key stacking) is '
      f'{(dt - de) * 1e3:.1f} ms = {100 * (dt - de) / dt:.0f} % of the call')
