"""The content-mode BKLM route on the device (lcb_content_order_batch, lcb_gather_rows_batch, lcb_gather_ragged_batch and
wire.aggregate_batch_content / aggregate_verify_batch_content) against the host route it replaces, on a B200 with the
shipped BKLM parameters (ag_cap = 2).

  k_content_order, device-resident random 57-byte rows: 2^16 .. 2^20 items in groups of two (the per-item path, with
        the k_group_ids launch beside it), and one group of 2^16 items (the radix path); an L2-sized buffer is
        overwritten before every launch, so no input is read from L2
  k_gather_rows, device-resident, 2^19 rows of 57 / 896 / 4,576 / 9,568 bytes in a random order: achieved bytes/s
        (bytes read + bytes written over kernel time) against the 7.7 TB/s of HBM3e
  the whole route at 2^19 items (2^18 groups of two), secpar 128 and 256: aggregate and aggregate-verify from unsorted
        packed keys, raw 32-bit messages and packed signatures (aggregates), all on the device, against the host route
        (wire.aggregation_inputs + numpy permutation of the packed records + the packed batch call on host arrays);
        the outputs of the two routes are asserted equal in the same run

  python tools/content_order_timing.py [reps] [output file]
"""
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from lattice_cryptography_b200 import bklm_one_time_agg_sigs as bk
from lattice_cryptography_b200 import wire

REPS = int(sys.argv[1]) if len(sys.argv) > 1 else 5
OUT = open(sys.argv[2], 'w') if len(sys.argv) > 2 else sys.stdout
HBM = 7.7e12
N_ROUTE = 1 << 19
FLUSH = torch.empty(256 << 20, dtype=torch.uint8, device='cuda')


def say(s=''):
    print(s, file=OUT, flush=True)


smi = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                     capture_output=True, text=True).stdout.strip().splitlines()
say(f'card: {torch.cuda.get_device_name(0)}; nvidia-smi name, power limit, max SM clock: {smi[0] if smi else "n/a"}')
say(f'kernel times: mean of {REPS} launches (lcb_profile_read, CUDA events), a 256 MB buffer overwritten before each; '
    f'route times: median of {REPS} (device, CUDA events) / of 2 (host, wall clock to a synchronised end)')


def kernel_ms(e, fn, names):
    fn()
    e.synchronize()
    e.profile(True)
    e.profile_reset()
    for _ in range(REPS):
        FLUSH.zero_()
        fn()
    e.synchronize()
    out = {k: e.profile_read(k) for k in names}
    e.profile(False)
    return {k: (ms / REPS, n // REPS) for k, (ms, n) in out.items()}


def device_ms(fn):
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(REPS):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts))


def host_s(fn):
    ts = []
    for _ in range(2):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts))


pp = bk.make_setup_parameters(128)
e, _ = bk._ctx(pp)
e.use_torch_stream()
gen = torch.Generator(device='cuda').manual_seed(1)

# ---- k_content_order
say()
say('=== k_content_order (random rows)')
for lg in range(16, 21):
    n = 1 << lg
    rows = torch.randint(0, 256, (n, 57), dtype=torch.uint8, device='cuda', generator=gen)
    off = torch.arange(n // 2 + 1, dtype=torch.int64, device='cuda') * 2
    got = e.content_order(off, rows, device=True).cpu().numpy()
    h = rows.cpu().numpy()
    assert np.array_equal(got, np.lexsort((h.view('S57').reshape(-1), np.arange(n) // 2)))
    ms = kernel_ms(e, lambda: e.content_order(off, rows, device=True), ('content_order', 'group_ids'))
    call = device_ms(lambda: e.content_order(off, rows, device=True))
    say(f'2^{lg} items in groups of two: k_content_order {ms["content_order"][0]:.3f} ms ({n / ms["content_order"][0] / 1e6:.2f} G '
        f'items/s), k_group_ids {ms["group_ids"][0]:.3f} ms; whole call {call:.3f} ms (agg_off read back on the host)')
n = 1 << 16
rows = torch.randint(0, 256, (n, 57), dtype=torch.uint8, device='cuda', generator=gen)
off = torch.tensor([0, n], dtype=torch.int64, device='cuda')
got = e.content_order(off, rows, device=True).cpu().numpy()
assert np.array_equal(got, np.lexsort((rows.cpu().numpy().view('S57').reshape(-1),)))
ms = kernel_ms(e, lambda: e.content_order(off, rows, device=True), ('content_order',))
call = device_ms(lambda: e.content_order(off, rows, device=True))
say(f'one group of 2^16 items (radix path: 9 CUB passes + key and scatter kernels, {ms["content_order"][1]} timed launch): '
    f'{ms["content_order"][0]:.3f} ms; whole call {call:.3f} ms')

# ---- k_gather_rows
say()
say('=== k_gather_rows, 2^19 rows in a random order (bytes read + written over kernel time)')
n = 1 << 19
idx = torch.randperm(n, device='cuda', generator=gen)
for row in (57, 896, 4576, 9568):
    src = torch.randint(0, 256, (n, row), dtype=torch.uint8, device='cuda', generator=gen)
    out = e.gather_rows(src, idx, device=True)
    assert torch.equal(out, src[idx])
    del out
    ms = kernel_ms(e, lambda: e.gather_rows(src, idx, device=True), ('gather_rows',))['gather_rows'][0]
    moved = 2 * n * row + 8 * n
    say(f'{row:5d}-byte rows ({n * row / 1e9:.2f} GB): {ms:.3f} ms = {moved / ms / 1e9:.2f} TB/s = {moved / ms / 1e9 / (HBM / 1e12):.2f} '
        f'of 7.7 TB/s')
    del src
torch.cuda.empty_cache()

# ---- the whole route
for secpar in (128, 256):
    pp = bk.make_setup_parameters(secpar)
    e, sch = bk._ctx(pp)
    e.use_torch_stream()
    kb, sb = wire.key_bits(pp), wire.sig_bits(pp)
    say()
    say(f'=== secpar {secpar}: 2^19 items in 2^18 groups of two, 32-bit messages, keys {kb} bits, signatures {sb} bits')
    seeds = e.expand_seeds(bytes(range(32)), N_ROUTE, device=True)
    skp, _, vkp = e.lm_keygen_packed(sch, seeds, wire.signing_key_bits(pp), pp['sk_bd'], kb, device=True)
    mblob = torch.randint(48, 50, (N_ROUTE * 32,), dtype=torch.uint8, device='cuda', generator=gen)
    moff = torch.arange(N_ROUTE + 1, dtype=torch.int64, device='cuda') * 32
    chm = wire.challenge_inputs(pp, vkp, (mblob, moff), device=True)
    sigp = e.lm_sign_packed_sk(sch, skp, wire.signing_key_bits(pp), pp['sk_bd'], chm, sb, pp['vf_bd'], device=True)
    del skp, chm
    off = torch.arange(N_ROUTE // 2 + 1, dtype=torch.int64, device='cuda') * 2
    h_off, h_vkp, h_sigp = off.cpu().numpy(), vkp.cpu().numpy(), sigp.cpu().numpy()
    h_msgs = [bytes(r).decode() for r in mblob.view(N_ROUTE, 32).cpu().numpy()]

    def host_aggregate():
        order, _, agmsgs = wire.aggregation_inputs(pp, h_off, h_vkp, h_msgs)
        return wire.aggregate_batch_packed(pp, h_off, np.ascontiguousarray(h_sigp[order]), agmsgs)

    def host_verify(agp):
        order, chmsgs, agmsgs = wire.aggregation_inputs(pp, h_off, h_vkp, h_msgs)
        return wire.aggregate_verify_batch_packed(pp, h_off, np.ascontiguousarray(h_vkp[order]), chmsgs, agmsgs, agp)

    def dev_aggregate():
        return wire.aggregate_batch_content(pp, off, vkp, (mblob, moff), sigp, device=True)

    h_ag = host_aggregate()
    d_ag = dev_aggregate()
    assert np.array_equal(d_ag[0].cpu().numpy(), h_ag[0]) and np.array_equal(d_ag[1].cpu().numpy(), h_ag[1])
    assert h_ag[1].all()
    agp = d_ag[0]
    h_v = host_verify(h_ag[0])
    d_v = wire.aggregate_verify_batch_content(pp, off, vkp, (mblob, moff), agp, device=True)
    assert np.array_equal(d_v.cpu().numpy(), h_v) and h_v.all()
    t_ha = host_s(host_aggregate)
    t_hv = host_s(lambda: host_verify(h_ag[0]))
    t_da = device_ms(dev_aggregate)
    t_dv = device_ms(lambda: wire.aggregate_verify_batch_content(pp, off, vkp, (mblob, moff), agp, device=True))
    ms = kernel_ms(e, dev_aggregate, ('content_str', 'content_order', 'gather_rows', 'gather_ragged', 'aggregation_inputs',
                                      'agg_coefs_seg', 'agg_partial_seg', 'agg_finish_pack'))
    say(f'aggregate:        device route {t_da:.2f} ms, host route {t_ha * 1e3:.0f} ms: {t_ha * 1e3 / t_da:.0f}x; outputs equal')
    say(f'aggregate-verify: device route {t_dv:.2f} ms, host route {t_hv * 1e3:.0f} ms: {t_hv * 1e3 / t_dv:.0f}x; verdicts equal '
        f'(all 1)')
    say('  kernels of the device aggregate (ms per call): ' + ', '.join(f'{k} {v[0]:.3f}' for k, v in ms.items()))
    del seeds, vkp, sigp, mblob, moff, off, d_ag, d_v, agp
    torch.cuda.empty_cache()
