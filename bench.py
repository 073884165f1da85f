#!/usr/bin/env python
"""bench.py — headline benchmark of the lcb200 engine.

Metric (BASELINE.json): LM-OTS verifies/sec.  Workload (BASELINE.json configs[1]): batched LM-OTS
verify of 2^20 independent (vk, msg, sig) triples at secpar = 128 per B200.  A "step" is one pass
of the verify path (challenge sampler kernel + verify kernel) over the whole batch.  With N > 1 GPUs
every rank verifies its own 2^20 triples (independent units, no data-path collective): weak scaling.

  python bench.py [--gpus N] [--steps K] [--warmup W]            # engine arm
  python bench.py --impl reference [--gpus N] [--steps K] ...    # the reference's CPU algorithm (oracle port)
  python bench.py --dump-outputs DIR ...                         # also write the last timed step's verdicts to DIR
"""
import argparse
import json
import os
import sys
import time

# the benchmark may run from a read-only tree: no bytecode caches are written next to the sources
sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SHIPPED = {128: dict(q=11777, l=13, sk_bd=45, ch_wt=20, vf_bd=945, vf_wt=256),
           256: dict(q=39937, l=23, sk_bd=65, ch_wt=50, vf_bd=3315, vf_wt=256)}
D = 256
KEY_CH_SEED = 'lcb200 bench key_ch v1'
METRIC = 'LM-OTS verifies/sec'
UNIT = 'verifies/s'


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='engine', choices=['engine', 'reference'])
    ap.add_argument('--secpar', type=int, default=128, choices=[128, 256])
    ap.add_argument('--log2n', type=int, default=20, help='log2 of triples per GPU')
    ap.add_argument('--e2e-steps', type=int, default=2)
    ap.add_argument('--cpu-per-core', type=int, default=32, help='CPU baseline: verifies per host core')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-secondary', action='store_true', help='skip the keygen+sign / BKLM / adaptor measurements')
    ap.add_argument('--bklm-log2n', type=int, default=16, help='log2 of signatures per aggregate (whole job)')
    ap.add_argument('--keygen-log2n', type=int, default=20, help='configs[2]: log2 of seeds, whole job (split over the GPUs)')
    ap.add_argument('--adaptor-log2n', type=int, default=18, help='configs[4]: log2 of instances, whole job')
    ap.add_argument('--cpu-bklm-log2n', type=int, default=8, help='CPU baseline: largest BKLM aggregate actually run')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='engine arm: write the verdicts of the last timed step as DIR/verdict.npy (float32; '
                         'verdict_rank<r>.npy per rank when several run), so that two builds can be compared output '
                         'for output on the same seeded inputs')
    a = ap.parse_args()
    if a.dump_outputs and a.impl != 'engine':
        ap.error('--dump-outputs writes what the engine arm computes')
    return a


def workload_name(a):
    return f'lm_ots_verify_batch secpar={a.secpar} n=2^{a.log2n} triples per GPU'


def engine_config(a):
    p = SHIPPED[a.secpar]
    n = 1 << a.log2n
    gb = (n * p['l'] * D * 2 + n * 2 * D * 2 + n * (86 + a.secpar)) / 1e9
    return {'workload': workload_name(a), 'secpar': a.secpar, 'q': p['q'], 'd': D, 'l': p['l'], 'triples_per_gpu': n,
            'tampered_every': 64, 'l2': f'inputs {gb:.2f} GB per pass >> 126 MB L2, no flush needed'}


# ---------------------------------------------------------------------------------------------------
def cpu_leg(secpar, per_core, extras=None):
    """The oracle port on every host core, bounded sample (see oracle/cpu_baseline.py).  `extras` = args: also time
    the other halves of the metric (keygen / sign phases, BKLM with the a*N^2 + b*N extrapolation of BASELINE.md
    section 3, the adaptor flow) for the `also` / `secondary` figures of the line."""
    sys.path.insert(0, os.path.join(ROOT, 'oracle'))
    import cpu_baseline
    cores = os.cpu_count() or 1
    sample = per_core * cores
    r = cpu_baseline.lm_verify_throughput(secpar, sample, cores)
    leg = {'value': r['value'], 'unit': UNIT, 'cores': r['cores'], 'kind': 'port',
           'sample': f'{sample} honest LM-OTS triples at secpar {secpar} ({per_core} per core), verify() only timed, '
                     f'pure-Python port of lattice_algebra (oracle/), slowest worker {r["elapsed_s"]:.2f} s'}
    if extras is not None:
        t0 = time.perf_counter()
        ns = tuple(n for n in (2, 16, 64, 256, 1024) if n <= (1 << extras.cpu_bklm_log2n))
        leg['phases_secpar256'] = cpu_baseline.lm_phase_throughput(256, max(cores, 8), cores)
        leg['bklm'] = cpu_baseline.bklm_extrapolation(128, ns=ns, target=1 << extras.bklm_log2n, nproc=cores)
        leg['adaptor'] = cpu_baseline.adaptor_throughput(128, 64, cores)
        leg['extras_wall_s'] = time.perf_counter() - t0
    return leg


def reference_arm(a):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    vals, t0 = [], time.perf_counter()
    leg = None
    for step in range(a.warmup + a.steps):
        leg = cpu_leg(a.secpar, max(1, a.cpu_per_core // 2))
        if step >= a.warmup:
            vals.append(leg['value'])
    v = sum(vals) / len(vals)
    leg['value'] = v
    line = {'impl': 'reference', 'metric': METRIC, 'value': v, 'unit': UNIT, 'n_gpus': a.gpus, 'steps': a.steps,
            'warmup': a.warmup, 'ms_per_step': 1e3 * (time.perf_counter() - t0) / (a.warmup + a.steps),
            'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'python-int', 'data': 'synthetic',
            # the engine arm's config, key for key (each step here is a bounded sample of that workload, see cpu_baseline.sample)
            'config': engine_config(a),
            'cpu_baseline': leg,
            'e2e': {'value': v, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'gpu_launches': 0}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------
def bind_to_gpu_numa_node(local):
    """Pin this rank's host threads to the CPUs NVML reports as local to its GPU, BEFORE any pinned host buffer is
    allocated: the end-to-end legs stream 6-8 GB per step from pinned memory, and first-touch placement on the
    GPU's own NUMA node keeps that traffic off the inter-socket link.  Best effort; returns what it did."""
    try:
        import pynvml
        import torch
        pynvml.nvmlInit()
        try:
            h = pynvml.nvmlDeviceGetHandleByUUID(('GPU-' + str(torch.cuda.get_device_properties(local).uuid)).encode())
        except Exception:
            h = pynvml.nvmlDeviceGetHandleByIndex(local)
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = {64 * i + b for i, w in enumerate(words) for b in range(64) if (int(w) >> b) & 1}
        cpus &= set(os.sched_getaffinity(0))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


class ClockSampler(object):
    """SM clock / power / throttle reasons sampled every 5 ms by NVML in a thread DURING the timed region."""
    REASONS = {0x8: 'hw_slowdown', 0x40: 'hw_thermal_slowdown', 0x20: 'sw_thermal_slowdown', 0x4: 'sw_power_cap'}

    def __init__(self, device):
        import threading
        self.rows, self.stop_flag, self.h = [], False, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            try:        # by UUID, so that CUDA_VISIBLE_DEVICES remapping cannot point NVML at another GPU
                import torch
                self.h = pynvml.nvmlDeviceGetHandleByUUID(('GPU-' + str(torch.cuda.get_device_properties(device).uuid)).encode())
            except Exception:
                self.h = pynvml.nvmlDeviceGetHandleByIndex(device)
            self.max_sm = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            return
        self.t = threading.Thread(target=self._loop, daemon=True)
        self.t.start()

    def _loop(self):
        nv = self.nv
        while not self.stop_flag:
            try:
                try:
                    reasons = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    reasons = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.rows.append((nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM),
                                  nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0, reasons))
            except Exception:
                pass
            time.sleep(0.005)

    def stop(self):
        out = {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': []}
        if self.h is None:
            return out
        self.stop_flag = True
        self.t.join(timeout=2)
        if not self.rows:
            return out
        sm = sorted(r[0] for r in self.rows)
        out['sm_mhz'] = float(sm[len(sm) // 2])
        out['sm_min_mhz'] = float(sm[0])
        out['sm_max_mhz'] = float(self.max_sm)
        out['power_w_max'] = max(r[1] for r in self.rows)
        seen = 0
        for r in self.rows:
            seen |= r[2]
        out['reasons'] = [name for bit, name in self.REASONS.items() if seen & bit]
        out['samples'] = len(self.rows)
        return out


def build_inputs(a, rank, torch, np):
    """Synthetic seeds / messages of the benchmark's shape, built as byte matrices (no Python loops)."""
    n = 1 << a.log2n
    rng = np.random.default_rng(20260101 + rank)
    seeds = (rng.integers(0, 2, (n, a.secpar), dtype=np.uint8) + ord('0')).astype(np.uint8)
    head = np.frombuffer(b'<lattice_cryptography.one_time_keys.OneTimeVerificationKey object at 0x7f', dtype=np.uint8)
    idx = (np.arange(n, dtype=np.int64) + rank * n) * 16
    hexd = np.frombuffer(b'0123456789abcdef', dtype=np.uint8)
    addr = np.stack([hexd[(idx >> (4 * (9 - k))) & 15] for k in range(10)], axis=1)
    tail = np.frombuffer(b'>, ', dtype=np.uint8)
    bits = (rng.integers(0, 2, (n, a.secpar), dtype=np.uint8) + ord('0')).astype(np.uint8)
    ch = np.concatenate([np.broadcast_to(head, (n, head.size)), addr, np.broadcast_to(tail, (n, 3)), bits], axis=1)
    ch = np.ascontiguousarray(ch)
    seed_off = np.arange(n + 1, dtype=np.int64) * a.secpar
    ch_off = np.arange(n + 1, dtype=np.int64) * ch.shape[1]
    return seeds.reshape(-1), seed_off, ch, ch_off


DUMP_BYTES = 64 << 20


def dump_outputs(dirname, arrays, world, np):
    """Writes every array of `arrays` (name -> array) as <dirname>/<name>.npy in float32.  All ranks together write at
    most DUMP_BYTES: a larger output is replaced by a fixed sample, its elements at indices drawn by a generator seeded
    with 0 (the same indices on every run with the same arguments)."""
    os.makedirs(dirname, exist_ok=True)
    cap = DUMP_BYTES // 4 // (world * len(arrays))
    for name, arr in arrays.items():
        if arr.size > cap:
            arr = arr.reshape(-1)[np.sort(np.random.default_rng(0).choice(arr.size, cap, replace=False))]
        np.save(os.path.join(dirname, name + '.npy'), arr.astype(np.float32))


# ---------------------------------------------------------------------------------------------------
# Secondary measurements (BASELINE.json configs[2..4] at sizes that keep the default run short).  Timed
# with CUDA events on the engine's stream, max over ranks; none of them is the headline metric.
def _timed(torch, dist, world, dev, fn, reps=3):
    """Median device time of `reps` calls after one warm-up call (max over ranks).  The median keeps a one-off
    allocator hiccup (torch or the stream-ordered pool growing) out of the secondary figures."""
    fn()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    times = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        times.append(e0.elapsed_time(e1))
    times.sort()
    ms = torch.tensor([times[len(times) // 2]], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return float(ms.item())


def _peaks():
    """Roofline denominators: measured HBM copy bandwidth (driver-written MEASURED_PEAKS.json, else the profiling
    recipe's fallback) and the integer issue limit 148 SMs x 4 schedulers x 32 lanes x max SM clock."""
    peaks, src = {}, 'fallback (B200_PROFILING.md)'
    try:
        with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as f:
            peaks, src = json.load(f), 'MEASURED_PEAKS.json'
    except OSError:
        pass
    mhz = peaks.get('sm_max_mhz', 1965.0)
    return {'hbm_gbs': peaks.get('hbm_gbs', 6650.0), 'source': src, 'sm_max_mhz': mhz,
            'int_tinstr_s': 148 * 128 * mhz * 1e6 / 1e12}


def _ncu_summary(kernel):
    """Figures of the newest committed ncu --set full digest of `kernel` (profiles/prof_r*_<kernel>.summary.txt), or
    None.  Only a digest that names its capture batch and commit (tools/digest_profiles.sh writes a `# capture:`
    line) is used: numbers of an older build must not ride along silently."""
    import glob
    import re
    best = None
    for path in sorted(glob.glob(os.path.join(ROOT, 'profiles', f'prof_r*_{kernel}.summary.txt'))):
        txt = open(path).read()
        cap = re.search(r'# capture: units=(\d+) commit=(\w+)', txt)
        if not cap:
            continue
        num = lambda key: (lambda m: float(m.group(1).replace(',', '')) if m else None)(re.search(re.escape(key) + r'\s+([\d.,]+)', txt))
        unit = lambda key: (lambda m: m.group(1) if m else '')(re.search(re.escape(key) + r'\s+[\d.,]+\s+(\w+)', txt))
        scale = {'Gbyte': 1e9, 'Mbyte': 1e6, 'Kbyte': 1e3, 'byte': 1.0}
        rd, wr = num('dram__bytes_read.sum'), num('dram__bytes_write.sum')
        if rd is None or wr is None:
            continue
        units = int(cap.group(1))
        best = {'source': os.path.relpath(path, ROOT), 'commit': cap.group(2), 'units_per_captured_launch': units,
                'dram_bytes_per_unit': (rd * scale.get(unit('dram__bytes_read.sum'), 1.0) +
                                        wr * scale.get(unit('dram__bytes_write.sum'), 1.0)) / units,
                'warp_instr_per_unit': (num('smsp__inst_executed.sum') or 0) / units,
                'issue_active_pct': num('smsp__issue_active.avg.pct_of_peak_sustained_active'),
                'pipe_alu_pct': num('sm__inst_executed_pipe_alu.avg.pct_of_peak_sustained_active'),
                'pipe_fma_pct': num('sm__inst_executed_pipe_fma.avg.pct_of_peak_sustained_active'),
                'pipe_lsu_pct': num('sm__inst_executed_pipe_lsu.avg.pct_of_peak_sustained_active')}
    return best


def _engine(secpar, local, np):
    from lattice_cryptography_b200 import Engine, make_scheme
    p = SHIPPED[secpar]
    eng = Engine(secpar, p['q'], D, p['l'], device=local)
    eng.use_torch_stream()
    key_ch, _ = eng.hash2polyvec('KEY_CH_SEED', [KEY_CH_SEED], p['q'] // 2, D, p['l'])
    eng.set_key_ch(np.ascontiguousarray(key_ch[0]))
    sch = make_scheme(sk_bd=p['sk_bd'], sk_wt=256, ch_bd=1, ch_wt=p['ch_wt'], wit_bd=1, wit_wt=20)
    return eng, sch, p


def _c_oracle():
    """oracle/lcb_oracle.c through ctypes: the CHECKER of the secondary legs (never timed, never on the product path)."""
    sys.path.insert(0, os.path.join(ROOT, 'oracle'))
    import c_oracle
    return c_oracle


def _chmsg_str(ch_row):
    return bytes(ch_row.tolist())


def secondary_keygen_sign(a, rank, local, world, torch, np, dist):
    """configs[2]: keygen + sign from 2^20 synthetic seeds at secpar 256, split over the GPUs (2^20 on one GPU at
    N = 1); a random subsample of keys and signatures is compared coefficient by coefficient with the C oracle."""
    class A: secpar, log2n = 256, max(0, a.keygen_log2n - (world.bit_length() - 1))
    eng, sch, p = _engine(256, local, np)
    dev = f'cuda:{local}'
    n = 1 << A.log2n
    seeds, seed_off, ch, ch_off = build_inputs(A, rank, torch, np)
    d_seeds = (torch.from_numpy(seeds).to(dev), torch.from_numpy(seed_off).to(dev))
    d_ch = (torch.from_numpy(ch).to(dev).view(-1), torch.from_numpy(ch_off).to(dev))
    out = {}

    def run():
        out.clear()
        _, sk_ntt, vk_ntt, _ = eng.lm_keygen(sch, d_seeds, want_sk_coef=False, want_vk_coef=False, device=True)
        out['sig'] = eng.lm_sign(sch, sk_ntt, d_ch, device=True)
        out['vk'] = vk_ntt
    ms = _timed(torch, dist, world, dev, run, reps=3)
    ok = bool(eng.lm_verify(sch, out['vk'], d_ch, out['sig'], p['vf_bd'], p['vf_wt'], device=True).all().item())
    # ---- checker: 12 random instances against the C oracle (keys from the seed, signature from the hash input)
    orc = _c_oracle()
    op = orc.params(256, p['q'], p['l'], p['sk_bd'], p['ch_wt'])
    key_ch, _ = eng.hash2polyvec('KEY_CH_SEED', [KEY_CH_SEED], p['q'] // 2, D, p['l'])
    pick = np.sort(np.random.default_rng(99 + rank).choice(n, 12, replace=False))
    d_pick = torch.from_numpy(pick).to(dev)
    vk_coef = eng.ntt_inv(out['vk'].view(torch.int16)[d_pick].contiguous().view(torch.uint16))
    sig_pick = out['sig'][d_pick].cpu().numpy()
    matches = 0
    for j, i in enumerate(pick):
        skl, skr, vkl, vkr = orc.lm_keygen(op, np.ascontiguousarray(key_ch[0]), bytes(seeds[i * 256:(i + 1) * 256].tolist()))
        osig = orc.lm_sign(op, skl, skr, _chmsg_str(ch[i]))
        matches += int(np.array_equal(vkl, vk_coef[j, 0]) and np.array_equal(vkr, vk_coef[j, 1]) and
                       np.array_equal(osig, sig_pick[j]))
    eng.close()
    perms = 2 * 2853 + 26
    return {'keys_per_s': world * n / (ms * 1e-3), 'ms': ms, 'n_per_gpu': n, 'n_total': world * n, 'all_verify': ok,
            'oracle_subsample': {'checked': len(pick), 'bit_exact': matches, 'checker': 'oracle/lcb_oracle.c'},
            'keccak_gperm_s_per_gpu': n * perms / (ms * 1e-3) / 1e9, 'keccak_roofline_gperm_s': 4.28}


def secondary_verify_secpar256(a, rank, local, world, torch, np, dist):
    """The headline path on the other shipped parameter set: 2^18 (vk, msg, sig) triples per GPU at secpar 256
    (q = 39937, l = 23, ch_wt = 50; 13.2 KB and 26 permutations per verify)."""
    class A: secpar, log2n = 256, 18
    eng, sch, p = _engine(256, local, np)
    dev = f'cuda:{local}'
    n = 1 << A.log2n
    seeds, seed_off, ch, ch_off = build_inputs(A, rank, torch, np)
    d_seeds = (torch.from_numpy(seeds).to(dev), torch.from_numpy(seed_off).to(dev))
    d_ch = (torch.from_numpy(ch).to(dev).view(-1), torch.from_numpy(ch_off).to(dev))
    _, sk_ntt, vk_ntt, _ = eng.lm_keygen(sch, d_seeds, want_sk_coef=False, want_vk_coef=False, device=True)
    sig = eng.lm_sign(sch, sk_ntt, d_ch, device=True)
    del sk_ntt
    torch.cuda.synchronize()
    bad = torch.arange(0, n, 64, device=dev)
    sig.view(torch.int16)[bad, bad % p['l'], (3 * bad) % D] += 1
    torch.cuda.synchronize()
    verdict = torch.empty(n, dtype=torch.uint8, device=dev)
    ms = _timed(torch, dist, world, dev, lambda: eng.lm_verify(sch, vk_ntt, d_ch, sig, p['vf_bd'], p['vf_wt'], out=verdict))
    expect = torch.ones(n, dtype=torch.uint8, device=dev)
    expect[bad] = 0
    ok = bool(torch.equal(verdict, expect))
    eng.profile(True)
    eng.profile_reset()
    eng.lm_verify(sch, vk_ntt, d_ch, sig, p['vf_bd'], p['vf_wt'], out=verdict)
    v_ms, _ = eng.profile_read('verify')
    s_ms, _ = eng.profile_read('sampler')
    eng.profile(False)
    eng.close()
    return {'verifies_per_s': world * n / (ms * 1e-3), 'ms': ms, 'n_per_gpu': n, 'verdicts_as_constructed': ok,
            'k_verify_ms': v_ms, 'k_sampler_ms': s_ms,
            'keccak_gperm_s_per_gpu': n * 26 / (s_ms * 1e-3) / 1e9, 'keccak_roofline_gperm_s': 4.28}


def secondary_bklm(a, rank, local, world, torch, np, dist):
    """configs[3]: aggregate + aggregate-verify of 2^k signatures per aggregate (secpar 128), the sorted list
    sharded over the ranks, ONE reduce of int32 partial sums each.  Two rows (SURVEY.md 8d):
      (i)  exact reference semantics, including the O(N^2) aggregation-coefficient hashing (Keccak-bound);
      (ii) the algebra alone with the coefficients supplied: k_agg_partial (a pure HBM stream, 6,656 B per
           signature) and challenge sampler + k_aggv_partial, on 2^k signatures PER GPU.
    A hashlib subsample checks the coefficients and the aggregate is compared with a numpy statement of the sum."""
    import hashlib
    from lattice_cryptography_b200.distributed import reduce_partial, shard_range
    class A: secpar, log2n = 128, a.bklm_log2n
    eng, sch, p = _engine(128, local, np)
    dev = f'cuda:{local}'
    total = 1 << A.log2n
    start, count = shard_range(total, rank, world)
    # synthetic keys / 32-bit messages; object addresses ascend, so sorted order == index order
    rng = np.random.default_rng(777)
    bits = rng.integers(0, 2, (total, 32), dtype=np.uint8) + ord('0')
    msgs = [bytes(r).decode() for r in bits]
    ident = [f'<lattice_cryptography.one_time_keys.OneTimeVerificationKey object at 0x7f{16 * i:010x}>' for i in range(total)]
    agmsg_b = ('[' + ', '.join(f"({k}, '{m}')" for k, m in zip(ident, msgs)) + ']').encode()
    agmsg = np.frombuffer(agmsg_b, dtype=np.uint8)
    d_agmsg = torch.from_numpy(agmsg.copy()).to(dev)
    seeds = [bin((0x9E3779B97F4A7C15 * (i + 1)) % (1 << 128))[2:].zfill(128) for i in range(start, start + count)]
    chm = [k + ', ' + m for k, m in zip(ident[start:start + count], msgs[start:start + count])]
    from lattice_cryptography_b200 import ragged
    cb, co = ragged(chm)
    d_chm = (torch.from_numpy(cb.copy()).to(dev), torch.from_numpy(co).to(dev))
    _, sk_ntt, vk_ntt, _ = eng.lm_keygen(sch, seeds, want_sk_coef=False, want_vk_coef=False, device=True)
    sigs = eng.lm_sign(sch, sk_ntt, d_chm, device=True)
    del sk_ntt
    res = {}

    # ---- row (i): exact
    def agg():
        ag = eng.agg_coefs(sch, d_agmsg, start, count, device=True)
        part = eng.aggregate_partial(sch, sigs, ag, device=True)
        part = reduce_partial(part)
        res['ag'] = ag
        if rank == 0:
            res['ag_sig'] = eng.aggregate_finish(part, device=True)
    ms_agg = _timed(torch, dist, world, dev, agg, reps=1)
    ag_sig = res.get('ag_sig')
    if world > 1:
        if rank != 0:
            ag_sig = torch.empty((p['l'], D), dtype=torch.int16, device=dev)
        dist.broadcast(ag_sig.view(torch.uint8), src=0)      # NCCL has no int16
    avf_bd = min(p['q'] // 2, total * p['vf_bd'])

    def aggv():
        ag = eng.agg_coefs(sch, d_agmsg, start, count, device=True)
        part = eng.aggverify_partial(sch, vk_ntt, d_chm, ag, device=True)
        part = reduce_partial(part)
        if rank == 0:
            res['ok'] = eng.aggverify_finish(part, ag_sig, total, total, avf_bd, 256)
    ms_aggv = _timed(torch, dist, world, dev, aggv, reps=1)
    eng.profile(True)
    eng.profile_reset()
    eng.agg_coefs(sch, d_agmsg, start, count, device=True)
    coef_ms, _ = eng.profile_read('agg_coefs')
    eng.profile(False)

    # ---- checker (untimed): coefficients against hashlib on this rank's shard, the aggregate against numpy
    coefs = res['ag'].cpu().numpy()
    pick = sorted({0, 1, count // 2, count - 1} | set(int(i) for i in rng.integers(0, count, 8)))
    h0 = hashlib.shake_256(b'AG_SALT')
    coef_ok = 0
    for i in pick:
        h = h0.copy()
        h.update(str(start + i).encode() + agmsg_b)
        dg = h.digest(2)
        coef_ok += int((int(coefs[i, 0, 0]), int(coefs[i, 0, 1])) == (dg[0], 1 if dg[1] & 0x80 else -1))
    sum_ok = None
    if world == 1 and total <= (1 << 16):
        h_sig = sigs.cpu().numpy()
        acc = np.zeros((p['l'], D), dtype=np.int64)
        pp_ = np.arange(D)
        for a0 in range(0, total, 2048):
            k = coefs[a0:a0 + 2048, 0, 0].astype(np.int64)[:, None]
            src = (pp_[None, :] - k) & (D - 1)
            sign = np.where(pp_[None, :] < k, -1, 1) * coefs[a0:a0 + 2048, 0, 1].astype(np.int64)[:, None]
            rot = np.take_along_axis(h_sig[a0:a0 + 2048].astype(np.int64),
                                     np.broadcast_to(src[:, None, :], (src.shape[0], p['l'], D)), axis=2)
            acc += (rot * sign[:, None, :]).sum(axis=0)
        want = acc % p['q']
        want = np.where(want > (p['q'] - 1) // 2, want - p['q'], want).astype(np.int16)
        sum_ok = bool(np.array_equal(want, ag_sig.cpu().numpy()))
        del h_sig

    # ---- row (ii): coefficients supplied, 2^k signatures per GPU
    reps_ = total // count
    sig_ii = sigs if reps_ == 1 else sigs.repeat(reps_, 1, 1)
    vk_ii = vk_ntt if reps_ == 1 else vk_ntt.view(torch.int16).repeat(reps_, 1, 1).view(torch.uint16)
    ag_ii = res['ag'] if reps_ == 1 else res['ag'].repeat(reps_, 1, 1)
    chm_ii = d_chm if reps_ == 1 else (d_chm[0].repeat(reps_), torch.arange(total + 1, device=dev, dtype=torch.int64) * (cb.shape[0] // count))
    n_ii = int(sig_ii.shape[0])
    eng.profile(True)
    ii = {}
    for name, fn, kern in (('aggregate', lambda: eng.aggregate_partial(sch, sig_ii, ag_ii, device=True), 'agg_partial'),
                           ('aggregate_verify', lambda: eng.aggverify_partial(sch, vk_ii, chm_ii, ag_ii, device=True), 'aggv_partial')):
        fn()
        eng.profile_reset()
        ms = _timed(torch, dist, world, dev, fn, reps=3)
        k_ms, k_n = eng.profile_read(kern)
        ii[name] = {'ms': ms, 'sigs_per_s_per_gpu': n_ii / (ms * 1e-3), 'kernel': 'k_' + kern,
                    'kernel_ms_per_launch': k_ms / max(k_n, 1)}
    eng.profile(False)
    peaks = _peaks()
    sig_bytes = p['l'] * D * 2
    k = ii['aggregate']
    k['roofline'] = {'bound': 'hbm', 'algorithmic_bytes_per_unit': sig_bytes + 4,
                     'achieved': (sig_bytes + 4) * n_ii / (k['kernel_ms_per_launch'] * 1e-3) / 1e9, 'peak': peaks['hbm_gbs'],
                     'unit': 'GB/s'}
    k['roofline']['frac'] = k['roofline']['achieved'] / k['roofline']['peak']
    k = ii['aggregate_verify']
    instr = 8192 + 3 * 256 * 6          # SURVEY 8(d): one NTT-256 + three pointwise passes per signature (Keccak is the sampler's)
    k['roofline'] = {'bound': 'int_issue', 'algorithmic_instr_per_unit': instr,
                     'achieved': instr * n_ii / (k['kernel_ms_per_launch'] * 1e-3) / 1e12, 'peak': peaks['int_tinstr_s'],
                     'unit': 'Tinstr/s'}
    k['roofline']['frac'] = k['roofline']['achieved'] / k['roofline']['peak']
    # ---- row (iii): the linear-time NON-REFERENCE mode (SURVEY 8(f)4; bklm_one_time_agg_sigs 'tree' mode): the message
    # is bound into a two-level SHAKE256 tree commitment on the GPU, every coefficient then hashes one block
    from lattice_cryptography_b200.bklm_one_time_agg_sigs import TREE_DOMAIN, TREE_LEAF_BYTES
    cuts = list(range(0, len(agmsg_b), TREE_LEAF_BYTES)) + [len(agmsg_b)]
    d_cuts = torch.tensor(cuts, dtype=torch.int64, device=dev)
    head = torch.from_numpy(np.frombuffer(TREE_DOMAIN + len(agmsg_b).to_bytes(8, 'little'), dtype=np.uint8).copy()).to(dev)
    d_top_off = torch.tensor([0, head.numel() + 32 * (len(cuts) - 1)], dtype=torch.int64, device=dev)

    def commit():
        leaves = eng.shake256((d_agmsg, d_cuts), 32, device=True)
        top = torch.cat([head, leaves.reshape(-1)])
        return bytes(eng.shake256((top, d_top_off), 32, device=True)[0].cpu().numpy()).hex().encode()

    def agg_tree():
        ag = eng.agg_coefs(sch, commit(), start, count, device=True)
        part = reduce_partial(eng.aggregate_partial(sch, sigs, ag, device=True))
        if rank == 0:
            res['ag_sig_tree'] = eng.aggregate_finish(part, device=True)
    agg_tree()
    ms_agg_t = _timed(torch, dist, world, dev, agg_tree, reps=3)
    ag_sig_t = res.get('ag_sig_tree')
    if world > 1:
        if rank != 0:
            ag_sig_t = torch.empty((p['l'], D), dtype=torch.int16, device=dev)
        dist.broadcast(ag_sig_t.view(torch.uint8), src=0)

    def aggv_tree():
        ag = eng.agg_coefs(sch, commit(), start, count, device=True)
        part = reduce_partial(eng.aggverify_partial(sch, vk_ntt, d_chm, ag, device=True))
        if rank == 0:
            res['ok_tree'] = eng.aggverify_finish(part, ag_sig_t, total, total, avf_bd, 256)
    aggv_tree()
    ms_aggv_t = _timed(torch, dist, world, dev, aggv_tree, reps=3)
    leaves_h = b''.join(hashlib.shake_256(agmsg_b[c0:c1]).digest(32) for c0, c1 in zip(cuts[:-1], cuts[1:]))
    root_h = hashlib.shake_256(TREE_DOMAIN + len(agmsg_b).to_bytes(8, 'little') + leaves_h).digest(32).hex().encode()
    tree = {'mode': "pp['ag_mode'] = 'tree': NOT the reference's coefficients (explicit opt-in), same algebra",
            'aggregate_ms': ms_agg_t, 'aggregate_verify_ms': ms_aggv_t,
            'aggregate_sigs_per_s': total / (ms_agg_t * 1e-3), 'aggregate_verify_sigs_per_s': total / (ms_aggv_t * 1e-3),
            'verdict': res.get('ok_tree') if rank == 0 else None, 'commitment_vs_hashlib': commit() == root_h,
            'reference_mode_rejects_it': (not eng.aggverify_finish(reduce_partial(eng.aggverify_partial(
                sch, vk_ntt, d_chm, res['ag'], device=True)), ag_sig_t, total, total, avf_bd, 256)) if world == 1 else None}
    eng.close()
    perms = count * ((len(agmsg) + 12) // 136 + 1)
    return {'sigs_per_aggregate': total, 'aggregate_sigs_per_s': total / (ms_agg * 1e-3),
            'aggregate_verify_sigs_per_s': total / (ms_aggv * 1e-3), 'aggregate_ms': ms_agg,
            'aggregate_verify_ms': ms_aggv, 'verdict': res.get('ok') if rank == 0 else None,
            'checker': {'coefficients_vs_hashlib': f'{coef_ok}/{len(pick)}', 'aggregate_vs_numpy_sum': sum_ok},
            'agmsg_bytes': int(len(agmsg)), 'agg_coefs_ms_rank0': coef_ms, 'streams_per_gpu': count,
            'agg_coefs_gperm_s_per_gpu': perms / (coef_ms * 1e-3) / 1e9, 'keccak_roofline_gperm_s': 4.28,
            'row_ii_coefficients_supplied': dict(ii, signatures_per_gpu=n_ii),
            'row_iii_tree_mode_nonreference': tree}


def secondary_single_ops(a, rank, local, world, torch, np, dist):
    """configs[0]: one key / one signature / one verification through the drop-in Python API (the reference's own
    calls, benchmarks/demo_signing.py), median wall-clock latency of 20 calls per secpar on rank 0."""
    if rank != 0:
        return None
    import statistics
    from lattice_cryptography_b200 import lattice_algebra as gla
    from lattice_cryptography_b200 import lm_one_time_sigs as lm
    gla.set_default_device(local)
    out = {}
    for secpar in (128, 256):
        pp = lm.make_setup_parameters(secpar)
        key = lm.keygen(pp=pp, num_keys_to_gen=1)[0]
        sig = lm.sign(pp=pp, otk=key, msg='QRL is awesome!')
        assert lm.verify(pp=pp, otvk=key[2], msg='QRL is awesome!', sig=sig)
        t = {'keygen': [], 'sign': [], 'verify': []}
        for _ in range(20):
            t0 = time.perf_counter()
            key = lm.keygen(pp=pp, num_keys_to_gen=1)[0]
            t1 = time.perf_counter()
            sig = lm.sign(pp=pp, otk=key, msg='QRL is awesome!')
            t2 = time.perf_counter()
            ok = lm.verify(pp=pp, otvk=key[2], msg='QRL is awesome!', sig=sig)
            t3 = time.perf_counter()
            assert ok
            t['keygen'].append(t1 - t0)
            t['sign'].append(t2 - t1)
            t['verify'].append(t3 - t2)
        out[f'secpar{secpar}_ms'] = {k: 1e3 * statistics.median(v) for k, v in t.items()}
    out['note'] = ('host-visible latency of single drop-in calls (Python objects in, Python objects out); the published '
                   'CPU log of the reference has 122 / 20 / 65-106 ms (secpar 128) for the same three calls')
    return out


def secondary_adaptor(a, rank, local, world, torch, np, dist):
    """configs[4]: adaptor pre-sign / pre-verify / adapt / verify / extract / witness-verify over 2^18 instances, split
    over the GPUs (2^18 on one GPU at N = 1); a random subsample of every object and verdict is compared with the
    C oracle."""
    class A: secpar, log2n = 128, max(0, a.adaptor_log2n - (world.bit_length() - 1))
    eng, sch, p = _engine(128, local, np)
    dev = f'cuda:{local}'
    n = 1 << A.log2n
    seeds, seed_off, ch, ch_off = build_inputs(A, rank, torch, np)
    d_seeds = (torch.from_numpy(seeds).to(dev), torch.from_numpy(seed_off).to(dev))
    d_ch = (torch.from_numpy(ch).to(dev).view(-1), torch.from_numpy(ch_off).to(dev))
    _, sk_ntt, vk_ntt, _ = eng.lm_keygen(sch, d_seeds, want_sk_coef=False, want_vk_coef=False, device=True)
    pvf_bd, vf_bd, ext_bd = p['vf_bd'], p['vf_bd'] + 1, 2 * p['vf_bd'] + 1
    st = {}
    t = {}
    t['witgen'] = _timed(torch, dist, world, dev, lambda: st.update(zip(('wit', 'st_ntt', 'st_coef'), eng.witgen(sch, d_seeds, device=True))))
    t['presign'] = _timed(torch, dist, world, dev, lambda: st.__setitem__('presig', eng.lm_sign(sch, sk_ntt, d_ch, device=True)))
    t['preverify'] = _timed(torch, dist, world, dev, lambda: st.__setitem__('pv', eng.lm_verify(sch, vk_ntt, d_ch, st['presig'], pvf_bd, 256, device=True)))
    t['adapt'] = _timed(torch, dist, world, dev, lambda: st.__setitem__('sig', eng.vec_add(st['presig'], st['wit'], device=True)))
    t['verify'] = _timed(torch, dist, world, dev, lambda: st.__setitem__('vv', eng.lm_verify(sch, vk_ntt, d_ch, st['sig'], vf_bd, 256, st_ntt=st['st_ntt'], device=True)))
    t['extract'] = _timed(torch, dist, world, dev, lambda: st.__setitem__('ext', eng.vec_sub(st['sig'], st['presig'], device=True)))
    t['witness_verify'] = _timed(torch, dist, world, dev, lambda: st.__setitem__('wv', eng.witness_verify(st['ext'], st['st_ntt'], ext_bd, 256, device=True)))
    ok = bool(st['pv'].all().item() and st['vv'].all().item() and st['wv'].all().item())
    # ---- checker: 12 random instances end to end against the C oracle (adaptor_sigs.py:80-101,191-266)
    orc = _c_oracle()
    op = orc.params(128, p['q'], p['l'], p['sk_bd'], p['ch_wt'])
    key_ch, _ = eng.hash2polyvec('KEY_CH_SEED', [KEY_CH_SEED], p['q'] // 2, D, p['l'])
    key_ch = np.ascontiguousarray(key_ch[0])
    pick = np.sort(np.random.default_rng(7 + rank).choice(n, 12, replace=False))
    d_pick = torch.from_numpy(pick).to(dev)
    got = {k: st[k][d_pick].cpu().numpy() for k in ('wit', 'st_coef', 'presig', 'sig', 'ext')}
    q = p['q']
    centre = lambda x: ((x.astype(np.int64) + q // 2) % q - q // 2).astype(np.int16)
    matches = 0
    for j, i in enumerate(pick):
        seed = bytes(seeds[i * 128:(i + 1) * 128].tolist())
        skl, skr, vkl, vkr = orc.lm_keygen(op, key_ch, seed)
        wit, _ = orc.hash2polyvec(128, D, 'WIT_SALT', seed, 1, 20, p['l'])
        stc = orc.dot(q, key_ch, wit)
        m = _chmsg_str(ch[i])
        presig = orc.lm_sign(op, skl, skr, m)
        sig = centre(presig.astype(np.int64) + wit)
        good = (np.array_equal(wit, got['wit'][j]) and np.array_equal(stc, got['st_coef'][j]) and
                np.array_equal(presig, got['presig'][j]) and np.array_equal(sig, got['sig'][j]) and
                np.array_equal(centre(sig.astype(np.int64) - presig), got['ext'][j]) and
                orc.lm_verify(op, key_ch, vkl, vkr, m, presig, pvf_bd, 256) and
                orc.lm_verify(op, key_ch, vkl, vkr, m, sig, vf_bd, 256, st=stc) and
                not orc.lm_verify(op, key_ch, vkl, vkr, m, presig, vf_bd, 256, st=stc))
        matches += int(good)
    eng.close()
    return {'n_per_gpu': n, 'n_total': world * n, 'all_verdicts_true': ok,
            'oracle_subsample': {'checked': len(pick), 'bit_exact': matches, 'checker': 'oracle/lcb_oracle.c'},
            'ops_per_s': {k: world * n / (v * 1e-3) for k, v in t.items()}, 'ms': t}


def engine_arm(a):
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    p = SHIPPED[a.secpar]

    cpu = None
    if rank == 0 and a.gpus == 1 and not a.no_cpu_baseline:
        cpu = cpu_leg(a.secpar, a.cpu_per_core, None if a.no_secondary else a)   # before CUDA is initialised (forks workers)

    import numpy as np
    import torch
    import torch.distributed as dist
    from lattice_cryptography_b200 import Engine, make_scheme

    torch.cuda.set_device(local)
    numa_cpus = bind_to_gpu_numa_node(local) if world > 1 else None
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device(f'cuda:{local}'))
    eng = Engine(a.secpar, p['q'], D, p['l'], device=local)
    eng.use_torch_stream()
    sch = make_scheme(sk_bd=p['sk_bd'], sk_wt=256, ch_bd=1, ch_wt=p['ch_wt'])
    key_ch, _ = eng.hash2polyvec('KEY_CH_SEED', [KEY_CH_SEED], p['q'] // 2, D, p['l'])
    eng.set_key_ch(np.ascontiguousarray(key_ch[0]))

    n = 1 << a.log2n
    seeds, seed_off, ch, ch_off = build_inputs(a, rank, torch, np)
    dev = f'cuda:{local}'
    d_ch = torch.from_numpy(ch).to(dev)
    d_ch_off = torch.from_numpy(ch_off).to(dev)
    # keys and signatures come from the engine itself (tests/ pin them to the oracle)
    t0 = time.perf_counter()
    _, sk_ntt, vk_ntt, _ = eng.lm_keygen(sch, (torch.from_numpy(seeds).to(dev), torch.from_numpy(seed_off).to(dev)),
                                         want_sk_coef=False, want_vk_coef=False, device=True)
    torch.cuda.synchronize()
    t_keygen = time.perf_counter() - t0
    t0 = time.perf_counter()
    sig = eng.lm_sign(sch, sk_ntt, (d_ch.view(-1), d_ch_off), device=True)
    torch.cuda.synchronize()
    t_sign = time.perf_counter() - t0
    del sk_ntt
    torch.cuda.empty_cache()
    # every 64th triple is tampered: coefficient +1 / coefficient out of bound / message byte flipped
    bad = torch.arange(0, n, 64, device=dev)
    kind = (bad // 64) % 3
    sig_v = sig.view(torch.int16)
    i0, i1 = bad[kind == 0], bad[kind == 1]
    sig_v[i0, i0 % p['l'], (3 * i0) % D] += 1
    sig_v[i1, (i1 + 1) % p['l'], (7 * i1) % D] = p['vf_bd'] + 1
    i2 = bad[kind == 2]
    d_ch[i2, -1] ^= 1           # '0' <-> '1'
    expect = torch.ones(n, dtype=torch.uint8, device=dev)
    expect[bad] = 0
    verdict = torch.empty(n, dtype=torch.uint8, device=dev)
    chm = (d_ch.view(-1), d_ch_off)

    def step():
        eng.lm_verify(sch, vk_ntt, chm, sig, p['vf_bd'], p['vf_wt'], out=verdict)

    step()
    torch.cuda.synchronize()
    if not torch.equal(verdict, expect):
        raise SystemExit(f'rank {rank}: verdicts differ from the construction rule '
                         f'({int((verdict != expect).sum())} of {n})')

    for _ in range(a.warmup):
        step()
    eng.profile(True)
    eng.profile_reset()
    launches0 = eng.launch_count
    clocks = ClockSampler(local) if rank == 0 else None
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ev0.record()
    for _ in range(a.steps):
        step()
    ev1.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    ms = torch.tensor([ev0.elapsed_time(ev1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    clk = clocks.stop() if clocks else None
    launches = eng.launch_count - launches0
    v_ms, v_n = eng.profile_read('verify')
    s_ms, s_n = eng.profile_read('sampler')
    eng.profile(False)
    total_ms = float(ms.item())
    value = world * n * a.steps / (total_ms * 1e-3)
    if a.dump_outputs:          # before the packed leg below reuses `verdict`
        dump_outputs(a.dump_outputs, {'verdict' if world == 1 else f'verdict_rank{rank}': verdict.cpu().numpy()}, world, np)

    # ---- end to end: the same call with pinned HOST buffers (H2D of every input + D2H of the verdicts inside)
    h_sig = torch.empty(sig.shape, dtype=torch.int16, pin_memory=True)
    h_sig.copy_(sig_v)
    h_vk = torch.empty(vk_ntt.shape, dtype=torch.uint16, pin_memory=True)
    h_vk.copy_(vk_ntt)
    h_ch = torch.empty(d_ch.shape, dtype=torch.uint8, pin_memory=True)
    h_ch.copy_(d_ch)
    h_off = torch.empty(d_ch_off.shape, dtype=torch.int64, pin_memory=True)
    h_off.copy_(d_ch_off)
    h_verdict = torch.empty(n, dtype=torch.uint8, pin_memory=True)
    torch.cuda.synchronize()
    np_sig, np_vk, np_ch, np_off, np_verdict = (h_sig.numpy(), h_vk.view(torch.int16).numpy().view(np.uint16),
                                                h_ch.numpy().reshape(-1), h_off.numpy(), h_verdict.numpy())

    def e2e_step():
        eng.lm_verify(sch, np_vk, (np_ch, np_off), np_sig, p['vf_bd'], p['vf_wt'], out=np_verdict)

    e2e_step()
    if not np.array_equal(np_verdict, expect.cpu().numpy()):
        raise SystemExit(f'rank {rank}: end-to-end verdicts differ from the construction rule')
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(a.e2e_steps):
        e2e_step()
    e2e_s = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    e2e_value = world * n * a.e2e_steps / float(e2e_s.item())
    h2d = np_sig.nbytes + np_vk.nbytes + np_ch.nbytes + np_off.nbytes
    d2h = np_verdict.nbytes

    # ---- the same end-to-end call on the packed wire format (opt-in, SURVEY 8(f)2): 11/13-bit signature
    # coefficients and 14/16-bit key slots cross PCIe instead of 16-bit ones
    import math
    sbits, kbits = math.ceil(math.log2(2 * p['vf_bd'] + 1)), math.ceil(math.log2(p['q']))
    d_sig_p = eng.pack(sig_v, sbits, p['vf_bd'], device=True)
    d_vk_p = eng.pack(vk_ntt, kbits, 0, device=True)
    eng.lm_verify_packed(sch, d_vk_p, kbits, chm, d_sig_p, sbits, p['vf_bd'], p['vf_bd'], p['vf_wt'], out=verdict)
    torch.cuda.synchronize()
    if not torch.equal(verdict, expect):
        raise SystemExit(f'rank {rank}: packed verdicts differ from the construction rule')
    pk0, pk1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    pk0.record()
    eng.lm_verify_packed(sch, d_vk_p, kbits, chm, d_sig_p, sbits, p['vf_bd'], p['vf_bd'], p['vf_wt'], out=verdict)
    pk1.record()
    torch.cuda.synchronize()
    packed_resident_ms = pk0.elapsed_time(pk1)
    h_sig_p = torch.empty(d_sig_p.shape, dtype=torch.uint8, pin_memory=True)
    h_sig_p.copy_(d_sig_p)
    h_vk_p = torch.empty(d_vk_p.shape, dtype=torch.uint8, pin_memory=True)
    h_vk_p.copy_(d_vk_p)
    torch.cuda.synchronize()
    del d_sig_p, d_vk_p
    np_sig_p, np_vk_p = h_sig_p.numpy(), h_vk_p.numpy()

    def e2e_packed_step():
        eng.lm_verify_packed(sch, np_vk_p, kbits, (np_ch, np_off), np_sig_p, sbits, p['vf_bd'], p['vf_bd'], p['vf_wt'],
                             out=np_verdict)

    np_verdict[:] = 2
    e2e_packed_step()
    if not np.array_equal(np_verdict, expect.cpu().numpy()):
        raise SystemExit(f'rank {rank}: packed end-to-end verdicts differ from the construction rule')
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(a.e2e_steps):
        e2e_packed_step()
    e2e_p_s = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(e2e_p_s, op=dist.ReduceOp.MAX)
    e2e_packed = {'value': world * n * a.e2e_steps / float(e2e_p_s.item()), 'unit': UNIT,
                  'h2d_bytes_per_step': np_sig_p.nbytes + np_vk_p.nbytes + np_ch.nbytes + np_off.nbytes,
                  'd2h_bytes_per_step': d2h, 'steps': a.e2e_steps, 'sig_bits': sbits, 'key_bits': kbits,
                  'resident_ms_per_step': packed_resident_ms,
                  'h2d_gbs_per_rank': (np_sig_p.nbytes + np_vk_p.nbytes + np_ch.nbytes + np_off.nbytes) * a.e2e_steps /
                                      float(e2e_p_s.item()) / 1e9,
                  'note': 'lcb_lm_verify_packed_batch on pinned host buffers: the documented route for host-resident '
                          'callers (INTEGRATION.md); the contract e2e above keeps the unpacked int16 format'}
    del h_sig_p, h_vk_p, np_sig_p, np_vk_p

    if rank == 0:
        peaks = _peaks()
        k_ms = v_ms / max(v_n, 1)
        # ---- primary roofline: integer instruction issue (SURVEY.md 8d; DESIGN.md 3.5).  Algorithmic work of ONE verify
        # inside k_verify at secpar 128 / 256 by the survey's work model: (l + 1) negacyclic NTT-256 of 8,192
        # int32 instructions (1,024 butterflies x 8), (l + 1) x 256 multiply-accumulates of 6, bounds 2 per coefficient,
        # comparison 2 per slot.  (The Keccak share of a verify, 6 / 26 permutations, is the sampler kernel's.)
        ntts = p['l'] + 1
        unit_instr = ntts * 8192 + ntts * D * 6 + p['l'] * D * 2 + D * 2
        step_instr = unit_instr + {128: 6, 256: 26}[a.secpar] * 4560 + p['ch_wt'] * 40
        achieved_t = unit_instr * n / (k_ms * 1e-3) / 1e12
        # algorithmic bytes of one verify inside k_verify: signature + vk + challenge pairs + verdict
        unit_bytes = p['l'] * D * 2 + 2 * D * 2 + p['ch_wt'] * 4 + 1
        hbm_achieved = unit_bytes * n / (k_ms * 1e-3) / 1e9
        ncu = _ncu_summary('verify') if a.secpar == 128 else None
        line = {
            'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': a.steps, 'warmup': a.warmup,
            'ms_per_step': total_ms / a.steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
            'dtype': 'u32 (mod-q integer arithmetic, q < 2^16)', 'data': 'synthetic',
            'config': engine_config(a),
            'roofline': {'bound': 'int_issue', 'kernel': 'k_verify', 'achieved': achieved_t, 'peak': peaks['int_tinstr_s'],
                         'unit': 'Tinstr/s', 'frac': achieved_t / peaks['int_tinstr_s'],
                         # DRAM bytes per launch of this kernel from its ncu --set full capture, scaled from the
                         # capture's batch to this launch's (None when no capture of this build's kernel is committed)
                         'traffic': ncu['dram_bytes_per_unit'] * n if ncu else None,
                         'algorithmic_instr_per_unit': unit_instr,
                         'work_model': f'{ntts} NTT-256 x 8192 + {ntts} x 256 x 6 (multiply-accumulate) + '
                                       f'{p["l"]} x 256 x 2 (bounds) + 512 (compare) int32 instructions per verify '
                                       f'(SURVEY.md 8d); peak = 148 SMs x 128 lanes x {peaks["sm_max_mhz"]:.0f} MHz',
                         'peak_source': peaks['source'] + ' sm_max_mhz',
                         'note': 'frac = algorithmic work by the SURVEY 8(d) model / peak issue rate; it can exceed 1 because '
                                 'the kernel needs fewer instructions than the model counts (4.5 instead of 8 per butterfly, '
                                 'FP32-assisted multiplication and two-stage quadruples): the share of issue slots actually '
                                 'used is executed.issue_slot_frac, the ncu counters are under ncu',
                         'kernel_ms_per_launch': k_ms, 'kernel_share_of_step': v_ms / total_ms,
                         'sampler_ms_per_launch': s_ms / max(s_n, 1),
                         'whole_step': {'algorithmic_instr_per_unit': step_instr,
                                        'frac': step_instr * (value / world) / 1e12 / peaks['int_tinstr_s']},
                         'hbm': {'bound': 'hbm', 'achieved': hbm_achieved, 'peak': peaks['hbm_gbs'], 'unit': 'GB/s',
                                 'frac': hbm_achieved / peaks['hbm_gbs'], 'algorithmic_bytes_per_unit': unit_bytes,
                                 'algorithmic_bytes_per_launch': unit_bytes * n, 'peak_source': peaks['source'] + ' hbm_gbs',
                                 'note': 'secondary figure: the kernel needs 7.8 KB per ~140 k instructions, HBM does not bind'},
                         'ncu': ncu,
                         # what the kernel really issues (committed ncu digest of this kernel x this launch's live time):
                         # the model above counts 8 instructions per butterfly, the kernel needs 4.5, so `frac` (work
                         # done per peak issue rate) sits above the share of issue slots actually used
                         'executed': ({'thread_instr_per_unit': ncu['warp_instr_per_unit'] * 32,
                                       'issue_slot_frac': ncu['warp_instr_per_unit'] * n / (k_ms * 1e-3) /
                                                          (148 * 4 * peaks['sm_max_mhz'] * 1e6)} if ncu else None)},
            'e2e': {'value': e2e_value, 'unit': UNIT, 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h,
                    'steps': a.e2e_steps, 'host_cpus_bound_per_rank': numa_cpus,
                    'h2d_gbs_per_rank': h2d * a.e2e_steps / float(e2e_s.item()) / 1e9,
                    'note': 'host-resident int16 signatures: bound by the host link (PCIe / host memory), see '
                            'h2d_gbs_per_rank; e2e_packed moves 28 % fewer bytes for the same verdicts'},
            'e2e_packed': e2e_packed,
            'gpu_launches': launches,
            'clocks': clk,
            'setup': {'keygen_s': t_keygen, 'sign_s': t_sign, 'keygen_keys_per_s': n / t_keygen,
                      'sign_sigs_per_s': n / t_sign,
                      'note': 'cold first calls of this process (memory-pool growth and output allocation inside); '
                              'warm rates are in secondary and profiles/README.md'},
        }
        if cpu is not None:
            line['cpu_baseline'] = cpu
    del sig, sig_v, vk_ntt, d_ch, h_sig, h_vk, h_ch, np_sig, np_vk, np_ch
    torch.cuda.empty_cache()
    secondary = {}
    if not a.no_secondary:
        for name, fn in (('keygen_sign_secpar256', secondary_keygen_sign),
                         ('lm_verify_secpar256', secondary_verify_secpar256), ('bklm', secondary_bklm),
                         ('adaptor', secondary_adaptor), ('single_ops', secondary_single_ops)):
            try:
                secondary[name] = fn(a, rank, local, world, torch, np, dist)
            except Exception as exc:          # the headline line must survive a secondary failure
                secondary[name] = {'error': repr(exc)[:300]}
    if rank == 0:
        line['secondary'] = secondary
        bk = secondary.get('bklm') or {}
        if 'aggregate_verify_sigs_per_s' in bk:       # the second half of BASELINE.json's metric, on the same line
            line['also'] = {'metric': 'BKLM aggregate-verify sigs/sec', 'value': bk['aggregate_verify_sigs_per_s'],
                            'unit': 'signatures/s', 'n_gpus': world,
                            'config': {'workload': f"bklm aggregate-verify, N = {bk['sigs_per_aggregate']} signatures per "
                                                   f"aggregate sharded over {world} GPU(s), secpar 128, exact reference "
                                                   f"semantics incl. the O(N^2) aggregation-coefficient hashing"},
                            'aggregate_sigs_per_s': bk.get('aggregate_sigs_per_s'),
                            'agg_coefs_gperm_s_per_gpu': bk.get('agg_coefs_gperm_s_per_gpu'),
                            'roofline': {'bound': 'alu_pipe (Keccak LOP3/SHF)', 'kernel': 'k_agg_coefs / k_agg_coefs_il',
                                         'achieved': bk.get('agg_coefs_gperm_s_per_gpu'), 'peak': 4.28, 'unit': 'Gperm/s',
                                         'frac': (bk.get('agg_coefs_gperm_s_per_gpu') or 0) / 4.28,
                                         'peak_source': 'tools/keccak_bench2.cu (measured, 100 % ALU pipe)'},
                            'row_ii_coefficients_supplied': bk.get('row_ii_coefficients_supplied')}
            if cpu is not None and 'bklm' in cpu:
                cb = cpu['bklm']
                line['also']['cpu_baseline'] = {
                    'value': cb['aggregate_verify']['sigs_per_s'], 'unit': 'signatures/s', 'cores': cb['cores'], 'kind': 'port',
                    'aggregate_sigs_per_s': cb['aggregate']['sigs_per_s'],
                    'sample': f"aggregate + aggregate-verify timed at N in {[q_['n'] for q_ in cb['points']]} on {cb['cores']} cores, "
                              f"t(N) = a N^2 + b N extrapolated to N = {cb['target_n']} (BASELINE.md section 3): b fitted, "
                              f"a = 124 B / (hashlib SHAKE256 rate measured on a {124 * cb['target_n']}-byte message on all cores)"}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    eng.close()


if __name__ == '__main__':
    args = parse()
    if args.impl == 'reference':
        reference_arm(args)
    else:
        engine_arm(args)
