"""The content-mode BKLM route on the device (include/lcb200.h: lcb_content_order_batch, lcb_gather_rows_batch,
lcb_gather_ragged_batch; Engine.content_order / gather_rows / gather_ragged; wire.sorted_aggregation_inputs /
aggregate_batch_content / aggregate_verify_batch_content): the per-group order against Python's stable sorted() and
numpy's lexsort on every path (LCB_ORDER_SMALL_MAX / LCB_ORDER_BLOCK_MAX force each one), the gathers against numpy
indexing and concatenation, and the whole route against the host route and the drop-in objects, bit for bit."""
import os
import subprocess
import sys
from ctypes import c_void_p

import numpy as np
import pytest

from test_gpu_content_inputs import _bitmsgs, _dev, _misaligned, _seed_objs, content_mode   # noqa: F401  (fixture re-export)
from test_gpu_parity import engines   # noqa: F401  (fixture re-export)

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# per item (default), per block (groups above 32 items), radix (every non-empty group)
PATHS = {'default': {}, 'block': {'LCB_ORDER_SMALL_MAX': '0'},
         'radix': {'LCB_ORDER_SMALL_MAX': '0', 'LCB_ORDER_BLOCK_MAX': '0'}}
BLOCK_MAX = 1024
EDGE_SIZES = [0, 1, 2, 0, 31, 32, 33, BLOCK_MAX - 1, BLOCK_MAX, BLOCK_MAX + 1, 3, 0]


def _off(sizes):
    return np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)


def _ref_order(rows, off):
    out = []
    for g in range(len(off) - 1):
        a, b = int(off[g]), int(off[g + 1])
        out.extend(sorted(range(a, b), key=lambda i: bytes(rows[i])))
    return np.array(out, dtype=np.int64)


def _lex_order(rows, off):
    gid = np.repeat(np.arange(len(off) - 1), np.diff(off))
    return np.lexsort((rows.view('S57').reshape(-1), gid)).astype(np.int64)


def _row_sets(total, seed):
    rng = np.random.default_rng(seed)
    rnd = rng.integers(0, 256, (total, 57), dtype=np.uint8)
    first = np.full((total, 57), 0x61, np.uint8)
    first[:, 0] = rng.choice(np.array([0x00, 0x01, 0x7F, 0x80, 0xFE, 0xFF], np.uint8), total)
    last = np.full((total, 57), 0x61, np.uint8)
    last[:, 56] = rng.choice(np.array([0x00, 0x01, 0x7F, 0x80, 0xFE, 0xFF], np.uint8), total)
    extremes = rng.choice(np.array([0x00, 0xFF], np.uint8), (total, 57))
    equal = np.full((total, 57), 0xA7, np.uint8)
    pool = rng.integers(0, 256, (5, 57), dtype=np.uint8)
    dups = pool[rng.integers(0, 5, total)]
    return {'random': rnd, 'first_byte': first, 'last_byte': last, 'bytes_00_ff': extremes, 'all_equal': equal,
            'duplicates': dups}


def _orders(e, off, rows):
    """Host and device buffers: both orders, as numpy."""
    host = e.content_order(off, rows)
    dev = e.content_order(_dev(off), _dev(rows), device=True)
    e.synchronize()
    return host, dev.cpu().numpy()


# ------------------------------------------------------------------------------------------- 1. order
@pytest.mark.parametrize('path', sorted(PATHS))
def test_order_edge_layouts_every_path(engines, monkeypatch, path):
    e = engines[128]
    for k, v in PATHS[path].items():
        monkeypatch.setenv(k, v)
    off = _off(EDGE_SIZES)
    total = int(off[-1])
    for name, rows in _row_sets(total, 7).items():
        want = _ref_order(rows, off)
        assert np.array_equal(_lex_order(rows, off), want), name
        for got in _orders(e, off, rows):
            assert got.dtype == np.int64 and np.array_equal(got, want), (path, name)
    assert np.array_equal(_orders(e, off, _row_sets(total, 7)['all_equal'])[0], np.arange(total))   # stability


@pytest.mark.parametrize('path', sorted(PATHS))
def test_order_one_group_of_2_16(engines, monkeypatch, path):
    e = engines[128]
    for k, v in PATHS[path].items():
        monkeypatch.setenv(k, v)
    off = _off([1 << 16])
    sets = _row_sets(1 << 16, 9)
    for name in ('random', 'duplicates', 'last_byte'):
        want = _ref_order(sets[name], off)
        for got in _orders(e, off, sets[name]):
            assert np.array_equal(got, want), (path, name)


def test_order_many_groups_of_two(engines):
    """2^18 groups of two with empty groups interleaved: the shipped ag_cap = 2 layout at size."""
    e = engines[128]
    sizes = np.full(5 << 16, 2, np.int64)
    sizes[4::5] = 0                                                # 2^18 groups of two, every fifth group empty
    off = _off(sizes)
    rng = np.random.default_rng(2)
    rows = rng.integers(0, 256, (int(off[-1]), 57), dtype=np.uint8)
    rows[1::7] = rows[0::7][:rows[1::7].shape[0]]                  # some equal pairs
    want = _lex_order(rows, off)
    for got in _orders(e, off, rows):
        assert np.array_equal(got, want)


@pytest.mark.parametrize('secpar', [128, 256])
def test_order_of_content_strings(content_mode, secpar):
    from lattice_cryptography_b200 import bklm_one_time_agg_sigs as bk
    from lattice_cryptography_b200 import wire
    pp = bk.make_setup_parameters(secpar)
    sizes = [0, 1, 2, 31, 32, 33, 40, 0, 2]
    total = sum(sizes)
    seeds = _seed_objs(pp, total, secpar)
    seeds[5] = seeds[4]                                            # one key twice in the group of 31
    _, vkp = wire.keygen_batch_packed(pp, seeds)
    rows = wire.content_strs(pp, vkp)
    off = _off(sizes)
    e = wire._engine(pp)
    want = _ref_order(rows, off)
    assert np.array_equal(_lex_order(rows, off), want)
    for got in _orders(e, off, rows):
        assert np.array_equal(got, want)


def test_order_empty_and_errors(engines):
    from lattice_cryptography_b200 import LcbError, _ffi
    e = engines[128]
    assert e.content_order(np.zeros(1, np.int64), np.zeros((0, 57), np.uint8)).shape == (0,)
    assert e.content_order(_off([0, 0]), np.zeros((0, 57), np.uint8)).shape == (0,)
    assert e._lib.lcb_content_order_batch(e._ctx, c_void_p(np.zeros(1, np.int64).ctypes.data), 0, None, None) == _ffi.LCB_OK
    rows = np.zeros((4, 57), np.uint8)
    for bad in (np.array([0, 3, 2, 4], np.int64), np.array([1, 2, 4], np.int64)):
        with pytest.raises(LcbError) as x:
            e._ck(e._lib.lcb_content_order_batch(e._ctx, c_void_p(bad.ctypes.data), len(bad) - 1, c_void_p(rows.ctypes.data),
                                                 c_void_p(np.zeros(4, np.int64).ctypes.data)))
        assert x.value.status == _ffi.LCB_ERR_INVALID


# ------------------------------------------------------------------------------------------- 2. gathers
@pytest.mark.parametrize('row', [1, 57, 333, 896, 1024, 4576, 9568])
def test_gather_rows(engines, row):
    e = engines[128]
    rng = np.random.default_rng(row)
    src = rng.integers(0, 256, (50, row), dtype=np.uint8)
    index = rng.integers(0, 50, 300).astype(np.int64)             # repeated indices
    want = src[index]
    assert np.array_equal(e.gather_rows(src, index), want)
    got = e.gather_rows(_dev(src), _dev(index), device=True)
    e.synchronize()
    assert np.array_equal(got.cpu().numpy(), want)
    got = e.gather_rows(_misaligned(src), _dev(index), device=True)   # 4-byte but not 16-byte aligned source
    e.synchronize()
    assert np.array_equal(got.cpu().numpy(), want)
    # a misaligned destination, through the ABI
    import torch
    raw = torch.zeros(300 * row + 16, dtype=torch.uint8, device='cuda')
    dst = raw[4:4 + 300 * row]
    e._ck(e._lib.lcb_gather_rows_batch(e._ctx, c_void_p(src.ctypes.data), 50, row, c_void_p(index.ctypes.data), 300,
                                       c_void_p(dst.data_ptr())))
    e.synchronize()
    assert np.array_equal(dst.cpu().numpy().reshape(300, row), want)
    # trailing shape kept
    sig = rng.integers(0, 256, (20, 13, 352), dtype=np.uint8)
    assert np.array_equal(e.gather_rows(sig, index[:40] % 20), sig[index[:40] % 20])


def test_gather_rows_out_of_range(engines):
    from lattice_cryptography_b200 import LcbError, _ffi
    e = engines[128]
    src = np.arange(1, 1 + 10 * 57, dtype=np.int64).astype(np.uint8).reshape(10, 57)
    index = np.array([0, -1, 10, 9, 1 << 40, -(1 << 40), 3], np.int64)
    got = e.gather_rows(_dev(src), _dev(index), device=True)
    e.synchronize()
    want = np.zeros((7, 57), np.uint8)
    for k, s in enumerate(index):
        if 0 <= s < 10:
            want[k] = src[s]
    assert np.array_equal(got.cpu().numpy(), want)
    with pytest.raises(LcbError) as x:
        e.gather_rows(src, index)
    assert x.value.status == _ffi.LCB_ERR_INVALID
    assert e.gather_rows(src, np.zeros(0, np.int64)).shape == (0, 57)


def _items(rng):
    lens = [0, 1, 15, 16, 17, 0, 31, 32, 33, 47, 48, 49, 0, 127, 128, 129, 300]
    return [bytes(rng.integers(0, 256, n, dtype=np.uint8)) for n in lens]


def test_gather_ragged(engines):
    from lattice_cryptography_b200 import ragged
    e = engines[128]
    rng = np.random.default_rng(4)
    items = _items(rng)
    index = rng.integers(0, len(items), 3000).astype(np.int64)
    want_b = [items[i] for i in index]
    wb, wo = ragged(want_b)
    blob, off = e.gather_ragged(items, index)
    assert np.array_equal(off, wo) and bytes(blob) == bytes(wb)
    dblob, doff = e.gather_ragged((_dev(ragged(items)[0]), _dev(ragged(items)[1])), _dev(index), device=True)
    e.synchronize()
    assert np.array_equal(doff.cpu().numpy(), wo) and bytes(dblob.cpu().numpy()) == bytes(wb)
    # every item empty
    blob, off = e.gather_ragged([b'', b''], np.array([1, 0, 1], np.int64))
    assert off.tolist() == [0, 0, 0, 0] and blob.shape == (0,)


def test_gather_ragged_abi_offsets_cap_and_range(engines):
    """off[0] != 0 on host and device buffers, out_cap one byte short, host and device out-of-range indices."""
    from lattice_cryptography_b200 import _ffi
    e = engines[128]
    rng = np.random.default_rng(5)
    items = _items(rng)
    lens = np.array([len(i) for i in items], np.int64)
    off = (777 + np.concatenate([[0], np.cumsum(lens)])).astype(np.int64)
    blob = np.concatenate([rng.integers(0, 256, 777, dtype=np.uint8), np.frombuffer(b''.join(items), np.uint8),
                           rng.integers(0, 256, 9, dtype=np.uint8)])
    n_src = len(items)
    index = rng.integers(0, n_src, 500).astype(np.int64)
    want = b''.join(items[i] for i in index)
    wo = np.concatenate([[0], np.cumsum(lens[index])]).astype(np.int64)
    p = lambda x: c_void_p(x.ctypes.data)   # noqa: E731
    d = lambda x: c_void_p(x.data_ptr())    # noqa: E731
    for dev in (False, True):
        b, o, i = (_dev(blob), _dev(off), _dev(index)) if dev else (blob, off, index)
        ptr = d if dev else p
        out = np.zeros(len(want), np.uint8)
        out_off = np.zeros(501, np.int64)
        assert e._lib.lcb_gather_ragged_batch(e._ctx, ptr(b), ptr(o), n_src, ptr(i), 500, p(out), len(want),
                                              p(out_off)) == _ffi.LCB_OK
        assert bytes(out) == want and np.array_equal(out_off, wo)
        assert e._lib.lcb_gather_ragged_batch(e._ctx, ptr(b), ptr(o), n_src, ptr(i), 500, p(out), len(want) - 1,
                                              p(out_off)) == _ffi.LCB_ERR_INVALID
        assert b'out_cap' in e._lib.lcb_last_error(e._ctx)
    bad = index.copy()
    bad[7] = n_src
    out = np.zeros(len(want) + 1000, np.uint8)
    assert e._lib.lcb_gather_ragged_batch(e._ctx, p(blob), p(off), n_src, p(bad), 500, p(out), out.shape[0],
                                          p(np.zeros(501, np.int64))) == _ffi.LCB_ERR_INVALID
    # device indices outside [0, n_src): empty items
    bad[3], bad[9] = -1, 1 << 40
    ok = (bad >= 0) & (bad < n_src)
    dblob, doff = e.gather_ragged((_dev(blob[777:]), _dev(off - 777)), _dev(bad), device=True)
    e.synchronize()
    assert bytes(dblob.cpu().numpy()) == b''.join(items[s] if k else b'' for s, k in zip(bad, ok))
    assert int(doff[-1].item()) == int(lens[bad[ok]].sum())
    assert e._lib.lcb_gather_ragged_batch(e._ctx, p(blob), p(off), n_src, None, 0, None, 0, p(out_off)) == _ffi.LCB_OK


# ------------------------------------------------------------------------------------------- 3. end to end
def _batch(pp, sizes, seed, tamper_msg=None):
    from lattice_cryptography_b200 import wire
    total = sum(sizes)
    seeds = _seed_objs(pp, total, seed)
    seeds[2] = seeds[1]                                            # one key twice in a group (sizes[1] >= 2)
    rng = np.random.default_rng(seed)
    msgs = _bitmsgs(rng, total, lens=(32, 0, 100, 150, 7))
    skp, vkp = wire.keygen_batch_packed(pp, seeds)
    sigp, ok = wire.sign_batch_packed_sk(pp, skp, wire.challenge_inputs(pp, vkp, msgs))
    assert ok.all()
    return seeds, vkp, msgs, sigp, _off(sizes)


@pytest.mark.parametrize('secpar', [128, 256])
def test_sorted_inputs_and_aggregates_equal_host_route(content_mode, secpar):
    from lattice_cryptography_b200 import bklm_one_time_agg_sigs as bk
    from lattice_cryptography_b200 import ragged, wire
    pp = bk.set_aggregation_capacity(bk.make_setup_parameters(secpar), 8)
    sizes = [1, 3, 2, 1, 5, 1, 2, 8, 2, 4]                         # aggregates need non-empty groups
    _, vkp, msgs, sigp, off = _batch(pp, sizes, 3 + secpar)
    order, chm, agmsgs = wire.aggregation_inputs(pp, off, vkp, msgs)
    want_ag = ragged(agmsgs)
    for dev in (False, True):
        args = (_dev(off), _dev(vkp), tuple(_dev(x) for x in ragged(msgs))) if dev else (off, vkp, msgs)
        o2, vks, chm2, ag2 = wire.sorted_aggregation_inputs(pp, *args, device=dev)
        wire._engine(pp).synchronize()
        h = (lambda x: x.cpu().numpy()) if dev else (lambda x: x)
        assert np.array_equal(h(o2), order) and np.array_equal(h(vks), vkp[order])
        assert np.array_equal(h(chm2[1]), chm[1]) and bytes(h(chm2[0])) == bytes(chm[0])
        assert np.array_equal(h(ag2[1]), want_ag[1]) and bytes(h(ag2[0])) == bytes(want_ag[0])
    agp, inr = wire.aggregate_batch_packed(pp, off, np.ascontiguousarray(sigp[order]), agmsgs)
    got, got_r = wire.aggregate_batch_content(pp, off, vkp, msgs, sigp)
    assert np.array_equal(got, agp) and np.array_equal(got_r, inr)
    dgot, dgot_r = wire.aggregate_batch_content(pp, _dev(off), _dev(vkp), ragged(msgs), _dev(sigp), device=True)
    wire._engine(pp).synchronize()
    assert dgot.is_cuda and np.array_equal(dgot.cpu().numpy(), agp) and np.array_equal(dgot_r.cpu().numpy(), inr)
    want_v = wire.aggregate_verify_batch_packed(pp, off, np.ascontiguousarray(vkp[order]), chm, agmsgs, agp)
    assert want_v.all()
    v = wire.aggregate_verify_batch_content(pp, off, vkp, msgs, agp)
    assert np.array_equal(v, want_v)
    dv = wire.aggregate_verify_batch_content(pp, _dev(off), _dev(vkp), ragged(msgs), _dev(agp), device=True)
    wire._engine(pp).synchronize()
    assert dv.is_cuda and np.array_equal(dv.cpu().numpy(), want_v)
    # tampers flip their own group only: one aggregate bit, one message of an item
    bad = agp.copy()
    bad[4, 0, 0] ^= 1
    assert wire.aggregate_verify_batch_content(pp, off, vkp, msgs, bad).tolist() == [int(g != 4)
                                                                                     for g in range(len(sizes))]
    tm = list(msgs)
    tm[int(off[7]) + 3] = tm[int(off[7]) + 3] + '1'
    t_order, t_chm, t_ag = wire.aggregation_inputs(pp, off, vkp, tm)
    want_t = wire.aggregate_verify_batch_packed(pp, off, np.ascontiguousarray(vkp[t_order]), t_chm, t_ag, agp)
    got_t = wire.aggregate_verify_batch_content(pp, off, vkp, tm, agp)
    assert np.array_equal(got_t, want_t) and got_t.tolist() == [int(g != 7) for g in range(len(sizes))]


def test_content_route_agrees_with_dropin_objects(content_mode):
    from lattice_cryptography_b200 import bklm_one_time_agg_sigs as bk
    from lattice_cryptography_b200 import lm_one_time_sigs as lm
    from lattice_cryptography_b200 import wire
    pp = bk.make_setup_parameters(128)
    sizes = [2, 2, 1, 2]
    seeds, vkp, msgs, sigp, off = _batch(pp, sizes, 21)
    agp, ok = wire.aggregate_batch_content(pp, off, vkp, msgs, sigp)
    assert ok.all()
    keys = lm.keygen(pp, sum(sizes), seeds=seeds, multiprocessing=False)
    sigs = [lm.sign(pp, k, m) for k, m in zip(keys, msgs)]
    for g in range(len(sizes)):
        a, b = int(off[g]), int(off[g + 1])
        ag = bk.aggregate(pp, [k[2] for k in keys[a:b]], msgs[a:b], sigs[a:b])
        assert np.array_equal(agp[g], wire.pack_signatures(pp, ag.coef[None], bound_key='avf_bd')[0][0])
        assert bk.aggregate_verify(pp, [k[2] for k in keys[a:b]], msgs[a:b], ag)
    assert wire.aggregate_verify_batch_content(pp, off, vkp, msgs, agp).all()


def test_content_route_refuses_tree_mode_and_bad_messages(content_mode):
    from lattice_cryptography_b200 import bklm_one_time_agg_sigs as bk
    from lattice_cryptography_b200 import wire
    pp = bk.make_setup_parameters(128)
    _, vkp, msgs, sigp, off = _batch(pp, [1, 2], 5)
    with pytest.raises(ValueError, match='Input messages must be bitstrings.'):
        wire.sorted_aggregation_inputs(pp, off, vkp, [msgs[0], 'hello', msgs[2]])
    bk.set_aggregation_mode(pp, 'tree')
    for call in (lambda: wire.sorted_aggregation_inputs(pp, off, vkp, msgs),
                 lambda: wire.aggregate_batch_content(pp, off, vkp, msgs, sigp),
                 lambda: wire.aggregate_verify_batch_content(pp, off, vkp, msgs, sigp[:2, :, :0])):
        with pytest.raises(ValueError, match='ag_mode'):
            call()


# ------------------------------------------------------------------------------------------- 4. checked build
def test_order_and_gathers_pass_on_the_checked_build():
    """The edge cases above, small, on liblcb200_checked.so (device-side asserts on every new global access)."""
    code = r'''
import os, numpy as np, torch
from lattice_cryptography_b200 import Engine, ragged
e = Engine(128, 11777, 256, 13)
assert e._lib.lcb_build_is_checked() == 1
rng = np.random.default_rng(1)
sizes = [0, 1, 2, 31, 32, 33, 40, 1200, 0, 2]
off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
rows = rng.integers(0, 256, (int(off[-1]), 57), dtype=np.uint8)
rows[100:300] = rows[100]
gid = np.repeat(np.arange(len(sizes)), sizes)
want = np.lexsort((rows.view('S57').reshape(-1), gid))
for env in ({}, {'LCB_ORDER_SMALL_MAX': '0'}, {'LCB_ORDER_SMALL_MAX': '0', 'LCB_ORDER_BLOCK_MAX': '0'}):
    for k in ('LCB_ORDER_SMALL_MAX', 'LCB_ORDER_BLOCK_MAX'):
        os.environ.pop(k, None)
    os.environ.update(env)
    assert np.array_equal(e.content_order(off, rows), want), env
    d = e.content_order(torch.from_numpy(off).cuda(), torch.from_numpy(rows).cuda(), device=True)
    e.synchronize()
    assert np.array_equal(d.cpu().numpy(), want), env
idx = np.array([3, -1, 1 << 40, 0, 5, 5], np.int64)
for row in (1, 57, 896, 4576):
    src = rng.integers(0, 256, (6, row), dtype=np.uint8)
    raw = torch.zeros(6 * row + 16, dtype=torch.uint8, device='cuda')
    mis = raw[4:4 + 6 * row]
    mis.copy_(torch.from_numpy(src.reshape(-1)).cuda())
    torch.cuda.synchronize()
    for s in (torch.from_numpy(src).cuda(), mis.view(6, row)):
        g = e.gather_rows(s, torch.from_numpy(idx).cuda(), device=True)
        e.synchronize()
        g = g.cpu().numpy()
        assert not g[1].any() and not g[2].any() and np.array_equal(g[[0, 3, 4, 5]], src[[3, 0, 5, 5]])
items = [b'x' * n for n in (0, 15, 16, 17, 33, 0)]
b, o = ragged(items)
gb, go = e.gather_ragged((torch.from_numpy(b).cuda(), torch.from_numpy(o).cuda()), torch.from_numpy(idx).cuda(), device=True)
e.synchronize()
assert go.cpu().numpy().tolist() == [0, 17, 17, 17, 17, 17, 17] and bytes(gb.cpu().numpy()) == b'x' * 17
hb, ho = e.gather_ragged(items, np.arange(6, dtype=np.int64)[::-1].copy())
assert bytes(hb) == b''.join(items[::-1])
print('ok')
'''
    env = dict(os.environ, LCB200_LIB=os.path.join(ROOT, 'lattice_cryptography_b200', 'liblcb200_checked.so'))
    r = subprocess.run([sys.executable, '-c', code], cwd=ROOT, env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and 'ok' in r.stdout, r.stdout + r.stderr
