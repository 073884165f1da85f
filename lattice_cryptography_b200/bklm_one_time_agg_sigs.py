"""Boneh-Kim style aggregation of LM one-time signatures: the reference's entry points
(lattice_cryptography/bklm_one_time_agg_sigs.py:27-116) on the CUDA engine, plus sharded variants.

Drop-in: make_setup_parameters, prepare_make_agg_coefs, prepare_hash2polyinput, make_agg_coefs,
         prepare_aggregate, aggregate, aggregate_verify
Sharded: aggregate_shard / aggregate_finish, aggregate_verify_shard / aggregate_verify_finish -
         each rank (GPU) handles a contiguous range of the SORTED list and the int32 partial sums
         are added across ranks (one NCCL reduce; see lattice_cryptography_b200.distributed).
Batched: aggregate_batch, aggregate_verify_batch - many independent aggregates (the reference caps one at
         ag_cap = 2 signatures) in one engine call; element g equals aggregate / aggregate_verify of group g.

Sorting by str(otvk) and building the hash-input strings stay on the host: they depend on CPython
object identity (SURVEY.md section 0.4).  The shipped parameters have ag_wt = ag_bd = 1, i.e. every
aggregation coefficient is a signed monomial (a signed rotation of the signature: the HBM-bound fast kernels);
other values of the module tables BDs / WTs (the reference leaves them editable, :15-19) take the general
NTT-domain product kernels.
"""
from typing import Dict, List, Tuple

import numpy as np

from .lattice_algebra import Polynomial, PolynomialVector, is_bitstring
from .lm_one_time_sigs import (BDs, Message, PublicParameters, SALTs, SecurityParameter, Signature, WTs, _ctx,
                               challenge_messages, make_setup_parameters as setup_pars, make_signature_challenge, well_formed)
from .one_time_keys import ALLOWABLE_SECPARS, OneTimeVerificationKey, bits_to_decode, bits_to_indices

AggCoef = Polynomial

for _s in ALLOWABLE_SECPARS:
    BDs[_s]['ag_bd'] = 1
    WTs[_s]['ag_wt'] = 1
    SALTs[_s]['ag_salt'] = 'AG_SALT'
CAPs: Dict[int, int] = {i: 2 for i in ALLOWABLE_SECPARS}


def make_setup_parameters(secpar: SecurityParameter) -> PublicParameters:
    pp = setup_pars(secpar=secpar)
    lp = pp['scheme_parameters'].lp
    pp['ag_cap'], pp['ag_salt'] = CAPs[secpar], SALTs[secpar]['ag_salt']
    pp['ag_bd'], pp['ag_wt'] = BDs[secpar]['ag_bd'], WTs[secpar]['ag_wt']
    pp['avf_wt'] = max(1, min(lp.degree, pp['ag_cap'] * pp['ag_wt'] * pp['vf_wt']))
    pp['avf_bd'] = max(1, min(lp.modulus // 2, pp['ag_cap'] * min(pp['ag_wt'], pp['vf_wt']) * pp['ag_bd'] * pp['vf_bd']))
    return pp


def set_aggregation_capacity(pp: PublicParameters, ag_cap: int) -> PublicParameters:
    """Raise/lower pp['ag_cap'] and recompute avf_bd / avf_wt by the reference's formulas
    (bklm_one_time_agg_sigs.py:36-43).  Not a reference function: the reference hard-codes cap = 2."""
    lp = pp['scheme_parameters'].lp
    pp['ag_cap'] = ag_cap
    pp['avf_wt'] = max(1, min(lp.degree, ag_cap * pp['ag_wt'] * pp['vf_wt']))
    pp['avf_bd'] = max(1, min(lp.modulus // 2, ag_cap * min(pp['ag_wt'], pp['vf_wt']) * pp['ag_bd'] * pp['vf_bd']))
    return pp


# ------------------------------------------------------------------------------- non-reference: linear-time mode
# The reference derives coefficient i from ag_salt || str(i) || M with M = str(list(zip(keys, msgs))) - every one of
# the N coefficients absorbs the whole O(N)-byte message (bklm_one_time_agg_sigs.py:60-81): 3.9e9 Keccak permutations
# at N = 2^16, which is all of the aggregate's cost.  SURVEY.md 8(f)4 asks for a sub-quadratic VARIANT "offered as an
# explicitly non-reference mode": with pp['ag_mode'] = 'tree' the message is first bound into a 32-byte commitment
#     leaf_j = SHAKE256(M[j*8192 : (j+1)*8192])[:32]                   (every 8,192-byte chunk, the last one shorter)
#     root   = SHAKE256(b'LCB200-AGTREE' || le64(len(M)) || leaf_0 || leaf_1 || ...)[:32]
# and coefficient i hashes ag_salt || str(i) || root.hex() - one permutation each.  The coefficients still depend on
# every key and message of the sorted list (through the commitment), so the rogue-key argument is unchanged, but they
# are NOT the reference's coefficients: aggregates made in one mode do not verify in the other.  Off by default.
AG_MODES = ('reference', 'tree')
TREE_LEAF_BYTES = 8192
TREE_DOMAIN = b'LCB200-AGTREE'


def set_aggregation_mode(pp: PublicParameters, mode: str) -> PublicParameters:
    if mode not in AG_MODES:
        raise ValueError(f"ag_mode must be one of {AG_MODES}")
    pp['ag_mode'] = mode
    return pp


def commit_aggregation_message(pp: PublicParameters, agmsg) -> str:
    """The 64-hex-digit tree commitment of an aggregation message (both levels hashed on the GPU)."""
    eng, _ = _ctx(pp)
    raw = agmsg.encode() if isinstance(agmsg, str) else bytes(agmsg)
    blob = np.frombuffer(raw, dtype=np.uint8) if raw else np.zeros(0, dtype=np.uint8)
    cuts = np.arange(0, len(raw), TREE_LEAF_BYTES, dtype=np.int64)
    off = np.concatenate([cuts, np.array([len(raw)], dtype=np.int64)]) if len(raw) else np.zeros(1, dtype=np.int64)
    leaves = eng.shake256((np.ascontiguousarray(blob), off), 32) if len(raw) else np.zeros((0, 32), dtype=np.uint8)
    top = TREE_DOMAIN + len(raw).to_bytes(8, 'little') + leaves.tobytes()
    return bytes(eng.shake256([top], 32)[0]).hex()


def _agg_message(pp: PublicParameters, agmsg):
    """What the aggregation coefficients hash behind ag_salt || str(i): the message itself (reference) or its commitment."""
    return commit_aggregation_message(pp, agmsg) if pp.get('ag_mode', 'reference') == 'tree' else agmsg


# ------------------------------------------------------------------------------- host-side preparation
def prepare_make_agg_coefs(otvks: List[OneTimeVerificationKey], msgs: List[Message]) -> Tuple[
        List[OneTimeVerificationKey], List[Message]]:
    if len(otvks) != len(msgs):
        raise ValueError("Cannot prepare_make_agg_coefs without two input vectors of equal length.")
    elif not all(is_bitstring(msg) for msg in msgs):
        raise ValueError("Input messages must be bitstrings.")
    order = sorted(range(len(otvks)), key=lambda i: str(otvks[i]))      # stable, like sorted() on the zip
    return [otvks[i] for i in order], [msgs[i] for i in order]


def prepare_hash2polyinput(pp: PublicParameters, otvks: List[OneTimeVerificationKey], msgs: List[Message]) -> dict:
    srt_keys, srt_msgs = prepare_make_agg_coefs(otvks=otvks, msgs=msgs)
    sp = pp['scheme_parameters']
    return {'secpar': sp.secpar, 'lp': sp.lp, 'distribution': sp.distribution,
            'dist_pars': {'bd': pp['ag_bd'], 'wt': pp['ag_wt']}, 'num_coefs': pp['ag_wt'],
            'bti': bits_to_indices(secpar=sp.secpar, degree=sp.lp.degree, wt=pp['ag_wt']),
            'btd': bits_to_decode(secpar=sp.secpar, bd=pp['ag_bd']),
            'msg': str(list(zip(srt_keys, srt_msgs))), 'const_time_flag': False}


def _monomials(lp, pairs: np.ndarray) -> List[AggCoef]:
    """(index, value) pairs int16[n][ag_wt][2] -> the n aggregation coefficients as Polynomials."""
    return [Polynomial(lp, {int(k): int(v) for k, v in row}, const_time_flag=False) for row in pairs]


def make_agg_coefs(pp: PublicParameters, otvks: List[OneTimeVerificationKey], msgs: List[Message]) -> List[AggCoef]:
    h2p = prepare_hash2polyinput(pp=pp, otvks=otvks, msgs=msgs)
    eng, sch = _ctx(pp)
    return _monomials(h2p['lp'], eng.agg_coefs(sch, _agg_message(pp, h2p['msg']), 0, len(otvks)))


def prepare_aggregate(otvks: List[OneTimeVerificationKey], msgs: List[Message], sigs: List[Signature]) -> Tuple[
        List[OneTimeVerificationKey], List[Message], List[Signature]]:
    order = sorted(range(len(otvks)), key=lambda i: str(otvks[i]))
    return [otvks[i] for i in order], [msgs[i] for i in order], [sigs[i] for i in order]


# ------------------------------------------------------------------------------- sharded engine API
# Aggregation coefficients are a function of (ag_salt, ag_bd, ag_wt, ring, the aggregation message, the index range)
# alone, and deriving them is the O(N^2) part of both aggregate and aggregate_verify (bklm_one_time_agg_sigs.py:60-81).
# A process that aggregates and then verifies the same list (the reference's own test_all does) would hash every
# coefficient twice; the last few derivations are therefore kept, keyed by a digest of the message CONTENT.
_AG_CACHE: Dict[tuple, object] = {}
_AG_CACHE_SLOTS = 4


def clear_agg_coef_cache() -> None:
    _AG_CACHE.clear()


def _agg_coefs_cached(pp: PublicParameters, eng, sch, agmsg, first: int, count: int, device: bool):
    import hashlib
    raw = agmsg.encode() if isinstance(agmsg, str) else (bytes(agmsg) if isinstance(agmsg, (bytes, bytearray)) else None)
    if raw is None:                                    # device / array messages: no content key, derive
        return eng.agg_coefs(sch, agmsg, first, count, device=device)
    lp = pp['scheme_parameters'].lp
    key = (hashlib.blake2b(raw, digest_size=20).digest(), len(raw), first, count, device, pp['scheme_parameters'].secpar,
           lp.modulus, lp.degree, pp.get('ag_salt', 'AG_SALT'), pp.get('ag_bd', 1), pp.get('ag_wt', 1))
    hit = _AG_CACHE.get(key)
    if hit is None:
        hit = eng.agg_coefs(sch, raw, first, count, device=device)
        while len(_AG_CACHE) >= _AG_CACHE_SLOTS:
            _AG_CACHE.pop(next(iter(_AG_CACHE)))
        _AG_CACHE[key] = hit
    return hit


def aggregate_shard(pp: PublicParameters, sig_sorted, agmsg, first: int, device: bool = False):
    """int32[l,d] partial sum over the shard of the SORTED signature list that starts at global
    position `first` (sig_sorted int16[count,l,d]); aggregation coefficients are derived here."""
    eng, sch = _ctx(pp)
    count = int(sig_sorted.shape[0])
    ag = _agg_coefs_cached(pp, eng, sch, _agg_message(pp, agmsg), first, count, device)
    return eng.aggregate_partial(sch, sig_sorted, ag, device=device)


def aggregate_finish(pp: PublicParameters, partial_sum, device: bool = False):
    eng, _ = _ctx(pp)
    return eng.aggregate_finish(partial_sum, device=device)


def aggregate_verify_shard(pp: PublicParameters, vk_ntt_sorted, chmsgs_sorted, agmsg, first: int, device: bool = False):
    """int32[d] partial sum (NTT form) of (vk_left*c + vk_right) * ag over one shard of the sorted list."""
    eng, sch = _ctx(pp)
    count = int(vk_ntt_sorted.shape[0])
    ag = _agg_coefs_cached(pp, eng, sch, _agg_message(pp, agmsg), first, count, device)
    return eng.aggverify_partial(sch, vk_ntt_sorted, chmsgs_sorted, ag, device=device)


def aggregate_verify_finish(pp: PublicParameters, partial_sum, ag_sig, total: int) -> bool:
    eng, _ = _ctx(pp)
    return eng.aggverify_finish(partial_sum, ag_sig, total, pp['ag_cap'], pp['avf_bd'], pp['avf_wt'])


# ------------------------------------------------------------------------------- drop-in API
def aggregate(pp: PublicParameters, otvks: List[OneTimeVerificationKey], msgs: List[Message],
              sigs: List[Signature]) -> Signature:
    srt_keys, srt_msgs, srt_sigs = prepare_aggregate(otvks=otvks, msgs=msgs, sigs=sigs)
    agmsg = prepare_hash2polyinput(pp=pp, otvks=otvks, msgs=msgs)['msg']
    sig_sorted = np.ascontiguousarray(np.stack([s.coef for s in srt_sigs]))
    partial = aggregate_shard(pp, sig_sorted, agmsg, 0)
    return PolynomialVector(pp['scheme_parameters'].lp, const_time_flag=False, _coef=aggregate_finish(pp, partial))


def aggregate_verify(pp: PublicParameters, otvks: List[OneTimeVerificationKey], msgs: List[Message],
                     ag_sig: Signature) -> bool:
    if len(otvks) < 1 or len(otvks) > pp['ag_cap'] or len(otvks) != len(msgs):
        return False
    if not well_formed(pp['scheme_parameters'].lp, ag_sig):
        return False
    srt_keys, srt_msgs = prepare_make_agg_coefs(otvks=otvks, msgs=msgs)
    agmsg = str(list(zip(srt_keys, srt_msgs)))
    vk_sorted = np.ascontiguousarray(np.stack([np.stack([k[0].ntt, k[1].ntt]) for k in srt_keys]))
    partial = aggregate_verify_shard(pp, vk_sorted, challenge_messages(srt_keys, srt_msgs), agmsg, 0)
    return aggregate_verify_finish(pp, partial, np.ascontiguousarray(ag_sig.coef), len(otvks))


# ------------------------------------------------------------------------------- batched drop-in API
def _commit_batch(pp: PublicParameters, agmsgs: List[str]) -> List[str]:
    """commit_aggregation_message of every message, with two hash calls in all: every leaf of every message, then
    every root."""
    eng, _ = _ctx(pp)
    raws = [m.encode() for m in agmsgs]
    lens = [len(r) for r in raws]
    base = np.concatenate([[0], np.cumsum(lens, dtype=np.int64)]).astype(np.int64)
    cuts = [np.arange(base[g], base[g + 1], TREE_LEAF_BYTES, dtype=np.int64) for g in range(len(raws))]
    nleaf = [len(c) for c in cuts]
    leaves = np.zeros((0, 32), dtype=np.uint8)
    if sum(nleaf):
        blob = np.frombuffer(b''.join(raws), dtype=np.uint8)
        off = np.concatenate(cuts + [base[-1:]]).astype(np.int64)
        leaves = eng.shake256((np.ascontiguousarray(blob), off), 32)
    first = np.concatenate([[0], np.cumsum(nleaf)]).astype(np.int64)
    tops = [TREE_DOMAIN + lens[g].to_bytes(8, 'little') + leaves[first[g]:first[g + 1]].tobytes() for g in range(len(raws))]
    if not tops:
        return []
    return [bytes(r).hex() for r in eng.shake256(tops, 32)]


def _batch_messages(pp: PublicParameters, agmsgs: List[str]) -> List[str]:
    return _commit_batch(pp, agmsgs) if pp.get('ag_mode', 'reference') == 'tree' else agmsgs


def _check_messages(otvks, msgs) -> None:
    """The argument checks of prepare_make_agg_coefs, without its sort."""
    if len(otvks) != len(msgs):
        raise ValueError("Cannot prepare_make_agg_coefs without two input vectors of equal length.")
    elif not all(is_bitstring(msg) for msg in msgs):
        raise ValueError("Input messages must be bitstrings.")


def aggregate_batch(pp: PublicParameters, otvks: List[List[OneTimeVerificationKey]], msgs: List[List[Message]],
                    sigs: List[List[Signature]]) -> List[Signature]:
    """[aggregate(pp, otvks[g], msgs[g], sigs[g]) for every g] in one engine call (same errors, raised for the first
    group that has one).  Sorting and the aggregation message stay on the host, once per group."""
    if not len(otvks) == len(msgs) == len(sigs):
        raise ValueError('aggregate_batch needs one list of keys, messages and signatures per aggregate')
    sp = pp['scheme_parameters']
    rows, agmsgs, counts = [], [], []
    for keys_g, msgs_g, sigs_g in zip(otvks, msgs, sigs):
        srt_keys, srt_msgs, srt_sigs = prepare_aggregate(otvks=keys_g, msgs=msgs_g, sigs=sigs_g)
        _check_messages(keys_g, msgs_g)
        if not srt_sigs:
            raise ValueError('need at least one array to stack')      # what aggregate() raises for an empty group
        rows.extend(s.coef for s in srt_sigs)
        agmsgs.append(str(list(zip(srt_keys, srt_msgs))))
        counts.append(len(srt_sigs))
    if not counts:
        return []
    eng, sch = _ctx(pp)
    agg_off = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
    out = eng.aggregate_batch(sch, agg_off, np.ascontiguousarray(np.stack(rows)), _batch_messages(pp, agmsgs))
    return [PolynomialVector(sp.lp, const_time_flag=False, _coef=out[g]) for g in range(len(counts))]


def aggregate_verify_batch(pp: PublicParameters, otvks: List[List[OneTimeVerificationKey]], msgs: List[List[Message]],
                           ag_sigs: List[Signature]) -> List[bool]:
    """[aggregate_verify(pp, otvks[g], msgs[g], ag_sigs[g]) for every g]: the host-side early False (length mismatch,
    over capacity, ill-formed aggregate) per group, then every remaining group in one engine call."""
    if not len(otvks) == len(msgs) == len(ag_sigs):
        raise ValueError('aggregate_verify_batch needs one list of keys and messages and one aggregate per group')
    lp = pp['scheme_parameters'].lp
    verdicts = [False] * len(otvks)
    live, vks, chmsgs, agmsgs, counts, ags = [], [], [], [], [], []
    for g, (keys_g, msgs_g, ag_g) in enumerate(zip(otvks, msgs, ag_sigs)):
        if len(keys_g) < 1 or len(keys_g) > pp['ag_cap'] or len(keys_g) != len(msgs_g):
            continue
        if not well_formed(lp, ag_g):
            continue
        srt_keys, srt_msgs = prepare_make_agg_coefs(otvks=keys_g, msgs=msgs_g)
        vks.extend(np.stack([k[0].ntt, k[1].ntt]) for k in srt_keys)
        chmsgs.extend(challenge_messages(srt_keys, srt_msgs))
        agmsgs.append(str(list(zip(srt_keys, srt_msgs))))
        counts.append(len(srt_keys))
        ags.append(ag_g.coef)
        live.append(g)
    if not live:
        return verdicts
    eng, sch = _ctx(pp)
    agg_off = np.concatenate([[0], np.cumsum(counts)]).astype(np.int64)
    got = eng.aggregate_verify_batch(sch, agg_off, np.ascontiguousarray(np.stack(vks)), chmsgs, _batch_messages(pp, agmsgs),
                                     np.ascontiguousarray(np.stack(ags)), pp['ag_cap'], pp['avf_bd'], pp['avf_wt'])
    for g, v in zip(live, got):
        verdicts[g] = bool(v)
    return verdicts
