"""Packed wire format for verification keys and signatures, and a public-seed `key_ch` (SURVEY.md 8(f)2-3).

The reference has neither: keys and signatures are live Python objects whose `str()` is a memory address
(`one_time_keys.py:197-237`) and the public row `key_ch` is drawn from `secrets`
(`one_time_keys.py:284-290`), so it has to be shipped as 6.6 / 11.8 KB of coefficients.  Everything in this
module is therefore OPT-IN and does not change what the drop-in API computes:

* `pack_signatures` / `unpack_signatures`: centred coefficients in `sig_bits(pp)` bits (11 at secpar 128,
  13 at 256) instead of 16 - 4,576 / 9,568 bytes per signature instead of 6,656 / 11,776;
* `pack_keys` / `unpack_keys`: NTT-form verification keys in `key_bits(pp)` bits (14 / 16);
* `verify_batch_packed`: `lm_one_time_sigs.verify_batch` straight from the packed records;
* `sign_batch_packed`: `lm_one_time_sigs.sign_batch` straight into packed signatures (bias `vf_bd`), without the int16
  signatures making a round trip;
* adaptor signatures (`adaptor_sigs`) on packed records, every width and bias taken from the adaptor `pp`:
  `presign_batch_packed` (presignatures in `sig_bits(pp, 'pvf_bd')` bits, bias `pvf_bd`: 11 / 13), `preverify_batch_packed`,
  `adapt_batch_packed` (adaptor signatures in `sig_bits(pp)` bits, bias `vf_bd`: 11 / 13), `adaptor_verify_batch_packed`
  (statements packed like keys with `pack_keys`) and `extract_batch_packed` (int16 witnesses);
* adaptor witnesses on packed records, so that the adaptor lifecycle runs on packed records only.  A witness is packed
  like a signature with a witness bound: `pack_witnesses` / `unpack_witnesses` (`bound_key='wit_bd'`: 2 bits, bias 1 -
  832 / 1,472 bytes per witness instead of 6,656 / 11,776; `'ext_wit_bd'`: 12 / 14 bits, lossless for every witness
  that witness verification can accept); `witgen_batch_packed` (packed witnesses and statements straight from the
  seeds), `adapt_batch_packed_wit` (adapt with a packed witness), `extract_batch_packed_wit` (packed witnesses out of
  extract, with in_range flags: a 2-bit extraction cannot hold a valid witness that is not the genuine one) and
  `witness_verify_batch_packed` (bound ext_wit_bd, weight ext_wit_wt);
* signing keys in COEFFICIENT form, `signing_key_bits(pp)` bits (7 at secpar 128, 8 at 256) with bias sk_bd - 5,824 /
  11,776 bytes per key instead of 13,312 / 23,552 for the uint16 NTT form: `pack_signing_keys` / `unpack_signing_keys`,
  `keygen_batch_packed` (packed signing and verification keys straight from the seeds) and `sign_batch_packed_sk` /
  `presign_batch_packed_sk` (packed signatures / presignatures straight from packed signing keys), so that the one-time
  signature lifecycle runs on packed records only;
* `aggregate_batch_packed` / `aggregate_verify_batch_packed`: the batched BKLM calls of `bklm_one_time_agg_sigs`
  (many independent aggregates, sorted signatures / keys of group g at agg_off[g] .. agg_off[g+1]) from packed
  signatures and keys, with packed aggregates.  An aggregate is encoded as a signature with the aggregate bound:
  `pack_signatures(pp, ag, bound_key='avf_bd')`, `sig_bits(pp, 'avf_bd')` bits (12 at secpar 128, 14 at 256), bias
  `avf_bd`;
* `setup_parameters_from_seed`: `make_setup_parameters` with `key_ch = H2PV('KEY_CH_SALT' || seed)` sampled on
  the GPU with the reference's own distribution parameters (bd = q//2, wt = d), so that two parties derive
  the same row from a short public string.

* `one_time_keys.set_content_str(True)` (re-exported here as `set_content_str`): `str()` / `repr()` of
  verification keys and public statements become content digests, so signatures verify against pickled or
  re-created key objects (changes the challenge bytes, hence every signature; off by default).  In that mode a packed
  key received over the wire identifies its key, and the hash inputs are built on the GPU from packed records and raw
  messages: `content_strs` (the 57-byte repr() of packed keys or statements), `challenge_inputs` (the `chmsgs` of every
  packed sign / verify / adaptor call) and `aggregation_inputs` (the per-group sort order, sorted `chmsgs` and
  aggregation messages of the packed BKLM calls; the order is sorted on the GPU over the 57-byte strings).
  `sorted_aggregation_inputs`, `aggregate_batch_content` and `aggregate_verify_batch_content` take UNSORTED packed keys,
  raw messages and packed signatures (aggregates) and do the sort and the permutation of the records on the GPU too, so
  that with device=True a batch never leaves the device (reference ag_mode only).  The drop-in `challenge_messages` and
  `aggregate_batch` keep building them on the host.

Bit layout (include/lcb200.h): value i of a polynomial at bit offset i*bits, least significant bit first.
"""
from math import ceil, log2
from typing import Any, Dict

import numpy as np

from .engine import Engine, _want, ragged
from .lattice_algebra import PolynomialVector, engine_for
from .one_time_keys import SchemeParameters, set_content_str  # noqa: F401

KEY_CH_SALT = 'KEY_CH_SALT'


def sig_bits(pp: Dict[str, Any], bound_key: str = 'vf_bd') -> int:
    """Bits per signature coefficient: the range [-bd, bd] has 2*bd + 1 values."""
    return max(1, ceil(log2(2 * pp[bound_key] + 1)))


def key_bits(pp: Dict[str, Any]) -> int:
    return ceil(log2(pp['scheme_parameters'].lp.modulus))


def signing_key_bits(pp: Dict[str, Any]) -> int:
    """Bits per signing-key coefficient: the sampler draws them from [-sk_bd, sk_bd]."""
    return max(1, ceil(log2(2 * pp['sk_bd'] + 1)))


def _engine(pp):
    sp = pp['scheme_parameters']
    return engine_for(sp.lp, sp.secpar)


def pack_signatures(pp, sig, device: bool = False, bound_key: str = 'vf_bd'):
    """sig int16[..., l, 256] -> (uint8[..., l, 32*bits], in_range uint8[..., l]).  A polynomial with a
    coefficient outside [-bd, 2^bits - 1 - bd] cannot be represented; its in_range flag is 0."""
    return _engine(pp).pack(sig, sig_bits(pp, bound_key), pp[bound_key], device=device, want_range=True)


def unpack_signatures(pp, packed, device: bool = False, bound_key: str = 'vf_bd'):
    return _engine(pp).unpack(packed, sig_bits(pp, bound_key), pp[bound_key], dtype=np.int16, device=device)


def pack_keys(pp, vk_ntt, device: bool = False):
    """vk_ntt uint16[..., 256] (engine NTT form, values < q) -> uint8[..., 32*key_bits]."""
    return _engine(pp).pack(vk_ntt, key_bits(pp), 0, device=device)


def unpack_keys(pp, packed, device: bool = False):
    return _engine(pp).unpack(packed, key_bits(pp), 0, dtype=np.uint16, device=device)


def pack_signing_keys(pp, sk_coef, device: bool = False):
    """sk_coef int16[..., 2, l, 256] (coefficient form, as `lm_keygen` returns it) -> (uint8[..., 2, l, 32*signing_key_bits],
    in_range uint8[..., 2, l]), bias sk_bd."""
    return _engine(pp).pack(sk_coef, signing_key_bits(pp), pp['sk_bd'], device=device, want_range=True)


def unpack_signing_keys(pp, packed, device: bool = False):
    return _engine(pp).unpack(packed, signing_key_bits(pp), pp['sk_bd'], dtype=np.int16, device=device)


def keygen_batch_packed(pp, seeds, device: bool = False):
    """Packed keys straight from the seeds (the seed forms of `lm_one_time_sigs.keygen_batch`, including the output of
    `random_seed_batch`): -> (sk_packed uint8[N, 2, l, 32*signing_key_bits(pp)], vk_packed uint8[N, 2, 32*key_bits(pp)]),
    exactly `pack_signing_keys` / `pack_keys` of the keys `keygen_batch` makes; no 16-bit key leaves the engine."""
    from .lm_one_time_sigs import SecretSeed, _ctx
    eng, sch = _ctx(pp)
    if isinstance(seeds, tuple) and len(seeds) == 2 and not isinstance(seeds[0], (str, SecretSeed)):
        strs = seeds                # already (byte blob, int64 offsets), e.g. from random_seed_batch
    else:
        strs = [s.seed if isinstance(s, SecretSeed) else s for s in seeds]
    sk, _, vk = eng.lm_keygen_packed(sch, strs, signing_key_bits(pp), pp['sk_bd'], key_bits(pp), device=device)
    return sk, vk


def sign_batch_packed_sk(pp, sk_packed, chmsgs, device: bool = False):
    """LM signatures from packed signing keys straight into the wire format: -> (uint8[N, l, 32*sig_bits], in_range
    uint8[N, l]), bias vf_bd; exactly `sign_batch_packed(pp, ntt_fwd(unpack_signing_keys(pp, sk_packed)), chmsgs)`."""
    from .lm_one_time_sigs import _ctx
    eng, sch = _ctx(pp)
    return eng.lm_sign_packed_sk(sch, sk_packed, signing_key_bits(pp), pp['sk_bd'], chmsgs, sig_bits(pp), pp['vf_bd'],
                                 device=device, want_range=True)


def presign_batch_packed_sk(pp, sk_packed, chmsgs, device: bool = False):
    """Adaptor presignatures (adaptor `pp`) from packed signing keys -> (uint8[N, l, 32*sig_bits(pp, 'pvf_bd')], in_range
    uint8[N, l]), bias pvf_bd."""
    from .adaptor_sigs import _ctx
    eng, sch = _ctx(pp)
    return eng.lm_sign_packed_sk(sch, sk_packed, signing_key_bits(pp), pp['sk_bd'], chmsgs, sig_bits(pp, 'pvf_bd'),
                                 pp['pvf_bd'], device=device, want_range=True)


def verify_batch_packed(pp, vk_packed, chmsgs, sig_packed, device: bool = False):
    """N verdicts (uint8) from packed keys uint8[N, 2, 32*key_bits] and signatures uint8[N, l, 32*sig_bits]."""
    from .lm_one_time_sigs import _ctx
    eng, sch = _ctx(pp)
    return eng.lm_verify_packed(sch, vk_packed, key_bits(pp), chmsgs, sig_packed, sig_bits(pp), pp['vf_bd'],
                                pp['vf_bd'], pp['vf_wt'], device=device)


def sign_batch_packed(pp, sk_ntt, chmsgs, device: bool = False):
    """LM signatures straight into the wire format: sk_ntt uint16[N, 2, l, 256] -> (uint8[N, l, 32*sig_bits], in_range
    uint8[N, l]), exactly `pack_signatures(pp, sign_batch(pp, sk_ntt, chmsgs))`."""
    from .lm_one_time_sigs import _ctx
    eng, sch = _ctx(pp)
    return eng.lm_sign_packed(sch, sk_ntt, chmsgs, sig_bits(pp), pp['vf_bd'], device=device, want_range=True)


def presign_batch_packed(pp, sk_ntt, chmsgs, device: bool = False):
    """Adaptor presignatures (adaptor `pp`; chmsgs from `adaptor_sigs.challenge_messages`) -> (uint8[N, l,
    32*sig_bits(pp, 'pvf_bd')], in_range uint8[N, l]), bias pvf_bd."""
    from .adaptor_sigs import _ctx
    eng, sch = _ctx(pp)
    return eng.lm_sign_packed(sch, sk_ntt, chmsgs, sig_bits(pp, 'pvf_bd'), pp['pvf_bd'], device=device, want_range=True)


def preverify_batch_packed(pp, vk_packed, chmsgs, presig_packed, device: bool = False):
    """N preverify verdicts from packed keys and packed presignatures (bound pvf_bd, weight pvf_wt)."""
    from .adaptor_sigs import _ctx
    eng, sch = _ctx(pp)
    return eng.lm_verify_packed(sch, vk_packed, key_bits(pp), chmsgs, presig_packed, sig_bits(pp, 'pvf_bd'), pp['pvf_bd'],
                                pp['pvf_bd'], pp['pvf_wt'], device=device)


def adapt_batch_packed(pp, presig_packed, wit_coef, device: bool = False):
    """Packed presignatures + witnesses int16[N, l, 256] -> (adaptor signatures uint8[N, l, 32*sig_bits(pp)], in_range
    uint8[N, l]), bias vf_bd."""
    from .adaptor_sigs import _ctx
    eng, _ = _ctx(pp)
    return eng.adapt_packed(presig_packed, sig_bits(pp, 'pvf_bd'), pp['pvf_bd'], wit_coef, sig_bits(pp), pp['vf_bd'],
                            device=device, want_range=True)


def extract_batch_packed(pp, presig_packed, sig_packed, device: bool = False):
    """Witnesses int16[N, l, 256] = signature - presignature, from the two packed records."""
    from .adaptor_sigs import _ctx
    eng, _ = _ctx(pp)
    return eng.extract_packed(sig_packed, sig_bits(pp), pp['vf_bd'], presig_packed, sig_bits(pp, 'pvf_bd'), pp['pvf_bd'],
                              device=device)


def adaptor_verify_batch_packed(pp, vk_packed, chmsgs, st_packed, sig_packed, device: bool = False):
    """N adaptor verify verdicts from packed keys, packed statements uint8[N, 32*key_bits] (`pack_keys(pp, st_ntt)`)
    and packed adaptor signatures (bound vf_bd, weight vf_wt)."""
    from .adaptor_sigs import _ctx
    eng, sch = _ctx(pp)
    return eng.adaptor_verify_packed(sch, vk_packed, key_bits(pp), chmsgs, sig_packed, sig_bits(pp), pp['vf_bd'], st_packed,
                                     key_bits(pp), pp['vf_bd'], pp['vf_wt'], device=device)


def pack_witnesses(pp, wit_coef, device: bool = False, bound_key: str = 'wit_bd'):
    """Adaptor witnesses int16[..., l, 256] -> (uint8[..., l, 32*sig_bits(pp, bound_key)], in_range uint8[..., l]), bias
    pp[bound_key]."""
    return _engine(pp).pack(wit_coef, sig_bits(pp, bound_key), pp[bound_key], device=device, want_range=True)


def unpack_witnesses(pp, packed, device: bool = False, bound_key: str = 'wit_bd'):
    return _engine(pp).unpack(packed, sig_bits(pp, bound_key), pp[bound_key], dtype=np.int16, device=device)


def witgen_batch_packed(pp, seeds, device: bool = False):
    """Adaptor witnesses and statements straight from the seeds (the seed forms of `adaptor_sigs.witgen_batch`) ->
    (wit_packed uint8[N, l, 32*sig_bits(pp, 'wit_bd')], st_packed uint8[N, 32*key_bits(pp)]), exactly
    `pack_witnesses` / `pack_keys` of what `witgen_batch` makes; no 16-bit witness leaves the engine."""
    from .adaptor_sigs import SecretSeed, _ctx
    eng, sch = _ctx(pp)
    if isinstance(seeds, tuple) and len(seeds) == 2 and not isinstance(seeds[0], (str, SecretSeed)):
        strs = seeds                # already (byte blob, int64 offsets)
    else:
        strs = [s.seed if isinstance(s, SecretSeed) else s for s in seeds]
    wit, _, st = eng.witgen_packed(sch, strs, sig_bits(pp, 'wit_bd'), pp['wit_bd'], key_bits(pp), device=device)
    return wit, st


def adapt_batch_packed_wit(pp, presig_packed, wit_packed, device: bool = False):
    """Packed presignatures + packed witnesses (`pack_witnesses`) -> (adaptor signatures uint8[N, l, 32*sig_bits(pp)],
    in_range uint8[N, l]), bias vf_bd; exactly `adapt_batch_packed(pp, presig_packed, unpack_witnesses(pp, wit_packed))`."""
    from .adaptor_sigs import _ctx
    eng, _ = _ctx(pp)
    return eng.adapt_packed_wit(presig_packed, sig_bits(pp, 'pvf_bd'), pp['pvf_bd'], wit_packed, sig_bits(pp, 'wit_bd'),
                                pp['wit_bd'], sig_bits(pp), pp['vf_bd'], device=device, want_range=True)


def extract_batch_packed_wit(pp, presig_packed, sig_packed, device: bool = False, bound_key: str = 'ext_wit_bd'):
    """Packed witnesses = signature - presignature, from the two packed records -> (uint8[N, l, 32*sig_bits(pp,
    bound_key)], in_range uint8[N, l]), bias pp[bound_key].  The default width holds every witness that
    `witness_verify_batch_packed` can accept; at bound_key='wit_bd' a valid witness that is not the genuine one reads
    in_range 0."""
    from .adaptor_sigs import _ctx
    eng, _ = _ctx(pp)
    return eng.extract_packed_wit(sig_packed, sig_bits(pp), pp['vf_bd'], presig_packed, sig_bits(pp, 'pvf_bd'),
                                  pp['pvf_bd'], sig_bits(pp, bound_key), pp[bound_key], device=device, want_range=True)


def witness_verify_batch_packed(pp, wit_packed, st_packed, device: bool = False, bound_key: str = 'wit_bd'):
    """N witness verdicts (uint8) from packed witnesses uint8[N, l, 32*sig_bits(pp, bound_key)] (bias pp[bound_key]) and
    packed statements uint8[N, 32*key_bits(pp)], with bound ext_wit_bd and weight ext_wit_wt as
    `adaptor_sigs.witness_verify_batch`."""
    from .adaptor_sigs import _ctx
    eng, _ = _ctx(pp)
    return eng.witness_verify_packed(wit_packed, sig_bits(pp, bound_key), pp[bound_key], st_packed, key_bits(pp),
                                     pp['ext_wit_bd'], pp['ext_wit_wt'], device=device)


def aggregate_batch_packed(pp, agg_off, sig_packed, agmsgs, device: bool = False):
    """Aggregates of many groups from packed sorted signatures uint8[total, l, 32*sig_bits] (agmsgs[g]: the aggregation
    message of group g, committed first in tree mode as `bklm_one_time_agg_sigs.aggregate_batch` does) ->
    (ag_packed uint8[n_agg, l, 32*sig_bits(pp, 'avf_bd')], in_range uint8[n_agg, l])."""
    from .bklm_one_time_agg_sigs import _batch_messages, _ctx
    eng, sch = _ctx(pp)
    return eng.aggregate_packed_batch(sch, agg_off, sig_packed, sig_bits(pp), pp['vf_bd'], _batch_messages(pp, list(agmsgs)),
                                      sig_bits(pp, 'avf_bd'), pp['avf_bd'], device=device, want_range=True)


def aggregate_verify_batch_packed(pp, agg_off, vk_packed, chmsgs_sorted, agmsgs, ag_packed, device: bool = False):
    """uint8[n_agg] verdicts of many aggregates from packed sorted keys uint8[total, 2, 32*key_bits] and packed aggregates
    uint8[n_agg, l, 32*sig_bits(pp, 'avf_bd')]; an empty group or one above ag_cap verifies as 0."""
    from .bklm_one_time_agg_sigs import _batch_messages, _ctx
    eng, sch = _ctx(pp)
    return eng.aggregate_verify_packed_batch(sch, agg_off, vk_packed, key_bits(pp), chmsgs_sorted,
                                             _batch_messages(pp, list(agmsgs)), ag_packed, sig_bits(pp, 'avf_bd'),
                                             pp['avf_bd'], pp['ag_cap'], pp['avf_bd'], pp['avf_wt'], device=device)


def content_strs(pp, packed, kind: str = 'vk', device: bool = False):
    """Content-mode repr() of packed keys uint8[N, 2, 32*key_bits] (kind 'vk') or packed statements uint8[N, 32*key_bits]
    ('st') -> uint8[N, 57], byte for byte what `repr()` of the drop-in objects gives after `set_content_str(True)`."""
    return _engine(pp).content_str(kind, packed, key_bits(pp), device=device)


def challenge_inputs(pp, vk_packed, msgs, st_packed=None, device: bool = False):
    """Content-mode challenge messages of packed keys (and packed statements for the adaptor challenge) and raw messages
    -> (blob, offsets): exactly `lm_one_time_sigs.challenge_messages` (or `adaptor_sigs.challenge_messages`) of the
    drop-in objects in content mode, ready as `chmsgs` for `sign_batch_packed_sk`, `verify_batch_packed`,
    `presign_batch_packed_sk`, `preverify_batch_packed` and `adaptor_verify_batch_packed`."""
    eng = _engine(pp)
    vk_str = content_strs(pp, vk_packed, 'vk', device=device)
    st_str = content_strs(pp, st_packed, 'st', device=device) if st_packed is not None else None
    return eng.challenge_inputs(vk_str, msgs, st_str=st_str, device=device)


def aggregation_inputs(pp, agg_off, vk_packed, msgs, device: bool = False):
    """The BKLM inputs of many groups (items agg_off[g] .. agg_off[g+1] of packed keys uint8[total, 2, 32*key_bits] and
    bitstring messages) in content mode -> (order, chmsgs_sorted, agmsgs):
      order          int64[total], within every group the stable sort by content string of `prepare_make_agg_coefs`;
      chmsgs_sorted  (blob, offsets) challenge messages of the sorted items;
      agmsgs         list of the n_agg aggregation messages str(list(zip(sorted keys, sorted messages))).
    Permute the packed signatures / keys by `order` and pass these to `aggregate_batch_packed` /
    `aggregate_verify_batch_packed`, or use `aggregate_batch_content` / `aggregate_verify_batch_content`, which do all of
    it on the device.  Each key is hashed once and the order is sorted on the GPU (`Engine.content_order`)."""
    from .lattice_algebra import is_bitstring
    msgs = list(msgs)
    if not all(is_bitstring(m) for m in msgs):
        raise ValueError("Input messages must be bitstrings.")
    agg_off = np.ascontiguousarray(agg_off, dtype=np.int64)
    total = len(msgs)
    if agg_off.ndim != 1 or agg_off.shape[0] < 1 or int(agg_off[0]) != 0 or int(agg_off[-1]) != total or \
            bool((np.diff(agg_off) < 0).any()):
        raise ValueError(f'agg_off must start at 0, never decrease and end at the number of messages ({total})')
    eng = _engine(pp)
    vk_str = content_strs(pp, vk_packed, 'vk')
    order = eng.content_order(agg_off, vk_str)
    vk_sorted = np.ascontiguousarray(vk_str[order])
    msgs_sorted = [msgs[i] for i in order]
    chmsgs = eng.challenge_inputs(vk_sorted, msgs_sorted, device=device)
    blob, off = eng.aggregation_inputs(agg_off, vk_sorted, msgs_sorted)
    raw = blob.tobytes()
    agmsgs = [raw[int(off[g]):int(off[g + 1])].decode() for g in range(off.shape[0] - 1)]
    return order, chmsgs, agmsgs


def _content_messages(msgs):
    """Messages of the content-mode BKLM routes as (blob, offsets): a list of bitstrings is checked with the error of
    `prepare_make_agg_coefs` and packed; a (blob, offsets) pair, host or device, is taken as it is."""
    from .lattice_algebra import is_bitstring
    if isinstance(msgs, tuple) and len(msgs) == 2 and not isinstance(msgs[0], str):
        return Engine._rag(msgs)
    msgs = list(msgs)
    if not all(is_bitstring(m) for m in msgs):
        raise ValueError("Input messages must be bitstrings.")
    return ragged(msgs)


def _sorted_content(pp, agg_off, vk_packed, msgs, device):
    """-> (order, content strings and messages of the sorted items, aggregation messages (blob, offsets)), on the device
    when `device`."""
    if pp.get('ag_mode', 'reference') != 'reference':
        raise ValueError("the content-mode BKLM routes support ag_mode 'reference' only: in tree mode the commitment of "
                         "each aggregation message is built on the host")
    eng = _engine(pp)
    rag = _content_messages(msgs)
    vk_str = content_strs(pp, vk_packed, 'vk', device=device)
    if eng._count(rag[1]) != int(vk_str.shape[0]):
        raise ValueError(f'{eng._count(rag[1])} messages for {int(vk_str.shape[0])} keys')
    order = eng.content_order(agg_off, vk_str, device=device)
    str_sorted = eng.gather_rows(vk_str, order, device=device)
    msgs_sorted = eng.gather_ragged(rag, order, device=device)
    agmsgs = eng.aggregation_inputs(agg_off, str_sorted, msgs_sorted, device=device)
    return order, str_sorted, msgs_sorted, agmsgs


def sorted_aggregation_inputs(pp, agg_off, vk_packed, msgs, device: bool = False):
    """The BKLM inputs of many groups in content mode, sorted on the GPU from unsorted records: packed keys uint8[total, 2,
    32*key_bits] and messages (a list of bitstrings or a (blob, offsets) pair, items agg_off[g] .. agg_off[g+1] in group
    g) -> (order, vk_packed_sorted, chmsgs_sorted, agmsgs):
      order             int64[total], `aggregation_inputs`'s order;
      vk_packed_sorted  vk_packed[order];
      chmsgs_sorted     (blob, offsets) challenge messages of the sorted items;
      agmsgs            (blob, offsets) aggregation messages of the groups.
    The two message sets go to `Engine.aggregate_packed_batch` / `aggregate_verify_packed_batch` as they are.  With
    device=True every output is a device tensor and no record leaves the device.  Reference ag_mode only."""
    eng = _engine(pp)
    order, str_sorted, msgs_sorted, agmsgs = _sorted_content(pp, agg_off, vk_packed, msgs, device)
    vk_sorted = eng.gather_rows(vk_packed, order, device=device)
    chmsgs = eng.challenge_inputs(str_sorted, msgs_sorted, device=device)
    return order, vk_sorted, chmsgs, agmsgs


def aggregate_batch_content(pp, agg_off, vk_packed, msgs, sig_packed, device: bool = False):
    """Aggregates of many groups in content mode from UNSORTED packed keys, messages and packed signatures
    uint8[total, l, 32*sig_bits] -> (ag_packed uint8[n_agg, l, 32*sig_bits(pp, 'avf_bd')], in_range uint8[n_agg, l]):
    exactly `aggregate_batch_packed(pp, agg_off, sig_packed[order], agmsgs)` with `aggregation_inputs`'s order and
    messages, sorted and gathered on the GPU.  Reference ag_mode only."""
    from .bklm_one_time_agg_sigs import _ctx
    eng, sch = _ctx(pp)
    total = int(vk_packed.shape[0]) if len(getattr(vk_packed, 'shape', ())) else 0
    _want(sig_packed, 'sig_packed', np.uint8, (total, eng.l, eng.d * sig_bits(pp) // 8))
    order, _, _, agmsgs = _sorted_content(pp, agg_off, vk_packed, msgs, device)
    sig_sorted = eng.gather_rows(sig_packed, order, device=device)
    return eng.aggregate_packed_batch(sch, agg_off, sig_sorted, sig_bits(pp), pp['vf_bd'], agmsgs, sig_bits(pp, 'avf_bd'),
                                      pp['avf_bd'], device=device, want_range=True)


def aggregate_verify_batch_content(pp, agg_off, vk_packed, msgs, ag_packed, device: bool = False):
    """uint8[n_agg] verdicts of many aggregates in content mode from UNSORTED packed keys and messages and packed
    aggregates uint8[n_agg, l, 32*sig_bits(pp, 'avf_bd')]: exactly `aggregate_verify_batch_packed` on the inputs of
    `sorted_aggregation_inputs`, all of them made on the GPU.  Reference ag_mode only."""
    from .bklm_one_time_agg_sigs import _ctx
    eng, sch = _ctx(pp)
    _, vk_sorted, chmsgs, agmsgs = sorted_aggregation_inputs(pp, agg_off, vk_packed, msgs, device=device)
    return eng.aggregate_verify_packed_batch(sch, agg_off, vk_sorted, key_bits(pp), chmsgs, agmsgs, ag_packed,
                                             sig_bits(pp, 'avf_bd'), pp['avf_bd'], pp['ag_cap'], pp['avf_bd'], pp['avf_wt'],
                                             device=device)


def key_ch_from_seed(lp, secpar: int, seed: str) -> PolynomialVector:
    """Public row from a public string: H2PV(KEY_CH_SALT || seed) with bd = q//2, wt = d (the parameters of
    `SchemeParameters.__init__`, one_time_keys.py:284-290, with the hash in place of `secrets`)."""
    coef, _ = engine_for(lp, secpar).hash2polyvec(KEY_CH_SALT, [seed], lp.modulus // 2, lp.degree, lp.length)
    return PolynomialVector(lp, const_time_flag=False, _coef=coef[0])


def setup_parameters_from_seed(make_setup_parameters, secpar: int, seed: str):
    """`make_setup_parameters(secpar)` of any of the three scheme modules, with key_ch derived from `seed`."""
    pp = make_setup_parameters(secpar)
    sp = pp['scheme_parameters']
    pp['scheme_parameters'] = SchemeParameters(secpar=sp.secpar, lp=sp.lp, distribution=sp.distribution,
                                               key_ch=key_ch_from_seed(sp.lp, sp.secpar, seed))
    return pp
