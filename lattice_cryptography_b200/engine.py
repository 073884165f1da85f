"""Array-level Python face of the lcb200 C ABI.

Every method takes host (numpy) or device (torch.cuda) arrays; the library detects which.
Outputs are numpy arrays unless ``device=True`` (then torch CUDA tensors on the engine's
GPU, left on its stream).  Layouts are the ones documented in include/lcb200.h.
"""
import functools
import hashlib
import threading
from ctypes import byref, c_void_p
from typing import List, Optional, Sequence, Tuple, Union

import numpy as np

from . import _ffi
from ._ffi import LcbError, LcbScheme

D = 256
Bytes = Union[bytes, bytearray, str]


def ragged(items: Sequence[Bytes]) -> Tuple[np.ndarray, np.ndarray]:
    """list of byte strings (str is UTF-8 encoded, as lattice_algebra does) -> (blob, offsets)."""
    enc = [i.encode() if isinstance(i, str) else bytes(i) for i in items]
    off = np.zeros(len(enc) + 1, dtype=np.int64)
    if enc:
        np.cumsum([len(e) for e in enc], out=off[1:])
    blob = np.frombuffer(b''.join(enc), dtype=np.uint8) if off[-1] else np.zeros(0, dtype=np.uint8)
    return np.ascontiguousarray(blob), off


def _is_torch(x) -> bool:
    return type(x).__module__.startswith('torch')


def _addr(x):
    if x is None:
        return None
    if _is_torch(x):
        if not x.is_contiguous():
            raise ValueError('device tensors must be contiguous')
        return c_void_p(x.data_ptr())
    if not isinstance(x, np.ndarray) or not x.flags['C_CONTIGUOUS']:
        raise ValueError('host buffers must be C-contiguous numpy arrays')
    return c_void_p(x.ctypes.data)


_NP_OF_TORCH = {'torch.int16': np.int16, 'torch.uint16': np.uint16, 'torch.uint8': np.uint8, 'torch.int32': np.int32,
                'torch.uint32': np.uint32, 'torch.int64': np.int64}


def _want(x, name: str, dtypes, shape):
    """Raise ValueError unless `x` (numpy array or torch tensor) has one of `dtypes` and exactly `shape`
    (None entries match any extent).  The C side trusts the extents it is given and reads n*l*d elements from
    every pointer, so a short or mistyped buffer must stop here (ADVICE r1: out-of-bounds read on a short signature)."""
    if x is None:
        raise ValueError(f'{name} is required')
    if _is_torch(x):
        dt = _NP_OF_TORCH.get(str(x.dtype))
        shp = tuple(x.shape)
    elif isinstance(x, np.ndarray):
        dt, shp = x.dtype.type, x.shape
    else:
        raise ValueError(f'{name} must be a numpy array or a torch tensor, not {type(x).__name__}')
    if not isinstance(dtypes, tuple):
        dtypes = (dtypes,)
    if dt not in dtypes:
        raise ValueError(f'{name} must have dtype {" or ".join(np.dtype(d).name for d in dtypes)}, not {x.dtype}')
    if len(shp) != len(shape) or any(w is not None and int(g) != int(w) for g, w in zip(shp, shape)):
        raise ValueError(f'{name} must have shape {tuple("*" if w is None else int(w) for w in shape)}, not {tuple(shp)}')
    return x


def _lead(x, name: str, dtypes, last: int):
    """Like _want for arrays of shape (..., last); returns the number of rows."""
    shp = tuple(x.shape) if hasattr(x, 'shape') else ()
    if len(shp) < 1:
        raise ValueError(f'{name} must have shape (..., {last})')
    _want(x, name, dtypes, (None,) * (len(shp) - 1) + (last,))
    return int(np.prod(shp[:-1])) if len(shp) > 1 else 1


def make_scheme(sk_bd=1, sk_wt=1, ch_bd=1, ch_wt=1, ag_bd=1, ag_wt=1, wit_bd=1, wit_wt=1, sk_salt='SK_SALT',
                ch_salt='CH_SALT', ag_salt='AG_SALT', wit_salt='WIT_SALT') -> LcbScheme:
    s = LcbScheme()
    s.sk_bd, s.sk_wt, s.ch_bd, s.ch_wt = sk_bd, sk_wt, ch_bd, ch_wt
    s.ag_bd, s.ag_wt, s.wit_bd, s.wit_wt = ag_bd, ag_wt, wit_bd, wit_wt
    for name, val in (('sk_salt', sk_salt), ('ch_salt', ch_salt), ('ag_salt', ag_salt), ('wit_salt', wit_salt)):
        raw = val.encode()
        if len(raw) >= _ffi.LCB_SALT_MAX:
            raise ValueError(f'{name} longer than {_ffi.LCB_SALT_MAX - 1} bytes')
        setattr(s, name, raw)
    return s


def _locked(cls):
    """Serialise every public method of an Engine on its own re-entrant lock: one context = one stream, one key_ch
    row and one set of scratch buffers, and ctypes releases the GIL inside a call (include/lcb200.h: "a ctx is not
    re-entrant")."""
    for name, fn in list(vars(cls).items()):
        if callable(fn) and not name.startswith('_') and not isinstance(fn, (staticmethod, classmethod, property)):
            def wrap(f):
                @functools.wraps(f)
                def inner(self, *a, **k):
                    with self.lock:
                        return f(self, *a, **k)
                return inner
            setattr(cls, name, wrap(fn))
    return cls


@_locked
class Engine(object):
    """One GPU context: LatticeParameters (q, d, l) + secpar + the NTT-resident public row key_ch.
    Thread-safe at the granularity of one call (see `lock`); callers that must pair a particular key_ch with a call
    hold `lock` around ensure_key_ch() + the call (lattice_algebra.BoundEngine does)."""

    def __init__(self, secpar: int, modulus: int, degree: int, length: int, device: int = 0):
        self.lock = threading.RLock()
        self._key_ch_token = None
        self._lib = _ffi.load()
        self._ctx = c_void_p()
        st = self._lib.lcb_ctx_create(byref(self._ctx), device, secpar, modulus, degree, length)
        if st != _ffi.LCB_OK:
            detail = self._lib.lcb_last_error(None).decode() or self._lib.lcb_strerror(st).decode()
            self._ctx = c_void_p()
            raise LcbError(st, detail)
        self.secpar, self.q, self.d, self.l, self.device = secpar, modulus, degree, length, device
        # element formats (include/lcb200.h): 16-bit for q < 2^16, 32-bit ("wide") otherwise; BKLM partial sums are
        # int32 / int64 accordingly
        self.wide = modulus >= 65536
        self.ct, self.nt, self.pt = (np.int32, np.uint32, np.int64) if self.wide else (np.int16, np.uint16, np.int32)

    # ------------------------------------------------------------------ plumbing
    def close(self):
        if getattr(self, '_ctx', None) is not None and self._ctx.value:
            self._lib.lcb_ctx_destroy(self._ctx)
            self._ctx = c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, st: int):
        if st != _ffi.LCB_OK:
            detail = self._lib.lcb_last_error(self._ctx).decode() or self._lib.lcb_strerror(st).decode()
            raise LcbError(st, f'{self._lib.lcb_strerror(st).decode()} ({detail})')

    def _out(self, shape, dtype, device: bool):
        if device:
            import torch
            tdt = {np.int16: torch.int16, np.uint16: torch.uint16, np.uint8: torch.uint8, np.int32: torch.int32,
                   np.uint32: torch.uint32, np.int64: torch.int64}[dtype]
            return torch.empty(shape, dtype=tdt, device=f'cuda:{self.device}')
        return np.empty(shape, dtype=dtype)

    def use_torch_stream(self):
        """Run on torch's current CUDA stream (so torch.cuda.Event timing sees the kernels)."""
        import torch
        self._ck(self._lib.lcb_ctx_set_stream(self._ctx, c_void_p(torch.cuda.current_stream(self.device).cuda_stream)))

    def synchronize(self):
        self._ck(self._lib.lcb_synchronize(self._ctx))

    @property
    def root_of_unity(self) -> int:
        return self._lib.lcb_ctx_root_of_unity(self._ctx)

    @property
    def launch_count(self) -> int:
        return self._lib.lcb_launch_count(self._ctx)

    def profile(self, on: bool = True):
        self._ck(self._lib.lcb_profile_enable(self._ctx, 1 if on else 0))

    def profile_reset(self):
        self._ck(self._lib.lcb_profile_reset(self._ctx))

    def profile_read(self, kernel: str):
        """-> (total milliseconds, launches) of one kernel since the last reset (CUDA events)."""
        import ctypes
        ms, n = ctypes.c_double(0), ctypes.c_int64(0)
        self._ck(self._lib.lcb_profile_read(self._ctx, kernel.encode(), byref(ms), byref(n)))
        return ms.value, n.value

    @staticmethod
    def _rag(items):
        if isinstance(items, tuple) and len(items) == 2:
            blob, off = items       # already (blob, offsets); host or device
            _want(blob, 'ragged blob', np.uint8, (None,))
            _want(off, 'ragged offsets', np.int64, (None,))
            if int(off.shape[0]) < 1:
                raise ValueError('ragged offsets need n + 1 entries')
            if isinstance(off, np.ndarray) and (int(off[0]) != 0 or int(off[-1]) > int(blob.shape[0]) or
                                                (off.shape[0] > 1 and bool((np.diff(off) < 0).any()))):
                raise ValueError('ragged offsets must start at 0, ascend and end inside the blob')
            return items
        return ragged(items)

    @staticmethod
    def _count(off) -> int:
        return int(off.shape[0]) - 1

    # ------------------------------------------------------------------ K1 / K2
    def set_key_ch(self, key_ch_coef):
        _want(key_ch_coef, 'key_ch', self.ct, (self.l, self.d))
        self._key_ch_token = None
        self._ck(self._lib.lcb_set_key_ch(self._ctx, _addr(key_ch_coef)))
        if isinstance(key_ch_coef, np.ndarray):
            self._key_ch_token = hashlib.blake2b(key_ch_coef.tobytes(), digest_size=16).digest()

    def ensure_key_ch(self, key_ch_coef: np.ndarray):
        """Upload `key_ch_coef` unless it already is this context's resident public row."""
        if self._key_ch_token != hashlib.blake2b(np.ascontiguousarray(key_ch_coef).tobytes(), digest_size=16).digest():
            self.set_key_ch(np.ascontiguousarray(key_ch_coef))

    def shake256(self, items, out_len: int, device: bool = False):
        blob, off = self._rag(items)
        n = self._count(off)
        out = self._out((n, out_len), np.uint8, device)
        self._ck(self._lib.lcb_shake256_batch(self._ctx, _addr(blob), _addr(off), n, _addr(out), out_len))
        return out

    def expand_seeds(self, secret32: bytes, n: int, first: int = 0, device: bool = False):
        """n seed bitstrings (uint8[n, secpar], ASCII '0'/'1') from ONE 32-byte secret: seed i = first secpar bits of
        SHAKE256(secret32 || le64(first + i)) (include/lcb200.h, lcb_expand_seeds).  -> (blob, offsets) as keygen takes."""
        if not isinstance(secret32, (bytes, bytearray)) or len(secret32) != 32:
            raise ValueError('secret32 must be 32 bytes')
        sec = np.frombuffer(bytes(secret32), dtype=np.uint8).copy()
        out = self._out((n, self.secpar), np.uint8, device)
        self._ck(self._lib.lcb_expand_seeds(self._ctx, _addr(sec), first, n, _addr(out)))
        sec[:] = 0
        if device:
            import torch
            off = torch.arange(n + 1, dtype=torch.int64, device=out.device) * self.secpar
            return out.view(-1), off
        return out.reshape(-1), np.arange(n + 1, dtype=np.int64) * self.secpar

    def hash2polyvec(self, salt: str, msgs, bd: int, wt: int, vec_len: int, want_dense: bool = True,
                     want_pairs: bool = False, device: bool = False):
        blob, off = self._rag(msgs)
        n = self._count(off)
        dense = self._out((n, vec_len, self.d), self.ct, device) if want_dense else None
        pairs = self._out((n, vec_len, wt, 2), self.ct, device) if want_pairs else None
        self._ck(self._lib.lcb_hash2polyvec_batch(self._ctx, salt.encode(), _addr(blob), _addr(off), n, bd, wt,
                                                  vec_len, _addr(dense), _addr(pairs)))
        return dense, pairs

    # ------------------------------------------------------------------ K3 / K4 / K6
    def ntt_fwd(self, coef, device: bool = False):
        npoly = _lead(coef, 'coef', self.ct, self.d)
        out = self._out(tuple(coef.shape), self.nt, device)
        self._ck(self._lib.lcb_ntt_fwd_batch(self._ctx, _addr(coef), npoly, _addr(out)))
        return out

    def ntt_inv(self, ntt, device: bool = False):
        npoly = _lead(ntt, 'ntt', self.nt, self.d)
        out = self._out(tuple(ntt.shape), self.ct, device)
        self._ck(self._lib.lcb_ntt_inv_batch(self._ctx, _addr(ntt), npoly, _addr(out)))
        return out

    def ntt_reference_repr(self, coef, device: bool = False):
        """lattice_algebra's Polynomial.ntt_representation: int16[..., 2d], rep[k] = a(rou^k), centred."""
        npoly = _lead(coef, 'coef', self.ct, self.d)
        out = self._out(tuple(coef.shape[:-1]) + (2 * self.d,), self.ct, device)
        self._ck(self._lib.lcb_ntt_reference_repr_batch(self._ctx, _addr(coef), npoly, _addr(out)))
        return out

    def poly_mul(self, a, b, device: bool = False):
        npoly = _lead(a, 'a', self.ct, self.d)
        _want(b, 'b', self.ct, tuple(a.shape))
        out = self._out(tuple(a.shape), self.ct, device)
        self._ck(self._lib.lcb_poly_mul_batch(self._ctx, _addr(a), _addr(b), npoly, _addr(out)))
        return out

    # ------------------------------------------------------------------ LM one-time signatures
    def lm_keygen(self, sch: LcbScheme, seeds, want_sk_coef: bool = True, want_sk_ntt: bool = True,
                  want_vk_ntt: bool = True, want_vk_coef: bool = True, device: bool = False):
        blob, off = self._rag(seeds)
        n = self._count(off)
        sk_coef = self._out((n, 2, self.l, self.d), self.ct, device) if want_sk_coef else None
        sk_ntt = self._out((n, 2, self.l, self.d), self.nt, device) if want_sk_ntt else None
        vk_ntt = self._out((n, 2, self.d), self.nt, device) if want_vk_ntt else None
        vk_coef = self._out((n, 2, self.d), self.ct, device) if want_vk_coef else None
        self._ck(self._lib.lcb_lm_keygen_batch(self._ctx, byref(sch), _addr(blob), _addr(off), n, _addr(sk_coef),
                                               _addr(sk_ntt), _addr(vk_ntt), _addr(vk_coef)))
        return sk_coef, sk_ntt, vk_ntt, vk_coef

    def challenge(self, sch: LcbScheme, chmsgs, device: bool = False):
        blob, off = self._rag(chmsgs)
        n = self._count(off)
        pairs = self._out((n, sch.ch_wt, 2), self.ct, device)
        self._ck(self._lib.lcb_challenge_batch(self._ctx, byref(sch), _addr(blob), _addr(off), n, _addr(pairs)))
        return pairs

    def lm_sign(self, sch: LcbScheme, sk_ntt, chmsgs, device: bool = False):
        blob, off = self._rag(chmsgs)
        n = self._count(off)
        _want(sk_ntt, 'sk_ntt', self.nt, (n, 2, self.l, self.d))
        sig = self._out((n, self.l, self.d), self.ct, device)
        self._ck(self._lib.lcb_lm_sign_batch(self._ctx, byref(sch), _addr(sk_ntt), _addr(blob), _addr(off), n,
                                             _addr(sig)))
        return sig

    def lm_verify(self, sch: LcbScheme, vk_ntt, chmsgs, sig, bd: int, wt: int, st_ntt=None, device: bool = False,
                  out=None):
        blob, off = self._rag(chmsgs)
        n = self._count(off)
        _want(vk_ntt, 'vk_ntt', self.nt, (n, 2, self.d))
        _want(sig, 'sig', self.ct, (n, self.l, self.d))
        if st_ntt is not None:
            _want(st_ntt, 'st_ntt', self.nt, (n, self.d))
        verdict = _want(out, 'out', np.uint8, (n,)) if out is not None else self._out((n,), np.uint8, device)
        self._ck(self._lib.lcb_lm_verify_batch(self._ctx, byref(sch), _addr(vk_ntt), _addr(blob), _addr(off),
                                               _addr(sig), _addr(st_ntt), n, bd, wt, _addr(verdict)))
        return verdict

    # ------------------------------------------------------------------ packed wire format
    def pack(self, values, bits: int, bias: int, device: bool = False, want_range: bool = False):
        """values int16/uint16 [..., 256] -> uint8 [..., 32*bits] (include/lcb200.h, lcb_pack_batch)."""
        npoly = _lead(values, 'values', (np.int16, np.uint16), self.d)
        lead = tuple(values.shape[:-1])
        packed = self._out(lead + (self.d * bits // 8,), np.uint8, device)
        ok = self._out(lead, np.uint8, device) if want_range else None
        self._ck(self._lib.lcb_pack_batch(self._ctx, _addr(values), npoly, bits, bias, _addr(packed), _addr(ok)))
        return (packed, ok) if want_range else packed

    def unpack(self, packed, bits: int, bias: int, dtype=np.int16, device: bool = False):
        npoly = _lead(packed, 'packed', np.uint8, self.d * bits // 8)
        lead = tuple(packed.shape[:-1])
        out = self._out(lead + (self.d,), dtype, device)
        self._ck(self._lib.lcb_unpack_batch(self._ctx, _addr(packed), npoly, bits, bias, _addr(out)))
        return out

    def lm_verify_packed(self, sch: LcbScheme, vk_packed, vk_bits: int, chmsgs, sig_packed, sig_bits: int,
                         sig_bias: int, bd: int, wt: int, device: bool = False, out=None):
        blob, off = self._rag(chmsgs)
        n = self._count(off)
        _want(vk_packed, 'vk_packed', np.uint8, (n, 2, self.d * vk_bits // 8))
        _want(sig_packed, 'sig_packed', np.uint8, (n, self.l, self.d * sig_bits // 8))
        verdict = _want(out, 'out', np.uint8, (n,)) if out is not None else self._out((n,), np.uint8, device)
        self._ck(self._lib.lcb_lm_verify_packed_batch(self._ctx, byref(sch), _addr(vk_packed), vk_bits, _addr(blob),
                                                      _addr(off), _addr(sig_packed), sig_bits, sig_bias, n, bd, wt,
                                                      _addr(verdict)))
        return verdict

    def lm_sign_packed(self, sch: LcbScheme, sk_ntt, chmsgs, sig_bits: int, sig_bias: int, device: bool = False,
                       want_range: bool = False):
        """lm_sign straight into the wire format: -> uint8[n, l, 32*sig_bits] (and in_range uint8[n, l] when want_range),
        exactly pack(lm_sign(...), sig_bits, sig_bias)."""
        blob, off = self._rag(chmsgs)
        n = self._count(off)
        _want(sk_ntt, 'sk_ntt', self.nt, (n, 2, self.l, self.d))
        sig = self._out((n, self.l, self.d * sig_bits // 8), np.uint8, device)
        ok = self._out((n, self.l), np.uint8, device) if want_range else None
        self._ck(self._lib.lcb_lm_sign_packed_batch(self._ctx, byref(sch), _addr(sk_ntt), _addr(blob), _addr(off), n,
                                                    sig_bits, sig_bias, _addr(sig), _addr(ok)))
        return (sig, ok) if want_range else sig

    def lm_keygen_packed(self, sch: LcbScheme, seeds, sk_bits: int, sk_bias: int, vk_bits: int, want_sk: bool = True,
                         want_sk_range: bool = False, want_vk: bool = True, device: bool = False):
        """lm_keygen straight into the wire format: -> (sk_packed uint8[n, 2, l, 32*sk_bits] (coefficient form, bias sk_bias),
        sk_in_range uint8[n, 2, l], vk_packed uint8[n, 2, 32*vk_bits] (NTT form, bias 0)), each None unless wanted; exactly
        pack(sk_coef, sk_bits, sk_bias) and pack(vk_ntt, vk_bits, 0) of lm_keygen."""
        blob, off = self._rag(seeds)
        n = self._count(off)
        sk = self._out((n, 2, self.l, self.d * sk_bits // 8), np.uint8, device) if want_sk else None
        ok = self._out((n, 2, self.l), np.uint8, device) if want_sk and want_sk_range else None
        vk = self._out((n, 2, self.d * vk_bits // 8), np.uint8, device) if want_vk else None
        self._ck(self._lib.lcb_lm_keygen_packed_batch(self._ctx, byref(sch), _addr(blob), _addr(off), n, sk_bits, sk_bias,
                                                      _addr(sk), _addr(ok), vk_bits, _addr(vk)))
        return sk, ok, vk

    def lm_sign_packed_sk(self, sch: LcbScheme, sk_packed, sk_bits: int, sk_bias: int, chmsgs, sig_bits: int,
                          sig_bias: int, device: bool = False, want_range: bool = False):
        """lm_sign from packed coefficient-form signing keys uint8[n, 2, l, 32*sk_bits] into the wire format: -> uint8[n, l,
        32*sig_bits] (and in_range uint8[n, l] when want_range), exactly lm_sign_packed(ntt_fwd(unpack(sk_packed, sk_bits,
        sk_bias)), ...)."""
        blob, off = self._rag(chmsgs)
        n = self._count(off)
        _want(sk_packed, 'sk_packed', np.uint8, (n, 2, self.l, self.d * sk_bits // 8))
        sig = self._out((n, self.l, self.d * sig_bits // 8), np.uint8, device)
        ok = self._out((n, self.l), np.uint8, device) if want_range else None
        self._ck(self._lib.lcb_lm_sign_packed_sk_batch(self._ctx, byref(sch), _addr(sk_packed), sk_bits, sk_bias, _addr(blob),
                                                       _addr(off), n, sig_bits, sig_bias, _addr(sig), _addr(ok)))
        return (sig, ok) if want_range else sig

    def adaptor_verify_packed(self, sch: LcbScheme, vk_packed, vk_bits: int, chmsgs, sig_packed, sig_bits: int,
                              sig_bias: int, st_packed, st_bits: int, bd: int, wt: int, device: bool = False, out=None):
        """lm_verify(..., st_ntt=...) from packed keys uint8[n, 2, 32*vk_bits], signatures uint8[n, l, 32*sig_bits] and
        statements uint8[n, 32*st_bits] (bias 0)."""
        blob, off = self._rag(chmsgs)
        n = self._count(off)
        _want(vk_packed, 'vk_packed', np.uint8, (n, 2, self.d * vk_bits // 8))
        _want(sig_packed, 'sig_packed', np.uint8, (n, self.l, self.d * sig_bits // 8))
        _want(st_packed, 'st_packed', np.uint8, (n, self.d * st_bits // 8))
        verdict = _want(out, 'out', np.uint8, (n,)) if out is not None else self._out((n,), np.uint8, device)
        self._ck(self._lib.lcb_adaptor_verify_packed_batch(self._ctx, byref(sch), _addr(vk_packed), vk_bits, _addr(blob),
                                                           _addr(off), _addr(sig_packed), sig_bits, sig_bias,
                                                           _addr(st_packed), st_bits, n, bd, wt, _addr(verdict)))
        return verdict

    def adapt_packed(self, presig_packed, presig_bits: int, presig_bias: int, wit_coef, sig_bits: int, sig_bias: int,
                     device: bool = False, want_range: bool = False):
        """presig uint8[..., 32*presig_bits] + wit int16[..., 256] -> uint8[..., 32*sig_bits] (and in_range uint8[...]),
        exactly pack(vec_add(unpack(presig), wit))."""
        npoly = _lead(presig_packed, 'presig_packed', np.uint8, self.d * presig_bits // 8)
        lead = tuple(presig_packed.shape[:-1])
        _want(wit_coef, 'wit_coef', self.ct, lead + (self.d,))
        sig = self._out(lead + (self.d * sig_bits // 8,), np.uint8, device)
        ok = self._out(lead, np.uint8, device) if want_range else None
        self._ck(self._lib.lcb_adaptor_adapt_packed_batch(self._ctx, _addr(presig_packed), presig_bits, presig_bias,
                                                          _addr(wit_coef), npoly, sig_bits, sig_bias, _addr(sig), _addr(ok)))
        return (sig, ok) if want_range else sig

    def extract_packed(self, sig_packed, sig_bits: int, sig_bias: int, presig_packed, presig_bits: int, presig_bias: int,
                       device: bool = False):
        """-> int16[..., 256] = vec_sub(unpack(sig), unpack(presig))."""
        npoly = _lead(sig_packed, 'sig_packed', np.uint8, self.d * sig_bits // 8)
        lead = tuple(sig_packed.shape[:-1])
        _want(presig_packed, 'presig_packed', np.uint8, lead + (self.d * presig_bits // 8,))
        wit = self._out(lead + (self.d,), self.ct, device)
        self._ck(self._lib.lcb_adaptor_extract_packed_batch(self._ctx, _addr(sig_packed), sig_bits, sig_bias,
                                                            _addr(presig_packed), presig_bits, presig_bias, npoly,
                                                            _addr(wit)))
        return wit

    def adapt_packed_wit(self, presig_packed, presig_bits: int, presig_bias: int, wit_packed, wit_bits: int, wit_bias: int,
                         sig_bits: int, sig_bias: int, device: bool = False, want_range: bool = False):
        """presig uint8[..., 32*presig_bits] + packed wit uint8[..., 32*wit_bits] -> uint8[..., 32*sig_bits] (and in_range
        uint8[...]), exactly pack(vec_add(unpack(presig), unpack(wit)))."""
        npoly = _lead(presig_packed, 'presig_packed', np.uint8, self.d * presig_bits // 8)
        lead = tuple(presig_packed.shape[:-1])
        _want(wit_packed, 'wit_packed', np.uint8, lead + (self.d * wit_bits // 8,))
        sig = self._out(lead + (self.d * sig_bits // 8,), np.uint8, device)
        ok = self._out(lead, np.uint8, device) if want_range else None
        self._ck(self._lib.lcb_adaptor_adapt_packed_wit_batch(self._ctx, _addr(presig_packed), presig_bits, presig_bias,
                                                              _addr(wit_packed), wit_bits, wit_bias, npoly, sig_bits, sig_bias,
                                                              _addr(sig), _addr(ok)))
        return (sig, ok) if want_range else sig

    def extract_packed_wit(self, sig_packed, sig_bits: int, sig_bias: int, presig_packed, presig_bits: int,
                           presig_bias: int, wit_bits: int, wit_bias: int, device: bool = False, want_range: bool = False):
        """-> packed witnesses uint8[..., 32*wit_bits] (and in_range uint8[...]), exactly
        pack(vec_sub(unpack(sig), unpack(presig)), wit_bits, wit_bias)."""
        npoly = _lead(sig_packed, 'sig_packed', np.uint8, self.d * sig_bits // 8)
        lead = tuple(sig_packed.shape[:-1])
        _want(presig_packed, 'presig_packed', np.uint8, lead + (self.d * presig_bits // 8,))
        wit = self._out(lead + (self.d * wit_bits // 8,), np.uint8, device)
        ok = self._out(lead, np.uint8, device) if want_range else None
        self._ck(self._lib.lcb_adaptor_extract_packed_wit_batch(self._ctx, _addr(sig_packed), sig_bits, sig_bias,
                                                                _addr(presig_packed), presig_bits, presig_bias, npoly,
                                                                wit_bits, wit_bias, _addr(wit), _addr(ok)))
        return (wit, ok) if want_range else wit

    # ------------------------------------------------------------------ content-mode hash inputs
    _CONTENT_KINDS = {'vk': (_ffi.LCB_CONTENT_VK, 2), 'st': (_ffi.LCB_CONTENT_ST, 1)}

    def content_str(self, kind: str, packed, bits: int, device: bool = False):
        """Content-mode repr() of packed NTT-form keys (kind 'vk': uint8[n, 2, 32*bits]) or statements ('st': uint8[n,
        32*bits]), bias 0 -> uint8[n, 57] (include/lcb200.h, lcb_content_str_batch).  At bits = 16 a plain uint16 NTT array
        (uint16[n, 2, 256] / uint16[n, 256]) is accepted as it is."""
        if kind not in self._CONTENT_KINDS:
            raise ValueError(f"kind must be 'vk' or 'st', not {kind!r}")
        code, rows = self._CONTENT_KINDS[kind]
        if not isinstance(bits, int) or not 1 <= bits <= 16:
            raise ValueError(f'bits must be in 1..16, not {bits}')
        n = int(packed.shape[0]) if len(getattr(packed, 'shape', ())) else 0
        lead = (n, 2) if rows == 2 else (n,)
        if bits == 16 and (packed.dtype == np.uint16 or str(packed.dtype) == 'torch.uint16'):
            _want(packed, 'packed', np.uint16, lead + (self.d,))
        else:
            _want(packed, 'packed', np.uint8, lead + (self.d * bits // 8,))
        out = self._out((n, 57), np.uint8, device)
        self._ck(self._lib.lcb_content_str_batch(self._ctx, code, _addr(packed), bits, n, _addr(out)))
        return out

    def challenge_inputs(self, vk_str, msgs, st_str=None, device: bool = False):
        """Challenge messages [st_str_i + ', '] + vk_str_i + ', ' + msg_i from 57-byte content strings uint8[n, 57] and
        ragged messages -> (blob uint8[total], offsets int64[n+1]), the chmsgs form every sign / verify call takes."""
        mblob, moff = self._rag(msgs)
        n = self._count(moff)
        _want(vk_str, 'vk_str', np.uint8, (n, 57))
        if st_str is not None:
            _want(st_str, 'st_str', np.uint8, (n, 57))
        total = int(moff[-1]) - int(moff[0]) + n * (118 if st_str is not None else 59)
        out = self._out((total,), np.uint8, device)
        out_off = self._out((n + 1,), np.int64, device)
        self._ck(self._lib.lcb_challenge_inputs_batch(self._ctx, _addr(st_str), _addr(vk_str), _addr(mblob), _addr(moff), n,
                                                      _addr(out), _addr(out_off)))
        return out, out_off

    def aggregation_inputs(self, agg_off, vk_str_sorted, msgs_sorted, device: bool = False):
        """BKLM aggregation messages '[' + ', '.join("(" + vk_str + ", '" + msg + "')") + ']' of many groups (sorted items
        agg_off[g] .. agg_off[g+1]) -> (blob uint8[total], offsets int64[n_agg+1])."""
        mblob, moff = self._rag(msgs_sorted)
        total = self._count(moff)
        _want(vk_str_sorted, 'vk_str_sorted', np.uint8, (total, 57))
        n_agg = self._groups(agg_off, total)
        ha = agg_off.cpu().numpy() if _is_torch(agg_off) else agg_off
        hm = moff.cpu().numpy() if _is_torch(moff) else moff
        counts = np.diff(ha)
        size = int((2 + 63 * counts + (hm[ha[1:]] - hm[ha[:-1]]) + 2 * np.maximum(counts - 1, 0)).sum()) if n_agg else 0
        out = self._out((size,), np.uint8, device)
        out_off = self._out((n_agg + 1,), np.int64, device)
        self._ck(self._lib.lcb_aggregation_inputs_batch(self._ctx, _addr(agg_off), n_agg, _addr(vk_str_sorted), _addr(mblob),
                                                        _addr(moff), _addr(out), _addr(out_off)))
        return out, out_off

    # ------------------------------------------------------------------ sorted order of content-mode batches
    def content_order(self, agg_off, rows, device: bool = False):
        """-> int64[total]: at agg_off[g] .. agg_off[g+1] the items of group g sorted by their 57-byte rows uint8[total, 57]
        (unsigned byte order, equal rows in ascending index; include/lcb200.h, lcb_content_order_batch)."""
        total = int(rows.shape[0]) if len(getattr(rows, 'shape', ())) else 0
        _want(rows, 'rows', np.uint8, (total, 57))
        n_agg = self._groups(agg_off, total)
        order = self._out((total,), np.int64, device)
        self._ck(self._lib.lcb_content_order_batch(self._ctx, _addr(agg_off), n_agg, _addr(rows), _addr(order)))
        return order

    def gather_rows(self, src, index, device: bool = False):
        """src[index] for a uint8 array with a leading item dimension: -> uint8[n, *src.shape[1:]]; an index outside
        [0, len(src)) gives an all-zero row (device indices; host ones are refused)."""
        shp = tuple(src.shape) if hasattr(src, 'shape') else ()
        if len(shp) < 1:
            raise ValueError('src must have a leading item dimension')
        _want(src, 'src', np.uint8, shp)
        _want(index, 'index', np.int64, (None,))
        n = int(index.shape[0])
        row = int(np.prod(shp[1:])) if len(shp) > 1 else 1
        out = self._out((n,) + shp[1:], np.uint8, device)
        if row == 0:
            return out
        self._ck(self._lib.lcb_gather_rows_batch(self._ctx, _addr(src), shp[0], row, _addr(index), n, _addr(out)))
        return out

    def gather_ragged(self, items, index, device: bool = False):
        """Items index[k] of ragged items (a list of byte strings or a (blob, offsets) pair) -> (blob, offsets int64[n+1]);
        an index outside [0, n_src) gives an empty item (device indices; host ones are refused)."""
        blob, off = self._rag(items)
        n_src = self._count(off)
        _want(index, 'index', np.int64, (None,))
        n = int(index.shape[0])
        if _is_torch(off) or _is_torch(index):          # size the output: the lengths of the valid indices, summed
            import torch
            o = off if _is_torch(off) else torch.from_numpy(np.ascontiguousarray(off))
            i = index if _is_torch(index) else torch.from_numpy(np.ascontiguousarray(index))
            i = i.to(o.device)
            lens = o[1:] - o[:-1]
            ok = (i >= 0) & (i < n_src)
            need = int((lens[i.clamp(0, max(n_src - 1, 0))] * ok).sum().item()) if n_src else 0
        else:
            lens = np.diff(off)
            ok = (index >= 0) & (index < n_src)
            need = int(lens[index[ok]].sum())
        out = self._out((need,), np.uint8, device)
        out_off = self._out((n + 1,), np.int64, device)
        self._ck(self._lib.lcb_gather_ragged_batch(self._ctx, _addr(blob), _addr(off), n_src, _addr(index), n, _addr(out),
                                                   need, _addr(out_off)))
        return out, out_off

    # ------------------------------------------------------------------ BKLM aggregation
    def agg_coefs(self, sch: LcbScheme, agmsg, first: int, count: int, device: bool = False):
        if isinstance(agmsg, (str, bytes, bytearray)):
            agmsg = np.frombuffer(agmsg.encode() if isinstance(agmsg, str) else bytes(agmsg), dtype=np.uint8)
        _want(agmsg, 'agmsg', np.uint8, (None,))
        pairs = self._out((count, sch.ag_wt, 2), self.ct, device)
        self._ck(self._lib.lcb_bklm_agg_coefs(self._ctx, byref(sch), _addr(agmsg), int(agmsg.shape[0]), first,
                                              count, _addr(pairs)))
        return pairs

    def aggregate_partial(self, sch: LcbScheme, sig_sorted, ag_pairs, device: bool = False):
        count = int(sig_sorted.shape[0])
        _want(sig_sorted, 'sig_sorted', self.ct, (count, self.l, self.d))
        _want(ag_pairs, 'ag_pairs', self.ct, (count, sch.ag_wt, 2))
        partial = self._out((self.l, self.d), self.pt, device)
        self._ck(self._lib.lcb_bklm_aggregate_partial(self._ctx, byref(sch), _addr(sig_sorted), _addr(ag_pairs),
                                                      None, 0, 0, count, _addr(partial)))
        return partial

    def aggregate_finish(self, partial_sum, device: bool = False):
        _want(partial_sum, 'partial_sum', self.pt, (self.l, self.d))
        out = self._out((self.l, self.d), self.ct, device)
        self._ck(self._lib.lcb_bklm_aggregate_finish(self._ctx, _addr(partial_sum), _addr(out)))
        return out

    def aggverify_partial(self, sch: LcbScheme, vk_ntt_sorted, chmsgs_sorted, ag_pairs, device: bool = False):
        blob, off = self._rag(chmsgs_sorted)
        count = self._count(off)
        _want(vk_ntt_sorted, 'vk_ntt_sorted', self.nt, (count, 2, self.d))
        _want(ag_pairs, 'ag_pairs', self.ct, (count, sch.ag_wt, 2))
        partial = self._out((self.d,), self.pt, device)
        self._ck(self._lib.lcb_bklm_aggverify_partial(self._ctx, byref(sch), _addr(vk_ntt_sorted), _addr(blob),
                                                      _addr(off), _addr(ag_pairs), None, 0, 0, count,
                                                      _addr(partial)))
        return partial

    def aggverify_finish(self, partial_sum, ag_sig, total: int, ag_cap: int, avf_bd: int, avf_wt: int) -> bool:
        _want(partial_sum, 'partial_sum', self.pt, (self.d,))
        _want(ag_sig, 'ag_sig', self.ct, (self.l, self.d))
        verdict = np.zeros(1, dtype=np.uint8)
        self._ck(self._lib.lcb_bklm_aggverify_finish(self._ctx, _addr(partial_sum), _addr(ag_sig), total, ag_cap,
                                                     avf_bd, avf_wt, _addr(verdict)))
        return bool(verdict[0])

    # many independent aggregates per call (include/lcb200.h, lcb_bklm_aggregate_batch): group g covers the sorted rows
    # agg_off[g] .. agg_off[g+1] and hashes agmsgs[g]
    @staticmethod
    def _groups(agg_off, total: int) -> int:
        _want(agg_off, 'agg_off', np.int64, (None,))
        if int(agg_off.shape[0]) < 1:
            raise ValueError('agg_off needs n_agg + 1 entries')
        if isinstance(agg_off, np.ndarray) and int(agg_off[-1]) != total:
            raise ValueError(f'agg_off must end at the number of sorted items ({total}), not {int(agg_off[-1])}')
        return int(agg_off.shape[0]) - 1

    def aggregate_batch(self, sch: LcbScheme, agg_off, sig_sorted, agmsgs, device: bool = False):
        """-> int16[n_agg, l, d]: aggregate g of the sorted signatures agg_off[g] .. agg_off[g+1] under agmsgs[g]."""
        total = int(sig_sorted.shape[0]) if hasattr(sig_sorted, 'shape') and len(sig_sorted.shape) else 0
        _want(sig_sorted, 'sig_sorted', self.ct, (total, self.l, self.d))
        n_agg = self._groups(agg_off, total)
        mblob, moff = self._rag(agmsgs)
        if self._count(moff) != n_agg:
            raise ValueError(f'{self._count(moff)} aggregation messages for {n_agg} aggregates')
        out = self._out((n_agg, self.l, self.d), self.ct, device)
        self._ck(self._lib.lcb_bklm_aggregate_batch(self._ctx, byref(sch), _addr(agg_off), n_agg, _addr(sig_sorted),
                                                    _addr(mblob), _addr(moff), _addr(out)))
        return out

    def aggregate_verify_batch(self, sch: LcbScheme, agg_off, vk_ntt_sorted, chmsgs_sorted, agmsgs, ag_sig, ag_cap: int,
                               avf_bd: int, avf_wt: int, device: bool = False):
        """-> uint8[n_agg]: verdict g = aggregate_verify of group g (0 for an empty group or one above ag_cap)."""
        cblob, coff = self._rag(chmsgs_sorted)
        total = self._count(coff)
        _want(vk_ntt_sorted, 'vk_ntt_sorted', self.nt, (total, 2, self.d))
        n_agg = self._groups(agg_off, total)
        _want(ag_sig, 'ag_sig', self.ct, (n_agg, self.l, self.d))
        mblob, moff = self._rag(agmsgs)
        if self._count(moff) != n_agg:
            raise ValueError(f'{self._count(moff)} aggregation messages for {n_agg} aggregates')
        verdict = self._out((n_agg,), np.uint8, device)
        self._ck(self._lib.lcb_bklm_aggregate_verify_batch(self._ctx, byref(sch), _addr(agg_off), n_agg, _addr(vk_ntt_sorted),
                                                           _addr(cblob), _addr(coff), _addr(mblob), _addr(moff),
                                                           _addr(ag_sig), ag_cap, avf_bd, avf_wt, _addr(verdict)))
        return verdict

    def aggregate_packed_batch(self, sch: LcbScheme, agg_off, sig_packed, sig_bits: int, sig_bias: int, agmsgs,
                               ag_bits: int, ag_bias: int, device: bool = False, want_range: bool = False):
        """aggregate_batch on the packed wire format: sig_packed uint8[total, l, 32*sig_bits] -> ag_packed
        uint8[n_agg, l, 32*ag_bits] (and in_range uint8[n_agg, l] when want_range), exactly pack(aggregate_batch(unpack))."""
        total = int(sig_packed.shape[0]) if hasattr(sig_packed, 'shape') and len(sig_packed.shape) else 0
        _want(sig_packed, 'sig_packed', np.uint8, (total, self.l, self.d * sig_bits // 8))
        n_agg = self._groups(agg_off, total)
        mblob, moff = self._rag(agmsgs)
        if self._count(moff) != n_agg:
            raise ValueError(f'{self._count(moff)} aggregation messages for {n_agg} aggregates')
        out = self._out((n_agg, self.l, self.d * ag_bits // 8), np.uint8, device)
        ok = self._out((n_agg, self.l), np.uint8, device) if want_range else None
        self._ck(self._lib.lcb_bklm_aggregate_packed_batch(self._ctx, byref(sch), _addr(agg_off), n_agg, _addr(sig_packed),
                                                           sig_bits, sig_bias, _addr(mblob), _addr(moff), ag_bits, ag_bias,
                                                           _addr(out), _addr(ok)))
        return (out, ok) if want_range else out

    def aggregate_verify_packed_batch(self, sch: LcbScheme, agg_off, vk_packed, vk_bits: int, chmsgs_sorted, agmsgs,
                                      ag_packed, ag_bits: int, ag_bias: int, ag_cap: int, avf_bd: int, avf_wt: int,
                                      device: bool = False):
        """aggregate_verify_batch from packed keys uint8[total, 2, 32*vk_bits] and aggregates uint8[n_agg, l, 32*ag_bits]."""
        cblob, coff = self._rag(chmsgs_sorted)
        total = self._count(coff)
        _want(vk_packed, 'vk_packed', np.uint8, (total, 2, self.d * vk_bits // 8))
        n_agg = self._groups(agg_off, total)
        _want(ag_packed, 'ag_packed', np.uint8, (n_agg, self.l, self.d * ag_bits // 8))
        mblob, moff = self._rag(agmsgs)
        if self._count(moff) != n_agg:
            raise ValueError(f'{self._count(moff)} aggregation messages for {n_agg} aggregates')
        verdict = self._out((n_agg,), np.uint8, device)
        self._ck(self._lib.lcb_bklm_aggregate_verify_packed_batch(
            self._ctx, byref(sch), _addr(agg_off), n_agg, _addr(vk_packed), vk_bits, _addr(cblob), _addr(coff), _addr(mblob),
            _addr(moff), _addr(ag_packed), ag_bits, ag_bias, ag_cap, avf_bd, avf_wt, _addr(verdict)))
        return verdict

    # ------------------------------------------------------------------ adaptor signatures
    def witgen(self, sch: LcbScheme, seeds, want_wit: bool = True, want_st_ntt: bool = True,
               want_st_coef: bool = True, device: bool = False):
        blob, off = self._rag(seeds)
        n = self._count(off)
        wit = self._out((n, self.l, self.d), self.ct, device) if want_wit else None
        st_ntt = self._out((n, self.d), self.nt, device) if want_st_ntt else None
        st_coef = self._out((n, self.d), self.ct, device) if want_st_coef else None
        self._ck(self._lib.lcb_adaptor_witgen_batch(self._ctx, byref(sch), _addr(blob), _addr(off), n, _addr(wit),
                                                    _addr(st_ntt), _addr(st_coef)))
        return wit, st_ntt, st_coef

    def witgen_packed(self, sch: LcbScheme, seeds, wit_bits: int, wit_bias: int, st_bits: int, want_wit: bool = True,
                      want_wit_range: bool = False, want_st: bool = True, device: bool = False):
        """witgen straight into the wire format: -> (wit_packed uint8[n, l, 32*wit_bits] (coefficient form, bias wit_bias),
        wit_in_range uint8[n, l], st_packed uint8[n, 32*st_bits] (NTT form, bias 0)), each None unless wanted; exactly
        pack(wit, wit_bits, wit_bias) and pack(st_ntt, st_bits, 0) of witgen."""
        blob, off = self._rag(seeds)
        n = self._count(off)
        wit = self._out((n, self.l, self.d * wit_bits // 8), np.uint8, device) if want_wit else None
        ok = self._out((n, self.l), np.uint8, device) if want_wit and want_wit_range else None
        st = self._out((n, self.d * st_bits // 8), np.uint8, device) if want_st else None
        self._ck(self._lib.lcb_adaptor_witgen_packed_batch(self._ctx, byref(sch), _addr(blob), _addr(off), n, wit_bits,
                                                           wit_bias, _addr(wit), _addr(ok), st_bits, _addr(st)))
        return wit, ok, st

    def vec_add(self, a, b, device: bool = False):
        npoly = _lead(a, 'a', self.ct, self.d)
        _want(b, 'b', self.ct, tuple(a.shape))
        out = self._out(tuple(a.shape), self.ct, device)
        self._ck(self._lib.lcb_vec_add_batch(self._ctx, _addr(a), _addr(b), npoly, _addr(out)))
        return out

    def vec_sub(self, a, b, device: bool = False):
        npoly = _lead(a, 'a', self.ct, self.d)
        _want(b, 'b', self.ct, tuple(a.shape))
        out = self._out(tuple(a.shape), self.ct, device)
        self._ck(self._lib.lcb_vec_sub_batch(self._ctx, _addr(a), _addr(b), npoly, _addr(out)))
        return out

    def witness_verify(self, wit_coef, st_ntt, bd: int, wt: int, device: bool = False):
        n = int(wit_coef.shape[0])
        _want(wit_coef, 'wit_coef', self.ct, (n, self.l, self.d))
        _want(st_ntt, 'st_ntt', self.nt, (n, self.d))
        verdict = self._out((n,), np.uint8, device)
        self._ck(self._lib.lcb_adaptor_witness_verify_batch(self._ctx, _addr(wit_coef), _addr(st_ntt), n, bd, wt,
                                                            _addr(verdict)))
        return verdict

    def witness_verify_packed(self, wit_packed, wit_bits: int, wit_bias: int, st_packed, st_bits: int, bd: int, wt: int,
                              device: bool = False):
        """witness_verify from packed witnesses uint8[n, l, 32*wit_bits] and statements uint8[n, 32*st_bits] (bias 0):
        exactly witness_verify(unpack(wit), unpack(st))."""
        n = int(wit_packed.shape[0]) if len(getattr(wit_packed, 'shape', ())) else 0
        _want(wit_packed, 'wit_packed', np.uint8, (n, self.l, self.d * wit_bits // 8))
        _want(st_packed, 'st_packed', np.uint8, (n, self.d * st_bits // 8))
        verdict = self._out((n,), np.uint8, device)
        self._ck(self._lib.lcb_adaptor_witness_verify_packed_batch(self._ctx, _addr(wit_packed), wit_bits, wit_bias,
                                                                   _addr(st_packed), st_bits, n, bd, wt, _addr(verdict)))
        return verdict


class MultiEngine(object):
    """Single-process multi-GPU face of the C ABI (lcb_mctx_*, include/lcb200.h): host-resident batches are sharded
    over `devices` inside ONE call; BKLM partial sums are reduced on the devices.  One process per GPU with
    torch.distributed (lattice_cryptography_b200.distributed) is the other way to use several GPUs."""

    def __init__(self, secpar: int, modulus: int, degree: int, length: int, devices: Sequence[int]):
        import ctypes
        self._lib = _ffi.load()
        self._m = c_void_p()
        arr = (ctypes.c_int * len(devices))(*devices)
        st = self._lib.lcb_mctx_create(byref(self._m), arr, len(devices), secpar, modulus, degree, length)
        if st != _ffi.LCB_OK:
            detail = self._lib.lcb_last_error(None).decode() or self._lib.lcb_strerror(st).decode()
            self._m = c_void_p()
            raise LcbError(st, detail)
        self.secpar, self.q, self.d, self.l, self.devices = secpar, modulus, degree, length, list(devices)
        self.wide = modulus >= 65536
        self.ct, self.nt = (np.int32, np.uint32) if self.wide else (np.int16, np.uint16)

    def close(self):
        if getattr(self, '_m', None) is not None and self._m.value:
            self._lib.lcb_mctx_destroy(self._m)
            self._m = c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _ck(self, st: int):
        if st != _ffi.LCB_OK:
            raise LcbError(st, f'{self._lib.lcb_strerror(st).decode()} ({self._lib.lcb_mctx_last_error(self._m).decode()})')

    @property
    def launch_count(self) -> int:
        return sum(self._lib.lcb_launch_count(self._lib.lcb_mctx_ctx(self._m, i)) for i in range(len(self.devices)))

    def set_key_ch(self, key_ch_coef):
        _want(key_ch_coef, 'key_ch', self.ct, (self.l, self.d))
        self._ck(self._lib.lcb_mctx_set_key_ch(self._m, _addr(key_ch_coef)))

    def lm_keygen(self, sch: LcbScheme, seeds, want_sk_coef: bool = True, want_sk_ntt: bool = True):
        blob, off = Engine._rag(seeds)
        n = Engine._count(off)
        sk_coef = np.empty((n, 2, self.l, self.d), self.ct) if want_sk_coef else None
        sk_ntt = np.empty((n, 2, self.l, self.d), self.nt) if want_sk_ntt else None
        vk_ntt, vk_coef = np.empty((n, 2, self.d), self.nt), np.empty((n, 2, self.d), self.ct)
        self._ck(self._lib.lcb_mctx_lm_keygen_batch(self._m, byref(sch), _addr(blob), _addr(off), n, _addr(sk_coef),
                                                    _addr(sk_ntt), _addr(vk_ntt), _addr(vk_coef)))
        return sk_coef, sk_ntt, vk_ntt, vk_coef

    def lm_sign(self, sch: LcbScheme, sk_ntt, chmsgs):
        blob, off = Engine._rag(chmsgs)
        n = Engine._count(off)
        _want(sk_ntt, 'sk_ntt', self.nt, (n, 2, self.l, self.d))
        sig = np.empty((n, self.l, self.d), self.ct)
        self._ck(self._lib.lcb_mctx_lm_sign_batch(self._m, byref(sch), _addr(sk_ntt), _addr(blob), _addr(off), n, _addr(sig)))
        return sig

    def lm_verify(self, sch: LcbScheme, vk_ntt, chmsgs, sig, bd: int, wt: int, st_ntt=None, out=None):
        blob, off = Engine._rag(chmsgs)
        n = Engine._count(off)
        _want(vk_ntt, 'vk_ntt', self.nt, (n, 2, self.d))
        _want(sig, 'sig', self.ct, (n, self.l, self.d))
        if st_ntt is not None:
            _want(st_ntt, 'st_ntt', self.nt, (n, self.d))
        verdict = _want(out, 'out', np.uint8, (n,)) if out is not None else np.empty(n, np.uint8)
        self._ck(self._lib.lcb_mctx_lm_verify_batch(self._m, byref(sch), _addr(vk_ntt), _addr(blob), _addr(off), _addr(sig),
                                                    _addr(st_ntt), n, bd, wt, _addr(verdict)))
        return verdict

    def lm_verify_packed(self, sch: LcbScheme, vk_packed, vk_bits: int, chmsgs, sig_packed, sig_bits: int, sig_bias: int,
                         bd: int, wt: int, out=None):
        blob, off = Engine._rag(chmsgs)
        n = Engine._count(off)
        _want(vk_packed, 'vk_packed', np.uint8, (n, 2, self.d * vk_bits // 8))
        _want(sig_packed, 'sig_packed', np.uint8, (n, self.l, self.d * sig_bits // 8))
        verdict = _want(out, 'out', np.uint8, (n,)) if out is not None else np.empty(n, np.uint8)
        self._ck(self._lib.lcb_mctx_lm_verify_packed_batch(self._m, byref(sch), _addr(vk_packed), vk_bits, _addr(blob), _addr(off),
                                                           _addr(sig_packed), sig_bits, sig_bias, n, bd, wt, _addr(verdict)))
        return verdict

    @staticmethod
    def _msg(agmsg):
        if isinstance(agmsg, (str, bytes, bytearray)):
            agmsg = np.frombuffer(agmsg.encode() if isinstance(agmsg, str) else bytes(agmsg), dtype=np.uint8)
        return _want(agmsg, 'agmsg', np.uint8, (None,))

    def bklm_aggregate(self, sch: LcbScheme, sig_sorted, agmsg):
        agmsg = self._msg(agmsg)
        n = int(sig_sorted.shape[0])
        _want(sig_sorted, 'sig_sorted', self.ct, (n, self.l, self.d))
        out = np.empty((self.l, self.d), self.ct)
        self._ck(self._lib.lcb_mctx_bklm_aggregate(self._m, byref(sch), _addr(sig_sorted), _addr(agmsg), int(agmsg.shape[0]), n,
                                                   _addr(out)))
        return out

    def bklm_aggregate_verify(self, sch: LcbScheme, vk_ntt_sorted, chmsgs_sorted, agmsg, ag_sig, ag_cap: int, avf_bd: int,
                              avf_wt: int) -> bool:
        agmsg = self._msg(agmsg)
        blob, off = Engine._rag(chmsgs_sorted)
        n = Engine._count(off)
        _want(vk_ntt_sorted, 'vk_ntt_sorted', self.nt, (n, 2, self.d))
        _want(ag_sig, 'ag_sig', self.ct, (self.l, self.d))
        verdict = np.zeros(1, dtype=np.uint8)
        self._ck(self._lib.lcb_mctx_bklm_aggregate_verify(self._m, byref(sch), _addr(vk_ntt_sorted), _addr(blob), _addr(off),
                                                          _addr(agmsg), int(agmsg.shape[0]), n, _addr(ag_sig), ag_cap, avf_bd,
                                                          avf_wt, _addr(verdict)))
        return bool(verdict[0])
