"""The limb reduction of k_verify_tc (ring.cu, tc_limbs_reduce), checked on the host for every modulus it can meet.

A converter thread of k_verify_tc turns the biased halves hi = a_hi + 32768, lo = a_lo + 32768 of two int16 coefficients
into u = reduce(hi * z + lo + kz) with kz = -(32768 + 32768 z) mod q, for z = zeta and z = q - zeta (the two square roots
of -1 mod q), and splits u into two u8 limbs.  u must be congruent to a_lo + z a_hi mod q and below 2^16, or a limb loses a
bit.  reduce is the device Barrett step x + umulhi(x, floor((2^32 - 1) / q)) * (-q) mod 2^32, followed by one conditional
subtraction of q when q > 32768.  Here the same 32-bit arithmetic runs in numpy over every (hi, lo) pair, for every NTT
prime q < 2^16 (q = 1 mod 512) and both roots.

Exhaustive in the default run: x = hi z + lo + kz covers exactly the interval [kz, 65535 z + 65535 + kz], because z < 65536
makes the lo ranges of consecutive hi overlap.  On it the Barrett quotient t(x) = (x * barrett) >> 32 never decreases, and
where t is constant the result rises by one per step of x.  So the largest result of each run of equal t is at the run's
last x, ceil((t + 1) 2^32 / barrett) - 1.  Checking those ends, about 65536 values per modulus, bounds every pair.  A literal
sweep over (hi, lo) in chunks of hi cross-checks that argument: by default it covers the lowest and highest hi at the
moduli either side of 32768 and the largest modulus.  LCB_FULL_LIMB_SWEEP=1 sweeps all 2^32 pairs of every modulus, which
takes hours."""
import os

import numpy as np
import pytest

M32 = (1 << 32) - 1


def _ntt_primes():
    return [q for q in range(513, 65536, 512) if all(q % f for f in range(2, int(q ** 0.5) + 1))]


def _roots(q):
    """Both square roots of -1 mod q: psi^128 and q - psi^128, psi the least primitive 512-th root of unity."""
    psi = next(g for g in range(2, q) if pow(g, 256, q) == q - 1)
    z = pow(psi, 128, q)
    assert z * z % q == q - 1
    return [z, q - z]


def _kz(q, z):
    """launch_verify's offset: -(32768 + 32768 z) mod q, so that hi z + lo + kz = a_lo + z a_hi (mod q)."""
    b15 = 32768 % q
    return (2 * q - b15 - b15 * z % q) % q


def _device_reduce(x, q, lazy=None):
    """tc_limbs_reduce on uint64 arrays holding 32-bit values, in the device's 32-bit arithmetic.  lazy defaults to
    launch_verify's choice, q <= 32768."""
    barrett = np.uint64(M32 // q)
    t = (x * barrett) >> np.uint64(32)
    r = (x + t * np.uint64((1 << 32) - q)) & np.uint64(M32)
    if not (q <= 32768 if lazy is None else lazy):
        r = np.where(r >= np.uint64(q), r - np.uint64(q), r)
    return r


def _check(x, q):
    u = _device_reduce(x, q)
    bad = (u >= np.uint64(1 << 16)) | (u % np.uint64(q) != x % np.uint64(q))
    assert not bad.any(), f'q={q}: x={int(x[bad][0])} -> u={int(u[bad][0])}'
    return int(u.max())


def _run_end_inputs(q, z):
    """The last input of every run of equal Barrett quotient over the limb inputs of (q, z), and the first input."""
    kz = _kz(q, z)
    x0, x1 = kz, 65535 * z + 65535 + kz
    assert x1 <= M32                      # the sum never wraps: 65535 (q - 1) + 65535 + q - 1 < 2^32
    barrett = M32 // q
    t = np.arange((x0 * barrett) >> 32, ((x1 * barrett) >> 32) + 1, dtype=np.uint64)
    ends = ((t + np.uint64(1)) * np.uint64(1 << 32) + np.uint64(barrett - 1)) // np.uint64(barrett) - np.uint64(1)
    ends = np.minimum(ends, np.uint64(x1))
    ends = ends[ends >= np.uint64(x0)]
    # the end of run t really is the last x with quotient t: its successor has a larger quotient
    assert (((ends * np.uint64(barrett)) >> np.uint64(32)) == t[-len(ends):]).all()
    nxt = ends[:-1] + np.uint64(1)
    assert (((nxt * np.uint64(barrett)) >> np.uint64(32)) > t[-len(ends):-1]).all()
    return np.concatenate([ends, np.array([x0], np.uint64)])


def _run_ends(q, z):
    return _check(_run_end_inputs(q, z), q)


def _sweep(q, z, his, chunk=64):
    """Every (hi, lo) pair for hi in his, chunk hi values at a time."""
    kz = np.uint64(_kz(q, z))
    lo = np.arange(65536, dtype=np.uint64)
    top = 0
    for a in range(0, len(his), chunk):
        hi = np.asarray(his[a:a + chunk], np.uint64)
        x = (hi[:, None] * np.uint64(z) + lo[None, :] + kz).reshape(-1)
        top = max(top, _check(x, q))
    return top


def test_every_ntt_prime_is_24():
    ps = _ntt_primes()
    assert len(ps) == 24 and ps[0] == 7681 and ps[-1] == 64513
    assert max(p for p in ps if p <= 32768) == 32257 and min(p for p in ps if p > 32768) == 36353


@pytest.mark.parametrize('q', _ntt_primes())
def test_limbs_below_2_16_for_every_pair(q):
    for z in _roots(q):
        top = _run_ends(q, z)
        # barrett_lazy lands in [0, 2q): the quotient estimate is short by at most one for every 32-bit x
        assert top < (2 * q if q <= 32768 else q)


def test_moduli_where_the_lazy_form_drops_a_bit():
    """Without the subtraction, u reaches 2^16 at exactly these moduli (each at some (hi, lo) pair); the lazy form is
    exact below 45569.  tests/test_gpu_verify_tc_extremes.py sends such pairs through k_verify_tc at 45569, 51713 and
    64513, so a kernel that chose the lazy form there rejects valid signatures in those cases."""
    need = [q for q in _ntt_primes()
            if max(int(_device_reduce(_run_end_inputs(q, z), q, lazy=True).max()) for z in _roots(q)) >= 1 << 16]
    assert need == [45569, 51713, 59393, 61441, 64513]


@pytest.mark.parametrize('q', [32257, 36353, 64513])
def test_literal_sweep_agrees_at_the_ends_of_the_range(q):
    his = list(range(256)) + list(range(65536 - 256, 65536))
    for z in _roots(q):
        assert _sweep(q, z, his) < 1 << 16


@pytest.mark.skipif(os.environ.get('LCB_FULL_LIMB_SWEEP') != '1', reason='hours of CPU: set LCB_FULL_LIMB_SWEEP=1')
@pytest.mark.parametrize('q', _ntt_primes())
def test_literal_sweep_of_every_pair(q):
    for z in _roots(q):
        assert _sweep(q, z, range(65536)) == _run_ends(q, z)
