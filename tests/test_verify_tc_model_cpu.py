"""CPU model of the tensor-core verify (ring.cu, k_verify_tc): the zeta stage on the CUDA cores, the two-limb u8 GEMM against
the per-context matrices B_0 / B_1 (k_verify_tc_matrix), and the recombination x = D_lo + 256 D_hi.  The model must give
the residues of the verify equation's left side, sum_k key_ch_k * s_k in Z_q[X]/(X^256 + 1), at all 256 NTT slots, bit
for bit, for the smallest, the shipped and the largest 16-bit moduli of the fast path, every int16 row (the witness-verify
and aggregate-verify callers accept all of them), key slots at q - 1, and l up to the largest the context accepts (64).
It also pins the int32 accumulator bound that makes the GEMM exact."""
import numpy as np
import pytest

D = 256


def is_prime(q):
    return q > 1 and all(q % f for f in range(2, int(q ** 0.5) + 1))


def moduli():
    fast = [q for q in range(D * 2 + 1, 1 << 16, 2 * D) if is_prime(q)]     # q = 1 mod 2d, q < 2^16: the fast path
    return [fast[0], 11777, 39937, fast[-1]]


def psi_of(q):
    """Least element of order 2d (api.cu, lcb_ctx_create)."""
    root = next(r for r in (pow(h, (q - 1) // (2 * D), q) for h in range(2, q)) if pow(r, D, q) == q - 1)
    return min(pow(root, k, q) for k in range(1, 2 * D, 2))


def bitrev8(p):
    return int(f'{p:08b}'[::-1], 2)


def slot_powers(q, psi):
    """V[P, j] = x_P^j with x_P = psi^(2 bitrev8(P) + 1): slot P of the NTT is the evaluation at x_P."""
    odd = np.array([2 * bitrev8(p) + 1 for p in range(D)], np.int64)
    pw = np.array([pow(psi, e, q) for e in range(2 * D)], np.int64)
    return pw[(odd[:, None] * np.arange(D, dtype=np.int64)[None, :]) % (2 * D)]


def matrices(key_hat, q, psi):
    """B_b [N = 256][K = 256 l], b = 0, 1, as k_verify_tc_matrix builds them: column n = (limb hl, slot p of block b),
    K = (poly k, A limb L, m); entry = byte hl of (256^L * key_hat[k][128 b + p] * x_(128 b + p)^m mod q)."""
    l = key_hat.shape[0]
    V = slot_powers(q, psi)
    out = []
    for b in range(2):
        P = np.arange(128) + 128 * b
        M = (key_hat[:, P][:, :, None] * V[P][None, :, :128]) % q           # [k][p][m]
        rows = []
        for hl in range(2):
            per_k = []
            for k in range(l):
                cols = [(M[k] * (256 ** L % q)) % q for L in range(2)]     # [p][m] each
                per_k.append(np.concatenate([(c >> (8 * hl)) & 255 for c in cols], axis=1))
            rows.append(np.concatenate(per_k, axis=1))                     # [p][K]
        out.append(np.concatenate(rows, axis=0))                           # [256][K]
    return out


def zeta_stage(sig, q, psi):
    """u^b_k[m] = a[m] +- zeta a[128 + m] in [0, q), from the biased halves (a + 32768) exactly as the converter warps
    form them: one multiply-add and one reduction per block and coefficient pair."""
    zeta = pow(psi, 128, q)
    lo = sig[..., :128].astype(np.int64) + 32768
    hi = sig[..., 128:].astype(np.int64) + 32768
    us = []
    for z in (zeta, q - zeta):
        k0 = (-32768 - z * 32768) % q
        x = lo + z * hi + k0
        assert x.max() < 1 << 32                                           # one 32-bit Barrett reduction
        us.append(x % q)
    return us                                                              # [rows][l][128] each


def model(sig, key_hat, q, psi):
    B = matrices(key_hat, q, psi)
    n, l = sig.shape[:2]
    x = np.zeros((n, D), np.int64)
    for b, u in enumerate(zeta_stage(sig, q, psi)):
        A = np.concatenate([np.concatenate([u[:, k] & 255, u[:, k] >> 8], axis=1) for k in range(l)], axis=1)
        assert A.max() <= 255 and B[b].max() <= 255
        Dm = A @ B[b].T                                                    # [rows][256]: (lo | hi) x 128 slots
        assert Dm.max() < 1 << 31                                          # exact in the int32 accumulators
        x[:, 128 * b:128 * (b + 1)] = Dm[:, :128] + 256 * Dm[:, 128:]
    return x


def negacyclic(a, b, q):
    full = np.convolve(a, b)
    return (full[:D] - np.concatenate([full[D:], [0]])) % q


@pytest.mark.parametrize('q', moduli())
@pytest.mark.parametrize('l', [1, 13, 23, 64])
def test_limb_gemm_equals_ring_product(q, l):
    rng = np.random.default_rng(q * 100 + l)
    psi = psi_of(q)
    V = slot_powers(q, psi)
    key = rng.integers(0, q, (l, D), dtype=np.int64)
    key_hat = (key @ V.T) % q
    rows = 3
    sig = rng.integers(-32768, 32768, (rows, l, D), dtype=np.int64)
    sig[0, :, :] = -32768
    sig[1, :, ::2] = 32767
    sig[1, :, 1::2] = -32768
    x = model(sig, key_hat, q, psi)
    for r in range(rows):
        prod = np.zeros(D, np.int64)
        for k in range(l):
            prod = (prod + negacyclic(key[k], sig[r, k] % q, q)) % q
        assert np.array_equal(x[r] % q, (prod @ V.T) % q)


@pytest.mark.parametrize('q', moduli())
def test_key_slots_at_q_minus_one(q):
    rng = np.random.default_rng(q)
    psi = psi_of(q)
    V = slot_powers(q, psi)
    l = 13
    key_hat = np.full((l, D), q - 1, np.int64)
    sig = rng.integers(-32768, 32768, (2, l, D), dtype=np.int64)
    sig[1] = 32767
    x = model(sig, key_hat, q, psi)
    want = ((key_hat[None] * ((sig % q) @ V.T % q)).sum(axis=1)) % q
    assert np.array_equal(x % q, want)


def test_accumulator_bound_at_the_worst_case():
    # every A and B byte at 255, K = 2 limbs x 128 coefficients x l: the largest l a context accepts is 64, and the
    # bound holds up to l = 128
    for l in (64, 128):
        assert 255 * 255 * 2 * 128 * l < 1 << 31
