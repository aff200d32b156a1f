"""Reference helpers of the many-LUT tests: sample extraction at any monomial (glwe_sample_extraction.rs:91-147 with t != 0)."""
import numpy as np


def extraction_step(p, F):
    total = p.msg_mod * p.carry_mod
    return (total // F) * (p.poly_size // total)


def mask_from_row0(p, row0):
    """the k mask polynomials of the GLWE that an extraction at monomial 0 came from: A_r[0] = w[rN], A_r[j] = -w[rN + N - j]"""
    N, k = p.poly_size, p.glwe_dim
    w = row0[:k * N].reshape(k, N)
    A = np.empty_like(w)
    A[:, 0] = w[:, 0]
    A[:, 1:] = np.uint64(0) - w[:, :0:-1]
    return A


def extract_mask_at(A, t):
    """mask words of the extraction at monomial t: word q of polynomial r = A_r[t - q] for q <= t, -A_r[N + t - q] otherwise"""
    k, N = A.shape
    q = np.arange(N)
    src = (t - q) % N
    out = A[:, src].copy()
    neg = q > t
    out[:, neg] = np.uint64(0) - out[:, neg]
    return out.ravel()


# ---- exact blind rotation returning the whole GLWE ------------------------------------------------------------------------------------
# The oracle's exact PBS (orc_pbs_exact_steps) extracts monomial 0 only.  This restates the same integer rotation in numpy, vectorised over
# ciphertexts, and keeps every coefficient, so that extraction at any monomial can be taken from the exact GLWE.  The polynomial products
# iterate over the key's nonzero coefficients (sparse lattice keys); tests/test_many_lut.py checks monomial 0 against orc_pbs_exact_batch.

_U64 = np.uint64


def _ms(x, lg_n):
    """orc_modulus_switch: round(x * 2N / 2^64), mod 2N"""
    return (((x >> _U64(64 - lg_n - 2)) + _U64(1)) >> _U64(1)).astype(np.int64) % (2 << lg_n)


def _rot_rows(a, deg, N):
    """a * X^deg per row (negacyclic), a: (R, ..., N), deg: (R,) in [0, 2N)"""
    j = np.arange(N)
    src = (j[None, :] - deg[:, None]) % (2 * N)
    shape = (a.shape[0],) + (1,) * (a.ndim - 2) + (N,)
    idx = np.broadcast_to((src % N).reshape(shape), a.shape)
    out = np.take_along_axis(a, idx, axis=-1)
    neg = np.broadcast_to((src >= N).reshape(shape), a.shape)
    return np.where(neg, _U64(0) - out, out)


def _rot_const(d, b):
    """d * X^b for one b in [0, N) (negacyclic), d: (R, N)"""
    r = np.roll(d, b, axis=-1)
    r[:, :b] = _U64(0) - r[:, :b]
    return r


def _sparse(poly):
    nz = np.flatnonzero(poly)
    return [(int(b), poly[b]) for b in nz]


def _ext_prod(p, ggsw_sparse, glwe):
    """orc_add_external_product_exact over rows: returns ggsw (x) glwe, glwe (R, k1, N)"""
    B, L = p.pbs_base_log, p.pbs_level
    k1, N = p.glwe_dim + 1, p.poly_size
    shift = 64 - B * L
    state = ((((glwe >> _U64(shift - 1)) + _U64(1)) & ~_U64(1)) << _U64(shift - 1)) >> _U64(shift)   # closest_representable >> shift
    mask = _U64((1 << B) - 1)
    out = np.zeros_like(glwe)
    for lv in range(L, 0, -1):
        res = state & mask
        state = state >> _U64(B)
        carry = (((res - _U64(1)) | state) & res) >> _U64(B - 1)
        state = state + carry
        digits = res - (carry << _U64(B))
        for row in range(k1):
            d = digits[:, row]
            for col in range(k1):
                for b, c in ggsw_sparse[((lv - 1) * k1 + row) * k1 + col]:
                    out[:, col] += _rot_const(d, b) * c
    return out


def exact_glwe_batch(p, bsk, small, luts, lut_idx, max_steps=None):
    """the exact GLWE after the blind rotation of every row of `small` (classic and multi-bit), (R, k + 1, N); max_steps as for
    orc_pbs_exact_steps"""
    N, k1, n, L = p.poly_size, p.glwe_dim + 1, p.lwe_dim, p.pbs_level
    lg = N.bit_length() - 1
    gl = L * k1 * k1 * N
    bsk = np.asarray(bsk, dtype=np.uint64).reshape(-1, N)
    small = np.asarray(small, dtype=np.uint64)
    R = small.shape[0]
    acc = np.asarray(luts, dtype=np.uint64).reshape(-1, k1, N)[np.asarray(lut_idx, dtype=np.int64)]
    b_hat = _ms(small[:, n], lg)
    ct0 = _rot_rows(acc, (2 * N - b_hat) % (2 * N), N)
    polys = gl // N
    with np.errstate(over="ignore"):
        if not p.grouping_factor:
            for i in range(n if max_steps is None else min(n, max_steps)):
                live = small[:, i] != 0
                if not live.any():
                    continue
                a = _ms(small[:, i], lg)
                ct1 = _rot_rows(ct0, a, N) - ct0
                ct1[~live] = 0
                key = [_sparse(bsk[i * polys + q]) for q in range(polys)]
                ct0 = ct0 + _ext_prod(p, key, ct1)
        else:
            g = p.grouping_factor
            per = 1 << g
            for grp in range(n // g if max_steps is None else min(n // g, max_steps)):
                dst = np.zeros_like(ct0)
                for j in range(per):
                    key = [_sparse(bsk[(grp * per + j) * polys + q]) for q in range(polys)]
                    part = _ext_prod(p, key, ct0)
                    if j == 0:
                        dst += part
                        continue
                    deg = np.zeros(R, dtype=np.uint64)
                    for mi in range(g):
                        if (j >> (g - 1 - mi)) & 1:
                            deg += small[:, grp * g + mi]
                    dst += _rot_rows(part, _ms(deg, lg), N)
                ct0 = dst
    return ct0


def extract_at(glwe, t):
    """the LWE extracted at monomial t from each row's GLWE (R, k + 1, N): mask as extract_mask_at, body B[t]"""
    return np.stack([np.concatenate([extract_mask_at(g[:-1], t), g[-1, t:t + 1]]) for g in glwe])
