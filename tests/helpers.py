"""Shared helpers for the parity tests (oracle side)."""
import ctypes as C

import numpy as np


def oracle_partial_pbs(orc, sk, lwe_small, lut, n_iters, log2_q=64):
    """bootstrap.rs:254-316 restated with the oracle primitives, stopping after n_iters mask elements;
    returns the sample-extracted LWE (same shape as a full PBS output)."""
    L = orc.lib()
    p = sk.p
    N, k1 = p.poly_size, p.glwe_dim + 1
    lg = int(N).bit_length() - 1
    b_hat = L.orc_modulus_switch(int(lwe_small[p.lwe_dim]), lg)
    acc = np.zeros(k1 * N, dtype=np.uint64)
    for q in range(k1):
        tmp = np.zeros(N, dtype=np.uint64)
        L.orc_monomial_div(tmp, np.ascontiguousarray(lut[q * N:(q + 1) * N]), N, b_hat)
        acc[q * N:(q + 1) * N] = tmp
    for i in range(n_iters):
        if int(lwe_small[i]) == 0:
            continue
        a_hat = L.orc_modulus_switch(int(lwe_small[i]), lg)
        ct1 = np.zeros_like(acc)
        for q in range(k1):
            tmp = np.zeros(N, dtype=np.uint64)
            L.orc_monomial_mul_and_subtract(tmp, np.ascontiguousarray(acc[q * N:(q + 1) * N]), N, a_hat)
            ct1[q * N:(q + 1) * N] = tmp
        L.orc_add_external_product_f64(C.byref(p), sk.fourier, i, acc, ct1)
    if log2_q < 64:   # bootstrap.rs:318-330: SignedDecomposer(log2_q, 1).closest_representable on every coefficient, then extract
        shift = np.uint64(64 - log2_q - 1)
        acc = (((acc >> shift) + np.uint64(1)) & ~np.uint64(1)) << shift
    out = np.zeros(p.big_dim + 1, dtype=np.uint64)
    L.orc_sample_extract0(C.byref(p), np.ascontiguousarray(acc), out)
    return out


def engine_params(orc_params):
    return dict(lwe_dim=orc_params.lwe_dim, glwe_dim=orc_params.glwe_dim, poly_size=orc_params.poly_size,
                pbs_base_log=orc_params.pbs_base_log, pbs_level=orc_params.pbs_level,
                ks_base_log=orc_params.ks_base_log, ks_level=orc_params.ks_level,
                grouping_factor=orc_params.grouping_factor, msg_mod=orc_params.msg_mod, carry_mod=orc_params.carry_mod)


def phase_error(ck, cts, expected_values):
    """|decrypted phase - expected plaintext| in u64 torus units, per ciphertext."""
    errs = []
    for ct, v in zip(cts, expected_values):
        ph = ck.decrypt_raw(ct)
        d = (ph - (int(v) << 59)) % 2**64
        errs.append(min(d, 2**64 - d))
    return np.array(errs, dtype=np.float64)


def simulate_program_clear(ir, inputs_clear, total_mod):
    """Noise-free execution of a recorded program on PLAINTEXT values: a slot holds its value modulo 2 * total_mod (message space plus
    the padding bit), leveled instructions are exact, a PBS is the table lookup the blind rotation performs -- f(x) below the padding
    bit, -f(x - total_mod) above it (negacyclic LUT, shortint/server_key/mod.rs:763-781).  Any operand that reaches the padding bit is
    reported: returns (outputs, n_padding_hits).  Used for programs far too large for the CPU oracle's real PBS."""
    M = 2 * total_mod
    delta = (1 << 63) // total_mod
    val = np.zeros(ir.n_slots, dtype=np.int64)
    val[: ir.n_inputs] = np.asarray(inputs_clear, dtype=np.int64)
    hits = 0
    for lv in range(len(ir.level_lin_off) - 1):
        for li in range(int(ir.level_lin_off[lv]), int(ir.level_lin_off[lv + 1])):
            out, tb, te = (int(v) for v in ir.lin[li])
            body = int(ir.lin_body[li])
            assert body % delta == 0, "plaintext bodies are multiples of delta"
            acc = body // delta
            for t in range(tb, te):
                acc += int(ir.term_coef[t]) * int(val[ir.term_slot[t]])
            val[out] = acc % M
        for j in range(int(ir.level_pbs_off[lv]), int(ir.level_pbs_off[lv + 1])):
            src, dst, lut = (int(v) for v in ir.pbs[j])
            x = int(val[src])
            if x >= total_mod:
                hits += 1
                val[dst] = (-int(ir.lut_tables[lut][x - total_mod])) % M
            else:
                val[dst] = int(ir.lut_tables[lut][x])
    return val[ir.outputs], hits


def string_blocks_clear(s: bytes):
    """4 little-endian 2-bit blocks per char"""
    return [(ch >> (2 * b)) & 3 for ch in s for b in range(4)]


# ---- lattice-valued test keys (DESIGN section 4): every value a multiple of 2^s, s = 64 - pbs_base_log * pbs_level ----------------------
# A BSK of small integers c * 2^s (not an encryption: the test only needs the algebra) and LUTs on the same lattice keep every accumulator
# coefficient on the lattice after every step: digits are integers, digit * c * 2^s lands on it again.  The FFT error of a correct kernel
# stays far below 2^(s-1), so rounding the kernel's output to the lattice must give the exact integer PBS word for word, after all n steps.

def lattice_shift(p):
    return 64 - p.pbs_base_log * p.pbs_level


def pbs_steps(p):
    """blind-rotation steps of a full PBS: mask elements (classic) or groups (multi-bit)"""
    return p.lwe_dim // p.grouping_factor if p.grouping_factor else p.lwe_dim


def lattice_bsk(orc, p, seed, nnz=8, cmax=127):
    """standard-domain (multi-bit) BSK of small multiples c * 2^s, 0 < |c| <= cmax, at nnz random positions per polynomial (nnz=None: every
    coefficient drawn from [-cmax, cmax])"""
    N, s = p.poly_size, lattice_shift(p)
    n_polys = lib_bsk_len(orc, p) // N
    rng = np.random.default_rng(seed)
    if nnz is None:
        c = rng.integers(-cmax, cmax + 1, size=(n_polys, N))
        return (c * 2**s).astype(np.int64).view(np.uint64).ravel()
    bsk = np.zeros((n_polys, N), dtype=np.uint64)
    pos = rng.integers(0, N, size=(n_polys, nnz))
    c = rng.integers(1, cmax + 1, size=(n_polys, nnz)) * rng.choice([-1, 1], size=(n_polys, nnz))
    np.put_along_axis(bsk, pos, (c * 2**s).astype(np.int64).view(np.uint64), axis=1)
    return bsk.ravel()


def lib_bsk_len(orc, p):
    return int(orc.lib().orc_bsk_len(C.byref(p)))


def lattice_tie_words(p, rng, count):
    """words on the lattice whose signed decomposition meets a digit tie: 2^63 (top digit exactly 2^(B-1)) and, for two or more levels,
    words whose lowest-level digit is exactly 2^(B-1) with both parities of the next level (the tie rounds up or down by that parity)"""
    s, B = lattice_shift(p), p.pbs_base_log
    words = [np.full(count, 2**63, dtype=np.uint64)]
    if p.pbs_level >= 2:
        hi = rng.integers(0, 2**(64 - s - B), size=(2, count), dtype=np.uint64)
        for parity in (0, 1):
            nxt = (hi[parity] & ~np.uint64(1)) | np.uint64(parity)
            words.append((nxt << np.uint64(s + B)) | np.uint64(2**(B - 1) << s))
    w = np.concatenate(words)
    return w[rng.permutation(len(w))[:count]]


def lattice_luts(p, n_luts, seed):
    """n_luts accumulators, all k+1 polynomials random multiples of 2^s with about one coefficient in eight replaced by a tie word; LUT 0
    is zero apart from the tie words, so the first CMUX decomposes ties and zeros only"""
    s = lattice_shift(p)
    rng = np.random.default_rng(seed)
    luts = rng.integers(0, 2**(64 - s), size=(n_luts, p.lut_len), dtype=np.uint64) << np.uint64(s)
    luts[0] = 0
    at = rng.random(luts.shape) < 0.125
    luts[at] = lattice_tie_words(p, rng, int(at.sum()))
    return luts


def modulus_switch_ties(p, rng, size):
    """odd multiples of 2^(62 - log2 N): x * 2N / 2^64 is exactly half-way between two integers"""
    lg = int(p.poly_size).bit_length() - 1
    return ((2 * rng.integers(0, 2**(lg + 1), size=size, dtype=np.uint64) + np.uint64(1)) << np.uint64(62 - lg)).astype(np.uint64)


def lattice_inputs(p, batch, seed):
    """small LWEs: random 64-bit words with a quarter replaced by edge words (0, 1, 2^64 - 1, 2^63 and modulus-switch ties); row 0 has an
    all-zero mask, row 1 a mask of ties only, row 2 the four fixed edge words in turn"""
    rng = np.random.default_rng(seed)
    n = p.lwe_dim
    x = rng.integers(0, 2**64, size=(batch, n + 1), dtype=np.uint64)
    fixed = np.array([0, 1, 2**64 - 1, 2**63], dtype=np.uint64)
    edge = np.where(rng.random(x.shape) < 0.5, fixed[rng.integers(0, 4, size=x.shape)], modulus_switch_ties(p, rng, x.shape))
    pick = rng.random(x.shape) < 0.25
    x[pick] = edge[pick]
    if batch > 0:
        x[0, :n] = 0
    if batch > 1:
        x[1] = modulus_switch_ties(p, rng, n + 1)
    if batch > 2:
        x[2, :n] = fixed[np.arange(n) % 4]
    return x


def round_to_lattice(x, s):
    half = np.uint64(1 << (s - 1))
    return ((x + half) >> np.uint64(s)) << np.uint64(s)


def max_residual(got, exact):
    """max |got - exact| in u64 torus units (signed difference)"""
    return int(np.abs((got - exact).view(np.int64)).max()) if got.size else 0


def exact_unique(orc, p, bsk, small, luts, idx, max_steps=None):
    """orc.pbs_exact_batch over the distinct (input, LUT index) rows only, expanded back to the batch"""
    key = np.concatenate([small, np.asarray(idx, dtype=np.uint64)[:, None]], axis=1)
    uniq, inv = np.unique(key, axis=0, return_inverse=True)
    out = orc.pbs_exact_batch(p, bsk, uniq[:, :-1], luts, uniq[:, -1].astype(np.uint32), max_steps=max_steps)
    return out[np.ravel(inv)]


def first_bad_step(run, ref, n_steps, s):
    """Bisect the blind rotation of one failing row: run(k) / ref(k) return that row's words after k steps (candidate, exact).  Returns
    (k, number of differing words after k steps), k the first step after which the candidate, rounded to 2^s, leaves the exact result."""
    def bad(k):
        return int((round_to_lattice(run(k), s) != ref(k)).sum())
    lo, hi = 0, n_steps          # invariant: bad(hi) > 0; lo = 0 is checked on its own (LUT rotation)
    if bad(0):
        return 0, bad(0)
    while hi - lo > 1:
        mid = (lo + hi) // 2
        if bad(mid):
            hi = mid
        else:
            lo = mid
    return hi, bad(hi)


def assert_on_lattice(got, exact, s, label, run_rows=None, ref_rows=None, n_steps=None, bound_log2=None):
    """(a) every row of got, rounded to 2^s, equals the exact PBS word for word; (b) max residual <= 2^bound_log2 (default s - 4).
    On a failure of (a), run_rows(k, rows) / ref_rows(k, rows) (outputs after k steps) name the first failing step of the first bad row.
    Returns the maximum residual."""
    bad_rows = np.flatnonzero((round_to_lattice(got, s) != exact).any(axis=1))
    if len(bad_rows):
        msg = f"{label}: {len(bad_rows)} of {len(got)} rows leave the exact PBS (first rows {bad_rows[:8].tolist()})"
        if run_rows is not None:
            r = int(bad_rows[0])
            k, words = first_bad_step(lambda k: run_rows(k, [r])[0], lambda k: ref_rows(k, [r])[0], n_steps, s)
            msg += f"; row {r} first differs after step {k} of {n_steps} ({words} words differ)"
        raise AssertionError(msg)
    res = max_residual(got, exact)
    bound = s - 4 if bound_log2 is None else bound_log2
    print(f"{label}: {len(got)} rows word for word after the full rotation, 0 mismatches; max residual 2^{np.log2(max(res, 1)):.1f} "
          f"(half lattice 2^{s - 1}, bound 2^{bound})")
    assert res <= 2**bound, f"{label}: residual 2^{np.log2(res):.1f} > 2^{bound}"
    return res
