"""The R1CS witness-map path, stage by stage, against exact references, at every NTT pass plan it runs.

  stage                  entry point                                 reference
  rows                   b2z_r1cs_eval (run_plan: products, row sums) cpu_oracle.constraint_evals, itself checked
                                                                     against Python integers on a tiny system
  coset evaluations      b2z_r1cs_coset_evals (eval_one, then         n coset_fft(ifft(rows)) from cpu_oracle.ntt:
                         witness_map_transform)                      the unscaled inverse is a permutation of the
                                                                     forward transform, so no multiplication
  whole-key proof        b2z_groth16_prove_partial_r1cs              the six sums of a key of known multiples
  uneven slices          b2z_pk_upload_slice + coset_evals,           per sum, the slices' partials add up to the
                         shard_begin / shard_finish (quotient with    whole key's value
                         natural_out = false, h slice from h_lo)
  tile-sharded prover    b2z_dist_prove (wm_dist_step1..4)            every rank returns the proof of the known
                                                                     multipliers

The systems are synthetic R1CS built straight from CSR arrays with exact (nc, l, m): empty rows, coefficient-one
copies, rows of 2..40 entries with coefficients 0, 2, r - 1, one, random and a coefficient whose Montgomery limb 0
equals one's (plan_matrix must not take it for one), repeated columns, columns 0 and m - 1, and one row of 2^16
entries per matrix.  The assignments are uniform, witness-like, all r - 1 (the largest lazy row sums) and zero.

Pass plans of make_plan (k0 = the low pass, t:k/logC = a high pass), asserted per case through the NTT-pass
launches of profile phase 0: 2 npass - 1 per coset evaluation, 3 npass - 1 per proof (per rank when sharded):

  log_n   single GPU                  sharded
   0      no pass (n = 1)
  10      10
  11      10, 10:1/9
  13      10, 10:3/7
  14                                  W = 8: 10, 7:4/6
  19      11, 11:8/3                  W = 2: 10, 9:9/1
  20                                  W = 4: 10, 8:10/0
  21      11, 11:10/1                 W = 8: 10, 7:6/4, 13:5/5   (three passes)
  22      11, 11:11/0
  23      11, 11:6/5, 17:6/5          W = 4: 11, 9:6/5, 15:6/5   (three passes)

The whole file, the 2^23 cases included, runs in about 100 s on one B200 (1000 W power limit), so none of it waits
for B2Z_SLOW_TESTS.
"""
import random

import numpy as np
import pytest

from oracle import bls12_381 as O
from helpers import (NAMES, R, KnownKey, add_point, c_point, check_partial, decode_partial, dist_prove_virtual_ranks,
                     ntt_pass_launches, point, scalar_mix)

gpu = pytest.mark.gpu
ZMIXES = ("uniform", "witness", "max", "zero")
X, Y = 0x1b2c3d4e5f60718293a4b5c6d7e8f90a1b2c3d4e5f6071829, 0x5a4b3c2d1e0f1a2b3c4d5e6f708192a3b4c5d6e7f8091a2b


@pytest.fixture(scope="module")
def codec(b2z):
    return b2z.codec


# ------------------------------------------------------------------------------- synthetic systems
ONE = 1                    # index of the coefficient one in the pool
NEAR_ONE = 4               # Montgomery limb 0 equal to one's, limb 1 different


def _coef_pool(codec, rs):
    """Montgomery coefficients: 0, 1, 2, r - 1, near-one, then 11 random values."""
    rand = [int(rs.randint(1, 1 << 30)) << 200 | int(rs.randint(1, 1 << 62)) for _ in range(11)]
    pool = codec.fr_to_mont_limbs([0, 1, 2, R - 1, 0] + rand)
    pool[NEAR_ONE] = pool[ONE]
    pool[NEAR_ONE, 1] ^= np.uint64(1 << 7)           # still below r: the top limb is one's
    assert pool[NEAR_ONE, 0] == pool[ONE, 0] and not np.array_equal(pool[NEAR_ONE], pool[ONE])
    return pool


def synth_csr(codec, nc, m, seed, big_row=True, empty=False):
    """One matrix of nc rows over m columns as (row_ptr uint64, cols uint32, coeffs (nnz, 4) Montgomery).  83 % of
    the rows hold one entry (70 % of those with coefficient one: the copy path), 14 % are empty, 3 % hold 2..40
    entries from the whole pool with their first column repeated; row 0 starts with the five special coefficients;
    one row holds 2^16 entries.  empty: nc rows without entries."""
    rs = np.random.RandomState(seed)
    pool = _coef_pool(codec, rs)
    if empty or nc == 0:
        return np.zeros(nc + 1, np.uint64), np.zeros(0, np.uint32), np.zeros((0, 4), np.uint64)
    u = rs.rand(nc)
    lens = np.where(u < 0.03, rs.randint(2, 41, size=nc), np.where(u < 0.17, 0, 1)).astype(np.int64)
    lens[0] = rs.randint(5, 41)
    if big_row:
        lens[rs.randint(nc)] = 1 << 16
    rp = np.zeros(nc + 1, np.uint64)
    np.cumsum(lens, out=rp[1:])
    nnz = int(rp[-1])
    cols = rs.randint(0, m, size=nnz).astype(np.uint32)
    idx = rs.randint(0, len(pool), size=nnz)
    single = np.repeat(lens == 1, lens)
    idx[single & (rs.rand(nnz) < 0.7)] = ONE
    starts = rp[:-1][lens >= 2].astype(np.int64)
    cols[starts + 1] = cols[starts]                   # a repeated column in every long row
    idx[:5] = np.arange(5)                            # 0, 1, 2, r - 1 and near-one in row 0
    hit = rs.randint(0, nnz, size=8)
    cols[hit[:4]], cols[hit[4:]] = 0, m - 1
    return rp, cols, np.ascontiguousarray(pool[idx])


class System:
    """A synthetic R1CS with exact (nc, l, m); `empty` names the matrices (0 A, 1 B, 2 C) without entries."""

    def __init__(self, codec, nc, l, m, seed, empty=(), big_row=True):
        self.codec, self.nc, self.l, self.m, self.seed = codec, nc, l, m, seed
        self.log_n = (nc + l - 1).bit_length()
        self.csr = tuple(synth_csr(codec, nc, m, seed + k, big_row, k in empty) for k in range(3))
        self._rows = (None, None)

    def matrices(self, b2z):
        """A fresh ConstraintMatrices (uploads belong to one context and are freed by the caller)."""
        return b2z.ConstraintMatrices(self.l, self.m - self.l, self.nc, *self.csr)

    def assignment(self, kind):
        """z as (canonical limbs, Montgomery limbs); z[0] = 1."""
        vals = scalar_mix(random.Random(self.seed * 7 + ZMIXES.index(kind)), self.m, kind)
        vals[0] = 1
        return self.codec.fr_to_bigint_limbs(vals), self.codec.fr_to_mont_limbs(vals)

    def rows(self, cpu_oracle, kind):
        """The oracle's a, b, c for assignment `kind` (the last one asked for is kept)."""
        if self._rows[0] != kind:
            zm = self.assignment(kind)[1]
            self._rows = (kind, cpu_oracle.constraint_evals(*self.csr, self.nc, self.l, zm))
        return self._rows[1]


# log_n -> (nc, l, m): nc + l a few short of 2^log_n, m small (the keys of known multiples hold m points per query).
# m = 5 < W = 8 at 2^14 (ranks without query points or z slice); 777, 1027, 2051 and 1029 are no multiple of W.
SIZES = {0: (0, 1, 3), 10: (1019, 3, 517), 11: (2043, 2, 1100), 13: (8185, 5, 2000), 14: ((1 << 14) - 4, 2, 5),
         19: ((1 << 19) - 9, 4, 777), 20: ((1 << 20) - 6, 3, 1027), 21: ((1 << 21) - 11, 6, 2051),
         22: ((1 << 22) - 5, 3, 999), 23: ((1 << 23) - 7, 4, 1029)}
# special shapes: name -> (nc, l, m, empty matrices)
SHAPES = {"B-empty": (1000, 3, 300, (1,)), "C-empty": (1000, 3, 300, (2,)), "all-empty": (1000, 3, 300, (0, 1, 2)),
          "nc-0": (0, 6, 40, ()), "m-eq-l": (500, 9, 9, ()), "l-gt-nc": (7, 60, 100, ()),
          "no-padding": ((1 << 12) - 5, 5, 300, ()), "near-half": ((1 << 11) + 1 - 5, 5, 300, ())}
SINGLE = (0, 10, 11, 13, 19, 21, 22, 23)
NPASS = {0: 0, 10: 1, 11: 2, 13: 2, 19: 2, 21: 2, 22: 2, 23: 3}
SHARDED = {(14, 8): 2, (19, 2): 2, (20, 4): 2, (21, 8): 3, (23, 4): 3}
_SYSTEMS, _KEYS = {}, {}


def _system(codec, case):
    if case not in _SYSTEMS:
        if case in SHAPES:
            nc, l, m, empty = SHAPES[case]
            _SYSTEMS[case] = System(codec, nc, l, m, 900 + 10 * list(SHAPES).index(case), empty)
        else:
            nc, l, m = SIZES[case]
            _SYSTEMS[case] = System(codec, nc, l, m, 100 + 10 * case)
            assert _SYSTEMS[case].log_n == case
    return _SYSTEMS[case]


def _key(b2z, ctx, S):
    """The key of known multiples of S's shape (one per log_n, shared by the tests of that size)."""
    if S.log_n not in _KEYS:
        _KEYS[S.log_n] = KnownKey(b2z, ctx, S.m, S.l, S.log_n, seed=7000 + S.log_n)
    return _KEYS[S.log_n]


def _prepare(key, S, cpu_oracle, kind="witness"):
    """Point the key's H sum at S's rows for assignment `kind`; returns (canonical z, Montgomery z)."""
    rows = S.rows(cpu_oracle, kind)
    if key.abc is not rows:
        key.abc, key.h_k = rows, None
    return S.assignment(kind)


def _profiled(ctx, fn):
    """fn() with the profiler on: (its result, the NTT-pass launches it made)."""
    ctx.check(ctx._lib.b2z_profile_enable(ctx.handle, 1))
    try:
        ntt_pass_launches(ctx)
        out = fn()
        return out, ntt_pass_launches(ctx)
    finally:
        ctx.check(ctx._lib.b2z_profile_enable(ctx.handle, 0))


def _coset_launches(npass):
    return 2 * npass - 1 if npass else 0


def _proof_launches(npass):
    return 3 * npass - 1 if npass else 0


# ------------------------------------------------------------------------------- 256-bit limb arithmetic (vectorised)
def _below(x, v):
    """x < v per row of an (n, 4) uint64 array."""
    lt, eq = np.zeros(x.shape[0], bool), np.ones(x.shape[0], bool)
    for i in (3, 2, 1, 0):
        vi = np.uint64((v >> (64 * i)) & ((1 << 64) - 1))
        lt |= eq & (x[:, i] < vi)
        eq &= x[:, i] == vi
    return lt


def _mod_r(x):
    """x mod r for rows below 2r."""
    out = x.copy()
    big = ~_below(x, R)
    borrow = np.zeros(x.shape[0], bool)
    for i in range(4):
        ri = np.uint64((R >> (64 * i)) & ((1 << 64) - 1))
        a = x[:, i]
        d = a - ri - borrow.astype(np.uint64)
        borrow = (a < ri) | ((a == ri) & borrow)
        out[big, i] = d[big]
    return out


# ------------------------------------------------------------------------------- CPU: the builder and the oracle
def test_synthetic_system_has_its_shape(b2z):
    codec = b2z.codec
    S = System(codec, 1 << 13, 5, 300, seed=1)
    assert (S.nc, S.l, S.m, S.log_n) == (1 << 13, 5, 300, 14)
    one = codec.fr_to_mont_limbs([1])[0]
    for rp, cols, cf in S.csr:
        lens = np.diff(rp.astype(np.int64))
        assert rp.shape == (S.nc + 1,) and cols.shape[0] == cf.shape[0] == int(rp[-1])
        assert (lens == 0).any() and (lens == 1).any() and (lens == 1 << 16).sum() == 1
        assert ((lens >= 2) & (lens <= 40)).sum() > 100
        assert 1.2 < (lens.sum() - (1 << 16)) / S.nc < 1.8
        assert cols.min() == 0 and cols.max() == S.m - 1
        is_one = (cf == one).all(axis=1)
        near = (cf[:, 0] == one[0]) & ~is_one
        assert near.any() and is_one[np.repeat(lens == 1, lens)].mean() > 0.6
        starts = rp[:-1][lens >= 2].astype(np.int64)
        assert (cols[starts] == cols[starts + 1]).all()
        vals = set(codec.fr_from_mont_limbs(np.unique(cf, axis=0)))
        assert {0, 1, 2, R - 1} <= vals
    empty = System(codec, 50, 2, 20, seed=2, empty=(1, 2))
    assert all(int(rp[-1]) == 0 and rp.shape == (51,) for rp, _, _ in empty.csr[1:]) and int(empty.csr[0][0][-1]) > 0


def test_oracle_rows_equal_python_integers(b2z, cpu_oracle):
    """The row reference itself, on a tiny system with every coefficient kind and the 2^16-entry row."""
    codec = b2z.codec
    S = System(codec, 12, 3, 10, seed=3)
    for kind in ZMIXES:
        zc, zm = S.assignment(kind)
        z = [int.from_bytes(r.tobytes(), "little") for r in zc]
        want = []
        for k, (rp, cols, cf) in enumerate(S.csr):
            c = codec.fr_from_mont_limbs(cf)
            row = [sum(c[e] * z[cols[e]] for e in range(int(rp[i]), int(rp[i + 1]))) % R for i in range(S.nc)]
            row += (z[:S.l] if k == 0 else [0] * S.l) + [0] * ((1 << S.log_n) - S.nc - S.l)
            want.append(codec.fr_to_mont_limbs(row))
        got = S.rows(cpu_oracle, kind)
        for k in range(3):
            assert np.array_equal(got[k], want[k]), "matrix %d, z = %s" % (k, kind)


# ------------------------------------------------------------------------------- rows
@gpu
@pytest.mark.parametrize("case", SINGLE + tuple(SHAPES))
def test_rows_equal_oracle(b2z, ctx, cpu_oracle, case):
    """b2z_r1cs_eval is canonical: limb for limb the oracle's rows, for every assignment mix."""
    S = _system(b2z.codec, case)
    if case in SIZES:
        assert S.log_n == case
    cm = S.matrices(b2z)
    try:
        def run():
            bad = []
            for kind in ZMIXES:
                got = b2z.LibsnarkReduction.constraint_evaluations_device(ctx, cm, S.assignment(kind)[1])
                want = S.rows(cpu_oracle, kind)
                bad += ["%s z=%s" % ("ABC"[k], kind) for k in range(3) if not np.array_equal(got[k], want[k])]
            return bad
        bad, launches = _profiled(ctx, run)
    finally:
        cm.free()
    assert launches == 0
    assert not bad, "%s (nc=%d l=%d m=%d): rows differ: %s" % (case, S.nc, S.l, S.m, ", ".join(bad))


# ------------------------------------------------------------------------------- coset evaluations
@gpu
@pytest.mark.parametrize("log_n", SINGLE)
def test_coset_evals_equal_unscaled_transforms(b2z, ctx, codec, cpu_oracle, log_n):
    """b2z_r1cs_coset_evals(which) = n coset_fft(ifft(rows[which])), lazily reduced: every element below 2r."""
    import torch
    S = _system(codec, log_n)
    kind = ZMIXES[SINGLE.index(log_n) % len(ZMIXES)]
    zm = S.assignment(kind)[1]
    n = 1 << log_n
    buf = torch.empty((n, 4), dtype=torch.int64, device="cuda")
    cm = S.matrices(b2z)
    try:
        def run():
            out = []
            for which in range(3):
                b2z.Groth16.coset_evals(ctx, cm, which, buf.data_ptr(), zm if which == 0 else None)
                out.append(buf.cpu().numpy().view(np.uint64).copy())
            return out
        got, launches = _profiled(ctx, run)
    finally:
        cm.free()
    assert cm.domain_size == n and launches == 3 * _coset_launches(NPASS[log_n])
    g = codec.fr_to_mont_limbs([7])
    for which, x in enumerate(S.rows(cpu_oracle, kind)):
        if n == 1:
            want = x
        else:
            unscaled_inv = cpu_oracle.ntt(x)[(n - np.arange(n)) % n]
            want = cpu_oracle.ntt(unscaled_inv, False, g)
        assert _below(got[which], 2 * R).all(), "%s: element not below 2r" % "ABC"[which]
        assert np.array_equal(_mod_r(got[which]), want), "%s z=%s: coset evaluations differ" % ("ABC"[which], kind)


# ------------------------------------------------------------------------------- whole-key proof from the matrices
@gpu
@pytest.mark.parametrize("log_n", SINGLE)
def test_whole_key_proof_from_matrices(b2z, ctx, cpu_oracle, log_n):
    S = _system(b2z.codec, log_n)
    key = _key(b2z, ctx, S)
    zc, zm = _prepare(key, S, cpu_oracle)
    pk = key.copy_pk(b2z).upload(ctx)
    cm = S.matrices(b2z)
    try:
        part, launches = _profiled(ctx, lambda: b2z.Groth16.create_proof_partial_with_matrices(ctx, pk, cm, zm, X, Y))
    finally:
        pk.free()
        cm.free()
    assert pk.domain_size == 1 << log_n and launches == _proof_launches(NPASS[log_n])
    wrong = check_partial(b2z, part, key.sums(cpu_oracle, zc, X, Y))
    assert not wrong, "2^%d: %s mismatch" % (log_n, "/".join(wrong))


# ------------------------------------------------------------------------------- uneven slices through the shard calls
@gpu
@pytest.mark.parametrize("log_n", [13, 23])
def test_uneven_slices_through_shard_calls(b2z, ctx, cpu_oracle, log_n):
    """Slices [1, 5, 2] of the key: per slice three coset_evals and shard_begin / shard_finish, in both orders, z
    with the first call.  Per sum the decoded partials add up to the whole key's value; combine agrees."""
    import torch
    G = b2z.Groth16
    S = _system(b2z.codec, log_n)
    key = _key(b2z, ctx, S)
    zc, zm = _prepare(key, S, cpu_oracle)
    want = key.sums(cpu_oracle, zc, X, Y)
    npass = NPASS[log_n]
    bufs = [torch.empty((1 << log_n, 4), dtype=torch.int64, device="cuda") for _ in range(3)]
    ptrs = [b.data_ptr() for b in bufs]
    cm = S.matrices(b2z)
    bad = []
    try:
        for order in ("evals-first", "begin-first"):
            total, parts = dict.fromkeys(NAMES), []
            for rank in range(3):
                pk = key.copy_pk(b2z).upload(ctx, rank=rank, world=3, weights=[1, 5, 2])

                def run():
                    if order == "evals-first":
                        for j in range(3):
                            G.coset_evals(ctx, cm, j, ptrs[j], zm if j == 0 else None)
                        keep = G.shard_begin(ctx, pk, cm, None, X, Y)
                    else:
                        keep = G.shard_begin(ctx, pk, cm, zm, X, Y)
                        for j in range(3):
                            G.coset_evals(ctx, cm, j, ptrs[j], None)
                    part = G.shard_finish(ctx, pk, *ptrs)
                    del keep
                    return part
                try:
                    part, launches = _profiled(ctx, run)
                finally:
                    pk.free()
                assert launches == 3 * _coset_launches(npass) + npass, (order, rank, launches)
                parts.append(part)
                got = decode_partial(b2z, part)
                for n in NAMES:
                    total[n] = add_point(n, total[n], got[n])
            assert G.combine(parts) == O.proof_serialize_compressed(total["A"], total["B"], c_point(total)), \
                "%s: partial-sum decoder disagrees with b2z_groth16_combine" % order
            bad += ["%s: %s" % (order, n) for n in NAMES if total[n] != point(n, want[n])]
    finally:
        cm.free()
    assert S.log_n == log_n and not bad, "2^%d slices [1, 5, 2]: %s mismatch" % (log_n, ", ".join(bad))


# ------------------------------------------------------------------------------- tile-sharded prover
def _proof_bytes(sums):
    C = (sums["sA"] + sums["rB1"] + sums["L"] + sums["H"]) % R
    return O.proof_serialize_compressed(point("A", sums["A"]), point("B", sums["B"]), point("C", C))


@gpu
@pytest.mark.parametrize("log_n,world", list(SHARDED))
def test_tile_sharded_prover_equals_known_multipliers(b2z, ctx, codec, cpu_oracle, log_n, world):
    """Two proofs in a row by `world` virtual ranks on the same handles: every rank returns the proof of the key's
    multipliers.  (14, 8) has m = 5 < W; the others have m no multiple of W."""
    S = _system(codec, log_n)
    key = _key(b2z, ctx, S)
    zc, zm = _prepare(key, S, cpu_oracle)
    want = [_proof_bytes(key.sums(cpu_oracle, zc, X + i, Y + i)) for i in range(2)]
    launches = [None] * world
    got = dist_prove_virtual_ranks(b2z, codec, S.matrices(b2z), key.pk, zm, X, Y, world, proofs=2,
                                   ntt_launches=launches)
    wrong = [rank for rank in range(world) if got[rank] != want]
    if wrong:
        pk, cm = key.copy_pk(b2z), S.matrices(b2z)
        try:
            single = b2z.Groth16.create_proof_with_matrices(ctx, pk, cm, zm, X, Y)
        finally:
            pk.free()
            cm.free()
        where = "the sharded path (the single-GPU proof is right)" if single == want[0] else \
            "the common path (the single-GPU proof is wrong too)"
        pytest.fail("2^%d over %d ranks: ranks %s differ; broken: %s" % (log_n, world, wrong, where))
    assert S.log_n == log_n and launches == [2 * _proof_launches(SHARDED[(log_n, world)])] * world, launches
