"""The prover's MSMs one sum at a time, in the mode the prover runs them, at every window size it can pick.

b2z_pk_upload builds every base set of a key with precomputed window copies (copy w = 2^(c w) P, one bucket set
shared by all windows, bit-plane sums finished by the host's Horner pass), while b2z_msm_g1 / _g2 always build
generic bases.  The keys here are made of known multiples: every query point and alpha, beta, delta is k G for a
multiplier k kept by the test (FixedBase on the GPU), so each of the six partial sums b2z_groth16_prove_partial
returns has an answer computed with Python integers:

  A   = (sum z_i a_i + alpha + r delta) G1          sA  = s A
  rB1 = r (sum z_i b_i + beta + s delta) G1          L   = (sum_{i>=l} z_i l_{i-l} - r s delta) G1
  H   = (sum_{j<n-1} h_j eta_j) G1                   B   = (sum z_i b'_i + beta_2 + s delta_2) G2

with h the CPU oracle's witness map of the (arbitrary) evaluation vectors; the last coefficient of h meets the
padded identity.  A failure names the sum that broke.  Every check also decodes the 1344 partial bytes
(A | sA | rB1 | L | H | B, XYZZ, lazily reduced Montgomery Fq, G2 as (c0, c1)) and checks the decoder against
b2z_groth16_combine.

Window sizes c reached (msm_pick_c; every test asserts its c with b2z_host_msm_window_bits):

  precomputed   a/b1/G2 set (m + 2 = 2^(c+1) + 3, the bottom of each range; 2^16 + 3 for c = 16)
                  c = 4 5 6 7 8 9 10 11 12 13 14 16 18 19 20        test_prover_sums_at_every_window_size
                L set (m - l + 1 = 2^(c+2), the top of each range)
                  c = 4 5 6 7 8 9 10 11 12 13 14 16 18 19
                H set (2^log_n)
                  c = 4 5 6 7 8 9 10 11 12 13 14 16 (2^19) 18 19 20 (2^23, three-pass NTT plan)
                adversarial keys, both accumulation kernels: c = 9, 14, 18 (sparse z: the colliding pairs
                  alone in their buckets; dense z: the collisions inside long runs)
                shards (block-cyclic over 3, uneven slices) of a c = 16 key
  generic       G1 c = 5 7 11 14, G2 c = 5 6 10 12 14, each at both ends of its range, with scalars that
                  reach the top window (c = 5 is the one generic size with an extra window)

The whole file, the m = 2^21 + 1 key with its 2^23 H set included, runs in about a minute on one B200 (1000 W power
limit), so none of it waits for B2Z_SLOW_TESTS.
"""
import random

import numpy as np
import pytest

from oracle import bls12_381 as O
from helpers import NAMES, R, KnownKey, add_point, c_point, check_partial, decode_partial, dot_mod_r, point, rand_k, scalar_mix

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def codec(b2z):
    return b2z.codec


# ------------------------------------------------------------------------------- window-size rules
def _digits(b2z, k, c):
    """The library's signed-window recoding of scalar k (for_each_digit, shared with the device): one digit per
    window, msm_windows(c) of them."""
    d = np.zeros(64, dtype=np.int32)
    k32 = np.frombuffer((k % R).to_bytes(32, "little"), dtype=np.uint32)
    w = b2z._ffi.lib().b2z_host_msm_digits(k32.ctypes.data, c, d.ctypes.data)
    return [int(x) for x in d[:w]]


def _windows(b2z, c):
    return len(_digits(b2z, 0, c))


def _c_of(b2z, n, precomputed):
    return int(b2z._ffi.lib().b2z_host_msm_window_bits(n, 1 if precomputed else 0))


def _assert_precomputed(b2z, m, l, log_n):
    """pk_upload builds precomputed copies when twice their size fits in the free device memory."""
    import torch
    cost = lambda n, pt: n * pt * _windows(b2z, _c_of(b2z, n, True)) if n else 0
    need = 2 * cost(m + 2, 96) + cost(m - l + 1, 96) + cost(m + 2, 192) + cost(1 << log_n, 96)
    free, _ = torch.cuda.mem_get_info()
    assert 2 * need < free, "key of %d bytes would not be precomputed (%d bytes free)" % (need, free)


# ------------------------------------------------------------------------------- scalars and exact sums
def _limb(v):
    return np.frombuffer((v % R).to_bytes(32, "little"), dtype=np.uint64)


def _int(row):
    return int.from_bytes(np.ascontiguousarray(row).tobytes(), "little")


def _boundary(rnd, cs, count):
    """Scalars built window by window from the digits where the signed recoding turns: 0, 1, nb - 1, nb, nb + 1 and
    2^c - 1 (nb = 2^(c-1)), for the window sizes `cs` in turn, up to the top window (bit 254 included), then reduced
    mod r (which leaves those below r, most of them, as they were built)."""
    out = []
    for i in range(count):
        c = cs[i % len(cs)]
        nb = 1 << (c - 1)
        digits = (0, 1, nb - 1, nb, nb + 1, (1 << c) - 1)
        v = 0
        for w in range(0, 255, c):
            v |= rnd.choice(digits) << w
        out.append((v & ((1 << 255) - 1)) % R)
    return out


def _z_mix(codec, kind, m, cs, seed):
    """z as (canonical limbs, Montgomery limbs).  Large assignments repeat 2^15 distinct values.  "sparse" is all zero
    here: the caller places its few non-zero scalars."""
    rnd = random.Random(seed)
    u = min(m, 1 << 15)
    vals = _boundary(rnd, cs, u) if kind == "boundary" else scalar_mix(rnd, u, "zero" if kind == "sparse" else kind)
    return (np.resize(codec.fr_to_bigint_limbs(vals), (m, 4)), np.resize(codec.fr_to_mont_limbs(vals), (m, 4)))


X, Y = 0x1b2c3d4e5f60718293a4b5c6d7e8f90a1b2c3d4e5f6071829, 0x5a4b3c2d1e0f1a2b3c4d5e6f708192a3b4c5d6e7f8091a2b
MIXES = (("uniform", 0, X), ("witness", X, 0), ("max", R - 1, R - 1), ("zero", X, Y), ("boundary", Y, X))


def _run_mixes(b2z, ctx, codec, cpu_oracle, key, cs, seed, mixes=MIXES, edit_z=None, label=""):
    """One partial proof per (scalar mix, r, s) on the uploaded key; returns the failures as readable strings."""
    bad = []
    for i, (kind, r, s) in enumerate(mixes):
        zc, zm = _z_mix(codec, kind, key.m, cs, seed + i)
        if edit_z is not None:
            edit_z(kind, zc, zm)
        part = key.prove(b2z, ctx, key.pk, zm, r, s)
        wrong = check_partial(b2z, part, key.sums(cpu_oracle, zc, r, s))
        if wrong:
            bad.append("%s z=%s r=%#x s=%#x: %s mismatch" % (label, kind, r, s, "/".join(wrong)))
    return bad


# ------------------------------------------------------------------------------- 3. the window-size sweep
PRE_C = (4, 5, 6, 7, 8, 9, 10, 11, 12, 13, 14, 16, 18, 19, 20)


def _sweep_cases():
    """(m, l, log_n, (c of the a/b1/G2 set, of the L set, of the H set)) per precomputed c: the a/b1/G2 set sits
    just past a power of two (bottom of c's range), the L set exactly on 2^(c'+2) for the previous c' (top of its
    range), the H set on 2^(c+2) (2^19 for c = 16, 2^23 for c = 20)."""
    out, prev = [], None
    for c in PRE_C:
        m = (1 << 16) + 1 if c == 16 else (1 << (c + 1)) + 1
        n_l = 1 << (prev + 2) if prev else m - 1
        log_n = {16: 19, 20: 23}.get(c, c + 2)
        out.append(pytest.param(m, m + 1 - n_l, log_n, (c, prev or 4, c), id="c%d-L%d-H%d" % (c, prev or 4, c)))
        prev = c
    return out


@pytest.mark.parametrize("m,l,log_n,want_c", _sweep_cases())
def test_prover_sums_at_every_window_size(b2z, ctx, codec, cpu_oracle, m, l, log_n, want_c):
    got_c = (_c_of(b2z, m + 2, True), _c_of(b2z, m - l + 1, True), _c_of(b2z, 1 << log_n, True))
    assert got_c == want_c, "msm_pick_c moved: this case no longer covers the window sizes it was chosen for"
    _assert_precomputed(b2z, m, l, log_n)
    key = KnownKey(b2z, ctx, m, l, log_n, seed=1000 + want_c[0])
    key.pk.upload(ctx)
    try:
        bad = _run_mixes(b2z, ctx, codec, cpu_oracle, key, want_c[:2], seed=want_c[0] * 10, label="c=%s" % (want_c,))
    finally:
        key.pk.free()
    assert not bad, bad


# ------------------------------------------------------------------------------- 4. adversarial keys
AFFINE = dict(B2Z_AFFINE_MIN_SEG="0", B2Z_AFFINE_G2="1", B2Z_ACCUM_MAX_SEGS="257")
XYZZ = dict(B2Z_AFFINE_MIN_SEG="4000000000")
ADV_M = {9: 2000, 14: 60000, 18: (1 << 20) - 100}


class _Adversary:
    """Identity points in every query; repeated (k_j = k_i) and negated (k_j = -k_i) bases with z_j = z_i; and
    shifted twins k_j = +-2^(c d) k_i with z_j = z_i >> (c d): copy w + d of P_i and copy w of P_j are the same point
    (or its negation) and meet in one bucket of the shared set.  All indices are witness variables, so the L set
    (same c) sees the same collisions."""

    def __init__(self, b2z, c, m, l):
        self.b2z, self.c, self.l = b2z, c, l
        self.W = W = _windows(b2z, c)
        self.identity = [l, l + 1, m - 1]
        self.same = [(l + 2, l + 3, 1), (l + 4, m - 2, -1), (l + 5, l + 6, -1)]
        self.twins = []
        for t, d in enumerate((1, 2, W - 2)):
            self.twins.append((l + 10 + 2 * t, l + 11 + 2 * t, d, 1))
            self.twins.append((l + 20 + 2 * t, m - 10 - t, d, -1))

    def edit_key(self, key):
        k = key.k
        for q in ("a", "b1", "b2", "l"):
            off = self.l if q == "l" else 0
            for i in self.identity:
                k[q][i - off] = 0
            for i, j, sign in self.same:
                k[q][j - off] = _limb(sign * _int(k[q][i - off]))
            for i, j, d, sign in self.twins:
                k[q][j - off] = _limb(sign * _int(k[q][i - off]) << (self.c * d))
        for j in (0, 3, key.n - 2):
            k["h"][j] = 0
        k["h"][5] = k["h"][4]
        k["h"][7] = _limb(-_int(k["h"][6]))

    def edit_z(self, codec):
        """For every mix: z_j = z_i on the repeated / negated pairs and z_j = z_i >> (c d) on the twins.  The sparse
        mix is zero except on those pairs, where z_i is a single digit v (nb, nb - 1, ... : one value per pair) in one
        window.  Each bucket it touches then holds exactly the two colliding references, so both accumulation
        kernels have to add P + P or P + (-P) themselves instead of meeting the collision inside a long running sum."""
        def put(zc, zm, i, v):
            zc[i], zm[i] = _limb(v), codec.fr_to_mont_limbs([v])[0]

        def edit(kind, zc, zm):
            nb = 1 << (self.c - 1)
            if kind == "sparse":
                for i in self.identity:              # identity bases take no bucket whatever their scalar
                    put(zc, zm, i, R - 1)
                for g, (i, _, _) in enumerate(self.same):
                    put(zc, zm, i, (nb - g) << self.c)
                for g, (i, _, d, _) in enumerate(self.twins, len(self.same)):
                    put(zc, zm, i, (nb - g) << (self.c * (d + (0 if d == self.W - 2 else 1))))
            for i, j, _ in self.same:
                zc[j], zm[j] = zc[i], zm[i]
            for i, j, d, _ in self.twins:
                put(zc, zm, j, _int(zc[i]) >> (self.c * d))
            if kind == "sparse":                     # what the library's recoding makes of it: two references per digit
                refs = [v for i in np.nonzero(zc.any(axis=1))[0] if i not in self.identity
                        for v in _digits(self.b2z, _int(zc[i]), self.c) if v]
                assert sorted(refs) == sorted(2 * [nb - g for g in range(len(self.same) + len(self.twins))])
        return edit


@pytest.mark.parametrize("kernel", ["affine", "xyzz"])
@pytest.mark.parametrize("c", [9, 14, 18])
def test_adversarial_precomputed_key(b2z, ctx, codec, cpu_oracle, monkeypatch, c, kernel):
    m, l, log_n = ADV_M[c], 3, 12
    assert (_c_of(b2z, m + 2, True), _c_of(b2z, m - l + 1, True)) == (c, c)
    _assert_precomputed(b2z, m, l, log_n)
    adv = _Adversary(b2z, c, m, l)
    key = KnownKey(b2z, ctx, m, l, log_n, seed=2000 + c, edit=adv.edit_key)
    for name, v in (AFFINE if kernel == "affine" else XYZZ).items():
        monkeypatch.setenv(name, v)
    key.pk.upload(ctx)
    try:
        mixes = (("sparse", 0, 0), ("uniform", X, Y), ("boundary", R - 1, X), ("max", Y, R - 1))
        bad = _run_mixes(b2z, ctx, codec, cpu_oracle, key, (c,), seed=c, mixes=mixes, edit_z=adv.edit_z(codec),
                         label="c=%d %s" % (c, kernel))
    finally:
        key.pk.free()
    assert not bad, bad


# ------------------------------------------------------------------------------- 5. edge shapes
@pytest.mark.parametrize("m,l,log_n", [(5, 5, 3), (6, 2, 0), (1, 1, 0)], ids=["no-witness", "domain-1", "both"])
def test_edge_shapes(b2z, ctx, codec, cpu_oracle, m, l, log_n):
    """m = l: l_query is empty and L = -rs delta; log_domain = 0: h_query is NULL and H is the identity."""
    key = KnownKey(b2z, ctx, m, l, log_n, seed=3000 + m)
    key.pk.upload(ctx)
    try:
        bad = _run_mixes(b2z, ctx, codec, cpu_oracle, key, (4,), seed=m)
    finally:
        key.pk.free()
    assert not bad, bad


@pytest.mark.parametrize("layout", ["cyclic3", "uneven"])
def test_shard_partials_sum_to_whole_key(b2z, ctx, codec, cpu_oracle, layout):
    """A c = 16 key as three block-cyclic shards and as uneven slices (the shards' own sets run at c = 11 to 16): per
    sum, the decoded shard partials add up to the whole key's known value, and their sum is what
    b2z_groth16_combine makes of the shards."""
    m, l, log_n = (1 << 16) + 1, 3, 18
    assert (_c_of(b2z, m + 2, True), _c_of(b2z, 1 << log_n, True)) == (16, 16)
    _assert_precomputed(b2z, m, l, log_n)
    key = KnownKey(b2z, ctx, m, l, log_n, seed=4000)
    zc, zm = _z_mix(codec, "boundary", m, (16, 13), 4001)
    r, s = X, Y
    want = key.sums(cpu_oracle, zc, r, s)
    weights = [5, 1, 3] if layout == "uneven" else None
    total = dict.fromkeys(NAMES)
    parts = []
    for rank in range(3):
        pk = key.copy_pk(b2z).upload(ctx, rank=rank, world=3, weights=weights)
        try:
            parts.append(key.prove(b2z, ctx, pk, zm, r, s))
        finally:
            pk.free()
        got = decode_partial(b2z, parts[-1])
        for n in NAMES:
            total[n] = add_point(n, total[n], got[n])
    assert b2z.Groth16.combine(parts) == O.proof_serialize_compressed(total["A"], total["B"], c_point(total)), \
        "partial-sum decoder disagrees with b2z_groth16_combine"
    bad = [n for n in NAMES if total[n] != point(n, want[n])]
    assert not bad, "%s: %s mismatch" % (layout, "/".join(bad))


# ------------------------------------------------------------------------------- 6. generic standalone MSM
GENERIC = [(1, 5), (1, 7), (1, 11), (1, 14), (2, 5), (2, 6), (2, 10), (2, 12), (2, 14)]


@pytest.mark.parametrize("end", ["bottom", "top"])
@pytest.mark.parametrize("group,c", GENERIC, ids=["G%d-c%d" % gc for gc in GENERIC])
def test_generic_msm_window_sizes(b2z, ctx, codec, group, c, end):
    n = (1 << (c + 3)) + 5 if end == "bottom" else 1 << (c + 4)
    assert _c_of(b2z, n, False) == c
    rs = np.random.RandomState(5000 + 100 * group + c)
    ks = rand_k(rs, n)
    curve = O.G1 if group == 1 else O.G2
    bases, inf = (b2z.FixedBase.msm_g1 if group == 1 else b2z.FixedBase.msm_g2)(ctx, ks)
    msm = b2z.VariableBaseMSM.msm_bigint_g1 if group == 1 else b2z.VariableBaseMSM.msm_bigint_g2
    proj = codec.g1_projective_from_limbs if group == 1 else codec.g2_projective_from_limbs
    rnd = random.Random(c)
    for kind in ("uniform", "boundary"):
        vals = scalar_mix(rnd, n, "uniform") if kind == "uniform" else _boundary(rnd, (c,), min(n, 1 << 12))
        assert any(_digits(b2z, v, c)[-1] for v in vals[:64]), "no scalar reaches the top window"
        sc = np.resize(codec.fr_to_bigint_limbs(vals), (n, 4))
        got = curve.to_affine(proj(msm(ctx, bases, sc, inf)))
        assert got == curve.mul(curve.gen, dot_mod_r(ks, sc)), "G%d c=%d n=%d %s scalars" % (group, c, n, kind)
