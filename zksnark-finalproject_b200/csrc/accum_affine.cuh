// Batched-affine bucket accumulation: what ONE thread does with its segment of the sorted point references.
//
// The XYZZ accumulation (msm_impl.inc, msm_accum_kernel) walks a segment with mixed additions of 8M + 2S.  An affine
// addition costs 1 division + 2M + 1S; Montgomery's trick turns the divisions of many INDEPENDENT additions into one
// inversion + 3M each, i.e. 5M + 1S per addition.  Independent additions come from a pairwise tree over every run of
// equal keys in the segment:
//
//   round r: every run of R entries becomes floor(R/2) sums + (R odd ? the last entry : nothing);
//            forward pass  : denominators d_k = x2 - x1 (2 y1 for a doubling), prefix products, (in, out) descriptors;
//                            pairs that need no division (an operand is the identity marker, P + (-P)) and the odd
//                            entries are written straight to the output list;
//            one inversion : division steps (inv_gcd.cuh), ~35 product-equivalents, per thread, all lanes busy;
//            backward pass : d_k^-1 = inv * prefix_k, inv *= d_k, the affine sum, stored canonical.
//   Rounds continue while a round has at least kMinPairs pairs (below that the inversion costs more than it saves);
//   the entries that remain (a few per run) are summed by the XYZZ mixed addition exactly as the XYZZ kernel does
//   and go to the same places: the bucket itself for a run inside the segment, the (key, partial sum) list for a run
//   cut by a segment boundary.  Everything downstream (partial-list levels, merge, bucket reduction) is unchanged.
//
// Entry lists ping-pong between two per-thread scratch buffers (round 0 reads the key's points through the sorted
// references), so a backward pass never overwrites an input it still needs.  The identity is the marker (0, 0),
// which is not on y^2 = x^3 + 4 (nor on the twist).
//
// Host and device: the same code runs in hostcheck.cu against a naive sum (tests/test_host_logic.py).
#pragma once
#include "ec.cuh"
#include "inv_gcd.cuh"

namespace b2z {
namespace aff {

constexpr uint32_t kNegBit = 0x80000000u;     // sign bit of a sorted point reference
constexpr uint32_t kEmptyKey = 0xffffffffu;   // key of the partial slots of a segment past the end of the list
constexpr uint32_t kMinPairsDefault = 24;

// host emulation only: [0] completed rounds, [1] batched additions, [2] of which doublings, [3] division-free pairs
// (identity marker / cancellation), [4] abandoned forward passes, [5] mixed additions of the XYZZ finish
inline uint64_t* host_stats() {
  static thread_local uint64_t s[8] = {0};
  return s;
}
#if !defined(__CUDA_ARCH__)
#define B2Z_AFF_STAT(i, n) (b2z::aff::host_stats()[i] += (n))
#else
#define B2Z_AFF_STAT(i, n) ((void)0)
#endif

// ---- element access without parking values in local memory (constant limb indices after unrolling)
template <bool RO>
B2Z_HD FqEl ld_el(const FqEl* p) {
#if defined(__CUDA_ARCH__)
  FqEl e;
  const uint4* q = reinterpret_cast<const uint4*>(p);
#pragma unroll
  for (int i = 0; i < 3; i++) {
    const uint4 v = RO ? __ldg(q + i) : q[i];
    e.l[4 * i] = v.x; e.l[4 * i + 1] = v.y; e.l[4 * i + 2] = v.z; e.l[4 * i + 3] = v.w;
  }
  return e;
#else
  return *p;
#endif
}
template <bool RO>
B2Z_HD Fq2El ld_el(const Fq2El* p) {
  Fq2El e;
  e.c0 = ld_el<RO>(&p->c0);
  e.c1 = ld_el<RO>(&p->c1);
  return e;
}
B2Z_HD void st_el(FqEl* p, const FqEl& e) {
#if defined(__CUDA_ARCH__)
  uint4* q = reinterpret_cast<uint4*>(p);
#pragma unroll
  for (int i = 0; i < 3; i++) q[i] = make_uint4(e.l[4 * i], e.l[4 * i + 1], e.l[4 * i + 2], e.l[4 * i + 3]);
#else
  *p = e;
#endif
}
B2Z_HD void st_el(Fq2El* p, const Fq2El& e) {
  st_el(&p->c0, e.c0);
  st_el(&p->c1, e.c1);
}

B2Z_HD bool all_zero(const FqEl& a) {
  uint32_t z = 0;
#pragma unroll
  for (int i = 0; i < 12; i++) z |= a.l[i];
  return z == 0;
}
B2Z_HD bool all_zero(const Fq2El& a) { return all_zero(a.c0) && all_zero(a.c1); }

// the shared inversion
B2Z_HD FqEl inverse(const FqEl& a) { return gcdinv::inv(a); }
B2Z_HD Fq2El inverse(const Fq2El& a) {             // conj(a) / (a0^2 + a1^2)
  const FqEl n = gcdinv::inv(Fq::add(Fq::sqr(a.c0), Fq::sqr(a.c1)));
  return Fq2El{Fq::mul(a.c0, n), Fq::neg(Fq::mul(a.c1, n))};
}

B2Z_HD uint32_t umin(uint32_t a, uint32_t b) { return a < b ? a : b; }

B2Z_HD void raise_max(uint32_t* p, uint32_t v) {
#if defined(__CUDA_ARCH__)
  atomicMax(p, v);
#else
  if (*p < v) *p = v;
#endif
}

template <class C>
B2Z_HD void st_xyzz(typename C::Xyzz* dst, const typename C::Xyzz& v) {
  st_el(&dst->x, v.x);
  st_el(&dst->y, v.y);
  st_el(&dst->zz, v.zz);
  st_el(&dst->zzz, v.zzz);
}

// The segment protocol of both accumulation kernels (msm_impl.inc) and of the host emulation (hostcheck.cu).
// The `total` sorted references are cut into nseg segments of seg_len = max(8, ceil(total / nseg)), one per thread;
// segment `seg` covers [lo, hi).  The length follows the ACTUAL number of references (zero digits and identity bases
// are gone), so the fixed grid stays busy whatever fraction of the scalars is zero or small.  A run of one bucket
// that lies inside the segment goes straight to the bucket; a run cut by the segment's start goes to the leading
// partial slot 2 seg, one cut by its end to the trailing slot 2 seg + 1.  Both slots are always written -- the
// identity keyed by the first / last bucket when unused, kEmptyKey for a segment past the end -- so the partial list
// stays sorted by key.
template <class C>
struct Segment {
  using Xyzz = typename C::Xyzz;
  uint32_t seg, seg_len, lo, hi, total;
  uint32_t first, first_begin, first_end;   // first bucket: first_begin = offsets[first] <= lo < offsets[first + 1]
  bool active;                              // seg < nseg and lo < total
  bool wrote0, wrote1;
  Xyzz* bucket_out;
  uint32_t* part_keys;
  Xyzz* part_pts;
  uint32_t* maxrun;

  B2Z_HD Segment(const uint32_t* offsets, uint32_t nbuckets, uint32_t nseg, uint32_t seg_, Xyzz* bucket_out_,
                 uint32_t* part_keys_, Xyzz* part_pts_, uint32_t* maxrun_)
      : seg(seg_), lo(0), hi(0), first(0), first_begin(0), first_end(0), wrote0(false), wrote1(false),
        bucket_out(bucket_out_), part_keys(part_keys_), part_pts(part_pts_), maxrun(maxrun_) {
    total = offsets[nbuckets];
    seg_len = (total + nseg - 1) / nseg;
    if (seg_len < 8) seg_len = 8;
    active = seg < nseg && (uint64_t)seg * seg_len < total;
    if (!active) return;
    lo = seg * seg_len;
    hi = umin(lo + seg_len, total);
    uint32_t a = 0, z = nbuckets;   // largest bucket a with offsets[a] <= lo; invariant offsets[a] <= lo < offsets[z]
    while (z - a > 1) {
      const uint32_t mid = (a + z) >> 1;
      if (offsets[mid] <= lo) a = mid; else z = mid;
    }
    first = a;
    first_begin = offsets[a];
    first_end = offsets[a + 1];
    while (first_end <= lo) {        // skip empty buckets that share the same offset
      first++;
      first_begin = first_end;
      first_end = offsets[first + 1];
    }
  }

  // The run of bucket `key` (references [begin, end) of the whole list) ends inside this segment (end <= hi) with the
  // sum `acc`: it goes to the leading slot or to the bucket.  This is flush() for a run that is not the segment's
  // last: there (end - 1) / seg_len == seg, so its bound reduces to 2 (seg - begin / seg_len + 1).  The XYZZ kernel
  // calls it inside its hot loop, where the trailing case of flush() costs the G2 kernel registers.
  template <class Acc>
  B2Z_HD void flush_inside(uint32_t key, uint32_t begin, const Acc& acc) {
    if (begin < lo) {
      part_keys[2 * seg] = key;
      acc.store(part_pts + 2 * seg);
      wrote0 = true;
      raise_max(maxrun, 2 * (seg - begin / seg_len + 1));
    } else {
      acc.store(bucket_out + key);
    }
  }
  // The segment's last run, of bucket `key` (references [begin, end) of the whole list), with the sum `acc`.
  template <class Acc>
  B2Z_HD void flush(uint32_t key, uint32_t begin, uint32_t end, const Acc& acc) {
    if (begin < lo) {
      part_keys[2 * seg] = key;
      acc.store(part_pts + 2 * seg);
      wrote0 = true;
    } else if (end > hi) {
      part_keys[2 * seg + 1] = key;
      acc.store(part_pts + 2 * seg + 1);
      wrote1 = true;
    } else {
      acc.store(bucket_out + key);
    }
    // entries this bucket can have in the partial list: 2 per segment it touches
    if (begin < lo || end > hi) raise_max(maxrun, 2 * ((umin(end, total) - 1) / seg_len - begin / seg_len + 1));
  }
  // after the last run (keyed `last`) of an active segment
  B2Z_HD void close(uint32_t last) {
    if (!wrote0) { part_keys[2 * seg] = first; st_xyzz<C>(part_pts + 2 * seg, C::identity()); }
    if (!wrote1) { part_keys[2 * seg + 1] = last; st_xyzz<C>(part_pts + 2 * seg + 1, C::identity()); }
  }
  // an inactive segment that is still in the grid
  B2Z_HD void close_empty() {
    part_keys[2 * seg] = kEmptyKey;
    part_keys[2 * seg + 1] = kEmptyKey;
  }
};

// The running sum of the XYZZ finish.  Default: the XYZZ point in registers (G1: 48 words).  The G2 kernel passes its
// shared-memory sum instead (msm_impl.inc, RunningSum<G2>: 96 words do not fit beside an Fq2 product).
template <class C>
struct RegAcc {
  typename C::Xyzz v;
  B2Z_HD explicit RegAcc(uint32_t*) { v = C::identity(); }
  B2Z_HD void reset() { v = C::identity(); }
  // q = the entry at src, already loaded (and negated when `neg`); ro: src is read-only key data
  B2Z_HD void madd(const typename C::Affine& q, const typename C::Affine* src, bool neg, bool) {
    v = C::madd_inl_at(v, q, src, neg);
  }
  B2Z_HD void store(typename C::Xyzz* dst) const { st_xyzz<C>(dst, v); }
};

// Per-thread scratch (this thread's regions): two entry lists of as many entries as the segment is long (a round
// never grows a list: every unit consumes at least one entry and emits one), one prefix product and one
// descriptor per pair.
template <class C>
struct Scratch {
  typename C::Affine* pts[2];
  uint32_t* keys[2];
  typename C::El* pref;
  uint4* desc;                 // (handle of the first operand, handle of the second, output slot, unused)
};

// A vote over the warp.  Every decision that changes WHICH loop a lane is in (another round or not) is taken with it,
// so the lanes of a warp stay in the same pass and the passes run converged; every lane of the warp must get here
// (the kernel keeps idle threads alive with an empty list).
B2Z_HD bool warp_any(bool p) {
#if defined(__CUDA_ARCH__)
  return __any_sync(0xffffffffu, p);
#else
  return p;
#endif
}

// The current entry list: the sorted references (before the first round) or a scratch list.  An entry is named by
// a HANDLE -- the reference word itself (point index | sign bit) or the index into the scratch list -- so that the
// passes can fetch handles ahead of the points they name.
template <class C>
struct List {
  using F = typename C::Fld;
  using El = typename C::El;
  using Affine = typename C::Affine;
  const Affine* points;
  const uint32_t* sorted;     // + lo
  const uint32_t* offsets;
  uint32_t lo;
  const Affine* in;
  const uint32_t* kin;
  bool refs;
  uint32_t rc, rnext;         // run cursor over the references: bucket of the last queried position, its end

  B2Z_HD uint32_t handle(uint32_t i, uint32_t cnt) const { return i < cnt ? (refs ? sorted[i] : i) : 0u; }
  // The forward pass keeps a WINDOW of four words for entries i .. i + 3, fetched two units ahead of their use:
  // the reference words themselves, or the keys of the scratch entries (whose handles are just their indices).
  B2Z_HD uint32_t window_word(uint32_t i, uint32_t cnt) const { return i < cnt ? (refs ? sorted[i] : kin[i]) : 0u; }
  B2Z_HD uint32_t handle_of(uint32_t word, uint32_t i) const { return refs ? word : i; }
  B2Z_HD const Affine* ptr(uint32_t h) const { return refs ? points + (h & ~kNegBit) : in + h; }
  B2Z_HD bool negated(uint32_t h) const { return refs && (h & kNegBit) != 0; }
  B2Z_HD El x_of(uint32_t h) const {
    const Affine* p = ptr(h);
    return refs ? ld_el<true>(&p->x) : ld_el<false>(&p->x);
  }
  B2Z_HD El y_of(uint32_t h) const {
    const Affine* p = ptr(h);
    const El y = refs ? ld_el<true>(&p->y) : ld_el<false>(&p->y);
    return negated(h) ? F::reduce(F::neg(y)) : y;
  }
  B2Z_HD uint32_t key_at(uint32_t i) {          // i must not decrease between calls (until the cursor is rewound)
    if (!refs) return kin[i];
    const uint32_t pos = lo + i;
    while (pos >= rnext) {
      rc++;
      rnext = offsets[rc + 1];
    }
    return rc;
  }
  // entry j = i + 1 in the same run as entry i (whose key was just queried)?
  B2Z_HD bool same_run(uint32_t j, uint32_t key) const { return refs ? lo + j < rnext : kin[j] == key; }
};

// One thread's segment G of the sorted references: complete runs go to their buckets, cut runs to the partial slots
// (Segment).  An inactive segment only takes part in the warp votes.
template <class C, class Acc = RegAcc<C>>
B2Z_HD void accum_segment(const typename C::Affine* points, const uint32_t* sorted, const uint32_t* offsets,
                          Segment<C>& G, const Scratch<C>& S, uint32_t kMinPairs = kMinPairsDefault,
                          uint32_t* acc_ctx = nullptr) {
  using F = typename C::Fld;
  using El = typename C::El;
  using Affine = typename C::Affine;

  List<C> L;
  L.points = points;
  L.sorted = sorted + G.lo;
  L.offsets = offsets;
  L.lo = G.lo;
  L.in = nullptr;
  L.kin = nullptr;
  L.refs = true;
  L.rc = G.first;
  L.rnext = G.first_end;
  uint32_t cnt = G.active ? G.hi - G.lo : 0;
  int out_sel = 0;

  // ---- tree rounds
  for (;;) {
    if (!warp_any(cnt >= 2 * kMinPairs)) break;
    Affine* out = out_sel ? S.pts[1] : S.pts[0];          // (a dynamic index would park S in local memory)
    uint32_t* kout = out_sel ? S.keys[1] : S.keys[0];
    // -- forward pass, one UNIT per iteration: a pair of neighbours with equal keys, or a single entry.  The handles
    // of the next three entries and the x coordinates of the next unit are fetched before this unit's product.
    El acc = F::one();
    uint32_t npairs = 0, o = 0, i = 0;
    uint32_t w0 = L.window_word(0, cnt), w1 = L.window_word(1, cnt), w2 = L.window_word(2, cnt),
             w3 = L.window_word(3, cnt);
    El x1 = L.x_of(L.handle_of(w0, 0)), x2 = L.x_of(L.handle_of(w1, cnt > 1 ? 1u : 0u));
    while (i < cnt) {
      uint32_t key;
      bool pair;
      if (L.refs) {
        key = L.key_at(i);
        pair = i + 1 < cnt && L.lo + i + 1 < L.rnext;
      } else {
        key = w0;
        pair = i + 1 < cnt && w1 == w0;
      }
      const uint32_t ha = L.handle_of(w0, i), hb = L.handle_of(w1, i + 1);
      const uint32_t inext = i + (pair ? 2u : 1u);
      if (pair) {
        w0 = w2; w1 = w3;
        w2 = L.window_word(inext + 2, cnt);
      } else {
        w0 = w1; w1 = w2; w2 = w3;
      }
      w3 = L.window_word(inext + 3, cnt);
      const El nx1 = L.x_of(L.handle_of(w0, inext < cnt ? inext : 0u));
      const El nx2 = L.x_of(L.handle_of(w1, inext + 1 < cnt ? inext + 1 : 0u));
      kout[o] = key;
      if (pair) {
        El d = F::sub(x2, x1);
        bool batch = true;
        if (F::is_zero(d) || all_zero(x1) || all_zero(x2)) {
          // rare: an identity marker, a doubling, or P + (-P)
          const El y1 = L.y_of(ha), y2 = L.y_of(hb);
          const bool m1 = all_zero(x1) && all_zero(y1), m2 = all_zero(x2) && all_zero(y2);
          if (m1 || m2) {
            batch = false;
            st_el(&out[o].x, m1 ? x2 : x1);              // both markers: the marker again
            st_el(&out[o].y, m1 ? y2 : y1);
          } else if (F::is_zero(d)) {
            d = F::dbl(y1);
            if (!F::is_zero(F::sub(y2, y1)) || F::is_zero(d)) {   // P + (-P) (or a point of order two)
              batch = false;
              st_el(&out[o].x, F::zero());
              st_el(&out[o].y, F::zero());
            }
          }
        }
        if (batch) {
          st_el(S.pref + npairs, acc);
          S.desc[npairs] = make_uint4(ha, hb, o, 0u);
          acc = F::mul(acc, d);
          npairs++;
        } else {
          B2Z_AFF_STAT(3, 1);
        }
      } else {                                               // carried as it is
        st_el(&out[o].x, x1);
        st_el(&out[o].y, L.y_of(ha));
      }
      o++;
      i = inext;
      x1 = nx1;
      x2 = nx2;
    }
    if (!warp_any(npairs >= kMinPairs)) {
      B2Z_AFF_STAT(4, 1);
      // not worth an inversion: the XYZZ finish takes the CURRENT list; rewind the run cursor
      if (L.refs) { L.rc = G.first; L.rnext = G.first_end; }
      break;
    }
    // -- one inversion, then the sums from the last pair to the first
    // (software pipeline: the descriptor of pair k - 2 and the x coordinates and prefix product of pair k - 1 are
    // in flight while pair k is computed; the y coordinates are asked for at the top of their own iteration and
    // first needed two products later)
    El inv = inverse(acc);
    const uint4 none = make_uint4(0u, 0u, 0u, 0u);
    if (sizeof(El) > sizeof(FqEl)) {
      // Fq2: an element is 24 registers -- nothing is kept in flight; every operand is (re)loaded where it is
      // consumed (the second reads hit L1) so that at most inv, lambda, x3 and one operand are live beside a product
      uint4 de = npairs ? S.desc[npairs - 1] : none;
      for (uint32_t k = npairs; k-- > 0;) {
        const uint4 den = k ? S.desc[k - 1] : none;
        El d = F::sub(L.x_of(de.y), L.x_of(de.x));
        const bool dbl = F::is_zero(d);
        if (dbl) d = F::dbl(L.y_of(de.x));
        El lam = F::mul(inv, ld_el<false>(S.pref + k));       // 1 / d
        inv = F::mul(inv, d);
        if (dbl) {
          B2Z_AFF_STAT(2, 1);
          const El xx = F::sqr(L.x_of(de.x));
          lam = F::mul(F::add(F::dbl(xx), xx), lam);
        } else {
          lam = F::mul(F::sub(L.y_of(de.y), L.y_of(de.x)), lam);
        }
        const El x1r = L.x_of(de.x);
        const El x3 = F::sub(F::sub(F::sqr(lam), x1r), L.x_of(de.y));
        st_el(&out[de.z].x, F::reduce(x3));
        const El y3 = F::sub(F::mul(lam, F::sub(x1r, x3)), L.y_of(de.x));
        st_el(&out[de.z].y, F::reduce(y3));
        de = den;
      }
    } else {
    uint4 de = npairs ? S.desc[npairs - 1] : none;
    uint4 den = npairs > 1 ? S.desc[npairs - 2] : none;
    El x1b = L.x_of(de.x), x2b = L.x_of(de.y);
    El pf = ld_el<false>(S.pref + (npairs ? npairs - 1 : 0));
    for (uint32_t k = npairs; k-- > 0;) {
      const uint4 den2 = k > 1 ? S.desc[k - 2] : none;
      const El nx1 = L.x_of(den.x), nx2 = L.x_of(den.y);
      const El npf = ld_el<false>(S.pref + (k ? k - 1 : 0));
      const El y1 = L.y_of(de.x), y2 = L.y_of(de.y);
      El d = F::sub(x2b, x1b);
      const bool dbl = F::is_zero(d);
      if (dbl) d = F::dbl(y1);
      const El dinv = F::mul(inv, pf);
      inv = F::mul(inv, d);
      El num;
      if (dbl) {
        B2Z_AFF_STAT(2, 1);
        const El xx = F::sqr(x1b);
        num = F::add(F::dbl(xx), xx);
      } else {
        num = F::sub(y2, y1);
      }
      const El lam = F::mul(num, dinv);
      const El x3 = F::sub(F::sub(F::sqr(lam), x1b), x2b);
      const El y3 = F::sub(F::mul(lam, F::sub(x1b, x3)), y1);
      st_el(&out[de.z].x, F::reduce(x3));
      st_el(&out[de.z].y, F::reduce(y3));
      de = den;
      den = den2;
      x1b = nx1;
      x2b = nx2;
      pf = npf;
    }
    }
    B2Z_AFF_STAT(0, 1);
    B2Z_AFF_STAT(1, npairs);
    L.refs = false;
    L.in = out;
    L.kin = kout;
    cnt = o;
    out_sel ^= 1;
  }
  if (!G.active) return;

  // ---- XYZZ finish over the current list
  uint32_t cur_key = L.key_at(0);
  Acc acc(acc_ctx);
  for (uint32_t i = 0; i < cnt; i++) {
    const uint32_t key = L.key_at(i);
    if (key != cur_key) {
      G.flush_inside(cur_key, offsets[cur_key], acc);
      acc.reset();
      cur_key = key;
    }
    const uint32_t h = L.handle(i, cnt);
    Affine q;
    q.x = L.x_of(h);
    q.y = L.y_of(h);
    if (all_zero(q.x) && all_zero(q.y)) continue;          // identity marker
    B2Z_AFF_STAT(5, 1);
    acc.madd(q, L.ptr(h), L.negated(h), L.refs);
  }
  G.flush(cur_key, offsets[cur_key], offsets[cur_key + 1], acc);
  G.close(cur_key);
}

}  // namespace aff
}  // namespace b2z
