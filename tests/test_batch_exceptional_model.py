"""A model of the batch arithmetic on exceptional group elements, and the cases of test_gpu_batch_exceptional.py.

Every point of a case is a multiple a*B of one base point B of order N: B = G (N = q), B = G + T (N = m q) or B = T
(N = m), with T a torsion point of order m.  Scalar multiplication is a homomorphism, so every intermediate value of every
stage of the device pipeline is a known integer mod N: "same point" is "equal mod N", "opposite points" is "sum = 0",
"identity" is "= 0".  The model below replays the stages of batch.cuh on those integers, in the order the kernels
add, and records each addition that takes an exceptional branch (an identity operand, equal operands, opposite operands).

This file checks, without a GPU, that the model agrees with the oracle (its lhs multiple times B is the lhs of
cref.verify_batch) and that every case makes the events it is named after happen, in every geometry the GPU file forces.
The GPU file then compares the device with the oracle on the same inputs and checks that the device ran the plan the
model assumed.
"""
import functools

import numpy as np
import pytest

import cref
import pyref as o
from util import KAT96, pack_msgs, pt_to96

Q = o.Q
G96 = pt_to96(o.generator())
TORSION_ORDERS = (2, 29, 58, 181, 155833)


def _le32(k):
    return np.frombuffer(int(k).to_bytes(32, "little"), dtype=np.uint8).copy()


def _mul(pt96, inf, k):
    """k * point for 0 <= k < 2^256 (oracle #2)."""
    return cref.pt_mul(pt96, inf, _le32(k))


@functools.lru_cache(maxsize=None)
def torsion(m):
    """T_m = (COFACTOR q / m) KAT, a point of order exactly m."""
    assert o.COFACTOR % m == 0
    t, ti = _mul(KAT96, 0, o.COFACTOR // m)
    t, ti = _mul(t, ti, Q)
    assert not ti
    assert _mul(t, 0, m)[1] == 1, "order divides m"
    for p in {f for f in (2, 29, 181, 155833) if m % f == 0}:
        assert _mul(t, 0, m // p)[1] == 0, "order is exactly m"
    return t.tobytes()


class Base:
    """B = G (m = 1, with_g), G + T_m (m > 1, with_g) or T_m (not with_g); N = the order of B."""

    def __init__(self, m=1, with_g=True):
        self.m, self.with_g = m, with_g
        self.N = (Q if with_g else 1) * m
        self._cache = {}

    def point(self, a):
        """a * B -> (pt96, inf), split as (a mod q) G + (a mod m) T_m (the oracle takes 256-bit scalars)."""
        a %= self.N
        if a in self._cache:
            return self._cache[a]
        acc, ai = np.zeros(96, dtype=np.uint8), 1
        if self.with_g and a % Q:
            acc, ai = _mul(G96, 0, a % Q)
        if self.m > 1 and a % self.m:
            t, ti = _mul(np.frombuffer(torsion(self.m), dtype=np.uint8), 0, a % self.m)
            acc, ai = cref.pt_add(acc, ai, t, ti)
        self._cache[a] = (acc, ai)
        return acc, ai

    def lhs97(self, a):
        pt, inf = self.point(a)
        return np.concatenate([np.zeros(96, dtype=np.uint8) if inf else pt, np.array([inf], dtype=np.uint8)])


# ---- exceptional-branch events ----------------------------------------------------------------------------------------
class Events:
    def __init__(self, N):
        self.N = N
        self.seen = set()

    def add(self, stage, a, b):
        """a + b of one exact addition of `stage`; records the branch it takes."""
        N = self.N
        a %= N
        b %= N
        if a == 0 and b == 0:
            self.seen.add((stage, "O+O"))
        elif a == 0:
            self.seen.add((stage, "O+W"))
        elif b == 0:
            self.seen.add((stage, "W+O"))
        elif a == b:
            self.seen.add((stage, "equal"))
        elif (a + b) % N == 0:
            self.seen.add((stage, "cancel"))
        return (a + b) % N

    def dbl(self, stage, a):
        a %= self.N
        if a and (2 * a) % self.N == 0:
            self.seen.add((stage, "dbl_to_O"))
        return (2 * a) % self.N

    def note(self, stage, what):
        self.seen.add((stage, what))

    def __contains__(self, ev):
        return ev in self.seen


# ---- the Pippenger pipeline (batch.cuh) ------------------------------------------------------------------------------
def msm_plan(npoints, c_override=0):
    """msm_make_plan, batch.cuh:27-59 -> (c, K, B, chunk_sz, chunks)."""
    best, c_best = None, None
    for c in range(4, 17):
        K = (256 + c - 1) // c
        cost = float(npoints) * K + 3.0 * K * float(1 << (c - 1))
        if best is None or cost < best:
            best, c_best = cost, c
    c = c_best
    if npoints <= 8192:
        c = 8
    if 4 <= c_override <= 16:
        c = c_override
    K, B = (256 + c - 1) // c, 1 << (c - 1)
    want = int((B * K) / 8192.0)
    chunk_sz = 32 if want >= 32 else (16 if want >= 16 else 8)
    chunk_sz = min(chunk_sz, B)
    return c, K, B, chunk_sz, B // chunk_sz


def segment_len(npoints, K, t_override=0):
    """The segment length rule of batch_partial_impl, batch.cuh:1246-1252."""
    max_entries = npoints * K
    T = 32
    while T > 8 and max_entries // T < 65536:
        T //= 2
    if t_override:
        T = t_override
    while (max_entries + T - 1) // T > (1 << 20):
        T *= 2
    return T


def msm_digits(s, c, K):
    """msm_digit, batch.cuh:184-190: (bucket id 1..B or 0, negated) per window, least significant first."""
    out, carry, half = [], 0, 1 << (c - 1)
    for k in range(K):
        raw = ((s >> (k * c)) & ((1 << c) - 1)) + carry
        neg = raw > half
        carry = 1 if neg else 0
        out.append(((1 << c) - raw if neg else raw, neg))
    return out


def recode_signed_w4(s):
    """recode_signed_w4, curve.cuh:239-247: 64 signed 4-bit digits in -7..8."""
    out, carry = [], 0
    for i in range(64):
        raw = ((s >> (4 * i)) & 15) + carry
        carry = 1 if raw > 8 else 0
        out.append(raw - 16 if carry else raw)
    return out


FOLD_THREADS = 128
MSM_LONG_SPAN = 16


def _warp_tree(ev, stage, vals):
    """Lane 0 of `for d in 16..1: v[l] += shfl_down(v, d)` (lanes past 31 read the identity); records the additions that
    reach lane 0 (lanes l < d)."""
    v = list(vals) + [0] * (32 - len(vals))
    for d in (16, 8, 4, 2, 1):
        v = [ev.add(stage, v[l], v[l + d]) if l < d else v[l] for l in range(32)]
    return v[0]


def pippenger(points, N, c_override=0, t_override=0):
    """points: [(multiple, scalar)] in MSM order -> (partial multiple, Events, plan dict).  Replays k_msm_count/scatter
    (buckets), k_msm_segment_sum/fixup/fixup_long (segments), k_msm_window_sum, k_msm_window_fold and k_msm_horner."""
    ev = Events(N)
    npts = len(points)
    c, K, B, chunk_sz, chunks = msm_plan(npts, c_override)
    T = segment_len(npts, K, t_override)
    content = {}
    for j, (a, s) in enumerate(points):
        for k, (b, neg) in enumerate(msm_digits(s, c, K)):
            if b:
                content.setdefault((k, b), []).append(-a % N if neg else a % N)
    # bucket sums: the scatter order inside a bucket is not deterministic, so only order-free facts are recorded
    val = {}
    pos = 0
    for (k, b) in sorted(content):
        lst = content[(k, b)]
        val[(k, b)] = sum(lst) % N
        if len(lst) >= 2:
            ms = sorted(lst)
            if val[(k, b)] == 0:
                ev.note("bucket", "sum_O")
            if len(lst) == 2 and ms[0] == ms[1]:
                ev.note("bucket", "pair_equal")     # {X, X}: the second addition doubles, whatever the order
            if len(lst) == 2 and ms[0] and (ms[0] + ms[1]) % N == 0:
                ev.note("bucket", "pair_cancel")    # {X, -X}: the second addition cancels
            if any(x and (-x) % N in set(ms) for x in ms):
                ev.note("bucket", "has_opposite")
            if len(set(ms)) < len(ms):
                ev.note("bucket", "has_equal")
        # the sorted list holds the buckets in slot order; segment t owns positions [t T, (t + 1) T)
        lo_seg, hi_seg = pos // T, (pos + len(lst) - 1) // T
        if lo_seg != hi_seg:
            kind = "long" if hi_seg - lo_seg >= MSM_LONG_SPAN else "cross"
            ev.note("segment", kind)
            if len(lst) == 2:               # one entry on each side: the fixup adds the two points themselves
                if lst[0] == lst[1]:
                    ev.note("segment", kind + "_pair_equal")
                elif (lst[0] + lst[1]) % N == 0:
                    ev.note("segment", kind + "_pair_cancel")
            if kind == "long" and len(set(lst)) == 1:
                ev.note("segment", "long_uniform")   # full segments: equal partials, whatever the order
                if (T * lst[0]) % N == 0:
                    # T copies of a point of order 2: every full segment's partial is O, the others T2 = -T2
                    ev.note("segment", "long_partials_O")
        pos += len(lst)
    # k_msm_window_sum: chunk ch of window k covers buckets lo..lo+chunk_sz-1, from the top
    chunk_out = {}
    live = {(k, (b - 1) // chunk_sz) for (k, b) in val}
    for k in range(K):
        for ch in range(chunks):
            lo = ch * chunk_sz + 1
            if (k, ch) not in live:         # all buckets empty: identities only
                chunk_out[(k, ch)] = 0
                continue
            running = acc = 0
            for b in range(chunk_sz - 1, -1, -1):
                running = ev.add("ws_running", running, val.get((k, lo + b), 0))
                acc = ev.add("ws_acc", acc, running)
            if lo > 1:
                m = lo - 1
                mm = running
                for bit in range(m.bit_length() - 2, -1, -1):
                    mm = ev.dbl("ws_mul", mm)
                    if (m >> bit) & 1:
                        mm = ev.add("ws_mul", mm, running)
                if running % N and mm == 0:
                    ev.note("ws_mul", "small_order")   # (lo - 1) running = O with running != O
                acc = ev.add("ws_lo", acc, mm)
            chunk_out[(k, ch)] = acc
    # k_msm_window_fold: strided per thread, shuffle tree per warp, warps 1..3 onto warp 0
    windows = []
    for k in range(K):
        th = [0] * FOLD_THREADS
        for ch in range(chunks):
            th[ch % FOLD_THREADS] = ev.add("fold_strided", th[ch % FOLD_THREADS], chunk_out[(k, ch)])
        warp = [_warp_tree(ev, "fold_tree", th[32 * w:32 * w + 32]) for w in range(FOLD_THREADS // 32)]
        acc = warp[0]
        for w in range(1, FOLD_THREADS // 32):
            acc = ev.add("fold_warps", acc, warp[w])
        windows.append(acc)
    # k_msm_horner
    acc = windows[K - 1]
    for w in range(K - 2, -1, -1):
        acc = (acc << c) % N
        acc = ev.add("horner", acc, windows[w])
    assert acc == sum(a * s for a, s in points) % N
    return acc, ev, dict(c=c, K=K, B=B, T=T)


# ---- the block-per-signature form (k_batch_small, k_batch_small_reduce) ----------------------------------------------
SMALL_REDUCE_WARPS = 16


def small_reduce(ev, stage, terms):
    """k_batch_small_reduce: warp w adds terms w, w + 16, ... in order, then a tree over the 16 warps."""
    x = [0] * SMALL_REDUCE_WARPS
    for i, t in enumerate(terms):
        x[i % SMALL_REDUCE_WARPS] = ev.add(stage, x[i % SMALL_REDUCE_WARPS], t)
    d = SMALL_REDUCE_WARPS // 2
    while d:
        x = [ev.add(stage + "_tree", x[w], x[w + d]) if w < d else x[w] for w in range(SMALL_REDUCE_WARPS)]
        d //= 2
    return x[0]


def batch_small(items, N):
    """items: [(R multiple, s_r, -P multiple, s_p)] -> (partial multiple, Events).  Window points 16^w R and 16^w (-P),
    buckets |digit| = 1..8 in window order, running sums from bucket 8 down, T_i, then the reduce."""
    ev = Events(N)
    terms = []
    for ra, sr, pa, sp in items:
        agg = []
        for a, s in ((ra, sr), (pa, sp)):
            win = [(a * pow(16, w, N)) % N for w in range(64)]
            if a % N and any(x == 0 for x in win[1:]):
                ev.note("small_window", "O")
            digits = recode_signed_w4(s)
            bk = []
            for mag in range(1, 9):
                acc, first = 0, True
                for w in range(64):
                    d = digits[w]
                    if d and abs(d) == mag:
                        p = (-win[w] if d < 0 else win[w]) % N
                        acc = p if first else ev.add("small_bucket", acc, p)
                        first = False
                bk.append(acc)
            r = o_ = bk[7]
            for b in range(6, -1, -1):
                r = ev.add("small_running", r, bk[b])
                o_ = ev.add("small_agg", o_, r)
            agg.append(o_)
        t = ev.add("small_term", agg[0], agg[1])
        assert t == (ra * sr + pa * sp) % N
        terms.append(t)
    return small_reduce(ev, "small_reduce", terms), ev


# ---- the key side of a registered batch (k_keyset_scalar_sum, k_keyset_batch_term) ----------------------------------
KT_W, KT_WINDOWS, KEYTERM_WARPS = 8, 32, 4


def key_terms(ev, key_mult, key_t, N, sm_count=148):
    """key_mult[k]: the multiple of P_k; key_t[k]: the t_i of its items -> the key partial multiple.  Column sums and
    keyset_sum_reduce (keyset.cuh:262-275), the KT_W-bit recoding of keyset_window_term (keyset.cuh:279-303), the
    per-warp shuffle tree, the warp's running sum, the block fold, then k_batch_small_reduce over the block terms."""
    n_keys = len(key_mult)
    blocks = min(2 * sm_count, (n_keys + KEYTERM_WARPS - 1) // KEYTERM_WARPS)
    acc = [[0] * KEYTERM_WARPS for _ in range(blocks)]
    for k in range(n_keys):
        total = sum(key_t[k])                                 # the column sums carry the exact integer sum
        if total >> 256:
            ev.note("key_sum", "hi")
        c = total % Q
        if total and c == 0:
            ev.note("key_sum", "c_zero_nonzero_columns")
        if c == Q - 1:
            ev.note("key_sum", "c_q_minus_1")
        if c == 0:
            continue
        lanes, carry = [], 0
        for i in range(KT_WINDOWS):
            raw = ((c >> (KT_W * i)) & 0xFF) + carry
            neg = raw > 128
            carry = 1 if neg else 0
            dsig = raw - 256 if neg else raw
            lanes.append((-dsig * (1 << (KT_W * i)) * key_mult[k]) % N)
        t = _warp_tree(ev, "key_tree", lanes)
        assert t == (-c * key_mult[k]) % N
        b, w = (k // KEYTERM_WARPS) % blocks, k % KEYTERM_WARPS   # k = (block, warp), strided by blocks * 4
        acc[b][w] = ev.add("key_warp", acc[b][w], t)
    terms = []
    for b in range(blocks):
        x = acc[b][0]
        for w in range(1, KEYTERM_WARPS):
            x = ev.add("key_block", x, acc[b][w])
        terms.append(x)
    return small_reduce(ev, "key_reduce", terms)


# ---- building the inputs ---------------------------------------------------------------------------------------------
class Item:
    """One signature of a case.  r: multiple of R (None = the identity R); flip: negate R through its flag byte; flag:
    an explicit flag byte; p: multiple of P (None = the identity key); s: randomiser, or t: the key-side scalar
    t = s h mod q to solve s for; e: the signature scalar."""

    def __init__(self, r, p, s=None, t=None, e=0, flip=False, flag=None, msg=None):
        self.r, self.p, self.s, self.t, self.e, self.flip, self.flag, self.msg = r, p, s, t, e, flip, flag, msg


def build(base, items, seed=0):
    """-> dict of the oracle's / engine's arrays and the model's view of every item."""
    rng = np.random.default_rng(seed)
    n = len(items)
    N = base.N
    sigs = np.zeros((n, 81), dtype=np.uint8)
    pk = np.zeros((n, 96), dtype=np.uint8)
    inf = np.zeros(n, dtype=np.uint8)
    msgs = []
    r_mult = []
    for i, it in enumerate(items):
        if it.r is None:
            sigs[i, 48] = 0x80
            r_mult.append(None)
        else:
            pt, pi = base.point(it.r)
            x49 = cref.compress(pt, pi)
            sigs[i, :49] = x49
            r = it.r % N
            if it.flag is not None:
                sigs[i, 48] = it.flag
            elif it.flip:
                sigs[i, 48] ^= 0x40
                r = -r % N
            r_mult.append(r)
        if it.p is None:
            inf[i] = 1
        else:
            pk[i], inf[i] = base.point(it.p)
        msgs.append(it.msg if it.msg is not None else bytes(rng.integers(0, 256, 8, dtype=np.uint8)))
    blob, off = pack_msgs(msgs)
    dig = cref.hash_messages(sigs[:, :48], pk, blob, off, cref.default_threads())
    h = [o.scalar_from_digest(bytes(d)) for d in dig]
    s_list = []
    for i, it in enumerate(items):
        if it.t is not None:
            s = (it.t * pow(h[i], -1, Q)) % Q
        elif it.s is not None:
            s = it.s
        else:
            s = int.from_bytes(rng.bytes(32), "little") % Q
        s_list.append(s)
        sigs[i, 49:81] = _le32(it.e % Q)
    rand = np.stack([_le32(s) for s in s_list]) if n else np.zeros((0, 32), dtype=np.uint8)
    # the two MSM points of item i: R_i with s mod q (0 for an identity R), -P_i with s h mod q (0 for an identity key)
    sr = [0 if r is None else s % Q for r, s in zip(r_mult, s_list)]
    sp = [0 if it.p is None else (hh * s) % Q for it, hh, s in zip(items, h, s_list)]
    ra = [0 if r is None else r for r in r_mult]
    pa = [0 if it.p is None else (-it.p) % N for it in items]
    lhs = (sum(a * s for a, s in zip(ra, sr)) + sum(a * s for a, s in zip(pa, sp))) % N
    return dict(base=base, N=N, n=n, sigs=sigs, pk=pk, inf=inf, blob=blob, off=off, rand=rand, h=h, s=s_list,
                ra=ra, sr=sr, pa=pa, sp=sp, lhs=lhs, items=items)


def msm_points(w):
    return list(zip(w["ra"], w["sr"])) + list(zip(w["pa"], w["sp"]))


def model_run(w, form, c=0, T=0):
    """form 'msm' or 'small' -> (lhs multiple, Events, plan (c, K, B, T), MSM points)."""
    if form == "small":
        part, ev = batch_small(list(zip(w["ra"], w["sr"], w["pa"], w["sp"])), w["N"])
        plan = (4, 64, 8, 0)
        npts = 0
    else:
        part, ev, pl = pippenger(msm_points(w), w["N"], c, T)
        plan = (pl["c"], pl["K"], pl["B"], pl["T"])
        npts = 2 * w["n"]
    ev.add("finish", 0, part)          # k_batch_finish: identity + the one partial
    assert part == w["lhs"]
    return part, ev, plan, npts


def oracle(w):
    return cref.verify_batch(w["sigs"], w["pk"], w["inf"], w["blob"], w["off"], w["rand"], cref.default_threads())


def rand_q(rng):
    return int.from_bytes(rng.bytes(32), "little") % Q


# ---- the cases -------------------------------------------------------------------------------------------------------
# Each case: build() -> w, and the forms it runs in: (form, c override, T override, events the model must see).  'small'
# is the block-per-signature form (at most 256 signatures by default), 'msm' the Pippenger pipeline.


def case_rneg_pairs(n, seed):
    """Honest batch with R / -R pairs: a copy of an item with its y flag flipped and the same randomiser.  The R-side
    scalars are equal, so the two R points meet in one bucket of every window and cancel; the challenge hashes x only,
    so the key-side points -P are equal, with equal scalars, and double.  (The copies fail the batch: verdict 2.)"""
    rng = np.random.default_rng(seed)
    base = Base()
    npairs = max(4, n // 50)
    # nonces and keys from pools of 1024 and 256 (the messages differ): fewer points for the oracle to compute
    rs, ps = [rand_q(rng) for _ in range(1024)], [rand_q(rng) for _ in range(256)]
    items = [Item(rs[int(rng.integers(1024))], ps[int(rng.integers(256))], s=rand_q(rng), msg=rng.bytes(8))
             for _ in range(n - npairs)]
    for it, hh in zip(items, build(base, items, seed)["h"]):
        it.e = (it.r - it.p * hh) % Q          # honest: e = r - sk h
    for i in rng.choice(len(items), npairs, replace=False):
        a = items[int(i)]
        items.append(Item(a.r, a.p, s=a.s, e=a.e, flip=True, msg=a.msg))
    return build(base, items, seed)


def _search(make, want, forms, tries=400):
    """The first seed whose case shows every event of `want` in every form: cases on small-order points are dense in
    coincidences, so a short deterministic search finds one."""
    for seed in range(tries):
        w = make(seed)
        if all(want <= model_run(w, f, c, T)[1].seen for f, c, T in forms):
            return w
    raise AssertionError("no seed shows %r" % (want,))


def case_two_torsion():
    """R = T2 (y = 0) with flag 0x00 and 0x40 (both decompress to T2), keys T2 and G + T2, pairs with equal randomisers:
    the doubling of a y = 0 point (identity) in a bucket; in the block form every window point from w = 1 on is O."""
    base = Base(2)                  # B = G + T2, N = 2q; T2 = q B
    rng = np.random.default_rng(2)
    s0, s1 = rand_q(rng), rand_q(rng)
    items = [Item(Q, 1, s=s0, flag=0x00, e=rand_q(rng)), Item(Q, 1, s=s0, flag=0x40, e=rand_q(rng)),
             Item(Q, Q, s=s1, flag=0x00, e=rand_q(rng)), Item(Q, Q, s=s1, flag=0x00, e=rand_q(rng)),
             Item(5, Q, s=rand_q(rng), e=rand_q(rng)), Item(2 * rand_q(rng) + 1, 1, e=rand_q(rng))]
    return build(base, items, 2)


def case_small_order(m, seed):
    """Keys and R of order m (B = T_m) with random scalars.  m = 2: every point is T2, so (lo - 1) running = O for
    every chunk whose running sum is T2."""
    rng = np.random.default_rng(1000 * m + seed)
    base = Base(m, with_g=False)
    items = [Item(int(rng.integers(1, m)), int(rng.integers(1, m)), e=rand_q(rng)) for _ in range(6)]
    return build(base, items, 1000 * m + seed)


HORNER_EVENTS = {("horner", "cancel"), ("horner", "O+W"), ("horner", "equal"), ("horner", "W+O")}
WINDOW_EVENTS = {("ws_acc", "cancel"), ("ws_acc", "equal"), ("ws_lo", "cancel"), ("fold_tree", "cancel"),
                 ("fold_tree", "equal")}
SMALL_EVENTS = {("small_bucket", "equal"), ("small_bucket", "cancel"), ("small_running", "O+W"),
                ("small_agg", "equal"), ("small_term", "cancel"), ("small_reduce_tree", "cancel")}


def case_order29(want, forms):
    """A few items whose points all have order 29: every stage value is a residue mod 29, coincidences are dense."""
    def make(seed):
        rng = np.random.default_rng(29000 + seed)
        base = Base(29, with_g=False)
        items = [Item(int(rng.integers(1, 29)), int(rng.integers(1, 29)), e=rand_q(rng)) for _ in range(8)]
        return build(base, items, 29000 + seed)
    return _search(make, want, forms)


SEGMENT_EVENTS = {("segment", "cross_pair_cancel"), ("segment", "cross_pair_equal"), ("segment", "long_uniform"),
                  ("segment", "long_partials_O")}


def case_segments():
    """At T = 8: pairs R / -R with equal randomisers and identity keys (buckets {Q, -Q} across a segment boundary: the
    fixup adds Q and -Q), pairs of equal R with equal randomisers ({Q, Q}: a doubling), and 300 copies of one point of
    order 29 with one randomiser (buckets of 300 equal entries: k_msm_fixup_long, whose full segments hold equal
    partials), and 301 copies of T2 with one randomiser (long buckets whose full-segment partials are O and whose other
    partials are T2 = -T2: the tree adds O, and opposite points that are also equal).  A few single items give buckets
    of odd size: a pair can then start at the last entry of a segment.  B = T58: order 29 is the even multiples, T2 = 29 B."""
    def make(seed):
        base = Base(58, with_g=False)
        rng = np.random.default_rng(600 + seed)
        items = []
        for j in range(24):
            a, s = 2 * int(rng.integers(1, 29)), rand_q(rng)
            items += [Item(a, None, s=s, e=rand_q(rng)), Item(a, None, s=s, e=rand_q(rng), flip=j % 2 == 0)]
        items += [Item(2 * int(rng.integers(1, 29)), None, e=rand_q(rng)) for _ in range(5)]   # odd bucket sizes
        s = rand_q(rng)
        items += [Item(10, None, s=s, e=rand_q(rng)) for _ in range(300)]
        s = rand_q(rng)
        items += [Item(29, None, s=s, e=rand_q(rng)) for _ in range(301)]
        return build(base, items, 600 + seed)
    return _search(make, SEGMENT_EVENTS, [("msm", 0, 8)])


def case_whole_identity(n, zero_e):
    """Pairs R / -R with equal randomisers and identity keys: lhs = O from cancelling items.  e = 0: rhs = O too."""
    rng = np.random.default_rng(70 + n)
    base = Base()
    items = []
    for _ in range(n // 2):
        r, s = rand_q(rng), rand_q(rng)
        e1, e2 = (0, 0) if zero_e else (rand_q(rng), rand_q(rng))
        items += [Item(r, None, s=s, e=e1), Item(r, None, s=s, e=e2, flip=True)]
    return build(base, items, 70 + n)


def case_partials(n_half, seed):
    """Slice A: pairs R / -R with equal randomisers (its partial is O); slice B: the R of A's pairs negated item by item,
    with A's randomisers (B's partial is minus that of A's first halves)... both over identity keys."""
    rng = np.random.default_rng(seed)
    base = Base()
    a_items, b_items = [], []
    for _ in range(n_half // 2):
        r, s = rand_q(rng), rand_q(rng)
        a_items += [Item(r, None, s=s, e=rand_q(rng)), Item(r, None, s=s, e=rand_q(rng), flip=True)]
    for _ in range(n_half):
        r, s = rand_q(rng), rand_q(rng)
        b_items += [Item(r, None, s=s, e=rand_q(rng))]
    c_items = [Item(it.r, None, s=it.s, e=rand_q(rng), flip=True) for it in b_items]
    return build(base, a_items + b_items + c_items, seed), len(a_items), len(b_items)


LARGE = 1 << 16


def case_registered(kind, seed=10, n_large=LARGE):
    """Keys P, -P, 2P (honest, order q) registered; the items' key-side scalars t_i = s_i h_i chosen per key.
    -> (w over the gathered records, key list multiples, key index per item)."""
    rng = np.random.default_rng(seed)
    base = Base()
    p = rand_q(rng)
    keys = [p, (-p) % Q, (2 * p) % Q]
    ts = {0: [], 1: [], 2: []}
    if kind == "cancel":            # c_P == c_{-P}: the terms -c P and c P cancel
        c = rand_q(rng)
        ts[0] = [rand_q(rng) for _ in range(5)]
        ts[0].append((c - sum(ts[0])) % Q)
        ts[1] = [rand_q(rng) for _ in range(3)]
        ts[1].append((c - sum(ts[1])) % Q)
        ts[2] = [rand_q(rng) for _ in range(4)]
    elif kind == "double":          # c_{2P} 2P == c_P P: equal terms (no item on -P, whose term would come between)
        c = rand_q(rng)
        ts[0] = [c]
        ts[2] = [rand_q(rng) for _ in range(2)]
        ts[2].append((c * pow(2, -1, Q) - sum(ts[2])) % Q)
    elif kind == "zero":            # sums of exactly q and 2q: c = 0 with non-zero columns; c = q - 1; 3 (q - 1) >= 2^256
        a = rand_q(rng)
        ts[0] = [a, Q - a]
        b1, b2 = rand_q(rng), rand_q(rng)
        while b1 + b2 <= Q:
            b1, b2 = rand_q(rng), rand_q(rng)
        ts[1] = [b1, b2, 2 * Q - b1 - b2]
        ts[2] = [Q - 1, Q - 1, Q - 1, 2]   # 3q - 1: c = q - 1, and the sum needs hi
    elif kind == "large":           # 2^16 items of t = q - 1 on one key: columns far beyond 32 bits, the carry into hi
        ts[0] = [Q - 1] * n_large
        ts[1] = [rand_q(rng) for _ in range(7)]
        ts[2] = [Q - 1, Q - 1]
    items, idx = [], []
    for k in (0, 1, 2):
        for j, t in enumerate(ts[k]):
            # the many items of "large" carry the identity R: the case is about the key side, and their R points
            # would only cost the oracle time
            r = None if kind == "large" and k == 0 and j >= 8 else rand_q(rng)
            items.append(Item(r, keys[k], t=t, e=rand_q(rng)))
            idx.append(k)
    order = rng.permutation(len(items))
    items = [items[i] for i in order]
    idx = np.array([idx[i] for i in order], dtype=np.uint32)
    w = build(base, items, seed)
    return w, keys, idx


def model_registered(w, keys, idx):
    """The aggregated form: the MSM over the n points R_i, the key side per key, k_partial_add -> (lhs, Events, plan)."""
    N = w["N"]
    part, ev, pl = pippenger(list(zip(w["ra"], w["sr"])), N)
    key_t = [[] for _ in keys]
    for i, k in enumerate(idx):
        key_t[int(k)].append(w["sp"][i])
    kp = key_terms(ev, keys, key_t, N)
    tot = ev.add("partial_add", part, kp)
    ev.add("finish", 0, tot)
    assert tot == w["lhs"]
    return tot, ev, (pl["c"], pl["K"], pl["B"], pl["T"])


REGISTERED_EVENTS = {
    "cancel": {("key_block", "cancel")},
    "double": {("key_block", "equal")},
    "zero": {("key_sum", "c_zero_nonzero_columns"), ("key_sum", "c_q_minus_1"), ("key_sum", "hi")},
    "large": {("key_sum", "hi")},
}


MULTI_MIN_PER_SHARD = 4096   # multi.cuh: shards get whole 128-signature blocks, at least this many signatures each


def case_two_shards():
    """8192 signatures for a two-device engine, which gives each device 4096 (multi_slices, multi.cuh:23-31).  Shard 0:
    pairs R / -R with equal randomisers and identity keys, so its partial is O; shard 1: items over small pools of R and
    keys with random randomisers and e.  -> (w, size of shard 0)."""
    rng = np.random.default_rng(90)
    base = Base()
    items = []
    for _ in range(MULTI_MIN_PER_SHARD // 2):
        r, s = rand_q(rng), rand_q(rng)
        items += [Item(r, None, s=s, e=rand_q(rng)), Item(r, None, s=s, e=rand_q(rng), flip=True)]
    rs, ps = [rand_q(rng) for _ in range(64)], [rand_q(rng) for _ in range(64)]
    items += [Item(rs[int(rng.integers(64))], ps[int(rng.integers(64))], e=rand_q(rng)) for _ in range(MULTI_MIN_PER_SHARD)]
    return build(base, items, 90), MULTI_MIN_PER_SHARD


def subset(w, idx):
    """The case restricted to the items idx (in order), with the model's view of them."""
    idx = [int(i) for i in idx]
    msgs = [bytes(w["blob"][int(w["off"][i]):int(w["off"][i + 1])]) for i in idx]
    blob, off = pack_msgs(msgs)
    out = dict(w, n=len(idx), blob=blob, off=off, items=[w["items"][i] for i in idx])
    for k in ("sigs", "pk", "inf", "rand"):
        out[k] = w[k][idx]
    for k in ("h", "s", "ra", "sr", "pa", "sp"):
        out[k] = [w[k][i] for i in idx]
    N = w["N"]
    out["lhs"] = (sum(a * b for a, b in zip(out["ra"], out["sr"])) + sum(a * b for a, b in zip(out["pa"], out["sp"]))) % N
    return out


CLEAN, TORSION_EVEN, TORSION_ODD, ZERO_RAND, WRONG_E = range(5)


def case_torsion_culprits(n, density, seed, n_keys=16):
    """Honest items (keys from a pool of n_keys), and every `density`-th item a culprit, in turn: a wrong e (WRONG_E), a
    torsion-shifted nonce point R' = r G + T2 with e = r - sk h' (D_i = T2) and an even randomiser (TORSION_EVEN), a
    wrong e with randomiser 0 (ZERO_RAND); and exactly one R' with an odd randomiser (TORSION_ODD).  The item's own term
    s_i D_i is O for TORSION_EVEN and ZERO_RAND, so only WRONG_E and TORSION_ODD items can make the batch fail.
    -> (w, kind per item, key multiples of the pool, key index per item)."""
    rng = np.random.default_rng(seed)
    base = Base(2)                  # B = G + T2, N = 2q: a G is the multiple congruent to a mod q and to 0 mod 2

    def g_mult(a):
        a %= Q
        return a if a % 2 == 0 else a + Q
    pool = [g_mult(rand_q(rng)) for _ in range(n_keys)]
    kinds = [CLEAN] * n
    for j, i in enumerate(range(density // 2, n, density)):
        kinds[i] = (WRONG_E, TORSION_EVEN, ZERO_RAND)[j % 3]
    kinds[density // 2 + density * 4 + 1] = TORSION_ODD
    idx = rng.integers(0, n_keys, n).astype(np.uint32)
    items = []
    for i in range(n):
        s = rand_q(rng)
        if kinds[i] == TORSION_EVEN:
            s -= s % 2
        elif kinds[i] == TORSION_ODD:
            s |= 1
        elif kinds[i] == ZERO_RAND:
            s = 0
        r = g_mult(rand_q(rng)) + (Q if kinds[i] in (TORSION_EVEN, TORSION_ODD) else 0)
        items.append(Item(r, pool[idx[i]], s=s, msg=rng.bytes(8)))
    for it, hh, kd in zip(items, build(base, items, seed)["h"], kinds):
        it.e = (it.r - it.p * hh + (1 if kd in (ZERO_RAND, WRONG_E) else 0)) % Q    # honest: e = r - sk h (mod q)
    return build(base, items, seed), np.array(kinds), pool, idx


def oracle_item(w, i):
    """The oracle of test_gpu_locate.py for "item i is bad": the one-item batch {i} with its own randomiser."""
    off = np.array([0, int(w["off"][i + 1] - w["off"][i])], dtype=np.uint64)
    blob = w["blob"][int(w["off"][i]):int(w["off"][i + 1])]
    return cref.verify_batch(w["sigs"][i:i + 1], w["pk"][i:i + 1], w["inf"][i:i + 1], blob, off, w["rand"][i:i + 1], 1)[0]


# ---- CPU checks of the model and the cases ---------------------------------------------------------------------------
def _check(w, form, c=0, T=0, want=()):
    lhs, ev, plan, npts = model_run(w, form, c, T)
    v, l97, r97 = oracle(w)
    assert (l97 == w["base"].lhs97(lhs)).all(), "the model's lhs is the oracle's"
    missing = set(want) - ev.seen
    assert not missing, missing
    return v, ev


def test_torsion_points_have_the_stated_orders():
    for m in TORSION_ORDERS:
        torsion(m)
    # 5 divides the cofactor, but the KAT point has no component of order 5
    t, ti = _mul(KAT96, 0, o.COFACTOR // 5)
    assert _mul(t, ti, Q)[1] == 1


def test_plan_and_digits_restate_the_device():
    assert msm_plan(600) == (8, 32, 128, 8, 16)
    assert msm_plan(1 << 20)[0] != 8
    assert msm_plan(10, 13) == (13, 20, 4096, 8, 512)
    assert segment_len(600, 32) == 8 and segment_len(600, 32, 8) == 8
    for s in (0, 1, Q - 1, 2**255 + 12345, 0x8888888888):
        for c in (4, 5, 7, 8, 13, 16):
            K = (256 + c - 1) // c
            assert sum((-b if neg else b) << (k * c) for k, (b, neg) in enumerate(msm_digits(s, c, K))) == s
        assert sum(d << (4 * i) for i, d in enumerate(recode_signed_w4(s % Q))) == s % Q


@pytest.mark.parametrize("n", [300, 5000])
def test_rneg_pairs(n):
    w = case_rneg_pairs(n, n)
    v, _ = _check(w, "msm", want={("bucket", "has_opposite"), ("bucket", "has_equal")})
    assert v == 2
    if n <= 300:
        _check(w, "small")


def test_two_torsion():
    w = case_two_torsion()
    _check(w, "msm", want={("bucket", "pair_equal")})
    _check(w, "small", want={("small_window", "O")})


@pytest.mark.parametrize("m", [2, 29, 58, 181])
def test_small_order(m):
    w = case_small_order(m, 0)
    _check(w, "msm", want={("ws_mul", "small_order")} if m == 2 else ())
    _check(w, "small", want={("small_window", "O")} if m == 2 else {("small_bucket", "equal")})


HORNER_C = [0, 4, 5, 7, 13, 16]


@pytest.mark.parametrize("c", HORNER_C)
def test_horner(c):
    w = case_order29(HORNER_EVENTS, [("msm", c, 0)])
    _check(w, "msm", c, want=HORNER_EVENTS)


def test_window_sum_and_fold():
    w = case_order29(WINDOW_EVENTS, [("msm", 0, 0)])
    _check(w, "msm", want=WINDOW_EVENTS)


def test_block_form_events():
    w = case_order29(SMALL_EVENTS, [("small", 0, 0)])
    _check(w, "small", want=SMALL_EVENTS)


def test_segments():
    w = case_segments()
    _check(w, "msm", 0, 8, want=SEGMENT_EVENTS)


@pytest.mark.parametrize("n,zero_e,verdict", [(8, True, 0), (8, False, 2), (300, True, 0)])
def test_whole_batch_identity(n, zero_e, verdict):
    w = case_whole_identity(n, zero_e)
    assert w["lhs"] == 0
    for form in ("small", "msm"):
        v, ev = _check(w, form, want={("finish", "O+O")})
        assert v == verdict


def test_partials():
    w, na, nb = case_partials(64, 9)
    sl = [slice(0, na), slice(na, na + 2 * nb)]
    N = w["N"]
    part = [sum(w["ra"][i] * w["sr"][i] for i in range(s.start, s.stop)) % N for s in sl]
    assert part[0] == 0 and part[1] == 0
    b_part = sum(w["ra"][i] * w["sr"][i] for i in range(na, na + nb)) % N
    c_part = sum(w["ra"][i] * w["sr"][i] for i in range(na + nb, na + 2 * nb)) % N
    assert b_part and (b_part + c_part) % N == 0
    _check(w, "msm")


@pytest.mark.parametrize("kind", ["cancel", "double", "zero"])
def test_registered_key_side(kind):
    w, keys, idx = case_registered(kind)
    lhs, ev, _ = model_registered(w, keys, idx)
    _, l97, _ = oracle(w)
    assert (l97 == w["base"].lhs97(lhs)).all()
    assert REGISTERED_EVENTS[kind] <= ev.seen, REGISTERED_EVENTS[kind] - ev.seen


def test_registered_large_columns_carry_into_hi():
    """The GPU file's 2^16 items of t = q - 1 on one key, at 2^12 items here (CPU time): the same carry into hi."""
    w, keys, idx = case_registered("large", n_large=1 << 12)
    lhs, ev, _ = model_registered(w, keys, idx)
    assert (oracle(w)[1] == w["base"].lhs97(lhs)).all()
    assert REGISTERED_EVENTS["large"] <= ev.seen
    assert sum(w["sp"][i] for i in range(w["n"]) if idx[i] == 0) >> 256 > 1 << 10


def test_registered_set_with_a_torsion_key():
    """A set holding a torsion key runs the per-signature pipeline on the gathered records: 2n MSM points."""
    assert not cref.is_torsion_free(np.frombuffer(torsion(29), dtype=np.uint8))
    w, _, _ = case_registered("cancel")
    assert w["n"] <= 256
    _, _, _, npts = model_run(w, "msm")
    assert npts == 2 * w["n"]
    _check(w, "msm")


def test_two_shards_one_partial_identity():
    w, n0 = case_two_shards()
    assert w["n"] == 2 * n0 and n0 % 128 == 0
    N = w["N"]
    part0 = sum(w["ra"][i] * w["sr"][i] + w["pa"][i] * w["sp"][i] for i in range(n0)) % N
    part1 = sum(w["ra"][i] * w["sr"][i] + w["pa"][i] * w["sp"][i] for i in range(n0, w["n"])) % N
    assert part0 == 0 and part1 != 0
    assert (oracle(w)[1] == w["base"].lhs97(w["lhs"])).all()


LOCATE_SIZES = [(400, 40), (5120, 40)]   # 5120 > LOCATE_LEAF (batch.cuh): the bisection runs before the per-item pass


@pytest.mark.parametrize("n,density", LOCATE_SIZES)
def test_torsion_culprits_batch_semantics(n, density):
    w, kinds, _, _ = case_torsion_culprits(n, density, n)
    assert sorted(set(kinds)) == [CLEAN, TORSION_EVEN, TORSION_ODD, ZERO_RAND, WRONG_E]
    assert (kinds == TORSION_ODD).sum() == 1
    v, l97, _ = oracle(w)
    assert v == 2 and (l97 == w["base"].lhs97(w["lhs"])).all()
    step = 1 if n <= 400 else 11
    for i in range(0, w["n"], step):
        if kinds[i] != CLEAN or i % 37 == 0:
            assert oracle_item(w, i) == (2 if kinds[i] in (TORSION_ODD, WRONG_E) else 0), (i, kinds[i])
    # without the items that can fail the batch, the torsion-shifted ones with even randomisers pass as a batch
    ok = subset(w, np.nonzero(np.isin(kinds, [CLEAN, TORSION_EVEN, ZERO_RAND]))[0])
    v, l97, _ = oracle(ok)
    assert v == 0 and (l97 == ok["base"].lhs97(ok["lhs"])).all()
