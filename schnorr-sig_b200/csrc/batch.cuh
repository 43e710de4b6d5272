// Random-linear-combination batch verification (reference src/batch.rs:31-130) as a Pippenger
// bucket multi-scalar multiplication.  Included by schnorr_b200.cu (single translation unit).
//
//   check   sum s_i R_i - sum (s_i h_i) P_i == (sum s_i e_i) G      (x-only, src/batch.rs:121-129)
//
//   k_batch_prepare   K3: per signature: challenge hash, h_i mod q, s_i e_i, s_i h_i, decompress R_i,
//                     negate P_i -> 2n affine points + 2n scalars
//   k_msm_count / k_msm_scatter   signed c-bit digits -> counting sort of point indices by bucket
//   k_msm_segment_sum fixed-size segments of the sorted list per thread, mixed additions; buckets that
//                     straddle segments are completed by k_msm_segment_fixup (robust to skewed buckets)
//   k_msm_window_sum  running-sum reduction of bucket chunks + chunk offsets
//   k_msm_window_fold per-window total: one warp per window, warp-shuffle tree of point additions
//   k_msm_horner      sum_k 2^(ck) W_k  -> one Jacobian partial per GPU
//   k_batch_finish    adds the per-GPU partials, (sum lin) * G, x-only comparison
// The bucket sums are order-independent group elements, so the atomics-based (non-deterministic)
// slot assignment inside a bucket does not affect the bit-exact result.
#pragma once

struct msm_plan {
    int c;        // window bits
    int K;        // windows
    int B;        // buckets per window = 2^(c-1), ids 1..B
    int chunks;   // threads per window in the window-sum stage
    int chunk_sz; // buckets per chunk
};

static msm_plan msm_make_plan(size_t npoints, int c_override = 0) {
    double best = 1e300;
    msm_plan p{};
    for (int c = 4; c <= 16; c++) {
        int K = (256 + c - 1) / c;
        double B = (double)(1u << (c - 1));
        double cost = (double)npoints * K + 3.0 * K * B;
        if (cost < best) {
            best = cost;
            p.c = c;
            p.K = K;
            p.B = 1 << (c - 1);
        }
    }
    // Small batches are latency-bound (one launch chain, the Horner tail is serial): 8-bit windows -- 32 Horner additions
    // instead of the 52-64 of the work-optimal 4-5 bits -- measured best for 4..4096 signatures (tools/small_batch_c_scan.py)
    if (npoints <= 8192) {
        p.c = 8;
        p.K = 32;
        p.B = 128;
    }
    if (c_override >= 4 && c_override <= 16) {  // schnorr_b200_set_msm_geometry (tests): force the window width
        p.c = c_override;
        p.K = (256 + p.c - 1) / p.c;
        p.B = 1 << (p.c - 1);
    }
    // bucket-reduction chunks: aim at ~8k chunk threads in total (short serial chains), 8..32 buckets each
    int want = (int)(((double)p.B * p.K) / 8192.0);
    p.chunk_sz = want >= 32 ? 32 : (want >= 16 ? 16 : 8);
    if (p.chunk_sz > p.B) p.chunk_sz = p.B;
    p.chunks = p.B / p.chunk_sz;
    return p;
}

// ---- K3 ----------------------------------------------------------------------------------------
// pts: 2n affine points as 12 x u64 (x||y); scalars: 2n x 8 x u32; lin: n scalars s_i e_i
__global__ void __launch_bounds__(128, 4) k_batch_prepare(soa_batch in, const uint8_t* __restrict__ msgs,
                                                       const uint64_t* __restrict__ msg_off,
                                                       const uint8_t* __restrict__ rand32, uint64_t* __restrict__ pts,
                                                       uint32_t* __restrict__ scalars, uint32_t* __restrict__ lin,
                                                       int* __restrict__ bad, const uint32_t* __restrict__ h_in) {
    size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    size_t n = in.n;
    bool live = t < n;
    // threads past the end of the batch redo the block's first item (which always exists) and store nothing: every thread
    // of the block then reaches the barriers of the permutation
    size_t i = live ? t : (size_t)blockIdx.x * blockDim.x;
    uint64_t off = msg_off[i], len = msg_off[i + 1] - off;
    // h_in != nullptr: the challenges were computed by k_batch_challenge_dist (small batches)
    hash_vote hv = block_hash_vote(!h_in ? hash_message_permutations(len) : -1, off, len);
    uint8_t fl = in.flags[i];
    fp6 sx = load_fp6_planes(in.planes, 0, n, i);
    scalar e = load_scalar_planes(in.planes, 3, n, i);
    fp6 px = load_fp6_planes(in.planes, 5, n, i);
    fp6 py = load_fp6_planes(in.planes, 8, n, i);
    bool pk_inf = fl & FL_PK_INF;
    bool ok = !(fl & (FL_MALFORMED | FL_X_BAD));
    scalar s = sc_from_u256(sc_load_le(rand32 + 32 * i));
    scalar s_r = sc_zero(), s_p = sc_zero(), l = sc_zero();
    fp6 rx = fp6_zero(), ry = fp6_zero();
    bool r_inf = true;
    if (ok) ok = decompress_point(sx, in.sig_flag[i], rx, ry, r_inf);  // unwrap panic, src/batch.rs:104
    // every thread hashes (a malformed item's digest is simply unused): the permutation barriers stay matched,
    // and the barrier at its start re-aligns the warps after the divergent square-root loops
    scalar h;
    if (h_in) {
#pragma unroll
        for (int k = 0; k < 8; k++) h.l[k] = h_in[i * 8 + k];
    } else {
        h = challenge_scalar(sx, px, py, pk_inf, msgs + off, len, hv.sync);
    }
    if (!live) return;
    if (ok) {
        l = sc_mul(s, e);                     // src/batch.rs:92-97
        s_r = r_inf ? sc_zero() : s;          // identity contributes nothing
        s_p = pk_inf ? sc_zero() : sc_mul(h, s);  // src/batch.rs:109-111
    }
    if (!ok) atomicOr(bad, 1);
    fp6 npy = fp6_neg(py);  // src/batch.rs:106
    uint64_t* o = pts + i * 12;
    uint64_t* o2 = pts + (n + i) * 12;
#pragma unroll
    for (int k = 0; k < 6; k++) {
        o[k] = rx.c[k];
        o[6 + k] = ry.c[k];
        o2[k] = px.c[k];
        o2[6 + k] = npy.c[k];
    }
#pragma unroll
    for (int k = 0; k < 8; k++) {
        scalars[i * 8 + k] = s_r.l[k];
        scalars[(n + i) * 8 + k] = s_p.l[k];
        lin[i * 8 + k] = l.l[k];
    }
}

// Challenges of a SMALL batch: one signature per group of six lanes (dist.cuh) -- the hash is two thirds of the serial
// latency of k_batch_prepare, and a batch of a few thousand signatures cannot hide it behind other warps.
__global__ void __launch_bounds__(DIST_THREADS) k_batch_challenge_dist(soa_batch in, const uint8_t* __restrict__ msgs,
                                                                       const uint64_t* __restrict__ msg_off,
                                                                       uint32_t* __restrict__ h_out) {
    __shared__ uint32_t s_mds2[24];
    if (threadIdx.x < 24) s_mds2[threadIdx.x] = c_mds_row[threadIdx.x % 12];
    __syncthreads();
    int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int g = lane / 6, k = lane % 6;
    if (g >= 5) return;
    size_t n = in.n;
    size_t i = ((size_t)blockIdx.x * (DIST_THREADS / 32) + warp) * 5 + g;
    if (i >= n) return;
    int gbase = 6 * g;
    unsigned mask = 0x3fu << gbase;
    bool pk_inf = in.flags[i] & FL_PK_INF;  // the identity key hashes as x = y = 0 (challenge_scalar)
    const uint64_t* pl = reinterpret_cast<const uint64_t*>(in.planes);
    fp_t sx = pl[((size_t)(0 + (k >> 1)) * n + i) * 2 + (k & 1)];
    fp_t px = pk_inf ? 0 : pl[((size_t)(5 + (k >> 1)) * n + i) * 2 + (k & 1)];
    fp_t py = pk_inf ? 0 : pl[((size_t)(8 + (k >> 1)) * n + i) * 2 + (k & 1)];
    uint64_t off = msg_off[i];
    scalar h = dchallenge_scalar(mask, sx, px, py, msgs + off, msg_off[i + 1] - off, k, gbase, s_mds2);
    if (k == 0) {
#pragma unroll
        for (int j = 0; j < 8; j++) h_out[i * 8 + j] = h.l[j];
    }
}

// sum of m scalars mod q: each block writes one partial into out[blockIdx.x]
__global__ void __launch_bounds__(256) k_scalar_sum(const uint32_t* __restrict__ in, size_t m, uint32_t* __restrict__ out) {
    __shared__ uint32_t sh[256 * 8];
    scalar acc = sc_zero();
    for (size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x; j < m; j += (size_t)gridDim.x * blockDim.x) {
        scalar v;
#pragma unroll
        for (int k = 0; k < 8; k++) v.l[k] = in[j * 8 + k];
        acc = sc_add(acc, v);
    }
#pragma unroll
    for (int k = 0; k < 8; k++) sh[threadIdx.x * 8 + k] = acc.l[k];
    __syncthreads();
    for (int stride = 128; stride > 0; stride >>= 1) {
        if ((int)threadIdx.x < stride) {
            scalar a, b;
#pragma unroll
            for (int k = 0; k < 8; k++) {
                a.l[k] = sh[threadIdx.x * 8 + k];
                b.l[k] = sh[(threadIdx.x + stride) * 8 + k];
            }
            a = sc_add(a, b);
#pragma unroll
            for (int k = 0; k < 8; k++) sh[threadIdx.x * 8 + k] = a.l[k];
        }
        __syncthreads();
    }
    if (threadIdx.x < 8) out[blockIdx.x * 8 + threadIdx.x] = sh[threadIdx.x];
}

// ---- K4: Pippenger ---------------------------------------------------------------------------
// signed digit of window k given the running carry; returns bucket id (0 = none) and sign
__device__ __forceinline__ int msm_digit(const scalar& s, int k, int c, int& carry, bool& neg) {
    int raw = (int)sc_bits(s, k * c, c) + carry;
    int half = 1 << (c - 1);
    neg = raw > half;
    carry = neg ? 1 : 0;
    return neg ? (1 << c) - raw : raw;
}

__global__ void __launch_bounds__(256) k_msm_count(const uint32_t* __restrict__ scalars, size_t npts, msm_plan pl,
                                                   uint32_t* __restrict__ counts) {
    size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= npts) return;
    scalar s;
#pragma unroll
    for (int k = 0; k < 8; k++) s.l[k] = scalars[j * 8 + k];
    int carry = 0;
    for (int k = 0; k < pl.K; k++) {
        bool neg;
        int b = msm_digit(s, k, pl.c, carry, neg);
        if (b) atomicAdd(&counts[(size_t)k * (pl.B + 1) + b], 1u);
    }
}

// Exclusive scan of m counters (m = windows x (buckets + 1), up to a few million) in two grid-wide passes:
//   k_scan_local   every block scans its tile of SCAN_TILE counters in place (exclusive, relative to the tile) and
//                  records the tile total
//   k_scan_offsets every block adds the sum of the totals of the tiles before it (<= a few hundred values: one
//                  strided sum + a block reduction) to its tile
// (the single-block version took 82 us of a 3 ms batch at 2^16 signatures.)
static constexpr int SCAN_THREADS = 256;
static constexpr int SCAN_PER_THREAD = 8;
static constexpr int SCAN_TILE = SCAN_THREADS * SCAN_PER_THREAD;
__global__ void __launch_bounds__(SCAN_THREADS) k_scan_local(const uint32_t* __restrict__ counts, size_t m,
                                                             uint32_t* __restrict__ offsets, uint32_t* __restrict__ tile_total) {
    __shared__ uint32_t sh[SCAN_THREADS];
    size_t base = (size_t)blockIdx.x * SCAN_TILE + (size_t)threadIdx.x * SCAN_PER_THREAD;
    uint32_t v[SCAN_PER_THREAD], sum = 0;
#pragma unroll
    for (int k = 0; k < SCAN_PER_THREAD; k++) {
        v[k] = base + k < m ? counts[base + k] : 0;
        sum += v[k];
    }
    sh[threadIdx.x] = sum;
    __syncthreads();
    for (int d = 1; d < SCAN_THREADS; d <<= 1) {  // Hillis-Steele inclusive scan of the per-thread sums
        uint32_t t = (int)threadIdx.x >= d ? sh[threadIdx.x - d] : 0;
        __syncthreads();
        sh[threadIdx.x] += t;
        __syncthreads();
    }
    uint32_t run = sh[threadIdx.x] - sum;
#pragma unroll
    for (int k = 0; k < SCAN_PER_THREAD; k++) {
        if (base + k < m) offsets[base + k] = run;
        run += v[k];
    }
    if (threadIdx.x == SCAN_THREADS - 1) tile_total[blockIdx.x] = sh[threadIdx.x];
}
__global__ void __launch_bounds__(SCAN_THREADS) k_scan_offsets(size_t m, uint32_t* __restrict__ offsets,
                                                               const uint32_t* __restrict__ tile_total) {
    __shared__ uint32_t sh[SCAN_THREADS];
    uint32_t part = 0;
    for (unsigned t = threadIdx.x; t < blockIdx.x; t += SCAN_THREADS) part += tile_total[t];
    sh[threadIdx.x] = part;
    __syncthreads();
    for (int d = SCAN_THREADS / 2; d > 0; d >>= 1) {
        if ((int)threadIdx.x < d) sh[threadIdx.x] += sh[threadIdx.x + d];
        __syncthreads();
    }
    uint32_t add = sh[0];
    size_t base = (size_t)blockIdx.x * SCAN_TILE + (size_t)threadIdx.x * SCAN_PER_THREAD;
#pragma unroll
    for (int k = 0; k < SCAN_PER_THREAD; k++)
        if (base + k < m) offsets[base + k] += add;
}

__global__ void __launch_bounds__(256) k_msm_scatter(const uint32_t* __restrict__ scalars, size_t npts, msm_plan pl,
                                                     const uint32_t* __restrict__ offsets, uint32_t* __restrict__ cursor,
                                                     uint32_t* __restrict__ sorted) {
    size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= npts) return;
    scalar s;
#pragma unroll
    for (int k = 0; k < 8; k++) s.l[k] = scalars[j * 8 + k];
    int carry = 0;
    for (int k = 0; k < pl.K; k++) {
        bool neg;
        int b = msm_digit(s, k, pl.c, carry, neg);
        if (b) {
            size_t slot = (size_t)k * (pl.B + 1) + b;
            uint32_t pos = offsets[slot] + atomicAdd(&cursor[slot], 1u);
            sorted[pos] = (uint32_t)j | (neg ? 0x80000000u : 0u);
        }
    }
}

__device__ __forceinline__ void load_affine(const uint64_t* __restrict__ pts, size_t j, fp6& x, fp6& y) {
    const ulonglong2* p = reinterpret_cast<const ulonglong2*>(pts + j * 12);
    ulonglong2 a = p[0], b = p[1], c = p[2], d = p[3], e = p[4], f = p[5];
    x = fp6{{a.x, a.y, b.x, b.y, c.x, c.y}};
    y = fp6{{d.x, d.y, e.x, e.y, f.x, f.y}};
}

// Bucket accumulation by fixed-size SEGMENTS of the sorted list (robust to skewed bucket sizes: the
// sparse top window, repeated randomisers, adversarial scalars).  Thread t owns positions
// [t*T, (t+1)*T) of `sorted`; it walks them bucket by bucket.  A bucket that lies entirely inside
// the segment is written directly (sole writer); a bucket that crosses a segment boundary leaves a
// partial sum (head: the bucket began before the segment; tail: it continues after) that
// k_msm_segment_fixup adds up.  Empty buckets keep the zero fill (Z = 0 = identity).
struct seg_partial {
    jac_pt pt;
    int32_t slot;  // -1 = unused
    int32_t pad[3];
};
__device__ __forceinline__ size_t bucket_of_slot(const msm_plan& pl, uint32_t slot) {
    uint32_t k = slot / (uint32_t)(pl.B + 1), b = slot % (uint32_t)(pl.B + 1);
    return (size_t)k * pl.B + (b - 1);
}
// (X, Y, w) is a Jacobian point with Z = w in Fp: the arrays between the MSM stages hold jac_pt records whose Z has
// only its first coefficient set (identity: w = 0)
__device__ __forceinline__ void store_jf_as_jac(jac_pt* out, const jf_pt& p) {
    out->X = p.X;
    out->Y = p.Y;
    out->Z = fp6{{p.w, 0, 0, 0, 0, 0}};
}
__device__ __forceinline__ jf_pt load_jac_as_jf(const jac_pt* in) {
    jf_pt r;
    r.X = in->X;
    r.Y = in->Y;
    r.w = in->Z.c[0];
    return r;
}
__device__ __forceinline__ jf_pt jf_identity() { return jf_pt{fp6_one(), fp6_one(), 0}; }
__global__ void __launch_bounds__(128, 3) k_msm_segment_sum(const uint64_t* __restrict__ pts, msm_plan pl, uint32_t nslots,
                                                         uint32_t T, const uint32_t* __restrict__ offsets,
                                                         const uint32_t* __restrict__ counts,
                                                         const uint32_t* __restrict__ sorted, jac_pt* __restrict__ buckets,
                                                         seg_partial* __restrict__ parts /*[nseg][2]*/) {
    size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t M = offsets[nslots - 1] + counts[nslots - 1];
    uint64_t lo64 = (uint64_t)t * T;
    parts[2 * t + 0].slot = -1;
    parts[2 * t + 1].slot = -1;
    if (lo64 >= M) return;
    uint32_t lo = (uint32_t)lo64, hi = lo + T < M ? lo + T : M;
    // last slot whose offset is <= lo
    uint32_t a = 0, b = nslots;  // invariant: offsets[a] <= lo < offsets[b] (b = nslots: +inf)
    while (b - a > 1) {
        uint32_t m = (a + b) >> 1;
        if (offsets[m] <= lo) a = m; else b = m;
    }
    uint32_t s = a, beg_s = offsets[s], end_s = beg_s + counts[s];
    // the running bucket sum lives in (X, Y, w) coordinates with w in Fp (affine.cuh): an addition of an affine point
    // is 2M + 1S + cofactor + scalings instead of the 7M + 4S of a Jacobian mixed addition; (X, Y, w) IS a Jacobian
    // point with Z = w, which is how the later stages read it (identity: w = 0)
    jf_pt acc, tp;
    acc.X = fp6_one();
    acc.Y = fp6_one();
    acc.w = 0;
    tp.w = 1;
    for (uint32_t pos = lo; pos < hi; pos++) {
        if (pos >= end_s) {
            // flush bucket s (it ended inside this segment) and move to the bucket holding pos
            if (beg_s >= lo) store_jf_as_jac(&buckets[bucket_of_slot(pl, s)], acc);          // complete: began and ended here
            else { store_jf_as_jac(&parts[2 * t + 0].pt, acc); parts[2 * t + 0].slot = (int32_t)s; }   // head partial
            acc.w = 0;
            do { s++; beg_s = offsets[s]; end_s = beg_s + counts[s]; } while (pos >= end_s);
        }
        uint32_t v = sorted[pos];
        load_affine(pts, v & 0x7fffffffu, tp.X, tp.Y);
        jf_madd_exact(&acc, &tp, (v >> 31) != 0);
    }
    bool began_here = beg_s >= lo, ends_here = end_s <= hi;
    if (began_here && ends_here) store_jf_as_jac(&buckets[bucket_of_slot(pl, s)], acc);
    else if (!began_here) { store_jf_as_jac(&parts[2 * t + 0].pt, acc); parts[2 * t + 0].slot = (int32_t)s; }   // head (maybe whole segment)
    else { store_jf_as_jac(&parts[2 * t + 1].pt, acc); parts[2 * t + 1].slot = (int32_t)s; }                     // tail
}
// one thread per slot: buckets that straddle segment boundaries are the sum of their partials
static constexpr uint32_t MSM_LONG_SPAN = 16;  // segments; longer buckets go to k_msm_fixup_long
__global__ void __launch_bounds__(128) k_msm_segment_fixup(msm_plan pl, uint32_t nslots, uint32_t T,
                                                           const uint32_t* __restrict__ offsets,
                                                           const uint32_t* __restrict__ counts,
                                                           const seg_partial* __restrict__ parts, jac_pt* __restrict__ buckets,
                                                           uint32_t* __restrict__ long_list, uint32_t* __restrict__ long_count) {
    uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= nslots) return;
    uint32_t cnt = counts[s];
    if (cnt == 0) return;
    uint32_t beg = offsets[s], end = beg + cnt;
    uint32_t sa = beg / T, sb = (end - 1) / T;
    if (sa == sb) return;  // written directly by its segment
    if (sb - sa >= MSM_LONG_SPAN) {  // a bucket spanning many segments (sparse top window, repeated randomisers,
        long_list[atomicAdd(long_count, 1u)] = s;  // adversarial scalars): summed by a whole block, below
        return;
    }
    jf_pt acc = jf_identity();
    for (uint32_t g = sa; g <= sb; g++) {
#pragma unroll 1
        for (int w = 0; w < 2; w++) {
            const seg_partial* p = &parts[2 * (size_t)g + w];
            if (p->slot == (int32_t)s) {
                jf_pt t = load_jac_as_jf(&p->pt);
                jf_add_exact(&acc, &t);
            }
        }
    }
    store_jf_as_jac(&buckets[bucket_of_slot(pl, s)], acc);
}

// Buckets that span >= MSM_LONG_SPAN segments: one BLOCK per bucket.  The threads sum the partial records strided,
// then a warp-shuffle tree and a last step through shared memory fold the 128 running sums -- a bucket holding a
// quarter of all points (3-bit top window) costs ~25 serial additions instead of thousands.
__device__ __forceinline__ jf_pt shfl_down_jf(const jf_pt& p, int delta);
static constexpr int FIXUP_LONG_THREADS = 128;
__global__ void __launch_bounds__(FIXUP_LONG_THREADS) k_msm_fixup_long(msm_plan pl, uint32_t T,
                                                                      const uint32_t* __restrict__ offsets,
                                                                      const uint32_t* __restrict__ counts,
                                                                      const seg_partial* __restrict__ parts,
                                                                      jac_pt* __restrict__ buckets,
                                                                      const uint32_t* __restrict__ long_list,
                                                                      const uint32_t* __restrict__ long_count) {
    __shared__ jac_pt s_warp[FIXUP_LONG_THREADS / 32];
    int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (uint32_t li = blockIdx.x; li < *long_count; li += gridDim.x) {
        uint32_t s = long_list[li];
        uint32_t beg = offsets[s], end = beg + counts[s];
        uint32_t sa = beg / T, sb = (end - 1) / T;
        uint32_t np = 2 * (sb - sa + 1);  // head and tail record of every segment in range
        jf_pt acc = jf_identity();
        for (uint32_t r = threadIdx.x; r < np; r += FIXUP_LONG_THREADS) {
            const seg_partial* p = &parts[2 * (size_t)sa + r];
            if (p->slot == (int32_t)s) {
                jf_pt t = load_jac_as_jf(&p->pt);
                jf_add_exact(&acc, &t);
            }
        }
#pragma unroll 1
        for (int d = 16; d >= 1; d >>= 1) {
            jf_pt o = shfl_down_jf(acc, d);
            if (lane + d >= 32) o.w = 0;
            jf_add_exact(&acc, &o);
        }
        if (lane == 0) store_jf_as_jac(&s_warp[warp], acc);
        __syncthreads();
        if (threadIdx.x == 0) {
#pragma unroll 1
            for (int w = 1; w < FIXUP_LONG_THREADS / 32; w++) {
                jf_pt t = load_jac_as_jf(&s_warp[w]);
                jf_add_exact(&acc, &t);
            }
            store_jf_as_jac(&buckets[bucket_of_slot(pl, s)], acc);
        }
        __syncthreads();
    }
}

// chunk t of window k covers buckets lo..lo+chunk_sz-1 (1-based ids): contributes
//   sum_b b * B_b = sum_b (b - lo + 1) B_b + (lo - 1) * sum_b B_b
// A chunk is a serial chain of ~2 chunk_sz + log2(B) point operations and there are only a few thousand chunks, so each
// chunk runs on a group of six lanes (dist.cuh) -- three times shorter chains, six times the threads.
__global__ void __launch_bounds__(DIST_THREADS) k_msm_window_sum(msm_plan pl, const jac_pt* __restrict__ buckets,
                                                                 jac_pt* __restrict__ chunk_out) {
    int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int g = lane / 6, kc = lane % 6;
    if (g >= 5) return;
    int t = (blockIdx.x * (DIST_THREADS / 32) + warp) * 5 + g;
    if (t >= pl.K * pl.chunks) return;
    int gbase = 6 * g;
    unsigned mask = 0x3fu << gbase;
    int k = t / pl.chunks, ch = t % pl.chunks;
    int lo = ch * pl.chunk_sz + 1;
    const jac_pt* bk = buckets + (size_t)k * pl.B + (lo - 1);
    dpt running = dpt{1, 1, 0}, acc = dpt{1, 1, 0};  // identity: w = 0
#pragma unroll 1
    for (int b = pl.chunk_sz - 1; b >= 0; b--) {
        dpt bb = dpt{bk[b].X.c[kc], bk[b].Y.c[kc], bk[b].Z.c[0]};
        djf_add_exact(mask, &running, &bb, kc, gbase);
        djf_add_exact(mask, &acc, &running, kc, gbase);
    }
    if (lo > 1) {  // (lo - 1) * running by double-and-add from the top set bit
        uint32_t m = (uint32_t)(lo - 1);
        dpt mm = running;
#pragma unroll 1
        for (int bit = 30 - __clz(m); bit >= 0; bit--) {
            djf_dbl_exact(mask, &mm, kc, gbase);
            if ((m >> bit) & 1) djf_add_exact(mask, &mm, &running, kc, gbase);
        }
        djf_add_exact(mask, &acc, &mm, kc, gbase);
    }
    chunk_out[t].X.c[kc] = acc.X;
    chunk_out[t].Y.c[kc] = acc.Y;
    chunk_out[t].Z.c[kc] = kc == 0 ? acc.w : 0;
}
// one block per window: threads add strided chunk results, then a shuffle tree ("warp-shuffle bucket reduction")
// and a last step through shared memory
__device__ __forceinline__ jf_pt shfl_down_jf(const jf_pt& p, int delta) {
    jf_pt r;
#pragma unroll
    for (int c = 0; c < 6; c++) {
        r.X.c[c] = __shfl_down_sync(0xffffffffu, p.X.c[c], delta);
        r.Y.c[c] = __shfl_down_sync(0xffffffffu, p.Y.c[c], delta);
    }
    r.w = __shfl_down_sync(0xffffffffu, p.w, delta);
    return r;
}
static constexpr int FOLD_THREADS = 128;
__global__ void __launch_bounds__(FOLD_THREADS) k_msm_window_fold(msm_plan pl, const jac_pt* __restrict__ chunk_out,
                                                                  jac_pt* __restrict__ windows) {
    __shared__ jac_pt s_warp[FOLD_THREADS / 32];
    int k = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    jf_pt acc = jf_identity();
#pragma unroll 1
    for (int ch = threadIdx.x; ch < pl.chunks; ch += FOLD_THREADS) {
        jf_pt t = load_jac_as_jf(&chunk_out[(size_t)k * pl.chunks + ch]);
        jf_add_exact(&acc, &t);
    }
#pragma unroll 1
    for (int d = 16; d >= 1; d >>= 1) {
        jf_pt o = shfl_down_jf(acc, d);
        if (lane + d >= 32) o.w = 0;
        jf_add_exact(&acc, &o);
    }
    if (lane == 0) store_jf_as_jac(&s_warp[warp], acc);
    __syncthreads();
    if (threadIdx.x == 0) {
#pragma unroll 1
        for (int w = 1; w < FOLD_THREADS / 32; w++) {
            jf_pt t = load_jac_as_jf(&s_warp[w]);
            jf_add_exact(&acc, &t);
        }
        store_jf_as_jac(&windows[k], acc);
    }
}
// Horner over the windows is a serial chain of ~255 doublings, i.e. pure latency.  24 lanes of one warp share each
// doubling on two levels:
//  * an Fp6 value is DISTRIBUTED over a group of six lanes, lane k holding coefficient k; a product is then one
//    coefficient per lane (six 64x64 products + one reduction), the operands travelling by warp shuffles
//    (the source lane pre-selects b_j or 7 b_j for the wrap-around terms, so 12 x 64-bit shuffles per product);
//  * four such groups run the independent squarings of dbl-2007-bl side by side (two rounds), the linear parts
//    are coefficient-wise and computed redundantly by every group -> 4 short product rounds instead of 9 products.
static constexpr unsigned HORNER_MASK = 0x00ffffffu;  // lanes 0..23 = 4 groups x 6 coefficients
__device__ __forceinline__ fp_t shfl_fp(fp_t v, int src) { return __shfl_sync(HORNER_MASK, v, src); }
// (the six-lane product dfp6_mul lives in dist.cuh)
// one doubling of the point whose coefficients (x, y, z of lane k) are replicated over the four groups
__device__ void jac_dbl_dist(fp_t& x, fp_t& y, fp_t& z, int g, int k) {
    int gbase = 6 * g;
    fp_t yz = fp_add(y, z);
    fp_t op1 = g == 0 ? x : (g == 1 ? y : (g == 2 ? z : yz));
    fp_t s1 = dfp6_mul(HORNER_MASK, op1, op1, k, gbase);
    fp_t XX = shfl_fp(s1, k), YY = shfl_fp(s1, 6 + k), ZZ = shfl_fp(s1, 12 + k), W = shfl_fp(s1, 18 + k);
    fp_t op2 = g == 0 ? fp_add(x, YY) : (g == 1 ? YY : ZZ);
    fp_t s2 = dfp6_mul(HORNER_MASK, op2, op2, k, gbase);
    fp_t t = shfl_fp(s2, k), YYYY = shfl_fp(s2, 6 + k), Z4 = shfl_fp(s2, 12 + k);
    fp_t S = fp_dbl(fp_sub(fp_sub(t, XX), YYYY));
    fp_t M = fp_add(fp_add(fp_dbl(XX), XX), Z4);  // 3 XX + a ZZ^2, a = 1
    fp_t X3 = fp_sub(dfp6_mul(HORNER_MASK, M, M, k, gbase), fp_dbl(S));
    fp_t Y3 = fp_sub(dfp6_mul(HORNER_MASK, M, fp_sub(S, X3), k, gbase), fp_dbl(fp_dbl(fp_dbl(YYYY))));
    z = fp_sub(fp_sub(W, YY), ZZ);
    x = X3;
    y = Y3;
}
// add-2007-bl on the same 24 lanes: (x1, y1, z1) += (x2, y2, z2), every value = the lane's coefficient k, replicated
// over the four groups, which share the 16 products of the formula in five rounds.  Returns false (and leaves the
// accumulator untouched) on the exceptional inputs -- an identity operand or equal x -- which the caller resolves
// with the exact per-thread routine.
__device__ bool jac_add_dist(fp_t& x1, fp_t& y1, fp_t& z1, fp_t x2, fp_t y2, fp_t z2, int g, int k) {
    int gbase = 6 * g;
    auto pick = [&](fp_t a, fp_t b, fp_t c, fp_t d) { return g == 0 ? a : (g == 1 ? b : (g == 2 ? c : d)); };
    auto from = [&](fp_t v, int grp) { return shfl_fp(v, 6 * grp + k); };
    auto all24 = [&](bool v) { return __ballot_sync(HORNER_MASK, v) == HORNER_MASK; };
    if (all24(z1 == 0) || all24(z2 == 0)) return false;
    // round 1: Z1Z1, Z2Z2, Y1 Z2, Y2 Z1
    fp_t r1 = dfp6_mul(HORNER_MASK, pick(z1, z2, y1, y2), pick(z1, z2, z2, z1), k, gbase);
    fp_t Z1Z1 = from(r1, 0), Z2Z2 = from(r1, 1), Y1Z2 = from(r1, 2), Y2Z1 = from(r1, 3);
    // round 2: U1 = X1 Z2Z2, U2 = X2 Z1Z1, S1 = Y1 Z2 Z2Z2, S2 = Y2 Z1 Z1Z1
    fp_t r2 = dfp6_mul(HORNER_MASK, pick(x1, x2, Y1Z2, Y2Z1), pick(Z2Z2, Z1Z1, Z2Z2, Z1Z1), k, gbase);
    fp_t U1 = from(r2, 0), U2 = from(r2, 1), S1 = from(r2, 2), S2 = from(r2, 3);
    fp_t H = fp_sub(U2, U1), rr = fp_dbl(fp_sub(S2, S1));
    if (all24(H == 0)) return false;
    // round 3: I = (2H)^2, (Z1 + Z2)^2
    fp_t h2 = fp_dbl(H), zs = fp_add(z1, z2);
    fp_t r3 = dfp6_mul(HORNER_MASK, (g & 1) ? zs : h2, (g & 1) ? zs : h2, k, gbase);
    fp_t I = from(r3, 0), ZS = from(r3, 1);
    // round 4: J = H I, V = U1 I, rr^2, Z3 = ((Z1+Z2)^2 - Z1Z1 - Z2Z2) H
    fp_t zz = fp_sub(fp_sub(ZS, Z1Z1), Z2Z2);
    fp_t r4 = dfp6_mul(HORNER_MASK, pick(H, U1, rr, zz), pick(I, I, rr, H), k, gbase);
    fp_t J = from(r4, 0), V = from(r4, 1), RR = from(r4, 2), Z3 = from(r4, 3);
    fp_t X3 = fp_sub(fp_sub(RR, J), fp_dbl(V));
    // round 5: rr (V - X3), S1 J
    fp_t r5 = dfp6_mul(HORNER_MASK, (g & 1) ? S1 : rr, (g & 1) ? J : fp_sub(V, X3), k, gbase);
    fp_t Y3 = fp_sub(from(r5, 0), fp_dbl(from(r5, 1)));
    x1 = X3;
    y1 = Y3;
    z1 = Z3;
    return true;
}
// all coefficients of a distributed value, gathered from group 0
__device__ __forceinline__ fp6 gather_fp6(fp_t v) {
    fp6 r;
#pragma unroll
    for (int c = 0; c < 6; c++) r.c[c] = shfl_fp(v, c);
    return r;
}
// partial192 = Jacobian point (18 u64) || partial scalar sum (4 u64) || bad flag (u64) || pad
__global__ void __launch_bounds__(32) k_msm_horner(msm_plan pl, const jac_pt* __restrict__ windows,
                                                   const uint32_t* __restrict__ lin, const int* __restrict__ bad,
                                                   uint64_t* __restrict__ partial) {
    int lane = threadIdx.x;
    if (blockIdx.x != 0 || lane >= 24) return;
    int g = lane / 6, k = lane % 6;
    // the accumulator stays distributed (lane k of every group holds coefficient k) across doublings and additions
    fp_t x = windows[pl.K - 1].X.c[k], y = windows[pl.K - 1].Y.c[k], z = windows[pl.K - 1].Z.c[k];
#pragma unroll 1
    for (int w = pl.K - 2; w >= 0; w--) {
#pragma unroll 1
        for (int s = 0; s < pl.c; s++) jac_dbl_dist(x, y, z, g, k);
        if (!jac_add_dist(x, y, z, windows[w].X.c[k], windows[w].Y.c[k], windows[w].Z.c[k], g, k)) {
            // identity operand or equal x (empty window, adversarial batch): the exact routine, all lanes redundantly
            jac_pt acc;
            acc.X = gather_fp6(x);
            acc.Y = gather_fp6(y);
            acc.Z = gather_fp6(z);
            jac_add_mem(&acc, &windows[w], false);
            x = acc.X.c[k];
            y = acc.Y.c[k];
            z = acc.Z.c[k];
        }
    }
    jac_pt acc;
    acc.X = gather_fp6(x);
    acc.Y = gather_fp6(y);
    acc.Z = gather_fp6(z);
    if (lane != 0) return;
#pragma unroll
    for (int c = 0; c < 6; c++) {
        partial[c] = acc.X.c[c];
        partial[6 + c] = acc.Y.c[c];
        partial[12 + c] = acc.Z.c[c];
    }
#pragma unroll
    for (int c = 0; c < 4; c++) partial[18 + c] = ((uint64_t)lin[2 * c + 1] << 32) | lin[2 * c];
    partial[22] = (uint64_t)(*bad != 0);
    partial[23] = 0;
}

// lin * G on ONE WARP: lane i fetches the table point of window i (digits recoded as in fixed_base_accumulate), a
// shuffle tree of exact (X, Y, w) additions folds the 20 points in 5 steps, lane 0 normalises with one Fp inversion.
// Valid on lane 0 only.
__device__ __forceinline__ void warp_fixed_base_affine(const scalar& lin, const uint64_t* __restrict__ gtab, int lane,
                                                       fp6& rx, fp6& ry, bool& rinf) {
    jf_pt t = jf_identity();
    {
        int carry = 0, my_d = 0;
        bool my_neg = false;
        for (int i = 0; i < GTAB_WINDOWS; i++) {
            int raw = (int)sc_bits(lin, GTAB_W * i, GTAB_W) + carry;
            bool neg = raw > (1 << (GTAB_W - 1));
            carry = neg ? 1 : 0;
            int d = neg ? (1 << GTAB_W) - raw : raw;
            if (i == lane) {
                my_d = d;
                my_neg = neg;
            }
        }
        if (lane < GTAB_WINDOWS && my_d != 0) {
            load_affine(gtab, (size_t)lane * GTAB_ENTRIES + my_d, t.X, t.Y);
            if (my_neg) t.Y = fp6_neg(t.Y);
            t.w = 1;
        }
    }
#pragma unroll 1
    for (int d = 16; d >= 1; d >>= 1) {
        jf_pt o = shfl_down_jf(t, d);
        if (lane + d >= 32) o.w = 0;
        jf_add_exact(&t, &o);
    }
    rx = fp6_zero();
    ry = fp6_zero();
    rinf = t.w == 0;
    if (lane == 0 && !rinf) {
        fp_t wi = fp_inv(t.w), wi2 = fp_sqr(wi);
        rx = fp6_scale(t.X, wi2);
        ry = fp6_scale(t.Y, fp_mul(wi2, wi));
    }
}
// (sum s_i e_i) G of a SINGLE-device batch, launched on the second stream as soon as the scalar sum is known, so that it
// runs beside the MSM instead of behind it: rhs13 = x (6) | y (6) | infinity flag
__global__ void __launch_bounds__(32) k_lin_times_g(const uint32_t* __restrict__ lin8, const uint64_t* __restrict__ gtab,
                                                     uint64_t* __restrict__ rhs13) {
    if (blockIdx.x != 0) return;
    int lane = threadIdx.x;
    scalar lin;
#pragma unroll
    for (int k = 0; k < 8; k++) lin.l[k] = lin8[k];
    fp6 rx, ry;
    bool rinf;
    warp_fixed_base_affine(lin, gtab, lane, rx, ry, rinf);
    if (lane != 0) return;
#pragma unroll
    for (int c = 0; c < 6; c++) {
        rhs13[c] = rx.c[c];
        rhs13[6 + c] = ry.c[c];
    }
    rhs13[12] = rinf ? 1 : 0;
}

// result200: [0] verdict, [8..105) lhs97, [104..201)... laid out as verdict(1) pad(7) lhs(97) pad(7) rhs(97)
static constexpr size_t RESULT_BYTES = 216;
// One warp: adds the per-GPU partials, (sum lin) G (unless `rhs_pre` already holds it), x-only comparison.
__global__ void __launch_bounds__(32) k_batch_finish(size_t np, const uint64_t* __restrict__ partials,
                                                      const uint64_t* __restrict__ gtab, uint8_t* __restrict__ result,
                                                      const uint64_t* __restrict__ rhs_pre) {
    if (blockIdx.x != 0) return;
    int lane = threadIdx.x;
    scalar lin = sc_zero();
    bool bad = false;
    for (size_t r = 0; r < np; r++) {  // every lane: 32-byte scalars, cheap
        const uint64_t* p = partials + r * 24;
        lin = sc_add(lin, sc_from_u64x4(p[18], p[19], p[20], p[21]));
        bad |= p[22] != 0;
    }
    fp6 rx, ry;
    bool rinf;
    if (rhs_pre) {
#pragma unroll
        for (int c = 0; c < 6; c++) {
            rx.c[c] = rhs_pre[c];
            ry.c[c] = rhs_pre[6 + c];
        }
        rinf = rhs_pre[12] != 0;
    } else {
        warp_fixed_base_affine(lin, gtab, lane, rx, ry, rinf);
    }
    if (lane != 0) return;
    jac_pt acc = jac_identity();
    for (size_t r = 0; r < np; r++) {
        const uint64_t* p = partials + r * 24;
        jac_pt q;
#pragma unroll
        for (int c = 0; c < 6; c++) {
            q.X.c[c] = p[c];
            q.Y.c[c] = p[6 + c];
            q.Z.c[c] = p[12 + c];
        }
        jac_add_mem(&acc, &q, false);
    }
    fp6 lx, ly;
    bool linf;
    jac_to_affine(acc, lx, ly, linf);
    uint8_t v = bad ? VERDICT_MALFORMED : (fp6_eq(lx, rx) ? VERDICT_OK : VERDICT_INVALID_SIGNATURE);
    result[0] = v;
    uint64_t* l = reinterpret_cast<uint64_t*>(result + 8);
    uint64_t* rr = reinterpret_cast<uint64_t*>(result + 112);
#pragma unroll
    for (int c = 0; c < 6; c++) {
        l[c] = lx.c[c];
        l[6 + c] = ly.c[c];
        rr[c] = rx.c[c];
        rr[6 + c] = ry.c[c];
    }
    result[8 + 96] = linf ? 1 : 0;
    result[112 + 96] = rinf ? 1 : 0;
}

// ---- f3: failed-batch localisation --------------------------------------------------------------
// The reference returns ONE Err for the whole batch (src/batch.rs:125-129).  What the batch equation sums per item is
//     D_i = R_i - h_i P_i - e_i G          with R_i = from_compressed(sig_i.x) INCLUDING its flag byte (src/batch.rs:104)
// and no subgroup check on P_i (src/batch.rs:102-106).  The batch sums s_i D_i (the scalars reduced mod q), so "item i is
// what makes the batch fail" means its own term s_i D_i != O: a property of the item and its randomiser alone, whatever
// slice the bisection puts it in.  That is NOT the verdict of Signature::verify (x-only comparison, flag byte ignored,
// subgroup check first).  k_batch_item_check evaluates exactly that for the items of a work list (exact Jacobian
// arithmetic: adversarial inputs welcome).  Only items inside failing slices reach it: a slice whose non-O terms sum to
// O (two torsion-shifted items T2 + T2, say) passes the bisection and its items stay unflagged.
//     out[i] = 0  s_i D_i == O      2  s_i D_i != O      3  malformed (the reference panics: src/batch.rs:67,104)
// s R + (s h mod q)(-P) - (s e mod q) G == O: one item's term of the batch equation, exactly as k_batch_prepare forms
// its scalars.  Out of line: the rare path of k_batch_item_check, kept from adding to the kernel's register pressure.
SB_DEV_NOINLINE bool batch_term_is_identity(fp6 rx, fp6 ry, bool r_inf, fp6 px, fp6 py, bool pk_inf, scalar s, scalar h,
                                            scalar e, const uint64_t* __restrict__ gtab) {
    scalar t = pk_inf ? sc_zero() : sc_mul(h, s);
    jac_pt pr = jac_from_affine(rx, ry, r_inf), pp = jac_from_affine(px, fp6_neg(py), pk_inf), term = jac_identity();
#pragma unroll 1
    for (int b = 255; b >= 0; b--) {
        jac_dbl_mem(&term);
        if (sc_bits(s, b, 1)) jac_add_mem(&term, &pr, false);
        if (sc_bits(t, b, 1)) jac_add_mem(&term, &pp, false);
    }
    fixed_base_accumulate(&term, sc_neg(sc_mul(s, e)), gtab);
    return jac_is_identity(term);
}
__global__ void __launch_bounds__(VERIFY_THREADS, VERIFY_MIN_BLOCKS) k_batch_item_check(
    soa_batch in, const uint8_t* __restrict__ msgs, const uint64_t* __restrict__ msg_off, const uint8_t* __restrict__ rand32,
    const uint64_t* __restrict__ gtab, uint8_t* __restrict__ out) {
    struct d_slot {
        jac_pt p;
        uint64_t pad;
    };
    __shared__ d_slot s_d[VERIFY_THREADS];
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= in.n) return;
    uint8_t fl = in.flags[i];
    fp6 sx = load_fp6_planes(in.planes, 0, in.n, i);
    scalar e = load_scalar_planes(in.planes, 3, in.n, i);
    fp6 px = load_fp6_planes(in.planes, 5, in.n, i);
    fp6 py = load_fp6_planes(in.planes, 8, in.n, i);
    bool pk_inf = fl & FL_PK_INF;
    fp6 rx, ry;
    bool r_inf = true;
    bool ok = !(fl & (FL_MALFORMED | FL_X_BAD)) && decompress_point(sx, in.sig_flag[i], rx, ry, r_inf);
    if (!ok) {
        out[i] = VERDICT_MALFORMED;
        return;
    }
    uint64_t off = msg_off[i];
    scalar h = challenge_scalar(sx, px, py, pk_inf, msgs + off, msg_off[i + 1] - off);
    jac_pt r;
    bool torsion_free = torsion_check_and_mul(jac_from_affine(px, py, pk_inf), h, &r, &s_d[threadIdx.x].p);   // h P
    fixed_base_accumulate(&r, e, gtab);                                                                       // + e G
    bool same;
    if (jac_is_identity(r)) {
        same = r_inf;
    } else if (r_inf) {
        same = false;
    } else {  // (X, Y, Z) == (x, y):  X == x Z^2  and  Y == y Z^3
        fp6 zz = fp6_sqr(r.Z);
        same = fp6_eq(r.X, fp6_mul(rx, zz)) && fp6_eq(r.Y, fp6_mul(ry, fp6_mul(zz, r.Z)));
    }
    // D_i == O and [q]P_i == O: the item's term s_i D_i is O.  Otherwise (rare) evaluate the term exactly as the batch
    // sums it, s R_i + (s h mod q)(-P_i) - (s e mod q) G: an item with s_i D_i == O (s_i = 0, or D_i of small order
    // and a randomiser that kills it) cannot make the batch fail, and flagging it would make its flag depend on whether
    // its neighbours put it into a failing slice
    if (!same || !torsion_free)
        same = batch_term_is_identity(rx, ry, r_inf, px, py, pk_inf, sc_from_u256(sc_load_le(rand32 + 32 * i)), h, e, gtab);
    out[i] = same ? VERDICT_OK : VERDICT_INVALID_SIGNATURE;
}

// ---- small batches: one thread block per signature -------------------------------------------------------------------
// A batch of a few signatures (the reference's Criterion cases are 4 ... 128, benches/schnorr.rs:67-96) is pure latency in
// the Pippenger pipeline above: sixteen launches, a counting sort for a hundred points, a Horner tail of 255 serial
// doublings.  Here block i evaluates its own term of the batch equation (src/batch.rs:102-123),
//     T_i = s_i R_i + (s_i h_i) (-P_i),
// as k_verify_one does for a single verification (one.cuh): the two doubling chains of R_i and -P_i run side by side on
// two warps (24-lane Jacobian toolkit above, only the 64 window points of each chain are kept), a third warp hashes the
// challenge and forms the scalars, then the sixteen bucket accumulations (signed 4-bit windows: eight buckets per point)
// run four per warp and the two aggregations on two warps.  k_batch_small_reduce adds the T_i (eight per warp, then a tree)
// and writes the same 192-byte partial as k_msm_horner.  All arithmetic is exact (jac_add_dist_exact).
static constexpr int SMALL_THREADS = 128;
static constexpr int SMALL_WINDOWS = 64;   // signed 4-bit windows of a scalar < q < 2^255

// acc += (x2, y2, z2) on the 24 lanes, exact: the distributed formula, or -- identity operand / equal x -- the complete
// per-thread addition, every lane redundantly
__device__ __forceinline__ void jac_add_dist_exact(fp_t& x, fp_t& y, fp_t& z, fp_t x2, fp_t y2, fp_t z2, int g, int k) {
    if (__ballot_sync(HORNER_MASK, z2 == 0) == HORNER_MASK) return;   // + identity
    if (__ballot_sync(HORNER_MASK, z == 0) == HORNER_MASK) {          // identity + src
        x = x2;
        y = y2;
        z = z2;
        return;
    }
    if (!jac_add_dist(x, y, z, x2, y2, z2, g, k)) {
        jac_pt a, b;
        a.X = gather_fp6(x);
        a.Y = gather_fp6(y);
        a.Z = gather_fp6(z);
        b.X = gather_fp6(x2);
        b.Y = gather_fp6(y2);
        b.Z = gather_fp6(z2);
        jac_add_mem(&a, &b, false);
        x = a.X.c[k];
        y = a.Y.c[k];
        z = a.Z.c[k];
    }
}

struct small_shared {
    fp_t cx[2][SMALL_WINDOWS][6], cy[2][SMALL_WINDOWS][6], cz[2][SMALL_WINDOWS][6];  // window points 16^w R (0) and 16^w (-P) (1)
    fp_t bx[16][6], by[16][6], bz[16][6];                                             // bucket sums: 0..7 of R, 8..15 of -P
    fp_t ax[6], ay[6], az[6];                                                         // aggregated s_p (-P)
    fp_t rxy[12];                                                                     // decompressed R
    uint32_t mds2[24];
    int8_t hd[2][SMALL_WINDOWS];
    uint8_t lst[16][SMALL_WINDOWS], neg[16][SMALL_WINDOWS];
    int cnt[16];
    int ok, r_inf;
};

__global__ void __launch_bounds__(SMALL_THREADS) k_batch_small(soa_batch in, const uint8_t* __restrict__ msgs,
                                                               const uint64_t* __restrict__ msg_off,
                                                               const uint8_t* __restrict__ rand32, uint64_t* __restrict__ terms,
                                                               uint32_t* __restrict__ lin, int* __restrict__ bad) {
    __shared__ small_shared S;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const bool in24 = lane < 24;
    const int g = in24 ? lane / 6 : 0, k = lane % 6;
    const size_t i = blockIdx.x, n = in.n;
    const uint8_t fl = in.flags[i];
    const bool pk_inf = fl & FL_PK_INF;
    if (tid < 24) S.mds2[tid] = c_mds_row[tid % 12];
    if (tid < 16) S.cnt[tid] = 0;
    const uint64_t* pl = reinterpret_cast<const uint64_t*>(in.planes);
    fp_t sx = pl[((size_t)(0 + (k >> 1)) * n + i) * 2 + (k & 1)];
    fp_t px = pl[((size_t)(5 + (k >> 1)) * n + i) * 2 + (k & 1)];
    fp_t py = pl[((size_t)(8 + (k >> 1)) * n + i) * 2 + (k & 1)];
    if (tid == 0) {   // R = from_compressed(sig.x) incl. its flag byte: the reference unwraps it (src/batch.rs:104)
        bool ok = !(fl & (FL_MALFORMED | FL_X_BAD));
        fp6 rx = fp6_zero(), ry = fp6_zero();
        bool r_inf = true;
        if (ok) ok = decompress_point(load_fp6_planes(in.planes, 0, n, i), in.sig_flag[i], rx, ry, r_inf);
#pragma unroll
        for (int c = 0; c < 6; c++) {
            S.rxy[c] = rx.c[c];
            S.rxy[6 + c] = ry.c[c];
        }
        S.ok = ok;
        S.r_inf = r_inf;
        if (!ok) atomicOr(bad, 1);
    }
    __syncthreads();
    const bool ok = S.ok != 0, r_inf = S.r_inf != 0;

    // ---- phase A: the two doubling chains | challenge and scalars ----------------------------------------------------
    if (warp < 2) {
        const bool skip = warp == 0 ? (!ok || r_inf) : (!ok || pk_inf);   // identity contributes nothing
        if (in24 && !skip) {
            fp_t x = warp == 0 ? S.rxy[k] : px;
            fp_t y = warp == 0 ? S.rxy[6 + k] : fp_neg(py);               // -P, src/batch.rs:106
            fp_t z = k == 0 ? 1 : 0;
#pragma unroll 1
            for (int w = 0; w < SMALL_WINDOWS; w++) {
                if (g == 0) {
                    S.cx[warp][w][k] = x;
                    S.cy[warp][w][k] = y;
                    S.cz[warp][w][k] = z;
                }
                if (w < SMALL_WINDOWS - 1) {
                    jac_dbl_dist(x, y, z, g, k);
                    jac_dbl_dist(x, y, z, g, k);
                    jac_dbl_dist(x, y, z, g, k);
                    jac_dbl_dist(x, y, z, g, k);
                }
            }
        }
    } else if (warp == 2) {
        if (lane < 6) {
            uint64_t off = msg_off[i];
            scalar h = dchallenge_scalar(0x3fu, sx, pk_inf ? 0 : px, pk_inf ? 0 : py, msgs + off, msg_off[i + 1] - off, k, 0, S.mds2);
            if (k == 0) {
                scalar e = load_scalar_planes(in.planes, 3, n, i);
                scalar s = sc_from_u256(sc_load_le(rand32 + 32 * i));
                scalar s_r = sc_zero(), s_p = sc_zero(), l = sc_zero();
                if (ok) {
                    l = sc_mul(s, e);                         // src/batch.rs:92-97
                    s_r = r_inf ? sc_zero() : s;
                    s_p = pk_inf ? sc_zero() : sc_mul(h, s);  // src/batch.rs:109-111
                }
                recode_signed_w4(s_r, S.hd[0]);
                recode_signed_w4(s_p, S.hd[1]);
#pragma unroll
                for (int c = 0; c < 8; c++) lin[i * 8 + c] = l.l[c];
            }
        }
    }
    __syncthreads();

    // ---- phase B: sixteen bucket accumulations, four per warp --------------------------------------------------------
    if (in24) {
#pragma unroll 1
        for (int q4 = 0; q4 < 4; q4++) {
            const int slot = warp * 4 + q4, which = slot >> 3, mag = (slot & 7) + 1;
            if (lane == 0) {
                int c = 0;
#pragma unroll 1
                for (int w = 0; w < SMALL_WINDOWS; w++) {
                    int d = S.hd[which][w];
                    if (d != 0 && (d < 0 ? -d : d) == mag) {
                        S.lst[slot][c] = (uint8_t)w;
                        S.neg[slot][c] = d < 0;
                        c++;
                    }
                }
                S.cnt[slot] = c;
            }
            __syncwarp(HORNER_MASK);
            const int cnt = S.cnt[slot];
            fp_t x = 1, y = 1, z = 0;
#pragma unroll 1
            for (int t = 0; t < cnt; t++) {
                int w = S.lst[slot][t];
                fp_t x2 = S.cx[which][w][k], y2 = S.cy[which][w][k], z2 = S.cz[which][w][k];
                if (S.neg[slot][t]) y2 = fp_neg(y2);
                if (t == 0) {
                    x = x2;
                    y = y2;
                    z = z2;
                } else {
                    jac_add_dist_exact(x, y, z, x2, y2, z2, g, k);
                }
            }
            if (g == 0) {
                S.bx[slot][k] = x;
                S.by[slot][k] = y;
                S.bz[slot][k] = z;
            }
        }
    }
    __syncthreads();

    // ---- phase C: sum_m m B_m for both points (running sums), then T_i ------------------------------------------------
    fp_t ox = 1, oy = 1, oz = 0;
    if (warp < 2 && in24) {
        const int base = 8 * warp;
        fp_t rx = S.bx[base + 7][k], ry = S.by[base + 7][k], rz = S.bz[base + 7][k];
        ox = rx;
        oy = ry;
        oz = rz;
#pragma unroll 1
        for (int b = 6; b >= 0; b--) {
            jac_add_dist_exact(rx, ry, rz, S.bx[base + b][k], S.by[base + b][k], S.bz[base + b][k], g, k);
            jac_add_dist_exact(ox, oy, oz, rx, ry, rz, g, k);
        }
        if (warp == 1 && g == 0) {
            S.ax[k] = ox;
            S.ay[k] = oy;
            S.az[k] = oz;
        }
    }
    __syncthreads();
    if (warp == 0 && in24) {
        jac_add_dist_exact(ox, oy, oz, S.ax[k], S.ay[k], S.az[k], g, k);
        if (g == 0) {
            uint64_t* o = terms + i * 18;
            o[k] = ox;
            o[6 + k] = oy;
            o[12 + k] = oz;
        }
    }
}

// partial192 = sum of the n terms (Jacobian) || partial scalar sum || bad flag, as k_msm_horner writes it
static constexpr int SMALL_REDUCE_THREADS = 512;
__global__ void __launch_bounds__(SMALL_REDUCE_THREADS) k_batch_small_reduce(size_t n, const uint64_t* __restrict__ terms,
                                                                              const uint32_t* __restrict__ lin_total,
                                                                              const int* __restrict__ bad,
                                                                              uint64_t* __restrict__ partial) {
    __shared__ fp_t sx[SMALL_REDUCE_THREADS / 32][6], sy[SMALL_REDUCE_THREADS / 32][6], sz[SMALL_REDUCE_THREADS / 32][6];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nw = SMALL_REDUCE_THREADS / 32;
    const bool in24 = lane < 24;
    const int g = in24 ? lane / 6 : 0, k = lane % 6;
    fp_t x = 1, y = 1, z = 0;
    if (in24) {
#pragma unroll 1
        for (size_t i = warp; i < n; i += nw) {
            const uint64_t* t = terms + i * 18;
            jac_add_dist_exact(x, y, z, t[k], t[6 + k], t[12 + k], g, k);
        }
        if (g == 0) {
            sx[warp][k] = x;
            sy[warp][k] = y;
            sz[warp][k] = z;
        }
    }
#pragma unroll 1
    for (int d = nw / 2; d > 0; d >>= 1) {
        __syncthreads();
        if (warp < d && in24) {
            jac_add_dist_exact(x, y, z, sx[warp + d][k], sy[warp + d][k], sz[warp + d][k], g, k);
            if (g == 0) {
                sx[warp][k] = x;
                sy[warp][k] = y;
                sz[warp][k] = z;
            }
        }
    }
    if (warp == 0 && in24 && g == 0) {
        partial[k] = x;
        partial[6 + k] = y;
        partial[12 + k] = z;
        if (k < 4) partial[18 + k] = ((uint64_t)lin_total[2 * k + 1] << 32) | lin_total[2 * k];
        if (k == 4) partial[22] = (uint64_t)(*bad != 0);
        if (k == 5) partial[23] = 0;
    }
}

// ---- batches against a registered key set (keyset.cuh) ---------------------------------------------------------------
// k_batch_prepare writes t_i = s_i h_i mod q into scalars [n, 2n) (zero for identity keys and malformed items).  Instead
// of putting every -P_i into the MSM, the key side sums the t_i per key and adds c_k (-P_k) from the key's table, so the
// MSM runs over the n points R_i only.  The three kernels below run on the second stream, beside the MSM.
//
// Per key: the exact integer sum of its t_i as 64-bit column sums of the eight 32-bit limbs (keyset_sum_reduce).  Lanes
// of a warp with the same key add their limbs first (16-bit halves: 32 of them fit a 32-bit reduction), then one atomic
// per group and limb.  Integer addition commutes: the sums do not depend on the order of the atomics.  A malformed item
// (an index outside the set among them) never addresses the accumulator; its t_i is zero anyway.
// LOOKUP: the items of keyed records (k_keyed_split_lookup), after k_keyed_route: key_idx[i] == KEYSET_MISS marks a miss,
// whose t_i stays in the MSM and is skipped here, and `scalars` is the key-side copy, t_i at [i] instead of [n + i].
static constexpr int KEYSUM_THREADS = 256;
template <bool LOOKUP>
__global__ void __launch_bounds__(KEYSUM_THREADS) k_keyset_scalar_sum(soa_batch in, const uint32_t* __restrict__ key_idx,
                                                                      const uint32_t* __restrict__ scalars,
                                                                      unsigned long long* __restrict__ cols) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    size_t n = in.n;
    int lane = threadIdx.x & 31;
    bool live = i < n && !(in.flags[i] & FL_MALFORMED);   // every lane stays for the warp-wide match below
    uint32_t k = live ? key_idx[i] : 0xffffffffu;           // a live index is inside the set (k_keyset_gather)
    if (LOOKUP && k == KEYSET_MISS) live = false;          // a miss groups with the dead lanes (the same k)
    uint4 a = make_uint4(0, 0, 0, 0), b = a;
    if (live) {
        const uint4* t = reinterpret_cast<const uint4*>(scalars + (LOOKUP ? i : n + i) * 8);
        a = t[0];
        b = t[1];
    }
    uint32_t v[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
    unsigned grp = __match_any_sync(0xffffffffu, k);
    bool leader = lane == __ffs(grp) - 1;
#pragma unroll
    for (int j = 0; j < 8; j++) {
        unsigned lo = __reduce_add_sync(grp, v[j] & 0xffffu), hi = __reduce_add_sync(grp, v[j] >> 16);
        if (live && leader) atomicAdd(&cols[(size_t)k * 8 + j], (unsigned long long)lo + ((unsigned long long)hi << 16));
    }
}

// c_k (-P_k) for every key with a non-zero sum: one warp per key, lane i adds window i of the key's table
// (keyset_window_term), a shuffle tree of exact additions folds the 32 addends (the pattern of warp_fixed_base_affine).
// Warps stride over the keys and keep a running sum; each block writes the sum of its warps as one Jacobian term
// (18 u64, the layout k_batch_small_reduce adds up).  A zero sum needs no table: keys without one (the identity, status
// KEY_MALFORMED) only ever have zero sums, because their items contribute t_i = 0 or nothing.
static_assert(KT_WINDOWS <= 32, "one window per lane");
static constexpr int KEYTERM_THREADS = 128;
__global__ void __launch_bounds__(KEYTERM_THREADS) k_keyset_batch_term(size_t n_keys, const unsigned long long* __restrict__ cols,
                                                                       const uint64_t* __restrict__ ktab,
                                                                       uint64_t* __restrict__ terms) {
    __shared__ jac_pt s_warp[KEYTERM_THREADS / 32];
    int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const size_t wpb = KEYTERM_THREADS / 32;
    jf_pt acc = jf_identity();   // lane 0: the running sum of this warp's keys
#pragma unroll 1
    for (size_t k = blockIdx.x * wpb + warp; k < n_keys; k += gridDim.x * wpb) {
        uint64_t col[8];
#pragma unroll
        for (int j = 0; j < 8; j++) col[j] = cols[k * 8 + j];
        scalar c = keyset_sum_reduce(col);
        if (sc_is_zero(c)) continue;   // warp-uniform
        jf_pt t = lane < KT_WINDOWS ? keyset_window_term(c, lane, ktab + k * KT_KEY_U64) : jf_identity();
#pragma unroll 1
        for (int d = 16; d >= 1; d >>= 1) {
            jf_pt o = shfl_down_jf(t, d);
            if (lane + d >= 32) o.w = 0;
            jf_add_exact(&t, &o);
        }
        if (lane == 0) jf_add_exact(&acc, &t);
    }
    if (lane == 0) store_jf_as_jac(&s_warp[warp], acc);
    __syncthreads();
    if (threadIdx.x == 0) {
#pragma unroll 1
        for (int w = 1; w < KEYTERM_THREADS / 32; w++) {
            jf_pt t = load_jac_as_jf(&s_warp[w]);
            jf_add_exact(&acc, &t);
        }
        store_jf_as_jac(reinterpret_cast<jac_pt*>(terms) + blockIdx.x, acc);
    }
}

// out = a + b as 192-byte partials: point sum (exact), scalar sum mod q, bad flags or-ed.  Joins the MSM partial of a
// registered batch and its key side.  out may alias a or b.
__global__ void __launch_bounds__(32) k_partial_add(const uint64_t* __restrict__ a, const uint64_t* __restrict__ b,
                                                    uint64_t* out) {
    if (blockIdx.x != 0 || threadIdx.x != 0) return;
    jac_pt p, q;
#pragma unroll
    for (int c = 0; c < 6; c++) {
        p.X.c[c] = a[c];
        p.Y.c[c] = a[6 + c];
        p.Z.c[c] = a[12 + c];
        q.X.c[c] = b[c];
        q.Y.c[c] = b[6 + c];
        q.Z.c[c] = b[12 + c];
    }
    scalar lin = sc_add(sc_from_u64x4(a[18], a[19], a[20], a[21]), sc_from_u64x4(b[18], b[19], b[20], b[21]));
    uint64_t bad = (a[22] | b[22]) != 0;
    jac_add_mem(&p, &q, false);
#pragma unroll
    for (int c = 0; c < 6; c++) {
        out[c] = p.X.c[c];
        out[6 + c] = p.Y.c[c];
        out[12 + c] = p.Z.c[c];
    }
#pragma unroll
    for (int c = 0; c < 4; c++) out[18 + c] = sc_u64(lin, c);
    out[22] = bad;
    out[23] = 0;
}

// Keyed records against a registered set (k_keyed_split_lookup, reg_batch::miss_count): every item's key-side term goes
// to exactly one side.  k_batch_prepare has written (-P_i, t_i) into points and scalars [n, 2n).  A hit
// (key_idx[i] != KEYSET_MISS) is summed with its key: k_keyset_scalar_sum<true> reads t_i from the copy tk[i].  A miss
// stays in the MSM, compacted into [n, n + m) in record order (the exclusive scan of the miss flags, k_scan_local /
// k_scan_offsets); scalars [n + m, 2n) become zero, which gives no bucket entry (msm_digit 0).  A malformed item's t_i
// is zero: it adds nothing on either side.
// Two hazards are ruled out by construction:
//   - the key side never reads [n, 2n) while it is rewritten: it reads tk, and these kernels run on the main stream
//     ahead of the fork to the second stream;
//   - the compaction never overwrites a slot it has not read yet: k_keyed_route copies the misses out to mpts / msc,
//     and k_keyed_compact, a later launch, copies them back into [n, n + m).
__global__ void __launch_bounds__(256) k_keyed_miss_flags(size_t n, const uint32_t* __restrict__ key_idx,
                                                          uint32_t* __restrict__ miss) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) miss[i] = key_idx[i] == KEYSET_MISS;
}
__global__ void __launch_bounds__(256) k_keyed_route(size_t n, const uint32_t* __restrict__ key_idx,
                                                     const uint32_t* __restrict__ pos, const uint64_t* __restrict__ pts,
                                                     const uint32_t* __restrict__ scalars, uint32_t* __restrict__ tk,
                                                     uint64_t* __restrict__ mpts, uint32_t* __restrict__ msc) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint4* t = reinterpret_cast<const uint4*>(scalars + (n + i) * 8);
    uint4 a = t[0], b = t[1];
    uint4* o = reinterpret_cast<uint4*>(tk + i * 8);
    o[0] = a;
    o[1] = b;
    if (key_idx[i] != KEYSET_MISS) return;
    size_t p = pos[i];
    o = reinterpret_cast<uint4*>(msc + p * 8);
    o[0] = a;
    o[1] = b;
#pragma unroll
    for (int c = 0; c < 12; c++) mpts[p * 12 + c] = pts[(n + i) * 12 + c];
}
__global__ void __launch_bounds__(256) k_keyed_compact(size_t n, const uint32_t* __restrict__ miss_count,
                                                       const uint64_t* __restrict__ mpts, const uint32_t* __restrict__ msc,
                                                       uint64_t* __restrict__ pts, uint32_t* __restrict__ scalars) {
    size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    uint4* o = reinterpret_cast<uint4*>(scalars + (n + j) * 8);
    if (j >= *miss_count) {
        o[0] = o[1] = make_uint4(0, 0, 0, 0);
        return;
    }
    const uint4* t = reinterpret_cast<const uint4*>(msc + j * 8);
    o[0] = t[0];
    o[1] = t[1];
#pragma unroll
    for (int c = 0; c < 12; c++) pts[(n + j) * 12 + c] = mpts[j * 12 + c];
}

// the randomisers first ... first + n - 1 of a 32-byte seed (device) as n x 32 canonical LE bytes, one per thread
// (derive.cuh batch_randomizer): they fill the buffer the batch kernels read as rand32
__global__ void __launch_bounds__(128) k_batch_randomizers(size_t n, const uint8_t* __restrict__ seed32, uint64_t first,
                                                           uint8_t* __restrict__ out32) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    scalar s = batch_randomizer(seed32, first + i);
    uint8_t* o = out32 + 32 * i;
#pragma unroll
    for (int k = 0; k < 8; k++)
#pragma unroll
        for (int b = 0; b < 4; b++) o[4 * k + b] = (uint8_t)(s.l[k] >> (8 * b));
}

// key side of a registered batch (batch_partial_impl): the device buffers and the geometry of its launches
struct reg_batch {
    const uint32_t* key_idx;   // [n] device
    size_t n_keys;
    const uint64_t* ktab;      // the set's tables on this device
    unsigned long long* cols;  // [n_keys][8] column sums (zeroed by batch_partial_impl)
    uint64_t* terms;           // [term_blocks][18]
    unsigned term_blocks;
    uint64_t* key_partial;     // 192 B
    uint64_t* msm_partial;     // 192 B
    const uint32_t* zero;      // 64 zero bytes: the key partial's scalar sum and bad flag
    size_t msm_points;         // n; keyed records: n + m (m read on the host) or 2n (m not known when planning)
    // keyed records only (null otherwise): key_idx holds KEYSET_MISS for the m misses, *miss_count = m (device); the
    // route buffers of k_keyed_route: miss flags and their scan [n], scan tile totals, tk [n][8], mpts [n][12], msc [n][8]
    const uint32_t* miss_count;
    uint32_t *miss, *pos, *tile_total, *tk, *msc;
    uint64_t* mpts;
};

// ---- host orchestration ----------------------------------------------------------------------
// rhs_pre (optional, device, 13 x u64): single-device batches get (sum s_i e_i) G computed on the second stream beside the
// MSM.  Whatever runs on the second stream is joined into the context stream before this returns, so the regions it
// reads may be released then.
// reg (optional): a batch against a registered key set (pk96 = the gathered records of its items): the MSM runs over the
// n points R_i, the key terms c_k (-P_k) are computed on the second stream beside it and added to the MSM's partial;
// with reg->miss_count (keyed records) the MSM also keeps the misses' -P_i (k_keyed_route)
static int batch_partial_impl(schnorr_b200_ctx* ctx, size_t n, const uint8_t* sigs81, const uint8_t* pk96,
                              const uint8_t* pk_inf, const uint8_t* msgs, const uint64_t* msg_off,
                              const uint8_t* rand32, uint8_t* partial192, uint64_t* rhs_pre = nullptr,
                              const reg_batch* reg = nullptr) {
    scratch_scope scope(ctx->scratch, ctx->stream);
    soa_batch soa;
    if (int rc = alloc_soa(ctx, n, &soa)) return rc;
    if (n <= ctx->batch_small_max && !reg) {   // one thread block per signature (latency), see k_batch_small
        void *d_terms, *d_lin, *d_small;
        if (int rc = stage_in(ctx, {{nullptr, n * 18 * 8, &d_terms}, {nullptr, n * 32 + 512 * 32, &d_lin}, {nullptr, 64, &d_small}}))
            return rc;
        uint32_t* lin = (uint32_t*)d_lin;
        uint32_t* lin_part = lin + n * 8;
        uint32_t* lin_total = lin_part + 256 * 8;
        int* bad = (int*)d_small;
        cudaStream_t st = ctx->stream;
        CUDA_TRY(ctx, cudaMemsetAsync(d_small, 0, 64, st));
        k_ingest<<<grid_for(n, INGEST_THREADS), INGEST_THREADS, 0, st>>>(n, sigs81, pk96, pk_inf, soa);
        cudaEventRecord(ctx->ev_k0, st);
        k_batch_small<<<(unsigned)n, SMALL_THREADS, 0, st>>>(soa, msgs, msg_off, rand32, (uint64_t*)d_terms, lin, bad);
        cudaEventRecord(ctx->ev_k1, st);
        int sum_blocks = (int)((n + 255) / 256);
        k_scalar_sum<<<sum_blocks, 256, 0, st>>>(lin, n, lin_part);
        k_scalar_sum<<<1, 256, 0, st>>>(lin_part, (size_t)sum_blocks, lin_total);
        if (rhs_pre) {
            CUDA_TRY(ctx, cudaEventRecord(ctx->ev_chunk[1], st));
            CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->aux_stream, ctx->ev_chunk[1], 0));
            k_lin_times_g<<<1, 32, 0, ctx->aux_stream>>>(lin_total, ctx->gtab, rhs_pre);
            CUDA_TRY(ctx, cudaEventRecord(ctx->ev_aux, ctx->aux_stream));
            ctx->launches += 1;
        }
        k_batch_small_reduce<<<1, SMALL_REDUCE_THREADS, 0, st>>>(n, (uint64_t*)d_terms, lin_total, bad, (uint64_t*)partial192);
        if (rhs_pre) CUDA_TRY(ctx, cudaStreamWaitEvent(st, ctx->ev_aux, 0));
        ctx->last_msm_c = 4;
        ctx->last_msm_K = SMALL_WINDOWS;
        ctx->last_msm_T = 0;
        ctx->last_batch_points = 0;
        ctx->launches += 5;
        CUDA_TRY(ctx, cudaGetLastError());
        return SCHNORR_B200_OK;
    }
    size_t npts = reg ? reg->msm_points : 2 * n;   // k_batch_prepare writes 2n points and scalars either way
    if (2 * n >= 0x7fffffffu) {
        ctx->err = "batch too large for 31-bit point indices";
        return SCHNORR_B200_EARG;
    }
    msm_plan pl = msm_make_plan(npts, ctx->msm_c_override);
    if (npts * (size_t)pl.K >= 0xffffffffull) {  // sorted positions, offsets and counts are 32-bit
        ctx->err = "batch too large for 32-bit bucket offsets: split it (n * windows must stay below 2^31)";
        return SCHNORR_B200_EARG;
    }
    size_t nslots = (size_t)pl.K * (pl.B + 1);
    void *d_pts, *d_sc, *d_lin, *d_cnt, *d_sorted, *d_buckets, *d_small;
    size_t scan_tiles_max = (nslots + SCAN_TILE - 1) / SCAN_TILE;
    if (int rc = stage_in(ctx, {{nullptr, 2 * n * 96, &d_pts},
                                {nullptr, 2 * n * 32, &d_sc},
                                {nullptr, n * 32 + 512 * 32, &d_lin},
                                {nullptr, nslots * 4 * 3 + 4 * scan_tiles_max + 64, &d_cnt},
                                {nullptr, npts * pl.K * 4, &d_sorted},
                                {nullptr, sizeof(jac_pt) * ((size_t)pl.K * pl.B + (size_t)pl.K * pl.chunks + pl.K), &d_buckets},
                                {nullptr, 64, &d_small}}))
        return rc;
    // segment length: 8..32 entries per thread, longer for very large batches (bounds the partial arrays)
    size_t max_entries = npts * (size_t)pl.K;
    // 8 (small batches: more, shorter chains -- the accumulation is latency-bound there) .. 32 entries per thread
    uint32_t T = 32;
    while (T > 8 && max_entries / T < 65536) T /= 2;
    if (ctx->msm_t_override) T = ctx->msm_t_override;  // schnorr_b200_set_msm_geometry (tests)
    while ((max_entries + T - 1) / T > ((size_t)1 << 20)) T *= 2;
    ctx->last_msm_c = pl.c;
    ctx->last_msm_K = pl.K;
    ctx->last_msm_T = T;
    ctx->last_batch_points = npts;
    size_t nseg = ((max_entries + T - 1) / T + 127) / 128 * 128;
    void* d_parts;
    size_t max_long = nseg / MSM_LONG_SPAN + 1;  // buckets that can span >= MSM_LONG_SPAN segments
    if (int rc = stage_in(ctx, {{nullptr, nseg * 2 * sizeof(seg_partial) + 4 * max_long, &d_parts}})) return rc;
    uint32_t* long_list = (uint32_t*)((uint8_t*)d_parts + nseg * 2 * sizeof(seg_partial));
    uint32_t* long_count = (uint32_t*)d_small + 1;  // zeroed with the `bad` flag below
    uint32_t* counts = (uint32_t*)d_cnt;
    uint32_t* offsets = counts + nslots;
    uint32_t* cursor = offsets + nslots;
    uint32_t* tile_total = cursor + nslots;   // one total per scan tile (written before it is read: no clearing needed)
    jac_pt* buckets = (jac_pt*)d_buckets;
    jac_pt* chunk_out = buckets + (size_t)pl.K * pl.B;
    jac_pt* windows = chunk_out + (size_t)pl.K * pl.chunks;
    uint32_t* lin = (uint32_t*)d_lin;
    uint32_t* lin_part = lin + n * 8;       // 256 partials
    uint32_t* lin_total = lin_part + 256 * 8;
    int* bad = (int*)d_small;
    cudaStream_t st = ctx->stream;
    CUDA_TRY(ctx, cudaMemsetAsync(d_cnt, 0, nslots * 4 * 3, st));
    CUDA_TRY(ctx, cudaMemsetAsync(d_small, 0, 64, st));
    if (reg) CUDA_TRY(ctx, cudaMemsetAsync(reg->cols, 0, reg->n_keys * 8 * sizeof(unsigned long long), st));
    k_ingest<<<grid_for(n, INGEST_THREADS), INGEST_THREADS, 0, st>>>(n, sigs81, pk96, pk_inf, soa);
    uint32_t* h_pre = nullptr;
    // Challenges on six lanes per signature (k_batch_challenge_dist) ahead of a hash-free k_batch_prepare: up to a few
    // hundred thousand signatures the per-thread hash is a single, latency-bound wave (2^16: 1.06 ms against 0.92 ms on
    // six lanes); beyond that the per-thread form wins on throughput (84 M against 72 M hashes/s).  Reuses the `sorted`
    // buffer, which is written later.
    if (n <= ctx->batch_dist_max) {
        h_pre = (uint32_t*)d_sorted;
        k_batch_challenge_dist<<<grid_for(n, DIST_SIGS_PER_BLOCK), DIST_THREADS, 0, st>>>(soa, msgs, msg_off, h_pre);
        ctx->launches += 1;
    }
    k_batch_prepare<<<grid_for(n, 128), 128, 0, st>>>(soa, msgs, msg_off, rand32, (uint64_t*)d_pts, (uint32_t*)d_sc, lin, bad,
                                                      h_pre);
    int sum_blocks = (int)((n + 255) / 256);
    if (sum_blocks > 256) sum_blocks = 256;
    k_scalar_sum<<<sum_blocks, 256, 0, st>>>(lin, n, lin_part);
    k_scalar_sum<<<1, 256, 0, st>>>(lin_part, (size_t)sum_blocks, lin_total);
    if (reg && reg->miss_count) {   // keyed records: hits to the key side, misses compacted into [n, n + m) (k_keyed_route)
        unsigned tiles = (unsigned)((n + SCAN_TILE - 1) / SCAN_TILE);
        k_keyed_miss_flags<<<grid_for(n, 256), 256, 0, st>>>(n, reg->key_idx, reg->miss);
        k_scan_local<<<tiles, SCAN_THREADS, 0, st>>>(reg->miss, n, reg->pos, reg->tile_total);
        k_scan_offsets<<<tiles, SCAN_THREADS, 0, st>>>(n, reg->pos, reg->tile_total);
        k_keyed_route<<<grid_for(n, 256), 256, 0, st>>>(n, reg->key_idx, reg->pos, (uint64_t*)d_pts, (uint32_t*)d_sc, reg->tk,
                                                        reg->mpts, reg->msc);
        k_keyed_compact<<<grid_for(n, 256), 256, 0, st>>>(n, reg->miss_count, reg->mpts, reg->msc, (uint64_t*)d_pts,
                                                          (uint32_t*)d_sc);
        ctx->launches += 5;
    }
    if (rhs_pre || reg) {
        CUDA_TRY(ctx, cudaEventRecord(ctx->ev_chunk[1], st));
        CUDA_TRY(ctx, cudaStreamWaitEvent(ctx->aux_stream, ctx->ev_chunk[1], 0));
        if (rhs_pre) {
            k_lin_times_g<<<1, 32, 0, ctx->aux_stream>>>(lin_total, ctx->gtab, rhs_pre);
            ctx->launches += 1;
        }
        if (reg) {   // the key side: per-key scalar sums, key terms, their sum as a partial
            if (reg->miss_count)
                k_keyset_scalar_sum<true><<<grid_for(n, KEYSUM_THREADS), KEYSUM_THREADS, 0, ctx->aux_stream>>>(
                    soa, reg->key_idx, reg->tk, reg->cols);
            else
                k_keyset_scalar_sum<false><<<grid_for(n, KEYSUM_THREADS), KEYSUM_THREADS, 0, ctx->aux_stream>>>(
                    soa, reg->key_idx, (uint32_t*)d_sc, reg->cols);
            k_keyset_batch_term<<<reg->term_blocks, KEYTERM_THREADS, 0, ctx->aux_stream>>>(reg->n_keys, reg->cols, reg->ktab,
                                                                                            reg->terms);
            k_batch_small_reduce<<<1, SMALL_REDUCE_THREADS, 0, ctx->aux_stream>>>(reg->term_blocks, reg->terms, reg->zero,
                                                                                   (const int*)reg->zero, reg->key_partial);
            ctx->launches += 3;
        }
        CUDA_TRY(ctx, cudaEventRecord(ctx->ev_aux, ctx->aux_stream));
    }
    k_msm_count<<<grid_for(npts, 256), 256, 0, st>>>((uint32_t*)d_sc, npts, pl, counts);
    unsigned scan_tiles = (unsigned)((nslots + SCAN_TILE - 1) / SCAN_TILE);
    k_scan_local<<<scan_tiles, SCAN_THREADS, 0, st>>>(counts, nslots, offsets, tile_total);
    k_scan_offsets<<<scan_tiles, SCAN_THREADS, 0, st>>>(nslots, offsets, tile_total);
    k_msm_scatter<<<grid_for(npts, 256), 256, 0, st>>>((uint32_t*)d_sc, npts, pl, offsets, cursor, (uint32_t*)d_sorted);
    CUDA_TRY(ctx, cudaMemsetAsync(buckets, 0, sizeof(jac_pt) * (size_t)pl.K * pl.B, st));   // Z = 0: identity
    cudaEventRecord(ctx->ev_k0, st);
    k_msm_segment_sum<<<(unsigned)(nseg / 128), 128, 0, st>>>((uint64_t*)d_pts, pl, (uint32_t)nslots, T, offsets, counts,
                                                              (uint32_t*)d_sorted, buckets, (seg_partial*)d_parts);
    cudaEventRecord(ctx->ev_k1, st);
    k_msm_segment_fixup<<<grid_for(nslots, 128), 128, 0, st>>>(pl, (uint32_t)nslots, T, offsets, counts,
                                                               (seg_partial*)d_parts, buckets, long_list, long_count);
    // long buckets are rare (sparse top window, repeated randomisers): a grid of two blocks per SM strides over the list;
    // a larger grid only adds block-launch latency to the common case of an empty list (65 us at 1024 blocks)
    size_t long_grid = (size_t)2 * ctx->sm_count;
    k_msm_fixup_long<<<(unsigned)(max_long < long_grid ? max_long : long_grid), FIXUP_LONG_THREADS, 0, st>>>(
        pl, T, offsets, counts, (seg_partial*)d_parts, buckets, long_list, long_count);
    k_msm_window_sum<<<grid_for((size_t)pl.K * pl.chunks, DIST_SIGS_PER_BLOCK), DIST_THREADS, 0, st>>>(pl, buckets, chunk_out);
    k_msm_window_fold<<<pl.K, FOLD_THREADS, 0, st>>>(pl, chunk_out, windows);
    k_msm_horner<<<1, 32, 0, st>>>(pl, windows, lin_total, bad, reg ? reg->msm_partial : (uint64_t*)partial192);
    ctx->launches += 14;
    if (rhs_pre || reg) CUDA_TRY(ctx, cudaStreamWaitEvent(st, ctx->ev_aux, 0));
    if (reg) {
        k_partial_add<<<1, 32, 0, st>>>(reg->msm_partial, reg->key_partial, (uint64_t*)partial192);
        ctx->launches += 1;
    }
    CUDA_TRY(ctx, cudaGetLastError());
    return SCHNORR_B200_OK;
}

// the partial of an empty batch: identity point, zero scalar
static int batch_partial_empty(schnorr_b200_ctx* ctx, uint8_t* partial192) {
    ctx->last_batch_points = 0;
    uint64_t h[24] = {0};
    h[0] = 1;
    h[6] = 1;
    CUDA_TRY(ctx, cudaMemcpyAsync(partial192, h, 192, cudaMemcpyHostToDevice, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    return SCHNORR_B200_OK;
}

// A whole batch on one device (its device selected): partial_fn(partial, rhs_pre) reduces the n > 0 signatures to the
// partial with (sum s e) G computed beside it into rhs_pre (batch_partial_impl), and k_batch_finish writes the result
// to `result216` (device).
template <typename F>
static int batch_whole(schnorr_b200_ctx* ctx, size_t n, F partial_fn, uint8_t* result216) {
    scratch_scope scope(ctx->scratch, ctx->stream);
    uint8_t* partial;
    uint64_t* rhs_pre;
    if (int rc = stage_in(ctx, {{nullptr, 192, &partial}, {nullptr, 128, &rhs_pre}})) return rc;
    if (!n) rhs_pre = nullptr;
    if (int rc = n ? partial_fn(partial, rhs_pre) : batch_partial_empty(ctx, partial)) return rc;
    k_batch_finish<<<1, 32, 0, ctx->stream>>>(1, (const uint64_t*)partial, ctx->gtab, result216, rhs_pre);
    ctx->launches += 1;
    CUDA_TRY(ctx, cudaGetLastError());
    return SCHNORR_B200_OK;
}

static int read_result(schnorr_b200_ctx* ctx, const uint8_t* d_res, int* verdict, uint8_t* lhs97, uint8_t* rhs97) {
    uint8_t h[RESULT_BYTES];
    CUDA_TRY(ctx, cudaMemcpyAsync(h, d_res, RESULT_BYTES, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(ctx, cudaStreamSynchronize(ctx->stream));
    *verdict = h[0];
    if (lhs97) memcpy(lhs97, h + 8, 97);
    if (rhs97) memcpy(rhs97, h + 112, 97);
    return SCHNORR_B200_OK;
}
// batch_whole into a result region of this call, read back into the host outputs
template <typename F>
static int batch_whole_host(schnorr_b200_ctx* ctx, size_t n, F partial_fn, int* verdict, uint8_t* lhs97, uint8_t* rhs97) {
    scratch_scope scope(ctx->scratch, ctx->stream);
    uint8_t* res;
    if (int rc = stage_in(ctx, {{nullptr, RESULT_BYTES, &res}})) return rc;
    if (int rc = batch_whole(ctx, n, partial_fn, res)) return rc;
    return read_result(ctx, res, verdict, lhs97, rhs97);
}

// multi.cuh: a batch over every device of a multi-device context; partial(k, slice, rebased offsets, partial192) reduces
// the non-empty slice of shard k to its partial on that shard's device
template <typename F>
static int multi_verify_batch(schnorr_b200_ctx* ctx, size_t n, const uint64_t* msg_off, int* verdict, uint8_t* lhs97,
                              uint8_t* rhs97, F partial);

extern "C" {

int schnorr_b200_batch_partial_dev(schnorr_b200_ctx* ctx, size_t n, const uint8_t* sigs81, const uint8_t* pk96,
                                   const uint8_t* pk_inf, const uint8_t* msgs, const uint64_t* msg_off,
                                   const uint8_t* rand32, uint8_t* partial192) {
    if (!ctx || !partial192 || (n && (!sigs81 || !pk96 || !msg_off || !rand32))) return SCHNORR_B200_EARG;
    NOT_ON_MULTI(ctx);
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    if (n == 0) return batch_partial_empty(ctx, partial192);
    return batch_partial_impl(ctx, n, sigs81, pk96, pk_inf, msgs, msg_off, rand32, partial192);
}

int schnorr_b200_batch_finish_dev(schnorr_b200_ctx* ctx, size_t n_partials, const uint8_t* partials192,
                                  uint8_t* result216) {
    if (!ctx || !partials192 || !result216 || n_partials == 0) return SCHNORR_B200_EARG;
    NOT_ON_MULTI(ctx);
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    k_batch_finish<<<1, 32, 0, ctx->stream>>>(n_partials, (const uint64_t*)partials192, ctx->gtab, result216, nullptr);
    ctx->launches += 1;
    CUDA_TRY(ctx, cudaGetLastError());
    return SCHNORR_B200_OK;
}

// whole single-device batch on device buffers: partial MSM with (sum s e) G computed beside it, then the finish
int schnorr_b200_verify_batch_dev(schnorr_b200_ctx* ctx, size_t n, const uint8_t* sigs81, const uint8_t* pk96,
                                  const uint8_t* pk_inf, const uint8_t* msgs, const uint64_t* msg_off,
                                  const uint8_t* rand32, uint8_t* result216) {
    if (!ctx || !result216 || (n && (!sigs81 || !pk96 || !msg_off || !rand32))) return SCHNORR_B200_EARG;
    NOT_ON_MULTI(ctx);
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    return batch_whole(ctx, n, [&](uint8_t* partial, uint64_t* rhs_pre) {
        return batch_partial_impl(ctx, n, sigs81, pk96, pk_inf, msgs, msg_off, rand32, partial, rhs_pre);
    }, result216);
}

int schnorr_b200_batch_finish(schnorr_b200_ctx* ctx, size_t n_partials, const uint8_t* partials192_host, int* verdict,
                              uint8_t* lhs97, uint8_t* rhs97) {
    if (!ctx || !partials192_host || !verdict || n_partials == 0) return SCHNORR_B200_EARG;
    MULTI_DISPATCH(ctx, schnorr_b200_batch_finish(ctx->shards[0], n_partials, partials192_host, verdict, lhs97, rhs97));
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    scratch_scope scope(ctx->scratch, ctx->stream);
    uint8_t *d_p, *res;
    if (int rc = stage_in(ctx, {{partials192_host, n_partials * 192, &d_p}, {nullptr, RESULT_BYTES, &res}})) return rc;
    if (int rc = schnorr_b200_batch_finish_dev(ctx, n_partials, d_p, res)) return rc;
    return read_result(ctx, res, verdict, lhs97, rhs97);
}

// Where the randomisers of a host-form batch come from: the caller's n x 32 bytes (`host`), or, when `host` is null, the
// generator run on the device from the 32-byte `seed` for the indices first, first + 1, ...  Staging copies `host` into
// the randomiser region, or copies only the seed and reserves the region for rand_generate.
struct rand_source {
    const uint8_t* host;
    const uint8_t* seed;
    uint64_t first;
    // the source of the items from `lo` on (a shard's slice)
    rand_source from(size_t lo) const { return host ? rand_source{host + 32 * lo, nullptr, 0} : rand_source{nullptr, seed, first + lo}; }
    stage_region rand_region(size_t n, uint8_t** d_rand) const { return {host, n * 32, d_rand}; }
    stage_region seed_region(uint8_t** d_seed) const { return {seed, host ? (size_t)0 : (size_t)32, d_seed}; }
};
static rand_source rand_from_host(const uint8_t* rand32) { return {rand32, nullptr, 0}; }
static rand_source rand_from_seed(const uint8_t* seed32) { return {nullptr, seed32, 0}; }

// n randomisers of a seeded source into d_rand (device), enqueued on the context stream; nothing for host bytes
static int rand_generate(schnorr_b200_ctx* ctx, size_t n, const rand_source& rs, const uint8_t* d_seed, uint8_t* d_rand) {
    if (rs.host || n == 0) return SCHNORR_B200_OK;
    k_batch_randomizers<<<grid_for(n, 128), 128, 0, ctx->stream>>>(n, d_seed, rs.first, d_rand);
    ctx->launches += 1;
    CUDA_TRY(ctx, cudaGetLastError());
    return SCHNORR_B200_OK;
}

// host inputs (n > 0) -> staged on the device -> one 192-byte partial at `partial` (device memory of this context)
static int batch_partial_host(schnorr_b200_ctx* ctx, size_t n, const uint8_t* sigs81, const uint8_t* pk96,
                              const uint8_t* pk_inf, const uint8_t* msgs, const uint64_t* msg_off, const rand_source& rs,
                              uint8_t* partial, uint64_t* rhs_pre = nullptr) {
    CHECK_MSG_OFF(ctx, n, msg_off);
    size_t mb = msg_off[n];
    if (mb && !msgs) return SCHNORR_B200_EARG;
    scratch_scope scope(ctx->scratch, ctx->stream);
    uint8_t *d_sig, *d_pk, *d_m, *d_off, *d_rand, *d_inf, *d_seed;
    if (int rc = stage_in(ctx, {{sigs81, n * 81, &d_sig}, {pk96, n * 96, &d_pk}, {msgs, mb, &d_m}, {msg_off, (n + 1) * 8, &d_off},
                                rs.rand_region(n, &d_rand), {pk_inf, n, &d_inf}, rs.seed_region(&d_seed)}))
        return rc;
    if (int rc = rand_generate(ctx, n, rs, d_seed, d_rand)) return rc;
    return batch_partial_impl(ctx, n, d_sig, d_pk, pk_inf ? d_inf : nullptr, d_m, (uint64_t*)d_off, d_rand, partial, rhs_pre);
}

// the host forms of verify_batch (arguments checked)
static int verify_batch_host(schnorr_b200_ctx* ctx, size_t n, const uint8_t* sigs81, const uint8_t* pk96,
                             const uint8_t* pk_inf, const uint8_t* msgs, const uint64_t* msg_off, const rand_source& rs,
                             int* verdict, uint8_t* lhs97, uint8_t* rhs97) {
    if (!ctx->shards.empty())
        return multi_verify_batch(ctx, n, msg_off, verdict, lhs97, rhs97, [&](int k, auto s, const uint64_t* off, uint8_t* partial) {
            return batch_partial_host(ctx->shards[k], s.hi - s.lo, sigs81 + 81 * s.lo, pk96 + 96 * s.lo,
                                      pk_inf ? pk_inf + s.lo : nullptr, msgs ? msgs + msg_off[s.lo] : nullptr, off,
                                      rs.from(s.lo), partial);
        });
    CUDA_TRY(ctx, cudaSetDevice(ctx->device));
    return batch_whole_host(ctx, n, [&](uint8_t* partial, uint64_t* rhs_pre) {
        return batch_partial_host(ctx, n, sigs81, pk96, pk_inf, msgs, msg_off, rs, partial, rhs_pre);
    }, verdict, lhs97, rhs97);
}

int schnorr_b200_verify_batch(schnorr_b200_ctx* ctx, size_t n, const uint8_t* sigs81, const uint8_t* pk96,
                              const uint8_t* pk_inf, const uint8_t* msgs, const uint64_t* msg_off, const uint8_t* rand32,
                              int* verdict, uint8_t* lhs97, uint8_t* rhs97) {
    if (!ctx || !verdict || (n && (!sigs81 || !pk96 || !msg_off || !rand32))) return SCHNORR_B200_EARG;
    return verify_batch_host(ctx, n, sigs81, pk96, pk_inf, msgs, msg_off, rand_from_host(rand32), verdict, lhs97, rhs97);
}

int schnorr_b200_verify_batch_seeded(schnorr_b200_ctx* ctx, size_t n, const uint8_t* sigs81, const uint8_t* pk96,
                                     const uint8_t* pk_inf, const uint8_t* msgs, const uint64_t* msg_off, const uint8_t* seed32,
                                     int* verdict, uint8_t* lhs97, uint8_t* rhs97) {
    if (!ctx || !verdict || !seed32 || (n && (!sigs81 || !pk96 || !msg_off))) return SCHNORR_B200_EARG;
    return verify_batch_host(ctx, n, sigs81, pk96, pk_inf, msgs, msg_off, rand_from_seed(seed32), verdict, lhs97, rhs97);
}

}  // extern "C"
