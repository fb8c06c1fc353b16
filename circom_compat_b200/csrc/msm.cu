// msm.cu - kernels and launchers of the fixed-base-table Pippenger MSM described in msm.cuh.
#include <algorithm>
#include <vector>
#include "msm.cuh"
#include "util.cuh"

namespace b2g {

std::atomic<uint64_t> g_launch_count{0};

// ------------------------------------------------------------------------------------------------ key-load time
// T[w][i] = 2^(c*w) * P_i, affine.  One thread per base; the nwin XYZZ multiples live in local memory and are brought
// back to affine with one field inversion per thread (Montgomery's trick over ZZZ).
template <class C, class F>
__global__ void __launch_bounds__(128) msm_table_kernel(const void* __restrict__ bases, uint32_t n, int c, int nwin, void* __restrict__ table) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    using Pt = typename C::Pt; using Aff = typename C::Aff; using E = typename F::elem;
    Aff p = aff_load<F>(bases, i);
    if (C::aff_is_inf(p)) {
        Aff z; z.x = F::zero(); z.y = F::zero();
        for (int w = 0; w < nwin; w++) aff_store<F>(table, (size_t)w * n + i, z);
        return;
    }
    Pt pts[MSM_MAX_WIN];
    E pre[MSM_MAX_WIN];
    Pt cur = C::from_affine(p);
    E acc = F::one();
    for (int w = 0; w < nwin; w++) {
        pts[w] = cur;
        pre[w] = acc;
        acc = F::mul(acc, cur.zzz);                 // never zero: prime-order group, P != inf
        if (w + 1 < nwin) for (int j = 0; j < c; j++) cur = C::dbl(cur);
    }
    E inv = F::inv(acc);
    for (int w = nwin - 1; w >= 0; w--) {
        E iz = F::mul(inv, pre[w]);                 // 1/zzz_w
        inv = F::mul(inv, pts[w].zzz);
        Aff a;
        a.y = F::mul(pts[w].y, iz);
        a.x = F::mul(pts[w].x, F::mul(F::sqr(pts[w].zz), F::sqr(iz)));
        aff_store<F>(table, (size_t)w * n + i, a);
    }
}

// every base must be on the curve (or the all-zero point at infinity); *bad receives 1 + index of an offender
template <class C, class F>
__global__ void __launch_bounds__(256) msm_validate_kernel(const void* __restrict__ bases, uint32_t n, uint32_t* __restrict__ bad) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (!aff_on_curve<C, F>(aff_load<F>(bases, i))) atomicMax(bad, i + 1u);
}

// ------------------------------------------------------------------------------------------------ (1) digits + histogram
// (1a) scalars -> canonical integers (one Montgomery reduction each)
__global__ void __launch_bounds__(256) msm_canon_kernel(const fe* __restrict__ scalars, uint32_t n, int scalars_mont, fe* __restrict__ canon_out) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    fe k = fe_load_nc(&scalars[i]);
    if (scalars_mont) k = Fr::to_canonical(k);
    fe_store(&canon_out[i], k);
}

// raw c-bit window w of a canonical scalar held in global memory
__device__ __forceinline__ uint32_t msm_window_bits(const uint32_t* __restrict__ k, int c, int w) {
    const uint32_t off = (uint32_t)w * (uint32_t)c, limb = off >> 5, sh = off & 31u;
    if (limb >= 8) return 0u;
    uint64_t v = __ldg(&k[limb]);
    if (limb + 1 < 8 && sh + (uint32_t)c > 32u) v |= (uint64_t)__ldg(&k[limb + 1]) << 32;
    return (uint32_t)(v >> sh) & ((1u << c) - 1u);
}

// Signed digit of window w without walking the whole carry chain (ark-ec make_digits semantics): the carry into window
// w is 1 iff the window below holds >= 2^(c-1), 0 iff it holds < 2^(c-1) - 1, and only for the single value
// 2^(c-1) - 1 does it depend on the next window down.
__device__ __forceinline__ int32_t msm_digit_at(const uint32_t* __restrict__ k, int c, int w) {
    const uint32_t half = 1u << (c - 1);
    uint32_t carry = 0;
    for (int v = w - 1; v >= 0; v--) {
        const uint32_t b = msm_window_bits(k, c, v);
        if (b >= half) { carry = 1; break; }
        if (b < half - 1) break;
    }
    const uint32_t coef = msm_window_bits(k, c, w) + carry;
    // top window: k < r keeps coef < 2^(c-1) for c in [8, 22], so cout = 0 and dropping it loses nothing (test_msm_digit_model.py)
    const uint32_t cout = (coef + half) >> c;
    return (int32_t)coef - (int32_t)(cout << c);
}

// (1b) one thread per (window, scalar): bucket histogram.  Hot buckets (circom witnesses: most wires are 0 / 1, so one bucket
// receives a large share of all entries) must not cost one atomic per entry, but match.any - the general way to group equal
// lanes - was the kernel's main stall on uniform scalars (short-scoreboard 14.6 per issue, L2 at 48 %).  Two leader rounds do:
// the first pending lane broadcasts its bucket, every lane with the same bucket is counted by ONE atomic; a hot bucket is the
// leader's with high probability, and on uniform data the rounds cost four ballots.  Lanes still pending add individually.
constexpr int MSM_LEADER_ROUNDS = 2;

__global__ void __launch_bounds__(256) msm_count_kernel(const fe* __restrict__ canon, uint32_t n, int c, int nwin, uint32_t* __restrict__ counts) {
    const uint64_t tid = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t w = (uint32_t)(tid / n), i = (uint32_t)(tid % n);
    int32_t d = 0;
    if (w < (uint32_t)nwin) d = msm_digit_at(canon[i].l, c, (int)w);
    const uint32_t b = d ? (uint32_t)(d < 0 ? -d : d) - 1u : 0xffffffffu;
    const uint32_t lane = threadIdx.x & 31;
    bool pending = d != 0;
    {   // bucket 0 (digit +-1) is where the bits of a circom witness land: always grouped, one ballot
        const uint32_t hot = __ballot_sync(0xffffffffu, pending && b == 0u);
        if (hot) {
            if ((int)lane == __ffs(hot) - 1) atomicAdd(&counts[0], (uint32_t)__popc(hot));
            if (b == 0u) pending = false;
        }
    }
    #pragma unroll
    for (int round = 0; round < MSM_LEADER_ROUNDS; round++) {
        const uint32_t pend = __ballot_sync(0xffffffffu, pending);
        if (!pend) break;
        const int leader = __ffs(pend) - 1;
        const uint32_t lb = __shfl_sync(0xffffffffu, b, leader);
        const bool mine = pending && b == lb;
        const uint32_t same = __ballot_sync(0xffffffffu, mine);
        if ((int)lane == leader) atomicAdd(&counts[lb], (uint32_t)__popc(same));
        if (mine) pending = false;
    }
    if (pending) atomicAdd(&counts[b], 1u);
}

// ------------------------------------------------------------------------------------------------ (2) exclusive scan (one CTA)
__global__ void __launch_bounds__(1024) msm_scan_kernel(const uint32_t* __restrict__ counts, uint32_t nb, uint32_t* __restrict__ offsets,
                                                        uint32_t* __restrict__ cursor) {
    __shared__ uint32_t warp_sums[32];
    __shared__ uint32_t carry_s;
    const uint32_t tid = threadIdx.x, per = (nb + 1023u) / 1024u;
    const uint32_t lo = tid * per, hi = min(lo + per, nb);
    uint32_t s = 0;
    if ((per & 3u) == 0 && hi == lo + per) {                      // aligned chunk: independent 128-bit loads
        const uint4* v4 = reinterpret_cast<const uint4*>(counts + lo);
        #pragma unroll 4
        for (uint32_t j = 0; j < per / 4; j++) { const uint4 q = __ldg(&v4[j]); s += q.x + q.y + q.z + q.w; }
    } else {
        for (uint32_t j = lo; j < hi; j++) s += counts[j];
    }
    // block exclusive scan of s
    uint32_t v = s;
    #pragma unroll
    for (int d = 1; d < 32; d <<= 1) { uint32_t t = __shfl_up_sync(0xffffffffu, v, d); if ((tid & 31) >= (uint32_t)d) v += t; }
    if ((tid & 31) == 31) warp_sums[tid >> 5] = v;
    __syncthreads();
    if (tid < 32) {
        uint32_t w = warp_sums[tid], x = w;
        #pragma unroll
        for (int d = 1; d < 32; d <<= 1) { uint32_t t = __shfl_up_sync(0xffffffffu, x, d); if (tid >= (uint32_t)d) x += t; }
        warp_sums[tid] = x - w;
        if (tid == 31) carry_s = x;
    }
    __syncthreads();
    uint32_t run = warp_sums[tid >> 5] + v - s;
    for (uint32_t j = lo; j < hi; j++) { offsets[j] = run; cursor[j] = 0; run += counts[j]; }
    if (tid == 0) offsets[nb] = carry_s;
}

// ------------------------------------------------------------------------------------------------ (3) scatter
__global__ void __launch_bounds__(256) msm_scatter_kernel(const fe* __restrict__ canon, uint32_t n, uint32_t row_stride, int c, int nwin,
                                   const uint32_t* __restrict__ offsets, uint32_t* __restrict__ cursor, uint32_t* __restrict__ entries) {
    const uint64_t tid = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const uint32_t w = (uint32_t)(tid / n), i = (uint32_t)(tid % n);
    int32_t d = 0;
    if (w < (uint32_t)nwin) d = msm_digit_at(canon[i].l, c, (int)w);
    const uint32_t b = d ? (uint32_t)(d < 0 ? -d : d) - 1u : 0xffffffffu;
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t entry = (w * row_stride + i) | (d < 0 ? 0x80000000u : 0u);
    bool pending = d != 0;
    {   // hot bucket 0 first (see msm_count_kernel)
        const uint32_t hot = __ballot_sync(0xffffffffu, pending && b == 0u);
        if (hot) {
            const int leader = __ffs(hot) - 1;
            uint32_t base = 0;
            if ((int)lane == leader) base = atomicAdd(&cursor[0], (uint32_t)__popc(hot));
            base = __shfl_sync(0xffffffffu, base, leader);
            if (pending && b == 0u) {
                entries[offsets[0] + base + (uint32_t)__popc(hot & ((1u << lane) - 1u))] = entry;
                pending = false;
            }
        }
    }
    #pragma unroll
    for (int round = 0; round < MSM_LEADER_ROUNDS; round++) {            // same leader rounds as the histogram pass
        const uint32_t pend = __ballot_sync(0xffffffffu, pending);
        if (!pend) break;
        const int leader = __ffs(pend) - 1;
        const uint32_t lb = __shfl_sync(0xffffffffu, b, leader);
        const bool mine = pending && b == lb;
        const uint32_t same = __ballot_sync(0xffffffffu, mine);
        uint32_t base = 0;
        if ((int)lane == leader) base = atomicAdd(&cursor[lb], (uint32_t)__popc(same));
        base = __shfl_sync(0xffffffffu, base, leader);
        if (mine) {
            entries[offsets[b] + base + (uint32_t)__popc(same & ((1u << lane) - 1u))] = entry;
            pending = false;
        }
    }
    if (pending) entries[offsets[b] + atomicAdd(&cursor[b], 1u)] = entry;
}

// ------------------------------------------------------------------------------------------------ (4a) batched-affine pre-reduction
// Level structure (depends only on the sorted scalars).  cnt_k[b] = ceil(cnt_{k-1}[b] / 2); off_k = exclusive scan.
// One CTA; levels are processed one after the other (each needs the previous one's offsets).
__global__ void __launch_bounds__(1024) msm_aff_levels_kernel(uint32_t nb, int rounds, uint32_t* const* __restrict__ off) {
    __shared__ uint32_t warp_sums[32];
    __shared__ uint32_t carry_s;
    const uint32_t tid = threadIdx.x, per = (nb + 1023u) / 1024u;
    const uint32_t lo = min(tid * per, nb), hi = min(lo + per, nb);
    for (int k = 1; k <= rounds; k++) {
        const uint32_t* prev = off[k - 1];
        uint32_t* cur = off[k];
        uint32_t s = 0;
        for (uint32_t j = lo; j < hi; j++) s += (prev[j + 1] - prev[j] + 1u) >> 1;
        uint32_t v = s;
        #pragma unroll
        for (int d = 1; d < 32; d <<= 1) { uint32_t t = __shfl_up_sync(0xffffffffu, v, d); if ((tid & 31) >= (uint32_t)d) v += t; }
        if ((tid & 31) == 31) warp_sums[tid >> 5] = v;
        __syncthreads();
        if (tid < 32) {
            uint32_t w = warp_sums[tid], x = w;
            #pragma unroll
            for (int d = 1; d < 32; d <<= 1) { uint32_t t = __shfl_up_sync(0xffffffffu, x, d); if (tid >= (uint32_t)d) x += t; }
            warp_sums[tid] = x - w;
            if (tid == 31) carry_s = x;
        }
        __syncthreads();
        uint32_t run = warp_sums[tid >> 5] + v - s;
        for (uint32_t j = lo; j < hi; j++) { cur[j] = run; run += (prev[j + 1] - prev[j] + 1u) >> 1; }
        if (tid == 0) cur[nb] = carry_s;
        __syncthreads();                                   // cur is complete (and visible to the block) before it becomes prev
    }
}

// src[q] for every slot q of level k: first input slot in level k-1, bit 31 set when the slot is the sum of a pair
// (clear: the odd element of its bucket, copied through).
__global__ void __launch_bounds__(256) msm_aff_src_kernel(const uint32_t* __restrict__ off_prev, const uint32_t* __restrict__ off_cur, uint32_t nb,
                                                          uint32_t* __restrict__ src) {
    const uint32_t total = off_cur[nb];
    for (uint32_t q = blockIdx.x * blockDim.x + threadIdx.x; q < total; q += gridDim.x * blockDim.x) {
        uint32_t lo = 0, hi = nb;                          // invariant: off_cur[lo] <= q < off_cur[hi]
        while (hi - lo > 1) { const uint32_t mid = (lo + hi) >> 1; if (off_cur[mid] <= q) lo = mid; else hi = mid; }
        const uint32_t j = q - off_cur[lo];
        const uint32_t p0 = off_prev[lo], cnt = off_prev[lo + 1] - p0;
        src[q] = (p0 + 2u * j) | ((2u * j + 1u < cnt) ? 0x80000000u : 0u);
    }
}

// what one slot of a level is made of, and the denominator its affine addition needs
enum : int { AFF_COPY_P = 0, AFF_COPY_Q = 1, AFF_INF = 2, AFF_ADD = 3, AFF_DBL = 4 };

template <class C, class F, bool LEVEL0>
__device__ __forceinline__ int aff_fetch(const void* __restrict__ table, const uint32_t* __restrict__ entries, const void* __restrict__ prev,
                                         uint32_t s, typename C::Aff& P, typename C::Aff& Q, typename F::elem& d) {
    const uint32_t i0 = s & 0x7fffffffu;
    const bool pair = (s >> 31) != 0;
    if (LEVEL0) {
        const uint32_t e0 = entries[i0];
        P = aff_load<F>(table, (size_t)(e0 & 0x7fffffffu));
        if (e0 >> 31) P.y = F::neg(P.y);
        if (pair) {
            const uint32_t e1 = entries[i0 + 1];
            Q = aff_load<F>(table, (size_t)(e1 & 0x7fffffffu));
            if (e1 >> 31) Q.y = F::neg(Q.y);
        }
    } else {
        P = aff_load<F>(prev, (size_t)i0);
        if (pair) Q = aff_load<F>(prev, (size_t)i0 + 1);
    }
    if (!pair) return AFF_COPY_P;
    if (C::aff_is_inf(P)) return AFF_COPY_Q;
    if (C::aff_is_inf(Q)) return AFF_COPY_P;
    if (F::eq(P.x, Q.x)) {
        if (F::eq(P.y, Q.y) && !F::is_zero(P.y)) { d = F::dbl(P.y); return AFF_DBL; }
        return AFF_INF;                                    // P + (-P)
    }
    d = F::sub(Q.x, P.x);
    return AFF_ADD;
}

// pass 1: exclusive prefix products of the denominators along each thread's slots, thread total -> totals[t]
template <class C, class F, bool LEVEL0>
__global__ void __launch_bounds__(128) msm_aff_prod_kernel(const void* __restrict__ table, const uint32_t* __restrict__ entries, const void* __restrict__ prev,
                                                           const uint32_t* __restrict__ src, const uint32_t* __restrict__ off_cur, uint32_t nb,
                                                           void* __restrict__ pref, void* __restrict__ totals) {
    using E = typename F::elem; using Aff = typename C::Aff;
    const uint32_t total = off_cur[nb];
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x, stride = gridDim.x * blockDim.x;
    E run = F::one();
    #pragma unroll 1
    for (int i = 0; i < MSM_AFF_M; i++) {
        const uint64_t q64 = (uint64_t)t + (uint64_t)i * stride;
        if (q64 >= total) break;
        const uint32_t q = (uint32_t)q64;
        Aff P, Q; E d;
        const int kind = aff_fetch<C, F, LEVEL0>(table, entries, prev, src[q], P, Q, d);
        if (kind >= AFF_ADD) {
            elem_store((char*)pref + (size_t)q * Bytes<F>::ELEM, run);
            run = F::mul(run, d);
        }
    }
    elem_store((char*)totals + (size_t)t * Bytes<F>::ELEM, run);
}

// pass 2: totals[i] <- 1 / totals[i] for i < count (all non-zero by construction).  Thread u owns the strided set
// u, u + U, u + 2U, ... (coalesced across the warp), forms their product with the prefixes parked in `scratch`, inverts
// once, and unwinds.
template <class F>
__global__ void __launch_bounds__(64) msm_aff_invert_kernel(void* __restrict__ totals, void* __restrict__ scratch, uint32_t count, uint32_t U) {
    using E = typename F::elem;
    const uint32_t u = blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= U) return;
    constexpr size_t B = Bytes<F>::ELEM;
    E run = F::one();
    int last = -1;
    #pragma unroll 1
    for (int v = 0; v < MSM_AFF_S; v++) {
        const uint64_t idx = (uint64_t)u + (uint64_t)v * U;
        if (idx >= count) break;
        E x; elem_load(x, (const char*)totals + idx * B);
        elem_store((char*)scratch + idx * B, run);
        run = F::mul(run, x);
        last = v;
    }
    if (last < 0) return;
    E inv = F::inv(run);
    #pragma unroll 1
    for (int v = last; v >= 0; v--) {
        const uint64_t idx = (uint64_t)u + (uint64_t)v * U;
        E x, pre; elem_load(x, (const char*)totals + idx * B); elem_load(pre, (const char*)scratch + idx * B);
        elem_store((char*)totals + idx * B, F::mul(inv, pre));
        inv = F::mul(inv, x);
    }
}

// pass 3: back-substitution.  1/d_i = inv * pref_i, inv *= d_i; lambda = (yQ - yP) / d (or 3 xP^2 / (2 yP));
// x3 = lambda^2 - xP - xQ, y3 = lambda (xP - x3) - yP.
template <class C, class F, bool LEVEL0>
__global__ void __launch_bounds__(128) msm_aff_apply_kernel(const void* __restrict__ table, const uint32_t* __restrict__ entries, const void* __restrict__ prev,
                                                            const uint32_t* __restrict__ src, const uint32_t* __restrict__ off_cur, uint32_t nb,
                                                            const void* __restrict__ pref, const void* __restrict__ totals_inv, void* __restrict__ out) {
    using E = typename F::elem; using Aff = typename C::Aff;
    const uint32_t total = off_cur[nb];
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x, stride = gridDim.x * blockDim.x;
    if (t >= total) return;
    E inv; elem_load(inv, (const char*)totals_inv + (size_t)t * Bytes<F>::ELEM);
    int i = MSM_AFF_M - 1;
    while ((uint64_t)t + (uint64_t)i * stride >= total) i--;
    #pragma unroll 1
    for (; i >= 0; i--) {
        const uint32_t q = t + (uint32_t)i * stride;
        Aff P, Q; E d;
        const int kind = aff_fetch<C, F, LEVEL0>(table, entries, prev, src[q], P, Q, d);
        Aff r;
        if (kind >= AFF_ADD) {
            E pre; elem_load(pre, (const char*)pref + (size_t)q * Bytes<F>::ELEM);
            const E inv_d = F::mul(inv, pre);
            inv = F::mul(inv, d);
            E num;
            if (kind == AFF_ADD) num = F::sub(Q.y, P.y);
            else { const E xx = F::sqr(P.x); num = F::add(F::dbl(xx), xx); Q.x = P.x; }
            const E lam = F::mul(num, inv_d);
            r.x = F::sub(F::sub(F::sqr(lam), P.x), Q.x);
            r.y = F::sub(F::mul(lam, F::sub(P.x, r.x)), P.y);
        } else if (kind == AFF_COPY_P) r = P;
        else if (kind == AFF_COPY_Q) r = Q;
        else { r.x = F::zero(); r.y = F::zero(); }
        aff_store<F>(out, (size_t)q, r);
    }
}

// ------------------------------------------------------------------------------------------------ (4) accumulate
// Thread t owns sorted positions [t*chunk, (t+1)*chunk).  Buckets that lie entirely inside the run are written to
// buckets[]; a run's first / last segment that belongs to a bucket crossing the run boundary goes to frag_first[t] /
// frag_last[t].
// occupancy targets (measured, round 2: 5 / 6 CTAs per SM for G1 = 96 / 80 registers: 2.343 / 2.410 ms vs 2.361 ms; register caps
// of 120 / 160 that leave room for a co-resident sort CTA: e2e 49.3 vs 50.3 proofs/s - neither kept): G1 runs 4 CTAs/SM at 126 registers; G2 sits at 174 registers, 1 % over the 3-CTA limit (170), so it
// is capped there (ncu: 2 CTAs/SM left the IMAD pipe waiting on dependent-issue latency with 2 warps per scheduler)
template <class F> struct AccOcc;
#ifndef B2G_G1_CTAS
#define B2G_G1_CTAS 4
#endif
template <> struct AccOcc<Fq> { static constexpr int MIN_CTAS = B2G_G1_CTAS; };
#ifndef B2G_G2_CTAS
#define B2G_G2_CTAS 3
#endif
template <> struct AccOcc<Fq2> { static constexpr int MIN_CTAS = B2G_G2_CTAS; };

template <class C, class F>
__global__ void __launch_bounds__(128, AccOcc<F>::MIN_CTAS) msm_accumulate_kernel(const void* __restrict__ table, const uint32_t* __restrict__ entries,
                                      const uint32_t* __restrict__ offsets, uint32_t nb, uint32_t chunk,
                                      void* __restrict__ buckets, void* __restrict__ frag_first, void* __restrict__ frag_last, uint32_t slab_words) {
    using Pt = typename C::Pt; using Aff = typename C::Aff;
    const uint32_t total = offsets[nb];
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    const uint64_t start64 = (uint64_t)t * chunk;
    // slab_words != 0 (default for G1): the CTA's contiguous slab of the sorted entry list (128 runs = 32 KB at the default run
    // length) is brought into shared memory by ONE bulk asynchronous copy (cp.async.bulk -> UBLKCP, completion on an mbarrier)
    // instead of 64 strided 4-byte loads per thread
    extern __shared__ __align__(128) uint32_t slab[];
    __shared__ __align__(8) unsigned long long slab_bar;
    const uint64_t cta_first = (uint64_t)blockIdx.x * blockDim.x * chunk;
    if (slab_words) {
        const uint32_t bar = (uint32_t)__cvta_generic_to_shared(&slab_bar);
        if (threadIdx.x == 0) {
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(bar));
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncthreads();
        if (threadIdx.x == 0 && cta_first < total) {
            const uint64_t left = total - cta_first;
            const uint32_t bytes = (uint32_t)(((left < slab_words ? left : (uint64_t)slab_words) * 4 + 15) & ~15ull);    // the list is padded by 16 B
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(bar), "r"(bytes) : "memory");
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                         :: "r"((uint32_t)__cvta_generic_to_shared(slab)), "l"(entries + cta_first), "r"(bytes), "r"(bar) : "memory");
        }
        if (cta_first < total) {
            uint32_t done = 0;
            while (!done)
                asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], 0;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(done) : "r"(bar) : "memory");
        }
    }
    if (start64 >= total) return;
    const uint32_t start = (uint32_t)start64;
    const uint32_t end = (uint32_t)min((uint64_t)total, start64 + chunk);
    // bucket containing `start`: largest b with offsets[b] <= start (and non-empty by construction of the search)
    uint32_t lo = 0, hi = nb;                       // invariant: offsets[lo] <= start < offsets[hi]
    while (hi - lo > 1) { uint32_t mid = (lo + hi) >> 1; if (offsets[mid] <= start) lo = mid; else hi = mid; }
    uint32_t b = lo;
    uint32_t bucket_end = offsets[b + 1];
    while (bucket_end <= start) { b++; bucket_end = offsets[b + 1]; }    // skip empty buckets sharing the offset
    Pt acc = C::infinity();
    uint32_t seg_start = start;
    for (uint32_t pos = start; pos < end;) {
        const uint32_t e = slab_words ? slab[pos - (uint32_t)cta_first] : (entries ? entries[pos] : pos);   // entries == nullptr: `table` is a pre-reduced point list (4a)
        Aff p = aff_load<F>(table, (size_t)(e & 0x7fffffffu));
        if (e >> 31) p.y = F::neg(p.y);
        C::madd(acc, p);
        pos++;
        if (pos == bucket_end || pos == end) {
            const uint32_t bucket_start = offsets[b];
            if (bucket_start >= start && bucket_end <= end) pt_store<F>(buckets, b, acc);
            else if (seg_start == start) pt_store<F>(frag_first, t, acc);
            else pt_store<F>(frag_last, t, acc);
            acc = C::infinity();
            seg_start = pos;
            if (pos == bucket_end && pos < end) {
                do { b++; bucket_end = offsets[b + 1]; } while (bucket_end <= pos);
            }
        }
    }
}


// ------------------------------------------------------------------------------------------------ (5) fold fragments
template <class C, class F>
__global__ void __launch_bounds__(128) msm_fold_kernel(const uint32_t* __restrict__ offsets, uint32_t nb, uint32_t chunk, void* __restrict__ buckets,
                                const void* __restrict__ frag_first, const void* __restrict__ frag_last,
                                uint32_t* __restrict__ big_list, uint32_t* __restrict__ big_count) {
    using Pt = typename C::Pt;
    uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= nb) return;
    uint32_t s = offsets[b], e = offsets[b + 1];
    if (s == e) { pt_store<F>(buckets, b, C::infinity()); return; }
    uint32_t t0 = s / chunk, t1 = (e - 1) / chunk;
    if (t0 == t1) return;                                   // complete bucket, already written by (4)
    if (t1 - t0 + 1 > (uint32_t)MSM_BIG_FRAGS) { big_list[atomicAdd(big_count, 1u)] = b; return; }
    Pt acc = (s == t0 * chunk) ? pt_load<F>(frag_first, t0) : pt_load<F>(frag_last, t0);
    for (uint32_t t = t0 + 1; t <= t1; t++) { Pt q = pt_load<F>(frag_first, t); C::add(acc, q); }
    pt_store<F>(buckets, b, acc);
}

// sum of one point per thread; result valid in thread 0.  Inside a warp the partial sums travel by register shuffles
// (lane i adds lane i + d, d = 16 .. 1: the classic butterfly, every limb of the XYZZ point through __shfl_down_sync); the one
// or two warp results are then combined through shared memory.
template <class F> struct PtWords;
template <> struct PtWords<Fq> { static constexpr int N = 32; };
template <> struct PtWords<Fq2> { static constexpr int N = 64; };

template <class C, class F>
__device__ __forceinline__ typename C::Pt warp_sum_points(typename C::Pt v) {
    using Pt = typename C::Pt;
    static_assert(sizeof(Pt) == PtWords<F>::N * 4, "XYZZ point layout");
    #pragma unroll 1
    for (int d = 16; d > 0; d >>= 1) {
        Pt q;
        uint32_t* qw = reinterpret_cast<uint32_t*>(&q);
        const uint32_t* vw = reinterpret_cast<const uint32_t*>(&v);
        #pragma unroll
        for (int i = 0; i < PtWords<F>::N; i++) qw[i] = __shfl_down_sync(0xffffffffu, vw[i], d);
        if ((int)(threadIdx.x & 31) < d) C::add(v, q);
    }
    return v;
}

template <class C, class F, int NT>
__device__ __forceinline__ typename C::Pt block_sum_points(typename C::Pt v, typename C::Pt* sh) {
    static_assert(NT == 32 || NT == 64, "one or two warps");
    v = warp_sum_points<C, F>(v);
    if (NT == 32) return v;
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x == 0) { typename C::Pt q = sh[1]; C::add(v, q); }
    __syncthreads();                                       // sh may be reused by the caller's next round
    return v;
}

// Tail kernels (fold_big / reduce / sum) are latency chains on a few CTAs.  Their CTAs are kept smaller than one
// accumulation CTA (128 threads x 126 regs for G1) so that the block scheduler can slot them in as soon as a single
// accumulation CTA of a concurrently running query retires, instead of waiting for two slots on the same SM.
template <class F> struct TailThreads;
template <> struct TailThreads<Fq> { static constexpr int N = 64; };
template <> struct TailThreads<Fq2> { static constexpr int N = 32; };
constexpr int MSM_REDUCE_CHUNK_DEFAULT = 8;   // buckets per thread in the weighted reduction (B2G_MSM_REDUCE_CHUNK)

// buckets with many fragments: one CTA each
template <class C, class F>
__global__ void __launch_bounds__(TailThreads<F>::N) msm_fold_big_kernel(const uint32_t* __restrict__ offsets, uint32_t chunk, void* __restrict__ buckets,
                                    const void* __restrict__ frag_first, const void* __restrict__ frag_last,
                                    const uint32_t* __restrict__ big_list, const uint32_t* __restrict__ big_count) {
    using Pt = typename C::Pt;
    extern __shared__ __align__(32) unsigned char smem_raw[];
    Pt* sh = reinterpret_cast<Pt*>(smem_raw);
    const uint32_t nbig = *big_count;
    for (uint32_t bi = blockIdx.x; bi < nbig; bi += gridDim.x) {
        uint32_t b = big_list[bi];
        uint32_t s = offsets[b], e = offsets[b + 1];
        uint32_t t0 = s / chunk, t1 = (e - 1) / chunk;
        Pt acc = C::infinity();
        for (uint32_t t = t0 + threadIdx.x; t <= t1; t += TailThreads<F>::N) {
            Pt q = (t == t0 && s != t0 * chunk) ? pt_load<F>(frag_last, t0) : pt_load<F>(frag_first, t);
            C::add(acc, q);
        }
        Pt r = block_sum_points<C, F, TailThreads<F>::N>(acc, sh);
        if (threadIdx.x == 0) pt_store<F>(buckets, b, r);
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------------------ (6) weighted bucket sum
// sum_b (b+1) * B_b.  Thread t takes buckets [t*S, (t+1)*S): running sums give A_t = sum_j (j+1) B_{tS+j} and
// S_t = sum_j B_{tS+j}; its contribution is A_t + (t*S) * S_t (small double-and-add); a CTA tree adds them up.
template <class C, class F>
__global__ void __launch_bounds__(TailThreads<F>::N) msm_reduce_kernel(const void* __restrict__ buckets, uint32_t nb, uint32_t rchunk, void* __restrict__ partials) {
    using Pt = typename C::Pt;
    extern __shared__ __align__(32) unsigned char smem_raw[];
    Pt* sh = reinterpret_cast<Pt*>(smem_raw);
    const uint32_t t = blockIdx.x * TailThreads<F>::N + threadIdx.x;
    const uint32_t base = t * rchunk;
    Pt run = C::infinity(), acc = C::infinity();
    if (base < nb) {
        const uint32_t cnt = min(rchunk, nb - base);
        for (int j = (int)cnt - 1; j >= 0; j--) {
            Pt q = pt_load<F>(buckets, base + j);
            C::add(run, q);
            C::add(acc, run);
        }
        // acc += base * run
        if (base != 0 && !C::is_inf(run)) {
            Pt m = C::infinity();
            int top = 31 - __clz(base);
            for (int i = top; i >= 0; i--) { m = C::dbl(m); if ((base >> i) & 1u) C::add(m, run); }
            C::add(acc, m);
        }
    }
    Pt r = block_sum_points<C, F, TailThreads<F>::N>(acc, sh);
    if (threadIdx.x == 0) pt_store<F>(partials, blockIdx.x, r);
}

// sum of `count` points (count <= a few hundred) by one CTA
template <class C, class F>
__global__ void __launch_bounds__(TailThreads<F>::N) msm_sum_kernel(const void* __restrict__ pts, uint32_t count, void* __restrict__ out) {
    using Pt = typename C::Pt;
    extern __shared__ __align__(32) unsigned char smem_raw[];
    Pt* sh = reinterpret_cast<Pt*>(smem_raw);
    Pt acc = C::infinity();
    for (uint32_t i = threadIdx.x; i < count; i += TailThreads<F>::N) { Pt q = pt_load<F>(pts, i); C::add(acc, q); }
    Pt r = block_sum_points<C, F, TailThreads<F>::N>(acc, sh);
    if (threadIdx.x == 0) pt_store<F>(out, 0, r);
}

// ------------------------------------------------------------------------------------------------ host side
static uint32_t env_u32(const char* name, uint32_t dflt) {
    const char* v = getenv(name);
    if (!v || !*v) return dflt;
    long x = strtol(v, nullptr, 10);
    return x > 0 ? (uint32_t)x : dflt;
}

// reference behaviour: an off-curve point in a zkey makes G1Affine::new / G2Affine::new panic (src/zkey.rs:340-360); here
// the load fails with B2G_E_INPUT.  `what` names the points in the message.
void msm_validate_points(const void* pts_dev, uint32_t n, bool g2, cudaStream_t st, const char* what) {
    if (n == 0) return;
    struct Flag { uint32_t* d = nullptr; ~Flag() { if (d) cudaFree(d); } } flag;
    uint32_t bad = 0;
    CUDA_CHECK(cudaMalloc(&flag.d, 4));
    CUDA_CHECK(cudaMemsetAsync(flag.d, 0, 4, st));
    if (g2) msm_validate_kernel<G2, Fq2><<<(n + 255) / 256, 256, 0, st>>>(pts_dev, n, flag.d);
    else msm_validate_kernel<G1, Fq><<<(n + 255) / 256, 256, 0, st>>>(pts_dev, n, flag.d);
    g_launch_count += 1;
    CUDA_CHECK(cudaMemcpyAsync(&bad, flag.d, 4, cudaMemcpyDeviceToHost, st));
    CUDA_CHECK(cudaStreamSynchronize(st));
    if (bad) throw_error(B2G_E_INPUT, std::string(g2 ? "G2" : "G1") + " point " + std::to_string(bad - 1) + " of " + what + " is not on the curve");
}

template <class C, class F>
static void msm_build_table_t(MsmPlan& plan, const void* bases_dev, uint32_t n, cudaStream_t st) {
    const size_t aff = 2 * Bytes<F>::ELEM;
    // B2G_MSM_C is a tuning override; outside [8, 22] the window count would overflow MSM_MAX_WIN or the bucket count 2^31
    uint32_t c = env_u32("B2G_MSM_C", (uint32_t)msm_pick_c(n ? n : 1));
    if (c < 8 || c > 22) throw_error(B2G_E_SHAPE, "B2G_MSM_C must be in [8, 22]");
    plan.n = n; plan.c = (int)c; plan.nwin = msm_nwin(plan.c); plan.nbuckets = 1u << (plan.c - 1);
    if (n == 0) { plan.table = nullptr; return; }
    if ((uint64_t)n * plan.nwin >= (1ull << 31)) throw_error(B2G_E_SHAPE, "msm: n * windows exceeds 2^31 table rows");
    msm_validate_points(bases_dev, n, plan.g2, st, "the query slice");
    CUDA_CHECK(cudaMalloc(&plan.table, (size_t)n * plan.nwin * aff));
    msm_table_kernel<C, F><<<(n + 127) / 128, 128, 0, st>>>(bases_dev, n, plan.c, plan.nwin, plan.table);
    g_launch_count += 1;
    CUDA_CHECK(cudaGetLastError());
}

void msm_build_table(MsmPlan& plan, const void* bases_dev, uint32_t n, bool g2, cudaStream_t st) {
    plan.g2 = g2;
    if (g2) msm_build_table_t<G2, Fq2>(plan, bases_dev, n, st);
    else msm_build_table_t<G1, Fq>(plan, bases_dev, n, st);
}

void msm_free_table(MsmPlan& plan) { if (plan.table) cudaFree(plan.table); plan.table = nullptr; }

void msm_scratch_alloc(MsmScratch& s, uint32_t n, int nwin, uint32_t nbuckets, bool g2, bool with_sort) {
    s.g2 = g2; s.cap_n = n; s.cap_nwin = nwin; s.cap_buckets = nbuckets;
    s.chunk = env_u32(g2 ? "B2G_MSM_CHUNK_G2" : "B2G_MSM_CHUNK", env_u32("B2G_MSM_CHUNK", 64));
    const size_t pt = (g2 ? 4 * 64 : 4 * 32);
    const size_t nent = (size_t)n * nwin;
    const size_t nchunks = (nent + s.chunk - 1) / s.chunk + 1;
    s.reduce_chunk = env_u32("B2G_MSM_REDUCE_CHUNK", MSM_REDUCE_CHUNK_DEFAULT);
    const size_t npart = (size_t)nbuckets / (s.reduce_chunk * 32) + 64;
    if (with_sort) {
        CUDA_CHECK(cudaMalloc(&s.counts, (size_t)nbuckets * 4));
        CUDA_CHECK(cudaMalloc(&s.offsets, ((size_t)nbuckets + 1) * 4));
        CUDA_CHECK(cudaMalloc(&s.cursor, (size_t)nbuckets * 4));
        CUDA_CHECK(cudaMalloc(&s.entries, (nent + 8) * 4));          // + 16 B: the bulk copy of the last slab is rounded up
        CUDA_CHECK(cudaMalloc(&s.scalars_canon, ((size_t)n + 1) * sizeof(fe)));
    }
    CUDA_CHECK(cudaMalloc(&s.big_list, (size_t)nbuckets * 4));
    CUDA_CHECK(cudaMalloc(&s.big_count, 4));
    CUDA_CHECK(cudaMalloc(&s.frag_first, nchunks * pt));
    CUDA_CHECK(cudaMalloc(&s.frag_last, nchunks * pt));
    CUDA_CHECK(cudaMalloc(&s.buckets, (size_t)nbuckets * pt));
    CUDA_CHECK(cudaMalloc(&s.partials, (npart + 1) * pt));
    CUDA_CHECK(cudaMalloc(&s.result, pt)); s.result_owned = true;
    // batched-affine pre-reduction (4a): OFF by default.  Measured on B200 at 2^20 x 15 windows (profiles/r2_affine_rounds.md):
    // the 36 % multiply saving is eaten by the DRAM traffic of the three-pass structure (every 64-byte gather costs 128 B of
    // DRAM, twice per level, plus the intermediate lists) and by the latency of the shared inversion; R = 1..4 levels were
    // 20-50 % slower than the XYZZ kernel alone and throughput-neutral inside a whole proof.  B2G_MSM_AFFINE_ROUNDS=R opts in.
    {
        int rounds = 0;
        const char* ov = getenv("B2G_MSM_AFFINE_ROUNDS");
        if (ov && *ov) { long x = strtol(ov, nullptr, 10); rounds = x < 0 ? 0 : (x > MSM_AFF_MAX_ROUNDS ? MSM_AFF_MAX_ROUNDS : (int)x); }
        s.aff_cap_rounds = rounds;
        s.aff_nmax[0] = (uint32_t)nent;
        for (int k = 1; k <= rounds; k++) s.aff_nmax[k] = s.aff_nmax[k - 1] / 2 + nbuckets / 2 + 1;
        if (rounds) {
            const size_t elem = g2 ? 64 : 32, aff = 2 * elem;
            if (with_sort) {
                std::vector<uint32_t*> offs(MSM_AFF_MAX_ROUNDS + 1, nullptr);
                offs[0] = s.offsets;
                for (int k = 1; k <= rounds; k++) {
                    CUDA_CHECK(cudaMalloc(&s.aff_off[k], ((size_t)nbuckets + 1) * 4));
                    CUDA_CHECK(cudaMalloc(&s.aff_src[k], ((size_t)s.aff_nmax[k] + 1) * 4));
                    offs[k] = s.aff_off[k];
                }
                s.aff_off[0] = s.offsets;
                CUDA_CHECK(cudaMalloc(&s.aff_off_dev, (MSM_AFF_MAX_ROUNDS + 1) * sizeof(uint32_t*)));
                CUDA_CHECK(cudaMemcpy(s.aff_off_dev, offs.data(), (MSM_AFF_MAX_ROUNDS + 1) * sizeof(uint32_t*), cudaMemcpyHostToDevice));
            }
            CUDA_CHECK(cudaMalloc(&s.aff_list[0], ((size_t)s.aff_nmax[1] + 1) * aff));
            if (rounds > 1) CUDA_CHECK(cudaMalloc(&s.aff_list[1], ((size_t)s.aff_nmax[2] + 1) * aff));
            const size_t threads1 = ((size_t)s.aff_nmax[1] + MSM_AFF_M - 1) / MSM_AFF_M + 128;
            CUDA_CHECK(cudaMalloc(&s.aff_pref, ((size_t)s.aff_nmax[1] + 1) * elem));
            CUDA_CHECK(cudaMalloc(&s.aff_totals, threads1 * elem));
            CUDA_CHECK(cudaMalloc(&s.aff_tscratch, threads1 * elem));
        }
    }
    if (env_u32("B2G_MSM_TAIL_PRIORITY", 1) == 1) {
        // the tail kernels occupy a handful of CTAs for a long dependent chain: let them be dispatched ahead of the
        // thousands of pending accumulation CTAs of the other queries
        int least = 0, greatest = 0;
        CUDA_CHECK(cudaDeviceGetStreamPriorityRange(&least, &greatest));
        CUDA_CHECK(cudaStreamCreateWithPriority(&s.tail, cudaStreamNonBlocking, greatest));
        CUDA_CHECK(cudaEventCreateWithFlags(&s.ev_acc, cudaEventDisableTiming));
        CUDA_CHECK(cudaEventCreateWithFlags(&s.ev_tail, cudaEventDisableTiming));
    }
}

void msm_scratch_free(MsmScratch& s) {
    void* ptrs[] = {s.counts, s.offsets, s.cursor, s.entries, s.big_list, s.big_count, s.frag_first, s.frag_last,
                    s.buckets, s.partials, s.result_owned ? s.result : nullptr, s.scalars_canon,
                    s.aff_list[0], s.aff_list[1], s.aff_pref, s.aff_totals, s.aff_tscratch, s.aff_off_dev};
    for (void* p : ptrs) if (p) cudaFree(p);
    for (int k = 1; k <= MSM_AFF_MAX_ROUNDS; k++) { if (s.aff_off[k]) cudaFree(s.aff_off[k]); if (s.aff_src[k]) cudaFree(s.aff_src[k]); }
    if (s.tail) { cudaStreamDestroy(s.tail); cudaEventDestroy(s.ev_acc); cudaEventDestroy(s.ev_tail); }
    s = MsmScratch();
}

void msm_sort(const MsmPlan& plan, MsmScratch& s, const fe* scalars_dev, uint32_t n, bool scalars_mont, cudaStream_t st) {
    if (n > plan.n) n = plan.n;                                  // msm_bigint truncates to the shorter side
    s.sorted_n = n;
    if (n == 0 || plan.table == nullptr) return;
    if (n > s.cap_n || plan.nwin > s.cap_nwin || plan.nbuckets > s.cap_buckets || !s.entries) throw_error(B2G_E_SHAPE, "msm: sort scratch too small");
    const uint32_t nb = plan.nbuckets;
    constexpr unsigned SORT_CTA = 256;
    CUDA_CHECK(cudaMemsetAsync(s.counts, 0, (size_t)nb * 4, st));
    const unsigned pair_blocks = (unsigned)(((uint64_t)n * plan.nwin + SORT_CTA - 1) / SORT_CTA);
    msm_canon_kernel<<<(n + SORT_CTA - 1) / SORT_CTA, SORT_CTA, 0, st>>>(scalars_dev, n, scalars_mont ? 1 : 0, s.scalars_canon);
    msm_count_kernel<<<pair_blocks, SORT_CTA, 0, st>>>(s.scalars_canon, n, plan.c, plan.nwin, s.counts);
    msm_scan_kernel<<<1, 1024, 0, st>>>(s.counts, nb, s.offsets, s.cursor);
    // table rows are indexed w * plan.n + i (the table was built over plan.n bases, n may be shorter)
    msm_scatter_kernel<<<pair_blocks, SORT_CTA, 0, st>>>(s.scalars_canon, n, plan.n, plan.c, plan.nwin, s.offsets, s.cursor, s.entries);
    g_launch_count += 4;
    // level structure of the batched-affine pre-reduction (shared by every query accumulated against this sort)
    s.aff_rounds = s.aff_off_dev ? s.aff_cap_rounds : 0;
    if (s.aff_rounds) {
        msm_aff_levels_kernel<<<1, 1024, 0, st>>>(nb, s.aff_rounds, s.aff_off_dev);
        for (int k = 1; k <= s.aff_rounds; k++) {
            const unsigned blocks = (unsigned)std::min<uint64_t>(((uint64_t)s.aff_nmax[k] + 255) / 256, 1u << 20);
            msm_aff_src_kernel<<<blocks, 256, 0, st>>>(s.aff_off[k - 1], s.aff_off[k], nb, s.aff_src[k]);
        }
        g_launch_count += 1 + s.aff_rounds;
    }
    CUDA_CHECK(cudaGetLastError());
}

template <class C, class F>
static void msm_accumulate_t(const MsmPlan& plan, const MsmScratch& sorted, MsmScratch& s, cudaStream_t st) {
    using Pt = typename C::Pt;
    const size_t ptb = sizeof(Pt);
    const uint32_t n = sorted.sorted_n;
    if (n == 0 || plan.table == nullptr) { CUDA_CHECK(cudaMemsetAsync(s.result, 0, ptb, st)); return; }
    if (plan.nbuckets > s.cap_buckets || n > s.cap_n || plan.nwin > s.cap_nwin) throw_error(B2G_E_SHAPE, "msm: accumulate scratch too small");
    const uint32_t nb = plan.nbuckets, chunk = s.chunk;
    CUDA_CHECK(cudaMemsetAsync(s.big_count, 0, 4, st));
    const uint64_t nent = (uint64_t)n * plan.nwin;
    const uint32_t nthreads = (uint32_t)((nent + chunk - 1) / chunk);
    if (s.prof0) CUDA_CHECK(cudaEventRecord(s.prof0, st));
    int rounds = sorted.aff_rounds < s.aff_cap_rounds ? sorted.aff_rounds : s.aff_cap_rounds;
    if (rounds && (sorted.aff_nmax[1] > s.aff_nmax[1] || !s.aff_list[0])) rounds = 0;
    const uint32_t* offsets = sorted.offsets;
    if (rounds) {
        // (4a) R levels of pairwise affine additions inside the buckets; three kernels per level
        const void* prev = nullptr;
        for (int k = 1; k <= rounds; k++) {
            const uint32_t nk = sorted.aff_nmax[k];
            const unsigned blocks = (unsigned)(((uint64_t)nk + (uint64_t)MSM_AFF_M * 128 - 1) / ((uint64_t)MSM_AFF_M * 128));
            const uint32_t stride = blocks * 128u, U = (stride + MSM_AFF_S - 1) / MSM_AFF_S;
            void* out = s.aff_list[(k - 1) & 1];
            if (k == 1) {
                msm_aff_prod_kernel<C, F, true><<<blocks, 128, 0, st>>>(plan.table, sorted.entries, nullptr, sorted.aff_src[k], sorted.aff_off[k], nb, s.aff_pref, s.aff_totals);
                msm_aff_invert_kernel<F><<<(U + 63) / 64, 64, 0, st>>>(s.aff_totals, s.aff_tscratch, stride, U);
                msm_aff_apply_kernel<C, F, true><<<blocks, 128, 0, st>>>(plan.table, sorted.entries, nullptr, sorted.aff_src[k], sorted.aff_off[k], nb, s.aff_pref, s.aff_totals, out);
            } else {
                msm_aff_prod_kernel<C, F, false><<<blocks, 128, 0, st>>>(nullptr, nullptr, prev, sorted.aff_src[k], sorted.aff_off[k], nb, s.aff_pref, s.aff_totals);
                msm_aff_invert_kernel<F><<<(U + 63) / 64, 64, 0, st>>>(s.aff_totals, s.aff_tscratch, stride, U);
                msm_aff_apply_kernel<C, F, false><<<blocks, 128, 0, st>>>(nullptr, nullptr, prev, sorted.aff_src[k], sorted.aff_off[k], nb, s.aff_pref, s.aff_totals, out);
            }
            prev = out;
        }
        g_launch_count += 3 * rounds;
        offsets = sorted.aff_off[rounds];
        const uint32_t nthreads_r = (uint32_t)(((uint64_t)sorted.aff_nmax[rounds] + chunk - 1) / chunk);
        msm_accumulate_kernel<C, F><<<(nthreads_r + 127) / 128, 128, 0, st>>>(prev, nullptr, offsets, nb, chunk, s.buckets, s.frag_first, s.frag_last, 0u);
    } else
    {
        // measured at 2^20 (gpurun_out/r2_b20_*.json): G1 2.356 vs 2.372 ms with the bulk-staged slab, G2 7.157 vs 7.098 ms
        // -> on for G1, off for G2; B2G_ACC_BULK=0 / 1 forces it off / on for both
        static const char* bulk_env = getenv("B2G_ACC_BULK");
        const bool bulk = bulk_env && *bulk_env ? *bulk_env == '1' : !plan.g2;
        const uint32_t slab_words = bulk && (size_t)chunk * 128 * 4 <= 48 * 1024 ? chunk * 128u : 0u;
        msm_accumulate_kernel<C, F><<<(nthreads + 127) / 128, 128, (size_t)slab_words * 4, st>>>(plan.table, sorted.entries, sorted.offsets, nb, chunk, s.buckets, s.frag_first,
                                                                                                  s.frag_last, slab_words);
    }
    if (s.prof1) CUDA_CHECK(cudaEventRecord(s.prof1, st));
    cudaStream_t main_st = st;
    if (s.tail) { CUDA_CHECK(cudaEventRecord(s.ev_acc, st)); CUDA_CHECK(cudaStreamWaitEvent(s.tail, s.ev_acc, 0)); st = s.tail; }
    msm_fold_kernel<C, F><<<(nb + 127) / 128, 128, 0, st>>>(offsets, nb, chunk, s.buckets, s.frag_first, s.frag_last, s.big_list, s.big_count);
    constexpr int NT = TailThreads<F>::N;
    const size_t sh = (size_t)NT * ptb;
    msm_fold_big_kernel<C, F><<<128, NT, sh, st>>>(offsets, chunk, s.buckets, s.frag_first, s.frag_last, s.big_list, s.big_count);
    const uint32_t rchunk = s.reduce_chunk;
    const uint32_t nred = (nb + rchunk - 1) / rchunk;
    const uint32_t npart = (nred + NT - 1) / NT;
    msm_reduce_kernel<C, F><<<npart, NT, sh, st>>>(s.buckets, nb, rchunk, s.partials);
    msm_sum_kernel<C, F><<<1, NT, sh, st>>>(s.partials, npart, s.result);
    if (s.tail) { CUDA_CHECK(cudaEventRecord(s.ev_tail, s.tail)); CUDA_CHECK(cudaStreamWaitEvent(main_st, s.ev_tail, 0)); }
    g_launch_count += 5;
    CUDA_CHECK(cudaGetLastError());
}

// bucket accumulation + reduction of `plan`'s table against an already sorted scalar vector (`sorted` may be shared by
// several queries that pair the same scalars with different bases: A, B1, B2, L all use the witness)
void msm_accumulate(const MsmPlan& plan, const MsmScratch& sorted, MsmScratch& acc, cudaStream_t st) {
    if (plan.g2) msm_accumulate_t<G2, Fq2>(plan, sorted, acc, st);
    else msm_accumulate_t<G1, Fq>(plan, sorted, acc, st);
}

void msm_run(const MsmPlan& plan, MsmScratch& s, const fe* scalars_dev, uint32_t n, bool scalars_mont, cudaStream_t st) {
    msm_sort(plan, s, scalars_dev, n, scalars_mont, st);
    msm_accumulate(plan, s, s, st);
}

void msm_init_kernels() {}   // all tail kernels use < 48 KiB of dynamic shared memory

}  // namespace b2g
