// k_dist.cuh — batched distance-only kernels (BASELINE config 2; also the scorer under wf_score).
//
// Systolic warp design: a pair's matrix is cut into strips of C columns; a lane keeps one row of
// its strip in C registers and the lanes of a group run one row apart, so the only inter-lane
// traffic is ONE __shfl_up per row (the strip's right-most cell).  Rows of the source string are
// streamed from the packed words through L1; the destination codes of a strip are turned into
// per-column selector registers once.  No shared-memory matrix, no HBM traffic besides the
// packed inputs (2 or 4 bit / symbol) and 8 B / pair of output.  Work arrives as warp tasks laid
// out on a tape of 32*P lane slots (k_plan.cuh).
//
// Replaces (reference): the double loop of wagnerFisher SED:185-222 + min_cost SED:92-128,
// read-out IR:439.
#pragma once
#include <climits>
#include <type_traits>
#include "k_plan.cuh"

struct SeqView {
    const uint32_t *words;
    const int64_t *start;
    const int32_t *len;
};

// =============================================================================================
// Fast path: 2-bit codes (ACGU), scaled-int16 values, TWO pairs per register (hi/lo halves).
// Max form: N = -H' >= 0 and v = -w = ins + del - sub clamped to >= 0 (a substitution dearer than
// delete+insert never wins, so the clamp leaves every value unchanged):
//     N[i][j] = max(N[i][j-1], N[i-1][j], N[i-1][j-1] + v(a_i, b_j)),   D = m*del + n*ins - N.
// Per packed cell (= 2 matrix cells): PRMT (v lookup for both pairs, alu pipe), one plain 32-bit add
// (halves are non-negative and < 2^16, so no carry crosses; issued as IMAD on the fma pipe) and
// VIMNMX3.U16x2 (alu pipe): 2 alu + 1 fma instructions per two cells.
//
// Two work layouts share the pieces below: k_dist_twin16 (a tape of strips, the lanes of a group one row
// apart) and k_dist_band16 (one group per lane, only the diagonal band an optimal path can reach).
// =============================================================================================

// A lane's group in the orientation of the plan (plan_swap): the rows (the twins share m), the column counts,
// D = base - N, the packed rows and columns and the shared-memory row table (the transposed one for a swapped pair).
struct TwinLane {
    int m, nA, nB, baseA, baseB;
    const uint32_t *awA, *awB, *bwA, *bwB;
    uint32_t sbaseA, sbaseB;
};
template <int C>
__device__ __forceinline__ TwinLane twin_lane(bool on, int pA, int pB, const SeqView &A, const SeqView &B,
                                              const IntCosts &ic, uint32_t sbase) {
    TwinLane t;
    t.m = 0; t.nA = 0; t.nB = 0; t.baseA = 0; t.baseB = 0;
    t.awA = A.words; t.awB = A.words; t.bwA = B.words; t.bwB = B.words;
    t.sbaseA = sbase; t.sbaseB = sbase;
    if (on) {
        const int mA = A.len[pA], mB = A.len[pB];
        t.nA = B.len[pA]; t.nB = B.len[pB];
        t.baseA = mA * ic.del + t.nA * ic.ins; t.baseB = mB * ic.del + t.nB * ic.ins;      // D = base - N either way
        t.awA = A.words + A.start[pA]; t.awB = A.words + A.start[pB];
        t.bwA = B.words + B.start[pA]; t.bwB = B.words + B.start[pB];
        t.m = mA;
        if (plan_swap(mA, t.nA, C)) { const uint32_t *x = t.awA; t.awA = t.bwA; t.bwA = x; t.m = t.nA; t.nA = mA; t.sbaseA = sbase + 16u; }
        if (plan_swap(mB, t.nB, C)) { const uint32_t *x = t.awB; t.awB = t.bwB; t.bwB = x; t.nB = mB; t.sbaseB = sbase + 16u; }
    }
    return t;
}

// per-column PRMT selectors of both twins for the strip whose first column is col0
template <int C>
__device__ __forceinline__ void twin_selectors(uint32_t (&sel)[C], bool on, const TwinLane &t, int col0) {
    static_assert(C % 16 == 0, "strip width must be a multiple of the 2-bit word");
#pragma unroll
    for (int k = 0; k < C / 16; ++k) {
        uint32_t xa = on ? __ldg(t.bwA + (col0 >> 4) + k) : 0u;
        uint32_t xb = on ? __ldg(t.bwB + (col0 >> 4) + k) : 0u;
#pragma unroll
        for (int c = 0; c < 16; ++c) {
            uint32_t ca = (xa >> (2 * c)) & 3u, cb = (xb >> (2 * c)) & 3u;
            // nibbles: [byte ca of ra][sign of it][byte cb of rb][sign of it]
            sel[k * 16 + c] = 0xC480u + ca * 0x11u + cb * 0x1100u;
        }
    }
}

// Rows are consumed in blocks of 16 so the source codes of a block sit in one register per pair: an unaligned 16-code
// window (funnel shift of the packed words a0, a1 from bit `bit` of a0), rotated so the current code is at bits [3:2]
// and can be OR-ed into the shared-memory address of the 4-entry row table.
__device__ __forceinline__ uint32_t code_window(uint32_t a0, uint32_t a1, int bit) {
    return __funnelshift_l(__funnelshift_r(a0, a1, bit), __funnelshift_r(a0, a1, bit), 2);
}
__device__ __forceinline__ uint32_t row_table(uint32_t sbase, uint32_t cur) {
    uint32_t r;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(r) : "r"(sbase | (cur & 0xCu)));
    return r;
}

// one row of a strip for both twins; left / diag: column -1 of this row and of the row above.  -> column C-1
template <int C>
__device__ __forceinline__ uint32_t twin_row(uint32_t (&H)[C], const uint32_t (&sel)[C], uint32_t ra, uint32_t rb,
                                             uint32_t left, uint32_t diag, uint32_t one) {
#pragma unroll
    for (int c = 0; c < C; ++c) {
        const uint32_t v = prmt(ra, rb, sel[c]);
        const uint32_t x = add_fma(v, diag, one);
        diag = H[c];
        H[c] = max3u16x2(x, H[c], left);
        left = H[c];
    }
    return left;
}

template <int C>
__device__ __forceinline__ uint32_t pick_col(const uint32_t (&H)[C], int cl) {
    uint32_t v = 0;
#pragma unroll
    for (int c = 0; c < C; ++c) if (c == cl) v = H[c];
    return v;
}

template <int C>
__global__ void __launch_bounds__(128)
k_dist_twin16(PlanView pv, SeqView A, SeqView B, IntCosts ic, double *__restrict__ out,
              uint32_t *__restrict__ scratch, int scratch_stride, uint32_t one) {
    __shared__ __align__(32) uint32_t s_tab[8];          // [0..3] v[a][.], [4..7] the transposed table (swapped pairs)
    if (threadIdx.x < 8) s_tab[threadIdx.x] = ic.rowtab4[threadIdx.x];
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int n_tasks = pv.totals[1];
    // two boundary columns per warp (ping-pong between passes)
    uint32_t *scr = scratch + (size_t)(blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * 2 * scratch_stride;
    const double inv_scale = 1.0 / (double)(1 << ic.scale_log2);
    const uint32_t sbase = (uint32_t)__cvta_generic_to_shared(s_tab);

    for (;;) {
        int W = 0;
        if (lane == 0) W = atomicAdd(pv.work_counter, 1);
        W = __shfl_sync(RSD_FULL, W, 0);
        if (W >= n_tasks) break;
        const TapeTask tt = plan_decode(pv, W);
        int ns = tt.ns, P = tt.P;
        if (ns == 0) {                               // class of long pairs: one group, shape from the pair
            const int p0 = pv.groups[tt.gfirst].x;
            const int m0 = A.len[p0], n0 = B.len[p0];
            ns = ((plan_swap(m0, n0, C) ? m0 : n0) + C - 1) / C; P = (ns + 31) >> 5;
        }

        for (int pass = 0; pass < P; ++pass) {
            const LaneSlot ls = tape_slot(pv, tt, ns, pass, lane);
            const TwinLane t = twin_lane<C>(ls.on, ls.pA, ls.pB, A, B, ic, sbase);
            uint32_t sel[C];
            twin_selectors<C>(sel, ls.on, t, ls.s * C);
            uint32_t H[C];
#pragma unroll
            for (int c = 0; c < C; ++c) H[c] = 0u;
            uint32_t last = 0u, prev_recv = 0u, curA = 0u, curB = 0u;
            const int steps = warp_max(ls.on ? t.m + ls.sk : 0);
            const bool has_in = __shfl_sync(RSD_FULL, (int)ls.from_scratch, 0) != 0;
            const bool has_out = __shfl_sync(RSD_FULL, (int)ls.to_scratch, 31) != 0;
            const uint32_t *scr_in = scr + ((pass & 1) ? scratch_stride : 0);
            uint32_t *scr_out = scr + ((pass & 1) ? 0 : scratch_stride);

            // Two copies of the row loop: passes without a boundary hand-off (the common case) run the lean one.
            const int mrow = ls.on ? t.m : 0;
            auto run_rows = [&](auto handoff_tag) {
                constexpr bool HANDOFF = decltype(handoff_tag)::value;
                int i = -ls.sk;
#pragma unroll 1
                for (int t0 = 0; t0 < steps; t0 += 16) {
                    {
                        const int wi = i >> 4, bit = (i & 15) * 2;            // floor division also for i < 0
                        const int w0 = max(wi, 0), w1 = max(wi + 1, 0);
                        curA = code_window(__ldg(t.awA + w0), __ldg(t.awA + w1), bit);
                        curB = code_window(__ldg(t.awB + w0), __ldg(t.awB + w1), bit);
                    }
                    const int tend = min(16, steps - t0);
#pragma unroll 2
                    for (int k = 0; k < tend; ++k, ++i) {
                        uint32_t recv = __shfl_up_sync(RSD_FULL, last, 1);
                        if (ls.lead) recv = 0u;
                        const bool row_on = (unsigned)i < (unsigned)mrow;
                        if constexpr (HANDOFF) { if (ls.from_scratch && row_on) recv = scr_in[i]; }
                        const uint32_t ra = row_table(t.sbaseA, curA), rb = row_table(t.sbaseB, curB);
                        curA = __funnelshift_r(curA, curA, 2);
                        curB = __funnelshift_r(curB, curB, 2);
                        if (row_on) {
                            last = twin_row<C>(H, sel, ra, rb, recv, prev_recv, one);
                            prev_recv = recv;
                            if constexpr (HANDOFF) { if (ls.to_scratch) scr_out[i] = last; }
                        }
                    }
                }
            };
            if (has_in || has_out) run_rows(std::true_type{}); else run_rows(std::false_type{});
            if (ls.on) {
                if (ls.s == (t.nA - 1) / C)
                    out[ls.pA] = (double)(t.baseA - (int)(pick_col<C>(H, (t.nA - 1) - ls.s * C) & 0xffffu)) * inv_scale;
                if (ls.hasB && ls.s == (t.nB - 1) / C)
                    out[ls.pB] = (double)(t.baseB - (int)(pick_col<C>(H, (t.nB - 1) - ls.s * C) >> 16)) * inv_scale;
            }
            __syncwarp();
        }
    }
}

// =============================================================================================
// Band layout: one lane per group (a twin of pairs), 32 groups = up to 64 pairs per warp task.  A lane walks the strips
// of its group one after the other and computes only the rows of each strip that an optimal path can reach.
//
// Why D stays exact: substitutions cost >= 0, so v <= ins + del, and a path through cell (i, j) of an m x n matrix
// has at most min(i, j) + min(m - i, n - j) diagonal steps.  With k = j - i, d = n - m and L = min(m, n) that bounds its
// N by (ins + del) * (L - dist(k, [min(0, d), max(0, d)])).  The diagonal path (the length difference as trailing gaps)
// is a real path worth Ndiag = sum of v(a_t, b_t) over t < L, so N >= Ndiag, and every optimal path stays inside
//     min(0, d) - q <= k <= max(0, d) + q,   q = L - ceil(Ndiag / (ins + del)).
// (In cost terms: LB(k) = g(k) + g(d - k) <= UB.)  Every value the recurrence produces is the N of a real path and 0 is
// the all-gap path, so a cell outside the band may hold 0 or anything computed from such values; the cells of an
// optimal path see the exact values of their predecessors, so N[m][n] comes out exact.  ins and del enter only as
// their sum, so a pair processed with swapped roles (plan_swap) uses the same formula.
//
// A lane's band is the hull of its twins' bands; the rows a strip computes are the union over the warp (REDUX min /
// max), so all lanes run the same rows and rows past a lane's m are skipped.  A strip hands its column C-1 to the
// next through a per-warp global buffer laid out [row][lane]: a lane reads row i (4 rows ahead of use) before it
// overwrites it, so one buffer serves every strip.  Rows the previous strip did not compute read 0.
// =============================================================================================

// q of one pair: rows aw, columns bw in the plan's orientation (the words of both are aligned on the diagonal), the
// pair's row table at `tab`; gap = ins + del > 0
__device__ __forceinline__ int band_q(const uint32_t *aw, const uint32_t *bw, int m, int n, uint32_t tab, int gap) {
    const int L = min(m, n);
    int nd = 0;
#pragma unroll 1
    for (int w = 0; 16 * w < L; ++w) {
        const uint32_t x = __ldg(aw + w), y = __ldg(bw + w);
        const int cnt = L - 16 * w;
#pragma unroll
        for (int c = 0; c < 16; ++c) {
            const uint32_t v = __byte_perm(row_table(tab, (x >> (2 * c)) << 2), 0u, 0x4440u | ((y >> (2 * c)) & 3u));
            if (c < cnt) nd += (int)v;
        }
    }
    return L - (nd + gap - 1) / gap;
}

// trace (RSD_TRACE, else null): [0] cell slots computed, [1] sum of m*n, [2] cells of the strip-padded matrices
template <int C>
__global__ void __launch_bounds__(128)
k_dist_band16(PlanView pv, SeqView A, SeqView B, IntCosts ic, double *__restrict__ out,
              uint32_t *__restrict__ scratch, int scratch_rows, uint32_t one, unsigned long long *__restrict__ trace) {
    __shared__ __align__(32) uint32_t s_tab[8];          // [0..3] v[a][.], [4..7] the transposed table (swapped pairs)
    if (threadIdx.x < 8) s_tab[threadIdx.x] = ic.rowtab4[threadIdx.x];
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int n_tasks = pv.totals[1];
    // the warp's hand-off buffer, [row][lane]: this lane's column
    uint32_t *hb = scratch + (size_t)(blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * 32 * scratch_rows + lane;
    const double inv_scale = 1.0 / (double)(1 << ic.scale_log2);
    const uint32_t sbase = (uint32_t)__cvta_generic_to_shared(s_tab);
    const int gap = ic.ins + ic.del;

    for (;;) {
        int W = 0;
        if (lane == 0) W = atomicAdd(pv.work_counter, 1);
        W = __shfl_sync(RSD_FULL, W, 0);
        if (W >= n_tasks) break;
        const TapeTask tt = plan_decode(pv, W);      // tt.ns > 0: a band plan holds no class of longer pairs
        const bool on = lane < tt.ng;
        int pA = 0, pB = 0;
        bool hasB = false;
        if (on) {
            const int2 g = pv.groups[tt.gfirst + lane];
            pA = g.x; hasB = g.y >= 0; pB = hasB ? g.y : g.x;
        }
        const TwinLane t = twin_lane<C>(on, pA, pB, A, B, ic, sbase);
        const int m = t.m;
        int klo = 0, khi = 0;                         // the lane's band, k = column - row
        if (on) {
            const int qA = band_q(t.awA, t.bwA, m, t.nA, t.sbaseA, gap);
            const int qB = hasB ? band_q(t.awB, t.bwB, m, t.nB, t.sbaseB, gap) : qA;
            klo = min(min(0, t.nA - m) - qA, min(0, t.nB - m) - qB);
            khi = max(max(0, t.nA - m) + qA, max(0, t.nB - m) + qB);
        }
        // word of the last row code: rows past m (kept for longer rows of other lanes) are skipped, and the loads of
        // their codes stay inside the lane's rows
        const int wlast = max((m - 1) >> 4, 0);
        int plo = 0, phi = -1;                        // rows of the previous strip (none before strip 0: column -1 is 0)
        long long rows_done = 0;
        uint32_t H[C];
#pragma unroll 1
        for (int s = 0; s < tt.ns; ++s) {
            const int col0 = s * C;
            // rows r (matrix row r + 1) of this strip inside the band: k = col0 + c - r for c in [0, C)
            const int lo = __reduce_min_sync(RSD_FULL, on ? max(0, col0 - khi) : INT_MAX);
            const int hi = __reduce_max_sync(RSD_FULL, on ? min(m - 1, col0 + C - 1 - klo) : -1);
            uint32_t sel[C];
            twin_selectors<C>(sel, on, t, col0);
#pragma unroll
            for (int c = 0; c < C; ++c) H[c] = 0u;
            // hand-off rows lo .. lo + 3 in flight; row r + 4 is requested when row r is taken
            uint32_t h0 = lo <= phi ? __ldcg(hb + (size_t)lo * 32) : 0u;
            uint32_t h1 = lo + 1 <= phi ? __ldcg(hb + (size_t)(lo + 1) * 32) : 0u;
            uint32_t h2 = lo + 2 <= phi ? __ldcg(hb + (size_t)(lo + 2) * 32) : 0u;
            uint32_t h3 = lo + 3 <= phi ? __ldcg(hb + (size_t)(lo + 3) * 32) : 0u;
            uint32_t diag = lo - 1 >= plo && lo - 1 <= phi ? __ldcg(hb + (size_t)(lo - 1) * 32) : 0u;
            uint32_t *hrow = hb + (size_t)lo * 32;
            int r = lo;
#pragma unroll 1
            for (int r0 = lo; r0 <= hi; r0 += 16) {
                uint32_t curA, curB;
                {
                    const int wi = r0 >> 4, bit = (r0 & 15) * 2;
                    const int w0 = min(wi, wlast), w1 = min(wi + 1, wlast);
                    curA = code_window(__ldg(t.awA + w0), __ldg(t.awA + w1), bit);
                    curB = code_window(__ldg(t.awB + w0), __ldg(t.awB + w1), bit);
                }
                const int tend = min(16, hi + 1 - r0);
#pragma unroll 2
                for (int k = 0; k < tend; ++k, ++r, hrow += 32) {
                    const uint32_t left = h0;
                    h0 = h1; h1 = h2; h2 = h3;
                    h3 = r + 4 <= phi ? __ldcg(hrow + 4 * 32) : 0u;
                    const uint32_t ra = row_table(t.sbaseA, curA), rb = row_table(t.sbaseB, curB);
                    curA = __funnelshift_r(curA, curA, 2);
                    curB = __funnelshift_r(curB, curB, 2);
                    if (r < m) __stcg(hrow, twin_row<C>(H, sel, ra, rb, left, diag, one));
                    diag = left;
                }
            }
            rows_done += hi - lo + 1;
            plo = lo; phi = hi;
        }
        if (on) {                                     // rows past m were skipped: H holds row m - 1 of the last strip
            const int cl0 = (tt.ns - 1) * C;
            out[pA] = (double)(t.baseA - (int)(pick_col<C>(H, t.nA - 1 - cl0) & 0xffffu)) * inv_scale;
            if (hasB) out[pB] = (double)(t.baseB - (int)(pick_col<C>(H, t.nB - 1 - cl0) >> 16)) * inv_scale;
        }
        if (trace) {
            if (lane == 0) atomicAdd(trace, (unsigned long long)rows_done * 64 * C);
            if (on) {
                atomicAdd(trace + 1, (unsigned long long)m * t.nA + (hasB ? (unsigned long long)m * t.nB : 0ull));
                atomicAdd(trace + 2, (unsigned long long)m * tt.ns * C * (hasB ? 2 : 1));
            }
        }
    }
}


// =============================================================================================
// General path: any symbols (2- or 4-bit packing), T = int32 (scaled, H' transform, table lookup
// of w from shared memory) or T = double (reference operation order, SED:95-109; borders are
// products SED:159,177; no FMA contraction — every add/mul is an explicit _rn intrinsic).
// =============================================================================================
template <typename T, int BITS, int C>
__global__ void __launch_bounds__(128, (sizeof(T) == 8 ? 5 : 4))
k_dist_gen(PlanView pv, SeqView A, SeqView B, const IntCosts *__restrict__ icp,
           const F64Costs *__restrict__ fcp, double *__restrict__ out,
           T *__restrict__ scratch, int scratch_stride) {
    constexpr bool F64 = sizeof(T) == 8;
    constexpr int PER = 32 / BITS;               // symbols per packed word
    static_assert(C % PER == 0, "strip width must be a multiple of the packed word");
    // The 16x16 table is replicated once per bank (group): entry e of replica r lives at word-pair /
    // word e*REP + r, so lane l always reads bank (pair) l % REP and the per-cell lookups of a warp are
    // free of bank conflicts whatever symbols the lanes hold (one table would serialise 3-4 ways).
    constexpr int REP = 128 / (int)sizeof(T);    // 16 replicas of 8-byte entries, 32 of 4-byte entries
    __shared__ T s_w[256 * REP];
    for (int k = threadIdx.x; k < 256 * REP; k += blockDim.x) {
        const int e = k / REP;
        if constexpr (F64) s_w[k] = fcp->sub[e >> 4][e & 15];
        else s_w[k] = icp->w[e >> 4][e & 15];
    }
    __syncthreads();
    T c_ins, c_del;
    double inv_scale = 1.0;
    int i_ins = 0, i_del = 0;
    if constexpr (F64) { c_ins = fcp->ins; c_del = fcp->del; }
    else { c_ins = 0; c_del = 0; i_ins = icp->ins; i_del = icp->del; inv_scale = 1.0 / (double)(1 << icp->scale_log2); }
    const int lane = threadIdx.x & 31;
    const int n_tasks = pv.totals[1];
    T *scr = scratch + (size_t)(blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * 2 * scratch_stride;
    const uint32_t sbase = (uint32_t)__cvta_generic_to_shared(s_w);

    for (;;) {
        int W = 0;
        if (lane == 0) W = atomicAdd(pv.work_counter, 1);
        W = __shfl_sync(RSD_FULL, W, 0);
        if (W >= n_tasks) break;
        const TapeTask tt = plan_decode(pv, W);
        int ns = tt.ns, P = tt.P;
        if (ns == 0) {
            const int p0 = pv.groups[tt.gfirst].x;
            ns = (B.len[p0] + C - 1) / C; P = (ns + 31) >> 5;
        }

        for (int pass = 0; pass < P; ++pass) {
            const LaneSlot ls = tape_slot(pv, tt, ns, pass, lane);
            int m = 0, n = 0;
            const uint32_t *aw = A.words, *bw = B.words;
            if (ls.on) {
                m = A.len[ls.pA]; n = B.len[ls.pA];
                aw = A.words + A.start[ls.pA]; bw = B.words + B.start[ls.pA];
            }
            const int s = ls.s;
            const int col0 = s * C;
            int bc[C];                            // shared-memory byte address of each column's table column
#pragma unroll
            for (int k = 0; k < C / PER; ++k) {
                uint32_t x = ls.on ? __ldg(bw + col0 / PER + k) : 0u;
#pragma unroll
                for (int c = 0; c < PER; ++c)
                    bc[k * PER + c] = (int)(sbase + (((x >> (BITS * c)) & ((1u << BITS) - 1u)) * REP + (lane % REP)) * (uint32_t)sizeof(T));
            }
            T H[C];
#pragma unroll
            for (int c = 0; c < C; ++c) {
                if constexpr (F64) H[c] = __dmul_rn((double)(col0 + c + 1), c_ins);   // SED:159
                else H[c] = 0;
            }
            T last = 0, prev_recv = 0;
            uint32_t cur = 0u;
            const int steps = warp_max(ls.on ? m + ls.sk : 0);
            const bool has_in = __shfl_sync(RSD_FULL, (int)ls.from_scratch, 0) != 0;
            const bool has_out = __shfl_sync(RSD_FULL, (int)ls.to_scratch, 31) != 0;
            const T *scr_in = scr + ((pass & 1) ? scratch_stride : 0);
            T *scr_out = scr + ((pass & 1) ? 0 : scratch_stride);

            auto run_rows = [&](auto handoff_tag) {          // two copies: passes without a hand-off run the lean one
            constexpr bool HANDOFF = decltype(handoff_tag)::value;
#pragma unroll (F64 ? 1 : 2)
            for (int t = 0; t < steps; ++t) {
                T recv = __shfl_up_sync(RSD_FULL, last, 1);
                const int i = t - ls.sk;
                const bool row_on = ls.on && (unsigned)i < (unsigned)m;
                if (ls.lead) {
                    if constexpr (F64) recv = __dmul_rn((double)(i + 1), c_del);          // SED:177
                    else recv = 0;
                }
                if constexpr (HANDOFF) { if (ls.from_scratch && row_on) recv = scr_in[i]; }
                if (row_on) {
                    if (i % PER == 0) cur = __ldg(aw + i / PER);
                    const uint32_t rowoff = ((cur & ((1u << BITS) - 1u)) << 4) * (uint32_t)(REP * sizeof(T)); cur >>= BITS;
                    T left = recv, diag = prev_recv;
                    if constexpr (F64) {
                        if (i == 0) diag = (s == 0) ? 0.0 : __dmul_rn((double)col0, c_ins);   // row-0 border
                        else if (s == 0) diag = __dmul_rn((double)i, c_del);
                    }
#pragma unroll
                    for (int c = 0; c < C; ++c) {
                        T w;
                        if constexpr (F64) asm volatile("ld.shared.f64 %0, [%1];" : "=d"(w) : "r"((uint32_t)bc[c] + rowoff));
                        else asm volatile("ld.shared.s32 %0, [%1];" : "=r"(w) : "r"((uint32_t)bc[c] + rowoff));
                        if constexpr (F64) {
                            const double c0 = __dadd_rn(left, c_ins);      // SED:95
                            const double c1 = __dadd_rn(H[c], c_del);      // SED:97
                            const double c2 = __dadd_rn(diag, w);          // SED:99
                            diag = H[c];
                            // SED:106-107 min(c0, c1, c2): the value of a min does not depend on the association, so
                            // the two candidates that do not involve the left neighbour are combined first and only
                            // DADD + one compare-select sit on the row's dependency chain
                            H[c] = dmin2(c0, dmin2(c1, c2));
                        } else {
                            const int t2 = addmin32(diag, w, H[c]);
                            diag = H[c];
                            H[c] = min(t2, left);
                        }
                        left = H[c];
                    }
                    last = left; prev_recv = recv;
                    if constexpr (HANDOFF) { if (ls.to_scratch) scr_out[i] = last; }
                }
            }
            };
            if (has_in || has_out) run_rows(std::true_type{}); else run_rows(std::false_type{});
            if (ls.on && s == (n - 1) / C) {
                const int cl = (n - 1) - s * C;
                T res = 0;
#pragma unroll
                for (int c = 0; c < C; ++c) if (c == cl) res = H[c];
                if constexpr (F64) out[ls.pA] = res;
                else out[ls.pA] = (double)(res + m * i_del + n * i_ins) * inv_scale;
            }
            __syncwarp();
        }
    }
}
