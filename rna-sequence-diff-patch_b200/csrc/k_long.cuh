// k_long.cuh — one long pair whose keys do not fit the 32-bit keys of k_long2.cuh: the fallback for costs too large
// for that bound (the integer key held exactly in a double) and for non-dyadic costs (fp64 cost, int steps).  One pair
// per launch, the whole direction matrix resident.  Also the polling helpers both long-pair kernels use.
//
// Block-tiled diagonal wavefront: the matrix is cut into column panels of 32*C columns; panel w is
// owned by warp w (one warp per CTA so panels spread over all SMs) and, inside the panel, lane s
// owns C columns in registers — the same systolic row pipeline as the batched kernels.  Panels run
// concurrently as a second-level pipeline: the right-most column of panel w streams through a
// global boundary array to panel w+1, which follows ~48 rows behind (each boundary cell is its own
// ready flag: the array is preset to a sentinel and polled).  All CTAs are co-resident (cooperative launch), so the waits cannot
// deadlock.  Directions are 2 bit/cell, accumulated 16 rows per register and written with 128-bit
// stores; the traceback walks them from (m,n).
// Replaces (reference): wagnerFisher + create_paths(dp)[0] + generate_es for a pair the reference
// cannot hold in memory (~500 B per cell, SURVEY section 5).
#pragma once
#include "k_script.cuh"

struct LongArgs {
    const uint8_t *a; int m;           // 1 byte / symbol codes on the device
    const uint8_t *b; int n;
    int n_panels, n_pad;               // n_pad = n_panels * 32 * C
    uint32_t *dirs;                    // [ceil(m/16)][n_pad]
    void *bound;                       // [n_panels][m] keys (int64 or double)
    int *bound_steps;                  // [n_panels][m] (fp64 mode)
    double *dist;
    int S;
};

// boundary cells are their own "ready" flag: the array is preset to this bit pattern (memset 0x80,
// as a double a tiny negative number) which no key (an integer) and no cost (>= 0) can take, and a
// consumer polls until it changes — no fences on the integer path.
#define RSD_LONG_SENTINEL 0x8080808080808080ull

// polling must be a strong access: ptxas may (and does) collapse a loop of weak loads into one load.
// gpu scope is enough (producer and consumer are CTAs of one grid) and, unlike a volatile (= sys
// scope) load, it leaves this SM's L1 contents alone.
__device__ __forceinline__ unsigned long long ld_poll_u64(const unsigned long long *p) {
    unsigned long long v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
// the fp64 kernel publishes (steps, then fence, then key): its consumer reads the key with acquire semantics so the
// steps word it reads next is the one written before the key (PTX memory model; the relaxed poll is enough for the
// integer kernels, whose boundary cell is a single 64-bit word)
__device__ __forceinline__ unsigned long long ld_acquire_u64(const unsigned long long *p) {
    unsigned long long v;
    asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_cg_u64(unsigned long long *p, unsigned long long v) {
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}

// Values are doubles in both modes.  Integer (dyadic-cost) mode stores the int (cost<<S | steps) key
// of k_script.cuh *as a double*: |key| < 2^52, so every add is exact and DADD / DMNMX / DSETP act as a
// 53-bit integer ALU on the fp64 pipe (full rate on B200) — one instruction per min instead of the
// four a 64-bit integer min costs.  F64 mode keeps (fp64 cost, int steps) like k_script_fwd<true>.
template <bool F64, int C>
__global__ void __launch_bounds__(32)
k_long_fwd(LongArgs la, const IntCosts *__restrict__ icp, const F64Costs *__restrict__ fcp) {
    __shared__ double s_w[256];
    __shared__ double s_pub[16];
    __shared__ int s_pub_s[16];
    __shared__ uint8_t s_a[64];                    // source symbols of rows t0-31 .. t0+15 of the current block
    for (int k = threadIdx.x; k < 256; k += 32) {
        if constexpr (F64) s_w[k] = fcp->sub[k >> 4][k & 15];
        else s_w[k] = (double)(((long long)icp->w[k >> 4][k & 15] << la.S) - 1);   // (w << S) - 1, exact
    }
    __syncwarp();
    const int lane = threadIdx.x;
    const int w = blockIdx.x;                       // panel
    const int m = la.m, n = la.n;
    const int col0 = (w * 32 + lane) * C;
    const bool strip_on = col0 < n;
    double c_ins = 0, c_del = 0;
    if constexpr (F64) { c_ins = fcp->ins; c_del = fcp->del; }

    int bc[C];
#pragma unroll
    for (int c = 0; c < C; ++c) bc[c] = (col0 + c < n) ? la.b[col0 + c] : 0;
    double H[C]; int HS[F64 ? C : 1]; uint32_t acc[C];
#pragma unroll
    for (int c = 0; c < C; ++c) {
        acc[c] = 0u;
        if constexpr (F64) { H[c] = __dmul_rn((double)(col0 + c + 1), c_ins); HS[c] = col0 + c + 1; }
        else H[c] = 0.0;
    }
    double last = 0, prev_recv = 0; int last_s = 0, prev_recv_s = 0;
    const unsigned long long *bin = w > 0 ? (const unsigned long long *)la.bound + (size_t)(w - 1) * m : nullptr;
    unsigned long long *bout = (unsigned long long *)la.bound + (size_t)w * m;
    const volatile int *bin_s = (F64 && w > 0) ? la.bound_steps + (size_t)(w - 1) * m : nullptr;
    int *bout_s = F64 ? la.bound_steps + (size_t)w * m : nullptr;
    const bool publish = (w + 1 < la.n_panels);
    uint32_t *dcol = la.dirs + col0;
    const int steps = m + 31 + 16;                  // + one block so the last rows get published

#pragma unroll 1
    for (int t0 = 0; t0 < steps; t0 += 16) {
        // (0) rows finished by lane 31 during the previous block (t0-16-31 .. t0-1-31) go to the next panel:
        //     16 lanes, one coalesced non-blocking store each
        if (publish && lane < 16) {
            const int r = t0 - 47 + lane;
            if (r >= 0 && r < m) {
                if constexpr (F64) { bout_s[r] = s_pub_s[lane]; __threadfence(); }
                st_cg_u64(bout + r, (unsigned long long)__double_as_longlong(s_pub[lane]));
            }
        }
        __syncwarp();
        // (1) the 16 boundary cells lane 0 will consume in this block, fetched by lanes 0..15 in parallel
        //     The loop condition is a warp vote so all 32 lanes leave it together: a per-lane spin would
        //     leave the warp split in two for the rest of the block (every instruction issued twice).
        double bval = 0; int bval_s = 0;
        if (w > 0) {
            const bool mine = lane < 16 && t0 + lane < m;
            unsigned long long raw = 0ull;
            do {
                if (mine) raw = F64 ? ld_acquire_u64(bin + t0 + lane) : ld_poll_u64(bin + t0 + lane);
            } while (!__all_sync(RSD_FULL, raw != RSD_LONG_SENTINEL));
            if (mine) {
                bval = __longlong_as_double((long long)raw);
                if constexpr (F64) bval_s = bin_s[t0 + lane];
            }
        }
        // (2) this lane's 16 source symbols (rows t0-lane .. t0-lane+15), 4 bits each
        //     staged through shared memory: two coalesced byte loads per lane per block
        unsigned long long codes = 0ull;
        {
            const int r0 = t0 - 31 + lane, r1 = t0 + 1 + lane;
            s_a[lane] = ((unsigned)r0 < (unsigned)m) ? la.a[r0] : (uint8_t)0;
            if (lane < 15) s_a[32 + lane] = ((unsigned)r1 < (unsigned)m) ? la.a[r1] : (uint8_t)0;
            __syncwarp();
#pragma unroll
            for (int k = 0; k < 16; ++k) codes |= (unsigned long long)s_a[31 - lane + k] << (4 * k);
            __syncwarp();
        }
#pragma unroll 1
        for (int k = 0; k < 16; ++k) {
            const int t = t0 + k;
            double recv = __shfl_up_sync(RSD_FULL, last, 1);
            int recv_s = 0;
            if constexpr (F64) recv_s = __shfl_up_sync(RSD_FULL, last_s, 1);
            const double b0 = __shfl_sync(RSD_FULL, bval, k);
            int b0_s = 0;
            if constexpr (F64) b0_s = __shfl_sync(RSD_FULL, bval_s, k);
            const int i = t - lane;
            const bool row_on = strip_on && (unsigned)i < (unsigned)m;
            if (lane == 0) {
                if (w > 0) { recv = b0; recv_s = b0_s; }
                else if constexpr (F64) { recv = __dmul_rn((double)(i + 1), c_del); recv_s = i + 1; }
                else recv = 0.0;
            }
            const int rowbase = (int)((codes >> (4 * k)) & 15ull) << 4;
            if (row_on) {
                double left = recv, diag = prev_recv; int left_s = recv_s, diag_s = prev_recv_s;
                if constexpr (F64) {
                    if (i == 0) { diag = (col0 == 0) ? 0.0 : __dmul_rn((double)col0, c_ins); diag_s = col0; }
                    else if (col0 == 0) { diag = __dmul_rn((double)i, c_del); diag_s = i; }
                }
#pragma unroll
                for (int c = 0; c < C; ++c) {
                    const double wv = s_w[rowbase + bc[c]];
                    uint32_t code;
                    if constexpr (F64) {
                        const double c0 = __dadd_rn(left, c_ins), c1 = __dadd_rn(H[c], c_del), c2 = __dadd_rn(diag, wv);
                        const int s0 = left_s + 1, s1 = HS[c] + 1, s2 = diag_s + 1;
                        const double v = dmin2(c0, dmin2(c1, c2));         // same value; only one compare-select after left + ins
                        int bs = (c0 == v) ? s0 : 0x7fffffff; code = 0u;
                        if (c1 == v && s1 < bs) { bs = s1; code = 1u; }
                        if (c2 == v && s2 < bs) { bs = s2; code = 2u; }
                        diag = H[c]; diag_s = HS[c]; H[c] = v; HS[c] = bs; left = v; left_s = bs;
                    } else {
                        const double x = __dadd_rn(diag, wv);
                        const bool p_del = H[c] <= x;                 // DEL before UPD
                        const double t2 = p_del ? H[c] : x;           // (no NaNs here: select == fmin, one DSETP)
                        const bool p_ins = left <= t2;                // INS first
                        diag = H[c];
                        H[c] = p_ins ? left : t2;
                        left = H[c];
                        code = p_ins ? 0u : (p_del ? 1u : 2u);
                    }
                    acc[c] = (acc[c] << 2) | (code == 0u ? 0u : code + 1u);      // layout of k_script.cuh: 00 INS, 10 DEL, 11 UPD
                }
                last = left; prev_recv = recv;
                if constexpr (F64) { last_s = left_s; prev_recv_s = recv_s; }
                if ((i & 15) == 15 || i == m - 1) {
                    const int sh = 2 * (15 - (i & 15));
                    uint4 *dst = reinterpret_cast<uint4 *>(dcol + (size_t)(i >> 4) * la.n_pad);
#pragma unroll
                    for (int c = 0; c < C; c += 4)
                        dst[c >> 2] = make_uint4(acc[c] << sh, acc[c + 1] << sh, acc[c + 2] << sh, acc[c + 3] << sh);
                }
            }
            // lane 31 owns the panel's right-most column (row t-31 at this step): park it for the block-end store
            if (lane == 31) { s_pub[k] = last; if constexpr (F64) s_pub_s[k] = last_s; }
        }
        __syncwarp();
    }
    // the cell (m, n) lives in panel (n-1)/(32C), lane ((n-1)/C)%32, column (n-1)%C
    if (strip_on && col0 <= n - 1 && n - 1 < col0 + C) {
        const int cl = (n - 1) - col0;
        double res = 0;
#pragma unroll
        for (int c = 0; c < C; ++c) if (c == cl) res = H[c];
        if constexpr (F64) la.dist[0] = res;
        else {
            const long long key = (long long)res + (long long)m * (((long long)icp->del << la.S) + 1) + (long long)n * (((long long)icp->ins << la.S) + 1);
            la.dist[0] = (double)(key >> la.S) / (double)(1 << icp->scale_log2);
        }
    }
}

// Traceback of the long pair: one warp.  The walk is a chain of ~m+n dependent reads, so the warp
// stages a 64-row x 64-column tile of direction words around the current cell in shared memory with
// coalesced loads, the warp walks inside the tile (whole diagonal runs per iteration, shared-memory
// latency instead of an HBM miss per step), and reloads when the path leaves the tile.  Ops are written sink->origin from the
// end of tmp[0 .. m+n).
__global__ void __launch_bounds__(32) k_long_traceback(int m, int n, const uint32_t *__restrict__ dirs, int n_pad,
                                                       uint8_t *__restrict__ tmp, int32_t *__restrict__ n_ops) {
    constexpr int TR = 16, TC = 256;               // row blocks (16 rows each) x columns per tile
    __shared__ uint32_t tile[TR][TC];
    const int lane = threadIdx.x;
    int i = m, j = n;
    int pos = m + n;
    while (i > 0 && j > 0) {
        const int rb_hi = (i - 1) >> 4, rb_lo = max(rb_hi - TR + 1, 0);
        const int c_hi = j - 1, c_lo = max(c_hi - TC + 1, 0);
        const int nr = rb_hi - rb_lo + 1, nc = c_hi - c_lo + 1;
        {
            // all loads of the tile are issued before the first store: one memory latency per tile, not one per word
            uint32_t v[TR * (TC / 32)];
#pragma unroll
            for (int q = 0; q < TR * (TC / 32); ++q) {
                const int r = q / (TC / 32), c = lane + 32 * (q % (TC / 32));
                v[q] = (r < nr && c < nc) ? __ldg(dirs + (size_t)(rb_lo + r) * n_pad + c_lo + c) : 0u;
            }
#pragma unroll
            for (int q = 0; q < TR * (TC / 32); ++q) tile[q / (TC / 32)][lane + 32 * (q % (TC / 32))] = v[q];
        }
        __syncwarp();
        // Inside the tile the warp walks together: lane l looks at the cell l steps up the diagonal from
        // (i, j); the leading run of UPD cells (the common move between similar sequences) is emitted in
        // one go, then the single INS / DEL that ended it.  i, j, pos stay warp-uniform.
        const int i_min = rb_lo * 16;
        while (i > i_min && j > c_lo) {
            const int ii = i - lane, jj = j - lane;
            uint32_t code = 3u;                                            // outside the tile
            if (ii > i_min && jj > c_lo) code = dir_decode(tile[((ii - 1) >> 4) - rb_lo][(jj - 1) - c_lo], ii - 1);
            const unsigned diag_mask = __ballot_sync(RSD_FULL, code == 2u);
            const int run = diag_mask == 0xffffffffu ? 32 : __ffs(~diag_mask) - 1;
            if (lane < run) tmp[pos - 1 - lane] = (uint8_t)2;
            pos -= run; i -= run; j -= run;
            if (run < 32) {
                const uint32_t nxt = __shfl_sync(RSD_FULL, code, run);
                if (nxt == 0u) { if (lane == 0) tmp[pos - 1] = (uint8_t)0; --pos; --j; }
                else if (nxt == 1u) { if (lane == 0) tmp[pos - 1] = (uint8_t)1; --pos; --i; }
            }
        }
        __syncwarp();
    }
    if (lane == 0) {
        while (j > 0) { tmp[--pos] = 0; --j; }
        while (i > 0) { tmp[--pos] = 1; --i; }
        n_ops[0] = m + n - pos;
    }
}
