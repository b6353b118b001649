// k_long2.cuh — long pairs (>= a few kb per side; BASELINE config 4: 50 kb x 50 kb with traceback) on 32-bit keys.
//
// Block-tiled diagonal wavefront: the matrix is cut into column panels of 32*C columns; panel w is owned by one warp (one
// warp per CTA, so panels spread over all SMs) and, inside the panel, lane s owns C columns in registers and advances two
// rows per step (a 2 x C register tile).  The right-most column of panel w streams through a global boundary array to
// panel w+1, which follows one block behind; all CTAs are co-resident (cooperative launch), so the waits cannot deadlock.
// Keys are the (cost << S | steps) keys of k_script.cuh, modulo 2^32 (see long2_panel).  It is a *job* kernel, so that
// one cooperative launch can carry
//   * several pairs at once (BASELINE config 4 is a batch of 50 kb pairs): the CTAs of a *ring* run panel w of
//     one pair after the other, so the pipeline fill of pair k+1 overlaps the drain of pair k, and several rings
//     side by side give every SM scheduler more than one warp;
//   * a row block [r0, r1) of a pair, starting from a stored key row and leaving the key row of r1 behind
//     (`top` / `bottom`): the linear-space overflow path recomputes blocks from such checkpoint rows when the
//     direction matrix of the whole pair does not fit in HBM (rsd_long.inl);
//   * a range of column panels [w_lo, w_lo + CTAs) of a pair whose panels exceed the co-resident CTAs.
// Replaces (reference): wagnerFisher + create_paths(dp)[0] for pairs the reference cannot hold (SED:133-271).
#pragma once
#include "k_long.cuh"

struct LongJob2 {
    const uint8_t *a, *b;          // 1 byte / symbol codes on the device (whole sequences)
    int m, n;                      // whole lengths
    int r0, r1;                    // source rows of this launch (r0 a multiple of 32; r1 == m or a multiple of 32)
    int n_panels, n_pad;           // panels of the whole pair, n_pad = n_panels * 32 * C
    int w_lo, w_cnt;               // panels of this launch
    const uint32_t *top;           // keys (mod 2^32, H' form) of matrix row r0, columns 1 .. n_pad; NULL = border row (zeros)
    uint32_t *bottom;              // receives the keys of matrix row r1 (optional)
    uint32_t *dirs;                // [(r1 - r0) / 16 + 8][n_pad] direction words of this row block (DIRS kernels), *skewed*:
                                   // the word (g, column) of a column held by lane l holds the block rows 16 g - 2 l .. + 15,
                                   // i.e. what the lane computed in the steps 8 g .. 8 g + 7 — so a whole warp stores its
                                   // words at the same step, 32 * C * 4 contiguous bytes, with no per-row test
    unsigned long long *bound;     // [n_panels][bstride] right-most column of every panel, rows r0 .. r1-1: (gen << 32 | key)
    int bstride;
    unsigned gen;                  // generation tag of this launch group: a boundary word is ready when its high half equals it
                                   // (no per-call memset of the array: stale words carry older tags, a fresh pool is zeroed once)
    long long *keyacc;             // exact key of the pair's last column, carried from row block to row block
    double *dist;                  // written by the launch with r1 == m
    int S;
};

// rows of direction-word groups a row block of `rows` rows needs (skew of the last lane + the publication tail)
__host__ __device__ inline long long long2_dir_groups(long long rows) { return rows / 16 + 8; }

#define RSD_LONG2_MAX_RINGS 128
#ifndef RSD_LONG2_UNROLL
#define RSD_LONG2_UNROLL 2             // steps of the row loop unrolled together (build-time knob)
#endif
constexpr int LONG2_UNROLL = RSD_LONG2_UNROLL;
struct LongLaunch2 {
    const LongJob2 *jobs;                          // device array, ring after ring
    int n_rings;
    int ring_job0[RSD_LONG2_MAX_RINGS + 1];        // jobs [ring_job0[g], ring_job0[g+1]) run one after the other on ring g
    int ring_cta0[RSD_LONG2_MAX_RINGS + 1];        // CTAs [ring_cta0[g], ring_cta0[g+1]) form ring g
};

// One panel of one job: rows r0 .. r1-1 of the 32*C columns of panel w.
//
// The (cost << S | steps) key of a 50 kb pair needs ~36 bits.  Everything written to memory (boundary columns, checkpoint
// rows) is the key modulo 2^32.  In registers keys are held *relative to a per-lane base* (a lane's keys, and those its
// left neighbour hands over, lie within (C + 34) border steps of each other — the host checks that this stays below
// 2^30), so they compare as plain signed integers: min(left, up, diag + w) is one VIMNMX3 (distance only) or two VIMNMX
// with the two differences for the direction bits (their sign bits, as in k_script_fwd), and the chain from a cell to its
// right neighbour is one instruction — what a lone warp per scheduler waits on.  The base moves to the lane's first
// column at every block start; values cross lanes with the difference of the two bases added.  The exact key of cell
// (m, n), needed for the distance, is rebuilt from bounded row-to-row differences of the lane's last column (`full`).
template <int C, bool DIRS>
__device__ __forceinline__ void long2_panel(const LongJob2 &J, const int w, const int lane, const IntCosts *__restrict__ icp,
                                            uint32_t *s_w, uint32_t *s_pub, uint8_t *s_a) {
    __syncwarp();
    // table rows are 20 words apart: the 16 entries of an A/G/C/U pair fall into 16 different banks (rows of 16 words
    // put symbols 0 and 2, 1 and 3 on the same banks: 2-way conflicts on most lookups of ACGU data, ncu)
    for (int k = lane; k < 256; k += 32)
        s_w[(k >> 4) * 20 + (k & 15)] = (uint32_t)(((long long)icp->w[k >> 4][k & 15] << J.S) - 1);        // (w << S) - 1, fits (host check)
    __syncwarp();
    const int rows = J.r1 - J.r0, n = J.n, n_pad = J.n_pad;
    const uint8_t *arow = J.a + J.r0;
    const int col0 = (w * 32 + lane) * C;
    const bool strip_on = col0 < n;
    uint32_t H[C], acc[C], bca[C];
    const uint32_t sbase = (uint32_t)__cvta_generic_to_shared(s_w);
#pragma unroll
    for (int c = 0; c < C; ++c) {
        const int bc = (col0 + c < n) ? __ldg(J.b + col0 + c) : 0;
        H[c] = J.top ? __ldcg(J.top + col0 + c) : 0u; acc[c] = 0u; bca[c] = sbase + 4u * (uint32_t)bc;
    }
    uint32_t prev_recv1 = (J.top && col0 > 0) ? __ldcg(J.top + col0 - 1) : 0u;       // key of (row r0, the column left of this strip)
    uint32_t base = H[0], d_nb = 0u;                   // this lane's base; left neighbour's base minus this one
#pragma unroll
    for (int c = 0; c < C; ++c) H[c] -= base;
    prev_recv1 -= base;
    uint32_t last0 = 0u, last1 = H[C - 1];
    long long full = 0;
    const unsigned long long *bin = w > 0 ? J.bound + (size_t)(w - 1) * J.bstride : nullptr;
    unsigned long long *bout = J.bound + (size_t)w * J.bstride;
    const bool publish = (w + 1 < J.n_panels);
    // the tag is read from shared memory where it is needed (once per block): held in a register across the row loop it
    // changed the allocator's schedule enough to cost a lone warp 4-9 % (one 50 kb pair: 5.7 instead of 5.5 ms)
    volatile unsigned *s_gen = reinterpret_cast<volatile unsigned *>(s_pub + 32);
    if (lane == 0) *s_gen = J.gen;
    __syncwarp();
    uint32_t *dcol = DIRS ? J.dirs + col0 : nullptr;
    const int steps = (rows + 1) / 2 + 31 + 16;       // + one block so the last rows get published
    auto fetch = [&](int t0, int q) -> uint8_t { const int r = 2 * (t0 - 31) + lane + 32 * q; return ((unsigned)r < (unsigned)rows) ? __ldg(arow + r) : (uint8_t)0; };
    uint8_t pf0 = fetch(0, 0), pf1 = fetch(0, 1), pf2 = fetch(0, 2);
    unsigned long long raw_next = (w > 0 && lane < rows) ? ld_poll_u64(bin + lane) : 0ull;

#pragma unroll 1
    for (int t0 = 0; t0 < steps; t0 += 16) {
        {                                              // rebase: every key this lane holds moves with its first column
            const uint32_t delta = H[0];
            base += delta;
#pragma unroll
            for (int c = 0; c < C; ++c) H[c] -= delta;
            last0 -= delta; last1 -= delta; prev_recv1 -= delta;
            d_nb = __shfl_up_sync(RSD_FULL, base, 1) - base;
        }
        const uint32_t last_at_block_start = last1;
        if (publish) {
            const int r = 2 * (t0 - 47) + lane;
            if (r >= 0 && r < rows) st_cg_u64(bout + r, ((unsigned long long)*s_gen << 32) | (unsigned long long)s_pub[lane]);
        }
        __syncwarp();
        // The 32 boundary rows of this block were requested one block ahead (raw_next): once the panel runs far enough
        // behind its left neighbour they have arrived by now and the L2 round trip of the poll is off the critical
        // path; a sentinel means "not published yet" and is polled again.
        uint32_t bval = 0u;
        if (w > 0) {
            const bool mine = 2 * t0 + lane < rows;
            unsigned long long raw = raw_next;
            const unsigned gen = *s_gen;
            while (!__all_sync(RSD_FULL, !mine || (unsigned)(raw >> 32) == gen)) {       // warp-uniform exit (see k_long_fwd)
                if (mine) raw = ld_poll_u64(bin + 2 * t0 + lane);
            }
            bval = (uint32_t)raw;
            raw_next = (2 * (t0 + 16) + lane < rows) ? ld_poll_u64(bin + 2 * (t0 + 16) + lane) : 0ull;
        }
        unsigned long long codes0 = 0ull, codes1 = 0ull;
        {
            s_a[lane] = pf0; s_a[32 + lane] = pf1; s_a[64 + lane] = pf2;
            pf0 = fetch(t0 + 16, 0); pf1 = fetch(t0 + 16, 1); pf2 = fetch(t0 + 16, 2);
            __syncwarp();
#pragma unroll
            for (int k = 0; k < 16; ++k) {
                const uint32_t two = *reinterpret_cast<const uint16_t *>(s_a + 2 * (31 - lane + k));
                codes0 |= (unsigned long long)(two & 15u) << (4 * k);
                codes1 |= (unsigned long long)((two >> 8) & 15u) << (4 * k);
            }
            __syncwarp();
        }
        auto run16 = [&](auto steady_tag) {
        constexpr bool STEADY = decltype(steady_tag)::value;
        // steps unrolled together: 4 for the 8-column kernel with directions (a lone pair: 5.4 instead of 5.6 ms), 2 otherwise
        // (4 costs the distance-only kernel 3 %, 8 runs the 16-column kernel out of registers)
        constexpr int UNR = (LONG2_UNROLL == 2 && DIRS && C == 8) ? 4 : LONG2_UNROLL;
#pragma unroll 1
        for (int k8 = 0; k8 < 16; k8 += 8) {
#pragma unroll (UNR)
        for (int kk = 0; kk < 8; ++kk) {
            const int k = k8 + kk;
            const int i0 = 2 * (t0 + k - lane);
            const bool on0 = STEADY || (strip_on && (unsigned)i0 < (unsigned)rows);
            const bool on1 = STEADY || (strip_on && (unsigned)(i0 + 1) < (unsigned)rows);
            const uint32_t off0 = ((uint32_t)(codes0 >> (4 * k)) & 15u) * 80u, off1 = ((uint32_t)(codes1 >> (4 * k)) & 15u) * 80u;
            uint32_t w0[C], w1[C];
#pragma unroll
            for (int c = 0; c < C; ++c) {
                asm volatile("ld.shared.u32 %0, [%1];" : "=r"(w0[c]) : "r"(bca[c] + off0));
                asm volatile("ld.shared.u32 %0, [%1];" : "=r"(w1[c]) : "r"(bca[c] + off1));
            }
            uint32_t recv0 = __shfl_up_sync(RSD_FULL, last0, 1);
            uint32_t recv1 = __shfl_up_sync(RSD_FULL, last1, 1);
            const uint32_t b0 = __shfl_sync(RSD_FULL, bval, 2 * k), b1 = __shfl_sync(RSD_FULL, bval, 2 * k + 1);
            recv0 += d_nb; recv1 += d_nb;
            if (lane == 0) { recv0 = (w > 0 ? b0 : 0u) - base; recv1 = (w > 0 ? b1 : 0u) - base; }
            if (on0) {
                int left = (int)recv0, diag = (int)prev_recv1, h0[C];
#pragma unroll
                for (int c = 0; c < C; ++c) {
                    const int up = (int)H[c];
                    const int x = diag + (int)w0[c];
                    if constexpr (DIRS) {
                        const int t2 = min(up, x);                        // ties keep DEL
                        acc[c] = __funnelshift_l((uint32_t)(t2 - left), acc[c], 1);      // "not INS" (ties keep INS)
                        acc[c] = __funnelshift_l((uint32_t)(x - up), acc[c], 1);         // then "UPD rather than DEL"
                        h0[c] = min(left, t2);
                    } else h0[c] = __vimin3_s32(x, up, left);
                    diag = up; left = h0[c];
                }
                last0 = (uint32_t)left;
                if (on1) {
                    int diag1 = (int)recv0, left1 = (int)recv1;
#pragma unroll
                    for (int c = 0; c < C; ++c) {
                        const int up = h0[c];
                        const int x = diag1 + (int)w1[c];
                        int hn;
                        if constexpr (DIRS) {
                            const int t2 = min(up, x);
                            acc[c] = __funnelshift_l((uint32_t)(t2 - left1), acc[c], 1);
                            acc[c] = __funnelshift_l((uint32_t)(x - up), acc[c], 1);
                            hn = min(left1, t2);
                        } else hn = __vimin3_s32(x, up, left1);
                        diag1 = up; H[c] = (uint32_t)hn; left1 = hn;
                    }
                    last1 = (uint32_t)left1;
                } else {
#pragma unroll
                    for (int c = 0; c < C; ++c) { H[c] = (uint32_t)h0[c]; if constexpr (DIRS) acc[c] <<= 2; }
                    last1 = last0;
                }
                prev_recv1 = recv1;
            } else if constexpr (DIRS && !STEADY) {
#pragma unroll
                for (int c = 0; c < C; ++c) acc[c] <<= 4;
            }
            if (lane == 31) { s_pub[2 * k] = last0 + base; s_pub[2 * k + 1] = last1 + base; }      // absolute keys
        }
        if constexpr (DIRS) {
            // the 16 rows of the last 8 steps, all lanes at once: 32 * C consecutive words of group (t0 + k8) / 8
            uint4 *dst = reinterpret_cast<uint4 *>(dcol + (size_t)((t0 + k8) >> 3) * n_pad);
#pragma unroll
            for (int c = 0; c < C; c += 4) __stcg(dst + (c >> 2), make_uint4(acc[c], acc[c + 1], acc[c + 2], acc[c + 3]));
        }
        }
        };
        if (2 * (t0 - 31) >= 0 && 2 * (t0 + 15) + 1 <= rows - 1) run16(std::true_type{}); else run16(std::false_type{});
        __syncwarp();
        full += (long long)(int)(last1 - last_at_block_start);          // <= 32 bounded row-to-row differences (host check)
    }
    if (J.bottom) {
#pragma unroll
        for (int c = 0; c < C; ++c) __stcg(J.bottom + col0 + c, H[c] + base);
    }
    if (strip_on && col0 <= n - 1 && n - 1 < col0 + C) {
        // `full` follows column C-1 of this lane from row r0 to row r1; keyacc holds the exact key of that column at row r0
        const long long at_r1 = *J.keyacc + full;
        if (J.r1 == J.m) {
            const int cl = (n - 1) - col0;
            uint32_t res = 0u;
#pragma unroll
            for (int c = 0; c < C; ++c) if (c == cl) res = H[c];
            const long long hkey = at_r1 + (long long)(int)(res - H[C - 1]);      // column cl lies at most C-1 cells to the left
            const long long key = hkey + (long long)J.m * (((long long)icp->del << J.S) + 1) + (long long)n * (((long long)icp->ins << J.S) + 1);
            J.dist[0] = (double)(key >> J.S) / (double)(1 << icp->scale_log2);
        }
        *J.keyacc = at_r1;
    }
}

template <int C, bool DIRS>
__global__ void __launch_bounds__(32)
k_long2(const LongLaunch2 L, const IntCosts *__restrict__ icp) {
    __shared__ uint32_t s_w[320];
    __shared__ uint32_t s_pub[33];                  // [32]: the generation tag of the job in hand
    __shared__ __align__(4) uint8_t s_a[96];
    const int lane = threadIdx.x;
    int g = 0;
    while (g + 1 < L.n_rings && (int)blockIdx.x >= L.ring_cta0[g + 1]) ++g;
    const int wl = (int)blockIdx.x - L.ring_cta0[g];
    for (int j = L.ring_job0[g]; j < L.ring_job0[g + 1]; ++j) {
        const LongJob2 J = L.jobs[j];
        if (wl < J.w_cnt) long2_panel<C, DIRS>(J, J.w_lo + wl, lane, icp, s_w, s_pub, s_a);
    }
}

// Traceback of one row block of every pair of a batch: one warp per pair, the tile walk of k_long_traceback, from the
// state (i, j, pos) the block below left behind down to row r0.  Ops are written sink -> origin from the end of tmp.
struct LongTb2 {
    int m, n, r0, n_pad, C;        // C: columns per lane of the forward kernel (the skew of a column's words is 2 * its lane)
    const uint32_t *dirs;          // direction words of the rows r0 .. (block-relative and skewed, as the forward kernel wrote them)
    uint8_t *tmp;                  // [m + n]
    int *state;                    // {i, j, pos, started}; started == 0: begin at (m, n)
    int32_t *n_ops;
    int last;                      // this is the pair's top block (r0 == 0): finish the borders and count
};

__global__ void __launch_bounds__(32) k_long2_traceback(const LongTb2 *__restrict__ jobs) {
    // 32 groups (512 skewed row positions: the rows i-449 .. i of every column) x 384 columns = 48 KB of direction words,
    // brought in with cp.async (16 bytes per request, all of a tile in flight together, no staging registers): one
    // memory round trip per ~384 path steps.  (16 x 256 tiles through registers: 1.33 ms per 50 kb pair, of which
    // ~80 % was waiting for the 258 tile loads.)
    constexpr int TR = 32, TC = 384;
    __shared__ __align__(16) uint32_t tile[TR][TC];
    const LongTb2 J = jobs[blockIdx.x];
    const int lane = threadIdx.x;
    int i = J.state[0], j = J.state[1], pos = J.state[2];
    if (J.state[3] == 0) { i = J.m; j = J.n; pos = J.m + J.n; }
    const int r0 = J.r0, n_pad = J.n_pad;
    const int logC = J.C == 4 ? 2 : J.C == 8 ? 3 : 4;
    const uint32_t tile_s = (uint32_t)__cvta_generic_to_shared(&tile[0][0]);
    while (i > r0 && j > 0) {
        // groups that hold the rows <= i of every column of the tile: row r of a column of lane l sits at position r + 2 l
        const int rb_hi = (i - 1 - r0 + 62) >> 4, rb_lo = max(rb_hi - TR + 1, 0);
        // columns: a 16-byte aligned window that ends at or just after column j-1 (n_pad is a multiple of 128)
        const int c_lo = max(((j - 1) | 3) - (TC - 1), 0);
        const int nr = rb_hi - rb_lo + 1, nc4 = min(TC, n_pad - c_lo) >> 2;       // 16-byte pieces per row inside the matrix
        for (int r = 0; r < nr; ++r) {
            const uint32_t *src = J.dirs + (size_t)(rb_lo + r) * n_pad + c_lo;
#pragma unroll
            for (int q = 0; q < TC / 4 / 32; ++q) {
                const int c4 = lane + 32 * q;
                if (c4 < nc4)
                    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(tile_s + (uint32_t)((r * TC + 4 * c4) * 4)), "l"(src + 4 * c4) : "memory");
            }
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        __syncwarp();
        const int i_min = r0 + rb_lo * 16;               // rows above this (block-relative >= 16 rb_lo) are inside the tile for every lane
        while (i > i_min && j > c_lo) {
            const int ii = i - lane, jj = j - lane;
            uint32_t code = 3u;
            if (ii > i_min && jj > c_lo) {
                const int pos16 = (ii - 1 - r0) + 2 * (((jj - 1) >> logC) & 31);
                code = dir_decode(tile[(pos16 >> 4) - rb_lo][(jj - 1) - c_lo], pos16);
            }
            const unsigned diag_mask = __ballot_sync(RSD_FULL, code == 2u);
            const int run = diag_mask == 0xffffffffu ? 32 : __ffs(~diag_mask) - 1;
            if (lane < run) J.tmp[pos - 1 - lane] = (uint8_t)2;
            pos -= run; i -= run; j -= run;
            if (run < 32) {
                const uint32_t nxt = __shfl_sync(RSD_FULL, code, run);
                if (nxt == 0u) { if (lane == 0) J.tmp[pos - 1] = (uint8_t)0; --pos; --j; }
                else if (nxt == 1u) { if (lane == 0) J.tmp[pos - 1] = (uint8_t)1; --pos; --i; }
            }
        }
        __syncwarp();
    }
    if (J.last) {
        // borders: row 0 is all inserts (SED:146-164), column 0 all deletes (SED:167-182)
        const int nj = j, ni = i;
        for (int k = lane; k < nj; k += 32) J.tmp[pos - 1 - k] = 0;
        pos -= nj;
        for (int k = lane; k < ni; k += 32) J.tmp[pos - 1 - k] = 1;
        pos -= ni; i = 0; j = 0;
        if (lane == 0) J.n_ops[0] = J.m + J.n - pos;
    }
    if (lane == 0) { J.state[0] = i; J.state[1] = j; J.state[2] = pos; J.state[3] = 1; }
}

// packed scripts: one CTA per pair, op + entered cell via two block scans (same as k_finalize, unpacked input)
struct LongEmit2 { const uint8_t *tmp; int m, n; const int32_t *n_ops; uint8_t *op; int32_t *oi, *oj; };

__global__ void __launch_bounds__(1024) k_long2_emit(const LongEmit2 *__restrict__ jobs) {
    __shared__ int s_ai[1024], s_bj[1024];
    __shared__ int carry_i, carry_j;
    const LongEmit2 J = jobs[blockIdx.x];
    const int tid = threadIdx.x;
    const int k_ops = J.n_ops[0];
    const uint8_t *src = J.tmp + ((int64_t)J.m + J.n - k_ops);
    if (tid == 0) { carry_i = 0; carry_j = 0; }
    __syncthreads();
    for (int base = 0; base < k_ops; base += 1024) {
        const int k = base + tid;
        const int o = k < k_ops ? src[k] : 3;
        s_ai[tid] = (o == 1 || o == 2); s_bj[tid] = (o == 0 || o == 2);
        __syncthreads();
        for (int off = 1; off < 1024; off <<= 1) {
            int xi = tid >= off ? s_ai[tid - off] : 0, xj = tid >= off ? s_bj[tid - off] : 0;
            __syncthreads();
            s_ai[tid] += xi; s_bj[tid] += xj;
            __syncthreads();
        }
        const int vi = carry_i + s_ai[tid], vj = carry_j + s_bj[tid];
        if (k < k_ops) { J.op[k] = (uint8_t)o; if (J.oi) J.oi[k] = vi; if (J.oj) J.oj[k] = vj; }
        __syncthreads();
        if (tid == 1023) { carry_i = vi; carry_j = vj; }
        __syncthreads();
    }
}
