// rsd_api.cu — the C ABI of librsd.so (include/rsd.h): context, cost classification, packing,
// buffer management and kernel dispatch.  No torch types, no CPU fallback: every compute entry
// point needs a CUDA device and says so when there is none.
#include "../../include/rsd.h"
#include "rsd_ctx.cuh"

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <algorithm>
#include <atomic>
#include <string>
#include <thread>
#include <vector>
#include <chrono>

#include "k_dist.cuh"
#include "k_matrix.cuh"
#include "k_ubench.cuh"
#include "k_script.cuh"
#include "k_search.cuh"
#include "k_sim.cuh"
#include "k_long.cuh"
#include "k_long2.cuh"
#include "k_ingest.cuh"
#include "k_layout.cuh"

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>

// ------------------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";
int rsd_fail(int code, const char *fmt, ...) {
    va_list ap; va_start(ap, fmt); vsnprintf(g_err, sizeof g_err, fmt, ap); va_end(ap);
    return code;
}
extern "C" const char *rsd_last_error(void) { return g_err; }
extern "C" int rsd_abi_version(void) { return RSD_ABI_VERSION; }

extern "C" int rsd_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

// ------------------------------------------------------------------------------------------------
// context
// ------------------------------------------------------------------------------------------------
extern "C" int rsd_create(int device, rsd_ctx **out) {
    if (!out) return rsd_fail(RSD_EINVAL, "rsd_create: out is NULL");
    rsd_ctx *c = new (std::nothrow) rsd_ctx();
    if (!c) return rsd_fail(RSD_ENOMEM, "rsd_create: out of host memory");
    c->device = device;
    *out = c;
    return RSD_OK;
}

int rsd_ctx::ensure_device() {
    if (inited) {
        if (pid != getpid())
            return rsd_fail(RSD_EINVAL, "rsd: context used after fork(); create a new context in the child process");
        cudaError_t e = cudaSetDevice(device);
        if (e != cudaSuccess) return rsd_fail(RSD_ECUDA, "cudaSetDevice(%d): %s", device, cudaGetErrorString(e));
        return RSD_OK;
    }
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        cudaGetLastError();
        return rsd_fail(RSD_ENODEV, "rsd: no CUDA device available (%s); librsd has no CPU fallback",
                        e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
    }
    if (device < 0 || device >= n) return rsd_fail(RSD_EINVAL, "rsd: device %d out of range (0..%d)", device, n - 1);
    RSD_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    RSD_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10)
        return rsd_fail(RSD_ENODEV, "rsd: device %d is sm_%d%d; this library is built for sm_100a only", device,
                        prop.major, prop.minor);
    sm_count = prop.multiProcessorCount;
    RSD_CUDA(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
    RSD_CUDA(cudaStreamCreateWithFlags(&stream2, cudaStreamNonBlocking));
    RSD_CUDA(cudaStreamCreateWithFlags(&copy_stream, cudaStreamNonBlocking));
    RSD_CUDA(cudaStreamCreateWithFlags(&d2h_stream, cudaStreamNonBlocking));
    RSD_CUDA(cudaEventCreateWithFlags(&ev_len, cudaEventDisableTiming));
    RSD_CUDA(cudaEventCreateWithFlags(&ev_plans, cudaEventDisableTiming));
    RSD_CUDA(cudaEventCreateWithFlags(&ev_tab, cudaEventDisableTiming));
    RSD_CUDA(cudaEventCreateWithFlags(&ev_sync, cudaEventDisableTiming));
    for (int k = 0; k < RSD_MAX_CHUNKS; ++k) RSD_CUDA(cudaEventCreate(&ev_chunk[k]));
    RSD_CUDA(cudaEventCreate(&ev_begin));
    RSD_CUDA(cudaEventCreate(&ev0));
    RSD_CUDA(cudaEventCreate(&ev1));
    for (int k = 0; k < RSD_MAX_CHUNKS; ++k) {
        RSD_CUDA(cudaEventCreate(&ev_t0[k])); RSD_CUDA(cudaEventCreate(&ev_t1[k]));
        RSD_CUDA(cudaEventCreateWithFlags(&ev_done[k], cudaEventDisableTiming));
    }
    RSD_CUDA(cudaMalloc(&d_ic, sizeof(IntCosts)));
    RSD_CUDA(cudaMalloc(&d_fc, sizeof(F64Costs)));
    pid = getpid();
    inited = true;
    return RSD_OK;
}

extern "C" int rsd_destroy(rsd_ctx *c) {
    if (!c) return RSD_OK;
    if (c->inited && c->pid == getpid()) {
        cudaSetDevice(c->device);
        cudaStreamSynchronize(c->stream);
        c->free_all();
        cudaFree(c->d_ic); cudaFree(c->d_fc);
        cudaEventDestroy(c->ev0); cudaEventDestroy(c->ev1);
        cudaStreamDestroy(c->stream); cudaStreamDestroy(c->stream2); cudaStreamDestroy(c->copy_stream); cudaStreamDestroy(c->d2h_stream);
        cudaEventDestroy(c->ev_sync); cudaEventDestroy(c->ev_len); cudaEventDestroy(c->ev_plans); cudaEventDestroy(c->ev_tab); cudaEventDestroy(c->ev_begin);
        for (int k = 0; k < RSD_MAX_CHUNKS; ++k) { cudaEventDestroy(c->ev_chunk[k]); cudaEventDestroy(c->ev_t0[k]); cudaEventDestroy(c->ev_t1[k]); cudaEventDestroy(c->ev_done[k]); }
    }
    delete c;
    return RSD_OK;
}

extern "C" int rsd_host_alloc(void **out, int64_t bytes) {
    if (!out || bytes < 0) return rsd_fail(RSD_EINVAL, "rsd_host_alloc: bad arguments");
    cudaError_t e = cudaMallocHost(out, (size_t)std::max<int64_t>(bytes, 1));
    if (e != cudaSuccess) { cudaGetLastError(); return rsd_fail(RSD_ENOMEM, "cudaMallocHost(%lld): %s", (long long)bytes, cudaGetErrorString(e)); }
    return RSD_OK;
}
extern "C" int rsd_host_free(void *p) {
    if (p) cudaFreeHost(p);
    return RSD_OK;
}

extern "C" int64_t rsd_launch_count(rsd_ctx *c) { return c ? c->launches : 0; }
extern "C" int rsd_set_timing(rsd_ctx *c, int on) { if (!c) return rsd_fail(RSD_EINVAL, "ctx is NULL"); c->timing = on != 0; return RSD_OK; }
extern "C" double rsd_last_kernel_ms(rsd_ctx *c) {
    if (c && c->last_ms_override > 0.0) return c->last_ms_override;
    if (!c || !c->inited || !c->timed) return 0.0;
    float ms = 0.f;
    if (cudaEventSynchronize(c->ev1) != cudaSuccess) return 0.0;
    if (cudaEventElapsedTime(&ms, c->ev0, c->ev1) != cudaSuccess) return 0.0;
    return (double)ms;
}

// ------------------------------------------------------------------------------------------------
// costs + numeric-mode classifier
// ------------------------------------------------------------------------------------------------
extern "C" int rsd_set_costs(rsd_ctx *c, double ins, double del, const double *sub) {
    if (!c || !sub) return rsd_fail(RSD_EINVAL, "rsd_set_costs: NULL argument");
    auto bad = [](double v) { return !(v >= 0.0) || std::isinf(v); };
    if (bad(ins) || bad(del)) return rsd_fail(RSD_ECOSTS, "rsd_set_costs: insert/delete cost must be finite and >= 0");
    for (int a = 0; a < 15; ++a)
        for (int b = 0; b < 15; ++b)
            if (a != b && bad(sub[a * 15 + b]))
                return rsd_fail(RSD_ECOSTS, "rsd_set_costs: update cost [%d][%d] must be finite and >= 0", a, b);
    c->ins = ins; c->del = del;
    for (int a = 0; a < 15; ++a)
        for (int b = 0; b < 15; ++b) c->sub[a][b] = a == b ? 0.0 : sub[a * 15 + b];
    c->have_costs = true;
    return RSD_OK;
}

int rsd_ctx::classify(uint32_t symmask, int64_t max_m, int64_t max_n, int bits, int force_mode, ModeInfo &mi) const {
    if (!have_costs) return rsd_fail(RSD_EINVAL, "rsd: rsd_set_costs has not been called");
    memset(&mi, 0, sizeof mi);
    mi.fc.ins = ins; mi.fc.del = del;
    for (int a = 0; a < 15; ++a)
        for (int b = 0; b < 15; ++b) mi.fc.sub[a][b] = a == b ? 0.0 : sub[a][b];
    // reachable costs: ins, del, sub[a][b] for a != b both present
    double reach[2 + 15 * 15]; int nr = 0;
    reach[nr++] = ins; reach[nr++] = del;
    for (int a = 0; a < 15; ++a) if (symmask >> a & 1)
        for (int b = 0; b < 15; ++b) if (a != b && (symmask >> b & 1)) reach[nr++] = sub[a][b];
    int k = -1;
    for (int kk = 0; kk <= 16 && k < 0; ++kk) {
        bool ok = true;
        for (int r = 0; r < nr && ok; ++r) {
            double s = std::ldexp(reach[r], kk);
            ok = s == std::floor(s) && s < 1073741824.0;
        }
        if (ok) k = kk;
    }
    bool i32_ok = false, i16_ok = false, fast_ok = false;
    if (k >= 0) {
        IntCosts &ic = mi.ic;
        ic.scale_log2 = k;
        ic.ins = (int32_t)std::ldexp(ins, k); ic.del = (int32_t)std::ldexp(del, k);
        int64_t maxabsw = (int64_t)ic.ins + ic.del;
        bool w8 = true;
        for (int a = 0; a < 16; ++a)
            for (int b = 0; b < 16; ++b) {
                int64_t w;
                if (a == b) w = -((int64_t)ic.ins + ic.del);
                else if (a < 15 && b < 15 && (symmask >> a & 1) && (symmask >> b & 1))
                    w = (int64_t)std::ldexp(sub[a][b], k) - ic.ins - ic.del;
                else w = 0;                                   // unreachable entry
                if (std::llabs(w) > maxabsw) maxabsw = std::llabs(w);
                if (a < 4 && b < 4 && (w < -127)) w8 = false;            // v = max(0, -w) must fit a non-negative int8
                ic.w[a][b] = (int32_t)std::max<int64_t>(std::min<int64_t>(w, INT32_MAX), INT32_MIN);
            }
        // |H'| <= i*del + j*ins on the extended (strip-padded) matrix
        const int64_t pad_n = max_n + 64;
        const double bound = (double)max_m * ic.del + (double)pad_n * ic.ins + (double)maxabsw;
        i32_ok = bound < 2147483000.0;
        // the int16x2 kernel may swap the roles of the two sequences: both orientations must fit
        const double bound_sw = (double)max_n * ic.ins + (double)(max_m + 64) * ic.del + (double)maxabsw;
        i16_ok = std::max(bound, bound_sw) < 65000.0;             // unsigned 16-bit N = -H'
        fast_ok = i16_ok && w8 && bits == 2 && (symmask & ~0xFu) == 0;
        if (fast_ok)
            for (int a = 0; a < 4; ++a) {
                uint32_t r = 0;
                uint32_t rt = 0;
                for (int b = 0; b < 4; ++b) { r |= (uint32_t)std::max(0, -ic.w[a][b]) << (8 * b); rt |= (uint32_t)std::max(0, -ic.w[b][a]) << (8 * b); }
                ic.rowtab4[a] = r; ic.rowtab4[4 + a] = rt;
            }
    }
    int mode;
    if (force_mode == 0) mode = fast_ok ? RSD_MODE_I16X2 : (i32_ok ? RSD_MODE_I32 : RSD_MODE_F64);
    else if (force_mode == RSD_MODE_I16X2) {
        if (!fast_ok) return rsd_fail(RSD_EINVAL, "rsd: I16X2 mode not exact/applicable for these costs, symbols or lengths");
        mode = force_mode;
    } else if (force_mode == RSD_MODE_I32) {
        if (!i32_ok) return rsd_fail(RSD_EINVAL, "rsd: I32 mode not exact for these costs (not dyadic) or lengths");
        mode = force_mode;
    } else if (force_mode == RSD_MODE_F64) mode = force_mode;
    else return rsd_fail(RSD_EINVAL, "rsd: unknown force_mode %d", force_mode);
    mi.mode = mode;
    mi.k = k < 0 ? 0 : k;
    mi.dyadic = k >= 0; mi.i16_ok = i16_ok; mi.i32_ok = i32_ok;
    return RSD_OK;
}

extern "C" int rsd_classify(rsd_ctx *c, uint32_t symmask, int64_t max_m, int64_t max_n, int force_mode,
                            int *mode_out, int *scale_log2_out) {
    if (!c) return rsd_fail(RSD_EINVAL, "ctx is NULL");
    ModeInfo mi;
    int bits = (symmask & ~0xFu) == 0 ? 2 : 4;
    int rc = c->classify(symmask, max_m, max_n, bits, force_mode, mi);
    if (rc) return rc;
    if (mode_out) *mode_out = mi.mode;
    if (scale_log2_out) *scale_log2_out = mi.k;
    return RSD_OK;
}

int rsd_ctx::upload_costs(const ModeInfo &mi, cudaStream_t st) {
    // staged through pinned-free small copies; cudaMemcpyAsync from pageable memory copies the
    // source before returning, so the stack ModeInfo is safe.
    RSD_CUDA(cudaMemcpyAsync(d_ic, &mi.ic, sizeof(IntCosts), cudaMemcpyHostToDevice, st));
    RSD_CUDA(cudaMemcpyAsync(d_fc, &mi.fc, sizeof(F64Costs), cudaMemcpyHostToDevice, st));
    return RSD_OK;
}

// ------------------------------------------------------------------------------------------------
// packing (ingest)
// ------------------------------------------------------------------------------------------------
extern "C" int64_t rsd_pack_words(const int32_t *len, int64_t n, int bits) {
    if (!len || (bits != 2 && bits != 4)) return -1;
    const int per = 32 / bits;
    int64_t w = 0;
    for (int64_t i = 0; i < n; ++i) w += (len[i] + per - 1) / per;
    return w + 4;
}

extern "C" int rsd_pack(const uint8_t *codes, const int64_t *off, int64_t n, int bits,
                        uint32_t *words, int64_t *start, int32_t *len, uint32_t *symmask_inout) {
    if (!off || !words || !start || !len || (n > 0 && !codes)) return rsd_fail(RSD_EINVAL, "rsd_pack: NULL argument");
    if (bits != 2 && bits != 4) return rsd_fail(RSD_EINVAL, "rsd_pack: bits must be 2 or 4");
    const int per = 32 / bits;
    const uint32_t lim = 1u << bits;
    // pass 1 (serial, cheap): lengths and word offsets
    int64_t w = 0;
    for (int64_t i = 0; i < n; ++i) {
        const int64_t L = off[i + 1] - off[i];
        if (L < 0 || L > INT32_MAX) return rsd_fail(RSD_EINVAL, "rsd_pack: bad offsets at sequence %lld", (long long)i);
        start[i] = w; len[i] = (int32_t)L;
        w += (L + per - 1) / per;
    }
    for (int p = 0; p < 4; ++p) words[w + p] = 0;
    // pass 2: the packing itself, sequences split over the host threads (large batches only)
    const int64_t total = n ? off[n] - off[0] : 0;
    int n_thr = 1;
    if (total >= (1 << 22)) n_thr = (int)std::min<int64_t>(std::max(1u, std::thread::hardware_concurrency()), 32);
    std::vector<uint32_t> masks((size_t)n_thr, 0u);
    std::vector<int64_t> bad((size_t)n_thr, -1);
    // eight symbols at a time: one 64-bit load, a range check on all bytes, and a shift-or cascade that squeezes
    // the low `bits` of every byte together (2-bit: 8 symbols -> 16 bits, 4-bit: 8 symbols -> 32 bits)
    auto squeeze8 = [bits](uint64_t x) -> uint32_t {
        if (bits == 2) {
            x = (x | (x >> 6)) & 0x000F000F000F000Full;
            x = (x | (x >> 12)) & 0x000000FF000000FFull;
            x = (x | (x >> 24)) & 0xFFFFull;
        } else {
            x = (x | (x >> 4)) & 0x00FF00FF00FF00FFull;
            x = (x | (x >> 8)) & 0x0000FFFF0000FFFFull;
            x = (x | (x >> 16)) & 0xFFFFFFFFull;
        }
        return (uint32_t)x;
    };
    const uint64_t hi_bits = bits == 2 ? 0xFCFCFCFCFCFCFCFCull : 0xF0F0F0F0F0F0F0F0ull;
    auto work = [&](int t) {
        const int64_t i0 = n * t / n_thr, i1 = n * (t + 1) / n_thr;
        uint32_t mask = 0;
        for (int64_t i = i0; i < i1; ++i) {
            const int64_t L = len[i];
            const uint8_t *s = codes + off[i];
            uint32_t *dst = words + start[i];
            int64_t k = 0;
            for (; k + per <= L; k += per) {                       // full words
                uint64_t x0, x1 = 0;
                memcpy(&x0, s + k, 8);
                if (bits == 2) memcpy(&x1, s + k + 8, 8);
                if ((x0 | x1) & hi_bits) { if (bad[(size_t)t] < 0) bad[(size_t)t] = i; break; }
                const uint32_t word = bits == 2 ? (squeeze8(x0) | (squeeze8(x1) << 16)) : squeeze8(x0);
                if (bits == 2) {                                   // which of the four symbols occur: field-parallel
                    const uint32_t lo = word & 0x55555555u, hi = (word >> 1) & 0x55555555u;
                    if ((~lo & ~hi) & 0x55555555u) mask |= 1u;
                    if (lo & ~hi) mask |= 2u;
                    if (~lo & hi) mask |= 4u;
                    if (lo & hi) mask |= 8u;
                } else {
                    for (int c = 0; c < 8; ++c) mask |= 1u << ((word >> (4 * c)) & 15u);
                }
                *dst++ = word;
            }
            if (bad[(size_t)t] == i) continue;
            if (k < L) {                                           // the last, partial word
                uint32_t word = 0;
                for (int c = 0; k + c < L; ++c) {
                    const uint32_t v = s[k + c];
                    if (v >= lim) { if (bad[(size_t)t] < 0) bad[(size_t)t] = i; continue; }
                    mask |= 1u << v;
                    word |= v << (bits * c);
                }
                *dst++ = word;
            }
        }
        masks[(size_t)t] = mask;
    };
    if (n_thr == 1) work(0);
    else {
        std::vector<std::thread> pool;
        for (int t = 0; t < n_thr; ++t) pool.emplace_back(work, t);
        for (auto &th : pool) th.join();
    }
    uint32_t mask = 0;
    for (int t = 0; t < n_thr; ++t) {
        if (bad[(size_t)t] >= 0) {
            const int64_t i = bad[(size_t)t];
            uint32_t v = 0;
            for (int64_t k = off[i]; k < off[i + 1]; ++k) if (codes[k] >= lim) { v = codes[k]; break; }
            return rsd_fail(RSD_EINVAL, "rsd_pack: code %u at sequence %lld does not fit %d bits", v, (long long)i, bits);
        }
        mask |= masks[(size_t)t];
    }
    if (symmask_inout) *symmask_inout |= mask;
    return RSD_OK;
}

// ------------------------------------------------------------------------------------------------
// planning
// ------------------------------------------------------------------------------------------------
template <typename K>
static int persistent_grid(K kernel, int threads, int sm_count, int &blocks) {
    static thread_local const void *cached_k[16]; static thread_local int cached_v[16]; static thread_local int n_cached = 0;
    for (int i = 0; i < n_cached; ++i) if (cached_k[i] == (const void *)kernel) { blocks = cached_v[i] * sm_count; return RSD_OK; }
    int per_sm = 0;
    RSD_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, 0));
    if (per_sm < 1) per_sm = 1;
    if (n_cached < 16) { cached_k[n_cached] = (const void *)kernel; cached_v[n_cached] = per_sm; ++n_cached; }
    blocks = per_sm * sm_count;
    return RSD_OK;
}

int rsd_ctx::make_plan(PlanSlot &sl, const int32_t *d_alen, const int32_t *d_blen, int64_t n_pairs, int C, int allow_twin,
                       double *d_out, cudaStream_t st, PlanView &pv, int64_t max_m, int64_t max_n, int band) {
    RSD_OK_OR_RETURN(sl.pair_bin.ensure(sizeof(int) * (size_t)n_pairs));
    const size_t plan_ints = (size_t)(2 * RSD_PLAN_COPIES) * RSD_NB_MAX + 2 * (RSD_NB_MAX + 1) + 16;
    {
        const void *before = sl.bins.p;
        RSD_OK_OR_RETURN(sl.bins.ensure(sizeof(int) * plan_ints));
        if (sl.bins.p != before) sl.dirty = true;                                // fresh allocation: contents undefined
    }
    // twins need identical m; otherwise a task may mix pairs whose m differ a little (every lane keeps its
    // own row count), so rows are binned ~3 % of max_m at a time and sparse shapes still fill their tapes
    if (allow_twin) max_m = max_n = std::max(max_m, max_n);                      // either sequence may end up as the rows (plan_swap)
    int lg = 0;
    while (((int64_t)2 << lg) <= std::max<int64_t>(max_m, 1)) ++lg;              // floor(log2(max_m))
    pv.m_shift = allow_twin ? 0 : std::min(std::max(lg - 5, 0), 6);
    pv.MQ = (int)std::min<int64_t>((std::max<int64_t>(max_m, 1) >> pv.m_shift) + 2, RSD_MQ_MAX);
    pv.NSC = (int)std::min<int64_t>((std::max<int64_t>(max_n, 1) + C - 1) / C, RSD_NSQ_MAX + 1);
    pv.NB = pv.NSC * pv.MQ;
    RSD_OK_OR_RETURN(sl.groups.ensure(sizeof(int2) * (size_t)n_pairs));
    int *bins = (int *)sl.bins.p;
    pv.pair_bin = (int *)sl.pair_bin.p;
    pv.bin_cnt = bins;
    // fixed array bases (independent of this call's NB) so the zeroed-counter invariant survives a change of NB
    pv.bin_cursor = bins + (size_t)RSD_PLAN_COPIES * RSD_NB_MAX;
    pv.bin_group_off = bins + (size_t)(2 * RSD_PLAN_COPIES) * RSD_NB_MAX;
    pv.bin_warp_off = pv.bin_group_off + (RSD_NB_MAX + 1);
    pv.totals = pv.bin_warp_off + (RSD_NB_MAX + 1);
    pv.work_counter = pv.totals + 4;
    pv.groups = (int2 *)sl.groups.p;
    pv.C = C; pv.allow_twin = allow_twin; pv.band = band;
    pv.dbg = getenv("RSD_TRACE_PLAN") ? (unsigned long long *)(pv.totals + 6) : nullptr;      // synchronises after every plan
    // bin counters are zeroed again by the scan phase, which also resets cursors / ticket / odd-twin
    // slots — so a plan is three kernels and no memsets.  A call that failed between count and
    // fill leaves them dirty: start clean then.
    // The whole array is cleared (all RSD_PLAN_COPIES counter copies, cursors, offsets, totals, ticket): a slot's
    // first use sees whatever cudaMalloc handed out, which is not zero when the block was used before.
    if (sl.dirty) {
        RSD_CUDA(cudaMemsetAsync(bins, 0, sizeof(int) * plan_ints, st));
    }
    sl.dirty = true;
    {
        // one cooperative launch: every SM gets up to two 1024-thread blocks (grid-stride over the pairs)
        int per_sm = 0;
        RSD_OK_OR_RETURN(persistent_grid(k_plan_all, 1024, 1, per_sm));
        const int64_t want = (n_pairs + 1023) / 1024;
        const unsigned G = (unsigned)std::max<int64_t>(1, std::min<int64_t>(want, (int64_t)sm_count * std::min(per_sm, 2)));
        double c_ins = ins, c_del = del;
        void *args[] = {(void *)&d_alen, (void *)&d_blen, (void *)&n_pairs, (void *)&pv, (void *)&c_ins, (void *)&c_del, (void *)&d_out};
        RSD_CUDA(cudaLaunchCooperativeKernel((const void *)k_plan_all, dim3(G), dim3(1024), args, 0, st));
        launches += 1;
        if (pv.dbg) {
            unsigned long long d[3];
            cudaStreamSynchronize(st);
            cudaMemcpy(d, pv.dbg, sizeof d, cudaMemcpyDeviceToHost);
            fprintf(stderr, "[rsd trace] plan %lld pairs, %u blocks: count %.1f us, scan %.1f us, fill %.1f us\n", (long long)n_pairs, G,
                    d[0] * 1e-3, d[1] * 1e-3, d[2] * 1e-3);
        }
    }
    RSD_CUDA(cudaGetLastError());
    sl.dirty = false;
    return RSD_OK;
}

// ------------------------------------------------------------------------------------------------
// distance batch
// ------------------------------------------------------------------------------------------------
// Longest sequence of a batch the int16x2 distance takes the band kernel for by default (DESIGN §4): its hand-off buffer
// takes 128 bytes per row and warp of the longest sequence, in every plan slot of a call
#define RSD_BAND_MAX_LEN 512
// Plans a batch into `sl`: its numeric mode, the kernel layout and the plan arrays.  load_costs = false when the caller
// has already uploaded the cost tables of this classification.
int rsd_ctx::distance_plan(PlanSlot &sl, const int32_t *a_len, const int32_t *b_len, int64_t n_pairs, int64_t max_m, int64_t max_n,
                           int bits, uint32_t symmask, int force_mode, bool load_costs, double *d_out, int *mode_out, cudaStream_t st) {
    if (n_pairs < 0 || n_pairs > INT32_MAX) return rsd_fail(RSD_ERANGE, "rsd: n_pairs out of range");
    if (bits != 2 && bits != 4) return rsd_fail(RSD_EINVAL, "rsd: bits must be 2 or 4");
    if (bits == 2 && (symmask & ~0xFu)) return rsd_fail(RSD_EINVAL, "rsd: 2-bit packing with symbols outside ACGU");
    RSD_OK_OR_RETURN(classify(symmask, max_m, max_n, bits, force_mode, sl.mi));
    if (mode_out) *mode_out = sl.mi.mode;
    sl.n_pairs = n_pairs; sl.max_n = max_n;
    if (n_pairs == 0) return RSD_OK;
    if (load_costs) RSD_OK_OR_RETURN(upload_costs(sl.mi, st));
    const int C = sl.mi.mode == RSD_MODE_F64 ? 16 : 32;
    // Layout of the int16x2 kernel.  The band kernel needs ins > 0 and del > 0 (else the band has no bound) and every
    // pair in a strip class of its own (<= RSD_NSQ_MAX strips).  It takes 64 pairs per warp task, so by default it runs
    // when the batch gives every resident warp at least one task (measured crossover at C2 shapes: 1.5 * 10^5 pairs =
    // 2344 tasks on 2368 warps, DESIGN §4) and no sequence is longer than RSD_BAND_MAX_LEN.  RSD_DIST_BAND=0|1 forces
    // the choice wherever the band kernel applies.
    bool band = false;
    const int64_t longest = std::max(max_m, max_n);
    if (sl.mi.mode == RSD_MODE_I16X2 && sl.mi.ic.ins > 0 && sl.mi.ic.del > 0 && (longest + C - 1) / C <= RSD_NSQ_MAX) {
        int blocks = 0;
        RSD_OK_OR_RETURN(persistent_grid(k_dist_band16<32>, 128, sm_count, blocks));
        band = longest <= RSD_BAND_MAX_LEN && n_pairs >= (int64_t)64 * 4 * blocks;
        if (const char *e = getenv("RSD_DIST_BAND")) band = atoi(e) != 0;
    }
    return make_plan(sl, a_len, b_len, n_pairs, C, sl.mi.mode == RSD_MODE_I16X2 ? 1 : 0, d_out, st, sl.pv, max_m, max_n, band ? 1 : 0);
}

// The distance kernel of the batch planned into `sl`.  Events t0 / t1 (when not null) are recorded around the launch.
int rsd_ctx::distance_launch(PlanSlot &sl, const uint32_t *a_words, const int64_t *a_start, const int32_t *a_len,
                             const uint32_t *b_words, const int64_t *b_start, const int32_t *b_len,
                             int64_t max_m, int bits, double *d_out, cudaStream_t st, cudaEvent_t t0, cudaEvent_t t1) {
    if (sl.n_pairs == 0) return RSD_OK;
    const ModeInfo &mi = sl.mi;
    const PlanView &pv = sl.pv;
    SeqView A{a_words, a_start, a_len}, B{b_words, b_start, b_len};
    constexpr int THREADS = 128;
    const int wpb = THREADS / 32;
    int blocks = 0;
    if (mi.mode == RSD_MODE_I16X2 && pv.band) {
        RSD_OK_OR_RETURN(persistent_grid(k_dist_band16<32>, THREADS, sm_count, blocks));
        const int rows = (int)std::max<int64_t>(max_m, sl.max_n);       // rows after the orientation choice
        RSD_OK_OR_RETURN(sl.scratch.ensure(sizeof(uint32_t) * 32 * (size_t)rows * blocks * wpb + 16));
        unsigned long long *trace = nullptr;
        if (getenv("RSD_TRACE")) {
            RSD_OK_OR_RETURN(sl.trace.ensure(3 * sizeof(unsigned long long)));
            trace = (unsigned long long *)sl.trace.p;
            RSD_CUDA(cudaMemsetAsync(trace, 0, 3 * sizeof(unsigned long long), st));
        }
        if (t0) RSD_CUDA(cudaEventRecord(t0, st));
        k_dist_band16<32><<<blocks, THREADS, 0, st>>>(pv, A, B, mi.ic, d_out, (uint32_t *)sl.scratch.p, rows, 1u, trace);
        if (trace) {                      // synchronises after the launch: not for timing runs
            unsigned long long h[3];
            RSD_CUDA(cudaMemcpyAsync(h, trace, sizeof h, cudaMemcpyDeviceToHost, st));
            RSD_CUDA(cudaStreamSynchronize(st));
            fprintf(stderr, "[rsd trace] k_dist_band16: %lld pairs, cell slots %.4g = %.3f x sum(m*n) %.4g = %.3f x the strip-padded cells %.4g\n",
                    (long long)sl.n_pairs, (double)h[0], (double)h[0] / std::max(1.0, (double)h[1]), (double)h[1],
                    (double)h[0] / std::max(1.0, (double)h[2]), (double)h[2]);
        }
    } else if (mi.mode == RSD_MODE_I16X2) {
        RSD_OK_OR_RETURN(persistent_grid(k_dist_twin16<32>, THREADS, sm_count, blocks));
        const int stride2 = (int)std::max<int64_t>(max_m, sl.max_n);     // rows after the orientation choice
        RSD_OK_OR_RETURN(sl.scratch.ensure(sizeof(uint32_t) * 2 * (size_t)stride2 * blocks * wpb + 16));
        if (t0) RSD_CUDA(cudaEventRecord(t0, st));
        k_dist_twin16<32><<<blocks, THREADS, 0, st>>>(pv, A, B, mi.ic, d_out, (uint32_t *)sl.scratch.p, stride2, 1u);
    } else {
        // general kernels: two boundary columns of max_m rows per warp (tape passes); `elem` has the scratch element type
        auto launch_gen = [&](auto kernel, auto elem) -> int {
            using T = decltype(elem);
            const int stride = (int)max_m;
            RSD_OK_OR_RETURN(persistent_grid(kernel, THREADS, sm_count, blocks));
            RSD_OK_OR_RETURN(sl.scratch.ensure(sizeof(T) * 2 * (size_t)stride * blocks * wpb + 16));
            if (t0) RSD_CUDA(cudaEventRecord(t0, st));
            kernel<<<blocks, THREADS, 0, st>>>(pv, A, B, d_ic, d_fc, d_out, (T *)sl.scratch.p, stride);
            return RSD_OK;
        };
        if (mi.mode == RSD_MODE_I32) RSD_OK_OR_RETURN(launch_gen(bits == 2 ? k_dist_gen<int, 2, 32> : k_dist_gen<int, 4, 32>, 0));
        else RSD_OK_OR_RETURN(launch_gen(bits == 2 ? k_dist_gen<double, 2, 16> : k_dist_gen<double, 4, 16>, 0.0));
    }
    if (t1) RSD_CUDA(cudaEventRecord(t1, st));
    launches += 1;
    RSD_CUDA(cudaGetLastError());
    return RSD_OK;
}

int rsd_ctx::distance_dev(const uint32_t *a_words, const int64_t *a_start, const int32_t *a_len,
                          const uint32_t *b_words, const int64_t *b_start, const int32_t *b_len,
                          int64_t n_pairs, int64_t max_m, int64_t max_n, int bits, uint32_t symmask,
                          int force_mode, double *d_out, int *mode_out, cudaStream_t st, cudaEvent_t t0, cudaEvent_t t1) {
    PlanSlot &sl = slots[0];
    RSD_OK_OR_RETURN(distance_plan(sl, a_len, b_len, n_pairs, max_m, max_n, bits, symmask, force_mode, true, d_out, mode_out, st));
    return distance_launch(sl, a_words, a_start, a_len, b_words, b_start, b_len, max_m, bits, d_out, st, t0, t1);
}

extern "C" int rsd_distance_batch_dev(rsd_ctx *c,
                                      const uint32_t *a_words, const int64_t *a_start, const int32_t *a_len,
                                      const uint32_t *b_words, const int64_t *b_start, const int32_t *b_len,
                                      int64_t n_pairs, int64_t max_m, int64_t max_n, int bits, uint32_t symmask,
                                      int force_mode, double *out, int *mode_out, void *stream) {
    if (!c) return rsd_fail(RSD_EINVAL, "ctx is NULL");
    RSD_OK_OR_RETURN(c->ensure_device());
    // the kernel alone is timed
    c->timed = false; c->last_ms_override = 0.0;
    const bool timed = c->timing && n_pairs > 0;
    RSD_OK_OR_RETURN(c->distance_dev(a_words, a_start, a_len, b_words, b_start, b_len, n_pairs, max_m, max_n, bits, symmask,
                                     force_mode, out, mode_out, (cudaStream_t)stream, timed ? c->ev0 : nullptr, timed ? c->ev1 : nullptr));
    c->timed = timed;
    return RSD_OK;
}

static int64_t max_len(const int32_t *len, int64_t n) {
    int32_t m = 0;
    for (int64_t i = 0; i < n; ++i) m = std::max(m, len[i]);
    return m;
}

// true when the sequences [p0, p1) are stored in pair order without overlap: start[p] >= 0, start[p] + nwords(len[p]) <=
// start[p+1] (the last sequence of the batch ends inside the buffer).  Then the pairs [p0, p1) own exactly the words
// [start[p0], start[p1]).
static bool pair_ordered(const int64_t *start, const int32_t *len, int64_t p0, int64_t p1, int64_t n, int64_t n_words, int bits) {
    if (p1 <= p0) return true;
    const int sh = bits == 2 ? 4 : 3, add = (1 << sh) - 1;
    int64_t bad = start[p0] < 0;
    const int64_t e = std::min(p1, n - 1);
    for (int64_t p = p0; p < e; ++p)
        bad |= (int64_t)(start[p] + (((int64_t)len[p] + add) >> sh) > start[p + 1]) | (int64_t)(len[p] < 0);
    if (p1 == n) bad |= (int64_t)(len[n - 1] < 0) | (int64_t)(start[n - 1] + (((int64_t)len[n - 1] + add) >> sh) > n_words);
    return bad == 0;
}

int rsd_ctx::upload_seqs(SeqBufs &sb, const uint32_t *words, const int64_t *start, const int32_t *len, int64_t n,
                         int64_t n_words, cudaStream_t st) {
    RSD_OK_OR_RETURN(sb.words.ensure(sizeof(uint32_t) * (size_t)(n_words + 8)));
    RSD_OK_OR_RETURN(sb.start.ensure(sizeof(int64_t) * (size_t)std::max<int64_t>(n, 1)));
    RSD_OK_OR_RETURN(sb.len.ensure(sizeof(int32_t) * (size_t)std::max<int64_t>(n, 1)));
    RSD_CUDA(cudaMemcpyAsync(sb.words.p, words, sizeof(uint32_t) * (size_t)n_words, cudaMemcpyHostToDevice, st));
    RSD_CUDA(cudaMemsetAsync((uint32_t *)sb.words.p + n_words, 0, sizeof(uint32_t) * 8, st));
    RSD_CUDA(cudaMemcpyAsync(sb.start.p, start, sizeof(int64_t) * (size_t)n, cudaMemcpyHostToDevice, st));
    RSD_CUDA(cudaMemcpyAsync(sb.len.p, len, sizeof(int32_t) * (size_t)n, cudaMemcpyHostToDevice, st));
    return RSD_OK;
}

// One side of a host batch call.  Three input forms:
//   packed, explicit start[]   words + start + len          (any layout; validated before chunked copies)
//   packed, canonical          words + len, start == NULL   (rsd_pack layout: start[] is rebuilt on the device)
//   raw codes                  codes + len                  (1 byte per symbol, concatenated; packed on the device)
struct SideIn {
    const uint32_t *words; const int64_t *start; const int32_t *len; int64_t nwords; const uint8_t *codes;
    bool canonical() const { return codes != nullptr || start == nullptr; }
};

// per-block sums of nwords(len) (and of len, for raw codes) for the blocks [b0, b1): sum[b] = words of block b
// neg (optional) receives a negative value when one of the lengths is negative (the OR of all of them)
static void block_sums(const int32_t *len, int64_t n, int sh, int64_t b0, int64_t b1, int64_t *sum, int64_t *sym_sum, std::atomic<int32_t> *neg = nullptr) {
    const int add = (1 << sh) - 1;
    int32_t any = 0;
    for (int64_t b = b0; b < b1; ++b) {
        const int64_t e = std::min<int64_t>(n, (b + 1) * RSD_SCAN_BLOCK);
        int64_t s = 0, ss = 0;
        for (int64_t p = b * RSD_SCAN_BLOCK; p < e; ++p) { s += (len[p] + add) >> sh; ss += len[p]; any |= len[p]; }
        sum[b] = s; if (sym_sum) sym_sum[b] = ss;
    }
    if (neg && any < 0) neg->store(any);
}
// in place: per-block sums -> exclusive prefix, entry nblk = total
static void block_prefix(int64_t *tab, int64_t nblk) {
    int64_t acc = 0;
    for (int64_t b = 0; b < nblk; ++b) { const int64_t v = tab[b]; tab[b] = acc; acc += v; }
    tab[nblk] = acc;
}

static int distance_host(rsd_ctx *c, const SideIn in[2], int64_t n_pairs, int64_t max_m_hint, int64_t max_n_hint, int bits,
                         uint32_t symmask, int force_mode, double *out, int *mode_out) {
    const bool trace = getenv("RSD_TRACE") != nullptr;
    auto now = [] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    const double t_in = now();
    double t_len = 0, t_cost = 0, t_first = 0, t_comp = 0;
    cudaStream_t st = c->stream, cp = c->copy_stream;
    const int64_t max_m = max_m_hint > 0 ? max_m_hint : max_len(in[0].len, n_pairs);
    const int64_t max_n = max_n_hint > 0 ? max_n_hint : max_len(in[1].len, n_pairs);
    const int sh = bits == 2 ? 4 : 3;
    const bool any_canon = in[0].canonical() || in[1].canonical();
    const bool any_codes = in[0].codes || in[1].codes;
    // costs go up first: a small pageable copy issued later would queue behind the big H2D copies on
    // the copy engine and stall the first kernel until every chunk has arrived.
    {
        ModeInfo mi0;
        RSD_OK_OR_RETURN(c->classify(symmask, max_m, max_n, bits, force_mode, mi0));
        RSD_OK_OR_RETURN(c->upload_costs(mi0, st));
    }
    t_cost = now();
    SeqBufs *dS[2] = {&c->bufA, &c->bufB};
    for (int s = 0; s < 2; ++s) {
        RSD_OK_OR_RETURN(dS[s]->start.ensure(sizeof(int64_t) * (size_t)n_pairs));
        RSD_OK_OR_RETURN(dS[s]->len.ensure(sizeof(int32_t) * (size_t)n_pairs));
        if (!in[s].codes) RSD_OK_OR_RETURN(dS[s]->words.ensure(sizeof(uint32_t) * (size_t)(in[s].nwords + 8)));
    }
    RSD_OK_OR_RETURN(c->out_f64.ensure(sizeof(double) * (size_t)n_pairs));
    // the previous call's kernels may still read these buffers: order the copy stream after them
    RSD_CUDA(cudaEventRecord(c->ev_sync, st));
    RSD_CUDA(cudaStreamWaitEvent(cp, c->ev_sync, 0));
    RSD_CUDA(cudaEventRecord(c->ev_begin, cp));
    // Lengths of the whole batch go first (8 bytes per pair): every chunk is planned from them right away, so
    // afterwards the compute streams hold nothing but the chunk kernels.
    for (int s = 0; s < 2; ++s)
        RSD_CUDA(cudaMemcpyAsync(dS[s]->len.p, in[s].len, sizeof(int32_t) * (size_t)n_pairs, cudaMemcpyHostToDevice, cp));
    RSD_CUDA(cudaEventRecord(c->ev_len, cp));
    const int64_t nblk = (n_pairs + RSD_SCAN_BLOCK - 1) / RSD_SCAN_BLOCK;
    int64_t *tab[2][2] = {{nullptr, nullptr}, {nullptr, nullptr}};      // [side][0 words, 1 symbols], nblk + 1 entries each
    int64_t nwords[2] = {in[0].nwords, in[1].nwords};
    const size_t tab_bytes = sizeof(int64_t) * 4 * (size_t)(nblk + 1);
    std::atomic<int32_t> neg_len{0};                    // (declared before the helper threads that write it)
    std::thread helpers[2];
    struct Joiner { std::thread *t; ~Joiner() { for (int s = 0; s < 2; ++s) if (t[s].joinable()) t[s].join(); } } joiner{helpers};
    if (any_canon) {
        if (tab_bytes + 64 > c->h_stage_cap) {
            if (c->h_stage) cudaFreeHost(c->h_stage);
            c->h_stage = nullptr; c->h_stage_cap = 0;
            RSD_CUDA(cudaMallocHost(&c->h_stage, tab_bytes + 4096));
            c->h_stage_cap = tab_bytes + 4096;
        }
        RSD_OK_OR_RETURN(c->d_stage.ensure(tab_bytes + 64));
        for (int s = 0; s < 2; ++s) for (int q = 0; q < 2; ++q) tab[s][q] = (int64_t *)c->h_stage + (size_t)(2 * s + q) * (nblk + 1);
    }
    // Large batches are cut into chunks of pairs so the H2D copy of chunk k+1 (copy stream) overlaps
    // the kernels of chunk k (compute stream); sequences are word-aligned and stored in pair order, so
    // a chunk is a contiguous slice of every array.  Pinned host buffers make the copies asynchronous.
    // Packed input: chunk sizes grow geometrically so the first copy is short; the growth stays below the
    // compute/copy time ratio so that no later chunk waits for its data.  Raw codes are four times the bytes and
    // copy-bound: 16 chunks that shrink by 0.85, so that little work is left when the last byte has arrived.
    int n_chunks = 1;
    int64_t bounds[RSD_MAX_CHUNKS + 1];
    bounds[0] = 0;
    if (n_pairs >= (1 << 16)) {
        n_chunks = any_codes ? 16 : 5;
        double ratio = any_codes ? 0.85 : 1.5;                 // codes: shrinking chunks, so little compute is left behind the last byte
        if (const char *e = getenv("RSD_CHUNKS")) n_chunks = std::min(std::max(atoi(e), 1), RSD_MAX_CHUNKS);
        if (const char *e = getenv("RSD_CHUNK_RATIO")) ratio = std::min(std::max(atof(e), 0.5), 4.0);
        double wsum = 0, w = 1.0, acc = 0;
        for (int k = 0; k < n_chunks; ++k) { wsum += w; w *= ratio; }
        w = 1.0;
        for (int k = 0; k < n_chunks; ++k) {
            acc += w; w *= ratio;
            int64_t b = (int64_t)((double)n_pairs * acc / wsum);
            if (any_canon) b = b / RSD_SCAN_BLOCK * RSD_SCAN_BLOCK;           // word offsets are known at block boundaries
            bounds[k + 1] = std::max(b, bounds[k]);
        }
    }
    bounds[n_chunks] = n_pairs;
    t_len = now();
    // the chunk kernels are timed (ev_t0 / ev_t1 of each chunk) and their times summed
    const bool timing = c->timing;
    float kernel_ms = 0.f;
    c->timed = false; c->last_ms_override = 0.0;
    RSD_CUDA(cudaStreamWaitEvent(st, c->ev_len, 0));
    auto enqueue_plans = [&]() -> int {
        for (int k = 0; k < n_chunks; ++k) {
            const int64_t p0 = bounds[k], p1 = bounds[k + 1];
            if (p1 <= p0) continue;
            RSD_OK_OR_RETURN(c->distance_plan(c->slots[k], (const int32_t *)dS[0]->len.p + p0, (const int32_t *)dS[1]->len.p + p0, p1 - p0, max_m, max_n,
                                              bits, symmask, force_mode, false, (double *)c->out_f64.p + p0, mode_out, st));
        }
        RSD_CUDA(cudaEventRecord(c->ev_plans, st));
        RSD_CUDA(cudaStreamWaitEvent(c->stream2, c->ev_plans, 0));
        return RSD_OK;
    };
    unsigned long long *d_bad = (unsigned long long *)((unsigned char *)c->d_stage.p + tab_bytes);       // {bad sequence + 1, symbols seen}
    // the distance kernel of chunk k and the copy of its results; chunk kernels alternate between two streams: the next
    // chunk's blocks move in while the last tasks of the previous chunk drain, so a chunk boundary costs no idle SMs
    auto launch_chunk = [&](int k, cudaStream_t sk) -> int {
        const int64_t p0 = bounds[k], p1 = bounds[k + 1];
        RSD_OK_OR_RETURN(c->distance_launch(c->slots[k], (const uint32_t *)dS[0]->words.p, (const int64_t *)dS[0]->start.p + p0, (const int32_t *)dS[0]->len.p + p0,
                                            (const uint32_t *)dS[1]->words.p, (const int64_t *)dS[1]->start.p + p0, (const int32_t *)dS[1]->len.p + p0,
                                            max_m, bits, (double *)c->out_f64.p + p0, sk, timing ? c->ev_t0[k] : nullptr, timing ? c->ev_t1[k] : nullptr));
        // results go back on their own stream, behind nothing but the chunk's kernel
        RSD_CUDA(cudaEventRecord(c->ev_done[k], sk));
        RSD_CUDA(cudaStreamWaitEvent(c->d2h_stream, c->ev_done[k], 0));
        RSD_CUDA(cudaMemcpyAsync(out + p0, (double *)c->out_f64.p + p0, sizeof(double) * (size_t)(p1 - p0), cudaMemcpyDeviceToHost, c->d2h_stream));
        return RSD_OK;
    };
    volatile unsigned long long *h_bad = nullptr;

    if (!any_codes) {
        // ---- packed words: everything a chunk needs is prepared, copied and launched chunk by chunk -----------------
        // Host-side preparation of a chunk, per side.  Canonical layout (start == NULL): the word count of every block
        // of RSD_SCAN_BLOCK sequences — their running sum gives the chunk's word range and seeds the device scan that
        // rebuilds start[] (so start[], 8 bytes per sequence, never crosses PCIe).  Caller-supplied start[]: a chunk's
        // copy is the word range [start[p0], start[p1]), which is only right when every sequence ends at or before the
        // start of the next one — one branch-free pass over start[] and len[]; from the first chunk that fails it the
        // whole word buffer is sent instead.  Both passes are memory-bound reads of the caller's arrays (0.3-1 ms per
        // 10^6 pairs and side): done per chunk on this thread they hide behind the kernels of the chunks before, and
        // only the first chunk's share (7 % of the batch) sits in front of the first copy.
        int64_t wacc[2] = {0, 0};
        bool whole[2] = {false, false};                  // side sent as one buffer (not in pair order, or a single chunk)
        bool plans_done = false;
        for (int k = 0; k < n_chunks; ++k) {
            const int64_t p0 = bounds[k], p1 = bounds[k + 1];
            if (p1 <= p0) continue;
            const int64_t b0 = p0 / RSD_SCAN_BLOCK, b1 = p1 >= n_pairs ? nblk : p1 / RSD_SCAN_BLOCK;
            for (int s = 0; s < 2; ++s) {
                if (in[s].canonical()) {
                    block_sums(in[s].len, n_pairs, sh, b0, b1, tab[s][0], nullptr, &neg_len);
                    if (neg_len.load() < 0) return rsd_fail(RSD_EINVAL, "rsd_distance_batch: negative length");
                    const int64_t w0 = wacc[s];
                    for (int64_t b = b0; b < b1; ++b) { const int64_t v = tab[s][0][b]; tab[s][0][b] = wacc[s]; wacc[s] += v; }
                    if (wacc[s] > in[s].nwords)
                        return rsd_fail(RSD_EINVAL, "rsd_distance_batch: side %d holds %lld words but its lengths need at least %lld (canonical layout)", s,
                                        (long long)in[s].nwords, (long long)wacc[s]);
                    int64_t *dtab = (int64_t *)c->d_stage.p + (size_t)(2 * s) * (nblk + 1);
                    RSD_CUDA(cudaMemcpyAsync(dtab + b0, tab[s][0] + b0, sizeof(int64_t) * (size_t)(b1 - b0), cudaMemcpyHostToDevice, cp));
                    if (wacc[s] > w0) RSD_CUDA(cudaMemcpyAsync((uint32_t *)dS[s]->words.p + w0, in[s].words + w0, sizeof(uint32_t) * (size_t)(wacc[s] - w0), cudaMemcpyHostToDevice, cp));
                    if (p1 >= n_pairs) { nwords[s] = wacc[s]; RSD_CUDA(cudaMemsetAsync((uint32_t *)dS[s]->words.p + nwords[s], 0, sizeof(uint32_t) * 8, cp)); }
                } else {
                    if (!whole[s] && (n_chunks == 1 || !pair_ordered(in[s].start, in[s].len, p0, p1, n_pairs, in[s].nwords, bits))) {
                        whole[s] = true;
                        if (nwords[s] > 0) RSD_CUDA(cudaMemcpyAsync(dS[s]->words.p, in[s].words, sizeof(uint32_t) * (size_t)nwords[s], cudaMemcpyHostToDevice, cp));
                    }
                    if (!whole[s]) {
                        const int64_t w0 = in[s].start[p0], w1 = p1 >= n_pairs ? nwords[s] : in[s].start[p1];
                        if (w1 > w0) RSD_CUDA(cudaMemcpyAsync((uint32_t *)dS[s]->words.p + w0, in[s].words + w0, sizeof(uint32_t) * (size_t)(w1 - w0), cudaMemcpyHostToDevice, cp));
                    }
                    RSD_CUDA(cudaMemcpyAsync((int64_t *)dS[s]->start.p + p0, in[s].start + p0, sizeof(int64_t) * (size_t)(p1 - p0), cudaMemcpyHostToDevice, cp));
                    if (p1 >= n_pairs) RSD_CUDA(cudaMemsetAsync((uint32_t *)dS[s]->words.p + nwords[s], 0, sizeof(uint32_t) * 8, cp));
                }
            }
            RSD_CUDA(cudaEventRecord(c->ev_chunk[k], cp));
            if (!plans_done) { t_first = now(); RSD_OK_OR_RETURN(enqueue_plans()); plans_done = true; }
            cudaStream_t sk = (k & 1) ? c->stream2 : st;
            RSD_CUDA(cudaStreamWaitEvent(sk, c->ev_chunk[k], 0));
            for (int s = 0; s < 2; ++s) if (in[s].canonical()) {
                const int64_t *dtab = (const int64_t *)c->d_stage.p + (size_t)(2 * s) * (nblk + 1);
                k_starts_from_len<<<(unsigned)(b1 - b0), 1024, 0, sk>>>((const int32_t *)dS[s]->len.p + p0, p1 - p0, sh, dtab + b0, (int64_t *)dS[s]->start.p + p0, nullptr, nullptr);
                c->launches += 1;
            }
            RSD_OK_OR_RETURN(launch_chunk(k, sk));
        }
    } else {
        // ---- raw codes: copy-bound (1 byte per symbol: 4x the packed bytes), so the copies go out first ------------------
        // The first chunk's block sums are done here and its codes leave at once; the other blocks are summed on helper
        // threads meanwhile.  Device buffers are sized by the length bound (n_pairs x longest sequence) so that nothing
        // has to wait for the totals.
        const int64_t b_first = n_chunks > 1 ? bounds[1] / RSD_SCAN_BLOCK : nblk;
        const int per_w = 32 / bits;
        // (a batch of very uneven lengths would make that bound huge: then the buffers wait for the totals)
        const bool early = n_chunks > 1 && (double)n_pairs * (double)std::max(max_m, max_n) <= 2147483648.0;
        for (int s = 0; s < 2; ++s) if (in[s].codes && early) {
            const int64_t mx = s == 0 ? max_m : max_n;
            RSD_OK_OR_RETURN(c->raw_codes[s].ensure((size_t)n_pairs * (size_t)mx + 64));
            RSD_OK_OR_RETURN(dS[s]->words.ensure(sizeof(uint32_t) * ((size_t)n_pairs * (size_t)((mx + per_w - 1) / per_w) + 8)));
        }
        for (int s = 0; s < 2; ++s) if (in[s].canonical()) {
            auto job = [&in, &tab, &neg_len, n_pairs, sh, nblk, b_first, s] { block_sums(in[s].len, n_pairs, sh, b_first, nblk, tab[s][0], in[s].codes ? tab[s][1] : nullptr, &neg_len); };
            if (b_first < nblk) { if (n_pairs >= (1 << 17)) helpers[s] = std::thread(job); else job(); }
        }
        int64_t sent0[2] = {0, 0};                       // symbols of chunk 0 already on their way
        for (int s = 0; s < 2; ++s) if (in[s].canonical()) {
            block_sums(in[s].len, n_pairs, sh, 0, b_first, tab[s][0], in[s].codes ? tab[s][1] : nullptr, &neg_len);
            if (neg_len.load() < 0) return rsd_fail(RSD_EINVAL, "rsd_distance_batch: negative length");
            if (in[s].codes && early) {
                for (int64_t b = 0; b < b_first; ++b) sent0[s] += tab[s][1][b];
                if (sent0[s] > (int64_t)n_pairs * (s == 0 ? max_m : max_n)) return rsd_fail(RSD_EINVAL, "rsd_distance_batch_codes: a length exceeds the max length hint");
                if (sent0[s] > 0) RSD_CUDA(cudaMemcpyAsync(c->raw_codes[s].p, in[s].codes, (size_t)sent0[s], cudaMemcpyHostToDevice, cp));
            }
        }
        for (int s = 0; s < 2; ++s) if (helpers[s].joinable()) helpers[s].join();
        if (neg_len.load() < 0) return rsd_fail(RSD_EINVAL, "rsd_distance_batch: negative length");
        bool whole[2] = {false, false};
        for (int s = 0; s < 2; ++s) {
            if (in[s].canonical()) {
                block_prefix(tab[s][0], nblk);
                if (in[s].codes) block_prefix(tab[s][1], nblk);
                if (!in[s].codes && tab[s][0][nblk] > in[s].nwords)
                    return rsd_fail(RSD_EINVAL, "rsd_distance_batch: side %d holds %lld words but its lengths need %lld (canonical layout)", s,
                                    (long long)in[s].nwords, (long long)tab[s][0][nblk]);
                if (in[s].codes && tab[s][1][nblk] > (int64_t)n_pairs * (s == 0 ? max_m : max_n))
                    return rsd_fail(RSD_EINVAL, "rsd_distance_batch_codes: a length exceeds the max length hint");
                nwords[s] = tab[s][0][nblk];
                if (in[s].codes) {
                    if (!early) {
                        RSD_OK_OR_RETURN(c->raw_codes[s].ensure((size_t)tab[s][1][nblk] + 64));
                        RSD_OK_OR_RETURN(dS[s]->words.ensure(sizeof(uint32_t) * (size_t)(nwords[s] + 8)));
                    }
                    RSD_OK_OR_RETURN(c->sym_start[s].ensure(sizeof(int64_t) * (size_t)n_pairs));
                }
            } else if (n_chunks == 1 || !pair_ordered(in[s].start, in[s].len, 0, n_pairs, n_pairs, in[s].nwords, bits)) whole[s] = true;
        }
        RSD_CUDA(cudaMemcpyAsync(c->d_stage.p, c->h_stage, tab_bytes, cudaMemcpyHostToDevice, cp));
        RSD_CUDA(cudaEventRecord(c->ev_tab, cp));
        for (int s = 0; s < 2; ++s) {
            RSD_CUDA(cudaMemsetAsync((uint32_t *)dS[s]->words.p + nwords[s], 0, sizeof(uint32_t) * 8, cp));
            if (whole[s] && nwords[s] > 0) RSD_CUDA(cudaMemcpyAsync(dS[s]->words.p, in[s].words, sizeof(uint32_t) * (size_t)nwords[s], cudaMemcpyHostToDevice, cp));
        }
        RSD_CUDA(cudaMemsetAsync(d_bad, 0, 16, st));
        auto word_at = [&](int s, int64_t p) -> int64_t {
            if (p >= n_pairs) return nwords[s];
            return in[s].canonical() ? tab[s][0][p / RSD_SCAN_BLOCK] : in[s].start[p];
        };
        for (int k = 0; k < n_chunks; ++k) {
            const int64_t p0 = bounds[k], p1 = bounds[k + 1];
            if (p1 <= p0) continue;
            for (int s = 0; s < 2; ++s) {
                if (in[s].codes) {
                    int64_t s0 = tab[s][1][p0 / RSD_SCAN_BLOCK];
                    const int64_t s1 = p1 >= n_pairs ? tab[s][1][nblk] : tab[s][1][p1 / RSD_SCAN_BLOCK];
                    s0 = std::max(s0, sent0[s]);                   // chunk 0 left before the block sums were complete
                    if (s1 > s0) RSD_CUDA(cudaMemcpyAsync((uint8_t *)c->raw_codes[s].p + s0, in[s].codes + s0, (size_t)(s1 - s0), cudaMemcpyHostToDevice, cp));
                    continue;
                }
                const int64_t w0 = word_at(s, p0), w1 = word_at(s, p1);
                if (!whole[s] && w1 > w0) RSD_CUDA(cudaMemcpyAsync((uint32_t *)dS[s]->words.p + w0, in[s].words + w0, sizeof(uint32_t) * (size_t)(w1 - w0), cudaMemcpyHostToDevice, cp));
                if (!in[s].canonical())
                    RSD_CUDA(cudaMemcpyAsync((int64_t *)dS[s]->start.p + p0, in[s].start + p0, sizeof(int64_t) * (size_t)(p1 - p0), cudaMemcpyHostToDevice, cp));
            }
            RSD_CUDA(cudaEventRecord(c->ev_chunk[k], cp));
        }
        t_first = now();
        RSD_CUDA(cudaStreamWaitEvent(st, c->ev_tab, 0));
        for (int s = 0; s < 2; ++s) if (in[s].canonical()) {
            const int64_t *dtab = (const int64_t *)c->d_stage.p + (size_t)(2 * s) * (nblk + 1);
            k_starts_from_len<<<(unsigned)nblk, 1024, 0, st>>>((const int32_t *)dS[s]->len.p, n_pairs, sh, dtab, (int64_t *)dS[s]->start.p,
                                                              in[s].codes ? dtab + (nblk + 1) : nullptr, in[s].codes ? (int64_t *)c->sym_start[s].p : nullptr);
            c->launches += 1;
        }
        RSD_OK_OR_RETURN(enqueue_plans());
        for (int k = 0; k < n_chunks; ++k) {
            const int64_t p0 = bounds[k], p1 = bounds[k + 1];
            if (p1 <= p0) continue;
            cudaStream_t sk = (k & 1) ? c->stream2 : st;
            RSD_CUDA(cudaStreamWaitEvent(sk, c->ev_chunk[k], 0));
            for (int s = 0; s < 2; ++s) if (in[s].codes) {                  // raw codes of the chunk -> packed words, on the device
                const int64_t w0 = word_at(s, p0), w1 = word_at(s, p1);
                if (w1 <= w0) continue;
                const unsigned grid = (unsigned)((w1 - w0 + 255) / 256);
                if (bits == 2) k_pack_codes<2><<<grid, 256, 0, sk>>>((const uint8_t *)c->raw_codes[s].p, (const int64_t *)c->sym_start[s].p, (const int64_t *)dS[s]->start.p,
                                                                   (const int32_t *)dS[s]->len.p, n_pairs, w0, w1, 0, (uint32_t *)dS[s]->words.p, d_bad, nullptr);
                else k_pack_codes<4><<<grid, 256, 0, sk>>>((const uint8_t *)c->raw_codes[s].p, (const int64_t *)c->sym_start[s].p, (const int64_t *)dS[s]->start.p,
                                                          (const int32_t *)dS[s]->len.p, n_pairs, w0, w1, 0, (uint32_t *)dS[s]->words.p, d_bad, nullptr);
                c->launches += 1;
            }
            RSD_OK_OR_RETURN(launch_chunk(k, sk));
        }
        // the d2h stream already waits for every chunk's kernels (ev_done[k]), pack kernels included
        h_bad = (volatile unsigned long long *)((unsigned char *)c->h_stage + tab_bytes);
        RSD_CUDA(cudaMemcpyAsync((void *)h_bad, d_bad, 16, cudaMemcpyDeviceToHost, c->d2h_stream));
    }
    t_comp = now();
    RSD_CUDA(cudaStreamSynchronize(c->d2h_stream));
    RSD_CUDA(cudaStreamSynchronize(cp));
    RSD_CUDA(cudaStreamSynchronize(c->stream2));
    RSD_CUDA(cudaStreamSynchronize(st));
    if (h_bad && h_bad[0])
        return rsd_fail(RSD_EINVAL, "rsd_distance_batch_codes: a symbol code of sequence %llu does not fit %d bits", (unsigned long long)h_bad[0] - 1ull, bits);
    if (trace) fprintf(stderr, "[rsd trace] host ms: classify+costs %.3f, lengths enqueued %.3f, first chunk prepared and sent %.3f, all chunks enqueued %.3f, wait %.3f\n",
                       t_cost - t_in, t_len - t_cost, t_first - t_len, t_comp - t_first, now() - t_comp);
    if (timing) {
        for (int k = 0; k < n_chunks; ++k) {
            if (bounds[k + 1] <= bounds[k]) continue;
            float ms = 0.f;
            RSD_CUDA(cudaEventElapsedTime(&ms, c->ev_t0[k], c->ev_t1[k]));
            kernel_ms += ms;
        }
        c->last_ms_override = kernel_ms;
        if (trace) {
            for (int k = 0; k < n_chunks; ++k) {
                if (bounds[k + 1] <= bounds[k]) continue;
                float a = 0, b = 0, d = 0;
                cudaEventElapsedTime(&a, c->ev_begin, c->ev_chunk[k]);
                cudaEventElapsedTime(&b, c->ev_begin, c->ev_t0[k]);
                cudaEventElapsedTime(&d, c->ev_begin, c->ev_t1[k]);
                fprintf(stderr, "[rsd trace] chunk %d pairs %lld: copy done %.3f ms, kernel %.3f -> %.3f ms\n", k,
                        (long long)(bounds[k + 1] - bounds[k]), a, b, d);
            }
        }
    }
    return RSD_OK;
}

// packed words -> one byte per symbol (word by word: no division per symbol)
static void unpack_symbols(const uint32_t *words, int64_t word0, int32_t len, int bits, uint8_t *out) {
    const int per = 32 / bits; const uint32_t msk = (1u << bits) - 1u;
    int32_t j = 0;
    for (int64_t w = word0; j + per <= len; ++w, j += per) {
        uint32_t x = words[w];
        for (int q = 0; q < per; ++q) { out[j + q] = (uint8_t)(x & msk); x >>= bits; }
    }
    if (j < len) { uint32_t x = words[word0 + j / per]; for (; j < len; ++j) { out[j] = (uint8_t)(x & msk); x >>= bits; } }
}

// Per-pair edit scripts of a batch that route_long sends to the panel kernels: rows of max_ops entries (rsd_script_batch).
struct LongScripts { int64_t max_ops; uint8_t *op; int32_t *oi, *oj, *n_ops; };

// Batches whose cells lie mostly in pairs of at least T symbols go to the panel-wavefront kernels (rsd_long_pairs).  One
// warp per pair with tape passes, the design of k_dist_* / k_script_fwd for 1-2 kb pairs, runs distances at 1.0 / 0.5 /
// 0.25 TCUPS and scripts at 450 / 240 / 35 GCUPS at 5 / 10 / 20 kb, where the panel pipeline runs at 2.7 and 1.0-1.4
// TCUPS (tools/dbg_mid_pairs.py).  With `scripts` the scripts come back too; T <= 0 never routes; `who` prefixes the
// messages.  -> 1 routed (out filled), 0 not applicable, < 0 error.
static int route_long(rsd_ctx *c, const char *who, int64_t T, const SideIn in[2], int64_t n_pairs, int bits, int force_mode,
                      const LongScripts *scripts, double *out, int *mode_out) {
    if (T <= 0 || n_pairs > 65536 || force_mode == RSD_MODE_I16X2) return 0;      // (a forced int16x2 mode keeps its own applicability error)
    double cells_all = 0, cells_long = 0; int64_t total[2] = {0, 0};
    for (int64_t p = 0; p < n_pairs; ++p) {
        const int32_t m = in[0].len[p], n = in[1].len[p];
        if (m < 0 || n < 0) return -rsd_fail(RSD_EINVAL, "%s: negative length", who);
        const double cells = (double)m * (double)n;
        cells_all += cells; total[0] += m; total[1] += n;
        if (std::max(m, n) >= T) cells_long += cells;
    }
    if (!(cells_long > 0.5 * cells_all)) return 0;
    const int per = 32 / bits;
    std::vector<uint8_t> codes[2];
    std::vector<const uint8_t *> ptr[2]; std::vector<int64_t> len64[2];
    int64_t at[2] = {0, 0}, wat[2] = {0, 0};          // symbol / word offset of the canonical layouts
    for (int s = 0; s < 2; ++s) {
        ptr[s].resize((size_t)n_pairs); len64[s].resize((size_t)n_pairs);
        if (!in[s].codes) codes[s].resize((size_t)total[s] + 16);
    }
    for (int64_t p = 0; p < n_pairs; ++p) {
        for (int s = 0; s < 2; ++s) {
            const int32_t len = in[s].len[p];
            len64[s][(size_t)p] = len;
            if (in[s].codes) { ptr[s][(size_t)p] = in[s].codes + at[s]; at[s] += len; continue; }
            const int64_t st0 = in[s].start ? in[s].start[p] : wat[s];
            const int64_t nw = ((int64_t)len + per - 1) / per;
            if (st0 < 0 || st0 + nw > in[s].nwords) return -rsd_fail(RSD_EINVAL, "%s: pair %lld lies outside the word buffer", who, (long long)p);
            ptr[s][(size_t)p] = codes[s].data() + at[s];
            unpack_symbols(in[s].words, st0, len, bits, codes[s].data() + at[s]); at[s] += len;
            wat[s] += nw;
        }
        if (scripts && (int64_t)in[0].len[p] + in[1].len[p] > scripts->max_ops)
            return -rsd_fail(RSD_EINVAL, "%s: max_ops too small for pair %lld", who, (long long)p);
    }
    const size_t n_rows = scripts ? (size_t)n_pairs : 0;
    std::vector<int64_t> mo(n_rows, scripts ? scripts->max_ops : 0), no64(n_rows, 0);
    std::vector<uint8_t *> pop(n_rows); std::vector<int32_t *> poi(n_rows), poj(n_rows);
    for (size_t p = 0; p < n_rows; ++p) {
        const size_t row = p * (size_t)scripts->max_ops;
        pop[p] = scripts->op + row;
        poi[p] = scripts->oi ? scripts->oi + row : nullptr; poj[p] = scripts->oj ? scripts->oj + row : nullptr;
    }
    std::vector<int> modes((size_t)n_pairs, 0);
    const int rc = rsd_long_pairs(c, (int)n_pairs, ptr[0].data(), len64[0].data(), ptr[1].data(), len64[1].data(), force_mode, scripts != nullptr,
                                  mo.data(), pop.data(), poi.data(), poj.data(), no64.data(), out, modes.data());
    if (rc) return -rc;
    for (size_t p = 0; p < n_rows; ++p) scripts->n_ops[p] = (int32_t)no64[p];
    if (mode_out) { int mm = 0; for (int x : modes) mm = std::max(mm, x); *mode_out = mm; }
    return 1;
}

// Length threshold of route_long for an entry point: 0 (never route) when the knob `off` is set, else the knob `min` or
// the default.  By wall time the tape-pass distance kernels still win at 4-5 kb (tools/dbg_crossover.py).
constexpr int64_t DIST_LONG_MIN = 6144, SCRIPT_LONG_MIN = 4096;
static int64_t long_min(const char *off, const char *min, int64_t dflt) {
    if (getenv(off)) return 0;
    const char *e = getenv(min);
    return e ? std::max<int64_t>(atoll(e), 1) : dflt;
}

extern "C" int rsd_distance_batch(rsd_ctx *c,
                                  const uint32_t *a_words, const int64_t *a_start, const int32_t *a_len, int64_t a_nwords,
                                  const uint32_t *b_words, const int64_t *b_start, const int32_t *b_len, int64_t b_nwords,
                                  int64_t n_pairs, int64_t max_m_hint, int64_t max_n_hint, int bits, uint32_t symmask, int force_mode,
                                  double *out, int *mode_out) {
    if (!c) return rsd_fail(RSD_EINVAL, "ctx is NULL");
    if (n_pairs < 0) return rsd_fail(RSD_EINVAL, "rsd_distance_batch: n_pairs < 0");
    if (n_pairs > 0 && (!a_words || !a_len || !b_words || !b_len || !out))
        return rsd_fail(RSD_EINVAL, "rsd_distance_batch: NULL buffer");
    if (bits != 2 && bits != 4) return rsd_fail(RSD_EINVAL, "rsd: bits must be 2 or 4");
    RSD_OK_OR_RETURN(c->ensure_device());
    if (n_pairs == 0) return RSD_OK;
    const SideIn in[2] = {{a_words, a_start, a_len, a_nwords, nullptr}, {b_words, b_start, b_len, b_nwords, nullptr}};
    const int64_t T = long_min("RSD_DIST_NO_LONG", "RSD_DIST_LONG_MIN", DIST_LONG_MIN);
    if (const int r = route_long(c, "rsd_distance_batch", T, in, n_pairs, bits, force_mode, nullptr, out, mode_out)) return r > 0 ? RSD_OK : -r;
    return distance_host(c, in, n_pairs, max_m_hint, max_n_hint, bits, symmask, force_mode, out, mode_out);
}

extern "C" int rsd_distance_batch_codes(rsd_ctx *c, const uint8_t *a_codes, const int32_t *a_len,
                                        const uint8_t *b_codes, const int32_t *b_len, int64_t n_pairs,
                                        int64_t max_m_hint, int64_t max_n_hint, int bits, uint32_t symmask, int force_mode,
                                        double *out, int *mode_out) {
    if (!c) return rsd_fail(RSD_EINVAL, "ctx is NULL");
    if (n_pairs < 0) return rsd_fail(RSD_EINVAL, "rsd_distance_batch_codes: n_pairs < 0");
    if (n_pairs > 0 && (!a_codes || !a_len || !b_codes || !b_len || !out))
        return rsd_fail(RSD_EINVAL, "rsd_distance_batch_codes: NULL buffer");
    if (bits != 2 && bits != 4) return rsd_fail(RSD_EINVAL, "rsd: bits must be 2 or 4");
    if (symmask == 0) symmask = bits == 2 ? 0xFu : 0x7FFFu;              // unknown: every symbol the packing can hold
    if (bits == 2 && (symmask & ~0xFu)) return rsd_fail(RSD_EINVAL, "rsd: 2-bit packing with symbols outside ACGU");
    RSD_OK_OR_RETURN(c->ensure_device());
    if (n_pairs == 0) return RSD_OK;
    // (negative lengths are caught by the block sums of distance_host: no extra pass over the 8 bytes per pair)
    const SideIn in[2] = {{nullptr, nullptr, a_len, 0, a_codes}, {nullptr, nullptr, b_len, 0, b_codes}};
    const int64_t T = long_min("RSD_DIST_NO_LONG", "RSD_DIST_LONG_MIN", DIST_LONG_MIN);
    if (const int r = route_long(c, "rsd_distance_batch", T, in, n_pairs, bits, force_mode, nullptr, out, mode_out)) return r > 0 ? RSD_OK : -r;
    return distance_host(c, in, n_pairs, max_m_hint, max_n_hint, bits, symmask, force_mode, out, mode_out);
}

// ------------------------------------------------------------------------------------------------
// one pair, whole matrix
// ------------------------------------------------------------------------------------------------
extern "C" int rsd_matrix(rsd_ctx *c, const uint8_t *a, int32_t m, const uint8_t *b, int32_t n,
                          double *values, uint8_t *mask) {
    if (!c) return rsd_fail(RSD_EINVAL, "ctx is NULL");
    if (m < 0 || n < 0 || !values || !mask || (m > 0 && !a) || (n > 0 && !b))
        return rsd_fail(RSD_EINVAL, "rsd_matrix: bad arguments");
    if ((int64_t)(m + 1) * (n + 1) > ((int64_t)1 << 31)) return rsd_fail(RSD_ERANGE, "rsd_matrix: matrix too large; use the batch entry points");
    RSD_OK_OR_RETURN(c->ensure_device());
    ModeInfo mi;
    RSD_OK_OR_RETURN(c->classify(0x7FFF, m, n, 4, RSD_MODE_F64, mi));
    cudaStream_t st = c->stream;
    RSD_OK_OR_RETURN(c->upload_costs(mi, st));
    const size_t cells = (size_t)(m + 1) * (n + 1);
    RSD_OK_OR_RETURN(c->mat_vals.ensure(sizeof(double) * cells));
    RSD_OK_OR_RETURN(c->mat_mask.ensure(cells));
    RSD_OK_OR_RETURN(c->mat_ab.ensure((size_t)m + n + 2));
    uint8_t *da = (uint8_t *)c->mat_ab.p, *db = da + m + 1;
    if (m) RSD_CUDA(cudaMemcpyAsync(da, a, m, cudaMemcpyHostToDevice, st));
    if (n) RSD_CUDA(cudaMemcpyAsync(db, b, n, cudaMemcpyHostToDevice, st));
    k_matrix_f64<<<1, 1024, 0, st>>>(da, m, db, n, c->d_fc, (double *)c->mat_vals.p, (uint8_t *)c->mat_mask.p);
    c->launches += 1;
    RSD_CUDA(cudaGetLastError());
    RSD_CUDA(cudaMemcpyAsync(values, c->mat_vals.p, sizeof(double) * cells, cudaMemcpyDeviceToHost, st));
    RSD_CUDA(cudaMemcpyAsync(mask, c->mat_mask.p, cells, cudaMemcpyDeviceToHost, st));
    RSD_CUDA(cudaStreamSynchronize(st));
    return RSD_OK;
}

// ------------------------------------------------------------------------------------------------
// issue-rate microbenchmark
// ------------------------------------------------------------------------------------------------
extern "C" int rsd_ubench(rsd_ctx *c, int which, double *ops_per_s) {
    if (!c || !ops_per_s) return rsd_fail(RSD_EINVAL, "rsd_ubench: NULL argument");
    RSD_OK_OR_RETURN(c->ensure_device());
    cudaStream_t st = c->stream;
    DevBuf &scratch = c->slots[0].scratch;
    RSD_OK_OR_RETURN(scratch.ensure(64));
    const int threads = 256, blocks = c->sm_count * 8, iters = 2000;
    const uint32_t y = 0x00010003u, z = 0x00070002u;
    float best = 1e30f;
    for (int rep = 0; rep < 4; ++rep) {
        RSD_CUDA(cudaEventRecord(c->ev0, st));
        switch (which) {
            case 0: k_ubench_u32<0><<<blocks, threads, 0, st>>>(iters, y, z, (uint32_t *)scratch.p); break;
            case 1: k_ubench_u32<1><<<blocks, threads, 0, st>>>(iters, y, z, (uint32_t *)scratch.p); break;
            case 2: k_ubench_u32<2><<<blocks, threads, 0, st>>>(iters, y, z, (uint32_t *)scratch.p); break;
            case 3: k_ubench_u32<3><<<blocks, threads, 0, st>>>(iters, y, z, (uint32_t *)scratch.p); break;
            case 4: k_ubench_f64<<<blocks, threads, 0, st>>>(iters, 1.5, (double *)scratch.p); break;
            case 5: k_ubench_u32<5><<<blocks, threads, 0, st>>>(iters, y, z, (uint32_t *)scratch.p); break;
            case 6: k_ubench_u32<6><<<blocks, threads, 0, st>>>(iters, y, z, (uint32_t *)scratch.p); break;
            case 7: k_ubench_mix<<<blocks, threads, 0, st>>>(iters, y, z, (uint32_t *)scratch.p); break;
            case 8: k_ubench_u32<8><<<blocks, threads, 0, st>>>(iters, y, z, (uint32_t *)scratch.p); break;
            case 9: k_ubench_u32<9><<<blocks, threads, 0, st>>>(iters, y, z, (uint32_t *)scratch.p); break;
            case 10: k_ubench_u32<10><<<blocks, threads, 0, st>>>(iters, y, z, (uint32_t *)scratch.p); break;
            case 11: k_ubench_u32<11><<<blocks, threads, 0, st>>>(iters, y, z, (uint32_t *)scratch.p); break;
            default: return rsd_fail(RSD_EINVAL, "rsd_ubench: unknown kind %d", which);
        }
        RSD_CUDA(cudaEventRecord(c->ev1, st));
        RSD_CUDA(cudaEventSynchronize(c->ev1));
        float ms = 0.f;
        RSD_CUDA(cudaEventElapsedTime(&ms, c->ev0, c->ev1));
        if (rep > 0) best = std::min(best, ms);
        c->launches += 1;
    }
    const double per_thread = (double)iters * RSD_UB_CHAINS * RSD_UB_REPS * (which == 7 ? 3.0 : 1.0);
    *ops_per_s = per_thread * threads * blocks / (best * 1e-3);
    return RSD_OK;
}

// ------------------------------------------------------------------------------------------------
// top-k merge after the gather (host; O(G*k) per query).  Key: score descending, global index
// ascending == the stable descending sort of performance.py:12-15 over the whole collection.
// ------------------------------------------------------------------------------------------------
extern "C" int rsd_topk_merge(const int64_t *idx, const double *score, int n_shards, int64_t n_queries, int k,
                              int64_t *out_idx, double *out_score) {
    if (!idx || !score || !out_idx || !out_score || n_shards < 1 || k < 1 || n_queries < 0)
        return rsd_fail(RSD_EINVAL, "rsd_topk_merge: bad arguments");
    std::vector<int> cur((size_t)n_shards);
    for (int64_t q = 0; q < n_queries; ++q) {
        std::fill(cur.begin(), cur.end(), 0);
        for (int r = 0; r < k; ++r) {
            int best = -1; int64_t bi = -1; double bs = 0;
            for (int g = 0; g < n_shards; ++g) {
                if (cur[g] >= k) continue;
                const size_t o = ((size_t)g * n_queries + q) * k + cur[g];
                const int64_t ci = idx[o];
                if (ci < 0) continue;                       // shard exhausted
                const double cs = score[o];
                if (best < 0 || cs > bs || (cs == bs && ci < bi)) { best = g; bi = ci; bs = cs; }
            }
            out_idx[q * k + r] = bi;
            out_score[q * k + r] = best < 0 ? 0.0 : bs;
            if (best >= 0) ++cur[best];
        }
    }
    return RSD_OK;
}


// ------------------------------------------------------------------------------------------------
// edit scripts + patch (BASELINE config 3)
// ------------------------------------------------------------------------------------------------
static int ceil_log2_i64(int64_t v) { int s = 0; while (((int64_t)1 << s) < v) ++s; return s; }

// Shared pipeline: forward (direction codes) -> traceback -> finalize, chunked so the direction
// words of one chunk fit the device budget.  Device inputs are in c->bufA / c->bufB (and c->bufX).
int rsd_ctx::script_pipeline(const int32_t *a_len, const int32_t *b_len, int64_t n_pairs, int bits, uint32_t symmask,
                             int force_mode, int64_t max_ops, bool with_x,
                             uint8_t *op, int32_t *oi, int32_t *oj, int32_t *n_ops, double *dist, uint8_t *ok,
                             int *mode_out) {
    cudaStream_t st = stream;
    last_ms_override = 0.0;
    const bool trace = getenv("RSD_TRACE") != nullptr;
    auto now = [] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    const double t_in = now();
    const int64_t max_m = [&] { int32_t v = 0; for (int64_t i = 0; i < n_pairs; ++i) v = std::max(v, a_len[i]); return (int64_t)v; }();
    const int64_t max_n = [&] { int32_t v = 0; for (int64_t i = 0; i < n_pairs; ++i) v = std::max(v, b_len[i]); return (int64_t)v; }();
    if (max_ops < max_m + max_n && n_pairs > 0) {
        for (int64_t i = 0; i < n_pairs; ++i)
            if ((int64_t)a_len[i] + b_len[i] > max_ops)
                return rsd_fail(RSD_EINVAL, "rsd_script: max_ops (%lld) < m+n (%lld) for pair %lld", (long long)max_ops,
                                (long long)((int64_t)a_len[i] + b_len[i]), (long long)i);
    }
    ModeInfo mi;
    RSD_OK_OR_RETURN(classify(symmask, max_m, max_n, bits, force_mode == RSD_MODE_I16X2 ? RSD_MODE_I32 : force_mode, mi));
    int mode = mi.mode == RSD_MODE_I16X2 ? RSD_MODE_I32 : mi.mode;
    const int S = ceil_log2_i64(max_m + max_n + 66);
    if (mode == RSD_MODE_I32) {
        int64_t maxabsw = 0;
        for (int a = 0; a < 16; ++a) for (int b = 0; b < 16; ++b) maxabsw = std::max<int64_t>(maxabsw, std::llabs((long long)mi.ic.w[a][b]));
        const double bound = ((double)max_m * mi.ic.del + (double)(max_n + 64) * mi.ic.ins + (double)maxabsw + 2.0) * std::ldexp(1.0, S)
                             + (double)(max_m + max_n + 66);
        if (bound >= 1073741000.0) {          // < 2^30: differences of two keys must not overflow either
            if (force_mode == RSD_MODE_I32) return rsd_fail(RSD_ERANGE, "rsd_script: int32 (cost,steps) key would overflow for these lengths");
            mode = RSD_MODE_F64;
        }
    }
    if (mode_out) *mode_out = mode;
    if (n_pairs == 0) return RSD_OK;
    RSD_OK_OR_RETURN(upload_costs(mi, st));
    const bool f64 = mode == RSD_MODE_F64;
    const int C = f64 ? 16 : 32;

    // per-pair direction-word counts and chunking
    // The chunk budget is what the direction buffer already holds when that was sized by an earlier call with
    // outputs of at least this size (cudaMemGetInfo costs ~15 ms with tens of GB allocated — measured); otherwise
    // 70 % of the free memory, at most 24 GiB of direction words per chunk.  RSD_SCRIPT_BUDGET_WORDS sets the budget of
    // this call alone (tests: forces the chunked path on small batches); it neither reads nor updates the measured one.
    const int64_t out_bytes = n_pairs * max_ops * (int64_t)((op ? 1 : 0) + (oi ? 4 : 0) + (oj ? 4 : 0)) + n_pairs * 32;
    const char *forced_budget = getenv("RSD_SCRIPT_BUDGET_WORDS");
    int64_t budget_words;
    if (forced_budget) budget_words = atoll(forced_budget);
    else if (dirs.p && dirs_budget_words > 0 && out_bytes <= dirs_budget_out_bytes) budget_words = dirs_budget_words;
    else {
        size_t free_b = 0, total_b = 0;
        RSD_CUDA(cudaMemGetInfo(&free_b, &total_b));
        budget_words = ((int64_t)((free_b + dirs.cap) * 0.70) - out_bytes) / 4;
        budget_words = std::min<int64_t>(budget_words, (int64_t)6 << 30);
        dirs_budget_words = budget_words; dirs_budget_out_bytes = out_bytes;
    }
    std::vector<int64_t> dir_off((size_t)n_pairs);
    std::vector<int64_t> chunk_start; chunk_start.push_back(0);
    int64_t acc = 0, chunk_max_words = 0;
    for (int64_t p = 0; p < n_pairs; ++p) {
        const int64_t n_pad = (((int64_t)b_len[p] + C - 1) / C) * C;
        const int64_t words = (((int64_t)a_len[p] + 15) / 16) * n_pad;
        const int64_t tmp_bytes_so_far = (p - chunk_start.back() + 1) * max_ops;
        if (acc > 0 && (acc + words + tmp_bytes_so_far / 4 > budget_words)) {
            chunk_max_words = std::max(chunk_max_words, acc);
            chunk_start.push_back(p); acc = 0;
        }
        if (words + max_ops / 4 > budget_words)
            return rsd_fail(RSD_ENOMEM, "rsd_script: pair %lld needs %lld direction words, device budget is %lld", (long long)p,
                            (long long)words, (long long)budget_words);
        dir_off[(size_t)p] = acc; acc += words;
    }
    chunk_max_words = std::max(chunk_max_words, acc);
    chunk_start.push_back(n_pairs);
    int64_t chunk_max_pairs = 0;
    for (size_t k = 0; k + 1 < chunk_start.size(); ++k) chunk_max_pairs = std::max(chunk_max_pairs, chunk_start[k + 1] - chunk_start[k]);

    const double t_plan = now();
    if (int rc = dirs.ensure(sizeof(uint32_t) * (size_t)(chunk_max_words + 64))) {
        if (!forced_budget) dirs_budget_words = 0;                                          // re-measure next time
        return rc;
    }
    RSD_OK_OR_RETURN(misc.ensure(sizeof(int64_t) * (size_t)n_pairs));                      // dir_off
    RSD_OK_OR_RETURN(s_tmp.ensure((size_t)chunk_max_pairs * max_ops + 16));
    RSD_OK_OR_RETURN(s_nops.ensure(sizeof(int32_t) * (size_t)n_pairs));
    RSD_OK_OR_RETURN(out_f64.ensure(sizeof(double) * (size_t)n_pairs));
    if (op) RSD_OK_OR_RETURN(s_op.ensure((size_t)n_pairs * max_ops));
    if (oi) RSD_OK_OR_RETURN(s_oi.ensure(sizeof(int32_t) * (size_t)n_pairs * max_ops));
    if (oj) RSD_OK_OR_RETURN(s_oj.ensure(sizeof(int32_t) * (size_t)n_pairs * max_ops));
    if (ok) RSD_OK_OR_RETURN(s_ok.ensure((size_t)n_pairs));
    RSD_CUDA(cudaMemcpyAsync(misc.p, dir_off.data(), sizeof(int64_t) * (size_t)n_pairs, cudaMemcpyHostToDevice, st));

    constexpr int THREADS = 128;
    const int wpb = THREADS / 32;
    const auto fwd = f64 ? (bits == 2 ? k_script_fwd<true, 2, 16> : k_script_fwd<true, 4, 16>)
                         : (bits == 2 ? k_script_fwd<false, 2, 32> : k_script_fwd<false, 4, 32>);
    int blocks = 0;
    RSD_OK_OR_RETURN(persistent_grid(fwd, THREADS, sm_count, blocks));
    const int stride = (int)max_m;       // two boundary columns of max_m rows per warp (tape passes)
    PlanSlot &sl = slots[0];
    RSD_OK_OR_RETURN(sl.scratch.ensure((size_t)(f64 ? 12 : 4) * 2 * (size_t)stride * blocks * wpb + 64));

    const uint32_t *dA = (const uint32_t *)bufA.words.p, *dB = (const uint32_t *)bufB.words.p;
    const int64_t *sA = (const int64_t *)bufA.start.p, *sB = (const int64_t *)bufB.start.p;
    const int32_t *lA = (const int32_t *)bufA.len.p, *lB = (const int32_t *)bufB.len.p;
    if (timing) RSD_CUDA(cudaEventRecord(ev0, st));
    bool rows_copied = false;
    for (size_t k = 0; k + 1 < chunk_start.size(); ++k) {
        const int64_t p0 = chunk_start[k], np = chunk_start[k + 1] - p0;
        SeqView A{dA, sA + p0, lA + p0}, B{dB, sB + p0, lB + p0};
        PlanView pv;
        // trivial pairs (m == 0 or n == 0) get their distance from the planner and an all-INS / all-DEL script from the traceback
        RSD_OK_OR_RETURN(make_plan(sl, lA + p0, lB + p0, np, C, 0, (double *)out_f64.p + p0, st, pv, max_m, max_n, 0));
        ScriptView sv{(uint32_t *)dirs.p, (const int64_t *)misc.p + p0, (double *)out_f64.p + p0};
        fwd<<<blocks, THREADS, 0, st>>>(pv, A, B, d_ic, d_fc, sv, S, sl.scratch.p, stride, -1);
        k_traceback<<<(unsigned)((np + 63) / 64), 64, 0, st>>>(lA + p0, lB + p0, np, (const uint32_t *)dirs.p,
                                                               (const int64_t *)misc.p + p0, C, (uint8_t *)s_tmp.p, max_ops,
                                                               (int32_t *)s_nops.p + p0);
        FinalizeArgs fa{};
        fa.tmp = (const uint8_t *)s_tmp.p; fa.max_ops = max_ops; fa.n_ops = (const int32_t *)s_nops.p + p0; fa.end_aligned = 1;
        fa.A = A; fa.B = B; fa.bits = bits;
        fa.X = with_x ? SeqView{(const uint32_t *)bufX.words.p, (const int64_t *)bufX.start.p + p0, (const int32_t *)bufX.len.p + p0} : A;
        fa.op = op ? (uint8_t *)s_op.p + p0 * max_ops : nullptr;
        fa.oi = oi ? (int32_t *)s_oi.p + p0 * max_ops : nullptr;
        fa.oj = oj ? (int32_t *)s_oj.p + p0 * max_ops : nullptr;
        fa.out_stride = max_ops;
        fa.patched = nullptr; fa.max_out = 0; fa.out_len = nullptr; fa.err = nullptr;
        fa.ok = ok ? (uint8_t *)s_ok.p + p0 : nullptr;
        if (op || oi || oj || ok) { k_finalize<<<(unsigned)np, 256, 0, st>>>(fa, np); launches += 1; }
        launches += 2;
        RSD_CUDA(cudaGetLastError());
        // the chunk's script rows go back on the copy stream while the next chunk computes
        if (chunk_start.size() > 2 && (op || oi || oj)) {
            const int ev = (int)(k % RSD_MAX_CHUNKS);
            RSD_CUDA(cudaEventRecord(ev_done[ev], st));
            RSD_CUDA(cudaStreamWaitEvent(copy_stream, ev_done[ev], 0));
            const size_t r0 = (size_t)p0 * max_ops, rn = (size_t)np * max_ops;
            if (op) RSD_CUDA(cudaMemcpyAsync(op + r0, (uint8_t *)s_op.p + r0, rn, cudaMemcpyDeviceToHost, copy_stream));
            if (oi) RSD_CUDA(cudaMemcpyAsync(oi + r0, (int32_t *)s_oi.p + r0, sizeof(int32_t) * rn, cudaMemcpyDeviceToHost, copy_stream));
            if (oj) RSD_CUDA(cudaMemcpyAsync(oj + r0, (int32_t *)s_oj.p + r0, sizeof(int32_t) * rn, cudaMemcpyDeviceToHost, copy_stream));
            rows_copied = true;
        }
    }
    if (timing) { RSD_CUDA(cudaEventRecord(ev1, st)); timed = true; }
    const double t_enq = now();
    if (trace) { cudaStreamSynchronize(st); fprintf(stderr, "[rsd trace] script: host prep %.3f ms, alloc+enqueue %.3f ms, kernels done after %.3f ms, %zu chunk(s)\n",
                                                   t_plan - t_in, t_enq - t_plan, now() - t_in, chunk_start.size() - 1); }
    if (!rows_copied) {
        if (op) RSD_CUDA(cudaMemcpyAsync(op, s_op.p, (size_t)n_pairs * max_ops, cudaMemcpyDeviceToHost, st));
        if (oi) RSD_CUDA(cudaMemcpyAsync(oi, s_oi.p, sizeof(int32_t) * (size_t)n_pairs * max_ops, cudaMemcpyDeviceToHost, st));
        if (oj) RSD_CUDA(cudaMemcpyAsync(oj, s_oj.p, sizeof(int32_t) * (size_t)n_pairs * max_ops, cudaMemcpyDeviceToHost, st));
    }
    if (n_ops) RSD_CUDA(cudaMemcpyAsync(n_ops, s_nops.p, sizeof(int32_t) * (size_t)n_pairs, cudaMemcpyDeviceToHost, st));
    if (dist) RSD_CUDA(cudaMemcpyAsync(dist, out_f64.p, sizeof(double) * (size_t)n_pairs, cudaMemcpyDeviceToHost, st));
    if (ok) RSD_CUDA(cudaMemcpyAsync(ok, s_ok.p, (size_t)n_pairs, cudaMemcpyDeviceToHost, st));
    if (rows_copied) RSD_CUDA(cudaStreamSynchronize(copy_stream));
    RSD_CUDA(cudaStreamSynchronize(st));
    if (trace) fprintf(stderr, "[rsd trace] script: results on the host after %.3f ms\n", now() - t_in);
    return RSD_OK;
}

static int script_common(rsd_ctx *c, const uint32_t *a_words, const int64_t *a_start, const int32_t *a_len, int64_t a_nwords,
                         const uint32_t *b_words, const int64_t *b_start, const int32_t *b_len, int64_t b_nwords,
                         int64_t n_pairs, int bits, uint32_t symmask, int force_mode, int64_t max_ops,
                         uint8_t *op, int32_t *oi, int32_t *oj, int32_t *n_ops, double *dist, uint8_t *ok, int *mode_out) {
    if (!c) return rsd_fail(RSD_EINVAL, "ctx is NULL");
    if (n_pairs < 0 || n_pairs > INT32_MAX) return rsd_fail(RSD_EINVAL, "rsd_script: n_pairs out of range");
    if (bits != 2 && bits != 4) return rsd_fail(RSD_EINVAL, "rsd: bits must be 2 or 4");
    if (n_pairs > 0 && (!a_words || !a_start || !a_len || !b_words || !b_start || !b_len))
        return rsd_fail(RSD_EINVAL, "rsd_script: NULL input buffer");
    if (max_ops < 1) return rsd_fail(RSD_EINVAL, "rsd_script: max_ops must be >= 1");
    RSD_OK_OR_RETURN(c->ensure_device());
    if (n_pairs == 0) { if (mode_out) *mode_out = 0; return RSD_OK; }
    // not for the round-trip-checking variant (ok != NULL), which patches on the device
    if (!ok) {
        const SideIn in[2] = {{a_words, a_start, a_len, a_nwords, nullptr}, {b_words, b_start, b_len, b_nwords, nullptr}};
        const LongScripts scripts{max_ops, op, oi, oj, n_ops};
        const int64_t T = long_min("RSD_SCRIPT_NO_LONG", "RSD_SCRIPT_LONG_MIN", SCRIPT_LONG_MIN);
        if (const int r = route_long(c, "rsd_script", T, in, n_pairs, bits, force_mode, &scripts, dist, mode_out)) return r > 0 ? RSD_OK : -r;
    }
    RSD_OK_OR_RETURN(c->upload_seqs(c->bufA, a_words, a_start, a_len, n_pairs, a_nwords, c->stream));
    RSD_OK_OR_RETURN(c->upload_seqs(c->bufB, b_words, b_start, b_len, n_pairs, b_nwords, c->stream));
    return c->script_pipeline(a_len, b_len, n_pairs, bits, symmask, force_mode, max_ops, false, op, oi, oj, n_ops, dist, ok, mode_out);
}

extern "C" int rsd_script_batch(rsd_ctx *c,
                                const uint32_t *a_words, const int64_t *a_start, const int32_t *a_len, int64_t a_nwords,
                                const uint32_t *b_words, const int64_t *b_start, const int32_t *b_len, int64_t b_nwords,
                                int64_t n_pairs, int bits, uint32_t symmask, int force_mode, int64_t max_ops,
                                uint8_t *op, int32_t *oi, int32_t *oj, int32_t *n_ops, double *dist, int *mode_out) {
    return script_common(c, a_words, a_start, a_len, a_nwords, b_words, b_start, b_len, b_nwords, n_pairs, bits, symmask,
                         force_mode, max_ops, op, oi, oj, n_ops, dist, nullptr, mode_out);
}

extern "C" int rsd_script_patch_check_batch(rsd_ctx *c,
                                const uint32_t *a_words, const int64_t *a_start, const int32_t *a_len, int64_t a_nwords,
                                const uint32_t *b_words, const int64_t *b_start, const int32_t *b_len, int64_t b_nwords,
                                int64_t n_pairs, int bits, uint32_t symmask, int force_mode, int64_t max_ops,
                                uint8_t *op, int32_t *oi, int32_t *oj, int32_t *n_ops, double *dist, uint8_t *ok, int *mode_out) {
    if (!ok) return rsd_fail(RSD_EINVAL, "rsd_script_patch_check_batch: ok is NULL");
    return script_common(c, a_words, a_start, a_len, a_nwords, b_words, b_start, b_len, b_nwords, n_pairs, bits, symmask,
                         force_mode, max_ops, op, oi, oj, n_ops, dist, ok, mode_out);
}

// A script handed to rsd_patch_batch must be a path of its pair (m = a_len, n = b_len): op codes in {INS, DEL, UPD},
// ending at cell (m, n), and where oi / oj are given, the cell each op enters: oj on INS / UPD, oi on DEL / UPD, the
// indices the reference's sequential patching reads (SED:380-457).  k_finalize rebuilds the entered cells from prefix
// sums of the ops, so a script with other counts would read past the pair's sequences (extra inserts also write past
// its max_out slot), and one whose indices disagree with those sums would be patched unlike the reference.  Scripts of
// rsd_script_batch, their reverses (eswire.rev_packed; the j-2 source index of a reversed delete is on an INS, which
// is not checked) and any op sequence with the right counts pass; a hand-edited script goes through sed.patching.
template <bool I, bool J>
static bool is_patch_path(const uint8_t *op, const int32_t *oi, const int32_t *oj, int32_t k, int32_t m, int32_t n) {
    uint32_t bad = 0; int32_t ci = 0, cj = 0;
    for (int32_t t = 0; t < k; ++t) {       // branch-free: 2x (with oi, oj) to 5x (op only) faster than the loop below
        const uint32_t o = op[t];
        ci += o != 0u; cj += o != 1u;
        bad |= (uint32_t)(o > 2u);
        if constexpr (I) bad |= (uint32_t)(o != 0u) & (uint32_t)(oi[t] != ci);
        if constexpr (J) bad |= (uint32_t)(o != 1u) & (uint32_t)(oj[t] != cj);
    }
    return !bad && ci == m && cj == n;
}

static int check_patch_path(int64_t p, const uint8_t *op, const int32_t *oi, const int32_t *oj, int32_t k, int32_t m, int32_t n) {
    static const char *name[3] = {"INS", "DEL", "UPD"};
    if (oi ? (oj ? is_patch_path<true, true>(op, oi, oj, k, m, n) : is_patch_path<true, false>(op, oi, oj, k, m, n))
           : (oj ? is_patch_path<false, true>(op, oi, oj, k, m, n) : is_patch_path<false, false>(op, oi, oj, k, m, n)))
        return RSD_OK;
    // not a path: find the first offending op for the message
    int32_t ci = 0, cj = 0;
    for (int32_t t = 0; t < k; ++t) {
        const uint32_t o = op[t];
        if (o > 2u) return rsd_fail(RSD_EINVAL, "rsd_patch_batch: pair %lld op %d: code %u is not INS (0), DEL (1) or UPD (2)",
                                    (long long)p, t, o);
        ci += o != 0u; cj += o != 1u;
        if (ci > m || cj > n)
            return rsd_fail(RSD_EINVAL, "rsd_patch_batch: pair %lld op %d (%s) enters cell (%d, %d) outside the %d x %d matrix of the pair",
                            (long long)p, t, name[o], ci, cj, m, n);
        if (oi && o != 0u && oi[t] != ci)
            return rsd_fail(RSD_EINVAL, "rsd_patch_batch: pair %lld op %d (%s): oi = %d, the path enters source cell %d",
                            (long long)p, t, name[o], oi[t], ci);
        if (oj && o != 1u && oj[t] != cj)
            return rsd_fail(RSD_EINVAL, "rsd_patch_batch: pair %lld op %d (%s): oj = %d, the path enters destination cell %d",
                            (long long)p, t, name[o], oj[t], cj);
    }
    if (ci != m || cj != n)
        return rsd_fail(RSD_EINVAL, "rsd_patch_batch: pair %lld ends after its %d ops at cell (%d, %d), not (%d, %d)",
                        (long long)p, k, ci, cj, m, n);
    return RSD_OK;
}

extern "C" int rsd_patch_batch(rsd_ctx *c,
                               const uint8_t *op, const int32_t *oi, const int32_t *oj, const int32_t *n_ops, int64_t max_ops,
                               const uint32_t *a_words, const int64_t *a_start, const int32_t *a_len, int64_t a_nwords,
                               const uint32_t *b_words, const int64_t *b_start, const int32_t *b_len, int64_t b_nwords,
                               const uint32_t *x_words, const int64_t *x_start, const int32_t *x_len, int64_t x_nwords,
                               int64_t n_pairs, int bits, int64_t max_out, uint8_t *out, int32_t *out_len, int32_t *err) {
    if (!c) return rsd_fail(RSD_EINVAL, "ctx is NULL");
    if (n_pairs < 0) return rsd_fail(RSD_EINVAL, "rsd_patch_batch: n_pairs < 0");
    if (n_pairs > 0 && (!op || !n_ops || !a_words || !a_len || !b_words || !b_len || !x_words || !x_len || !out || !out_len || !err))
        return rsd_fail(RSD_EINVAL, "rsd_patch_batch: NULL buffer");
    if (bits != 2 && bits != 4) return rsd_fail(RSD_EINVAL, "rsd: bits must be 2 or 4");
    // host-side validation first, so that a bad script is refused the same way with or without a device
    for (int64_t p = 0; p < n_pairs; ++p) {
        if (n_ops[p] < 0 || n_ops[p] > max_ops) return rsd_fail(RSD_EINVAL, "rsd_patch_batch: n_ops[%lld] out of range", (long long)p);
        if ((int64_t)x_len[p] + b_len[p] > max_out) return rsd_fail(RSD_EINVAL, "rsd_patch_batch: max_out too small for pair %lld", (long long)p);
        const size_t row = (size_t)p * (size_t)max_ops;
        RSD_OK_OR_RETURN(check_patch_path(p, op + row, oi ? oi + row : nullptr, oj ? oj + row : nullptr, n_ops[p], a_len[p], b_len[p]));
    }
    RSD_OK_OR_RETURN(c->ensure_device());
    if (n_pairs == 0) return RSD_OK;
    cudaStream_t st = c->stream;
    RSD_OK_OR_RETURN(c->upload_seqs(c->bufA, a_words, a_start, a_len, n_pairs, a_nwords, st));
    RSD_OK_OR_RETURN(c->upload_seqs(c->bufB, b_words, b_start, b_len, n_pairs, b_nwords, st));
    RSD_OK_OR_RETURN(c->upload_seqs(c->bufX, x_words, x_start, x_len, n_pairs, x_nwords, st));
    RSD_OK_OR_RETURN(c->s_tmp.ensure((size_t)n_pairs * max_ops + 16));
    RSD_OK_OR_RETURN(c->s_nops.ensure(sizeof(int32_t) * (size_t)n_pairs));
    RSD_OK_OR_RETURN(c->p_out.ensure((size_t)n_pairs * max_out + 16));
    RSD_OK_OR_RETURN(c->p_len.ensure(sizeof(int32_t) * (size_t)n_pairs));
    RSD_OK_OR_RETURN(c->p_err.ensure(sizeof(int32_t) * (size_t)n_pairs));
    RSD_CUDA(cudaMemcpyAsync(c->s_tmp.p, op, (size_t)n_pairs * max_ops, cudaMemcpyHostToDevice, st));
    RSD_CUDA(cudaMemcpyAsync(c->s_nops.p, n_ops, sizeof(int32_t) * (size_t)n_pairs, cudaMemcpyHostToDevice, st));
    RSD_CUDA(cudaMemsetAsync(c->p_out.p, 0, (size_t)n_pairs * max_out, st));
    FinalizeArgs fa{};
    fa.tmp = (const uint8_t *)c->s_tmp.p; fa.max_ops = max_ops; fa.n_ops = (const int32_t *)c->s_nops.p; fa.end_aligned = 0;
    fa.A = SeqView{(const uint32_t *)c->bufA.words.p, (const int64_t *)c->bufA.start.p, (const int32_t *)c->bufA.len.p};
    fa.B = SeqView{(const uint32_t *)c->bufB.words.p, (const int64_t *)c->bufB.start.p, (const int32_t *)c->bufB.len.p};
    fa.X = SeqView{(const uint32_t *)c->bufX.words.p, (const int64_t *)c->bufX.start.p, (const int32_t *)c->bufX.len.p};
    fa.bits = bits; fa.op = nullptr; fa.oi = nullptr; fa.oj = nullptr; fa.out_stride = max_ops;
    fa.patched = (uint8_t *)c->p_out.p; fa.max_out = max_out; fa.out_len = (int32_t *)c->p_len.p; fa.err = (int32_t *)c->p_err.p;
    fa.ok = nullptr;
    k_finalize<<<(unsigned)n_pairs, 256, 0, st>>>(fa, n_pairs);
    c->launches += 1;
    RSD_CUDA(cudaGetLastError());
    RSD_CUDA(cudaMemcpyAsync(out, c->p_out.p, (size_t)n_pairs * max_out, cudaMemcpyDeviceToHost, st));
    RSD_CUDA(cudaMemcpyAsync(out_len, c->p_len.p, sizeof(int32_t) * (size_t)n_pairs, cudaMemcpyDeviceToHost, st));
    RSD_CUDA(cudaMemcpyAsync(err, c->p_err.p, sizeof(int32_t) * (size_t)n_pairs, cudaMemcpyDeviceToHost, st));
    RSD_CUDA(cudaStreamSynchronize(st));
    return RSD_OK;
}

// ------------------------------------------------------------------------------------------------
// database search (BASELINE config 5)
// ------------------------------------------------------------------------------------------------
// The tier policy of the stored order, shared by rsd_db_load (host counts) and rsd_db_append (device counts).
// holds[b] = the records that contain symbol b.  rank[b] = b's place when the symbols are ordered by holds, most held
// first (stable: ties keep code order); a record's tier is the rank of its rarest symbol.
static void tier_ranks(const int64_t holds[16], int rank[16]) {
    int order[16];
    for (int b = 0; b < 16; ++b) order[b] = b;
    std::stable_sort(order, order + 16, [&](int x, int y) { return holds[x] > holds[y]; });
    for (int r = 0; r < 16; ++r) rank[order[r]] = r;
}

// tcnt[t] = the records of unmerged tier t, n their total -> r0, the number of leading tiers merged into tier 0, and
// per merged tier t: tier_end[t] (stored records [0, tier_end[t]) are of tiers <= t) and tier_mask[t] (their symbols).
static int tier_cut(const int64_t holds[16], const int64_t tcnt[16], int64_t n, int64_t tier_end[16], uint32_t tier_mask[16]) {
    int rank[16], order[16];
    tier_ranks(holds, rank);
    for (int b = 0; b < 16; ++b) order[rank[b]] = b;
    uint32_t acc = 0, mask[16];
    int64_t cum[16], s = 0;
    for (int r = 0; r < 16; ++r) {
        if (holds[order[r]] > 0) acc |= 1u << order[r];
        mask[r] = acc; s += tcnt[r]; cum[r] = s;
    }
    // The first tiers are merged up to the one that brings the prefix to half of the records: the bulk of the database
    // (for RNA: everything made of A, G, C, U, whether or not a record happens to lack one of them) is then ONE tier
    // sorted by length, and the short chunk that seeds the top-k threshold holds typical records (seeding it from
    // the handful of records that lack a common symbol gave a useless threshold: 8.7 ms in the next fold, ncu).
    int r0 = 0;
    while (r0 < 15 && cum[r0] * 2 < n) ++r0;
    for (int t = 0; t < 16; ++t) { tier_end[t] = cum[std::min(15, t + r0)]; tier_mask[t] = mask[std::min(15, t + r0)]; }
    return r0;
}

extern "C" int rsd_db_load(rsd_ctx *c, const uint32_t *words, const int64_t *start, const int32_t *len,
                           int64_t n_records, int64_t n_words, int bits, uint32_t symmask, int64_t global_index_base) {
    if (!c) return rsd_fail(RSD_EINVAL, "ctx is NULL");
    if (n_records < 0 || (n_records > 0 && (!words || !start || !len))) return rsd_fail(RSD_EINVAL, "rsd_db_load: bad arguments");
    if (bits != 2 && bits != 4) return rsd_fail(RSD_EINVAL, "rsd: bits must be 2 or 4");
    if (bits == 2 && (symmask & ~0xFu)) return rsd_fail(RSD_EINVAL, "rsd_db_load: 2-bit packing with symbols outside ACGU");
    RSD_OK_OR_RETURN(c->ensure_device());
    c->idf_ready = false;
    // Records are stored sorted by length (stable, so equal lengths keep collection order): the warps of
    // the search kernel then hold records of one length and skip the padding columns.  perm[r] is the
    // collection index of stored record r; every key and every all_scores row uses it.
    const int per = 32 / bits;
    int32_t mx = 0;
    for (int64_t i = 0; i < n_records; ++i) { if (len[i] < 0) return rsd_fail(RSD_EINVAL, "rsd_db_load: negative length"); mx = std::max(mx, len[i]); }
    std::vector<int64_t> cnt((size_t)mx + 2, 0);
    for (int64_t i = 0; i < n_records; ++i) ++cnt[(size_t)len[i] + 1];
    for (size_t l = 1; l < cnt.size(); ++l) cnt[l] += cnt[l - 1];
    std::vector<int64_t> perm((size_t)std::max<int64_t>(n_records, 1)), s_start((size_t)std::max<int64_t>(n_records, 1));
    std::vector<int32_t> s_len((size_t)std::max<int64_t>(n_records, 1));
    for (int64_t i = 0; i < n_records; ++i) perm[(size_t)cnt[(size_t)len[i]]++] = i;
    // Second key, in front of the length: the record's *tier* = the rank of its rarest symbol when the symbols are ordered
    // by the number of records that contain them.  A collection of mostly A/G/C/U(+N) records with a few full-IUPAC ones
    // (SURVEY 8d, second C5 run) then stores the common-alphabet records as a prefix: a search runs the int16x2 kernel
    // over the longest prefix whose symbols (with the query's) keep every reachable cost dyadic, and only the rest
    // through the general kernels (search_dev) — instead of the whole database in fp64 because of 1 % of its records.
    {
        std::vector<uint16_t> rmask((size_t)std::max<int64_t>(n_records, 1), 0);
        const int n_thr = n_records >= (1 << 18) ? (int)std::min<int64_t>(std::max(1u, std::thread::hardware_concurrency()), 32) : 1;
        std::atomic<int> bad_rec{0};
        auto scan = [&](int t) {
            for (int64_t i = n_records * t / n_thr, i1 = n_records * (t + 1) / n_thr; i < i1; ++i) {
                const int64_t nw = ((int64_t)len[i] + per - 1) / per;
                if (start[i] < 0 || start[i] + nw > n_words) { bad_rec.store(1); continue; }
                uint32_t m = 0;
                for (int32_t j = 0; j < len[i]; ++j) m |= 1u << ((words[start[i] + j / per] >> ((j % per) * bits)) & ((1u << bits) - 1u));
                rmask[(size_t)i] = (uint16_t)m;
            }
        };
        if (n_thr == 1) scan(0);
        else { std::vector<std::thread> pool; for (int t = 0; t < n_thr; ++t) pool.emplace_back(scan, t); for (auto &th : pool) th.join(); }
        if (bad_rec.load()) return rsd_fail(RSD_EINVAL, "rsd_db_load: a record lies outside the word buffer");
        int64_t holds[16] = {0};
        for (int64_t i = 0; i < n_records; ++i) for (int b = 0; b < 16; ++b) holds[b] += (rmask[(size_t)i] >> b) & 1;
        int rank[16];
        tier_ranks(holds, rank);
        std::vector<uint8_t> tier((size_t)std::max<int64_t>(n_records, 1), 0);
        int64_t tcnt[16] = {0};
        for (int64_t i = 0; i < n_records; ++i) {
            int t = 0;
            for (int b = 0; b < 16; ++b) if ((rmask[(size_t)i] >> b) & 1) t = std::max(t, rank[b]);
            tier[(size_t)i] = (uint8_t)t; ++tcnt[t];
        }
        const int r0 = tier_cut(holds, tcnt, n_records, c->db_tier_end, c->db_tier_mask);
        int64_t pos[16];                                            // first stored record of each merged tier
        for (int t = 0; t < 16; ++t) pos[t] = t == 0 ? 0 : c->db_tier_end[t - 1];
        std::vector<int64_t> perm2((size_t)std::max<int64_t>(n_records, 1));
        for (int64_t r = 0; r < n_records; ++r) { const int64_t i = perm[(size_t)r]; perm2[(size_t)pos[std::max(0, tier[(size_t)i] - r0)]++] = i; }     // stable: lengths stay sorted inside a tier
        perm.swap(perm2);
    }
    std::vector<uint32_t> s_words((size_t)n_words + 8, 0u);
    int64_t w = 0;
    for (int64_t r = 0; r < n_records; ++r) {                       // offsets in stored order (serial, cheap)
        const int64_t i = perm[(size_t)r];
        const int64_t nw = ((int64_t)len[i] + per - 1) / per;
        if (start[i] < 0 || start[i] + nw > n_words) return rsd_fail(RSD_EINVAL, "rsd_db_load: record %lld lies outside the word buffer", (long long)i);
        s_start[(size_t)r] = w; s_len[(size_t)r] = len[i];
        w += nw;
    }
    {                                                               // the gather itself, split over the host threads
        const int n_thr = n_records >= (1 << 18) ? (int)std::min<int64_t>(std::max(1u, std::thread::hardware_concurrency()), 32) : 1;
        auto work = [&](int t) {
            for (int64_t r = n_records * t / n_thr, r1 = n_records * (t + 1) / n_thr; r < r1; ++r) {
                const int64_t i = perm[(size_t)r];
                memcpy(s_words.data() + s_start[(size_t)r], words + start[i], sizeof(uint32_t) * (size_t)(((int64_t)len[i] + per - 1) / per));
            }
        };
        if (n_thr == 1) work(0);
        else {
            std::vector<std::thread> pool;
            for (int t = 0; t < n_thr; ++t) pool.emplace_back(work, t);
            for (auto &th : pool) th.join();
        }
    }
    RSD_OK_OR_RETURN(c->upload_seqs(c->db, s_words.data(), s_start.data(), s_len.data(), n_records, std::max<int64_t>(w, 1), c->stream));
    RSD_OK_OR_RETURN(c->db_perm.ensure(sizeof(int64_t) * (size_t)std::max<int64_t>(n_records, 1)));
    for (int64_t r = 0; r < n_records; ++r) perm[(size_t)r] += global_index_base;        // global index of stored record r
    RSD_CUDA(cudaMemcpyAsync(c->db_perm.p, perm.data(), sizeof(int64_t) * (size_t)n_records, cudaMemcpyHostToDevice, c->stream));
    RSD_CUDA(cudaStreamSynchronize(c->stream));
    c->db_n = n_records; c->db_base = global_index_base; c->db_nwords = w; c->db_bits = bits; c->db_symmask = symmask;
    c->db_maxlen = mx;
    c->db_loaded = true;
    return RSD_OK;
}

extern "C" int rsd_db_free(rsd_ctx *c) {
    if (!c) return rsd_fail(RSD_EINVAL, "ctx is NULL");
    if (c->inited && c->pid == getpid()) { cudaSetDevice(c->device); c->db.release(); c->db_perm.release(); c->db_topi.release(); c->db_tops.release(); c->db_aux.release(); c->db_dist.release(); c->rng_keys.release(); c->rng_dist.release(); c->rng_tmp.release(); c->sim_scores.release(); c->sim_aux.release(); c->sim_work.release(); c->idf_work.release(); }
    c->db_loaded = false; c->db_n = 0; c->idf_ready = false;
    return RSD_OK;
}

// Fast path (int16x2 thread-per-record kernel) applicability, per prefix of the stored order: records [0, db_tier_end[t])
// use only the symbols db_tier_mask[t] (rsd_db_load).  -> the longest prefix [0, n_fast) whose symbols, together with the
// queries', keep every reachable cost dyadic and small; its integer tables (mi_fast) and the compact symbol maps
// (lut = {syms_lo, syms_hi, lut_lo, lut_hi}).
int rsd_ctx::fast_prefix(uint32_t q_symmask, int64_t max_qlen, int bits, int force_mode, ModeInfo &mi_fast, uint32_t lut[4], int64_t &n_fast) const {
    n_fast = 0;
    lut[0] = lut[1] = 0; lut[2] = lut[3] = 0x77777777u;
    const int QROWS = (int)((max_qlen + 7) / 8 * 8);
    if (!((force_mode == 0 || force_mode == RSD_MODE_I16X2) && db_maxlen <= 32 && max_qlen >= 1 && QROWS <= 64)) return RSD_OK;
    for (int t = 0; t < 16; ++t) {
        if (t > 0 && db_tier_end[t] == db_tier_end[t - 1]) continue;          // no record adds this symbol as its rarest
        const uint32_t sm = db_tier_mask[t] | q_symmask;
        ModeInfo m2;
        RSD_OK_OR_RETURN(classify(sm, max_qlen, db_maxlen, bits, 0, m2));
        int nsym = 0;
        bool w8 = true;
        uint32_t s_lo = 0, s_hi = 0, l_lo = 0x77777777u, l_hi = 0x77777777u;
        for (int a = 0; a < 16; ++a) if (sm >> a & 1) {
            if (nsym < 7) {
                uint64_t s64 = ((uint64_t)s_hi << 32) | s_lo; s64 |= (uint64_t)a << (4 * nsym); s_lo = (uint32_t)s64; s_hi = (uint32_t)(s64 >> 32);
                uint64_t l64 = ((uint64_t)l_hi << 32) | l_lo; l64 &= ~((uint64_t)15 << (4 * a)); l64 |= (uint64_t)nsym << (4 * a);
                l_lo = (uint32_t)l64; l_hi = (uint32_t)(l64 >> 32);
            }
            ++nsym;
        }
        if (m2.dyadic)
            for (int a = 0; a < 16; ++a) for (int b2 = 0; b2 < 16; ++b2)
                if ((sm >> a & 1) && (sm >> b2 & 1) && m2.ic.w[a][b2] < -127) w8 = false;
        if (!(m2.dyadic && m2.i16_ok && w8 && nsym <= 7)) break;
        mi_fast = m2; n_fast = db_tier_end[t];
        lut[0] = s_lo; lut[1] = s_hi; lut[2] = l_lo; lut[3] = l_hi;
    }
    return RSD_OK;
}

#define RSD_RANGE_HITS0 ((int64_t)1 << 20)

// queries already on the device; outputs to device buffers (top_idx/top_score [Q][k]) and optionally all scores, or,
// with `ro`, a range search: every record within ro->max_dist of each query, appended to ro batch by batch.  Timed from
// ev0 to ev1; record_start = false keeps the ev0 of an earlier search (the first query group of a host call).
int rsd_ctx::search_dev(const uint32_t *q_words, const int64_t *q_start, const int32_t *q_len, int64_t n_queries,
                        int64_t max_qlen, int bits, uint32_t q_symmask, int k, int force_mode,
                        int64_t *top_idx, double *top_score, double *all_scores_dev, int *mode_out, cudaStream_t st, RangeOut *ro,
                        bool record_start) {
    if (!db_loaded) return rsd_fail(RSD_EINVAL, "rsd_db_search: no database loaded (rsd_db_load)");
    if (bits != db_bits) return rsd_fail(RSD_EINVAL, "rsd_db_search: query packing (%d bit) differs from the database (%d bit)", bits, db_bits);
    if (k < 0 || k > RSD_TOPK_MAX) return rsd_fail(RSD_EINVAL, "rsd_db_search: k must be in 0..%d (ask for all_scores instead)", RSD_TOPK_MAX);
    if (n_queries < 0 || n_queries > 1 << 20) return rsd_fail(RSD_EINVAL, "rsd_db_search: n_queries out of range");
    if (ro && db_n > 0xffffffffLL) return rsd_fail(RSD_EINVAL, "rsd_db_search_range: a shard holds at most 2^32 - 1 records");
    const uint32_t symmask = db_symmask | q_symmask;
    ModeInfo mi;                                  // general kernels: every symbol of the database and the queries
    RSD_OK_OR_RETURN(classify(symmask, max_qlen, db_maxlen, bits, force_mode == RSD_MODE_I16X2 ? 0 : force_mode, mi));
    timed = false; last_ms_override = 0.0;
    // Fast path (int16x2 thread-per-record kernel) applicability, per prefix of the stored order: records [0, db_tier_end[t])
    // use only the t+1 most common symbols of the database (rsd_db_load).  The longest prefix whose symbols, together with
    // the queries', keep every reachable cost dyadic and small goes through the fast kernel; the remaining records through
    // the general kernels in `mi`'s mode.  A database of A/G/C/U(+N) records with a few full-IUPAC ones (non-dyadic 0.66 /
    // 0.83 under the default table) thus pays fp64 for those few only.
    const int QROWS = (int)((max_qlen + 7) / 8 * 8);
    ModeInfo mi_fast{};
    uint32_t lut4[4] = {0, 0, 0x77777777u, 0x77777777u};
    int64_t n_fast = 0;
    RSD_OK_OR_RETURN(fast_prefix(q_symmask, max_qlen, bits, force_mode, mi_fast, lut4, n_fast));
    const uint32_t syms_lo = lut4[0], syms_hi = lut4[1], lut_lo = lut4[2], lut_hi = lut4[3];
    const int64_t n_gen = db_n - n_fast;          // records for the general kernels (stored order [n_fast, db_n))
    if (force_mode == RSD_MODE_I16X2 && n_gen > 0) return rsd_fail(RSD_EINVAL, "rsd_db_search: int16x2 search kernel not applicable (symbols, costs or lengths)");
    const bool fast = n_fast > 0;
    if (mode_out) *mode_out = n_gen == 0 ? RSD_MODE_I16X2 : mi.mode;
    if (n_queries == 0) return RSD_OK;
    if (!fast) RSD_OK_OR_RETURN(upload_costs(mi, st));

    // chunking: a small first chunk seeds tau cheaply, then large ones; candidate capacity = chunk size
    // (candidate capacity 2^21 per query: a shard of up to 2 M records — 1/8 of BASELINE config 5 — is one main chunk)
    const int64_t CH0 = 4096, CH = (int64_t)1 << 21;
    const int QB = fast ? 64 : 16;                           // queries per batch
    const int64_t cap = std::min<int64_t>(std::max<int64_t>(db_n, 1), CH);
    RSD_OK_OR_RETURN(db_topi.ensure((size_t)QB * QROWS * 8 + 64));
    TopkState tk{};
    if (!ro) {                                     // a range search keeps no top-k state
        const size_t per_q = (size_t)cap * 16 + (size_t)std::max(k, 1) * 16 + 64;
        RSD_OK_OR_RETURN(db_aux.ensure(per_q * QB + (size_t)QB * 64 * 8 + 4096));
        unsigned char *aux = (unsigned char *)db_aux.p;
        tk.k = k; tk.cap = cap;
        tk.cand_s = (double *)aux; aux += (size_t)QB * cap * 8;
        tk.cand_i = (int64_t *)aux; aux += (size_t)QB * cap * 8;
        tk.best_s = (double *)aux; aux += (size_t)QB * std::max(k, 1) * 8;
        tk.best_i = (int64_t *)aux; aux += (size_t)QB * std::max(k, 1) * 8;
        tk.tau_s = (double *)aux; aux += (size_t)QB * 8;
        tk.tau_i = (int64_t *)aux; aux += (size_t)QB * 8;
        tk.cand_n = (int *)aux; aux += (size_t)QB * 4;
    }
    RangeHits rh{};
    if (ro) {
        // the fast kernel compares the scaled integer distance with floor(max_dist * 2^k) (exact: a power-of-two scale)
        const double t = std::floor(std::ldexp(ro->max_dist, mi_fast.ic.scale_log2));
        rh.thr = t >= (double)INT32_MAX ? INT32_MAX : (int)t;
        rh.max_dist = ro->max_dist;
        RSD_OK_OR_RETURN(range_reserve(std::max<int64_t>(RSD_RANGE_HITS0, range_cap()), QB));
    }
    uint2 *rowtab = (uint2 *)db_topi.p;
    const int64_t cap_gen = std::min<int64_t>(std::max<int64_t>(n_gen, 1), cap);
    const int64_t gen_pairs_max = (int64_t)1 << 23;                          // (query, record) pairs per launch train of the general path
    const int64_t gen_pairs_cap = std::max<int64_t>(cap_gen, std::min<int64_t>(gen_pairs_max, (int64_t)QB * cap_gen));
    if (n_gen > 0) {
        RSD_OK_OR_RETURN(db_dist.ensure((size_t)gen_pairs_cap * 8 + 64));
        RSD_OK_OR_RETURN(db_tops.ensure((size_t)gen_pairs_cap * 24 + 64));
    }
    SearchTab tab{};
    tab.ins = mi_fast.ic.ins; tab.del = mi_fast.ic.del; tab.inv_scale = 1.0 / (double)(1 << mi_fast.ic.scale_log2);
    tab.compact_lut_lo = lut_lo; tab.compact_lut_hi = lut_hi;
    const uint32_t *dbw = (const uint32_t *)db.words.p; const int64_t *dbs = (const int64_t *)db.start.p; const int32_t *dbl = (const int32_t *)db.len.p;
    if (timing && record_start) RSD_CUDA(cudaEventRecord(ev0, st));
    for (int64_t q0 = 0; q0 < n_queries; q0 += QB) {
        const int nq = (int)std::min<int64_t>(QB, n_queries - q0);
        if (k > 0) { k_topk_init<<<(nq + 63) / 64, 64, 0, st>>>(tk, nq); launches += 1; }
        if (ro) {
            rh.keys = (unsigned long long *)rng_keys.p; rh.dist = (double *)rng_dist.p; rh.n = (unsigned long long *)rng_n.p;
            rh.cap = range_cap();
            RSD_CUDA(cudaMemsetAsync(rh.n, 0, sizeof(unsigned long long), st));
        }
        double *alls = all_scores_dev ? all_scores_dev + (size_t)q0 * db_n : nullptr;
        if (fast) {
            // the integer tables of the fast prefix (the general part below uploads its own; stream order keeps them apart)
            RSD_OK_OR_RETURN(upload_costs(mi_fast, st));
            k_build_rowtab<<<(nq * QROWS + 127) / 128, 128, 0, st>>>(q_words, q_start + q0, q_len + q0, nq, bits, QROWS, d_ic, syms_lo, syms_hi, rowtab);
            launches += 1;
            // a short first chunk (its queries spread over blockIdx.y) seeds tau; the rest goes in equal chunks <= cap
            const int64_t rest = std::max<int64_t>(n_fast - CH0, 0);
            const int64_t n_main = (rest + cap - 1) / std::max<int64_t>(cap, 1);
            int64_t main_sz = n_main ? std::min<int64_t>(cap, ((rest + n_main - 1) / n_main + 255) / 256 * 256) : cap;
            int64_t wave = 0;
            if (!getenv("RSD_SEARCH_NOWAVE")) {
                // the CTAs of a chunk do equal work (the database is sorted by length), so they finish wave by wave: a chunk
                // that is a whole number of waves (resident CTAs x 256 records) leaves no partly filled last wave
                int per_sm = 0;
                const size_t smem_q = (size_t)nq * QROWS * 8 + (size_t)nq * 20 + 16;
                if (search_per_sm_nq != nq || search_per_sm_qrows != QROWS || search_per_sm_range != (ro != nullptr)) {
                    RSD_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, ro ? k_search_twin16<true> : k_search_twin16<false>, 128, smem_q));
                    search_per_sm = per_sm; search_per_sm_nq = nq; search_per_sm_qrows = QROWS; search_per_sm_range = ro != nullptr;
                }
                per_sm = search_per_sm;
                wave = (int64_t)std::max(per_sm, 1) * sm_count * 256;
                if (rest > cap && cap >= wave) main_sz = cap / wave * wave;       // a shard that fits one chunk goes in one launch (finer waves below)
            }
            for (int64_t r0 = 0; r0 < n_fast;) {
                const bool seed = !ro && r0 == 0 && n_fast > CH0;
                const int64_t nr = std::min<int64_t>(seed ? CH0 : main_sz, n_fast - r0);
                const int64_t threads = (nr + 1) / 2;
                const size_t smem = (size_t)nq * QROWS * 8 + (size_t)nq * 20 + 16;
                // A chunk of only a few waves (a small shard: 1/8 of the database per GPU) ends in a partly filled wave that
                // costs as much as a full one.  Splitting the query batch over blockIdx.y makes the CTAs shorter and the
                // waves more numerous (>= 12), so that tail shrinks with them; the selectors are rebuilt per CTA (cheap).
                unsigned gy = seed ? (unsigned)std::min(nq, 8) : 1u;
                int64_t want_waves = 12;              // measured on a 1.25 M-record shard: 12 -> 4.37 ms, 24 -> 4.43, 48 -> 4.64, 96 -> 5.12 (selectors are rebuilt per CTA)
                if (const char *e = getenv("RSD_SEARCH_WAVES")) want_waves = std::max(atoi(e), 1);
                if (!seed && wave > 0 && nr < want_waves * wave) gy = (unsigned)std::min<int64_t>(std::min(nq, 16), (want_waves * wave + nr - 1) / std::max<int64_t>(nr, 1));
                const dim3 grid((unsigned)((threads + 127) / 128), gy);
                if (ro) k_search_twin16<true><<<grid, 128, smem, st>>>(dbw, dbs, dbl, r0, nr, db_bits, (const int64_t *)db_perm.p, db_base, rowtab, QROWS,
                                                                       q_len + q0, nq, tab, tk, nullptr, db_n, 1u, rh);
                else k_search_twin16<false><<<grid, 128, smem, st>>>(dbw, dbs, dbl, r0, nr, db_bits, (const int64_t *)db_perm.p, db_base, rowtab, QROWS,
                                                                     q_len + q0, nq, tab, tk, alls, db_n, 1u, rh);
                launches += 1;
                if (k > 0) { k_topk_fold<<<nq, 256, 0, st>>>(tk); launches += 1; }
                RSD_CUDA(cudaGetLastError());
                r0 += nr;
            }
        }
        // records outside the fast prefix (or all of them) through the systolic distance kernels: (query, record) pairs of
        // several queries per launch train (fill views, plan, distance kernel, score filter), up to PAIRS_MAX pairs at a time
        for (int64_t r0 = n_fast; r0 < db_n;) {
            // without a fast prefix nothing has seeded the thresholds yet: a short first chunk does (every record of an
            // unseeded 2 M-record chunk was a candidate: 1.4 ms of atomics and a 30 ms fold, ncu)
            const bool seed_gen = !fast && r0 == 0 && k > 0 && db_n > CH0;
            const int64_t nr = std::min<int64_t>(seed_gen ? CH0 : cap_gen, db_n - r0);
            const int qb_max = (int)std::max<int64_t>(1, std::min<int64_t>(nq, gen_pairs_max / std::max<int64_t>(nr, 1)));
            for (int qa = 0; qa < nq; qa += qb_max) {
                const int nqb = std::min(qb_max, nq - qa);
                const int64_t np = (int64_t)nqb * nr;
                int64_t *va_s = (int64_t *)db_tops.p, *vb_s = va_s + gen_pairs_cap;
                int32_t *va_l = (int32_t *)(vb_s + gen_pairs_cap), *vb_l = va_l + gen_pairs_cap;
                k_fill_pairs_view<<<(unsigned)((np + 255) / 256), 256, 0, st>>>(q_start + q0, q_len + q0, qa, nqb, dbs, dbl, r0, nr, va_s, va_l, vb_s, vb_l);
                launches += 1;
                int mode_unused = 0;
                RSD_OK_OR_RETURN(distance_dev(q_words, va_s, va_l, dbw, vb_s, vb_l, np, max_qlen, db_maxlen, bits, symmask,
                                              force_mode == RSD_MODE_I16X2 ? 0 : force_mode, (double *)db_dist.p, &mode_unused, st, nullptr, nullptr));
                if (ro) k_range_filter_pairs<<<(unsigned)((np + 255) / 256), 256, 0, st>>>((const double *)db_dist.p, r0, nr, (const int64_t *)db_perm.p, db_base, qa, nqb, rh);
                else k_score_filter_pairs<<<(unsigned)((np + 255) / 256), 256, 0, st>>>((const double *)db_dist.p, r0, nr, (const int64_t *)db_perm.p, db_base, qa, nqb, tk, alls, db_n);
                launches += 1;
            }
            if (k > 0) { k_topk_fold<<<nq, 256, 0, st>>>(tk); launches += 1; }
            RSD_CUDA(cudaGetLastError());
            r0 += nr;
        }
        if (k > 0) {
            RSD_CUDA(cudaMemcpyAsync(top_idx + q0 * k, tk.best_i, sizeof(int64_t) * (size_t)nq * k, cudaMemcpyDeviceToDevice, st));
            RSD_CUDA(cudaMemcpyAsync(top_score + q0 * k, tk.best_s, sizeof(double) * (size_t)nq * k, cudaMemcpyDeviceToDevice, st));
        }
        if (ro) {
            bool rerun = false;
            RSD_OK_OR_RETURN(range_collect(nq, QB, *ro, rerun, st));
            if (rerun) q0 -= QB;                 // the buffer now holds the batch's exact count: the same batch again
        }
    }
    if (timing) { RSD_CUDA(cudaEventRecord(ev1, st)); timed = true; }
    return RSD_OK;
}

// Range search hit buffer: room for `hits` hits (keys and distances, each twice for the sort's double buffer), the
// counter and qb + 1 offsets.  Starts at RSD_RANGE_HITS0 hits and grows to the exact count of a batch that overflowed.
int rsd_ctx::range_reserve(int64_t hits, int qb) {
    RSD_OK_OR_RETURN(rng_keys.ensure(sizeof(unsigned long long) * 2 * (size_t)hits));
    RSD_OK_OR_RETURN(rng_dist.ensure(sizeof(double) * 2 * (size_t)hits));
    RSD_OK_OR_RETURN(rng_n.ensure(sizeof(int64_t) * (size_t)(qb + 2)));
    return RSD_OK;
}

// After a query batch of a range search: the hit count comes back; a count above the buffer grows it and asks for the
// batch again (rerun).  Otherwise the hits are sorted by key (query in batch, then collection index: the store order is
// (tier, length)), split per query, and appended to `ro`.
int rsd_ctx::range_collect(int nq, int qb, RangeOut &ro, bool &rerun, cudaStream_t st) {
    unsigned long long n = 0;
    RSD_CUDA(cudaMemcpyAsync(&n, rng_n.p, sizeof n, cudaMemcpyDeviceToHost, st));
    RSD_CUDA(cudaStreamSynchronize(st));
    const int64_t cap_h = range_cap();
    rerun = (int64_t)n > cap_h;
    if (rerun) return range_reserve((int64_t)n, qb);
    cub::DoubleBuffer<unsigned long long> kb((unsigned long long *)rng_keys.p, (unsigned long long *)rng_keys.p + cap_h);
    cub::DoubleBuffer<double> vb((double *)rng_dist.p, (double *)rng_dist.p + cap_h);
    if (n > 1) {
        int end_bit = 32;
        while ((1 << (end_bit - 32)) < nq) ++end_bit;
        size_t tmp = 0;
        RSD_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tmp, kb, vb, (int64_t)n, 0, end_bit, st));
        RSD_OK_OR_RETURN(rng_tmp.ensure(tmp));
        RSD_CUDA(cub::DeviceRadixSort::SortPairs(rng_tmp.p, tmp, kb, vb, (int64_t)n, 0, end_bit, st));
        launches += 1;
    }
    int64_t *off_d = (int64_t *)rng_n.p + 1, *idx_d = (int64_t *)kb.Alternate();
    const int64_t nt = std::max<int64_t>((int64_t)n, nq + 1);
    k_range_split<<<(unsigned)((nt + 255) / 256), 256, 0, st>>>(kb.Current(), (int64_t)n, nq, db_base, idx_d, off_d);
    launches += 1;
    RSD_CUDA(cudaGetLastError());
    std::vector<int64_t> off((size_t)nq + 1);
    const size_t h0 = ro.idx.size();
    ro.idx.resize(h0 + n); ro.dist.resize(h0 + n);
    RSD_CUDA(cudaMemcpyAsync(off.data(), off_d, sizeof(int64_t) * off.size(), cudaMemcpyDeviceToHost, st));
    if (n) {
        RSD_CUDA(cudaMemcpyAsync(ro.idx.data() + h0, idx_d, sizeof(int64_t) * n, cudaMemcpyDeviceToHost, st));
        RSD_CUDA(cudaMemcpyAsync(ro.dist.data() + h0, vb.Current(), sizeof(double) * n, cudaMemcpyDeviceToHost, st));
    }
    RSD_CUDA(cudaStreamSynchronize(st));
    for (int q = 0; q < nq; ++q) ro.cnt.push_back(off[(size_t)q + 1] - off[(size_t)q]);
    return RSD_OK;
}

extern "C" int rsd_db_search_topk_dev(rsd_ctx *c, const uint32_t *q_words_dev, const int64_t *q_start_dev,
                                      const int32_t *q_len_dev, int64_t n_queries, int64_t max_qlen, int bits,
                                      uint32_t q_symmask, int k, int force_mode,
                                      int64_t *top_idx_dev, double *top_score_dev, int *mode_out, void *stream) {
    if (!c) return rsd_fail(RSD_EINVAL, "ctx is NULL");
    RSD_OK_OR_RETURN(c->ensure_device());
    if (k < 1) return rsd_fail(RSD_EINVAL, "rsd_db_search_topk_dev: k must be >= 1");
    return c->search_dev(q_words_dev, q_start_dev, q_len_dev, n_queries, max_qlen, bits, q_symmask, k, force_mode,
                         top_idx_dev, top_score_dev, nullptr, mode_out, (cudaStream_t)stream, nullptr, true);
}

// order (empty: caller order) = the caller's query of every device row; rows [0, n_first) form the first group
struct QueryGroups {
    std::vector<int64_t> order;
    int64_t n_first = 0;
    uint32_t mask_first = 0, mask_rest = 0;
};

// the queries are already in c->bufQ; their start / len there are rewritten in group order
static int group_queries(rsd_ctx *c, const char *who, const uint32_t *q_words, const int64_t *q_start, const int32_t *q_len,
                         int64_t n_queries, int64_t q_nwords, int bits, uint32_t q_symmask, int force_mode, int64_t max_qlen,
                         QueryGroups &qg) {
    // A query that carries a symbol outside the fast kernel's reach (an ambiguity code whose costs are not dyadic) would
    // send every query of its batch through the general kernels for the whole database.  Queries are therefore grouped:
    // those that leave a fast prefix first, the others after them, one search per group.
    std::vector<int64_t> &order = qg.order;
    order.clear();
    qg.n_first = n_queries; qg.mask_first = q_symmask; qg.mask_rest = 0;
    if (n_queries > 1 && force_mode == 0) {
        const int per = 32 / bits;
        std::vector<uint32_t> qm((size_t)n_queries, 0u);
        for (int64_t q = 0; q < n_queries; ++q) {
            if (q_start[q] < 0 || q_start[q] + ((int64_t)q_len[q] + per - 1) / per > q_nwords) return rsd_fail(RSD_EINVAL, "%s: query %lld lies outside the word buffer", who, (long long)q);
            for (int32_t j = 0; j < q_len[q]; ++j) qm[(size_t)q] |= 1u << ((q_words[q_start[q] + j / per] >> ((j % per) * bits)) & ((1u << bits) - 1u));
        }
        std::vector<uint32_t> ok_masks, bad_masks;         // masks already classified (few distinct ones)
        std::vector<char> friendly((size_t)n_queries, 0);
        for (int64_t q = 0; q < n_queries; ++q) {
            const uint32_t m = qm[(size_t)q];
            bool known = false, ok = false;
            for (uint32_t x : ok_masks) if (x == m) { known = true; ok = true; }
            for (uint32_t x : bad_masks) if (x == m) known = true;
            if (!known) {
                ModeInfo mf; uint32_t l4[4]; int64_t nf = 0;
                RSD_OK_OR_RETURN(c->fast_prefix(m, max_qlen, bits, 0, mf, l4, nf));
                ok = nf > 0;
                (ok ? ok_masks : bad_masks).push_back(m);
            }
            friendly[(size_t)q] = ok;
        }
        int64_t n_ok = 0;
        for (int64_t q = 0; q < n_queries; ++q) n_ok += friendly[(size_t)q];
        // the union of the friendly queries' symbols must itself leave a fast prefix (it does when each one does and the
        // costs among their symbols are dyadic; checked, not assumed)
        if (n_ok > 0 && n_ok < n_queries) {
            uint32_t mu = 0;
            for (int64_t q = 0; q < n_queries; ++q) if (friendly[(size_t)q]) mu |= qm[(size_t)q];
            ModeInfo mf; uint32_t l4[4]; int64_t nf = 0;
            RSD_OK_OR_RETURN(c->fast_prefix(mu, max_qlen, bits, 0, mf, l4, nf));
            if (nf > 0) {
                order.reserve((size_t)n_queries);
                for (int64_t q = 0; q < n_queries; ++q) if (friendly[(size_t)q]) order.push_back(q);
                for (int64_t q = 0; q < n_queries; ++q) if (!friendly[(size_t)q]) { order.push_back(q); qg.mask_rest |= qm[(size_t)q]; }
                qg.n_first = n_ok; qg.mask_first = mu;
            }
        }
    }
    if (!order.empty()) {                             // queries in group order on the device (the words stay where they are)
        std::vector<int64_t> ps((size_t)n_queries); std::vector<int32_t> pl((size_t)n_queries);
        for (int64_t r = 0; r < n_queries; ++r) { ps[(size_t)r] = q_start[order[(size_t)r]]; pl[(size_t)r] = q_len[order[(size_t)r]]; }
        RSD_CUDA(cudaMemcpyAsync(c->bufQ.start.p, ps.data(), sizeof(int64_t) * (size_t)n_queries, cudaMemcpyHostToDevice, c->stream));
        RSD_CUDA(cudaMemcpyAsync(c->bufQ.len.p, pl.data(), sizeof(int32_t) * (size_t)n_queries, cudaMemcpyHostToDevice, c->stream));
        RSD_CUDA(cudaStreamSynchronize(c->stream));          // ps / pl are pageable temporaries
    }
    return RSD_OK;
}

// one search_dev per group (rows of c->bufQ); top-k rows go to c->s_oi / c->s_oj, all_scores rows to c->out_f64, and range
// hits (ro) are appended row by row
static int search_groups(rsd_ctx *c, const QueryGroups &qg, int64_t n_queries, int64_t max_qlen, int bits, int kk, int force_mode,
                         bool all_scores, RangeOut *ro, int &mode_all) {
    mode_all = 0;
    for (int g = 0; g < 2; ++g) {
        const int64_t g0 = g == 0 ? 0 : qg.n_first, g1 = g == 0 ? qg.n_first : n_queries;
        if (g1 <= g0) continue;
        int mo = 0;
        RSD_OK_OR_RETURN(c->search_dev((const uint32_t *)c->bufQ.words.p, (const int64_t *)c->bufQ.start.p + g0, (const int32_t *)c->bufQ.len.p + g0,
                                       g1 - g0, max_qlen, bits, g == 0 ? qg.mask_first : qg.mask_rest, kk, force_mode,
                                       ro ? nullptr : (int64_t *)c->s_oi.p + g0 * kk, ro ? nullptr : (double *)c->s_oj.p + g0 * kk,
                                       all_scores ? (double *)c->out_f64.p + (size_t)g0 * c->db_n : nullptr, &mo, c->stream, ro, g0 == 0));
        mode_all = std::max(mode_all, mo);
    }
    return RSD_OK;
}

extern "C" int rsd_db_search_topk(rsd_ctx *c, const uint32_t *q_words, const int64_t *q_start, const int32_t *q_len,
                                  int64_t n_queries, int64_t q_nwords, int bits, uint32_t q_symmask, int k, int force_mode,
                                  int64_t *top_idx, double *top_score, double *all_scores, int *mode_out) {
    if (!c) return rsd_fail(RSD_EINVAL, "ctx is NULL");
    if (n_queries < 0 || (n_queries > 0 && (!q_words || !q_start || !q_len))) return rsd_fail(RSD_EINVAL, "rsd_db_search_topk: bad arguments");
    if (k > 0 && (!top_idx || !top_score)) return rsd_fail(RSD_EINVAL, "rsd_db_search_topk: NULL top-k output");
    RSD_OK_OR_RETURN(c->ensure_device());
    if (n_queries == 0) return RSD_OK;
    cudaStream_t st = c->stream;
    RSD_OK_OR_RETURN(c->upload_seqs(c->bufQ, q_words, q_start, q_len, n_queries, q_nwords, st));
    const int kk = std::max(k, 0);
    RSD_OK_OR_RETURN(c->s_oi.ensure(sizeof(int64_t) * (size_t)n_queries * std::max(kk, 1)));
    RSD_OK_OR_RETURN(c->s_oj.ensure(sizeof(double) * (size_t)n_queries * std::max(kk, 1)));
    if (all_scores) RSD_OK_OR_RETURN(c->out_f64.ensure(sizeof(double) * (size_t)n_queries * std::max<int64_t>(c->db_n, 1)));
    int64_t max_qlen = 0;
    for (int64_t i = 0; i < n_queries; ++i) max_qlen = std::max<int64_t>(max_qlen, q_len[i]);
    QueryGroups qg;
    RSD_OK_OR_RETURN(group_queries(c, "rsd_db_search_topk", q_words, q_start, q_len, n_queries, q_nwords, bits, q_symmask, force_mode, max_qlen, qg));
    const std::vector<int64_t> &order = qg.order;
    int mode_all = 0;
    RSD_OK_OR_RETURN(search_groups(c, qg, n_queries, max_qlen, bits, kk, force_mode, all_scores != nullptr, nullptr, mode_all));
    if (mode_out) *mode_out = mode_all;
    if (order.empty()) {
        if (kk > 0) {
            RSD_CUDA(cudaMemcpyAsync(top_idx, c->s_oi.p, sizeof(int64_t) * (size_t)n_queries * kk, cudaMemcpyDeviceToHost, st));
            RSD_CUDA(cudaMemcpyAsync(top_score, c->s_oj.p, sizeof(double) * (size_t)n_queries * kk, cudaMemcpyDeviceToHost, st));
        }
        if (all_scores) RSD_CUDA(cudaMemcpyAsync(all_scores, c->out_f64.p, sizeof(double) * (size_t)n_queries * c->db_n, cudaMemcpyDeviceToHost, st));
    } else {
        for (int64_t r = 0; r < n_queries; ++r) {       // row r of the device results belongs to query order[r]
            const int64_t q = order[(size_t)r];
            if (kk > 0) {
                RSD_CUDA(cudaMemcpyAsync(top_idx + q * kk, (int64_t *)c->s_oi.p + r * kk, sizeof(int64_t) * (size_t)kk, cudaMemcpyDeviceToHost, st));
                RSD_CUDA(cudaMemcpyAsync(top_score + q * kk, (double *)c->s_oj.p + r * kk, sizeof(double) * (size_t)kk, cudaMemcpyDeviceToHost, st));
            }
            if (all_scores) RSD_CUDA(cudaMemcpyAsync(all_scores + (size_t)q * c->db_n, (double *)c->out_f64.p + (size_t)r * c->db_n, sizeof(double) * (size_t)c->db_n, cudaMemcpyDeviceToHost, st));
        }
    }
    RSD_CUDA(cudaStreamSynchronize(st));
    return RSD_OK;
}

// Range search of one shard, host queries in, hits out per query in caller order (rsd_db_search_range and every shard of
// rsd_multi_db_search_range).
static int range_shard(rsd_ctx *c, const uint32_t *q_words, const int64_t *q_start, const int32_t *q_len, int64_t n_queries,
                       int64_t q_nwords, int bits, uint32_t q_symmask, double max_dist, int force_mode, RangeOut &out, int *mode_out) {
    RSD_OK_OR_RETURN(c->upload_seqs(c->bufQ, q_words, q_start, q_len, n_queries, q_nwords, c->stream));
    int64_t max_qlen = 0;
    for (int64_t i = 0; i < n_queries; ++i) max_qlen = std::max<int64_t>(max_qlen, q_len[i]);
    QueryGroups qg;
    RSD_OK_OR_RETURN(group_queries(c, "rsd_db_search_range", q_words, q_start, q_len, n_queries, q_nwords, bits, q_symmask, force_mode, max_qlen, qg));
    RangeOut ro;
    ro.max_dist = max_dist;
    int mode_all = 0;
    RSD_OK_OR_RETURN(search_groups(c, qg, n_queries, max_qlen, bits, 0, force_mode, false, &ro, mode_all));
    if (mode_out) *mode_out = mode_all;
    if (qg.order.empty()) { out = std::move(ro); return RSD_OK; }
    std::vector<int64_t> row0((size_t)n_queries + 1, 0), row_of((size_t)n_queries);      // device row -> first hit; query -> row
    for (int64_t r = 0; r < n_queries; ++r) { row0[(size_t)r + 1] = row0[(size_t)r] + ro.cnt[(size_t)r]; row_of[(size_t)qg.order[(size_t)r]] = r; }
    out.cnt.assign((size_t)n_queries, 0); out.idx.resize(ro.idx.size()); out.dist.resize(ro.dist.size());
    int64_t h = 0;
    for (int64_t q = 0; q < n_queries; ++q) {
        const int64_t r = row_of[(size_t)q], n = ro.cnt[(size_t)r];
        std::copy_n(ro.idx.begin() + row0[(size_t)r], n, out.idx.begin() + h);
        std::copy_n(ro.dist.begin() + row0[(size_t)r], n, out.dist.begin() + h);
        out.cnt[(size_t)q] = n; h += n;
    }
    return RSD_OK;
}

// CSR output of a range search: each query's hits of shard 0, then shard 1, ... (the shards are index-contiguous, so
// this is collection order).  hit_off is always written; more hits than cap is RSD_ERANGE, never a silent cut.
static int range_emit(const char *who, const std::vector<RangeOut> &shards, int64_t n_queries, int64_t cap,
                      int64_t *hit_off, int64_t *hit_idx, double *hit_dist) {
    hit_off[0] = 0;
    for (int64_t q = 0; q < n_queries; ++q) {
        int64_t n = 0;
        for (const RangeOut &o : shards) n += o.cnt[(size_t)q];
        hit_off[q + 1] = hit_off[q] + n;
    }
    if (hit_off[n_queries] > cap)
        return rsd_fail(RSD_ERANGE, "%s: %lld hits exceed cap = %lld (hit_off holds every query's count)", who,
                        (long long)hit_off[n_queries], (long long)cap);
    std::vector<int64_t> pos(shards.size(), 0);
    int64_t h = 0;
    for (int64_t q = 0; q < n_queries; ++q)
        for (size_t g = 0; g < shards.size(); ++g) {
            const int64_t n = shards[g].cnt[(size_t)q];
            if (n) {
                memcpy(hit_idx + h, shards[g].idx.data() + pos[g], sizeof(int64_t) * (size_t)n);
                memcpy(hit_dist + h, shards[g].dist.data() + pos[g], sizeof(double) * (size_t)n);
            }
            pos[g] += n; h += n;
        }
    return RSD_OK;
}

// argument checks of both range entry points (before any device work)
static int range_args(const char *who, const uint32_t *q_words, const int64_t *q_start, const int32_t *q_len, int64_t n_queries,
                      double max_dist, int64_t cap, const int64_t *hit_off, const int64_t *hit_idx, const double *hit_dist) {
    if (n_queries < 0 || (n_queries > 0 && (!q_words || !q_start || !q_len))) return rsd_fail(RSD_EINVAL, "%s: bad arguments", who);
    if (!(max_dist >= 0.0)) return rsd_fail(RSD_EINVAL, "%s: max_dist must be >= 0 and not NaN (got %g)", who, max_dist);
    if (cap < 0 || !hit_off || (cap > 0 && (!hit_idx || !hit_dist))) return rsd_fail(RSD_EINVAL, "%s: bad output arrays", who);
    return RSD_OK;
}

extern "C" int rsd_db_search_range(rsd_ctx *c, const uint32_t *q_words, const int64_t *q_start, const int32_t *q_len,
                                   int64_t n_queries, int64_t q_nwords, int bits, uint32_t q_symmask, double max_dist,
                                   int force_mode, int64_t cap, int64_t *hit_off, int64_t *hit_idx, double *hit_dist,
                                   int *mode_out) {
    if (!c) return rsd_fail(RSD_EINVAL, "ctx is NULL");
    RSD_OK_OR_RETURN(range_args("rsd_db_search_range", q_words, q_start, q_len, n_queries, max_dist, cap, hit_off, hit_idx, hit_dist));
    RSD_OK_OR_RETURN(c->ensure_device());
    hit_off[0] = 0;
    if (n_queries == 0) return RSD_OK;
    std::vector<RangeOut> out(1);
    RSD_OK_OR_RETURN(range_shard(c, q_words, q_start, q_len, n_queries, q_nwords, bits, q_symmask, max_dist, force_mode, out[0], mode_out));
    return range_emit("rsd_db_search_range", out, n_queries, cap, hit_off, hit_idx, hit_dist);
}

// ------------------------------------------------------------------------------------------------
// set / multiset / TF-vector similarity search (SURVEY 8f rank 4)
// ------------------------------------------------------------------------------------------------
extern "C" int rsd_db_similarity(rsd_ctx *c, const uint8_t *q_codes, int32_t q_len, int method, int k,
                                 int64_t *top_idx, double *top_score, double *all_scores) {
    if (!c) return rsd_fail(RSD_EINVAL, "ctx is NULL");
    if (method < 0 || method >= RSD_SIM_COUNT) return rsd_fail(RSD_EINVAL, "rsd_db_similarity: unknown method %d", method);
    if (q_len < 0 || (q_len > 0 && !q_codes)) return rsd_fail(RSD_EINVAL, "rsd_db_similarity: bad query");
    if (k < 0 || k > RSD_TOPK_MAX) return rsd_fail(RSD_EINVAL, "rsd_db_similarity: k must be in 0..%d", RSD_TOPK_MAX);
    if (k > 0 && (!top_idx || !top_score)) return rsd_fail(RSD_EINVAL, "rsd_db_similarity: NULL top-k output");
    for (int32_t i = 0; i < q_len; ++i)
        if (q_codes[i] >= 15) return rsd_fail(RSD_EINVAL, "rsd_db_similarity: query code %u at %d is not a symbol", q_codes[i], i);
    RSD_OK_OR_RETURN(c->ensure_device());
    if (!c->db_loaded) return rsd_fail(RSD_EINVAL, "rsd_db_similarity: no database loaded (rsd_db_load)");
    cudaStream_t st = c->stream;
    c->timed = false; c->last_ms_override = 0.0;
    const int64_t n = c->db_n;
    RSD_OK_OR_RETURN(c->sim_codes.ensure((size_t)q_len + 16));
    RSD_OK_OR_RETURN(c->sim_q.ensure(sizeof(SimQuery)));
    RSD_OK_OR_RETURN(c->sim_scores.ensure(sizeof(double) * (size_t)std::max<int64_t>(n, 1)));
    if (q_len) RSD_CUDA(cudaMemcpyAsync(c->sim_codes.p, q_codes, (size_t)q_len, cudaMemcpyHostToDevice, st));
    if (c->timing) RSD_CUDA(cudaEventRecord(c->ev0, st));
    k_sim_query<<<1, 32, 0, st>>>((const uint8_t *)c->sim_codes.p, q_len, (SimQuery *)c->sim_q.p);
    c->launches += 1;
    const uint32_t *dbw = (const uint32_t *)c->db.words.p; const int64_t *dbs = (const int64_t *)c->db.start.p; const int32_t *dbl = (const int32_t *)c->db.len.p;
    double *scores = (double *)c->sim_scores.p;
    if (n > 0) {
        if (method < RSD_SIM_COSINE) {
            k_sim_small<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(dbw, dbs, dbl, n, c->db_bits, (const int64_t *)c->db_perm.p, c->db_base,
                                                                     (const SimQuery *)c->sim_q.p, method, scores);
        } else {
            // plain A/G/C/U records: one thread each; the rest (ambiguity codes) go through a worklist to the warp kernel
            RSD_OK_OR_RETURN(c->sim_work.ensure(sizeof(int) * (size_t)(n + 16)));
            int *wl_n = (int *)c->sim_work.p, *wl = wl_n + 4;
            RSD_CUDA(cudaMemsetAsync(wl_n, 0, sizeof(int), st));
            k_sim_tf_thread<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(dbw, dbs, dbl, n, c->db_bits, (const int64_t *)c->db_perm.p, c->db_base,
                                                                         (const SimQuery *)c->sim_q.p, method, scores, wl, wl_n);
            const unsigned grid = (unsigned)std::min<int64_t>((n + 3) / 4, (int64_t)c->sm_count * 16);
            k_sim_tf<<<grid, 128, 0, st>>>(dbw, dbs, dbl, n, c->db_bits, (const int64_t *)c->db_perm.p, c->db_base,
                                           (const SimQuery *)c->sim_q.p, method, scores, wl, wl_n);
            c->launches += 1;
        }
        c->launches += 1;
    }
    if (k > 0) {
        const int64_t CH0 = 4096, cap = std::min<int64_t>(std::max<int64_t>(n, 1), (int64_t)1 << 20);
        RSD_OK_OR_RETURN(c->sim_aux.ensure((size_t)cap * 16 + (size_t)k * 16 + 256));
        unsigned char *aux = (unsigned char *)c->sim_aux.p;
        TopkState tk{};
        tk.k = k; tk.cap = cap;
        tk.cand_s = (double *)aux; aux += (size_t)cap * 8;
        tk.cand_i = (int64_t *)aux; aux += (size_t)cap * 8;
        tk.best_s = (double *)aux; aux += (size_t)k * 8;
        tk.best_i = (int64_t *)aux; aux += (size_t)k * 8;
        tk.tau_s = (double *)aux; aux += 8;
        tk.tau_i = (int64_t *)aux; aux += 8;
        tk.cand_n = (int *)aux;
        k_topk_init<<<1, 64, 0, st>>>(tk, 1);
        c->launches += 1;
        for (int64_t r0 = 0; r0 < n;) {
            const int64_t nr = std::min<int64_t>(r0 == 0 ? std::min(CH0, cap) : cap, n - r0);
            k_sim_filter<<<(unsigned)((nr + 255) / 256), 256, 0, st>>>(scores, r0, nr, c->db_base, tk);
            k_topk_fold<<<1, 256, 0, st>>>(tk);
            c->launches += 2;
            r0 += nr;
        }
        RSD_CUDA(cudaMemcpyAsync(top_idx, tk.best_i, sizeof(int64_t) * (size_t)k, cudaMemcpyDeviceToHost, st));
        RSD_CUDA(cudaMemcpyAsync(top_score, tk.best_s, sizeof(double) * (size_t)k, cudaMemcpyDeviceToHost, st));
    }
    if (c->timing) { RSD_CUDA(cudaEventRecord(c->ev1, st)); c->timed = true; }
    if (all_scores && n > 0) RSD_CUDA(cudaMemcpyAsync(all_scores, scores, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost, st));
    RSD_CUDA(cudaGetLastError());
    RSD_CUDA(cudaStreamSynchronize(st));
    return RSD_OK;
}

// the host-side checks of a similarity query batch (every entry point, before any device work)
static int sim_batch_args(const char *fn, const uint8_t *q_codes, const int64_t *q_off, int64_t n_queries, int method, int k,
                          const int64_t *top_idx, const double *top_score) {
    if (method < 0 || method >= RSD_SIM_COUNT) return rsd_fail(RSD_EINVAL, "%s: unknown method %d", fn, method);
    if (k < 0 || k > RSD_TOPK_MAX) return rsd_fail(RSD_EINVAL, "%s: k must be in 0..%d", fn, RSD_TOPK_MAX);
    if (n_queries < 0 || (n_queries > 0 && !q_off)) return rsd_fail(RSD_EINVAL, "%s: bad query", fn);
    if (n_queries == 0) return RSD_OK;
    if (k > 0 && (!top_idx || !top_score)) return rsd_fail(RSD_EINVAL, "%s: NULL top-k output", fn);
    if (q_off[0] != 0) return rsd_fail(RSD_EINVAL, "%s: q_off[0] must be 0", fn);
    for (int64_t q = 0; q < n_queries; ++q) {
        const int64_t len = q_off[q + 1] - q_off[q];
        if (len < 0 || len > INT32_MAX) return rsd_fail(RSD_EINVAL, "%s: bad query offsets at query %lld", fn, (long long)q);
    }
    if (q_off[n_queries] > 0 && !q_codes) return rsd_fail(RSD_EINVAL, "%s: bad query", fn);
    for (int64_t i = 0; i < q_off[n_queries]; ++i)
        if (q_codes[i] >= 15) return rsd_fail(RSD_EINVAL, "%s: query code %u at %lld is not a symbol", fn, q_codes[i], (long long)i);
    return RSD_OK;
}

// Queries q_codes[q_off[q] .. q_off[q+1]) (host) up to the context's sim_codes / sim_off.
static int sim_upload_queries(rsd_ctx *c, const uint8_t *q_codes, const int64_t *q_off, int64_t n_queries) {
    const int64_t total = q_off[n_queries];
    RSD_OK_OR_RETURN(c->sim_codes.ensure((size_t)total + 16));
    RSD_OK_OR_RETURN(c->sim_off.ensure(sizeof(int64_t) * (size_t)(n_queries + 1)));
    if (total) RSD_CUDA(cudaMemcpyAsync(c->sim_codes.p, q_codes, (size_t)total, cudaMemcpyHostToDevice, c->stream));
    RSD_CUDA(cudaMemcpyAsync(c->sim_off.p, q_off, sizeof(int64_t) * (size_t)(n_queries + 1), cudaMemcpyHostToDevice, c->stream));
    return RSD_OK;
}

// The similarity of n_queries queries (on the device: sim_codes / sim_off) against the loaded shard, in query batches of
// QB: each batch is one pass over the records into scores [QB][db_n], then the top-k of each query with the chunk
// sequence of rsd_db_similarity (a 4096-record seed chunk, then chunks of min(db_n, 2^20)).  Outputs: top_idx_dev /
// top_score_dev [n_queries][k] on the device (k > 0); all_scores (host, may be NULL): query q's db_n scores at
// all_scores + q * all_stride + all_col.  Timed (rsd_set_timing) from the first kernel to the last copy.  vt: the
// vector type (RSD_VEC_TF, or RSD_VEC_IDF / RSD_VEC_TFIDF with the context's idf table uploaded, idf_upload).
static int sim_batch_dev(rsd_ctx *c, int vt, int64_t n_queries, int method, int k, int64_t *top_idx_dev, double *top_score_dev,
                         double *all_scores, int64_t all_stride, int64_t all_col) {
    cudaStream_t st = c->stream;
    const int64_t n = c->db_n;
    const int64_t CH0 = 4096, cap = std::min<int64_t>(std::max<int64_t>(n, 1), (int64_t)1 << 20);
    // QB: at most RSD_SIM_QB queries, and what half of the free device memory holds (the buffers this call reuses count
    // as free); RSD_SIM_QBATCH lowers it
    const size_t per_q = sizeof(double) * (size_t)std::max<int64_t>(n, 1) + sizeof(SimQuery) + 64
                       + (k > 0 ? (size_t)cap * 16 + (size_t)k * 16 : 0);
    size_t free_b = 0, total_b = 0;
    RSD_CUDA(cudaMemGetInfo(&free_b, &total_b));
    const size_t room = free_b / 2 + c->sim_scores.cap + c->sim_aux.cap + c->sim_q.cap;
    int64_t qb = std::min<int64_t>({n_queries, (int64_t)RSD_SIM_QB, (int64_t)(room / per_q)});
    if (const char *e = getenv("RSD_SIM_QBATCH")) qb = std::min<int64_t>(qb, atoi(e));
    qb = std::max<int64_t>(qb, 1);
    RSD_OK_OR_RETURN(c->sim_q.ensure(sizeof(SimQuery) * (size_t)qb));
    RSD_OK_OR_RETURN(c->sim_scores.ensure(sizeof(double) * (size_t)qb * (size_t)std::max<int64_t>(n, 1)));
    RSD_OK_OR_RETURN(c->sim_work.ensure(sizeof(int) * (size_t)(n + 16)));
    TopkState tk{};
    if (k > 0) {
        RSD_OK_OR_RETURN(c->sim_aux.ensure((size_t)qb * ((size_t)cap * 16 + (size_t)k * 16 + 24) + 256));
        unsigned char *aux = (unsigned char *)c->sim_aux.p;
        tk.k = k; tk.cap = cap;
        tk.cand_s = (double *)aux; aux += (size_t)qb * cap * 8;
        tk.cand_i = (int64_t *)aux; aux += (size_t)qb * cap * 8;
        tk.best_s = (double *)aux; aux += (size_t)qb * k * 8;
        tk.best_i = (int64_t *)aux; aux += (size_t)qb * k * 8;
        tk.tau_s = (double *)aux; aux += (size_t)qb * 8;
        tk.tau_i = (int64_t *)aux; aux += (size_t)qb * 8;
        tk.cand_n = (int *)aux;
    }
    const uint32_t *dbw = (const uint32_t *)c->db.words.p; const int64_t *dbs = (const int64_t *)c->db.start.p; const int32_t *dbl = (const int32_t *)c->db.len.p;
    const int64_t *perm = (const int64_t *)c->db_perm.p;
    const uint8_t *codes = (const uint8_t *)c->sim_codes.p;
    const int64_t *off = (const int64_t *)c->sim_off.p;
    SimQuery *simq = (SimQuery *)c->sim_q.p;
    double *scores = (double *)c->sim_scores.p;
    int *wl_n = (int *)c->sim_work.p, *wl = wl_n + 4;
    const double *idf = vt == RSD_VEC_TF ? nullptr : (const double *)c->idf_dev.p;
    const int a_nonneg = c->idf_nonneg;
    auto k_query = vt == RSD_VEC_IDF ? k_sim_query_batch<RSD_VEC_IDF> : vt == RSD_VEC_TFIDF ? k_sim_query_batch<RSD_VEC_TFIDF> : k_sim_query_batch<RSD_VEC_TF>;
    auto k_thread = vt == RSD_VEC_IDF ? k_sim_tf_thread_batch<RSD_VEC_IDF> : vt == RSD_VEC_TFIDF ? k_sim_tf_thread_batch<RSD_VEC_TFIDF>
                                                                                                 : k_sim_tf_thread_batch<RSD_VEC_TF>;
    auto k_warp = vt == RSD_VEC_IDF ? k_sim_tf_batch<RSD_VEC_IDF> : vt == RSD_VEC_TFIDF ? k_sim_tf_batch<RSD_VEC_TFIDF> : k_sim_tf_batch<RSD_VEC_TF>;
    if (c->timing) RSD_CUDA(cudaEventRecord(c->ev0, st));
    for (int64_t q0 = 0; q0 < n_queries; q0 += qb) {
        const int nq = (int)std::min<int64_t>(qb, n_queries - q0);
        k_query<<<nq, 32, 0, st>>>(codes, off + q0, simq, idf);
        c->launches += 1;
        if (n > 0) {
            if (method < RSD_SIM_COSINE) {
                k_sim_small_batch<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(dbw, dbs, dbl, n, c->db_bits, perm, c->db_base, simq, nq, method, scores, n);
                c->launches += 1;
            } else {
                // plain A/G/C/U records: one thread each; the rest (ambiguity codes, > 60000 symbols) through the worklist
                RSD_CUDA(cudaMemsetAsync(wl_n, 0, sizeof(int), st));
                k_thread<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(dbw, dbs, dbl, n, c->db_bits, perm, c->db_base, simq, nq, method,
                                                                  scores, n, wl, wl_n, idf, a_nonneg);
                const unsigned grid = (unsigned)std::min<int64_t>((n + 3) / 4, (int64_t)c->sm_count * 16);
                k_warp<<<grid, 128, 0, st>>>(dbw, dbs, dbl, c->db_bits, perm, c->db_base, simq, nq, method, scores, n, wl, wl_n, idf);
                c->launches += 2;
            }
        }
        if (k > 0) {
            k_topk_init<<<(nq + 63) / 64, 64, 0, st>>>(tk, nq);
            c->launches += 1;
            for (int64_t r0 = 0; r0 < n;) {
                const int64_t nr = std::min<int64_t>(r0 == 0 ? std::min(CH0, cap) : cap, n - r0);
                k_sim_filter_batch<<<dim3((unsigned)((nr + 255) / 256), (unsigned)nq), 256, 0, st>>>(scores, n, r0, nr, c->db_base, tk);
                k_topk_fold<<<nq, 256, 0, st>>>(tk);
                c->launches += 2;
                r0 += nr;
            }
            RSD_CUDA(cudaMemcpyAsync(top_idx_dev + q0 * k, tk.best_i, sizeof(int64_t) * (size_t)nq * k, cudaMemcpyDeviceToDevice, st));
            RSD_CUDA(cudaMemcpyAsync(top_score_dev + q0 * k, tk.best_s, sizeof(double) * (size_t)nq * k, cudaMemcpyDeviceToDevice, st));
        }
        RSD_CUDA(cudaGetLastError());
        if (all_scores && n > 0) {
            // a [nq][n] block: contiguous in the caller's [Q][n] rows, or placed at column all_col of wider rows (a shard)
            if (all_stride == n) RSD_CUDA(cudaMemcpyAsync(all_scores + q0 * n + all_col, scores, sizeof(double) * (size_t)nq * n, cudaMemcpyDeviceToHost, st));
            else RSD_CUDA(cudaMemcpy2DAsync(all_scores + q0 * all_stride + all_col, sizeof(double) * (size_t)all_stride, scores, sizeof(double) * (size_t)n,
                                            sizeof(double) * (size_t)n, (size_t)nq, cudaMemcpyDeviceToHost, st));
        }
    }
    if (c->timing) { RSD_CUDA(cudaEventRecord(c->ev1, st)); c->timed = true; }
    return RSD_OK;
}

// a query batch against the loaded database after its arguments were checked: queries up, sim_batch_dev, results down
static int sim_batch_host(rsd_ctx *c, int vt, const uint8_t *q_codes, const int64_t *q_off, int64_t n_queries, int method, int k,
                          int64_t *top_idx, double *top_score, double *all_scores) {
    cudaStream_t st = c->stream;
    c->timed = false; c->last_ms_override = 0.0;
    const size_t cells = (size_t)n_queries * (size_t)std::max(k, 1);
    RSD_OK_OR_RETURN(c->sim_top.ensure(sizeof(int64_t) * 2 * cells));
    int64_t *ti = (int64_t *)c->sim_top.p; double *ts = (double *)(ti + cells);
    RSD_OK_OR_RETURN(sim_upload_queries(c, q_codes, q_off, n_queries));
    RSD_OK_OR_RETURN(sim_batch_dev(c, vt, n_queries, method, k, ti, ts, all_scores, c->db_n, 0));
    if (k > 0) {
        RSD_CUDA(cudaMemcpyAsync(top_idx, ti, sizeof(int64_t) * (size_t)n_queries * k, cudaMemcpyDeviceToHost, st));
        RSD_CUDA(cudaMemcpyAsync(top_score, ts, sizeof(double) * (size_t)n_queries * k, cudaMemcpyDeviceToHost, st));
    }
    RSD_CUDA(cudaGetLastError());
    RSD_CUDA(cudaStreamSynchronize(st));
    return RSD_OK;
}

extern "C" int rsd_db_similarity_batch(rsd_ctx *c, const uint8_t *q_codes, const int64_t *q_off, int64_t n_queries,
                                       int method, int k, int64_t *top_idx, double *top_score, double *all_scores) {
    if (!c) return rsd_fail(RSD_EINVAL, "ctx is NULL");
    RSD_OK_OR_RETURN(sim_batch_args("rsd_db_similarity_batch", q_codes, q_off, n_queries, method, k, top_idx, top_score));
    RSD_OK_OR_RETURN(c->ensure_device());
    if (n_queries == 0) return RSD_OK;
    if (!c->db_loaded) return rsd_fail(RSD_EINVAL, "rsd_db_similarity_batch: no database loaded (rsd_db_load)");
    return sim_batch_host(c, RSD_VEC_TF, q_codes, q_off, n_queries, method, k, top_idx, top_score, all_scores);
}

// ------------------------------------------------------------------------------------------------
// idf / tf-idf vectors (IR:189-225, searched by IR:458-465)
// ------------------------------------------------------------------------------------------------
// possibilities(symbol) (IR:255-287): a base first with probability 1, then every ambiguity code that may stand for it
// (IR:20-46 order) with that code's weight; an ambiguity code: the bases it may stand for, each 1 / (their number),
// then the code itself with probability 1.
static int idf_possibilities(int s, int *sym, double *prob) {
    static const double W[15][4] = {
        {1, 0, 0, 0}, {0, 1, 0, 0}, {0, 0, 1, 0}, {0, 0, 0, 1},
        {0, 0, 0.5, 0.5}, {0.5, 0.5, 0, 0}, {0.5, 0, 0, 0.5}, {0, 0.5, 0.5, 0}, {0, 0.5, 0, 0.5}, {0.5, 0, 0.5, 0},
        {0.33, 0.33, 0, 0.33}, {0.33, 0.33, 0.33, 0}, {0.33, 0, 0.33, 0.33}, {0, 0.33, 0.33, 0.33}, {0.25, 0.25, 0.25, 0.25}};
    int n = 0;
    if (s < 4) {
        sym[n] = s; prob[n++] = 1.0;
        for (int x = 4; x < 15; ++x) if (W[x][s] != 0) { sym[n] = x; prob[n++] = W[x][s]; }
        return n;
    }
    for (int b = 0; b < 4; ++b) if (W[s][b] != 0) sym[n++] = b;
    for (int i = 0; i < n; ++i) prob[i] = 1.0 / (double)n;
    sym[n] = s; prob[n++] = 1.0;
    return n;
}

// the expansions of every pair (IdfExp, k_sim.cuh), built once per process
static const IdfExp &idf_expansions() {
    static const IdfExp X = [] {
        IdfExp x{};
        for (int p = 0; p < RSD_TF; ++p) {
            int sa[8], sb[8]; double pa[8], pb[8];
            const int na = idf_possibilities(p / 15, sa, pa), nb = idf_possibilities(p % 15, sb, pb);
            std::vector<std::pair<double, int>> ex;
            for (int i = 0; i < na; ++i) for (int j = 0; j < nb; ++j) ex.push_back({pa[i] * pb[j], sa[i] * 15 + sb[j]});
            std::stable_sort(ex.begin(), ex.end(), [](const std::pair<double, int> &u, const std::pair<double, int> &v) { return u.first > v.first; });
            x.n[p] = (int)ex.size();
            for (size_t m = 0; m < ex.size(); ++m) { x.w[p][m] = ex[m].first; x.e[p][m] = (uint8_t)ex[m].second; }
        }
        return x;
    }();
    return X;
}

// Continues the 225 df sums (host df, in and out) over the records [first, db_n) of the shard loaded in c (shard-local
// collection indices), in collection order.
static int idf_df_shard(rsd_ctx *c, double *df, int64_t first = 0) {
    cudaStream_t st = c->stream;
    const int64_t n = c->db_n;
    RSD_OK_OR_RETURN(c->idf_dev.ensure(sizeof(double) * 2 * RSD_TF));
    double *d_df = (double *)c->idf_dev.p + RSD_TF;
    RSD_CUDA(cudaMemcpyAsync(d_df, df, sizeof(double) * RSD_TF, cudaMemcpyHostToDevice, st));
    if (n > first) {
        RSD_OK_OR_RETURN(c->idf_exp.ensure(sizeof(IdfExp)));
        RSD_CUDA(cudaMemcpyAsync(c->idf_exp.p, &idf_expansions(), sizeof(IdfExp), cudaMemcpyHostToDevice, st));
        // chunks of 2^20 records: the presence sets take 32 bytes per record of the chunk
        const int64_t CH = std::min<int64_t>(n - first, (int64_t)1 << 20);
        RSD_OK_OR_RETURN(c->idf_work.ensure(32 * (size_t)CH + sizeof(int64_t) * (size_t)n));
        uint32_t *pres = (uint32_t *)c->idf_work.p;            // first: the kernels access it as 16-byte uint4
        int64_t *inv = (int64_t *)(pres + 8 * CH);
        const uint32_t *dbw = (const uint32_t *)c->db.words.p; const int64_t *dbs = (const int64_t *)c->db.start.p; const int32_t *dbl = (const int32_t *)c->db.len.p;
        k_idf_inv<<<(unsigned)((n + 255) / 256), 256, 0, st>>>((const int64_t *)c->db_perm.p, c->db_base, n, inv);
        c->launches += 1;
        for (int64_t i0 = first; i0 < n; i0 += CH) {
            const int64_t nn = std::min(CH, n - i0);
            k_idf_pres<<<(unsigned)((nn + 255) / 256), 256, 0, st>>>(dbw, dbs, dbl, c->db_bits, inv, i0, nn, pres);
            k_idf_chain<<<15, 32 + RSD_IDF_T, 0, st>>>(pres, nn, (const IdfExp *)c->idf_exp.p, d_df);
            c->launches += 2;
        }
    }
    RSD_CUDA(cudaGetLastError());
    RSD_CUDA(cudaMemcpyAsync(df, d_df, sizeof(double) * RSD_TF, cudaMemcpyDeviceToHost, st));
    RSD_CUDA(cudaStreamSynchronize(st));
    return RSD_OK;
}

// IR:213-214: idf[p] = 0 if df[p] == 0 else math.log(N / df[p], 10), which CPython evaluates as log(N / df) / log(10.0)
// with the C library's log -- computed here on the host for that reason (the device log rounds differently).  Returns
// whether every entry is finite and >= +0 (always, as df[p] <= N; k_sim_tf_thread_batch relies on it when it holds).
static bool idf_from_df(const double *df, int64_t N, double *idf) {
    volatile double ten = 10.0;                    // evaluated at run time like CPython's, not folded by the compiler
    const double l10 = std::log((double)ten);
    bool nonneg = true;
    for (int p = 0; p < RSD_TF; ++p) {
        idf[p] = df[p] == 0 ? 0.0 : std::log((double)N / df[p]) / l10;
        nonneg = nonneg && std::isfinite(idf[p]) && !std::signbit(idf[p]);
    }
    return nonneg;
}

// the table to the device (idf_dev[0..225)) and the context's host copies
static int idf_upload(rsd_ctx *c, const double *df, const double *idf, bool nonneg) {
    RSD_OK_OR_RETURN(c->ensure_device());
    RSD_OK_OR_RETURN(c->idf_dev.ensure(sizeof(double) * 2 * RSD_TF));
    RSD_CUDA(cudaMemcpyAsync(c->idf_dev.p, idf, sizeof(double) * RSD_TF, cudaMemcpyHostToDevice, c->stream));
    RSD_CUDA(cudaStreamSynchronize(c->stream));
    memcpy(c->idf_df, df, sizeof c->idf_df); memcpy(c->idf_tab, idf, sizeof c->idf_tab);
    c->idf_nonneg = nonneg;
    return RSD_OK;
}

// the loaded database's table, built when the context does not hold it yet (timed on its own: rsd_set_timing)
static int idf_ensure(rsd_ctx *c, const char *fn) {
    if (!c->db_loaded) return rsd_fail(RSD_EINVAL, "%s: no database loaded (rsd_db_load)", fn);
    if (c->db_base != 0)
        return rsd_fail(RSD_EINVAL, "%s: the database was loaded with global_index_base %lld: a shard cannot know the collection's "
                        "document frequencies (rsd_multi holds every shard)", fn, (long long)c->db_base);
    if (c->idf_ready) return RSD_OK;
    c->timed = false; c->last_ms_override = 0.0;
    if (c->timing) RSD_CUDA(cudaEventRecord(c->ev0, c->stream));
    double df[RSD_TF] = {}, idf[RSD_TF];
    RSD_OK_OR_RETURN(idf_df_shard(c, df));
    if (c->timing) { RSD_CUDA(cudaEventRecord(c->ev1, c->stream)); RSD_CUDA(cudaEventSynchronize(c->ev1)); c->timed = true; }
    RSD_OK_OR_RETURN(idf_upload(c, df, idf, idf_from_df(df, c->db_n, idf)));
    c->idf_ready = true;
    return RSD_OK;
}

extern "C" int rsd_db_idf_table(rsd_ctx *c, double *df, double *idf) {
    if (!c) return rsd_fail(RSD_EINVAL, "ctx is NULL");
    RSD_OK_OR_RETURN(c->ensure_device());
    RSD_OK_OR_RETURN(idf_ensure(c, "rsd_db_idf_table"));
    if (df) memcpy(df, c->idf_df, sizeof c->idf_df);
    if (idf) memcpy(idf, c->idf_tab, sizeof c->idf_tab);
    return RSD_OK;
}

// the host-side checks of a vector-type batch, in front of sim_batch_args
static int vec_batch_args(const char *fn, int vector_type, int method) {
    if (vector_type != RSD_VEC_IDF && vector_type != RSD_VEC_TFIDF) return rsd_fail(RSD_EINVAL, "%s: unknown vector type %d", fn, vector_type);
    if (method < RSD_SIM_COSINE || method > RSD_SIM_DICE)
        return rsd_fail(RSD_EINVAL, "%s: method %d is not a vector measure (RSD_SIM_COSINE..RSD_SIM_DICE)", fn, method);
    return RSD_OK;
}

extern "C" int rsd_db_vector_similarity_batch(rsd_ctx *c, const uint8_t *q_codes, const int64_t *q_off, int64_t n_queries,
                                              int vector_type, int method, int k, int64_t *top_idx, double *top_score, double *all_scores) {
    const char *fn = "rsd_db_vector_similarity_batch";
    if (!c) return rsd_fail(RSD_EINVAL, "ctx is NULL");
    RSD_OK_OR_RETURN(vec_batch_args(fn, vector_type, method));
    RSD_OK_OR_RETURN(sim_batch_args(fn, q_codes, q_off, n_queries, method, k, top_idx, top_score));
    RSD_OK_OR_RETURN(c->ensure_device());
    if (!c->db_loaded) return rsd_fail(RSD_EINVAL, "%s: no database loaded (rsd_db_load)", fn);
    if (n_queries == 0) return RSD_OK;
    RSD_OK_OR_RETURN(idf_ensure(c, fn));
    return sim_batch_host(c, vector_type, q_codes, q_off, n_queries, method, k, top_idx, top_score, all_scores);
}

// ------------------------------------------------------------------------------------------------
// appending records to the loaded database
// ------------------------------------------------------------------------------------------------
// The buffers of one device rebuild: scratch, and the new store, which is swapped into the context when it is complete.
// Whatever the context does not take (the scratch, or the new store after a failure) is freed on the way out.
struct LayBufs {
    DevBuf inv, mask, lenc, keys, vals, nw, tmp, cnt, perm;
    SeqBufs db;
    ~LayBufs() { DevBuf *all[] = {&inv, &mask, &lenc, &keys, &vals, &nw, &tmp, &cnt, &perm}; for (DevBuf *b : all) b->release(); db.release(); }
};

extern "C" int rsd_db_append(rsd_ctx *c, const uint32_t *words, const int64_t *start, const int32_t *len,
                             int64_t n_records, int64_t n_words, int bits, uint32_t symmask) {
    if (!c) return rsd_fail(RSD_EINVAL, "ctx is NULL");
    if (!c->db_loaded) return rsd_fail(RSD_EINVAL, "rsd_db_append: no database loaded (rsd_db_load)");
    if (n_records < 0 || n_words < 0 || (n_records > 0 && (!words || !start || !len))) return rsd_fail(RSD_EINVAL, "rsd_db_append: bad arguments");
    if (bits != c->db_bits) return rsd_fail(RSD_EINVAL, "rsd_db_append: %d-bit records for a %d-bit database (reload it to change the packing)", bits, c->db_bits);
    if (bits == 2 && (symmask & ~0xFu)) return rsd_fail(RSD_EINVAL, "rsd_db_append: 2-bit packing with symbols outside ACGU");
    const int per = 32 / bits;
    int32_t mx = 0;
    int64_t add_w = 0;
    for (int64_t i = 0; i < n_records; ++i) {
        if (len[i] < 0) return rsd_fail(RSD_EINVAL, "rsd_db_append: negative length");
        const int64_t nw = ((int64_t)len[i] + per - 1) / per;
        if (start[i] < 0 || start[i] + nw > n_words) return rsd_fail(RSD_EINVAL, "rsd_db_append: record %lld lies outside the word buffer", (long long)i);
        mx = std::max(mx, len[i]); add_w += nw;
    }
    if (n_records == 0) return RSD_OK;
    RSD_OK_OR_RETURN(c->ensure_device());
    cudaStream_t st = c->stream;
    const int64_t n_old = c->db_n, N = n_old + n_records, W = c->db_nwords + add_w;
    const int64_t maxlen = std::max<int64_t>(c->db_maxlen, mx);
    LayBufs b;
    RSD_OK_OR_RETURN(c->upload_seqs(c->bufA, words, start, len, n_records, n_words, st));         // the staging copy
    RSD_OK_OR_RETURN(b.inv.ensure(sizeof(int64_t) * (size_t)std::max<int64_t>(n_old, 1)));
    RSD_OK_OR_RETURN(b.mask.ensure(sizeof(uint16_t) * (size_t)N));
    RSD_OK_OR_RETURN(b.lenc.ensure(sizeof(int32_t) * (size_t)N));
    RSD_OK_OR_RETURN(b.keys.ensure(2 * sizeof(uint64_t) * (size_t)N));
    RSD_OK_OR_RETURN(b.vals.ensure(2 * sizeof(int64_t) * (size_t)N));
    RSD_OK_OR_RETURN(b.nw.ensure(sizeof(int64_t) * (size_t)N));
    RSD_OK_OR_RETURN(b.cnt.ensure(sizeof(unsigned long long) * 32));
    RSD_OK_OR_RETURN(b.perm.ensure(sizeof(int64_t) * (size_t)N));
    RSD_OK_OR_RETURN(b.db.words.ensure(sizeof(uint32_t) * (size_t)(std::max<int64_t>(W, 1) + 8)));
    RSD_OK_OR_RETURN(b.db.start.ensure(sizeof(int64_t) * (size_t)N));
    RSD_OK_OR_RETURN(b.db.len.ensure(sizeof(int32_t) * (size_t)N));
    const unsigned g1 = (unsigned)((N + 255) / 256);
    if (n_old > 0) {
        k_idf_inv<<<(unsigned)((n_old + 255) / 256), 256, 0, st>>>((const int64_t *)c->db_perm.p, c->db_base, n_old, (int64_t *)b.inv.p);
        c->launches += 1;
    }
    const LaySrc src{(const uint32_t *)c->db.words.p, (const int64_t *)c->db.start.p, (const int32_t *)c->db.len.p, (const int64_t *)b.inv.p, n_old,
                     (const uint32_t *)c->bufA.words.p, (const int64_t *)c->bufA.start.p, (const int32_t *)c->bufA.len.p};
    unsigned long long *d_cnt = (unsigned long long *)b.cnt.p, h_cnt[32];
    RSD_CUDA(cudaMemsetAsync(d_cnt, 0, sizeof(unsigned long long) * 32, st));
    k_lay_mask<<<g1, 256, 0, st>>>(src, N, bits, (uint16_t *)b.mask.p, (int32_t *)b.lenc.p, d_cnt);
    c->launches += 1;
    RSD_CUDA(cudaGetLastError());
    RSD_CUDA(cudaMemcpyAsync(h_cnt, d_cnt, sizeof(unsigned long long) * 16, cudaMemcpyDeviceToHost, st));
    RSD_CUDA(cudaStreamSynchronize(st));
    int64_t holds[16], tcnt[16];
    for (int s = 0; s < 16; ++s) holds[s] = (int64_t)h_cnt[s];
    int rank[16];
    tier_ranks(holds, rank);
    uint64_t rk = 0;
    for (int s = 0; s < 16; ++s) rk |= (uint64_t)rank[s] << (4 * s);
    k_lay_tier<<<g1, 256, 0, st>>>((const uint16_t *)b.mask.p, N, rk, d_cnt + 16);
    c->launches += 1;
    RSD_CUDA(cudaGetLastError());
    RSD_CUDA(cudaMemcpyAsync(h_cnt + 16, d_cnt + 16, sizeof(unsigned long long) * 16, cudaMemcpyDeviceToHost, st));
    RSD_CUDA(cudaStreamSynchronize(st));
    for (int t = 0; t < 16; ++t) tcnt[t] = (int64_t)h_cnt[16 + t];
    int64_t tier_end[16];
    uint32_t tier_mask[16];
    const int r0 = tier_cut(holds, tcnt, N, tier_end, tier_mask);
    // stable radix sort by (merged tier, length) over the records in collection order = rsd_db_load's (tier, length,
    // collection index) order
    const int lenbits = ceil_log2_i64(maxlen + 1);
    uint64_t *keys = (uint64_t *)b.keys.p;
    int64_t *vals = (int64_t *)b.vals.p;
    k_lay_key<<<g1, 256, 0, st>>>((const uint16_t *)b.mask.p, (const int32_t *)b.lenc.p, N, rk, r0, lenbits, keys, vals);
    c->launches += 1;
    RSD_CUDA(cudaGetLastError());
    cub::DoubleBuffer<uint64_t> kb(keys, keys + N);
    cub::DoubleBuffer<int64_t> vb(vals, vals + N);
    size_t tmp_sort = 0, tmp_scan = 0;
    int64_t *d_nw = (int64_t *)b.nw.p, *d_start = (int64_t *)b.db.start.p;
    RSD_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tmp_sort, kb, vb, N, 0, 4 + lenbits, st));
    RSD_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tmp_scan, d_nw, d_start, N, st));
    RSD_OK_OR_RETURN(b.tmp.ensure(std::max(tmp_sort, tmp_scan)));
    RSD_CUDA(cub::DeviceRadixSort::SortPairs(b.tmp.p, tmp_sort, kb, vb, N, 0, 4 + lenbits, st));
    const int64_t *idx = vb.Current();
    k_lay_order<<<g1, 256, 0, st>>>(idx, (const int32_t *)b.lenc.p, N, bits, c->db_base, (int32_t *)b.db.len.p, d_nw, (int64_t *)b.perm.p);
    c->launches += 1;
    RSD_CUDA(cudaGetLastError());
    RSD_CUDA(cub::DeviceScan::ExclusiveSum(b.tmp.p, tmp_scan, d_nw, d_start, N, st));
    k_lay_copy<<<(unsigned)((N + 7) / 8), 256, 0, st>>>(src, idx, d_start, N, bits, (uint32_t *)b.db.words.p);
    c->launches += 1;
    RSD_CUDA(cudaGetLastError());
    RSD_CUDA(cudaMemsetAsync((uint32_t *)b.db.words.p + W, 0, sizeof(uint32_t) * (size_t)(std::max<int64_t>(W, 1) - W + 8), st));
    RSD_CUDA(cudaStreamSynchronize(st));
    // the new layout is complete: swap it in (the old store goes with b)
    std::swap(c->db, b.db);
    std::swap(c->db_perm, b.perm);
    c->db_n = N; c->db_nwords = W; c->db_maxlen = maxlen; c->db_symmask |= symmask;
    memcpy(c->db_tier_end, tier_end, sizeof tier_end); memcpy(c->db_tier_mask, tier_mask, sizeof tier_mask);
    // The df sums are chains in collection order: the appended records continue them.  A failure here leaves the
    // appended database standing and the table to be rebuilt on next use.
    if (c->idf_ready) {
        double df[RSD_TF], idf[RSD_TF];
        memcpy(df, c->idf_df, sizeof df);
        int rc = idf_df_shard(c, df, n_old);
        if (rc == RSD_OK) rc = idf_upload(c, df, idf, idf_from_df(df, N, idf));
        if (rc != RSD_OK) c->idf_ready = false;
    }
    return RSD_OK;
}

extern "C" int rsd_db_layout(rsd_ctx *c, int64_t *n_records, int64_t *perm, int64_t *tier_end, uint32_t *tier_mask) {
    if (!c || !n_records) return rsd_fail(RSD_EINVAL, "rsd_db_layout: bad arguments");
    if (!c->db_loaded) return rsd_fail(RSD_EINVAL, "rsd_db_layout: no database loaded (rsd_db_load)");
    *n_records = c->db_n;
    if (tier_end) memcpy(tier_end, c->db_tier_end, sizeof c->db_tier_end);
    if (tier_mask) memcpy(tier_mask, c->db_tier_mask, sizeof c->db_tier_mask);
    if (perm && c->db_n > 0) {
        RSD_OK_OR_RETURN(c->ensure_device());
        RSD_CUDA(cudaMemcpyAsync(perm, c->db_perm.p, sizeof(int64_t) * (size_t)c->db_n, cudaMemcpyDeviceToHost, c->stream));
        RSD_CUDA(cudaStreamSynchronize(c->stream));
    }
    return RSD_OK;
}

// ------------------------------------------------------------------------------------------------
// long pair (BASELINE config 4)
// ------------------------------------------------------------------------------------------------
// Pairs whose keys do not fit the 32-bit keys of k_long2 (costs too large for that bound, or not dyadic) run on
// k_long_fwd, one pair per launch with the whole direction matrix resident.  Called by rsd_long_pairs for one non-empty
// pair whose arguments and symbols (symmask) it has checked.
static int long_pair_wide(rsd_ctx *c, const uint8_t *a, int64_t m, const uint8_t *b, int64_t n, uint32_t symmask, int force_mode,
                          int want_script, uint8_t *op, int32_t *oi, int32_t *oj, int64_t *n_ops, double *dist, int *mode_out) {
    ModeInfo mi;
    RSD_OK_OR_RETURN(c->classify(symmask, m, n, 4, force_mode == RSD_MODE_I16X2 ? RSD_MODE_I32 : force_mode, mi));
    // integer keys (cost * 2^S + steps) are carried in doubles: they must stay below 2^52
    int S = ceil_log2_i64(m + n + 66);
    if (const char *e = getenv("RSD_LONG_S")) S = std::min(std::max(S, atoi(e)), 30);
    bool f64 = mi.mode == RSD_MODE_F64;
    if (!f64) {
        const double bound = ((double)m * mi.ic.del + (double)(n + 512) * mi.ic.ins + 4.0 * ((double)mi.ic.ins + mi.ic.del)) * std::ldexp(1.0, S);
        if (bound > 4.0e15) { if (force_mode == RSD_MODE_I32) return rsd_fail(RSD_ERANGE, "rsd_long_pair: int64 key would overflow"); f64 = true; }
    } else if (force_mode == RSD_MODE_I32) return rsd_fail(RSD_EINVAL, "rsd_long_pair: integer mode not exact for these costs");
    if (mode_out) *mode_out = f64 ? RSD_MODE_F64 : RSD_MODE_I32;
    c->timed = false; c->last_ms_override = 0.0;
    cudaStream_t st = c->stream;
    RSD_OK_OR_RETURN(c->upload_costs(mi, st));
    int C = 4;                                  // columns per lane
    if (const char *e = getenv("RSD_LONG_C")) { const int v = atoi(e); if (v == 4 || v == 8 || v == 16) C = v; }
    const int n_panels = (int)((n + 32 * C - 1) / (32 * C));
    const int64_t n_pad = (int64_t)n_panels * 32 * C;
    int per_sm = 0;
    const void *kfn = f64 ? (C == 4 ? (const void *)k_long_fwd<true, 4> : C == 16 ? (const void *)k_long_fwd<true, 16> : (const void *)k_long_fwd<true, 8>)
                          : (C == 4 ? (const void *)k_long_fwd<false, 4> : C == 16 ? (const void *)k_long_fwd<false, 16> : (const void *)k_long_fwd<false, 8>);
    RSD_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kfn, 32, 0));
    if ((int64_t)per_sm * c->sm_count < n_panels)
        return rsd_fail(RSD_ERANGE, "rsd_long_pair: %d column panels exceed the %d co-resident CTAs of this GPU (n too large for one wavefront launch)",
                        n_panels, per_sm * c->sm_count);
    const size_t dir_words = (size_t)((m + 15) / 16) * (size_t)n_pad;
    RSD_OK_OR_RETURN(c->dirs.ensure(dir_words * 4 + 64));
    DevBuf &scratch = c->slots[0].scratch;
    RSD_OK_OR_RETURN(scratch.ensure((size_t)n_panels * (size_t)m * 12 + 256));
    RSD_OK_OR_RETURN(c->mat_ab.ensure((size_t)m + n + 64));
    RSD_OK_OR_RETURN(c->out_f64.ensure(64));
    uint8_t *da = (uint8_t *)c->mat_ab.p, *db = da + ((m + 15) / 16) * 16;
    RSD_CUDA(cudaMemcpyAsync(da, a, (size_t)m, cudaMemcpyHostToDevice, st));
    RSD_CUDA(cudaMemcpyAsync(db, b, (size_t)n, cudaMemcpyHostToDevice, st));
    LongArgs la{};
    la.a = da; la.m = (int)m; la.b = db; la.n = (int)n; la.n_panels = n_panels; la.n_pad = (int)n_pad;
    la.dirs = (uint32_t *)c->dirs.p;
    la.bound = scratch.p;
    la.bound_steps = (int *)((unsigned char *)scratch.p + (size_t)n_panels * (size_t)m * 8);
    la.dist = (double *)c->out_f64.p;
    la.S = S;
    RSD_CUDA(cudaMemsetAsync(la.bound, 0x80, (size_t)n_panels * (size_t)m * 8, st));      // sentinel = "not published yet"
    if (want_script) {
        RSD_OK_OR_RETURN(c->s_tmp.ensure((size_t)(m + n) + 64));
        RSD_OK_OR_RETURN(c->s_nops.ensure(64));
        RSD_OK_OR_RETURN(c->s_op.ensure((size_t)(m + n) + 64));
        if (oi) RSD_OK_OR_RETURN(c->s_oi.ensure(sizeof(int32_t) * (size_t)(m + n) + 64));
        if (oj) RSD_OK_OR_RETURN(c->s_oj.ensure(sizeof(int32_t) * (size_t)(m + n) + 64));
        RSD_OK_OR_RETURN(c->long_jobs.ensure(sizeof(LongEmit2)));
        const LongEmit2 em{(const uint8_t *)c->s_tmp.p, (int)m, (int)n, (const int32_t *)c->s_nops.p, (uint8_t *)c->s_op.p,
                           oi ? (int32_t *)c->s_oi.p : nullptr, oj ? (int32_t *)c->s_oj.p : nullptr};
        RSD_CUDA(cudaMemcpyAsync(c->long_jobs.p, &em, sizeof em, cudaMemcpyHostToDevice, st));
    }
    const IntCosts *dic = c->d_ic; const F64Costs *dfc = c->d_fc;
    void *args[] = {&la, &dic, &dfc};
    if (c->timing) RSD_CUDA(cudaEventRecord(c->ev0, st));
    RSD_CUDA(cudaLaunchCooperativeKernel(kfn, dim3(n_panels), dim3(32), args, 0, st));
    c->launches += 1;
    if (want_script) {
        k_long_traceback<<<1, 32, 0, st>>>((int)m, (int)n, (const uint32_t *)c->dirs.p, (int)n_pad, (uint8_t *)c->s_tmp.p, (int32_t *)c->s_nops.p);
        k_long2_emit<<<1, 1024, 0, st>>>((const LongEmit2 *)c->long_jobs.p);
        c->launches += 2;
    }
    if (c->timing) { RSD_CUDA(cudaEventRecord(c->ev1, st)); c->timed = true; }
    RSD_CUDA(cudaGetLastError());
    RSD_CUDA(cudaMemcpyAsync(dist, c->out_f64.p, sizeof(double), cudaMemcpyDeviceToHost, st));
    if (want_script) {
        int32_t k32 = 0;
        RSD_CUDA(cudaMemcpyAsync(&k32, c->s_nops.p, sizeof(int32_t), cudaMemcpyDeviceToHost, st));
        RSD_CUDA(cudaStreamSynchronize(st));
        *n_ops = k32;
        RSD_CUDA(cudaMemcpyAsync(op, c->s_op.p, (size_t)k32, cudaMemcpyDeviceToHost, st));
        if (oi) RSD_CUDA(cudaMemcpyAsync(oi, c->s_oi.p, sizeof(int32_t) * (size_t)k32, cudaMemcpyDeviceToHost, st));
        if (oj) RSD_CUDA(cudaMemcpyAsync(oj, c->s_oj.p, sizeof(int32_t) * (size_t)k32, cudaMemcpyDeviceToHost, st));
    }
    RSD_CUDA(cudaStreamSynchronize(st));
    return RSD_OK;
}

// ------------------------------------------------------------------------------------------------
// several GPUs, one process: sharded database search with an NCCL gather
// ------------------------------------------------------------------------------------------------
#include "rsd_long.inl"
#include "rsd_multi.inl"
