// k_layout.cuh — the stored order of the resident database rebuilt on the device (rsd_db_append).
//
// The database is stored sorted by (merged tier, length, collection index) (rsd_db_load).  After an append the order of
// the concatenation (the loaded records, then the batch) is rebuilt here: the loaded records are read in place through
// the inverse of db_perm (k_idf_inv), the batch from a staging copy, so no loaded record crosses PCIe again.
//   k_lay_mask   one thread per record, collection order: symbol mask and length; the 16 "records holding symbol b" counts
//   k_lay_tier   the histogram of the unmerged tiers (rank of the record's rarest symbol), ranks from the host
//   k_lay_key    the sort key (merged tier, length) and the collection index, for a stable radix sort
//   k_lay_order  per stored record of the new order: length, word count (scanned into start), global index
//   k_lay_copy   one warp per stored record: its words from the old store or the staging copy, coalesced

// The records of the concatenation in collection order: i < n_old is stored record inv[i] of the loaded store, the
// others are record i - n_old of the staged batch.
struct LaySrc {
    const uint32_t *ow; const int64_t *os; const int32_t *ol; const int64_t *inv; int64_t n_old;
    const uint32_t *nw; const int64_t *ns; const int32_t *nl;
};

__device__ __forceinline__ void lay_rec(const LaySrc &s, int64_t i, const uint32_t *&w, int64_t &st, int32_t &len) {
    if (i < s.n_old) { const int64_t r = s.inv[i]; w = s.ow; st = s.os[r]; len = s.ol[r]; }
    else { const int64_t j = i - s.n_old; w = s.nw; st = s.ns[j]; len = s.nl[j]; }
}

// rank of the rarest symbol of mask m; rk holds the 16 ranks, 4 bits each
__device__ __forceinline__ int lay_tier(uint32_t m, uint64_t rk) {
    int t = 0;
    for (; m; m &= m - 1) t = max(t, (int)((rk >> (4 * (__ffs(m) - 1))) & 15u));
    return t;
}

__global__ void __launch_bounds__(256)
k_lay_mask(LaySrc s, int64_t n, int bits, uint16_t *__restrict__ mask, int32_t *__restrict__ lenc, unsigned long long *__restrict__ holds) {
    __shared__ unsigned int s_h[16];
    if (threadIdx.x < 16) s_h[threadIdx.x] = 0;
    __syncthreads();
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t m = 0;
    if (i < n) {
        const uint32_t *w; int64_t st; int32_t len;
        lay_rec(s, i, w, st, len);
        const int per = 32 / bits;
        const uint32_t sym = (1u << bits) - 1u;
        for (int32_t j0 = 0; j0 < len; j0 += per) {
            const uint32_t x = w[st + j0 / per];
            const int cnt = min(per, len - j0);               // the padding of the last word is not a symbol
            for (int j = 0; j < cnt; ++j) m |= 1u << ((x >> (j * bits)) & sym);
        }
        mask[i] = (uint16_t)m; lenc[i] = len;
    }
    const int lane = threadIdx.x & 31;
#pragma unroll
    for (int b = 0; b < 16; ++b) {
        const int c = __popc(__ballot_sync(0xffffffffu, (m >> b) & 1u));
        if (lane == 0 && c) atomicAdd(&s_h[b], (unsigned)c);
    }
    __syncthreads();
    if (threadIdx.x < 16 && s_h[threadIdx.x]) atomicAdd(&holds[threadIdx.x], (unsigned long long)s_h[threadIdx.x]);
}

__global__ void __launch_bounds__(256)
k_lay_tier(const uint16_t *__restrict__ mask, int64_t n, uint64_t rk, unsigned long long *__restrict__ tcnt) {
    __shared__ unsigned int s_h[16];
    if (threadIdx.x < 16) s_h[threadIdx.x] = 0;
    __syncthreads();
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) atomicAdd(&s_h[lay_tier(mask[i], rk)], 1u);
    __syncthreads();
    if (threadIdx.x < 16 && s_h[threadIdx.x]) atomicAdd(&tcnt[threadIdx.x], (unsigned long long)s_h[threadIdx.x]);
}

__global__ void __launch_bounds__(256)
k_lay_key(const uint16_t *__restrict__ mask, const int32_t *__restrict__ lenc, int64_t n, uint64_t rk, int r0, int lenbits,
          uint64_t *__restrict__ key, int64_t *__restrict__ val) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    key[i] = ((uint64_t)max(0, lay_tier(mask[i], rk) - r0) << lenbits) | (uint64_t)lenc[i];
    val[i] = i;
}

// idx[r] = collection index of new stored record r -> its length, word count and global index
__global__ void __launch_bounds__(256)
k_lay_order(const int64_t *__restrict__ idx, const int32_t *__restrict__ lenc, int64_t n, int bits, int64_t global_base,
            int32_t *__restrict__ len, int64_t *__restrict__ nw, int64_t *__restrict__ perm) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n) return;
    const int64_t i = idx[r];
    const int32_t l = lenc[i];
    const int per = 32 / bits;
    len[r] = l; nw[r] = ((int64_t)l + per - 1) / per; perm[r] = global_base + i;
}

__global__ void __launch_bounds__(256)
k_lay_copy(LaySrc s, const int64_t *__restrict__ idx, const int64_t *__restrict__ start, int64_t n, int bits, uint32_t *__restrict__ out) {
    const int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (r >= n) return;
    const int lane = threadIdx.x & 31;
    const uint32_t *w; int64_t st; int32_t len;
    lay_rec(s, idx[r], w, st, len);
    const int per = 32 / bits;
    const int64_t nwr = ((int64_t)len + per - 1) / per, o = start[r];
    for (int64_t k = lane; k < nwr; k += 32) out[o + k] = w[st + k];
}
