// K6 - next-level generation with superset pruning, plus the ordered compaction / scan plumbing around it.
//
// Replaces generate_children_sets + CombinationTester.check
// (/root/reference/src/ppopt/mp_solvers/solver_utils.py:29-55,154-166, called from mpqp_combinatorial.py:60-61) and the
// mpLP cardinality filter (mpqp_combinatorial.py:40-42).  The reference tests every child against EVERY stored
// infeasible tuple (linear scan, the measured bottleneck at MPC N=10).  Here a child C = P + {i} of a feasible parent P
// survives iff every k-subset C \ {j}, j in P, is itself in this level's FEASIBLE list - equivalent to "no subset of C is
// in the murder list" by induction over levels (DESIGN.md, K6).  Those subsets share P's structure: C \ {j} is P \ {j}
// plus C's highest row, so one bitmap intersection per parent over a prefix-group index of the feasible list decides all
// of P's children at once (children_count_kernel).
// Children are written parent by parent in ascending i, i.e. in the reference's order.
#include "common.cuh"
#include "launch.h"

namespace ppgpu {

constexpr int SCAN_THREADS = 256;
constexpr int SCAN_ITEMS = 8;
constexpr int SCAN_CHUNK = SCAN_THREADS * SCAN_ITEMS;
constexpr int MAXW = 4;

// words of K6's group table (int32 slots, a power of two >= 2 x groups, >= 1024), which first hold nf + 1 scan words
static long long table_words(long long nf) { return 2 * nf + 2 > 512 ? 2 * nf + 2 : 512; }

__device__ __forceinline__ long long block_exclusive_scan(long long v, long long* total) {
    __shared__ long long wsum[SCAN_THREADS / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    long long x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const long long y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
    }
    if (lane == 31) wsum[warp] = x;
    __syncthreads();
    long long wpre = 0, tot = 0;
#pragma unroll
    for (int w = 0; w < SCAN_THREADS / 32; ++w) {
        if (w < warp) wpre += wsum[w];
        tot += wsum[w];
    }
    __syncthreads();
    *total = tot;
    return wpre + x - v;
}

__global__ void __launch_bounds__(SCAN_THREADS) scan_block_sums_kernel(const long long* __restrict__ in, long long n,
                                                                        long long* __restrict__ bsum) {
    const long long base = (long long)blockIdx.x * SCAN_CHUNK;
    long long s = 0;
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; ++k) {
        const long long i = base + (long long)k * SCAN_THREADS + threadIdx.x;
        if (i < n) s += in[i];
    }
    long long tot;
    block_exclusive_scan(s, &tot);
    if (threadIdx.x == 0) bsum[blockIdx.x] = tot;
}

__global__ void __launch_bounds__(SCAN_THREADS) scan_bsums_kernel(long long* __restrict__ bsum, long long nb) {
    __shared__ long long carry_s;
    if (threadIdx.x == 0) carry_s = 0;
    __syncthreads();
    for (long long base = 0; base < nb; base += SCAN_THREADS) {
        const long long i = base + threadIdx.x;
        const long long v = i < nb ? bsum[i] : 0;
        long long tot;
        const long long ex = block_exclusive_scan(v, &tot);
        const long long carry = carry_s;
        if (i < nb) bsum[i] = carry + ex;
        __syncthreads();
        if (threadIdx.x == 0) carry_s = carry + tot;
        __syncthreads();
    }
    if (threadIdx.x == 0) bsum[nb] = carry_s;
}

// out[i] = exclusive prefix of in (in and out may alias); out[n] = total
__global__ void __launch_bounds__(SCAN_THREADS) scan_apply_kernel(const long long* in, long long n,
                                                                   const long long* __restrict__ bsum, long long nb,
                                                                   long long* out) {
    const long long base = (long long)blockIdx.x * SCAN_CHUNK + (long long)threadIdx.x * SCAN_ITEMS;
    long long v[SCAN_ITEMS];
    long long s = 0;
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; ++k) {
        const long long i = base + k;
        v[k] = i < n ? in[i] : 0;
        s += v[k];
    }
    long long tot;
    long long ex = block_exclusive_scan(s, &tot) + bsum[blockIdx.x];
#pragma unroll
    for (int k = 0; k < SCAN_ITEMS; ++k) {
        const long long i = base + k;
        if (i < n) out[i] = ex;
        ex += v[k];
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) out[n] = bsum[nb];
}

// NOTE: scan_block_sums_kernel sums items strided by thread while scan_apply_kernel assigns items contiguously per
// thread; both cover exactly the chunk [blockIdx*SCAN_CHUNK, +SCAN_CHUNK), so the block totals agree.

// ordered compaction: n + 1 offsets, block sums (+ total) and one result slot
size_t select_workspace_bytes(long long n) {
    return (size_t)(n + 1 + (n + SCAN_CHUNK - 1) / SCAN_CHUNK + 3) * sizeof(long long);
}

// exclusive scan of vals[0..n) in place -> vals[0..n], vals[n] = total; bsum = scratch of nb+1
static cudaError_t scan_inplace(long long* vals, long long n, long long* bsum, cudaStream_t st) {
    const long long nb = (n + SCAN_CHUNK - 1) / SCAN_CHUNK;
    if (n == 0) return cudaMemsetAsync(vals, 0, sizeof(long long), st);
    scan_block_sums_kernel<<<(unsigned)nb, SCAN_THREADS, 0, st>>>(vals, n, bsum);
    scan_bsums_kernel<<<1, SCAN_THREADS, 0, st>>>(bsum, nb);
    scan_apply_kernel<<<(unsigned)nb, SCAN_THREADS, 0, st>>>(vals, n, bsum, nb, vals);
    return cudaGetLastError();
}

__global__ void select_flag_kernel(const uint8_t* __restrict__ status, long long n, uint8_t bits, uint8_t value,
                                   long long* __restrict__ flag) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) flag[i] = ((status[i] & bits) == value) ? 1 : 0;
}

__global__ void select_scatter_kernel(const uint8_t* __restrict__ status, long long n, uint8_t bits, uint8_t value,
                                      const long long* __restrict__ offs, long long* __restrict__ idx_out) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n && ((status[i] & bits) == value)) idx_out[offs[i]] = i;
}

// ordered compaction: indices i with (status[i] & bits) == value, ascending; *d_count = how many
cudaError_t select_indices(const uint8_t* status, long long n, uint8_t bits, uint8_t value, long long* idx_out,
                           long long* d_count, void* ws, size_t ws_bytes, cudaStream_t st) {
    if (ws_bytes + sizeof(long long) < select_workspace_bytes(n)) return cudaErrorInvalidValue;
    long long* offs = (long long*)ws;
    long long* bsum = offs + n + 1;
    if (n == 0) return cudaMemsetAsync(d_count, 0, sizeof(long long), st);
    const unsigned blocks = (unsigned)((n + 255) / 256);
    select_flag_kernel<<<blocks, 256, 0, st>>>(status, n, bits, value, offs);
    cudaError_t e = scan_inplace(offs, n, bsum, st);
    if (e != cudaSuccess) return e;
    select_scatter_kernel<<<blocks, 256, 0, st>>>(status, n, bits, value, offs, idx_out);
    return cudaMemcpyAsync(d_count, offs + n, sizeof(long long), cudaMemcpyDeviceToDevice, st);
}

__global__ void root_level_kernel(int W, long long count, uint64_t* __restrict__ masks) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < count) {
        for (int w = 0; w < W; ++w) masks[i * W + w] = 0ull;
        masks[i * W + (i >> 6)] = 1ull << (i & 63);
    }
}

// level-1 candidates [eq..., i]; mpLP keeps only i that can still reach |A| = n (mpqp_combinatorial.py:40-42)
cudaError_t root_level(const DevProgram& P, uint64_t* masks, long long* h_count, cudaStream_t st) {
    long long count = P.mi;
    if (!P.is_qp) {
        long long lim = (long long)1 + P.m - P.n;  // kept iff ne + i < (ne + 1) + m - n
        if (lim < 0) lim = 0;
        if (count > lim) count = lim;
    }
    *h_count = count;
    if (count == 0) return cudaSuccess;
    root_level_kernel<<<(unsigned)((count + 255) / 256), 256, 0, st>>>(P.W, count, masks);
    return cudaGetLastError();
}

__global__ void gather_masks_kernel(const uint64_t* __restrict__ masks, const long long* __restrict__ idx, long long nf, int W,
                                    uint64_t* __restrict__ out) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e < nf * W) {
        const long long p = e / W;
        const int w = (int)(e - p * W);
        out[e] = masks[idx[p] * W + w];
    }
}

struct Mask4 { uint64_t w[MAXW]; };

// lexicographic compare of a stored key with a register-resident mask (fully unrolled: no dynamic indexing)
__device__ __forceinline__ int lex_cmp4(const uint64_t* __restrict__ a, const Mask4& b, int W) {
    int res = 0;
#pragma unroll
    for (int x = 0; x < MAXW; ++x) {
        if (x < W && res == 0) {
            const uint64_t av = a[x];
            const uint64_t d = av ^ b.w[x];
            if (d) {
                const uint64_t low = d & (~d + 1ull);
                res = (av & low) ? -1 : 1;
            }
        }
    }
    return res;
}

__device__ __forceinline__ unsigned hash_mask(const Mask4& k, int W) {
    uint64_t h = 0x9e3779b97f4a7c15ull;
#pragma unroll
    for (int x = 0; x < MAXW; ++x)
        if (x < W) { h ^= k.w[x]; h *= 0xff51afd7ed558ccdull; h ^= h >> 32; }
    return (unsigned)h;
}

__device__ __forceinline__ Mask4 load_mask(const uint64_t* __restrict__ m, long long i, int W) {
    Mask4 k;
#pragma unroll
    for (int x = 0; x < MAXW; ++x) k.w[x] = x < W ? __ldg(m + i * W + x) : 0ull;
    return k;
}

__device__ __forceinline__ bool mask_eq(const Mask4& a, const Mask4& b) {
    bool eq = true;
#pragma unroll
    for (int x = 0; x < MAXW; ++x) eq &= a.w[x] == b.w[x];
    return eq;
}

// removes the highest row from k and returns it (-1: k is empty)
__device__ __forceinline__ int pop_last(Mask4& k) {
    int last = -1;
#pragma unroll
    for (int x = MAXW - 1; x >= 0; --x)
        if (last < 0 && k.w[x]) {
            const int b = 63 - __clzll((long long)k.w[x]);
            k.w[x] &= ~(1ull << b);
            last = x * 64 + b;
        }
    return last;
}

__device__ __forceinline__ uint64_t low_bits(int b) { return b <= 0 ? 0ull : b >= 64 ? ~0ull : (1ull << b) - 1ull; }

// the rows [lo, hi)
__device__ __forceinline__ Mask4 row_range(int lo, int hi) {
    Mask4 r;
#pragma unroll
    for (int x = 0; x < MAXW; ++x) r.w[x] = low_bits(hi - 64 * x) & ~low_bits(lo - 64 * x);
    return r;
}

// ---- prefix-group index of a level's feasible list ---------------------------------------------------------------------------
// A level's feasible list is in lexicographic order (root_level, children parent by parent in ascending i, ordered
// compaction), so the sets that share their PREFIX Q (the set without its highest row) form one contiguous run, in
// ascending highest row.  children_prepare makes every run a group: the index of its first member (`start`, also its key:
// the prefix of that member is Q) and E_Q, the bitmap of its members' highest rows.  Then
//     Q + {x} is in the list  <=>  x in E_Q,  at index  start + |E_Q below x|.
// Groups are found through an open-addressing table keyed by Q (load <= 1/2).  There are as many groups as distinct
// prefixes: 158 k for the 3.78 M level-4 sets of the bench program, so table and records are a few MB that stay in L2;
// the key compare reads the group's first member from the mask array (one line per group probed), which keeps the
// workspace at W + 1 words per group instead of 2W + 1.
//
// Workspace after the scan block sums (nb + 2 long long words): hdr = {table mask, number of groups, order violated, -};
// the table, int32
// slots in table_words(nf) words (during children_prepare the same words first hold the run-start flags and their scan,
// nf + 1 words); one record of W + 1 words per group, {start, E}, so that one look-up reads both.  scan_workspace_bytes
// sizes it for nf groups of MAXW words.
struct GroupIndex {
    long long* hdr;
    int* table;
    uint64_t* rec;
};

static GroupIndex group_index(void* ws, long long nf) {
    long long* base = (long long*)ws + (nf + SCAN_CHUNK - 1) / SCAN_CHUNK + 2;
    GroupIndex gi;
    gi.hdr = base;
    gi.table = reinterpret_cast<int*>(base + 4);
    gi.rec = reinterpret_cast<uint64_t*>(base + 4 + table_words(nf));
    return gi;
}

static size_t group_index_bytes(long long nf, int W) {
    const long long nb = (nf + SCAN_CHUNK - 1) / SCAN_CHUNK;
    return (size_t)(nb + 6 + table_words(nf) + (long long)(W + 1) * nf) * sizeof(long long);
}

// K6 workspace: scan block sums and the prefix-group index of up to n groups of MAXW words
size_t scan_workspace_bytes(long long n) { return group_index_bytes(n, MAXW); }

// nonzero after children_prepare iff the parents were not strictly increasing sets of one cardinality
const long long* children_order_flag(const void* ws, long long nf) { return group_index(const_cast<void*>(ws), nf).hdr + 2; }

// flag[p] = 1 iff p starts a run (its prefix differs from that of p - 1).  The runs are the groups only if the list is
// in lexicographic order: an entry that does not follow its predecessor in that order, or differs in cardinality, sets
// hdr[2], and the host calls that read the child total report it
__global__ void group_flag_kernel(const uint64_t* __restrict__ feas, long long nf, int W, long long* __restrict__ flag,
                                  GroupIndex gi) {
    const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= nf) return;
    const Mask4 m = load_mask(feas, p, W);
    Mask4 q = m;
    pop_last(q);
    bool first = p == 0;
    if (!first) {
        const Mask4 prev = load_mask(feas, p - 1, W);
        int cp = 0, cm = 0;
#pragma unroll
        for (int x = 0; x < MAXW; ++x) { cp += __popcll(prev.w[x]); cm += __popcll(m.w[x]); }
        if (cp != cm || lex_cmp4(feas + (p - 1) * W, m, W) >= 0) gi.hdr[2] = 1;
        Mask4 r = prev;
        pop_last(r);
        first = !mask_eq(q, r);
    }
    flag[p] = first ? 1 : 0;
}

// gid = exclusive scan of the flags (gid[nf] = number of groups).  The first member of each run records the group and
// walks the run (at most mi members) for E; thread 0 sizes the table (a power of two >= 2 x groups).
__global__ void group_build_kernel(const uint64_t* __restrict__ feas, long long nf, int W, const long long* __restrict__ gid,
                                   GroupIndex gi) {
    const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= nf) return;
    if (p == 0) {
        const long long groups = gid[nf];
        long long cap = 1024;
        while (cap < 2 * groups) cap <<= 1;
        gi.hdr[0] = cap - 1;
        gi.hdr[1] = groups;
    }
    const long long g = gid[p];
    if (gid[p + 1] == g) return;
    Mask4 q = load_mask(feas, p, W);
    Mask4 e = row_range(0, 0);
    int last = pop_last(q);
    for (long long r = p + 1;; ++r) {
        const Mask4 bit = row_range(last, last + 1);
#pragma unroll
        for (int x = 0; x < MAXW; ++x) e.w[x] |= bit.w[x];
        if (r >= nf) break;
        Mask4 s = load_mask(feas, r, W);
        last = pop_last(s);
        if (!mask_eq(s, q)) break;
    }
    uint64_t* r = gi.rec + g * (W + 1);
    r[0] = (uint64_t)p;
#pragma unroll
    for (int x = 0; x < MAXW; ++x)
        if (x < W) r[1 + x] = e.w[x];
}

__global__ void group_clear_kernel(GroupIndex gi) {
    const long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (s <= gi.hdr[0]) gi.table[s] = -1;
}

__global__ void group_insert_kernel(const uint64_t* __restrict__ feas, int W, GroupIndex gi) {
    const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= gi.hdr[1]) return;
    const unsigned cap_mask = (unsigned)gi.hdr[0];
    Mask4 q = load_mask(feas, (long long)gi.rec[g * (W + 1)], W);
    pop_last(q);
    unsigned slot = hash_mask(q, W) & cap_mask;
    while (atomicCAS(&gi.table[slot], -1, (int)g) != -1) slot = (slot + 1) & cap_mask;
}

// E of the group of prefix q; false if no set of the list has that prefix
__device__ __forceinline__ bool find_group(const uint64_t* __restrict__ feas, int W, const GroupIndex& gi, unsigned cap_mask,
                                           const Mask4& q, Mask4& e) {
    unsigned slot = hash_mask(q, W) & cap_mask;
    for (;;) {
        const int g = __ldg(gi.table + slot);
        if (g < 0) return false;
        const uint64_t* r = gi.rec + (long long)g * (W + 1);
        e = load_mask(r + 1, 0, W);
        Mask4 k = load_mask(feas, (long long)__ldg(r), W);
        pop_last(k);
        if (mask_eq(k, q)) return true;
        slot = (slot + 1) & cap_mask;
    }
}

// One thread per parent P (highest row l).  A child C = P + {i} has i > l, so each k-subset C \ {j}, j in P, is
// (P \ {j}) + {i} with i as its highest row: it is in the feasible list iff i is in E_{P \ {j}}.  The surviving children
// are the rows i > l within the mpLP limits that lie in the intersection of those k bitmaps (j = l is P's own group):
// at most k group look-ups per parent (CNT_K6_LOOKUPS counts them) instead of k look-ups of a child's subsets per child.
// W (= P.W) is a template parameter so that masks hold W words in registers, not MAXW; 3 blocks per SM leave W = 4
// enough registers not to spill.
template <int W>
__global__ void __launch_bounds__(256, 3)
children_count_kernel(DevProgram P, const uint64_t* __restrict__ feas, long long p_lo, long long p_hi, int k_act,
                      uint64_t* __restrict__ survive, long long* __restrict__ counts,
                      unsigned long long* __restrict__ counters, GroupIndex gi) {
    const long long p = p_lo + (long long)blockIdx.x * blockDim.x + threadIdx.x;
    unsigned long long lookups = 0;
    if (p < p_hi) {
        const unsigned cap_mask = (unsigned)__ldg(gi.hdr);
        // mpLP: a list of length L whose last element is g is dropped iff g >= L + m - n.  The child exists iff
        // ne + i < child_limit; for ne + i >= sub_limit its k-subsets ending in i were dropped by that filter, not tested,
        // and the subset test is waived
        const bool lp = !P.is_qp;
        const long long child_limit = lp ? (long long)(P.ne + k_act + 1) + P.m - P.n : (long long)P.ne + P.mi;
        const long long sub_limit = lp ? child_limit - 1 : (long long)P.ne + P.mi;
        const Mask4 pm = load_mask(feas, p, W);
        Mask4 rest = pm;
        const int last = pop_last(rest);
        const int hi = (int)(child_limit - P.ne < P.mi ? child_limit - P.ne : P.mi);
        const int wlo = (int)(sub_limit - P.ne > last + 1 ? sub_limit - P.ne : last + 1);
        const Mask4 range = row_range(last + 1, hi), waived = row_range(wlo, hi);
        Mask4 acc;
#pragma unroll
        for (int x = 0; x < MAXW; ++x) acc.w[x] = x < W ? ~0ull : 0ull;
        bool open = true;   // some child whose test is not waived is still in acc
#pragma unroll
        for (int w = MAXW - 1; w >= 0; --w) {
            uint64_t bits = pm.w[w];
            while (bits && open) {
                uint64_t left = 0;
#pragma unroll
                for (int x = 0; x < MAXW; ++x) left |= range.w[x] & ~waived.w[x] & acc.w[x];
                open = left != 0;
                if (!open) break;
                const int b = 63 - __clzll((long long)bits);
                bits &= ~(1ull << b);
                Mask4 q = pm;
                q.w[w] &= ~(1ull << b);
                ++lookups;
                Mask4 e;
                const bool found = find_group(feas, W, gi, cap_mask, q, e);
#pragma unroll
                for (int x = 0; x < MAXW; ++x) acc.w[x] &= found ? e.w[x] : 0ull;
            }
        }
        long long cnt = 0;
#pragma unroll
        for (int x = 0; x < MAXW; ++x) {
            const uint64_t sv = range.w[x] & (waived.w[x] | acc.w[x]);
            cnt += __popcll(sv);
            if (x < W) survive[p * W + x] = sv;
        }
        counts[p] = cnt;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) lookups += __shfl_xor_sync(0xffffffffu, lookups, o);
    if ((threadIdx.x & 31) == 0 && lookups) atomicAdd(&counters[CNT_K6_LOOKUPS], lookups);
}

__global__ void __launch_bounds__(128)
children_write_kernel(int W, const uint64_t* __restrict__ feas, const uint64_t* __restrict__ survive,
                      const long long* __restrict__ offsets, long long nf, uint64_t* __restrict__ children) {
    const int lane = threadIdx.x & 31;
    const long long warp0 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long p = warp0; p < nf; p += nwarps) {
        long long off = offsets[p];
        for (int w = 0; w < W; ++w) {
            const uint64_t x = survive[p * W + w];
            const int tot = __popcll(x);
            for (int r = lane; r < tot; r += 32) {
                const int b = mask_nth(&x, 1, r);
                uint64_t* dst = children + (off + r) * W;
                for (int y = 0; y < W; ++y) dst[y] = feas[p * W + y] | (y == w ? (1ull << b) : 0ull);
            }
            off += tot;
        }
    }
}

// gathers the feasible parents (in the level's lexicographic order) and builds their prefix-group index in the workspace
cudaError_t children_prepare(const DevProgram& P, const uint64_t* masks, const long long* feas_idx, long long nf,
                             uint64_t* feas_masks, void* ws, size_t ws_bytes, cudaStream_t st) {
    if (P.W > MAXW) return cudaErrorInvalidValue;
    if (nf <= 0) return cudaSuccess;
    if (nf >= (1ll << 30)) return cudaErrorInvalidValue;
    if (ws_bytes < group_index_bytes(nf, P.W)) return cudaErrorInvalidValue;
    const GroupIndex gi = group_index(ws, nf);
    long long* gid = reinterpret_cast<long long*>(gi.table);   // nf + 1 words, dead before the table is cleared
    const long long ne = nf * P.W;
    const unsigned blocks = (unsigned)((nf + 255) / 256);
    gather_masks_kernel<<<(unsigned)((ne + 255) / 256), 256, 0, st>>>(masks, feas_idx, nf, P.W, feas_masks);
    cudaError_t e = cudaMemsetAsync(gi.hdr, 0, 4 * sizeof(long long), st);
    if (e != cudaSuccess) return e;
    group_flag_kernel<<<blocks, 256, 0, st>>>(feas_masks, nf, P.W, gid, gi);
    e = scan_inplace(gid, nf, (long long*)ws, st);
    if (e != cudaSuccess) return e;
    group_build_kernel<<<blocks, 256, 0, st>>>(feas_masks, nf, P.W, gid, gi);
    long long cap = 1024;   // the largest table group_build_kernel can size (nf groups)
    while (cap < 2 * nf) cap <<= 1;
    group_clear_kernel<<<(unsigned)(cap / 256), 256, 0, st>>>(gi);
    group_insert_kernel<<<blocks, 256, 0, st>>>(feas_masks, P.W, gi);
    return cudaGetLastError();
}

// surviving children (bit sets) and their number for the parents [p_lo, p_hi); other entries are left untouched
cudaError_t children_count_range(const DevProgram& P, const uint64_t* feas_masks, long long nf, int k_act, uint64_t* survive,
                                 long long* counts, long long p_lo, long long p_hi, void* ws, unsigned long long* counters,
                                 cudaStream_t st) {
    if (p_hi <= p_lo) return cudaSuccess;
    const unsigned blocks = (unsigned)((p_hi - p_lo + 255) / 256);
    const GroupIndex gi = group_index(ws, nf);
    switch (P.W) {
        case 1: children_count_kernel<1><<<blocks, 256, 0, st>>>(P, feas_masks, p_lo, p_hi, k_act, survive, counts, counters, gi); break;
        case 2: children_count_kernel<2><<<blocks, 256, 0, st>>>(P, feas_masks, p_lo, p_hi, k_act, survive, counts, counters, gi); break;
        case 3: children_count_kernel<3><<<blocks, 256, 0, st>>>(P, feas_masks, p_lo, p_hi, k_act, survive, counts, counters, gi); break;
        case 4: children_count_kernel<4><<<blocks, 256, 0, st>>>(P, feas_masks, p_lo, p_hi, k_act, survive, counts, counters, gi); break;
        default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}

cudaError_t children_scan(long long* counts_to_offsets, long long nf, void* ws, cudaStream_t st) {
    if (nf == 0) return cudaMemsetAsync(counts_to_offsets, 0, sizeof(long long), st);
    return scan_inplace(counts_to_offsets, nf, (long long*)ws, st);
}

cudaError_t children_count(const DevProgram& P, const uint64_t* masks, const long long* feas_idx, long long nf, int k_act,
                           uint64_t* feas_masks, uint64_t* survive, long long* offsets, void* ws, size_t ws_bytes,
                           unsigned long long* counters, cudaStream_t st) {
    if (nf == 0) return cudaMemsetAsync(offsets, 0, sizeof(long long), st);
    cudaError_t e = children_prepare(P, masks, feas_idx, nf, feas_masks, ws, ws_bytes, st);
    if (e != cudaSuccess) return e;
    if ((e = children_count_range(P, feas_masks, nf, k_act, survive, offsets, 0, nf, ws, counters, st)) != cudaSuccess) return e;
    return children_scan(offsets, nf, ws, st);
}

cudaError_t children_write(const DevProgram& P, const uint64_t* feas_masks, const uint64_t* survive, const long long* offsets,
                           long long nf, uint64_t* children, cudaStream_t st) {
    if (nf == 0) return cudaSuccess;
    long long blocks = (nf * 32 + 127) / 128;
    if (blocks > 148 * 64) blocks = 148 * 64;
    children_write_kernel<<<(unsigned)blocks, 128, 0, st>>>(P.W, feas_masks, survive, offsets, nf, children);
    return cudaGetLastError();
}

// ---- certificates inherited from the previous level ------------------------------------------------------------------------
// The vertex walk (k2w_walk.cu) leaves, for every candidate it certifies, the WITNESS: the mask of all rows active at the
// certifying vertex (~n' rows, the candidate's own among them), and next to it the mask of a later vertex of the walk that
// holds the candidate as well (PPG_WITNESS_SLOTS masks per candidate).  A candidate C of the next level is feasible as soon
// as a witness of ONE of its parents C \ {b} also has row b active: the same vertex, the same exact statement ("the rows of
// C are nonbasic at a vertex whose basic slacks are >= -1e-8").  On the 100x30x6 program 85 % of the candidates of levels
// 4-5 are certified this way (CPU model scripts/witness_coverage_model.py: 84 % / 86 %), which removes them - the ones
// that are easy to reach - from the walk.  Parents are found in the prefix-group index K6 built when it generated this
// level (children_prepare): the parent S = C \ {b} with highest row h and prefix Q sits at start(Q) + |E_Q below h| in
// the parent level's feasible list; parent_wit is the witness array gathered in that order.  One thread per candidate;
// rows are dropped from the highest down (CPU model: the middle positions inherit most often, the first one least).  An
// inherited witness is passed on (witness_out), so that certificates propagate down the levels without any further pivot.
template <int W>
__global__ void __launch_bounds__(256)
inherit_kernel(const uint64_t* __restrict__ masks, long long n, uint8_t* __restrict__ status,
               uint64_t* __restrict__ witness_out, const uint64_t* __restrict__ pfeas, GroupIndex gi,
               const uint64_t* __restrict__ pwit, unsigned long long* __restrict__ counters) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    unsigned long long lookups = 0;
    int got = 0;
    if (i < n) {
        const uint8_t sb = status[i];
        if ((sb & PPG_ST_RANK) && !(sb & PPG_ST_FEAS)) {
            const unsigned cap_mask = (unsigned)__ldg(gi.hdr);
            const Mask4 m = load_mask(masks, i, W);
#pragma unroll
            for (int w = MAXW - 1; w >= 0; --w) {
                if (w < W && !got) {
                    uint64_t bits = m.w[w];
                    while (bits && !got) {
                        const int b = 63 - __clzll((long long)bits);
                        bits &= ~(1ull << b);
                        Mask4 q = m;
                        q.w[w] &= ~(1ull << b);
                        const Mask4 sub = q;         // the parent S = C \ {b}
                        const int h = pop_last(q);   // its highest row; q = its prefix Q
                        if (h < 0) continue;         // a single row: level 1 has no parent level
                        ++lookups;
                        const Mask4 below = row_range(0, h), bit = row_range(h, h + 1);
                        // Q's probe sequence: a group whose E holds h names an entry of the list, and that entry is S
                        // iff the group is Q's - so S's mask and its witnesses load together, with no key compare first
                        unsigned slot = hash_mask(q, W) & cap_mask;
                        for (;;) {
                            const int g = __ldg(gi.table + slot);
                            if (g < 0) break;
                            slot = (slot + 1) & cap_mask;
                            const uint64_t* r = gi.rec + (long long)g * (W + 1);
                            const Mask4 eq = load_mask(r + 1, 0, W);
                            long long e = (long long)__ldg(r);
                            uint64_t in = 0;
#pragma unroll
                            for (int x = 0; x < MAXW; ++x) {
                                e += __popcll(eq.w[x] & below.w[x]);
                                in |= eq.w[x] & bit.w[x];
                            }
                            if (!in) continue;   // (for Q's own group only if S is not feasible: never for a child K6 let through)
                            const Mask4 pm = load_mask(pfeas, e, W);
                            uint64_t wv[PPG_WITNESS_SLOTS][MAXW];
#pragma unroll
                            for (int sl = 0; sl < PPG_WITNESS_SLOTS; ++sl)
#pragma unroll
                                for (int x = 0; x < MAXW; ++x)
                                    wv[sl][x] = x < W ? __ldg(pwit + ((e * PPG_WITNESS_SLOTS + sl) * W + x)) : 0ull;
                            if (!mask_eq(pm, sub)) continue;
                            // a parent's witnesses hold the parent (or are empty: certified by the relaxation / the simplex)
#pragma unroll
                            for (int sl = 0; sl < PPG_WITNESS_SLOTS; ++sl) {
                                bool inside = !got;
#pragma unroll
                                for (int x = 0; x < MAXW; ++x)
                                    if (m.w[x] & ~wv[sl][x]) inside = false;
                                if (inside) {
                                    got = 1;
                                    status[i] = sb | PPG_ST_FEAS;
                                    if (witness_out)
#pragma unroll
                                        for (int x = 0; x < MAXW; ++x)
                                            if (x < W) witness_out[i * (PPG_WITNESS_SLOTS * W) + x] = wv[sl][x];
                                }
                            }
                            break;
                        }
                    }
                }
            }
        }
    }
    got = __reduce_add_sync(0xffffffffu, got);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) lookups += __shfl_xor_sync(0xffffffffu, lookups, o);
    if ((threadIdx.x & 31) == 0 && lookups) {
        atomicAdd(&counters[CNT_INHERITED], (unsigned long long)got);
        atomicAdd(&counters[CNT_INHERIT_LOOKUPS], lookups);
    }
}

cudaError_t launch_inherit(const DevProgram& P, const uint64_t* masks, long long n, uint8_t* status, uint64_t* witness_out,
                           const uint64_t* parent_feas, long long parent_nf, const void* parent_ws, const uint64_t* parent_wit,
                           unsigned long long* counters, cudaStream_t st) {
    if (n <= 0 || parent_nf <= 0) return cudaSuccess;
    if (P.W > MAXW) return cudaErrorInvalidValue;
    // the index sits in the K6 workspace behind the scan scratch (children_prepare)
    const GroupIndex gi = group_index(const_cast<void*>(parent_ws), parent_nf);
    const unsigned blocks = (unsigned)((n + 255) / 256);
    switch (P.W) {
        case 1: inherit_kernel<1><<<blocks, 256, 0, st>>>(masks, n, status, witness_out, parent_feas, gi, parent_wit, counters); break;
        case 2: inherit_kernel<2><<<blocks, 256, 0, st>>>(masks, n, status, witness_out, parent_feas, gi, parent_wit, counters); break;
        case 3: inherit_kernel<3><<<blocks, 256, 0, st>>>(masks, n, status, witness_out, parent_feas, gi, parent_wit, counters); break;
        case 4: inherit_kernel<4><<<blocks, 256, 0, st>>>(masks, n, status, witness_out, parent_feas, gi, parent_wit, counters); break;
        default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}

// ---- FP64 FMA peak of the device (roofline denominator for the LP kernels; not in MEASURED_PEAKS.json)
__global__ void __launch_bounds__(256) dfma_peak_kernel(int iters, double* sink) {
    double a0 = threadIdx.x * 1e-3, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
    const double m = 0.999999, c = 1e-9;
    for (int i = 0; i < iters; ++i) {
        a0 = fma(a0, m, c); a1 = fma(a1, m, c); a2 = fma(a2, m, c); a3 = fma(a3, m, c);
        a4 = fma(a4, m, c); a5 = fma(a5, m, c); a6 = fma(a6, m, c); a7 = fma(a7, m, c);
    }
    const double s = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
    if (s == 123.456) sink[0] = s;
}

cudaError_t measure_fp64_peak(int iters, double* tflops, cudaStream_t st) {
    int dev = 0, sms = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    double* sink = nullptr;
    cudaError_t e = cudaMalloc(&sink, sizeof(double));
    if (e != cudaSuccess) return e;
    cudaEvent_t a, b;
    cudaEventCreate(&a); cudaEventCreate(&b);
    const int blocks = sms * 8;
    dfma_peak_kernel<<<blocks, 256, 0, st>>>(iters / 10 + 1, sink);
    float best = 1e30f;
    for (int rep = 0; rep < 3; ++rep) {
        cudaEventRecord(a, st);
        dfma_peak_kernel<<<blocks, 256, 0, st>>>(iters, sink);
        cudaEventRecord(b, st);
        cudaEventSynchronize(b);
        float ms = 0;
        cudaEventElapsedTime(&ms, a, b);
        if (ms < best) best = ms;
    }
    cudaEventDestroy(a); cudaEventDestroy(b);
    cudaFree(sink);
    e = cudaGetLastError();
    const double flops = 2.0 * 8.0 * (double)iters * 256.0 * blocks;
    *tflops = flops / (best * 1e-3) / 1e12;
    return e;
}

}  // namespace ppgpu
