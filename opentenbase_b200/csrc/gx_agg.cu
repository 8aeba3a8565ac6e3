// gx_agg.cu — K3+K4: [hash probe ->] hash aggregate.
//
// Replaces agg_fill_hash_table / lookup_hash_entries / advance_aggregates
// (nodeAgg.c:2609,2149,856), LookupTupleHashEntry (execGrouping.c:295) and —
// when a join feeds the aggregate — ExecHashJoinImpl's probe loop
// (nodeHashjoin.c:446-666) without materialising the join.
//
// State model.  A group is a record of 8-byte words
//      [meta | k0 | k1 | w0 .. w(nwords-1)]
// meta = null bits of the group columns, k0/k1 = the group columns packed by
// byte width, w0 = the group's row count, the other words belong to the
// aggregates (float8 sum, non-NULL input count, int8 sum, min/max).  Every word
// has a merge kind (add int64 / add float8 / min / max), so ONE merge operator
// serves the per-CTA shared-memory tables, the global table, the second radix
// pass and the cross-datanode Finalize step (int8pl / float8pl /
// float8_combine's N and Sx, utils/adt/float.c:2725).
//
// Strategies:
//   1  shared-memory privatised table per CTA, merged into an L2-resident
//      global table at CTA exit  (few groups: Q1, GROUP BY date)
//   2  two-pass radix: rows -> per-row records -> partition by key hash ->
//      one CTA aggregates one partition in shared memory (many groups: Q3)
//   3  global table only (atomics in L2)
#include "gx_internal.cuh"
#include <type_traits>

int gx_fill_dpreds(gx_ctx *ctx, const gx_table *t, int n_preds, const gx_pred *preds, gx_dpred *out);

enum { WK_ADD_I64 = 0, WK_ADD_F64 = 1, WK_MIN_F64 = 2, WK_MAX_F64 = 3 };

struct gx_agg_dev {
    gx_dplan P;
    long long winit[GX_MAX_WORDS];
    int wkind[GX_MAX_WORDS];
    // join table
    const gx_slot *slots; unsigned long long mask;
    const gx_cslot *cslots; unsigned long long cspan;      // compact form of the table (gx_k_runjoin reads it directly)
    const unsigned long long *special; int special_count; int _pad0; gx_slotfn sf;
    long long row0, row1;
    // shared-memory table
    int s_slots;             // power of two; 0 = none
    int s_log2;              // log2(s_slots)
    int s_tagkey;            // 1: the tag word holds the whole (<= 7 byte) key, no k0/k1 arrays
    int s_gmax;              // lane-private mode: max dense groups per CTA (0 = dense CAS mode)
    int need_w0;             // maintain w0 (rows per group)?
    int _pad1;
    // global table: g_cap records of (3 + nwords) words
    unsigned long long *g_tab; unsigned long long g_mask;
    // record sink (radix stage A)
    unsigned long long *recs; long long rec_cap;
    long long *counters;     // [0] ngroups in g_tab, [1] overflow flags, [2] record cursor
};

#define TAG_LOCK 1ULL

__device__ __forceinline__ unsigned long long group_hash(unsigned long long k0, unsigned long long k1, unsigned int nullmask)
{
    return gx_mix64(k0 ^ (k1 * 0x9E3779B97F4A7C15ULL) ^ ((unsigned long long) nullmask << 56) ^ 0x51ED270B27B4F3CFULL);
}
__device__ __forceinline__ unsigned long long make_tag(unsigned long long h, unsigned int nullmask)
{
    return (1ULL << 63) | ((unsigned long long) (nullmask & 0xF) << 59) | (h >> 5);
}

// merge one word into a (shared or global) location
__device__ __forceinline__ void atomic_min_f64(unsigned long long *addr, double v, bool want_min)
{
    unsigned long long old = *(volatile unsigned long long *) addr;
    for (;;) {
        double cur = __longlong_as_double((long long) old);
        int c = gx_f8cmp(v, cur);
        if (want_min ? (c >= 0) : (c <= 0)) return;
        unsigned long long prev = atomicCAS(addr, old, (unsigned long long) __double_as_longlong(v));
        if (prev == old) return;
        old = prev;
    }
}
__device__ __forceinline__ void merge_word(unsigned long long *addr, int kind, unsigned long long v)
{
    switch (kind) {
        case WK_ADD_I64: if (v) atomicAdd(addr, v); break;
        case WK_ADD_F64: atomicAdd((double *) addr, __longlong_as_double((long long) v)); break;
        case WK_MIN_F64: atomic_min_f64(addr, __longlong_as_double((long long) v), true); break;
        default:         atomic_min_f64(addr, __longlong_as_double((long long) v), false); break;
    }
}

// --------------------------------------------------------------- sinks
// CTA-shared directory (+ dense state words).  Measured on B200
// (profiles/r01_ubench_agg_update_mechanisms.txt): a CTA-shared table with
// CAS-loop fp64 adds sustains ~230 G rows/s; for a handful of groups
// lane-private accumulators ([word][group][lane], bank == lane, no atomics)
// reach ~440 G rows/s.  Both are used here.
struct SmemTable {
    unsigned long long *tag, *k0, *k1, *w;   // dense: w[slot * nwords + i]; lane-private: see lp_base()
    unsigned int *gidx;                      // lane-private: slot -> dense group number
    unsigned int *gcount;                    // lane-private: groups handed out so far
    int S, log2S, nwords, nkw, tagkey, gmax;
};

__device__ __forceinline__ unsigned long long smem_hash(unsigned long long k0, unsigned long long k1, unsigned int nullmask)
{
    return (k0 ^ (k0 >> 29) ^ (k1 * 0xC2B2AE3D27D4EB4FULL) ^ ((unsigned long long) nullmask << 50)) * 0x9E3779B97F4A7C15ULL;
}

// returns the slot, or -1 when the table (or the lane-private group budget) is full
template <bool LP>
__device__ __forceinline__ int smem_upsert(const SmemTable &T, unsigned long long k0, unsigned long long k1, unsigned int nullmask)
{
    unsigned long long h = smem_hash(k0, k1, nullmask);
    unsigned long long tag = T.tagkey ? ((1ULL << 63) | ((unsigned long long) (nullmask & 0xF) << 59) | (k0 & 0x00FFFFFFFFFFFFFFULL))
                                      : make_tag(h, nullmask);
    int s = (int) (h >> (64 - T.log2S));
    const int maxprobe = T.S < 64 ? T.S : 64;
    const bool direct = T.tagkey && !LP;          // the tag IS the key: claim with one CAS, no lock phase
    for (int n = 0; n < maxprobe; n++) {
        unsigned long long t = *(volatile unsigned long long *) &T.tag[s];
        if (t == tag) { if (T.tagkey || (T.k0[s] == k0 && (T.nkw == 1 || T.k1[s] == k1))) return s; }
        else if (t == 0) {
            unsigned long long old = atomicCAS(&T.tag[s], 0ULL, direct ? tag : TAG_LOCK);
            if (old == 0) {
                if (direct) return s;
                if (!T.tagkey) { T.k0[s] = k0; if (T.nkw > 1) T.k1[s] = k1; }
                if (LP) {
                    unsigned int gi = atomicAdd(T.gcount, 1u);
                    T.gidx[s] = gi;                 // gi >= gmax is caught by the caller
                }
                __threadfence_block();
                *(volatile unsigned long long *) &T.tag[s] = tag;
                return s;
            }
            t = old;
            while (t == TAG_LOCK) t = *(volatile unsigned long long *) &T.tag[s];
            if (t == tag && (T.tagkey || (T.k0[s] == k0 && (T.nkw == 1 || T.k1[s] == k1)))) return s;
        } else if (t == TAG_LOCK) {
            while (t == TAG_LOCK) t = *(volatile unsigned long long *) &T.tag[s];
            if (t == tag && (T.tagkey || (T.k0[s] == k0 && (T.nkw == 1 || T.k1[s] == k1)))) return s;
        }
        s = (s + 1) & (T.S - 1);
    }
    return -1;
}

// global table: record r at g_tab + r * (3 + nwords): [tag][k0][k1][w..]
__device__ __forceinline__ unsigned long long *global_upsert(const gx_agg_dev &A, unsigned long long k0, unsigned long long k1,
                                                             unsigned int nullmask)
{
    const int RW = 3 + A.P.nwords;
    unsigned long long h = group_hash(k0, k1, nullmask), tag = make_tag(h, nullmask);
    unsigned long long s = h & A.g_mask;
    for (unsigned long long n = 0; n <= A.g_mask; n++) {
        unsigned long long *rec = A.g_tab + s * RW;
        unsigned long long t = *(volatile unsigned long long *) rec;
        if (t == 0) {
            unsigned long long old = atomicCAS(rec, 0ULL, TAG_LOCK);
            if (old == 0) {
                rec[1] = k0; rec[2] = k1;
                for (int i = 0; i < A.P.nwords; i++) rec[3 + i] = (unsigned long long) A.winit[i];
                __threadfence();
                *(volatile unsigned long long *) rec = tag;
                atomicAdd((unsigned long long *) &A.counters[0], 1ULL);
                return rec;
            }
            t = old;
        }
        while (t == TAG_LOCK) t = *(volatile unsigned long long *) rec;
        if (t == tag && rec[1] == k0 && rec[2] == k1) return rec;
        s = (s + 1) & A.g_mask;
        if (n > 4096 && (n & 1023) == 0 && *(volatile long long *) &A.counters[1]) break;
    }
    return nullptr;
}

enum { SINK_SMEM = 1, SINK_RECORD = 2, SINK_GLOBAL = 3, SINK_SMEM_LP = 4 };

template <int SINK>
struct Sink {
    unsigned long long *w;          // base of the target's state words
    int wstride;                    // distance between consecutive words (lane-private: gmax * 32)
    __device__ __forceinline__ unsigned long long *at(int word) { return w + (size_t) word * wstride; }
    // +1 on a counter word
    __device__ __forceinline__ void inc(int word)
    {
        if (SINK == SINK_RECORD) *at(word) = 1ULL;
        else if (SINK == SINK_SMEM_LP) *at(word) += 1ULL;
        else if (SINK == SINK_SMEM) atomicAdd((unsigned int *) at(word), 1u);   // native ATOMS.ADD.32; < 2^32 rows per CTA
        else atomicAdd(at(word), 1ULL);
    }
    __device__ __forceinline__ void add_i64(int word, long long v)
    {
        if (SINK == SINK_RECORD) *at(word) = (unsigned long long) v;
        else if (SINK == SINK_SMEM_LP) *at(word) += (unsigned long long) v;
        else atomicAdd(at(word), (unsigned long long) v);
    }
    __device__ __forceinline__ void add_f64(int word, double v)
    {
        if (SINK == SINK_RECORD) *at(word) = (unsigned long long) __double_as_longlong(v);
        else if (SINK == SINK_SMEM_LP) { double *p = (double *) at(word); *p = __dadd_rn(*p, v); }
        else atomicAdd((double *) at(word), v);
    }
    __device__ __forceinline__ void minmax_f64(int word, double v, bool want_min)
    {
        if (SINK == SINK_RECORD) *at(word) = (unsigned long long) __double_as_longlong(v);
        else if (SINK == SINK_SMEM_LP) {
            double *p = (double *) at(word); int c = gx_f8cmp(v, *p);
            if (want_min ? (c < 0) : (c > 0)) *p = v;
        } else atomic_min_f64(at(word), v, want_min);
    }
};

// pack the group columns of one (joined) row
__device__ __forceinline__ void pack_group_key(const gx_dplan &P, long long r, unsigned long long payload,
                                               unsigned long long &k0, unsigned long long &k1, unsigned int &nullmask)
{
    k0 = 0; k1 = 0; nullmask = 0;
#pragma unroll
    for (int c = 0; c < GX_MAX_GROUP_COLS; c++) {
        if (c >= P.ngroup) break;
        const gx_dgroupcol &g = P.gcols[c];
        unsigned long long v;
        if (g.side == 0) {
            if (gx_is_null(g.col, r)) { nullmask |= 1u << c; continue; }
            v = (unsigned long long) gx_load_int(g.col, r);
            if (g.type == GX_FLOAT8) {                       // -0 = +0, all NaNs equal (float8eq)
                double d = __longlong_as_double((long long) v);
                if (d == 0.0) v = 0; else if (isnan(d)) v = 0x7FF8000000000000ULL;
            }
        } else {
            v = payload >> g.payload_idx;                     // payload_idx holds the bit offset
        }
        if (g.bytes < 8) v &= (1ULL << (8 * g.bytes)) - 1;
        if (g.word == 0) k0 |= v << g.shift; else k1 |= v << g.shift;
    }
}

template <int SINK>
__device__ __forceinline__ void apply_aggs(const gx_dplan &P, bool need_w0, long long r, Sink<SINK> &sink)
{
    if (need_w0 || SINK == SINK_RECORD) sink.inc(0);          // w0: rows in the group (count(*))
#pragma unroll
    for (int a = 0; a < GX_MAX_AGGS; a++) {
        if (a >= P.nagg) break;
        const gx_dagg &g = P.aggs[a];
        if (g.kind == GXU_NONE) continue;
        if (g.is_int) {
            if (gx_is_null(g.icol, r)) continue;
            if (g.kind == GXU_CNT) { sink.inc(g.word); continue; }
            sink.add_i64(g.word, gx_load_int(g.icol, r));     // int4_sum: widen to int8
            if (g.cnt_word) sink.inc(g.cnt_word);
        } else {
            bool isnull = false;
            double v = gx_eval_expr(g.expr, r, isnull);
            if (isnull) continue;                             // strict transition function
            if (g.kind == GXU_ADD_F64) sink.add_f64(g.word, v);
            else sink.minmax_f64(g.word, v, g.kind == GXU_MIN_F64);
            if (g.cnt_word) sink.inc(g.cnt_word);
        }
    }
}

template <int SINK>
__device__ __forceinline__ void consume_row(const gx_agg_dev &A, const SmemTable &T, long long r, unsigned long long payload, unsigned int cm = 0)
{
    unsigned long long k0, k1; unsigned int nullmask;
    pack_group_key(A.P, r, payload, k0, k1, nullmask);
    Sink<SINK> sink; sink.wstride = 1;
    // The table lookups below leave their probe loops at different iterations; without an explicit
    // reconvergence point the lanes then run the whole aggregate section in separate passes
    // (ncu, Q1 shape: 15 of 32 threads active per instruction).  cm = the lanes the caller KNOWS to be
    // in this call together (a ballot taken in warp-uniform code), 0 = unknown: no barrier.
    if (SINK == SINK_SMEM) {
        int s = smem_upsert<false>(T, k0, k1, nullmask);
        if (cm) __syncwarp(cm);
        if (s < 0) { atomicOr((unsigned long long *) &A.counters[1], 1ULL); return; }
        sink.w = T.w + (size_t) s * T.nwords;
    } else if (SINK == SINK_SMEM_LP) {
        int s = smem_upsert<true>(T, k0, k1, nullmask);
        if (cm) __syncwarp(cm);
        unsigned int gi = s < 0 ? 0xFFFFFFFFu : T.gidx[s];
        if (gi >= (unsigned) T.gmax) { atomicOr((unsigned long long *) &A.counters[1], 1ULL); return; }
        // [warp][word][group][lane]
        sink.wstride = T.gmax * 32;
        sink.w = T.w + ((size_t) (threadIdx.x >> 5) * T.nwords * T.gmax + gi) * 32 + (threadIdx.x & 31);
    } else if (SINK == SINK_GLOBAL) {
        unsigned long long *rec = global_upsert(A, k0, k1, nullmask);
        if (cm) __syncwarp(cm);
        if (!rec) { atomicOr((unsigned long long *) &A.counters[1], 2ULL); return; }
        sink.w = rec + 3;
    } else {
        const int RW = 3 + A.P.nwords;
        // warp-aggregated append: one atomic per converged group of lanes
        unsigned int am = __activemask();
        int leader = __ffs(am) - 1, lane = threadIdx.x & 31;
        long long idx = 0;
        if (lane == leader) idx = (long long) atomicAdd((unsigned long long *) &A.counters[2], (unsigned long long) __popc(am));
        idx = __shfl_sync(am, idx, leader) + __popc(am & ((1u << lane) - 1));
        if (idx >= A.rec_cap) { atomicOr((unsigned long long *) &A.counters[1], 4ULL); return; }
        unsigned long long *rec = A.recs + (size_t) idx * RW;
        rec[0] = nullmask; rec[1] = k0; rec[2] = k1;
        for (int i = 0; i < A.P.nwords; i++) rec[3 + i] = (unsigned long long) A.winit[i];
        sink.w = rec + 3;
    }
    apply_aggs<SINK>(A.P, A.need_w0 != 0, r, sink);
}

// merge a CTA's dense shared-memory table into the global table
__device__ __forceinline__ void smem_dense_merge(const SmemTable &T, const gx_agg_dev &A)
{
    for (int i = threadIdx.x; i < T.S; i += blockDim.x) {
        unsigned long long t = T.tag[i];
        if (t == 0) continue;
        unsigned int nullmask = (unsigned int) (t >> 59) & 0xF;
        unsigned long long k0 = T.tagkey ? (t & 0x00FFFFFFFFFFFFFFULL) : T.k0[i];
        unsigned long long *rec = global_upsert(A, k0, (!T.tagkey && T.nkw > 1) ? T.k1[i] : 0ULL, nullmask);
        if (!rec) { atomicOr((unsigned long long *) &A.counters[1], 2ULL); continue; }
        for (int j = 0; j < T.nwords; j++) merge_word(&rec[3 + j], A.wkind[j], T.w[(size_t) i * T.nwords + j]);
    }
}

// lane-private merge helper: combine one word over all warps and lanes of the CTA
__device__ __forceinline__ unsigned long long lp_reduce_word(const SmemTable &T, int nwarps, int word, unsigned int gi, int kind, int lane)
{
    unsigned long long acc = 0; bool first = true;
    for (int wp = 0; wp < nwarps; wp++) {
        unsigned long long v = T.w[(((size_t) wp * T.nwords + word) * T.gmax + gi) * 32 + lane];
        if (first) { acc = v; first = false; continue; }
        switch (kind) {
            case WK_ADD_I64: acc += v; break;
            case WK_ADD_F64: acc = (unsigned long long) __double_as_longlong(__dadd_rn(__longlong_as_double((long long) acc), __longlong_as_double((long long) v))); break;
            case WK_MIN_F64: if (gx_f8cmp(__longlong_as_double((long long) v), __longlong_as_double((long long) acc)) < 0) acc = v; break;
            default:         if (gx_f8cmp(__longlong_as_double((long long) v), __longlong_as_double((long long) acc)) > 0) acc = v; break;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        unsigned long long v = __shfl_down_sync(0xffffffffu, acc, o);
        switch (kind) {
            case WK_ADD_I64: acc += v; break;
            case WK_ADD_F64: acc = (unsigned long long) __double_as_longlong(__dadd_rn(__longlong_as_double((long long) acc), __longlong_as_double((long long) v))); break;
            case WK_MIN_F64: if (gx_f8cmp(__longlong_as_double((long long) v), __longlong_as_double((long long) acc)) < 0) acc = v; break;
            default:         if (gx_f8cmp(__longlong_as_double((long long) v), __longlong_as_double((long long) acc)) > 0) acc = v; break;
        }
    }
    return acc;                                   // valid in lane 0
}

template <int SINK>
__global__ void __launch_bounds__(1024, 1) gx_k_agg(const __grid_constant__ gx_agg_dev A)
{
    extern __shared__ unsigned long long smem[];
    constexpr bool IS_SMEM = SINK == SINK_SMEM || SINK == SINK_SMEM_LP;
    SmemTable T; T.S = A.s_slots; T.log2S = A.s_log2; T.nwords = A.P.nwords; T.nkw = A.P.nkw; T.tagkey = A.s_tagkey; T.gmax = A.s_gmax;
    T.tag = smem; T.k0 = T.tag + T.S; T.k1 = T.k0 + (T.tagkey ? 0 : T.S);
    unsigned long long *after_keys = T.k1 + ((!T.tagkey && A.P.nkw > 1) ? T.S : 0);
    T.gidx = nullptr; T.gcount = nullptr; T.w = after_keys;
    const int nwarps = blockDim.x >> 5;
    if (SINK == SINK_SMEM) {
        for (int i = threadIdx.x; i < T.S; i += blockDim.x) {
            T.tag[i] = 0;
            for (int j = 0; j < T.nwords; j++) T.w[(size_t) i * T.nwords + j] = (unsigned long long) A.winit[j];
        }
        __syncthreads();
    } else if (SINK == SINK_SMEM_LP) {
        T.gidx = (unsigned int *) after_keys;                       // S entries (+ the counter), padded to 8 bytes
        T.gcount = T.gidx + T.S;
        T.w = after_keys + (T.S + 2) / 2 + 1;
        for (int i = threadIdx.x; i < T.S; i += blockDim.x) T.tag[i] = 0;
        if (threadIdx.x == 0) *T.gcount = 0;
        const int per_warp = T.nwords * T.gmax * 32;
        for (int i = threadIdx.x; i < per_warp * nwarps; i += blockDim.x) {
            int word = (i % per_warp) / (T.gmax * 32);
            T.w[i] = (unsigned long long) A.winit[word];
        }
        __syncthreads();
    }
    const gx_dplan &P = A.P;
    long long stride = (long long) gridDim.x * blockDim.x;
    // warp-uniform loop: every lane of a warp makes the same number of trips (lanes past the end idle)
    const int lane = threadIdx.x & 31;
    for (long long r = A.row0 + (long long) blockIdx.x * blockDim.x + threadIdx.x; r - lane < A.row1; r += stride) {
        bool ok = r < A.row1;
#pragma unroll
        for (int p = 0; p < GX_MAX_PREDS; p++) if (p < P.npreds) ok = ok && gx_eval_pred(P.preds[p], ok ? r : A.row0);
        if (!P.has_join) {
            // exactly the lanes that consume a row now; the barrier only pays when a row has several
            // state words to update (with one counter it cost 20 % on the config-1 shape)
            const unsigned int m = P.nwords >= 3 ? __ballot_sync(0xffffffffu, ok) : 0u;
            if (ok) consume_row<SINK>(A, T, r, 0ULL, m);
            continue;
        }
        if (!ok) continue;
        if (gx_is_null(P.okey, r)) continue;                  // NULL outer key never joins
        long long key = gx_load_int(P.okey, r);
        if (key == GX_EMPTY_KEY) {
            for (int i = 0; i < A.special_count; i++) { consume_row<SINK>(A, T, r, A.special[i]); if (P.unique) break; }
            continue;
        }
        unsigned long long s = gx_slot_index(key, A.sf);
        for (;;) {
            gx_slot sl = A.slots[s];
            if (sl.key == GX_EMPTY_KEY) break;
            if (sl.key == key) { consume_row<SINK>(A, T, r, sl.payload); if (P.unique) break; }
            s = gx_next_slot(s, A.mask);
        }
    }
    if (!IS_SMEM) return;
    __syncthreads();
    // merge the CTA's table into the global one
    if (SINK == SINK_SMEM) {
        smem_dense_merge(T, A);
    } else {
        const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
        for (int i = wid; i < T.S; i += nwarps) {              // one warp per directory slot
            unsigned long long t = T.tag[i];
            if (t == 0) continue;
            unsigned int gi = T.gidx[i];
            if (gi >= (unsigned) T.gmax) continue;             // overflow already flagged
            unsigned int nullmask = (unsigned int) (t >> 59) & 0xF;
            unsigned long long k0 = T.tagkey ? (t & 0x00FFFFFFFFFFFFFFULL) : T.k0[i];
            unsigned long long *rec = nullptr;
            if (lane == 0) rec = global_upsert(A, k0, (!T.tagkey && T.nkw > 1) ? T.k1[i] : 0ULL, nullmask);
            for (int j = 0; j < T.nwords; j++) {
                unsigned long long v = lp_reduce_word(T, nwarps, j, gi, A.wkind[j], lane);
                if (lane == 0) { if (rec) merge_word(&rec[3 + j], A.wkind[j], v); else atomicOr((unsigned long long *) &A.counters[1], 2ULL); }
            }
        }
    }
}

// ---------------------------------------------------------------------------
// Few groups, many float8 aggregates, no join (the Q1 shape): lane-private accumulators as in
// gx_k_agg<SINK_SMEM_LP>, but the plan is walked once per TILE of LPT_K x 32 rows instead of
// once per row.  A lane holds LPT_K rows; for every aggregate the expression descriptor is
// decoded once and its terms are evaluated for the lane's LPT_K rows back to back (LPT_K
// independent loads in flight per term), then added to the rows' accumulators.  ncu on the
// row-at-a-time interpreter: 1000 warp instructions per 32 rows and 14 warps per SM with
// nothing to overlap the column loads (profiles/r01_bench_configs_sf100.json).
// Plan shape (checked by the host): no join, every aggregate is count(*) or a sum/avg over a
// chain expression of NOT-NULL float8 columns and constants.
// LPT_K = rows per lane and tile: 8 when the CTA is small enough for the registers (<= 640 threads), else 4
template <int LPT_K>
__device__ __forceinline__ void lpt_term(const gx_dterm &t, const long long (&r)[LPT_K], const bool (&ok)[LPT_K], double (&out)[LPT_K])
{
    const double *c = (const double *) t.col.data;
    const double k = t.k;
    if (t.kind == GXT_CONST) {
#pragma unroll
        for (int j = 0; j < LPT_K; j++) out[j] = k;
        return;
    }
    double x[LPT_K];
#pragma unroll
    for (int j = 0; j < LPT_K; j++) x[j] = ok[j] ? __ldg(c + r[j]) : 0.0;
    switch (t.kind) {
        case GXT_COL:
#pragma unroll
            for (int j = 0; j < LPT_K; j++) out[j] = x[j];
            break;
        case GXT_K_SUB_COL:
#pragma unroll
            for (int j = 0; j < LPT_K; j++) out[j] = __dsub_rn(k, x[j]);
            break;
        case GXT_K_ADD_COL:
#pragma unroll
            for (int j = 0; j < LPT_K; j++) out[j] = __dadd_rn(k, x[j]);
            break;
        case GXT_K_MUL_COL:
#pragma unroll
            for (int j = 0; j < LPT_K; j++) out[j] = __dmul_rn(k, x[j]);
            break;
        default:                                               // GXT_COL_SUB_K
#pragma unroll
            for (int j = 0; j < LPT_K; j++) out[j] = __dsub_rn(x[j], k);
            break;
    }
}

template <int LPT_K>
__global__ void __launch_bounds__(LPT_K == 8 ? 640 : 1024, 1) gx_k_agg_lptile(const __grid_constant__ gx_agg_dev A)
{
    extern __shared__ unsigned long long smem[];
    SmemTable T; T.S = A.s_slots; T.log2S = A.s_log2; T.nwords = A.P.nwords; T.nkw = A.P.nkw; T.tagkey = A.s_tagkey; T.gmax = A.s_gmax;
    T.tag = smem; T.k0 = T.tag + T.S; T.k1 = T.k0 + (T.tagkey ? 0 : T.S);
    unsigned long long *after_keys = T.k1 + ((!T.tagkey && A.P.nkw > 1) ? T.S : 0);
    T.gidx = (unsigned int *) after_keys;                       // same layout as gx_k_agg<SINK_SMEM_LP>
    T.gcount = T.gidx + T.S;
    T.w = after_keys + (T.S + 2) / 2 + 1;
    const int nwarps = blockDim.x >> 5, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int i = threadIdx.x; i < T.S; i += blockDim.x) T.tag[i] = 0;
    if (threadIdx.x == 0) *T.gcount = 0;
    {
        const int per_warp = T.nwords * T.gmax * 32;
        for (int i = threadIdx.x; i < per_warp * nwarps; i += blockDim.x) T.w[i] = (unsigned long long) A.winit[(i % per_warp) / (T.gmax * 32)];
    }
    __syncthreads();
    const gx_dplan &P = A.P;
    const int wstride = T.gmax * 32;
    unsigned long long *const wbase = T.w + (size_t) warp * T.nwords * T.gmax * 32 + lane;    // + gi * 32 + word * wstride
    const long long tile = 32LL * LPT_K, step = (long long) gridDim.x * nwarps * tile;
    for (long long base = A.row0 + ((long long) blockIdx.x * nwarps + warp) * tile; base < A.row1; base += step) {
        long long r[LPT_K]; bool ok[LPT_K]; unsigned long long *acc[LPT_K];
#pragma unroll
        for (int j = 0; j < LPT_K; j++) { r[j] = base + j * 32 + lane; ok[j] = r[j] < A.row1; acc[j] = wbase; }
        for (int p = 0; p < P.npreds; p++) {
#pragma unroll
            for (int j = 0; j < LPT_K; j++) if (ok[j]) ok[j] = gx_eval_pred(P.preds[p], r[j]);
        }
#pragma unroll
        for (int j = 0; j < LPT_K; j++) {
            if (!ok[j]) continue;
            unsigned long long k0, k1; unsigned int nullmask;
            pack_group_key(P, r[j], 0ULL, k0, k1, nullmask);
            const int s = smem_upsert<true>(T, k0, k1, nullmask);
            const unsigned int gi = s < 0 ? 0xFFFFFFFFu : T.gidx[s];
            if (gi >= (unsigned) T.gmax) { atomicOr((unsigned long long *) &A.counters[1], 1ULL); ok[j] = false; }
            else acc[j] = wbase + (size_t) gi * 32;
        }
        __syncwarp();                                          // the lookups leave their probe loops at different times
        if (A.need_w0) {
#pragma unroll
            for (int j = 0; j < LPT_K; j++) if (ok[j]) acc[j][0] += 1ULL;
        }
        for (int a = 0; a < P.nagg; a++) {
            const gx_dagg &g = P.aggs[a];
            if (g.kind == GXU_NONE) continue;
            double v[LPT_K];
            lpt_term<LPT_K>(g.expr.t[0], r, ok, v);
            for (int i = 1; i < g.expr.nterms; i++) {
                double x[LPT_K];
                lpt_term<LPT_K>(g.expr.t[i], r, ok, x);
                const int op = g.expr.t[i].op;
                if (op == GX_OP_ADD) {
#pragma unroll
                    for (int j = 0; j < LPT_K; j++) v[j] = __dadd_rn(v[j], x[j]);
                } else if (op == GX_OP_SUB) {
#pragma unroll
                    for (int j = 0; j < LPT_K; j++) v[j] = __dsub_rn(v[j], x[j]);
                } else {
#pragma unroll
                    for (int j = 0; j < LPT_K; j++) v[j] = __dmul_rn(v[j], x[j]);
                }
            }
            const int wo = g.word * wstride;
#pragma unroll
            for (int j = 0; j < LPT_K; j++) if (ok[j]) { double *pp = (double *) (acc[j] + wo); *pp = __dadd_rn(*pp, v[j]); }
        }
    }
    __syncthreads();
    for (int i = warp; i < T.S; i += nwarps) {                 // one warp per directory slot, as in gx_k_agg
        unsigned long long t = T.tag[i];
        if (t == 0) continue;
        unsigned int gi = T.gidx[i];
        if (gi >= (unsigned) T.gmax) continue;
        unsigned int nullmask = (unsigned int) (t >> 59) & 0xF;
        unsigned long long k0 = T.tagkey ? (t & 0x00FFFFFFFFFFFFFFULL) : T.k0[i];
        unsigned long long *rec = nullptr;
        if (lane == 0) rec = global_upsert(A, k0, (!T.tagkey && T.nkw > 1) ? T.k1[i] : 0ULL, nullmask);
        for (int j = 0; j < T.nwords; j++) {
            unsigned long long v = lp_reduce_word(T, nwarps, j, gi, A.wkind[j], lane);
            if (lane == 0) { if (rec) merge_word(&rec[3 + j], A.wkind[j], v); else atomicOr((unsigned long long *) &A.counters[1], 2ULL); }
        }
    }
}

// ---------------------------------------------------------------------------
// A handful of groups (<= FG_G), no join: the Q1 shape and config 1.  The accumulators live in
// REGISTERS: a thread keeps (row count, FG_NV float8 sums) for each of the FG_G groups the CTA
// has discovered, every row adds to the accumulators of its group through predicated adds
// (adding nothing to the other groups), and the threads' accumulators meet once, at the end
// (warp shuffles -> one shared-memory table per CTA -> the global table).  Against the
// lane-private shared-memory accumulators of gx_k_agg_lptile this needs no shared memory per
// lane (full occupancy instead of 18 warps/SM) and no load-add-store per word and row.
// The group directory is a FG_G-entry list in shared memory, claimed with a CAS on first
// sight of a key; a (FG_G+1)-th key raises the overflow flag and the host retries with the
// general kernels — the result never depends on the estimate.
// Plan shape (checked by the host): no join; group key <= 8 bytes without NULLs; aggregates are
// count(*) or sum/avg over chain expressions of NOT-NULL float8 columns and constants.
#define FG_G  4
#define FG_NV 5
/* FG_K = rows per lane and tile (independent loads in flight; the plan walk is paid once per tile) and the CTA size are
 * template parameters of gx_k_fewgroups: <8, 512> (128 registers, 16 warps/SM) and <4, 768> (85 registers, 24 warps/SM) */
#define FG_NC 4                         /* distinct float8 columns the aggregate arguments may read */
struct gx_fewgroups_args {
    int nv, nc;
    const double *col[FG_NC];           // the distinct argument columns: loaded ONCE per row into registers
    int vagg[FG_NV], vword[FG_NV];
    signed char tslot[FG_NV][4];        // column slot of term t of value w (-1: constant)
};

__device__ __forceinline__ int fg_insert(unsigned long long *s_keys, unsigned int *s_state, unsigned long long key)
{
    for (int gI = 0; gI < FG_G; gI++) {
        for (;;) {
            const unsigned int st = *(volatile unsigned int *) &s_state[gI];
            if (st == 2u) { if (*(volatile unsigned long long *) &s_keys[gI] == key) return gI; break; }
            if (st == 0u && atomicCAS(&s_state[gI], 0u, 1u) == 0u) {
                *(volatile unsigned long long *) &s_keys[gI] = key;
                __threadfence_block();
                *(volatile unsigned int *) &s_state[gI] = 2u;
                return gI;
            }
        }
    }
    return -1;
}

// one term of a chain expression over a register tile
template <int K>
__device__ __forceinline__ void reg_term(int kind, double k, const double (&x)[K], double (&out)[K])
{
    switch (kind) {
        case GXT_COL:
#pragma unroll
            for (int j = 0; j < K; j++) out[j] = x[j];
            break;
        case GXT_K_SUB_COL:
#pragma unroll
            for (int j = 0; j < K; j++) out[j] = __dsub_rn(k, x[j]);
            break;
        case GXT_K_ADD_COL:
#pragma unroll
            for (int j = 0; j < K; j++) out[j] = __dadd_rn(k, x[j]);
            break;
        case GXT_K_MUL_COL:
#pragma unroll
            for (int j = 0; j < K; j++) out[j] = __dmul_rn(k, x[j]);
            break;
        default:                                               // GXT_COL_SUB_K
#pragma unroll
            for (int j = 0; j < K; j++) out[j] = __dsub_rn(x[j], k);
            break;
    }
}
template <int K, int NC>
__device__ __forceinline__ void slot_term(const gx_dterm &t, int slot, const double (&x)[NC][K], double (&out)[K])
{
    if (slot < 0) {
#pragma unroll
        for (int j = 0; j < K; j++) out[j] = t.k;
        return;
    }
    // warp-uniform: picks the register tile of the column
    if (slot == 0 || NC == 1) reg_term<K>(t.kind, t.k, x[0], out);
    else if (slot == 1 || NC == 2) reg_term<K>(t.kind, t.k, x[NC > 1 ? 1 : 0], out);
    else if (slot == 2 || NC == 3) reg_term<K>(t.kind, t.k, x[NC > 2 ? 2 : 0], out);
    else reg_term<K>(t.kind, t.k, x[NC > 3 ? 3 : 0], out);
}

// BYTEKEY: the group key is one or two 1-byte columns without NULLs (Q1: l_returnflag, l_linestatus) — packed with
// two byte loads instead of the generic column walk.
template <bool BYTEKEY, int FG_K, int FG_THREADS>
__global__ void __launch_bounds__(FG_THREADS, 1) gx_k_fewgroups(const __grid_constant__ gx_agg_dev A, const __grid_constant__ gx_fewgroups_args F)
{
    extern __shared__ unsigned long long fg_smem[];            // [warp][word][group][lane]: a lane's own accumulators (bank == lane)
    __shared__ unsigned long long s_keys[FG_G];
    __shared__ unsigned int s_state[FG_G];
    __shared__ unsigned long long s_acc[FG_G][1 + FG_NV];
    __shared__ int s_over;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nv = F.nv, nw = 1 + nv;
    if (threadIdx.x < FG_G) { s_state[threadIdx.x] = 0u; s_keys[threadIdx.x] = 0ULL; }
    if (threadIdx.x < FG_G * (1 + FG_NV)) ((unsigned long long *) s_acc)[threadIdx.x] = 0ULL;
    if (threadIdx.x == 0) s_over = 0;
    // group slot FG_G is a trash can: rows that fail the quals are added there, so the tile body has no per-row branches
    constexpr int GS = FG_G + 1;
    unsigned long long *const acc = fg_smem + (size_t) warp * nw * GS * 32 + lane;     // + (word * GS + group) * 32
    for (int i = 0; i < nw * GS; i++) acc[i * 32] = 0ULL;
    __syncthreads();
    const gx_dplan &P = A.P;
    // keys the CTA has handed out so far; an unused entry holds a value no packed key can take (BYTEKEY keys are
    // below 2^16; the generic path also checks the valid bit)
    unsigned long long gk[FG_G]; unsigned int gvalid = 0u;
#pragma unroll
    for (int gI = 0; gI < FG_G; gI++) gk[gI] = ~0ULL;
    const unsigned char *kc0 = (const unsigned char *) P.gcols[0].col.data, *kc1 = (const unsigned char *) P.gcols[P.ngroup > 1 ? 1 : 0].col.data;
    const int two = P.ngroup > 1, sh1 = P.gcols[P.ngroup > 1 ? 1 : 0].shift;
    const long long tile = 32LL * FG_K, nwarp_total = (long long) gridDim.x * (blockDim.x >> 5);
    const long long wid = (long long) blockIdx.x * (blockDim.x >> 5) + warp;
    bool stop = false;
    // FULL = every row of the tile exists: loads and arithmetic are unconditional (the compiler sees no row predicate)
    auto tile_body = [&](long long base, auto FULL) {
        constexpr bool full = decltype(FULL)::value;
        long long r[FG_K]; bool ok[FG_K]; int gi[FG_K];
#pragma unroll
        for (int j = 0; j < FG_K; j++) { r[j] = base + j * 32 + lane; ok[j] = full || r[j] < A.row1; }
        // ---- every column the tile needs is requested before anything is used: argument columns first (no use
        // until the arithmetic below), then the group columns, then the qual columns
        double x[FG_NC][FG_K];
#pragma unroll
        for (int c = 0; c < FG_NC; c++) {
            const double *pc = F.col[c < F.nc ? c : 0] + base + lane;      // row j of the tile sits at a compile-time offset
            if (c < F.nc) {
#pragma unroll
                for (int j = 0; j < FG_K; j++) x[c][j] = (full || ok[j]) ? __ldg(pc + j * 32) : 0.0;
            } else {
#pragma unroll
                for (int j = 0; j < FG_K; j++) x[c][j] = 0.0;
            }
        }
        unsigned long long key[FG_K];
        if (BYTEKEY) {
            unsigned int b0[FG_K], b1[FG_K];
            const unsigned char *p0 = kc0 + base + lane, *p1 = kc1 + base + lane;
#pragma unroll
            for (int j = 0; j < FG_K; j++) { b0[j] = (full || ok[j]) ? __ldg(p0 + j * 32) : 0u; b1[j] = (two && (full || ok[j])) ? __ldg(p1 + j * 32) : 0u; }
#pragma unroll
            for (int j = 0; j < FG_K; j++) key[j] = (unsigned long long) (b0[j] | (b1[j] << sh1));
        } else {
#pragma unroll
            for (int j = 0; j < FG_K; j++) { unsigned long long k0 = 0, k1; unsigned int nm; if (ok[j]) pack_group_key(P, r[j], 0ULL, k0, k1, nm); key[j] = k0; }
        }
        for (int p = 0; p < P.npreds; p++) pred_tile<FG_K>(P.preds[p], r, ok);
        // group of every row: compare with the keys this CTA knows
        bool miss = false;
#pragma unroll
        for (int j = 0; j < FG_K; j++) {
            gi[j] = -1;
            if (BYTEKEY) {
#pragma unroll
                for (int gI = 0; gI < FG_G; gI++) if ((unsigned int) key[j] == (unsigned int) gk[gI]) gi[j] = gI;      // 32-bit compare; unused entries hold 0xffffffff
            } else {
#pragma unroll
                for (int gI = 0; gI < FG_G; gI++) if (((gvalid >> gI) & 1u) && key[j] == gk[gI]) gi[j] = gI;
            }
            miss |= ok[j] && gi[j] < 0;
        }
        if (__any_sync(0xffffffffu, miss)) {                       // first sight of a key (a handful of times per CTA)
#pragma unroll
            for (int j = 0; j < FG_K; j++) if (ok[j] && gi[j] < 0) { gi[j] = fg_insert(s_keys, s_state, key[j]); if (gi[j] < 0) { s_over = 1; ok[j] = false; } }
            __syncwarp();
#pragma unroll
            for (int gI = 0; gI < FG_G; gI++) if (*(volatile unsigned int *) &s_state[gI] == 2u) { gk[gI] = *(volatile unsigned long long *) &s_keys[gI]; gvalid |= 1u << gI; }
            if (*(volatile int *) &s_over) { stop = true; return; }    // more groups than accumulators: the host takes the general path
        }
        // ---- accumulate: word 0 = rows, word 1 + w = sum of value w; [word][group][lane], a lane touches only its own column
        unsigned long long *ap[FG_K];
#pragma unroll
        for (int j = 0; j < FG_K; j++) { ap[j] = acc + (size_t) ((ok[j] && gi[j] >= 0) ? gi[j] : FG_G) * 32; *ap[j] += 1ULL; }
#pragma unroll
        for (int w = 0; w < FG_NV; w++) {
            if (w >= nv) break;
            const gx_dexpr &e = P.aggs[F.vagg[w]].expr;
            double v[FG_K];
            slot_term<FG_K, FG_NC>(e.t[0], F.tslot[w][0], x, v);
            for (int i = 1; i < e.nterms; i++) {
                double y[FG_K];
                slot_term<FG_K, FG_NC>(e.t[i], F.tslot[w][i], x, y);
                const int op = e.t[i].op;
                if (op == GX_OP_ADD) {
#pragma unroll
                    for (int j = 0; j < FG_K; j++) v[j] = __dadd_rn(v[j], y[j]);
                } else if (op == GX_OP_SUB) {
#pragma unroll
                    for (int j = 0; j < FG_K; j++) v[j] = __dsub_rn(v[j], y[j]);
                } else {
#pragma unroll
                    for (int j = 0; j < FG_K; j++) v[j] = __dmul_rn(v[j], y[j]);
                }
            }
#pragma unroll
            for (int j = 0; j < FG_K; j++) { double *pp = (double *) (ap[j] + (size_t) (1 + w) * GS * 32); *pp = __dadd_rn(*pp, v[j]); }
        }
    };
    for (long long base = A.row0 + wid * tile; base < A.row1 && !stop; base += nwarp_total * tile) {
        if (*(volatile int *) &s_over) break;
        if (base + tile <= A.row1) tile_body(base, std::true_type());
        else tile_body(base, std::false_type());
    }
    // ---- lanes -> warp -> CTA -> global table
    __syncwarp();
    for (int i = 0; i < nw * GS; i++) {
        const int word = i / GS, gI = i % GS;
        if (gI == FG_G) continue;                                  // the trash can
        unsigned long long raw = acc[i * 32];
        if (word == 0) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) raw += __shfl_down_sync(0xffffffffu, raw, o);
            if (lane == 0 && raw) atomicAdd(&s_acc[gI][0], raw);
        } else {
            double xx = __longlong_as_double((long long) raw);
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) xx = __dadd_rn(xx, __shfl_down_sync(0xffffffffu, xx, o));
            if (lane == 0) atomicAdd((double *) &s_acc[gI][word], xx);
        }
    }
    __syncthreads();
    if (s_over) { if (threadIdx.x == 0) atomicOr((unsigned long long *) &A.counters[1], 1ULL); return; }
    if (threadIdx.x < FG_G && s_state[threadIdx.x] == 2u && s_acc[threadIdx.x][0] != 0ULL) {
        unsigned long long *rec = global_upsert(A, s_keys[threadIdx.x], 0ULL, 0u);
        if (!rec) { atomicOr((unsigned long long *) &A.counters[1], 2ULL); return; }
        atomicAdd(&rec[3], s_acc[threadIdx.x][0]);
        for (int w = 0; w < nv; w++) atomicAdd((double *) &rec[3 + F.vword[w]], __longlong_as_double((long long) s_acc[threadIdx.x][1 + w]));
    }
}

// config 1's shape exactly: count(*) GROUP BY one 1-byte column, no quals.  16 rows per 128-bit load; every byte is
// compared with the (<= 8) keys the CTA knows four bytes at a time (exact zero-byte test of word ^ replicated key:
// 0x80 in every matching byte), matches are counted with a population count.  1 B/row of traffic.  The key list is
// claimed with a single compare-and-swap per new key (0 = free, 0x100 | byte = taken): no lock, nothing spins.
#define CC_G 8
// a byte value this thread has not seen: claim / find it in the CTA's list; returns the number of keys now known
// (the ready slots form a prefix), or -1 when a ninth distinct value turns up
__device__ __noinline__ int cc_learn(unsigned int *s_keys, unsigned int w, unsigned int unseen)
{
    for (int b = 0; b < 4; b++) {
        if (!((unseen >> (8 * b)) & 0x80u)) continue;
        const unsigned int want = 0x100u | ((w >> (8 * b)) & 0xffu);
        int gI = 0;
        for (; gI < CC_G; gI++) {
            unsigned int cur = *(volatile unsigned int *) &s_keys[gI];
            if (cur == 0u) { cur = atomicCAS(&s_keys[gI], 0u, want); if (cur == 0u) cur = want; }
            if (cur == want) break;
        }
        if (gI == CC_G) return -1;
    }
    int n = 0;
    while (n < CC_G && *(volatile unsigned int *) &s_keys[n] != 0u) n++;
    return n;
}
__global__ void __launch_bounds__(512, 2) gx_k_count_char(const __grid_constant__ gx_agg_dev A, const signed char *__restrict__ col)
{
    __shared__ unsigned int s_keys[CC_G];
    __shared__ unsigned long long s_cnt[CC_G];
    __shared__ int s_over;
    if (threadIdx.x < CC_G) { s_keys[threadIdx.x] = 0u; s_cnt[threadIdx.x] = 0ULL; }
    if (threadIdx.x == 0) s_over = 0;
    __syncthreads();
    unsigned int cnt[CC_G], rep[CC_G];
    int ngk = 0;                                                    // keys this thread knows: a prefix of the CTA's list
#pragma unroll
    for (int gI = 0; gI < CC_G; gI++) { cnt[gI] = 0u; rep[gI] = 0u; }
    // bytes of w equal to the replicated key: 0x80 in every matching byte
    auto eqmask = [](unsigned int w, unsigned int rp) -> unsigned int { const unsigned int x = w ^ rp; return ~(((x & 0x7f7f7f7fu) + 0x7f7f7f7fu) | x | 0x7f7f7f7fu); };
    auto count_word = [&](unsigned int w, unsigned int keep /* 0x80 per byte that is a row */) {
        unsigned int seen = 0u;
#pragma unroll
        for (int gI = 0; gI < CC_G; gI++) {
            if (gI >= ngk) break;
            const unsigned int m = eqmask(w, rep[gI]) & keep;
            cnt[gI] += (unsigned int) __popc(m); seen |= m;
        }
        if (seen != keep) {                                        // rare: a value not seen by this thread before
            const unsigned int todo = keep & ~seen;
            const int n = cc_learn(s_keys, w, todo);
            if (n < 0) { s_over = 1; return; }
            const int old = ngk;
            ngk = n;
#pragma unroll
            for (int gI = 0; gI < CC_G; gI++) {
                if (gI >= ngk) break;
                if (gI >= old) rep[gI] = (s_keys[gI] & 0xffu) * 0x01010101u;
                if (gI >= old) cnt[gI] += (unsigned int) __popc(eqmask(w, rep[gI]) & todo);
            }
        }
    };
    const long long n = A.row1 - A.row0;
    const signed char *p0 = col + A.row0;
    // head: bytes up to the first 16-byte boundary; body: vectors; tail: the rest
    long long head = (long long) ((16 - ((unsigned long long) p0 & 15ULL)) & 15ULL); if (head > n) head = n;
    const long long nvec = (n - head) >> 4, tail0 = head + (nvec << 4);
    const long long tid = (long long) blockIdx.x * blockDim.x + threadIdx.x;
    if (tid < head) count_word((unsigned int) (unsigned char) p0[tid], 0x80u);
    if (tid < n - tail0) count_word((unsigned int) (unsigned char) p0[tail0 + tid], 0x80u);
    const uint4 *pv = (const uint4 *) (p0 + head);
    // a CTA reads one contiguous range of vectors, its threads two vectors at a time
    const long long per = (nvec + gridDim.x - 1) / gridDim.x, v0 = per * blockIdx.x, v1 = v0 + per < nvec ? v0 + per : nvec;
    for (long long i = v0 + threadIdx.x; i < v1; i += 2 * blockDim.x) {
        uint4 v, u = make_uint4(0, 0, 0, 0);
        const bool two = i + blockDim.x < v1;
        asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(pv + i));
        if (two) asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(u.x), "=r"(u.y), "=r"(u.z), "=r"(u.w) : "l"(pv + i + blockDim.x));
        count_word(v.x, 0x80808080u); count_word(v.y, 0x80808080u); count_word(v.z, 0x80808080u); count_word(v.w, 0x80808080u);
        if (two) { count_word(u.x, 0x80808080u); count_word(u.y, 0x80808080u); count_word(u.z, 0x80808080u); count_word(u.w, 0x80808080u); }
        if (*(volatile int *) &s_over) break;
    }
    const int lane = threadIdx.x & 31;                             // list positions are the CTA's: every thread counts key g in cnt[g]
#pragma unroll
    for (int gI = 0; gI < CC_G; gI++) {
        unsigned long long c = cnt[gI];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) c += __shfl_down_sync(0xffffffffu, c, o);
        if (lane == 0 && c) atomicAdd(&s_cnt[gI], c);
    }
    __syncthreads();
    if (s_over) { if (threadIdx.x == 0) atomicOr((unsigned long long *) &A.counters[1], 1ULL); return; }
    if (threadIdx.x < CC_G && s_keys[threadIdx.x] != 0u && s_cnt[threadIdx.x]) {
        // group key = the byte the way pack_group_key packs a 1-byte column
        unsigned long long *rec = global_upsert(A, (unsigned long long) (s_keys[threadIdx.x] & 0xffu), 0ULL, 0u);
        if (!rec) { atomicOr((unsigned long long *) &A.counters[1], 2ULL); return; }
        atomicAdd(&rec[3], s_cnt[threadIdx.x]);
    }
}

// ---------------------------------------------------------------------------
// Specialised kernel for the dominant plan shape (BASELINE configs 2 and 3):
//   [probe a unique-key join table with an int8 key ->] GROUP BY one 4-byte
//   column (a scanned int4/date column, or the 4-byte join payload), aggregates
//   drawn from { count(*), sum/avg(one float8 column) }, no quals, no NULLs.
// The generic kernel above interprets the plan per row (~220-580 instructions
// per row measured with ncu, profiles/r01_ncu_generic_kernel.txt): this one is
// what the same plan compiles to by hand.  Four consecutive rows per thread:
// 16-byte vector loads, four independent table probes in flight, equal
// neighbouring keys probed once (TPC-H lineitem is clustered on the order key)
// and their rows pre-combined in registers before touching shared memory.
struct gx_fast_args {
    const long long *okey;      // JOIN: outer key column (int8)
    const int *gcol;            // !JOIN: group column (int4/date)
    const double *vcol;         // value column of sum/avg (may be NULL)
    int sum_word;               // state word of the sum
    int pf;                     // gx_k_runjoin: 1/2 = prefetch the join-table lines of a tile into L2/L1 before its runs are folded
};

__device__ __forceinline__ longlong2 ld_stream_ll2(const long long *p)
{
    longlong2 v;
    asm volatile("ld.global.nc.L1::no_allocate.v2.s64 {%0, %1}, [%2];" : "=l"(v.x), "=l"(v.y) : "l"(p));
    return v;
}
__device__ __forceinline__ double2 ld_stream_d2(const double *p)
{
    double2 v;
    asm volatile("ld.global.nc.L1::no_allocate.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "l"(p));
    return v;
}
__device__ __forceinline__ int4 ld_stream_i4(const int *p)
{
    int4 v;
    asm volatile("ld.global.nc.L1::no_allocate.v4.s32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
    return v;
}
// two neighbouring slots (one aligned 32-byte sector) with a single 256-bit load
struct gx_slot2 { long long k0; unsigned long long p0; long long k1; unsigned long long p1; };
__device__ __forceinline__ gx_slot2 ld_slot2(const gx_slot *p)
{
    gx_slot2 s;
    asm volatile("ld.global.v4.u64 {%0, %1, %2, %3}, [%4];" : "=l"(s.k0), "=l"(s.p0), "=l"(s.k1), "=l"(s.p1) : "l"(p));
    return s;
}
__device__ __forceinline__ gx_slot ld_slot(const gx_slot *p)
{
    gx_slot s;
    asm volatile("ld.global.v2.u64 {%0, %1}, [%2];" : "=l"(s.key), "=l"(s.payload) : "l"(p));
    return s;
}

// Group-table update of the specialised kernel.  The key is one 4-byte value and the tag
// word holds it whole, so the slot is taken from the key's low bits directly: dates, codes
// and other dense domains then map without any collision (2406 consecutive dates into 4096
// slots), anything else falls back on linear probing; a table that still overflows is
// caught by the generic retry logic of gx_hash_agg.
template <bool HAS_CNT, bool HAS_SUM>
__device__ __forceinline__ void fast_flush(const SmemTable &T, const gx_agg_dev &A, int gkey, unsigned int cnt, double sum, int sum_word)
{
    const unsigned long long tag = (1ULL << 63) | (unsigned long long) (unsigned int) gkey;
    int s = (int) ((unsigned int) gkey & (unsigned int) (T.S - 1));
    int n = 0;
    for (;;) {
        unsigned long long t = *(volatile unsigned long long *) &T.tag[s];
        if (t == tag) break;
        if (t == 0) { unsigned long long old = atomicCAS(&T.tag[s], 0ULL, tag); if (old == 0 || old == tag) break; }
        s = (s + 1) & (T.S - 1);
        if (++n >= 64) { atomicOr((unsigned long long *) &A.counters[1], 1ULL); return; }
    }
    unsigned long long *w = T.w + (size_t) s * T.nwords;
    if (HAS_CNT) atomicAdd((unsigned int *) &w[0], cnt);
    if (HAS_SUM) atomicAdd((double *) &w[sum_word], sum);
}

template <bool JOIN, bool HAS_CNT, bool HAS_SUM>
__global__ void __launch_bounds__(1024, 1) gx_k_fast(const __grid_constant__ gx_agg_dev A, const gx_fast_args F)
{
    extern __shared__ unsigned long long smem[];
    SmemTable T; T.S = A.s_slots; T.log2S = A.s_log2; T.nwords = A.P.nwords; T.nkw = 1; T.tagkey = 1; T.gmax = 0;
    T.tag = smem; T.k0 = T.tag + T.S; T.k1 = T.k0; T.w = T.k0; T.gidx = nullptr; T.gcount = nullptr;
    for (int i = threadIdx.x; i < T.S; i += blockDim.x) {
        T.tag[i] = 0;
        for (int j = 0; j < T.nwords; j++) T.w[(size_t) i * T.nwords + j] = (unsigned long long) A.winit[j];
    }
    __syncthreads();
    const long long nvec = (A.row1 - A.row0) >> 2;              // groups of four rows
    const long long stride = (long long) gridDim.x * blockDim.x;
    for (long long q = (long long) blockIdx.x * blockDim.x + threadIdx.x; q < nvec; q += stride) {
        const long long r = A.row0 + (q << 2);
        int g[4]; bool hit[4]; double v[4];
        unsigned int rcnt = 0; double rsum = 0.0;                     // partial handed over by the lane above
        if (HAS_SUM) { double2 a = ld_stream_d2(F.vcol + r), b = ld_stream_d2(F.vcol + r + 2); v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y; }
        if (JOIN) {
            longlong2 ka = ld_stream_ll2(F.okey + r), kb = ld_stream_ll2(F.okey + r + 2);
            long long k[4] = { ka.x, ka.y, kb.x, kb.y };
            gx_slot2 sl[4];
            // A run of equal keys that started in the previous lane is not probed again:
            // ncu showed such cross-lane repeats re-fetching their sector from DRAM
            // (profiles/r01_ncu_fast_probe_and_bucket_build_sf100.csv).
            const unsigned int wmask = __activemask();
            const int lane = threadIdx.x & 31;
            long long prevk = __shfl_up_sync(wmask, k[3], 1);
            const bool lead_dup = lane > 0 && ((wmask >> (lane - 1)) & 1u) && k[0] == prevk;
            // a leading run that ends inside this lane is handed to the lane below as a partial
            // (count, sum): that lane has probed the key and does the one group update
            const bool give = lead_dup && k[3] != k[0];
            // first probe of every distinct neighbour: one 32-byte load fetches the key's home
            // pair of slots (gx_slot_index is even); up to four loads in flight
#pragma unroll
            for (int i = 0; i < 4; i++) {
                bool need = (i == 0) ? !lead_dup : (k[i] != k[i - 1]);
                if (need) sl[i] = ld_slot2(A.slots + gx_slot_index(k[i], A.sf));
            }
            bool valid0 = !lead_dup || give;
#pragma unroll
            for (int i = 0; i < 4; i++) {
                if (i > 0 && k[i] == k[i - 1]) { g[i] = g[i - 1]; hit[i] = hit[i - 1]; continue; }
                if (i == 0 && lead_dup) { g[0] = 0; hit[0] = give; continue; }        // give: counted below; else filled in by the hand-down
                if (k[i] == GX_EMPTY_KEY) {                    // lives in the side list, never in the table
                    hit[i] = A.special_count > 0; g[i] = hit[i] ? (int) A.special[0] : 0; continue;
                }
                gx_slot2 c = sl[i];
                if (c.k0 == k[i]) { hit[i] = true; g[i] = (int) (unsigned int) c.p0; }
                else if (c.k0 == GX_EMPTY_KEY) { hit[i] = false; g[i] = 0; }
                else if (c.k1 == k[i]) { hit[i] = true; g[i] = (int) (unsigned int) c.p1; }
                else if (c.k1 == GX_EMPTY_KEY) { hit[i] = false; g[i] = 0; }
                else {                                         // both home slots taken by other keys: walk on, a pair at a time
                    unsigned long long p = gx_slot_index(k[i], A.sf);
                    for (;;) {
                        p = gx_next_pair(p, A.mask); c = ld_slot2(A.slots + p);
                        if (c.k0 == k[i]) { hit[i] = true; g[i] = (int) (unsigned int) c.p0; break; }
                        if (c.k0 == GX_EMPTY_KEY) { hit[i] = false; g[i] = 0; break; }
                        if (c.k1 == k[i]) { hit[i] = true; g[i] = (int) (unsigned int) c.p1; break; }
                        if (c.k1 == GX_EMPTY_KEY) { hit[i] = false; g[i] = 0; break; }
                    }
                }
            }
            // whole-lane runs (the lane's four rows all continue the previous lane's key) take the
            // answer from below; such a run can span several lanes, so iterate until settled
            bool valid3 = valid0 || k[3] != k[0];
            while (__any_sync(wmask, !valid0)) {
                int pg = __shfl_up_sync(wmask, g[3], 1);
                bool ph = __shfl_up_sync(wmask, hit[3], 1), pv = __shfl_up_sync(wmask, valid3, 1);
                if (!valid0 && pv) {
                    valid0 = true;
#pragma unroll
                    for (int i = 0; i < 4; i++) if (k[i] == k[0]) { g[i] = pg; hit[i] = ph; }
                    valid3 = true;
                }
            }
            // partial of a handed-over leading run
            unsigned int gcnt = 0; double gsum = 0.0;
            if (give) {
#pragma unroll
                bool in = true;
#pragma unroll
                for (int i = 0; i < 3; i++) { in = in && k[i] == k[0]; if (in) { gcnt++; if (HAS_SUM) gsum = __dadd_rn(gsum, v[i]); hit[i] = false; } }
            }
            rcnt = __shfl_down_sync(wmask, gcnt, 1);
            if (HAS_SUM) rsum = __shfl_down_sync(wmask, gsum, 1);
            if (lane == 31 || !((wmask >> (lane + 1)) & 1u)) { rcnt = 0; rsum = 0.0; }
        } else {
            int4 gg = ld_stream_i4(F.gcol + r);
            g[0] = gg.x; g[1] = gg.y; g[2] = gg.z; g[3] = gg.w;
            hit[0] = hit[1] = hit[2] = hit[3] = true;
        }
        // combine equal neighbours in registers, then one shared-memory update per run
        int cur = 0; unsigned int cnt = 0; double sum = 0.0; bool open = false;
#pragma unroll
        for (int i = 0; i < 4; i++) {
            if (!hit[i]) continue;
            if (open && g[i] == cur) { cnt++; if (HAS_SUM) sum = __dadd_rn(sum, v[i]); continue; }
            if (open) fast_flush<HAS_CNT, HAS_SUM>(T, A, cur, cnt, sum, F.sum_word);
            open = true; cur = g[i]; cnt = 1; sum = HAS_SUM ? v[i] : 0.0;
        }
        if (open) { cnt += rcnt; if (HAS_SUM) sum = __dadd_rn(sum, rsum); fast_flush<HAS_CNT, HAS_SUM>(T, A, cur, cnt, sum, F.sum_word); }
    }
    // the (< 4) rows after the last full vector: one thread each
    {
        long long r = A.row0 + (nvec << 2) + (long long) blockIdx.x * blockDim.x + threadIdx.x;
        if (r < A.row1) {
            bool h = true; int gk;
            if (JOIN) {
                long long key = F.okey[r];
                if (key == GX_EMPTY_KEY) { h = A.special_count > 0; gk = h ? (int) A.special[0] : 0; }
                else {
                    unsigned long long p = gx_slot_index(key, A.sf); gx_slot c = ld_slot(A.slots + p);
                    while (c.key != key && c.key != GX_EMPTY_KEY) { p = gx_next_slot(p, A.mask); c = ld_slot(A.slots + p); }
                    h = c.key == key; gk = (int) (unsigned int) c.payload;
                }
            } else gk = F.gcol[r];
            if (h) fast_flush<HAS_CNT, HAS_SUM>(T, A, gk, 1u, HAS_SUM ? F.vcol[r] : 0.0, F.sum_word);
        }
    }
    __syncthreads();
    smem_dense_merge(T, A);
}

// ---------------------------------------------------------------------------
// Join + aggregate for an outer side whose equal keys sit next to each other (lineitem in
// order-key order: runs of 1..7 rows).  A warp takes 128 consecutive rows, four per lane,
// finds the run heads, and folds every run to ONE (key, count, sum) entry of a per-warp
// shared-memory list — the entries of a run that spans lanes are merged there.  Then the
// list is processed densely, one run per lane: slot function, one 256-bit load of the key's
// home pair, one group-table update.  Against the row-per-lane kernel above this removes
// the repeated probes, the divergent per-row code and three of four group updates; ncu had
// shown that kernel issue-bound at 13.8 of 32 threads per instruction
// (profiles/r01_ncu_probe_pairs_sf100.csv).
struct gx_runlist { long long key[128]; double sum[128]; unsigned int cnt[128]; };

// one key against the join table: the home group of slots arrives with a single 256-bit load
// Branch-free inside the group: a table that is only ever filled (never deleted from) has no
// match behind an empty slot, so "any slot matches" / "any slot empty" decide the step, and the
// function has ONE exit (several exits made the compiler clone the group update per exit).
template <bool COMPACT>
__device__ __forceinline__ bool runjoin_probe(const gx_agg_dev &A, long long key, int &g)
{
    bool found = false;
    if (COMPACT) {
        const unsigned long long dd = (unsigned long long) key - (unsigned long long) A.sf.kmin;
        if (dd < A.cspan) {                                    // else outside the build side's key span (also the reserved key)
            const unsigned int d = GX_CSLOT_D(key, A.sf.kmin);
            unsigned long long p = gx_slot_index(key, A.sf);
            for (;;) {
                const gx_slot2 c = ld_slot2((const gx_slot *) (A.cslots + p));   // four 8-byte slots {d, payload}
                const unsigned int d0 = (unsigned int) c.k0, d1 = (unsigned int) c.p0, d2 = (unsigned int) c.k1, d3 = (unsigned int) c.p1;
                const unsigned long long m = d0 == d ? (unsigned long long) c.k0 : d1 == d ? c.p0 : d2 == d ? (unsigned long long) c.k1 : c.p1;
                found = (d0 == d) | (d1 == d) | (d2 == d) | (d3 == d);
                g = (int) (m >> 32);
                if (found | (d0 == 0u) | (d1 == 0u) | (d2 == 0u) | (d3 == 0u)) break;
                p = gx_next_quad(p, A.mask);
            }
        }
    } else if (key == GX_EMPTY_KEY) {                          // side list, never in the table
        found = A.special_count > 0; if (found) g = (int) A.special[0];
    } else {
        unsigned long long p = gx_slot_index(key, A.sf);
        for (;;) {
            const gx_slot2 c = ld_slot2(A.slots + p);
            found = (c.k0 == key) | (c.k1 == key);
            g = (int) (unsigned int) (c.k0 == key ? c.p0 : c.p1);
            if (found | (c.k0 == GX_EMPTY_KEY) | (c.k1 == GX_EMPTY_KEY)) break;
            p = gx_next_pair(p, A.mask);
        }
    }
    return found;
}

template <bool HAS_CNT, bool HAS_SUM, bool COMPACT>
__global__ void __launch_bounds__(1024, 1) gx_k_runjoin(const __grid_constant__ gx_agg_dev A, const gx_fast_args F)
{
    extern __shared__ unsigned long long smem[];
    SmemTable T; T.S = A.s_slots; T.log2S = A.s_log2; T.nwords = A.P.nwords; T.nkw = 1; T.tagkey = 1; T.gmax = 0;
    T.tag = smem; T.k0 = T.tag + T.S; T.k1 = T.k0; T.w = T.k0; T.gidx = nullptr; T.gcount = nullptr;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    gx_runlist &Q = ((gx_runlist *) (smem + (size_t) T.S * (1 + T.nwords)))[warp];
    for (int i = threadIdx.x; i < T.S; i += blockDim.x) {
        T.tag[i] = 0;
        for (int j = 0; j < T.nwords; j++) T.w[(size_t) i * T.nwords + j] = (unsigned long long) A.winit[j];
    }
    __syncthreads();
    const long long nvec = (A.row1 - A.row0) >> 2;              // groups of four rows
    const long long stride = (long long) gridDim.x * blockDim.x;
    long long q = (long long) blockIdx.x * blockDim.x + threadIdx.x;
    long long k[4]; double v[4];
    bool act = q < nvec;
    if (act) {
        const long long r = A.row0 + (q << 2);
        longlong2 ka = ld_stream_ll2(F.okey + r), kb = ld_stream_ll2(F.okey + r + 2);
        k[0] = ka.x; k[1] = ka.y; k[2] = kb.x; k[3] = kb.y;
        if (HAS_SUM) { double2 a = ld_stream_d2(F.vcol + r), b = ld_stream_d2(F.vcol + r + 2); v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y; }
    }
    // the loop is warp-uniform: lanes past the end carry no rows
    while (__any_sync(0xffffffffu, act)) {
        // ---- the join-table lines this tile's runs will read: requested now, they arrive while the runs are folded
        if (COMPACT && F.pf && act) {
            const unsigned long long dd = (unsigned long long) k[0] - (unsigned long long) A.sf.kmin;
            if (dd < A.cspan) {
                const gx_cslot *pa = A.cslots + gx_slot_index(k[0], A.sf);
                if (F.pf == 2) asm volatile("prefetch.global.L1 [%0];" :: "l"(pa)); else asm volatile("prefetch.global.L2 [%0];" :: "l"(pa));
            }
        }
        // ---- run heads and their numbering inside the warp
        const long long prevk = __shfl_up_sync(0xffffffffu, k[3], 1);
        bool hd[4];
        hd[0] = lane == 0 || k[0] != prevk; hd[1] = k[1] != k[0]; hd[2] = k[2] != k[1]; hd[3] = k[3] != k[2];
        const int nh = act ? (int) hd[0] + (int) hd[1] + (int) hd[2] + (int) hd[3] : 0;
        int inc = nh;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { int t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
        const int base = inc - nh, R = __shfl_sync(0xffffffffu, inc, 31);
        // ---- fold: runs that start in this lane are stored, the rows that continue the previous
        // lane's run are added to that run afterwards
        unsigned int c0 = 0; double s0 = 0.0;
        if (act) {
            int rid = base - 1; unsigned int c = 0; double sacc = 0.0;
#pragma unroll
            for (int i = 0; i < 4; i++) {
                if (hd[i]) {
                    if (rid >= base) { Q.cnt[rid] = c; if (HAS_SUM) Q.sum[rid] = sacc; } else { c0 = c; s0 = sacc; }
                    rid++; Q.key[rid] = k[i]; c = 0; sacc = 0.0;
                }
                c++; if (HAS_SUM) sacc = __dadd_rn(sacc, v[i]);
            }
            if (rid >= base) { Q.cnt[rid] = c; if (HAS_SUM) Q.sum[rid] = sacc; } else { c0 = c; s0 = sacc; }
        }
        __syncwarp();
        if (c0) { atomicAdd(&Q.cnt[base - 1], c0); if (HAS_SUM) atomicAdd(&Q.sum[base - 1], s0); }
        __syncwarp();
        // ---- next rows: requested now, they arrive while the runs are probed
        q += stride; act = q < nvec;
        if (act) {
            const long long r = A.row0 + (q << 2);
            longlong2 ka = ld_stream_ll2(F.okey + r), kb = ld_stream_ll2(F.okey + r + 2);
            k[0] = ka.x; k[1] = ka.y; k[2] = kb.x; k[3] = kb.y;
            if (HAS_SUM) { double2 a = ld_stream_d2(F.vcol + r), b = ld_stream_d2(F.vcol + r + 2); v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y; }
        }
        // ---- one run per lane
        for (int j = lane; j < R; j += 32) {
            const long long key = Q.key[j];
            const unsigned int rc = Q.cnt[j];
            const double rs = HAS_SUM ? Q.sum[j] : 0.0;
            int g = 0;
            const bool hit = runjoin_probe<COMPACT>(A, key, g);
            if (hit) fast_flush<HAS_CNT, HAS_SUM>(T, A, g, rc, rs, F.sum_word);
        }
        __syncwarp();
    }
    // the (< 4) rows after the last full vector: one thread each
    {
        long long r = A.row0 + (nvec << 2) + (long long) blockIdx.x * blockDim.x + threadIdx.x;
        if (r < A.row1) {
            int gk = 0;
            if (runjoin_probe<COMPACT>(A, F.okey[r], gk)) fast_flush<HAS_CNT, HAS_SUM>(T, A, gk, 1u, HAS_SUM ? F.vcol[r] : 0.0, F.sum_word);
        }
    }
    __syncthreads();
    smem_dense_merge(T, A);
}

// ---------------------------------------------------------------------------
// gx_k_runjoin_seg: the same join + aggregate, with the join table STREAMED instead of gathered.
//
// What ncu said about gx_k_runjoin (profiles/r01_ncu_final_sf100_raw.csv, r02_runjoin_variants.txt): 54 % issue
// utilisation, 64 % of the DRAM peak, the warps parked on the dependent 256-bit slot load of their runs.  But with an
// order-preserving slot function and an outer side in key order those loads are not random at all: the CTA's 31 tiles
// of one iteration are 3968 consecutive rows, their keys lie in [first key, last key] of that chunk, and every home
// slot of such a key lies in ONE contiguous piece of the table — about 14 KB at TPC-H's densities.  So a producer warp
// reads the chunk's first and last key one chunk ahead, computes the slot range and copies it into shared memory with a
// single bulk-async copy (TMA, cp.async.bulk ... mbarrier::complete_tx, SASS UBLKCP) into a two-deep ring guarded by
// full/empty mbarriers; the 31 consumer warps fold their tiles exactly as gx_k_runjoin does and then probe SHARED memory.
// The table is still read from DRAM exactly once, now front to back in large requests, and no warp waits on a gather.
// Nothing depends on the layout for correctness: a probe whose slot group is not inside the staged window (keys out
// of order, a chain that walks past the window, a chunk denser than the ring buffer) reads global memory as before,
// and a chunk whose key range is far wider than the buffer is not staged at all.
// Every wait is bounded (GX_SEG_SPIN_LIMIT polls): a protocol error raises flag 16 and the host redoes the query with
// gx_k_runjoin instead of hanging the device.
#define GX_SEG_CW          31                     /* consumer warps; warp 31 is the producer */
#define GX_SEG_SPIN_LIMIT  (1u << 22)
#define GX_SEG_MAXBUF      4
struct gx_seg_ctl { unsigned long long full[GX_SEG_MAXBUF], empty[GX_SEG_MAXBUF], lo[GX_SEG_MAXBUF]; unsigned int len[GX_SEG_MAXBUF]; };

__device__ __forceinline__ unsigned int gx_smem_u32(const void *p) { return (unsigned int) __cvta_generic_to_shared(p); }
__device__ __forceinline__ void gx_mbar_init(void *bar, unsigned int count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(gx_smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void gx_mbar_arrive(void *bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(gx_smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void gx_mbar_arrive_expect_tx(void *bar, unsigned int bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(gx_smem_u32(bar)), "r"(bytes) : "memory");
}
// false when the phase did not complete within the poll budget (try_wait itself sleeps in hardware between polls)
__device__ __forceinline__ bool gx_mbar_wait(void *bar, unsigned int parity)
{
    const unsigned int a = gx_smem_u32(bar);
#pragma unroll 1
    for (unsigned int n = 0; n < GX_SEG_SPIN_LIMIT; n++) {
        unsigned int ok;
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(ok) : "r"(a), "r"(parity) : "memory");
        if (ok) return true;
    }
    return false;
}
// one bulk-async copy global -> shared (16-byte aligned addresses, size a multiple of 16); completion is counted on `bar`
__device__ __forceinline__ void gx_bulk_g2s(void *dst, const void *src, unsigned int bytes, void *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 :: "r"(gx_smem_u32(dst)), "l"(src), "r"(bytes), "r"(gx_smem_u32(bar)) : "memory");
}

// one key against the compact join table, the slot groups inside [lo, lo + len) taken from the staged copy `sg`
__device__ __forceinline__ bool runjoin_probe_seg(const gx_agg_dev &A, long long key, int &g,
                                                  const unsigned long long *sg, unsigned long long lo, unsigned int len)
{
    bool found = false;
    const unsigned long long dd = (unsigned long long) key - (unsigned long long) A.sf.kmin;
    if (dd < A.cspan) {
        const unsigned int d = GX_CSLOT_D(key, A.sf.kmin);
        unsigned long long p = gx_slot_index(key, A.sf);
        for (;;) {
            const unsigned long long off = p - lo;                 // p < lo wraps to a huge value
            unsigned long long s0, s1, s2, s3;                     // four 8-byte slots {d, payload}
            if (off < (unsigned long long) len) {                  // lo, len and p are multiples of 4: the group is inside or outside as a whole
                const ulonglong2 a = *(const ulonglong2 *) (sg + off), b = *(const ulonglong2 *) (sg + off + 2);
                s0 = a.x; s1 = a.y; s2 = b.x; s3 = b.y;
            } else {
                const gx_slot2 c = ld_slot2((const gx_slot *) (A.cslots + p));
                s0 = (unsigned long long) c.k0; s1 = c.p0; s2 = (unsigned long long) c.k1; s3 = c.p1;
            }
            const unsigned int d0 = (unsigned int) s0, d1 = (unsigned int) s1, d2 = (unsigned int) s2, d3 = (unsigned int) s3;
            const unsigned long long m = d0 == d ? s0 : d1 == d ? s1 : d2 == d ? s2 : s3;
            found = (d0 == d) | (d1 == d) | (d2 == d) | (d3 == d);
            g = (int) (m >> 32);
            if (found | (d0 == 0u) | (d1 == 0u) | (d2 == 0u) | (d3 == 0u)) break;
            p = gx_next_quad(p, A.mask);
        }
    }
    return found;
}

template <bool HAS_CNT, bool HAS_SUM>
__global__ void __launch_bounds__(1024, 1) gx_k_runjoin_seg(const __grid_constant__ gx_agg_dev A, const gx_fast_args F, const unsigned int seg_slots, const int nbuf)
{
    extern __shared__ __align__(128) unsigned long long smem_seg[];
    unsigned long long *const smem = smem_seg;
    SmemTable T; T.S = A.s_slots; T.log2S = A.s_log2; T.nwords = A.P.nwords; T.nkw = 1; T.tagkey = 1; T.gmax = 0;
    T.tag = smem; T.k0 = T.tag + T.S; T.k1 = T.k0; T.w = T.k0; T.gidx = nullptr; T.gcount = nullptr;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    gx_runlist *const lists = (gx_runlist *) (smem + (size_t) T.S * (1 + T.nwords));
    // table (S >= 16 slots of >= 16 bytes) and run lists (31 x 2560 bytes) are multiples of 128 bytes: the ring starts 128-byte aligned
    unsigned long long *const seg0 = smem + (size_t) T.S * (1 + T.nwords) + GX_SEG_CW * (sizeof(gx_runlist) / 8);
    gx_seg_ctl *const ctl = (gx_seg_ctl *) (seg0 + (size_t) nbuf * seg_slots);
    for (int i = threadIdx.x; i < T.S; i += blockDim.x) {
        T.tag[i] = 0;
        for (int j = 0; j < T.nwords; j++) T.w[(size_t) i * T.nwords + j] = (unsigned long long) A.winit[j];
    }
    if (threadIdx.x == 0) {
        for (int b = 0; b < nbuf; b++) { gx_mbar_init(&ctl->full[b], 1); gx_mbar_init(&ctl->empty[b], GX_SEG_CW); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    __syncthreads();
    const long long nvec = (A.row1 - A.row0) >> 2;              // groups of four rows
    const long long cvec = (long long) GX_SEG_CW * 32;          // vectors per chunk: one 128-row tile per consumer warp
    const long long nchunks = (nvec + cvec - 1) / cvec;
    const long long niter = (long long) blockIdx.x < nchunks ? (nchunks - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;   // chunks blockIdx.x + j * gridDim.x
    bool stuck = false;
    if (warp == GX_SEG_CW) {
        // ---- producer: chunk j's slot range into ring buffer j % nbuf, up to nbuf chunks ahead of the slowest consumer
        int b = 0; unsigned int use = 0;                       // buffer of chunk j, how often it has been filled before
        long long klo_n = 0, khi_n = 0;
        if (lane == 0 && niter > 0) {
            const long long v0 = (long long) blockIdx.x * cvec, v1 = v0 + cvec < nvec ? v0 + cvec : nvec;
            klo_n = __ldg(F.okey + A.row0 + (v0 << 2)); khi_n = __ldg(F.okey + A.row0 + (v1 << 2) - 1);
        }
        for (long long j = 0; j < niter; j++) {
            if (lane == 0 && !stuck) {
                const long long klo = klo_n, khi = khi_n;
                if (j + 1 < niter) {                             // the next chunk's end keys travel while this one is set up
                    const long long v0 = ((long long) blockIdx.x + (j + 1) * gridDim.x) * cvec, v1 = v0 + cvec < nvec ? v0 + cvec : nvec;
                    klo_n = __ldg(F.okey + A.row0 + (v0 << 2)); khi_n = __ldg(F.okey + A.row0 + (v1 << 2) - 1);
                }
                // the part of the chunk's key range that lies inside the build side's key span
                const long long kmax = (long long) ((unsigned long long) A.sf.kmin + A.cspan - 1ULL);
                const long long ka = klo < A.sf.kmin ? A.sf.kmin : klo, kz = khi > kmax ? kmax : khi;
                unsigned long long lo = 0; unsigned int len = 0;
                if (ka <= kz) {
                    const unsigned long long wm = (unsigned long long) (A.sf.win | A.sf.amask);     // the scatter window keeps a key inside its aligned block
                    lo = gx_slot_index(ka, A.sf) & ~wm;
                    unsigned long long hi = (gx_slot_index(kz, A.sf) | wm) + 1ULL + 32ULL;          // + one block for chains that walk on
                    if (hi > A.mask + 1ULL) hi = A.mask + 1ULL;
                    if (hi > lo) {
                        const unsigned long long n = hi - lo;
                        if (n <= 4ULL * seg_slots) len = (unsigned int) (n < seg_slots ? n : seg_slots);   // far wider: not clustered, stage nothing
                    }
                }
                if (use > 0 && !gx_mbar_wait(&ctl->empty[b], (use - 1) & 1u)) stuck = true;
                if (!stuck) {
                    ctl->lo[b] = lo; ctl->len[b] = len;
                    if (len) {
                        gx_mbar_arrive_expect_tx(&ctl->full[b], len * 8u);
                        gx_bulk_g2s(seg0 + (size_t) b * seg_slots, A.cslots + lo, len * 8u, &ctl->full[b]);
                    } else gx_mbar_arrive(&ctl->full[b]);
                }
            }
            if (++b == nbuf) { b = 0; use++; }
            __syncwarp();
        }
    } else {
        gx_runlist &Q = lists[warp];
        long long q = ((long long) blockIdx.x * GX_SEG_CW + warp) * 32 + lane;
        const long long qstride = (long long) gridDim.x * cvec;
        long long k[4]; double v[4];
        bool act = q < nvec;
        if (act) {
            const long long r = A.row0 + (q << 2);
            longlong2 ka = ld_stream_ll2(F.okey + r), kb = ld_stream_ll2(F.okey + r + 2);
            k[0] = ka.x; k[1] = ka.y; k[2] = kb.x; k[3] = kb.y;
            if (HAS_SUM) { double2 a = ld_stream_d2(F.vcol + r), b = ld_stream_d2(F.vcol + r + 2); v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y; }
        }
        int b = 0; unsigned int use = 0;
        for (long long j = 0; j < niter; j++) {
            // ---- run heads and their numbering inside the warp (as in gx_k_runjoin)
            const long long prevk = __shfl_up_sync(0xffffffffu, k[3], 1);
            bool hd[4];
            hd[0] = lane == 0 || k[0] != prevk; hd[1] = k[1] != k[0]; hd[2] = k[2] != k[1]; hd[3] = k[3] != k[2];
            const int nh = act ? (int) hd[0] + (int) hd[1] + (int) hd[2] + (int) hd[3] : 0;
            int inc = nh;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { int t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
            const int base = inc - nh, R = __shfl_sync(0xffffffffu, inc, 31);
            unsigned int c0 = 0; double s0 = 0.0;
            if (act) {
                int rid = base - 1; unsigned int c = 0; double sacc = 0.0;
#pragma unroll
                for (int i = 0; i < 4; i++) {
                    if (hd[i]) {
                        if (rid >= base) { Q.cnt[rid] = c; if (HAS_SUM) Q.sum[rid] = sacc; } else { c0 = c; s0 = sacc; }
                        rid++; Q.key[rid] = k[i]; c = 0; sacc = 0.0;
                    }
                    c++; if (HAS_SUM) sacc = __dadd_rn(sacc, v[i]);
                }
                if (rid >= base) { Q.cnt[rid] = c; if (HAS_SUM) Q.sum[rid] = sacc; } else { c0 = c; s0 = sacc; }
            }
            __syncwarp();
            if (c0) { atomicAdd(&Q.cnt[base - 1], c0); if (HAS_SUM) atomicAdd(&Q.sum[base - 1], s0); }
            __syncwarp();
            // ---- next rows: requested now, they arrive while the runs are probed
            q += qstride; act = q < nvec;
            if (act) {
                const long long r = A.row0 + (q << 2);
                longlong2 ka = ld_stream_ll2(F.okey + r), kb = ld_stream_ll2(F.okey + r + 2);
                k[0] = ka.x; k[1] = ka.y; k[2] = kb.x; k[3] = kb.y;
                if (HAS_SUM) { double2 a = ld_stream_d2(F.vcol + r), b = ld_stream_d2(F.vcol + r + 2); v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y; }
            }
            // ---- this chunk's piece of the join table has landed (or the wait gives up and the host is told)
            unsigned long long lo = 0; unsigned int len = 0;
            if (!stuck && !gx_mbar_wait(&ctl->full[b], use & 1u)) stuck = true;
            if (!stuck) { lo = ctl->lo[b]; len = ctl->len[b]; }
            const unsigned long long *const sg = seg0 + (size_t) b * seg_slots;
            // ---- one run per lane
            for (int jj = lane; jj < R; jj += 32) {
                const long long key = Q.key[jj];
                const unsigned int rc = Q.cnt[jj];
                const double rs = HAS_SUM ? Q.sum[jj] : 0.0;
                int g = 0;
                const bool hit = runjoin_probe_seg(A, key, g, sg, lo, len);
                if (hit) fast_flush<HAS_CNT, HAS_SUM>(T, A, g, rc, rs, F.sum_word);
            }
            __syncwarp();
            if (lane == 0) gx_mbar_arrive(&ctl->empty[b]);      // the buffer may be refilled for chunk j + nbuf
            if (++b == nbuf) { b = 0; use++; }
        }
        // the (< 4) rows after the last full vector: one thread each
        {
            long long r = A.row0 + (nvec << 2) + (long long) blockIdx.x * blockDim.x + threadIdx.x;
            if (r < A.row1) {
                int gk = 0;
                if (runjoin_probe<true>(A, F.okey[r], gk)) fast_flush<HAS_CNT, HAS_SUM>(T, A, gk, 1u, HAS_SUM ? F.vcol[r] : 0.0, F.sum_word);
            }
        }
    }
    if (stuck) atomicOr((unsigned long long *) &A.counters[1], 16ULL);
    __syncthreads();
    smem_dense_merge(T, A);
}

struct gx_runlist3 { long long key[160]; double sum[160]; unsigned int cnt[160]; };   // 31 waiting + 128 new runs
template <bool HAS_CNT, bool HAS_SUM, bool COMPACT>
__global__ void __launch_bounds__(1024, 1) gx_k_runjoin3(const __grid_constant__ gx_agg_dev A, const gx_fast_args F)
{
    extern __shared__ unsigned long long smem[];
    SmemTable T; T.S = A.s_slots; T.log2S = A.s_log2; T.nwords = A.P.nwords; T.nkw = 1; T.tagkey = 1; T.gmax = 0;
    T.tag = smem; T.k0 = T.tag + T.S; T.k1 = T.k0; T.w = T.k0; T.gidx = nullptr; T.gcount = nullptr;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    gx_runlist3 &Q = ((gx_runlist3 *) (smem + (size_t) T.S * (1 + T.nwords)))[warp];
    int nl = 0;                                                 // finished runs waiting at the front of the list for a full round of 32
    for (int i = threadIdx.x; i < T.S; i += blockDim.x) {
        T.tag[i] = 0;
        for (int j = 0; j < T.nwords; j++) T.w[(size_t) i * T.nwords + j] = (unsigned long long) A.winit[j];
    }
    __syncthreads();
    const long long nvec = (A.row1 - A.row0) >> 2;              // groups of four rows
    const long long stride = (long long) gridDim.x * blockDim.x;
    long long q = (long long) blockIdx.x * blockDim.x + threadIdx.x;
    long long k[4]; double v[4];
    bool act = q < nvec;
    if (act) {
        const long long r = A.row0 + (q << 2);
        longlong2 ka = ld_stream_ll2(F.okey + r), kb = ld_stream_ll2(F.okey + r + 2);
        k[0] = ka.x; k[1] = ka.y; k[2] = kb.x; k[3] = kb.y;
        if (HAS_SUM) { double2 a = ld_stream_d2(F.vcol + r), b = ld_stream_d2(F.vcol + r + 2); v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y; }
    }
    // the loop is warp-uniform: lanes past the end carry no rows
    while (__any_sync(0xffffffffu, act)) {
        // ---- run heads and their numbering inside the warp
        const long long prevk = __shfl_up_sync(0xffffffffu, k[3], 1);
        bool hd[4];
        hd[0] = lane == 0 || k[0] != prevk; hd[1] = k[1] != k[0]; hd[2] = k[2] != k[1]; hd[3] = k[3] != k[2];
        const int nh = act ? (int) hd[0] + (int) hd[1] + (int) hd[2] + (int) hd[3] : 0;
        int inc = nh;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { int t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
        const int base = nl + inc - nh, R = __shfl_sync(0xffffffffu, inc, 31);      // this tile's runs go behind the waiting ones
        // ---- fold: runs that start in this lane are stored, the rows that continue the previous
        // lane's run are added to that run afterwards
        unsigned int c0 = 0; double s0 = 0.0;
        if (act) {
            int rid = base - 1; unsigned int c = 0; double sacc = 0.0;
#pragma unroll
            for (int i = 0; i < 4; i++) {
                if (hd[i]) {
                    if (rid >= base) { Q.cnt[rid] = c; if (HAS_SUM) Q.sum[rid] = sacc; } else { c0 = c; s0 = sacc; }
                    rid++; Q.key[rid] = k[i]; c = 0; sacc = 0.0;
                }
                c++; if (HAS_SUM) sacc = __dadd_rn(sacc, v[i]);
            }
            if (rid >= base) { Q.cnt[rid] = c; if (HAS_SUM) Q.sum[rid] = sacc; } else { c0 = c; s0 = sacc; }
        }
        __syncwarp();
        if (c0) { atomicAdd(&Q.cnt[base - 1], c0); if (HAS_SUM) atomicAdd(&Q.sum[base - 1], s0); }
        __syncwarp();
        // ---- next rows: requested now, they arrive while the runs are probed
        q += stride; act = q < nvec;
        if (act) {
            const long long r = A.row0 + (q << 2);
            longlong2 ka = ld_stream_ll2(F.okey + r), kb = ld_stream_ll2(F.okey + r + 2);
            k[0] = ka.x; k[1] = ka.y; k[2] = kb.x; k[3] = kb.y;
            if (HAS_SUM) { double2 a = ld_stream_d2(F.vcol + r), b = ld_stream_d2(F.vcol + r + 2); v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y; }
        }
        // ---- one run per lane, in FULL rounds of 32 only: a tile of 128 rows holds ~33 runs, and a second round for
        // the last one or two of them costs the warp as many issue slots as a full one
        const int total = nl + R, full = total & ~31;
        for (int j = lane; j < full; j += 32) {
            const long long key = Q.key[j];
            const unsigned int rc = Q.cnt[j];
            const double rs = HAS_SUM ? Q.sum[j] : 0.0;
            int g = 0;
            const bool hit = runjoin_probe<COMPACT>(A, key, g);
            if (hit) fast_flush<HAS_CNT, HAS_SUM>(T, A, g, rc, rs, F.sum_word);
        }
        __syncwarp();
        nl = total - full;
        if (full > 0 && lane < nl) {                                // the remainder moves to the front (sources lie at index >= 32)
            const long long kk = Q.key[full + lane]; const unsigned int cq = Q.cnt[full + lane]; const double sq = HAS_SUM ? Q.sum[full + lane] : 0.0;
            Q.key[lane] = kk; Q.cnt[lane] = cq; if (HAS_SUM) Q.sum[lane] = sq;
        }
        __syncwarp();
    }
    for (int j = lane; j < nl; j += 32) {                           // what was still waiting when the rows ran out
        int g = 0;
        const bool hit = runjoin_probe<COMPACT>(A, Q.key[j], g);
        if (hit) fast_flush<HAS_CNT, HAS_SUM>(T, A, g, Q.cnt[j], HAS_SUM ? Q.sum[j] : 0.0, F.sum_word);
    }
    __syncwarp();
    // the (< 4) rows after the last full vector: one thread each
    {
        long long r = A.row0 + (nvec << 2) + (long long) blockIdx.x * blockDim.x + threadIdx.x;
        if (r < A.row1) {
            int gk = 0;
            if (runjoin_probe<COMPACT>(A, F.okey[r], gk)) fast_flush<HAS_CNT, HAS_SUM>(T, A, gk, 1u, HAS_SUM ? F.vcol[r] : 0.0, F.sum_word);
        }
    }
    __syncthreads();
    smem_dense_merge(T, A);
}

// 16-byte group slots for gx_k_runjoin2: word 0 = [bit 63 occupied | bits 62..32 rows | bits 31..0 the 4-byte key], the sum
// lives in a parallel array.  The row count is added to the word's upper half with a native 32-bit shared atomic.
#define PK_OCC   0x8000000000000000ULL
#define PK_MATCH 0x80000000FFFFFFFFULL
template <bool HAS_SUM>
__device__ __forceinline__ void packed_flush(unsigned long long *tab, double *tsum, int S, const gx_agg_dev &A, int gkey, unsigned int cnt, double sum)
{
    const unsigned long long want = PK_OCC | (unsigned long long) (unsigned int) gkey;
    int s = (int) ((unsigned int) gkey & (unsigned int) (S - 1));
    for (int n = 0;; n++) {
        const unsigned long long t = *(volatile unsigned long long *) &tab[s];
        if ((t & PK_MATCH) == want) break;
        if (t == 0) { const unsigned long long old = atomicCAS(&tab[s], 0ULL, want); if (old == 0 || (old & PK_MATCH) == want) break; }
        s = (s + 1) & (S - 1);
        if (n >= 64) { atomicOr((unsigned long long *) &A.counters[1], 1ULL); return; }
    }
    atomicAdd((unsigned int *) &tab[s] + 1, cnt);                  // little-endian: the upper half holds the row count
    if (HAS_SUM) atomicAdd(&tsum[s], sum);
}

template <bool HAS_SUM, bool COMPACT>
__global__ void __launch_bounds__(512, 2) gx_k_runjoin2(const __grid_constant__ gx_agg_dev A, const gx_fast_args F)
{
    extern __shared__ unsigned long long smem[];
    // group table: 16 bytes per slot — [occupied | rows (31 bits) | 4-byte key] and the float8 sum — so that two CTAs
    // of 512 threads fit one SM (gx_k_runjoin keeps 24-byte slots and one CTA of 1024)
    const int S = A.s_slots;
    unsigned long long *const tab = smem; double *const tsum = (double *) (smem + S);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    gx_runlist &Q = ((gx_runlist *) (smem + (size_t) S * 2))[warp];
    for (int i = threadIdx.x; i < S; i += blockDim.x) { tab[i] = 0ULL; tsum[i] = 0.0; }
    __syncthreads();
    const long long nvec = (A.row1 - A.row0) >> 2;              // groups of four rows
    const long long stride = (long long) gridDim.x * blockDim.x;
    long long q = (long long) blockIdx.x * blockDim.x + threadIdx.x;
    long long k[4]; double v[4];
    bool act = q < nvec;
    if (act) {
        const long long r = A.row0 + (q << 2);
        longlong2 ka = ld_stream_ll2(F.okey + r), kb = ld_stream_ll2(F.okey + r + 2);
        k[0] = ka.x; k[1] = ka.y; k[2] = kb.x; k[3] = kb.y;
        if (HAS_SUM) { double2 a = ld_stream_d2(F.vcol + r), b = ld_stream_d2(F.vcol + r + 2); v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y; }
    }
    // the loop is warp-uniform: lanes past the end carry no rows
    while (__any_sync(0xffffffffu, act)) {
        // ---- run heads and their numbering inside the warp
        const long long prevk = __shfl_up_sync(0xffffffffu, k[3], 1);
        bool hd[4];
        hd[0] = lane == 0 || k[0] != prevk; hd[1] = k[1] != k[0]; hd[2] = k[2] != k[1]; hd[3] = k[3] != k[2];
        const int nh = act ? (int) hd[0] + (int) hd[1] + (int) hd[2] + (int) hd[3] : 0;
        int inc = nh;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { int t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
        const int base = inc - nh, R = __shfl_sync(0xffffffffu, inc, 31);
        // ---- fold: runs that start in this lane are stored, the rows that continue the previous
        // lane's run are added to that run afterwards
        unsigned int c0 = 0; double s0 = 0.0;
        if (act) {
            int rid = base - 1; unsigned int c = 0; double sacc = 0.0;
#pragma unroll
            for (int i = 0; i < 4; i++) {
                if (hd[i]) {
                    if (rid >= base) { Q.cnt[rid] = c; if (HAS_SUM) Q.sum[rid] = sacc; } else { c0 = c; s0 = sacc; }
                    rid++; Q.key[rid] = k[i]; c = 0; sacc = 0.0;
                }
                c++; if (HAS_SUM) sacc = __dadd_rn(sacc, v[i]);
            }
            if (rid >= base) { Q.cnt[rid] = c; if (HAS_SUM) Q.sum[rid] = sacc; } else { c0 = c; s0 = sacc; }
        }
        __syncwarp();
        if (c0) { atomicAdd(&Q.cnt[base - 1], c0); if (HAS_SUM) atomicAdd(&Q.sum[base - 1], s0); }
        __syncwarp();
        // ---- next rows: requested now, they arrive while the runs are probed
        q += stride; act = q < nvec;
        if (act) {
            const long long r = A.row0 + (q << 2);
            longlong2 ka = ld_stream_ll2(F.okey + r), kb = ld_stream_ll2(F.okey + r + 2);
            k[0] = ka.x; k[1] = ka.y; k[2] = kb.x; k[3] = kb.y;
            if (HAS_SUM) { double2 a = ld_stream_d2(F.vcol + r), b = ld_stream_d2(F.vcol + r + 2); v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y; }
        }
        // ---- one run per lane
        for (int j = lane; j < R; j += 32) {
            const long long key = Q.key[j];
            const unsigned int rc = Q.cnt[j];
            const double rs = HAS_SUM ? Q.sum[j] : 0.0;
            int g = 0;
            const bool hit = runjoin_probe<COMPACT>(A, key, g);
            if (hit) packed_flush<HAS_SUM>(tab, tsum, S, A, g, rc, rs);
        }
        __syncwarp();
    }
    // the (< 4) rows after the last full vector: one thread each
    {
        long long r = A.row0 + (nvec << 2) + (long long) blockIdx.x * blockDim.x + threadIdx.x;
        if (r < A.row1) {
            int gk = 0;
            if (runjoin_probe<COMPACT>(A, F.okey[r], gk)) packed_flush<HAS_SUM>(tab, tsum, S, A, gk, 1u, HAS_SUM ? F.vcol[r] : 0.0);
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < S; i += blockDim.x) {             // the CTA's table into the global one
        const unsigned long long t = tab[i];
        if (t == 0) continue;
        unsigned long long *rec = global_upsert(A, t & 0xFFFFFFFFULL, 0ULL, 0u);
        if (!rec) { atomicOr((unsigned long long *) &A.counters[1], 2ULL); continue; }
        merge_word(&rec[3], WK_ADD_I64, (t >> 32) & 0x7FFFFFFFULL);
        if (HAS_SUM) merge_word(&rec[3 + F.sum_word], WK_ADD_F64, (unsigned long long) __double_as_longlong(tsum[i]));
    }
}

// ---------------------------------------------------------------------------
// gx_k_runjoin_tma: gx_k_runjoin with the outer rows delivered by the copy engine.
//
// The per-instruction stall samples of gx_k_runjoin (source page of the ncu capture behind profiles/r01_ncu_final_sf100.csv) put 14 % of all
// samples on ONE register move right behind the "prefetch" loads of the next tile: ptxas lands half of the 128-bit
// loads in temporaries and copies them into the loop-carried registers at once, so the warp waits out the DRAM latency
// of its rows BEFORE it starts the probe, whose dependent slot load then costs a second one (27 % of the samples).
// Here the rows never pass through registers on their way in: lane 0 of every warp asks the copy engine for the warp's
// next tile (two 1 KB cp.async.bulk transfers, keys and values, completion counted on the warp's own mbarrier) as soon
// as the lanes have read the current one out of shared memory — before the fold, a whole tile ahead — and nobody waits
// for anybody else: a warp only ever waits on its own barrier.  The 64 KB of row stages fit because the group table
// uses gx_k_runjoin2's packed 16-byte slots (64 KB instead of 96 KB for 4096 slots).
// Bounded waits as in gx_k_runjoin_seg: flag 16 sends the plan back to gx_k_runjoin.
struct gx_rowstage { long long key[128]; double val[128]; };

template <bool HAS_SUM, bool COMPACT, bool FOLD2, bool CARRY>
__global__ void __launch_bounds__(1024, 1) gx_k_runjoin_tma(const __grid_constant__ gx_agg_dev A, const gx_fast_args F)
{
    extern __shared__ __align__(128) unsigned long long smem_tma[];
    const int S = A.s_slots;
    unsigned long long *const tab = smem_tma; double *const tsum = (double *) (smem_tma + S);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    gx_runlist &Q = ((gx_runlist *) (smem_tma + (size_t) S * 2))[warp];
    gx_rowstage &R = ((gx_rowstage *) (smem_tma + (size_t) S * 2 + 32 * (sizeof(gx_runlist) / 8)))[warp];
    unsigned long long *const bar = smem_tma + (size_t) S * 2 + 32 * (sizeof(gx_runlist) / 8) + 32 * (sizeof(gx_rowstage) / 8) + warp;
    for (int i = threadIdx.x; i < S; i += blockDim.x) { tab[i] = 0ULL; tsum[i] = 0.0; }
    if (lane == 0) {
        gx_mbar_init(bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    __syncthreads();
    const long long nvec = (A.row1 - A.row0) >> 2;              // groups of four rows
    const long long stride = (long long) gridDim.x * blockDim.x;
    long long qw = (long long) blockIdx.x * blockDim.x + warp * 32;     // the warp's first vector of its current tile
    // the warp's tile [qw, qw + 32) vectors = up to 128 rows: one bulk copy per column.  The request is the only per-tile
    // code that was not in gx_k_runjoin and every instruction of it is issued by the whole warp, so it is kept short:
    // running byte pointers, 32-bit shared addresses, a running count of the vectors left, and elect.sync so that ptxas
    // knows a single lane feeds the uniform registers of UBLKCP (no per-operand broadcast loops).
    const char *kp = (const char *) (F.okey + A.row0) + (qw << 5);
    const char *vp = (const char *) (F.vcol + A.row0) + (qw << 5);
    const long long step = stride << 5;                         // bytes between a warp's consecutive tiles
    const unsigned int s_key = gx_smem_u32(R.key), s_val = gx_smem_u32(R.val), s_bar = gx_smem_u32(bar);
    long long left = nvec - qw;                                 // vectors from the start of the warp's current tile to the end of the input
    auto request = [&](unsigned int bytes) {
        unsigned int leader;
        asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(leader));
        if (leader) {
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(s_bar), "r"(HAS_SUM ? 2u * bytes : bytes) : "memory");
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                         :: "r"(s_key), "l"(kp), "r"(bytes), "r"(s_bar) : "memory");
            if (HAS_SUM)
                asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                             :: "r"(s_val), "l"(vp), "r"(bytes), "r"(s_bar) : "memory");
        }
    };
    if (left > 0) request(left >= 32 ? 1024u : (unsigned int) left << 5);
    unsigned int parity = 0;
    bool stuck = false;
    // one run against the join table and into the group table
    auto probe_one = [&](int j) {
        const long long key = Q.key[j];
        const unsigned int rc = Q.cnt[j];
        const double rs = HAS_SUM ? Q.sum[j] : 0.0;
        int g = 0;
        const bool hit = runjoin_probe<COMPACT>(A, key, g);
        if (hit) packed_flush<HAS_SUM>(tab, tsum, S, A, g, rc, rs);
    };
    // CARRY (GX_RUNJOIN_TMA=3): probe rounds only ever run with 32 lanes.  A tile holds ~33 runs, so half the tiles pay a second
    // round for one to three of them (~50 instructions per tile).  Here the list keeps its oldest T mod 32 entries at the front -
    // nothing is moved: the rounds take the NEWEST entries [T mod 32, T), the next tile appends behind what stayed, and the last
    // stragglers are probed when the warp runs out of rows.  (gx_k_runjoin3 moved the remainder to the front after every tile.)
    int nc = 0;                                                 // entries waiting at the front of the list
    while (left > 0) {                                          // warp-uniform
        const bool act = (long long) lane < left;
        long long k[4]; double v[4];
        if (!gx_mbar_wait(bar, parity)) { stuck = true; break; }
        parity ^= 1u;
        if (act) {
            const longlong2 ka = *(const longlong2 *) &R.key[lane * 4], kb = *(const longlong2 *) &R.key[lane * 4 + 2];
            k[0] = ka.x; k[1] = ka.y; k[2] = kb.x; k[3] = kb.y;
            if (HAS_SUM) {
                const double2 a = *(const double2 *) &R.val[lane * 4], b = *(const double2 *) &R.val[lane * 4 + 2];
                v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
            }
        }
        // ---- the stage is free again: the next tile travels while this one is folded and probed.  The copy engine's
        // writes are not ordered after the lanes' shared loads above by __syncwarp: a load still in flight could return
        // bytes of the next tile, and that lane would fold rows of the wrong tile (counts off by one in some groups, seen
        // with outer rows not in key order).  So the request DEPENDS on every lane's loaded values: a vote over them
        // (always 0 after the mask, which the compiler cannot know) is added to the byte count, and the vote cannot
        // execute before every load has returned.  Measured at SF100 on one B200 (1000 W limit) against a fence.proxy.async per tile
        // (4.09 ms/step) and against issuing the request after the fold (4.02): 3.93, the same as without any ordering.
        unsigned long long dx = 0;
        if (act) {
            dx = (unsigned long long) (k[0] ^ k[1] ^ k[2] ^ k[3]);
            if (HAS_SUM) dx ^= (unsigned long long) (__double_as_longlong(v[0]) ^ __double_as_longlong(v[1]) ^ __double_as_longlong(v[2]) ^ __double_as_longlong(v[3]));
        }
        const unsigned int dep = __ballot_sync(0xffffffffu, dx == 0x5a5a5a5a5a5a5a5aULL) & (unsigned int) (left >> 62);   // left < 2^62
        kp += step; vp += step; left -= stride;
        if (left > 0) request((left >= 32 ? 1024u : (unsigned int) left << 5) + dep);
        int NR;
        if (FOLD2) {
            // ---- the same fold without branches (GX_RUNJOIN_TMA=2): ptxas turned the four "if (head) { close the open run, open the
            // next }" steps of the loop below into four branch regions full of register shuffling (~100 instructions per tile).
            // Here every row knows its run (r_i), every run length and sum is a chain of selects that restarts at a head, and each
            // store is a single predicated instruction.
            const long long prevk = __shfl_up_sync(0xffffffffu, k[3], 1);
            const bool h0 = act && (lane == 0 || k[0] != prevk), h1 = act && k[1] != k[0], h2 = act && k[2] != k[1], h3 = act && k[3] != k[2];
            const int nh = (int) h0 + (int) h1 + (int) h2 + (int) h3;
            int inc = nh;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { int t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
            NR = __shfl_sync(0xffffffffu, inc, 31);
            if (CARRY && nc + NR > 128) {                       // more runs than the list has room for behind the waiting ones (rare): those first
                for (int j = lane; j < nc; j += 32) probe_one(j);
                nc = 0;
                __syncwarp();
            }
            const int base = inc - nh + (CARRY ? nc : 0);
            const int r0 = base + (int) h0 - 1, r1 = r0 + (int) h1, r2 = r1 + (int) h2, r3 = r2 + (int) h3;   // run of row i; base - 1 = the previous lane's last run
            const unsigned int c1 = h1 ? 1u : 2u, c2 = h2 ? 1u : c1 + 1u, c3 = h3 ? 1u : c2 + 1u;                // rows of row i's run up to row i, inside this lane
            double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
            if (HAS_SUM) { s0 = v[0]; s1 = h1 ? v[1] : __dadd_rn(s0, v[1]); s2 = h2 ? v[2] : __dadd_rn(s1, v[2]); s3 = h3 ? v[3] : __dadd_rn(s2, v[3]); }
            const bool q0 = h0, q1 = q0 || h1, q2 = q1 || h2, q3 = q2 || h3;                                     // row i's run started in this lane
            if (h0) Q.key[r0] = k[0];
            if (h1) Q.key[r1] = k[1];
            if (h2) Q.key[r2] = k[2];
            if (h3) Q.key[r3] = k[3];
            // a run of this lane ends at row i when row i + 1 is a head, the last one at row 3
            if (h1 && q0) { Q.cnt[r0] = 1u; if (HAS_SUM) Q.sum[r0] = s0; }
            if (h2 && q1) { Q.cnt[r1] = c1; if (HAS_SUM) Q.sum[r1] = s1; }
            if (h3 && q2) { Q.cnt[r2] = c2; if (HAS_SUM) Q.sum[r2] = s2; }
            if (q3) { Q.cnt[r3] = c3; if (HAS_SUM) Q.sum[r3] = s3; }
            // the rows before this lane's first head continue the previous lane's run: added once that run's own lane has stored it
            unsigned int cc = 0; double sc = 0.0;
            if (act && !h0) {
                cc = h1 ? 1u : h2 ? c1 : h3 ? c2 : c3;
                if (HAS_SUM) sc = h1 ? s0 : h2 ? s1 : h3 ? s2 : s3;
            }
            __syncwarp();
            if (cc) { atomicAdd(&Q.cnt[base - 1], cc); if (HAS_SUM) atomicAdd(&Q.sum[base - 1], sc); }
            __syncwarp();
        } else {
            // ---- run heads and their numbering inside the warp
            const long long prevk = __shfl_up_sync(0xffffffffu, k[3], 1);
            bool hd[4];
            hd[0] = lane == 0 || k[0] != prevk; hd[1] = k[1] != k[0]; hd[2] = k[2] != k[1]; hd[3] = k[3] != k[2];
            const int nh = act ? (int) hd[0] + (int) hd[1] + (int) hd[2] + (int) hd[3] : 0;
            int inc = nh;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { int t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
            const int base = inc - nh;
            NR = __shfl_sync(0xffffffffu, inc, 31);
            // ---- fold: runs that start in this lane are stored, the rows that continue the previous
            // lane's run are added to that run afterwards
            unsigned int c0 = 0; double s0 = 0.0;
            if (act) {
                int rid = base - 1; unsigned int c = 0; double sacc = 0.0;
#pragma unroll
                for (int i = 0; i < 4; i++) {
                    if (hd[i]) {
                        if (rid >= base) { Q.cnt[rid] = c; if (HAS_SUM) Q.sum[rid] = sacc; } else { c0 = c; s0 = sacc; }
                        rid++; Q.key[rid] = k[i]; c = 0; sacc = 0.0;
                    }
                    c++; if (HAS_SUM) sacc = __dadd_rn(sacc, v[i]);
                }
                if (rid >= base) { Q.cnt[rid] = c; if (HAS_SUM) Q.sum[rid] = sacc; } else { c0 = c; s0 = sacc; }
            }
            __syncwarp();
            if (c0) { atomicAdd(&Q.cnt[base - 1], c0); if (HAS_SUM) atomicAdd(&Q.sum[base - 1], s0); }
            __syncwarp();
        }
        // ---- one run per lane
        if (CARRY) {
            const int T = nc + NR, first = T & 31;
            for (int j = first + lane; j < T; j += 32) probe_one(j);
            nc = first;
        } else {
            for (int j = lane; j < NR; j += 32) probe_one(j);
        }
        __syncwarp();
    }
    if (CARRY) { for (int j = lane; j < nc; j += 32) probe_one(j); }        // what was still waiting when the rows ran out
    if (stuck) atomicOr((unsigned long long *) &A.counters[1], 16ULL);
    // the (< 4) rows after the last full vector: one thread each
    {
        long long r = A.row0 + (nvec << 2) + (long long) blockIdx.x * blockDim.x + threadIdx.x;
        if (r < A.row1) {
            int gk = 0;
            if (runjoin_probe<COMPACT>(A, F.okey[r], gk)) packed_flush<HAS_SUM>(tab, tsum, S, A, gk, 1u, HAS_SUM ? F.vcol[r] : 0.0);
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < S; i += blockDim.x) {             // the CTA's table into the global one
        const unsigned long long t = tab[i];
        if (t == 0) continue;
        unsigned long long *rec = global_upsert(A, t & 0xFFFFFFFFULL, 0ULL, 0u);
        if (!rec) { atomicOr((unsigned long long *) &A.counters[1], 2ULL); continue; }
        merge_word(&rec[3], WK_ADD_I64, (t >> 32) & 0x7FFFFFFFULL);
        if (HAS_SUM) merge_word(&rec[3 + F.sum_word], WK_ADD_F64, (unsigned long long) __double_as_longlong(tsum[i]));
    }
}

// ---------------------------------------------------------------------------
// GROUP BY keys that CONTAIN the join key of a unique build side (the Q3 shape: GROUP BY
// l_orderkey, o_orderdate, o_shippriority) over an outer side stored in key order: all rows of
// a group are one run of consecutive rows, so a run IS a group.  Each warp owns a contiguous
// chunk of rows; per slab of 32 rows it evaluates quals and aggregate arguments, finds the run
// heads, reduces (count, sums) per run with a segmented warp scan, and appends every finished
// run to a per-warp shared-memory list; the list is then processed densely, one run per lane:
// one probe of the join table, one FINAL record written.  No per-row records, no radix passes,
// no group table — except for the (at most two) runs per chunk that touch a chunk boundary and
// may continue in a neighbour's chunk: their pieces meet in a small global table through the
// ordinary merge operator.  The kernel verifies on every adjacent pair of rows (across slabs,
// tiles and chunks) that the keys do not descend; any violation raises a flag and the host
// takes the general path (records + radix), so the result never depends on the layout.
// Replaces ExecHashJoinImpl's probe loop + agg_fill_hash_table for this shape
// (nodeHashjoin.c:446-666, nodeAgg.c:2609-2648).
#define RA_NV   4                        /* float8 sum words per group (beyond the row count) */
#define RA_LIST 168                      /* <= 31 finished runs waiting for a full round + the carry + 128 new ones */
#define RA_BND  0x80000000u
struct gx_runagg_args {
    int nv, nc, pf, pf_n;             // pf_n: columns listed for the row prefetch (the first four the tile reads)
    const char *pf_ptr[4]; int pf_size[4], pf_lines[4];            // pf: bit 0 = rows two tiles ahead into L2, bit 1 = this tile's join-table lines into L2 before the fold
    int vagg[RA_NV], vword[RA_NV];
    const double *col[FG_NC];           // distinct argument columns, loaded once per row (as in gx_k_fewgroups)
    signed char tslot[RA_NV][4];
    unsigned long long *out; long long out_cap; long long *cursor;   // dense final records + cursor
    long long rows_per_warp;
    // group-key packing: the join key and/or payload bit fields
    int ngk; int gk_from_key[GX_MAX_GROUP_COLS]; int gk_word[GX_MAX_GROUP_COLS], gk_shift[GX_MAX_GROUP_COLS], gk_bytes[GX_MAX_GROUP_COLS], gk_pbit[GX_MAX_GROUP_COLS];
};

__device__ __forceinline__ bool runagg_probe(const gx_agg_dev &A, long long key, unsigned long long &payload)
{
    bool found = false;
    if (key == GX_EMPTY_KEY) { found = A.special_count > 0; if (found) payload = A.special[0]; return found; }
    unsigned long long p = gx_slot_index(key, A.sf);
    for (;;) {
        const gx_slot2 c = ld_slot2(A.slots + p);
        found = (c.k0 == key) | (c.k1 == key);
        payload = c.k0 == key ? c.p0 : c.p1;
        if (found | (c.k0 == GX_EMPTY_KEY) | (c.k1 == GX_EMPTY_KEY)) break;
        p = gx_next_pair(p, A.mask);
    }
    return found;
}

// quals of FOUR CONSECUTIVE rows starting at r0 (a multiple of 4): one 128-bit load per 4-byte column, two per 8-byte one
__device__ __forceinline__ void pred_vec4(const gx_dpred &p, long long r0, bool (&ok)[4])
{
    if (p.col.nulls == nullptr && (p.col.type == GX_INT4 || p.col.type == GX_DATE)) {
        const int4 v = ld_stream_i4((const int *) p.col.data + r0);
        const int x[4] = { v.x, v.y, v.z, v.w };
#pragma unroll
        for (int i = 0; i < 4; i++) ok[i] = ok[i] && gx_op_holds(p.op, (long long) x[i] > p.ival ? 1 : ((long long) x[i] < p.ival ? -1 : 0));
    } else if (p.col.nulls == nullptr && p.col.type == GX_FLOAT8) {
        const double2 a = ld_stream_d2((const double *) p.col.data + r0), b = ld_stream_d2((const double *) p.col.data + r0 + 2);
        const double x[4] = { a.x, a.y, b.x, b.y };
#pragma unroll
        for (int i = 0; i < 4; i++) ok[i] = ok[i] && gx_op_holds(p.op, gx_f8cmp(x[i], p.fval));
    } else {
#pragma unroll
        for (int i = 0; i < 4; i++) if (ok[i]) ok[i] = gx_eval_pred(p, r0 + i);
    }
}

// The kernel.  A lane owns FOUR CONSECUTIVE rows of a 128-row tile (128-bit loads for every column), folds them
// serially into runs, and only the runs' boundaries meet other lanes: a warp scan numbers the run heads, a run that
// starts in a lane is written to the per-warp list by that lane, the rows that continue a run begun further left
// are added to its list entry with a shared-memory atomic.  Entry 0 of the list is the run left open by the previous
// tile (the carry), so a run may span any number of lanes and tiles of the warp's chunk.  All entries but the last
// are then complete and are processed densely, one run per lane (probe, final record); the last becomes the carry.
template <int NV, int NC, int DENSE = 0>                      // DENSE: two CTAs of 512 threads per SM (64 registers) instead of two of 384 (80)
__global__ void __launch_bounds__(DENSE ? 512 : (NV <= 2 ? 384 : 512), (DENSE || NV <= 2) ? 2 : 1) gx_k_runagg(const __grid_constant__ gx_agg_dev A, const __grid_constant__ gx_runagg_args R)
{
    extern __shared__ unsigned long long smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    const int nv = R.nv;
    // per-warp list: key[RA_LIST], sum[nv][RA_LIST], cnt[RA_LIST]
    const size_t per_warp = (size_t) RA_LIST * (1 + nv) + RA_LIST / 2;
    unsigned long long *base = smem + (size_t) warp * per_warp;
    long long *Qkey = (long long *) base;
    double *Qsum = (double *) (base + RA_LIST);
    unsigned int *Qcnt = (unsigned int *) (base + (size_t) RA_LIST * (1 + nv));
    const gx_dplan &P = A.P;
    const long long *okey = (const long long *) P.okey.data;
    const int RW = 3 + P.nwords;
    const long long gw = (long long) blockIdx.x * nwarps + warp;
    const long long c0 = A.row0 + gw * R.rows_per_warp;
    long long c1 = c0 + R.rows_per_warp; if (c1 > A.row1) c1 = A.row1;
    if (c0 >= c1) return;
    const unsigned int lt = (1u << lane) - 1;
    bool bad = false;

    // entries [0, n) of the list: probe, then a final record (or, for a run that touches the chunk's edge, the global table)
    auto flush = [&](int n) {
        for (int b = 0; b < n; b += 32) {
            const int i = b + lane;
            const bool valid = i < n;
            const long long key = valid ? Qkey[i] : 0;
            const unsigned int craw = valid ? Qcnt[i] : 0u, cnt = craw & ~RA_BND;
            const bool bnd = (craw & RA_BND) != 0;
            unsigned long long payload = 0;
            const bool hit = valid && cnt > 0 && runagg_probe(A, key, payload);
            __syncwarp();
            unsigned long long k0 = 0, k1 = 0;
            if (hit) {
#pragma unroll
                for (int c = 0; c < GX_MAX_GROUP_COLS; c++) {
                    if (c >= R.ngk) break;
                    unsigned long long v = R.gk_from_key[c] ? (unsigned long long) key : (payload >> R.gk_pbit[c]);
                    if (R.gk_bytes[c] < 8) v &= (1ULL << (8 * R.gk_bytes[c])) - 1;
                    if (R.gk_word[c] == 0) k0 |= v << R.gk_shift[c]; else k1 |= v << R.gk_shift[c];
                }
            }
            const unsigned int dm = __ballot_sync(0xffffffffu, hit && !bnd);
            if (dm) {
                long long pos = 0;
                if (lane == 0) pos = (long long) atomicAdd((unsigned long long *) R.cursor, (unsigned long long) __popc(dm));
                pos = __shfl_sync(0xffffffffu, pos, 0) + __popc(dm & lt);
                if (hit && !bnd) {
                    if (pos < R.out_cap) {
                        unsigned long long *rec = R.out + (size_t) pos * RW;
                        rec[0] = 0; rec[1] = k0; rec[2] = k1;
                        for (int w = 0; w < P.nwords; w++) rec[3 + w] = (unsigned long long) A.winit[w];
                        rec[3] = (unsigned long long) cnt;
#pragma unroll
                        for (int q = 0; q < NV; q++) if (q < nv) rec[3 + R.vword[q]] = (unsigned long long) __double_as_longlong(Qsum[(size_t) q * RA_LIST + i]);
                    } else atomicOr((unsigned long long *) &A.counters[1], 4ULL);
                }
            }
            if (hit && bnd) {                                   // a run that may continue in the neighbouring chunk
                unsigned long long *rec = global_upsert(A, k0, k1, 0u);
                if (!rec) atomicOr((unsigned long long *) &A.counters[1], 2ULL);
                else {
                    atomicAdd(&rec[3], (unsigned long long) cnt);
#pragma unroll
                    for (int q = 0; q < NV; q++) if (q < nv) atomicAdd((double *) &rec[3 + R.vword[q]], Qsum[(size_t) q * RA_LIST + i]);
                }
            }
        }
        __syncwarp();
    };

    // entry cbase = the open run (the carry); entries [0, cbase) are finished runs waiting for a full round of 32.
    // At the start: the chunk's first key, nothing counted yet; it may have begun in the previous chunk.
    int cbase = 0;
    long long carry_key = __ldg(okey + c0);
    if (c0 > A.row0) bad |= carry_key < __ldg(okey + c0 - 1);
    if (lane == 0) {
        Qkey[0] = carry_key; Qcnt[0] = RA_BND;
#pragma unroll
        for (int q = 0; q < NV; q++) if (q < nv) Qsum[(size_t) q * RA_LIST] = 0.0;
    }
    __syncwarp();

    for (long long t0 = c0; t0 < c1; t0 += 128) {
        const long long r0 = t0 + lane * 4;
        long long k[4]; bool ok[4]; double x[NC][4];
        if ((R.pf & 1) && t0 + 384 <= c1) {
            // the warp walks its chunk front to back: the lines of the tile after the next one are asked for now
            // (8 lanes per column, one 128-byte line each; the host lists the columns), so the loads below find their rows in L2
            const int it = lane >> 3, li = lane & 7;
            if (it < R.pf_n && li < R.pf_lines[it]) asm volatile("prefetch.global.L2 [%0];" :: "l"(R.pf_ptr[it] + (t0 + 256) * R.pf_size[it] + li * 128));
        }
        if (t0 + 128 <= c1) {                                   // full tile: 128-bit loads, everything requested before use
            const longlong2 ka = ld_stream_ll2(okey + r0), kb = ld_stream_ll2(okey + r0 + 2);
            k[0] = ka.x; k[1] = ka.y; k[2] = kb.x; k[3] = kb.y;
#pragma unroll
            for (int c = 0; c < NC; c++) {
                if (c < R.nc) { const double2 a = ld_stream_d2(R.col[c] + r0), b = ld_stream_d2(R.col[c] + r0 + 2); x[c][0] = a.x; x[c][1] = a.y; x[c][2] = b.x; x[c][3] = b.y; }
                else { x[c][0] = x[c][1] = x[c][2] = x[c][3] = 0.0; }
            }
            ok[0] = ok[1] = ok[2] = ok[3] = true;
            for (int p = 0; p < P.npreds; p++) pred_vec4(P.preds[p], r0, ok);
        } else {                                                // the chunk's last, partial tile: rows past the end extend the last run with nothing
            const long long last = c1 - 1;
#pragma unroll
            for (int i = 0; i < 4; i++) {
                const long long r = r0 + i < c1 ? r0 + i : last;
                k[i] = __ldg(okey + r); ok[i] = r0 + i < c1;
#pragma unroll
                for (int c = 0; c < NC; c++) x[c][i] = c < R.nc ? __ldg(R.col[c] + r) : 0.0;
                for (int p = 0; p < P.npreds; p++) if (ok[i]) ok[i] = gx_eval_pred(P.preds[p], r);
            }
        }
        if ((R.pf & 2) && k[0] != GX_EMPTY_KEY) asm volatile("prefetch.global.L2 [%0];" :: "l"(A.slots + gx_slot_index(k[0], A.sf)));
        // aggregate arguments of the lane's four rows
        double v[NV][4];
#pragma unroll
        for (int q = 0; q < NV; q++) {
#pragma unroll
            for (int i = 0; i < 4; i++) v[q][i] = 0.0;
            if (q < nv) {
                const gx_dexpr &e = P.aggs[R.vagg[q]].expr;
                slot_term<4, NC>(e.t[0], R.tslot[q][0], x, v[q]);
                for (int t = 1; t < e.nterms; t++) {
                    double y[4];
                    slot_term<4, NC>(e.t[t], R.tslot[q][t], x, y);
                    const int op = e.t[t].op;
#pragma unroll
                    for (int i = 0; i < 4; i++) v[q][i] = op == GX_OP_ADD ? __dadd_rn(v[q][i], y[i]) : (op == GX_OP_SUB ? __dsub_rn(v[q][i], y[i]) : __dmul_rn(v[q][i], y[i]));
                }
            }
        }
        // ---- run heads, their numbering inside the warp, order check
        long long prevk = __shfl_up_sync(0xffffffffu, k[3], 1);
        if (lane == 0) prevk = carry_key;
        bad |= (k[0] < prevk) | (k[1] < k[0]) | (k[2] < k[1]) | (k[3] < k[2]);
        bool hd[4];
        hd[0] = k[0] != prevk; hd[1] = k[1] != k[0]; hd[2] = k[2] != k[1]; hd[3] = k[3] != k[2];
        const int nh = (int) hd[0] + (int) hd[1] + (int) hd[2] + (int) hd[3];
        int inc = nh;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
        const int ebase = cbase + inc - nh;                     // list entry of the run that is open when this lane starts (cbase = the carry)
        const int nheads = __shfl_sync(0xffffffffu, inc, 31);
        // ---- fold: runs that start in this lane are written, the rows continuing an earlier run are added to it afterwards
        unsigned int cc = 0; double cs[NV];                    // the continuing part
#pragma unroll
        for (int q = 0; q < NV; q++) cs[q] = 0.0;
        {
            int e = ebase; unsigned int c = 0; double sacc[NV];
#pragma unroll
            for (int q = 0; q < NV; q++) sacc[q] = 0.0;
#pragma unroll
            for (int i = 0; i < 4; i++) {
                if (hd[i]) {
                    if (e > ebase) { Qcnt[e] = c;
#pragma unroll
                        for (int q = 0; q < NV; q++) if (q < nv) Qsum[(size_t) q * RA_LIST + e] = sacc[q]; }
                    else { cc = c;
#pragma unroll
                        for (int q = 0; q < NV; q++) cs[q] = sacc[q]; }
                    e++; Qkey[e] = k[i]; c = 0;
#pragma unroll
                    for (int q = 0; q < NV; q++) sacc[q] = 0.0;
                }
                if (ok[i]) { c++;
#pragma unroll
                    for (int q = 0; q < NV; q++) if (q < nv) sacc[q] = __dadd_rn(sacc[q], v[q][i]); }
            }
            if (e > ebase) { Qcnt[e] = c;
#pragma unroll
                for (int q = 0; q < NV; q++) if (q < nv) Qsum[(size_t) q * RA_LIST + e] = sacc[q]; }
            else { cc = c;
#pragma unroll
                for (int q = 0; q < NV; q++) cs[q] = sacc[q]; }
        }
        __syncwarp();
        if (cc) {
            atomicAdd(&Qcnt[ebase], cc);
#pragma unroll
            for (int q = 0; q < NV; q++) if (q < nv) atomicAdd(&Qsum[(size_t) q * RA_LIST + ebase], cs[q]);
        }
        __syncwarp();
        // ---- entries [0, cbase + nheads) are finished, entry cbase + nheads is the new carry.  Finished runs are
        // processed in FULL rounds of 32 (one run per lane); the remainder waits at the front of the list.
        {
            const int done = cbase + nheads, full = done & ~31;
            if (full > 0) {
                flush(full);
                const int rest = done - full + 1;                   // unprocessed finished runs + the carry
                for (int i = lane; i < rest; i += 32) {             // rest <= 32: one pass, no overlap hazards (source index >= 32)
                    const long long kk = Qkey[full + i]; const unsigned int cq = Qcnt[full + i];
                    double sq[NV];
#pragma unroll
                    for (int q = 0; q < NV; q++) sq[q] = q < nv ? Qsum[(size_t) q * RA_LIST + full + i] : 0.0;
                    __syncwarp(__activemask());
                    Qkey[i] = kk; Qcnt[i] = cq;
#pragma unroll
                    for (int q = 0; q < NV; q++) if (q < nv) Qsum[(size_t) q * RA_LIST + i] = sq[q];
                }
                __syncwarp();
            }
            cbase = done - full;
        }
        carry_key = __shfl_sync(0xffffffffu, k[3], 31);
    }
    // the last run of the chunk may continue in the next chunk
    if (lane == 0) Qcnt[cbase] |= RA_BND;
    __syncwarp();
    flush(cbase + 1);
    if (__any_sync(0xffffffffu, bad) && lane == 0) atomicOr((unsigned long long *) &A.counters[1], 8ULL);
}

// global table -> dense records [meta][k0][k1][w..]
__global__ void gx_k_compact_groups(const unsigned long long *g_tab, long long g_cap, int nwords,
                                    unsigned long long *recs, long long *cursor)
{
    const int RW = 3 + nwords;
    long long stride = (long long) gridDim.x * blockDim.x;
    for (long long i = (long long) blockIdx.x * blockDim.x + threadIdx.x; i < g_cap; i += stride) {
        const unsigned long long *src = g_tab + i * RW;
        unsigned long long t = src[0];
        if (t == 0) continue;
        long long dst = (long long) atomicAdd((unsigned long long *) cursor, 1ULL);
        unsigned long long *d = recs + dst * RW;
        d[0] = (t >> 59) & 0xF;
        for (int j = 1; j < RW; j++) d[j] = src[j];
    }
}

// ----------------------------------------------------- radix pass 1 & 2
#define RADIX_MAX_BITS 13

__device__ __forceinline__ unsigned int rec_partition(const unsigned long long *rec, int bits)
{
    unsigned long long h = group_hash(rec[1], rec[2], (unsigned int) rec[0]);
    return (unsigned int) (h >> (64 - bits));
}

// histogram: hist[part * nblocks + block]
__global__ void __launch_bounds__(512) gx_k_radix_hist(const unsigned long long *recs, long long nrec, int RW, int bits, long long *hist)
{
    extern __shared__ unsigned int sh[];
    const int P = 1 << bits;
    for (int i = threadIdx.x; i < P; i += blockDim.x) sh[i] = 0;
    __syncthreads();
    long long per = (nrec + gridDim.x - 1) / gridDim.x, b = per * blockIdx.x, e = min(nrec, b + per);
    for (long long i = b + threadIdx.x; i < e; i += blockDim.x) atomicAdd(&sh[rec_partition(recs + i * RW, bits)], 1u);
    __syncthreads();
    for (int i = threadIdx.x; i < P; i += blockDim.x) hist[(long long) i * gridDim.x + blockIdx.x] = sh[i];
}
__global__ void __launch_bounds__(512) gx_k_radix_scatter(const unsigned long long *recs, long long nrec, int RW, int bits,
                                                         const long long *offs, unsigned long long *out)
{
    extern __shared__ unsigned int sh[];       // per-partition cursor within this block's slice
    const int P = 1 << bits;
    for (int i = threadIdx.x; i < P; i += blockDim.x) sh[i] = 0;
    __syncthreads();
    long long per = (nrec + gridDim.x - 1) / gridDim.x, b = per * blockIdx.x, e = min(nrec, b + per);
    for (long long i = b + threadIdx.x; i < e; i += blockDim.x) {
        const unsigned long long *src = recs + i * RW;
        unsigned int p = rec_partition(src, bits);
        unsigned int k = atomicAdd(&sh[p], 1u);
        unsigned long long *dst = out + (offs[(long long) p * gridDim.x + blockIdx.x] + k) * RW;
        for (int j = 0; j < RW; j++) dst[j] = src[j];
    }
}

// pass 2: one CTA per partition (grid-strided); aggregates the partition in a
// shared-memory table and appends its groups to the dense output.
__global__ void __launch_bounds__(512) gx_k_radix_agg(const gx_agg_dev A, const unsigned long long *recs, const long long *part_begin,
                                                      int nparts, int nblk, unsigned long long *out, long long *cursor, int *overflowed)
{
    extern __shared__ unsigned long long smem[];
    __shared__ long long s_base; __shared__ int s_cnt, s_over;
    const int RW = 3 + A.P.nwords;
    SmemTable T; T.S = A.s_slots; T.log2S = A.s_log2; T.nwords = A.P.nwords; T.nkw = 2; T.tagkey = 0; T.gmax = 0;
    T.gidx = nullptr; T.gcount = nullptr;
    T.tag = smem; T.k0 = T.tag + T.S; T.k1 = T.k0 + T.S; T.w = T.k1 + T.S;
    for (int part = blockIdx.x; part < nparts; part += gridDim.x) {
        long long b = part_begin[(long long) part * nblk];
        long long e = (part + 1 < nparts) ? part_begin[(long long) (part + 1) * nblk] : A.rec_cap;
        for (int i = threadIdx.x; i < T.S; i += blockDim.x) {
            T.tag[i] = 0;
            for (int j = 0; j < T.nwords; j++) T.w[(size_t) i * T.nwords + j] = (unsigned long long) A.winit[j];
        }
        if (threadIdx.x == 0) { s_cnt = 0; s_over = 0; }
        __syncthreads();
        for (long long i = b + threadIdx.x; i < e; i += blockDim.x) {
            const unsigned long long *rec = recs + i * RW;
            int s = smem_upsert<false>(T, rec[1], rec[2], (unsigned int) rec[0]);
            if (s < 0) { s_over = 1; continue; }
            for (int j = 0; j < T.nwords; j++) merge_word(&T.w[(size_t) s * T.nwords + j], A.wkind[j], rec[3 + j]);
        }
        __syncthreads();
        if (s_over) { if (threadIdx.x == 0) overflowed[part] = 1; __syncthreads(); continue; }
        int mine = 0;
        for (int i = threadIdx.x; i < T.S; i += blockDim.x) mine += T.tag[i] != 0;
        int pos = mine ? atomicAdd(&s_cnt, mine) : 0;
        __syncthreads();
        if (threadIdx.x == 0) s_base = (long long) atomicAdd((unsigned long long *) cursor, (unsigned long long) s_cnt);
        __syncthreads();
        for (int i = threadIdx.x; i < T.S; i += blockDim.x) {
            unsigned long long t = T.tag[i];
            if (t == 0) continue;
            unsigned long long *d = out + (s_base + pos++) * RW;
            d[0] = (t >> 59) & 0xF; d[1] = T.k0[i]; d[2] = T.k1[i];
            for (int j = 0; j < T.nwords; j++) d[3 + j] = T.w[(size_t) i * T.nwords + j];
        }
        __syncthreads();
    }
}

// fallback for partitions that did not fit shared memory, and the generic
// "merge records into the global table" used by gx_result_combine
__global__ void gx_k_merge_records(const gx_agg_dev A, const unsigned long long *recs, const long long *part_begin, int nblk,
                                   const int *sel /* may be NULL: all */, int nparts, long long nrec)
{
    const int RW = 3 + A.P.nwords;
    if (!sel) {
        long long stride = (long long) gridDim.x * blockDim.x;
        for (long long i = (long long) blockIdx.x * blockDim.x + threadIdx.x; i < nrec; i += stride) {
            const unsigned long long *rec = recs + i * RW;
            unsigned long long *g = global_upsert(A, rec[1], rec[2], (unsigned int) rec[0]);
            if (!g) { atomicOr((unsigned long long *) &A.counters[1], 2ULL); continue; }
            for (int j = 0; j < A.P.nwords; j++) merge_word(&g[3 + j], A.wkind[j], rec[3 + j]);
        }
        return;
    }
    for (int part = blockIdx.x; part < nparts; part += gridDim.x) {
        if (!sel[part]) continue;
        long long b = part_begin[(long long) part * nblk];
        long long e = (part + 1 < nparts) ? part_begin[(long long) (part + 1) * nblk] : nrec;
        for (long long i = b + threadIdx.x; i < e; i += blockDim.x) {
            const unsigned long long *rec = recs + i * RW;
            unsigned long long *g = global_upsert(A, rec[1], rec[2], (unsigned int) rec[0]);
            if (!g) { atomicOr((unsigned long long *) &A.counters[1], 2ULL); continue; }
            for (int j = 0; j < A.P.nwords; j++) merge_word(&g[3 + j], A.wkind[j], rec[3 + j]);
        }
    }
}

// Finalize over an all-gathered buffer of partial states (gx_result_combine's small-result
// path): segment p = [ngroups_p][flags_p][cap records of RW words].  Every rank sees every
// partial record and keeps the groups it OWNS (the same key hash the redistribute path
// uses), so the union over ranks holds each group exactly once — the contract of
// "Distribute results by S -> Finalize HashAggregate" (xc_groupby.out:193-205) without a
// partition step, a count exchange or a host round trip.
__global__ void gx_k_merge_gathered(const gx_agg_dev A, const unsigned long long *gathered, int nseg, long long cap, int rank, int nranks)
{
    const int RW = 3 + A.P.nwords;
    const long long seg_words = 2 + cap * RW, total = (long long) nseg * cap;
    const long long stride = (long long) gridDim.x * blockDim.x;
    for (long long i = (long long) blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        const int p = (int) (i / cap); const long long j = i - (long long) p * cap;
        const unsigned long long *seg = gathered + (long long) p * seg_words;
        if (seg[1]) { if (j == 0) atomicOr((unsigned long long *) &A.counters[3], 1ULL); continue; }   // that rank had more than cap groups
        if (j >= (long long) seg[0]) continue;
        const unsigned long long *rec = seg + 2 + j * RW;
        const unsigned long long h = gx_mix64(rec[1] ^ (rec[2] * 0x9E3779B97F4A7C15ULL) ^ (rec[0] << 56));
        if ((int) (h % (unsigned long long) nranks) != rank) continue;
        unsigned long long *g = global_upsert(A, rec[1], rec[2], (unsigned int) rec[0]);
        if (!g) { atomicOr((unsigned long long *) &A.counters[1], 2ULL); continue; }
        for (int w = 0; w < A.P.nwords; w++) merge_word(&g[3 + w], A.wkind[w], rec[3 + w]);
    }
}
__global__ void gx_k_pack_partial(const unsigned long long *recs, long long n, long long cap, int RW, unsigned long long *out)
{
    const long long stride = (long long) gridDim.x * blockDim.x;
    const bool big = n > cap;
    if (blockIdx.x == 0 && threadIdx.x == 0) { out[0] = big ? 0ULL : (unsigned long long) n; out[1] = big ? 1ULL : 0ULL; }
    if (big) return;
    for (long long i = (long long) blockIdx.x * blockDim.x + threadIdx.x; i < n * RW; i += stride) out[2 + i] = recs[i];
}

__global__ void gx_k_scan_i64(long long *v, long long n, long long *total);   // below

// ============================================================ host side
static gx_dcol dcol_of(const gx_table *t, int c)
{
    gx_dcol d; d.data = t->cols[c]; d.nulls = t->nulls[c]; d.type = t->types[c]; d._pad = 0; return d;
}

// postfix -> chain form; returns false when the shape is not representable
struct sym { int is_chain; gx_dexpr e; };
static bool compile_expr(gx_ctx *ctx, const gx_table *t, const gx_expr *in, gx_dexpr *out, bool *nullable)
{
    sym st[GX_MAX_EXPR_OPS]; int sp = 0;
    *nullable = false;
    for (int i = 0; i < in->nops; i++) {
        const gx_expr_op *op = &in->ops[i];
        if (op->op == GX_OP_COL) {
            if (op->col < 0 || op->col >= t->ncols) { GX_SET_ERR(ctx, "expression: column %d out of range", op->col); return false; }
            sym s; memset(&s, 0, sizeof(s)); s.e.nterms = 1; s.e.t[0].kind = GXT_COL; s.e.t[0].col = dcol_of(t, op->col);
            if (t->nulls[op->col]) *nullable = true;
            st[sp++] = s;
        } else if (op->op == GX_OP_CONST) {
            sym s; memset(&s, 0, sizeof(s)); s.e.nterms = 1; s.e.t[0].kind = GXT_CONST; s.e.t[0].k = op->k;
            st[sp++] = s;
        } else if (op->op == GX_OP_ADD || op->op == GX_OP_SUB || op->op == GX_OP_MUL) {
            if (sp < 2) { GX_SET_ERR(ctx, "expression: stack underflow"); return false; }
            sym b = st[--sp], a = st[--sp];
            if (b.is_chain) { GX_SET_ERR(ctx, "expression shape not supported (right operand is a compound expression)"); return false; }
            gx_dterm bt = b.e.t[0];
            if (!a.is_chain) {
                gx_dterm at = a.e.t[0];
                // leaf (op) leaf -> a single composite term where one exists
                if (at.kind == GXT_CONST && bt.kind == GXT_COL) {
                    sym s; memset(&s, 0, sizeof(s)); s.e.nterms = 1; s.e.t[0] = bt; s.e.t[0].k = at.k;
                    s.e.t[0].kind = op->op == GX_OP_ADD ? GXT_K_ADD_COL : op->op == GX_OP_SUB ? GXT_K_SUB_COL : GXT_K_MUL_COL;
                    st[sp++] = s; continue;
                }
                if (at.kind == GXT_COL && bt.kind == GXT_CONST) {
                    sym s; memset(&s, 0, sizeof(s)); s.e.nterms = 1; s.e.t[0] = at; s.e.t[0].k = bt.k;
                    s.e.t[0].kind = op->op == GX_OP_ADD ? GXT_K_ADD_COL : op->op == GX_OP_SUB ? GXT_COL_SUB_K : GXT_K_MUL_COL;
                    st[sp++] = s; continue;
                }
                if (at.kind == GXT_CONST && bt.kind == GXT_CONST) {
                    sym s; memset(&s, 0, sizeof(s)); s.e.nterms = 1; s.e.t[0].kind = GXT_CONST;
                    s.e.t[0].k = op->op == GX_OP_ADD ? at.k + bt.k : op->op == GX_OP_SUB ? at.k - bt.k : at.k * bt.k;
                    st[sp++] = s; continue;
                }
            }
            if (a.e.nterms >= 4) { GX_SET_ERR(ctx, "expression too long (more than 4 terms)"); return false; }
            a.is_chain = 1;
            bt.op = op->op;
            a.e.t[a.e.nterms++] = bt;
            st[sp++] = a;
        } else { GX_SET_ERR(ctx, "expression: unknown opcode %d", op->op); return false; }
    }
    if (sp != 1) { GX_SET_ERR(ctx, "expression: malformed postfix program"); return false; }
    *out = st[0].e;
    return true;
}

struct compiled_plan {
    gx_agg_dev A;
    int32_t group_types[GX_MAX_GROUP_COLS];
    int gword[GX_MAX_GROUP_COLS], gshift[GX_MAX_GROUP_COLS], gbytes[GX_MAX_GROUP_COLS];
    int agg_word[GX_MAX_AGGS], agg_cnt_word[GX_MAX_AGGS];
    int need_w0;
};

static int compile_plan(gx_ctx *ctx, const gx_table *outer, const gx_hash *h, const gx_agg_plan *plan, compiled_plan *cp)
{
    memset(cp, 0, sizeof(*cp));
    gx_dplan &P = cp->A.P;
    GX_CHECK_ARG(ctx, plan->n_aggs >= 0 && plan->n_aggs <= GX_MAX_AGGS, "agg plan: n_aggs %d", plan->n_aggs);
    GX_CHECK_ARG(ctx, plan->n_group_cols >= 0 && plan->n_group_cols <= GX_MAX_GROUP_COLS, "agg plan: n_group_cols %d", plan->n_group_cols);
    P.npreds = plan->n_preds;
    int rc = gx_fill_dpreds(ctx, outer, plan->n_preds, plan->preds, P.preds); if (rc) return rc;
    P.has_join = plan->outer_key_col >= 0;
    if (P.has_join) {
        GX_CHECK_ARG(ctx, h != nullptr, "agg plan: join requested but no hash table given");
        GX_CHECK_ARG(ctx, plan->outer_key_col < outer->ncols, "agg plan: outer key column out of range");
        int kt = outer->types[plan->outer_key_col];
        GX_CHECK_ARG(ctx, kt == GX_INT4 || kt == GX_INT8 || kt == GX_DATE, "agg plan: outer key type %d not supported", kt);
        P.okey = dcol_of(outer, plan->outer_key_col); P.key_type = kt; P.unique = h->unique;
        P.n_payload = h->n_payload;
        for (int i = 0; i < h->n_payload; i++) P.payload_types[i] = h->payload_types[i];
        cp->A.slots = h->slots; cp->A.mask = (unsigned long long) h->nslots - 1;
        cp->A.cslots = h->cslots; cp->A.cspan = h->cspan;
        cp->A.special = h->special_payload; cp->A.special_count = h->special_count;
        cp->A.sf.mode = h->mode; cp->A.sf.win = h->win; cp->A.sf.shift = h->shift; cp->A.sf.amask = h->amask; cp->A.sf.kmin = h->kmin; cp->A.sf.scale = h->scale; cp->A.sf.mask = (unsigned long long) h->nslots - 1;
    }
    // group columns: pack by byte width into k0 then k1
    int used[2] = { 0, 0 };
    P.ngroup = plan->n_group_cols;
    for (int c = 0; c < plan->n_group_cols; c++) {
        gx_dgroupcol &g = P.gcols[c];
        g.side = plan->group_cols[c].side;
        int type;
        if (g.side == 0) {
            int col = plan->group_cols[c].col;
            GX_CHECK_ARG(ctx, col >= 0 && col < outer->ncols, "agg plan: group column %d out of range", col);
            g.col = dcol_of(outer, col); type = outer->types[col];
        } else {
            GX_CHECK_ARG(ctx, h != nullptr && h->n_payload > 0, "agg plan: group column refers to a join payload but none is carried");
            int pi = plan->group_cols[c].col;
            GX_CHECK_ARG(ctx, pi >= 0 && pi < h->n_payload, "agg plan: payload index %d out of range", pi);
            int bit = 0;
            for (int i = 0; i < pi; i++) bit += 8 * gx_type_size(h->payload_types[i]);
            g.payload_idx = bit; type = h->payload_types[pi];
        }
        g.type = type; g.bytes = gx_type_size(type);
        int w = (used[0] + g.bytes <= 8) ? 0 : 1;
        GX_CHECK_ARG(ctx, used[w] + g.bytes <= 8, "agg plan: group key wider than 16 bytes");
        g.word = w; g.shift = 8 * used[w]; used[w] += g.bytes;
        cp->group_types[c] = type; cp->gword[c] = g.word; cp->gshift[c] = g.shift; cp->gbytes[c] = g.bytes;
    }
    P.nkw = used[1] ? 2 : 1;
    // aggregates
    int nw = 1;                                     // w0 = row count
    cp->A.wkind[0] = WK_ADD_I64; cp->A.winit[0] = 0;
    P.nagg = plan->n_aggs;
    for (int a = 0; a < plan->n_aggs; a++) {
        gx_dagg &g = P.aggs[a];
        const gx_agg &src = plan->aggs[a];
        bool nullable = false;
        auto new_word = [&](int kind, long long init) { cp->A.wkind[nw] = kind; cp->A.winit[nw] = init; return nw++; };
        if (nw + 2 > GX_MAX_WORDS) { GX_SET_ERR(ctx, "agg plan: too many state words"); return GX_ERR_ARG; }
        switch (src.fn) {
            case GX_AGG_COUNT_STAR: g.kind = GXU_NONE; cp->agg_word[a] = 0; cp->need_w0 = 1; break;
            case GX_AGG_COUNT: case GX_AGG_SUM_I4: case GX_AGG_SUM_I8: {
                GX_CHECK_ARG(ctx, src.arg.nops == 1 && src.arg.ops[0].op == GX_OP_COL, "agg %d: argument must be a plain column", a);
                int col = src.arg.ops[0].col;
                GX_CHECK_ARG(ctx, col >= 0 && col < outer->ncols, "agg %d: column out of range", a);
                int t = outer->types[col];
                if (src.fn == GX_AGG_SUM_I4) GX_CHECK_ARG(ctx, t == GX_INT4, "agg %d: sum(int4) needs an int4 column", a);
                if (src.fn == GX_AGG_SUM_I8) GX_CHECK_ARG(ctx, t == GX_INT8, "agg %d: sum(int8) needs an int8 column", a);
                g.is_int = 1; g.icol = dcol_of(outer, col); nullable = outer->nulls[col] != nullptr;
                if (src.fn == GX_AGG_COUNT) {
                    if (nullable) { g.kind = GXU_CNT; g.word = new_word(WK_ADD_I64, 0); cp->agg_word[a] = g.word; }
                    else { g.kind = GXU_NONE; cp->agg_word[a] = 0; cp->need_w0 = 1; }
                } else {
                    g.kind = GXU_ADD_I64; g.word = new_word(WK_ADD_I64, 0); cp->agg_word[a] = g.word;
                    g.cnt_word = nullable ? new_word(WK_ADD_I64, 0) : 0; cp->agg_cnt_word[a] = g.cnt_word;
                }
                break;
            }
            case GX_AGG_SUM_F8: case GX_AGG_AVG_F8: case GX_AGG_MIN_F8: case GX_AGG_MAX_F8: {
                GX_CHECK_ARG(ctx, src.arg.nops >= 1 && src.arg.nops <= GX_MAX_EXPR_OPS, "agg %d: missing argument expression", a);
                // sum(x) and avg(x) over the same argument keep ONE running sum (float8pl and float8_accum
                // add the same values in the same order: float.c:970, :2823) — Q1 has two such pairs
                if (src.fn == GX_AGG_SUM_F8 || src.fn == GX_AGG_AVG_F8) {
                    int twin = -1;
                    for (int b = 0; b < a && twin < 0; b++) {
                        const gx_agg &o = plan->aggs[b];
                        if ((o.fn != GX_AGG_SUM_F8 && o.fn != GX_AGG_AVG_F8) || o.arg.nops != src.arg.nops) continue;
                        bool same = true;
                        for (int k = 0; k < src.arg.nops && same; k++)
                            same = o.arg.ops[k].op == src.arg.ops[k].op && o.arg.ops[k].col == src.arg.ops[k].col &&
                                   memcmp(&o.arg.ops[k].k, &src.arg.ops[k].k, sizeof(double)) == 0;
                        if (same) twin = b;
                    }
                    if (twin >= 0) {
                        g.kind = GXU_NONE; cp->agg_word[a] = cp->agg_word[twin]; cp->agg_cnt_word[a] = cp->agg_cnt_word[twin];
                        if (cp->agg_cnt_word[a] == 0 && src.fn == GX_AGG_AVG_F8) cp->need_w0 = 1;
                        break;
                    }
                }
                if (!compile_expr(ctx, outer, &src.arg, &g.expr, &nullable)) return GX_ERR_ARG;
                if (src.fn == GX_AGG_MIN_F8) {        // identity of float8smaller under float8_cmp: NaN
                    double nan = __builtin_nan(""); long long bits; memcpy(&bits, &nan, 8);
                    g.kind = GXU_MIN_F64; g.word = new_word(WK_MIN_F64, bits);
                } else if (src.fn == GX_AGG_MAX_F8) { // identity of float8larger: -inf
                    double ninf = -__builtin_inf(); long long bits; memcpy(&bits, &ninf, 8);
                    g.kind = GXU_MAX_F64; g.word = new_word(WK_MAX_F64, bits);
                } else { g.kind = GXU_ADD_F64; g.word = new_word(WK_ADD_F64, 0); }
                cp->agg_word[a] = g.word;
                g.cnt_word = nullable ? new_word(WK_ADD_I64, 0) : 0; cp->agg_cnt_word[a] = g.cnt_word;
                if (!nullable && src.fn == GX_AGG_AVG_F8) cp->need_w0 = 1;    // N of float8_avg
                break;
            }
            default: GX_SET_ERR(ctx, "agg %d: unknown aggregate function %d", a, src.fn); return GX_ERR_ARG;
        }
    }
    P.nwords = nw;
    cp->A.row0 = 0; cp->A.row1 = outer->nrows;
    cp->A.counters = ctx->d_scratch + 8;
    return GX_OK;
}

int gx_result_alloc(gx_ctx *ctx, const gx_agg_plan *plan, const int32_t *group_types, int64_t cap, gx_result **out)
{
    gx_result *r = (gx_result *) calloc(1, sizeof(gx_result));
    r->ctx = ctx; r->plan = *plan; r->cap = cap < 1 ? 1 : cap;
    for (int c = 0; c < plan->n_group_cols; c++) r->group_types[c] = group_types[c];
    *out = r;
    return GX_OK;
}

static size_t smem_bytes_for(int S, int nkw, int nwords) { return (size_t) S * 8 * (1 + nkw + nwords); }

static int ilog2(long long x) { int l = 0; while ((1LL << l) < x) l++; return l; }

template <int SINK>
static int launch_agg(gx_ctx *ctx, const gx_agg_dev &A, size_t smem, const char *name, int threads = 1024)
{
    static bool attr_set[8] = { false };
    if (!attr_set[SINK]) {
        GX_CUDA(ctx, cudaFuncSetAttribute(gx_k_agg<SINK>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) ctx->smem_optin));
        attr_set[SINK] = true;
    }
    long long nrows = A.row1 - A.row0;
    long long nb = (nrows + threads - 1) / threads, maxb = (long long) ctx->sm_count;
    // the shared-memory counters are 32-bit per CTA
    while ((nrows + maxb - 1) / maxb >= (1LL << 32)) maxb *= 2;
    unsigned grid = (unsigned) (nb < maxb ? (nb > 0 ? nb : 1) : maxb);
    gx_launch_scope ls(ctx, name);
    gx_k_agg<SINK><<<grid, threads, smem, ctx->stream>>>(A);
    GX_CUDA(ctx, cudaGetLastError());
    return GX_OK;
}

template <int K>
static int launch_lptile_k(gx_ctx *ctx, const gx_agg_dev &A, size_t smem, const char *name, int threads)
{
    static bool attr_set = false;
    if (!attr_set) {
        GX_CUDA(ctx, cudaFuncSetAttribute(gx_k_agg_lptile<K>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) ctx->smem_optin));
        attr_set = true;
    }
    long long nrows = A.row1 - A.row0, per_block = (long long) (threads / 32) * 32 * K;
    long long nb = (nrows + per_block - 1) / per_block, maxb = (long long) ctx->sm_count;
    unsigned grid = (unsigned) (nb < maxb ? (nb > 0 ? nb : 1) : maxb);
    gx_launch_scope ls(ctx, name);
    gx_k_agg_lptile<K><<<grid, threads, smem, ctx->stream>>>(A);
    GX_CUDA(ctx, cudaGetLastError());
    return GX_OK;
}
static int launch_lptile(gx_ctx *ctx, const gx_agg_dev &A, size_t smem, const char *name, int threads)
{
    const char *k4 = getenv("GX_LPTILE_K4");
    if (threads <= 640 && !(k4 && k4[0] == '1')) return launch_lptile_k<8>(ctx, A, smem, name, threads);
    return launch_lptile_k<4>(ctx, A, smem, name, threads);
}

template <bool JOIN, bool HAS_CNT, bool HAS_SUM>
static int launch_fast_t(gx_ctx *ctx, const gx_agg_dev &A, const gx_fast_args &FA, size_t smem, const char *name)
{
    static bool attr_set = false;
    if (!attr_set) {
        GX_CUDA(ctx, cudaFuncSetAttribute(gx_k_fast<JOIN, HAS_CNT, HAS_SUM>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) ctx->smem_optin));
        attr_set = true;
    }
    long long nvec = (A.row1 - A.row0 + 3) / 4;
    long long nb = (nvec + 1023) / 1024, maxb = (long long) ctx->sm_count;
    while ((A.row1 - A.row0 + maxb - 1) / maxb >= (1LL << 32)) maxb *= 2;
    unsigned grid = (unsigned) (nb < maxb ? (nb > 0 ? nb : 1) : maxb);
    gx_launch_scope ls(ctx, name);
    gx_k_fast<JOIN, HAS_CNT, HAS_SUM><<<grid, 1024, smem, ctx->stream>>>(A, FA);
    GX_CUDA(ctx, cudaGetLastError());
    return GX_OK;
}
template <bool HAS_CNT, bool HAS_SUM, bool COMPACT>
static int launch_runjoin_t(gx_ctx *ctx, const gx_agg_dev &A, const gx_fast_args &FA, size_t smem, const char *name)
{
    static bool attr_set = false;
    if (!attr_set) {
        GX_CUDA(ctx, cudaFuncSetAttribute(gx_k_runjoin<HAS_CNT, HAS_SUM, COMPACT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) ctx->smem_optin));
        attr_set = true;
    }
    long long nvec = (A.row1 - A.row0 + 3) / 4;
    long long nb = (nvec + 1023) / 1024, maxb = (long long) ctx->sm_count;
    while ((A.row1 - A.row0 + maxb - 1) / maxb >= (1LL << 32)) maxb *= 2;
    unsigned grid = (unsigned) (nb < maxb ? (nb > 0 ? nb : 1) : maxb);
    gx_launch_scope ls(ctx, name);
    gx_k_runjoin<HAS_CNT, HAS_SUM, COMPACT><<<grid, 1024, smem, ctx->stream>>>(A, FA);
    GX_CUDA(ctx, cudaGetLastError());
    return GX_OK;
}
// Measured at SF100 on one B200 (profiles/r02_runjoin_variants.txt): gx_k_runjoin 2.787 ms, gx_k_runjoin_tma 2.660 ms, with the
// branch-free fold 2.617 ms, with full probe rounds only 2.514 ms (parity suite, the whole GPU suite, smoke and the bench checks
// green under it) -> 3 is the default; GX_RUNJOIN_TMA=0 restores gx_k_runjoin
#define GX_RUNJOIN_TMA_DEFAULT 3          /* 0 off, 1 gx_k_runjoin_tma, 2 + branch-free fold, 3 + probe rounds of 32 lanes only */
// gx_k_runjoin_seg: 31 consumer warps + 1 producer warp, the rest of the CTA's shared memory is the two-deep ring of
// join-table pieces.  0 slots = the ring does not fit next to this group table (the caller keeps gx_k_runjoin).
// Ring depth 3 when three buffers of the size a chunk is expected to need fit (table slots per outer row x 3968 rows, + 15 %
// and the two edge blocks), else 2 larger ones.
static unsigned int runjoin_seg_slots(const gx_ctx *ctx, size_t table_bytes, const gx_agg_dev &A, int *nbuf)
{
    const size_t fixed = table_bytes + GX_SEG_CW * sizeof(gx_runlist) + sizeof(gx_seg_ctl) + 1024;
    *nbuf = 2;
    if (fixed + 2 * 512 * 8 > ctx->smem_optin) return 0;
    const size_t avail = (ctx->smem_optin - fixed) / 8;
    const long long nrows = A.row1 - A.row0 > 0 ? A.row1 - A.row0 : 1;
    const double need = 1.15 * (double) (A.mask + 1ULL) / (double) nrows * (GX_SEG_CW * 128) + 96.0;
    const char *e = getenv("GX_RUNJOIN_SEG_BUFS");
    if (e && e[0]) { int v = atoi(e); if (v >= 2 && v <= GX_SEG_MAXBUF) *nbuf = v; }
    else if (need * 3.0 <= (double) avail) *nbuf = 3;
    size_t slots = avail / (size_t) *nbuf;
    if (slots > 4096) slots = 4096;                              // 32 KB per buffer
    return (unsigned int) (slots & ~(size_t) 31);
}
template <bool HAS_CNT, bool HAS_SUM>
static int launch_runjoin_seg_t(gx_ctx *ctx, const gx_agg_dev &A, const gx_fast_args &FA, size_t table_bytes, unsigned int seg_slots, int nbuf, const char *name)
{
    static bool attr_set = false;
    if (!attr_set) {
        GX_CUDA(ctx, cudaFuncSetAttribute(gx_k_runjoin_seg<HAS_CNT, HAS_SUM>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) ctx->smem_optin));
        attr_set = true;
    }
    const size_t smem = table_bytes + GX_SEG_CW * sizeof(gx_runlist) + (size_t) nbuf * seg_slots * 8 + sizeof(gx_seg_ctl);
    const long long nvec = (A.row1 - A.row0) >> 2, cvec = (long long) GX_SEG_CW * 32;
    long long nb = (nvec + cvec - 1) / cvec, maxb = (long long) ctx->sm_count;
    while ((A.row1 - A.row0 + maxb - 1) / maxb >= (1LL << 32)) maxb *= 2;      // 32-bit row counters per CTA
    unsigned grid = (unsigned) (nb < maxb ? (nb > 0 ? nb : 1) : maxb);
    gx_launch_scope ls(ctx, name);
    gx_launch_scope which(ctx, "probe_agg_seg", 0);              // same kernel under a second profile name: tells gx_profile_get() which variant ran
    gx_k_runjoin_seg<HAS_CNT, HAS_SUM><<<grid, 1024, smem, ctx->stream>>>(A, FA, seg_slots, nbuf);
    GX_CUDA(ctx, cudaGetLastError());
    return GX_OK;
}
template <bool HAS_CNT, bool HAS_SUM, bool COMPACT>
static int launch_runjoin3_t(gx_ctx *ctx, const gx_agg_dev &A, const gx_fast_args &FA, size_t table_bytes, const char *name)
{
    static bool attr_set = false;
    if (!attr_set) {
        GX_CUDA(ctx, cudaFuncSetAttribute(gx_k_runjoin3<HAS_CNT, HAS_SUM, COMPACT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) ctx->smem_optin));
        attr_set = true;
    }
    long long nvec = (A.row1 - A.row0 + 3) / 4;
    long long nb = (nvec + 1023) / 1024, maxb = (long long) ctx->sm_count;
    while ((A.row1 - A.row0 + maxb - 1) / maxb >= (1LL << 32)) maxb *= 2;
    unsigned grid = (unsigned) (nb < maxb ? (nb > 0 ? nb : 1) : maxb);
    gx_launch_scope ls(ctx, name);
    gx_k_runjoin3<HAS_CNT, HAS_SUM, COMPACT><<<grid, 1024, table_bytes + 32 * sizeof(gx_runlist3), ctx->stream>>>(A, FA);
    GX_CUDA(ctx, cudaGetLastError());
    return GX_OK;
}
template <bool HAS_SUM, bool COMPACT>
static int launch_runjoin_tma_t(gx_ctx *ctx, const gx_agg_dev &A, const gx_fast_args &FA, size_t smem, const char *name)
{
    static bool attr_set = false;
    if (!attr_set) {
        GX_CUDA(ctx, cudaFuncSetAttribute(gx_k_runjoin_tma<HAS_SUM, COMPACT, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) ctx->smem_optin));
        GX_CUDA(ctx, cudaFuncSetAttribute(gx_k_runjoin_tma<HAS_SUM, COMPACT, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) ctx->smem_optin));
        GX_CUDA(ctx, cudaFuncSetAttribute(gx_k_runjoin_tma<HAS_SUM, COMPACT, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) ctx->smem_optin));
        attr_set = true;
    }
    const char *fv = getenv("GX_RUNJOIN_TMA");
    const int variant = fv && fv[0] ? fv[0] - '0' : GX_RUNJOIN_TMA_DEFAULT;           // 2: the branch-free fold, 3: + full probe rounds only
    long long nvec = (A.row1 - A.row0 + 3) / 4;
    long long nb = (nvec + 1023) / 1024, maxb = (long long) ctx->sm_count;
    while ((A.row1 - A.row0 + maxb - 1) / maxb >= (1LL << 31)) maxb *= 2;      // 31-bit row counters per CTA
    unsigned grid = (unsigned) (nb < maxb ? (nb > 0 ? nb : 1) : maxb);
    gx_launch_scope ls(ctx, name);
    gx_launch_scope which(ctx, "probe_agg_tma", 0);              // second profile name: which variant ran
    if (variant == 3) gx_k_runjoin_tma<HAS_SUM, COMPACT, true, true><<<grid, 1024, smem, ctx->stream>>>(A, FA);
    else if (variant == 2) gx_k_runjoin_tma<HAS_SUM, COMPACT, true, false><<<grid, 1024, smem, ctx->stream>>>(A, FA);
    else gx_k_runjoin_tma<HAS_SUM, COMPACT, false, false><<<grid, 1024, smem, ctx->stream>>>(A, FA);
    GX_CUDA(ctx, cudaGetLastError());
    return GX_OK;
}
template <bool HAS_SUM, bool COMPACT>
static int launch_runjoin2_t(gx_ctx *ctx, const gx_agg_dev &A, const gx_fast_args &FA, const char *name)
{
    static bool attr_set = false;
    const size_t smem = (size_t) A.s_slots * 16 + 16 * sizeof(gx_runlist);
    if (!attr_set) {
        GX_CUDA(ctx, cudaFuncSetAttribute(gx_k_runjoin2<HAS_SUM, COMPACT>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem > 100 * 1024 ? (int) smem : 100 * 1024));
        attr_set = true;
    }
    long long nvec = (A.row1 - A.row0 + 3) / 4;
    long long nb = (nvec + 511) / 512, maxb = (long long) ctx->sm_count * 2;
    while ((A.row1 - A.row0 + maxb - 1) / maxb >= (1LL << 31)) maxb *= 2;      // 31-bit row counters per CTA
    unsigned grid = (unsigned) (nb < maxb ? (nb > 0 ? nb : 1) : maxb);
    gx_launch_scope ls(ctx, name);
    gx_k_runjoin2<HAS_SUM, COMPACT><<<grid, 512, smem, ctx->stream>>>(A, FA);
    GX_CUDA(ctx, cudaGetLastError());
    return GX_OK;
}
// GX_RUNJOIN_SEG=1/0 selects / forbids gx_k_runjoin_seg; a run that raised flag 16 (a bounded mbarrier wait gave up)
// switches it off for the rest of the process
#define GX_RUNJOIN_SEG_DEFAULT 0
static bool g_runjoin_seg_broken = false;
static bool gx_runjoin_seg_enabled()
{
    if (g_runjoin_seg_broken) return false;
    const char *e = getenv("GX_RUNJOIN_SEG");
    return e && e[0] ? e[0] != '0' : GX_RUNJOIN_SEG_DEFAULT != 0;
}
// GX_RUNJOIN_TMA=1/0 selects / forbids gx_k_runjoin_tma (same rules as GX_RUNJOIN_SEG)
static bool gx_runjoin_tma_enabled()
{
    if (g_runjoin_seg_broken) return false;
    const char *e = getenv("GX_RUNJOIN_TMA");
    return e && e[0] ? e[0] != '0' : GX_RUNJOIN_TMA_DEFAULT != 0;
}
static int launch_fast(gx_ctx *ctx, const gx_agg_dev &A, const gx_fast_args &FA, bool join, bool cnt, bool sum, size_t smem, const char *name, bool use_run)
{
    // gx_k_runjoin3: finished runs wait for a full round of 32 (GX_RUNJOIN_CARRY=1; A/B against gx_k_runjoin)
    {
        const char *cv = getenv("GX_RUNJOIN_CARRY");
        if (use_run && cv && cv[0] == '1' && smem + 32 * sizeof(gx_runlist3) <= ctx->smem_optin - 1024) {
            if (A.cslots) {
                if (cnt && sum) return launch_runjoin3_t<true, true, true>(ctx, A, FA, smem, name);
                if (cnt) return launch_runjoin3_t<true, false, true>(ctx, A, FA, smem, name);
                return launch_runjoin3_t<false, true, true>(ctx, A, FA, smem, name);
            }
            if (cnt && sum) return launch_runjoin3_t<true, true, false>(ctx, A, FA, smem, name);
            if (cnt) return launch_runjoin3_t<true, false, false>(ctx, A, FA, smem, name);
            return launch_runjoin3_t<false, true, false>(ctx, A, FA, smem, name);
        }
    }
    // gx_k_runjoin2: two CTAs of 512 threads per SM with 16-byte group slots (64 KB + 40 KB of run lists).  MEASURED SLOWER
    // than one CTA of 1024 threads with 24-byte slots (3.29 vs 2.76 ms at SF100, profiles/r02_runjoin_variants.txt), like the
    // other attempts to trade CTA size for occupancy on this kernel; kept behind GX_RUNJOIN_V2=1 for the record.
    {
        const char *v2 = getenv("GX_RUNJOIN_V2");
        if (use_run && v2 && v2[0] == '1' && A.s_slots <= 4096) {
            if (A.cslots) return sum ? launch_runjoin2_t<true, true>(ctx, A, FA, name) : launch_runjoin2_t<false, true>(ctx, A, FA, name);
            return sum ? launch_runjoin2_t<true, false>(ctx, A, FA, name) : launch_runjoin2_t<false, false>(ctx, A, FA, name);
        }
    }
    // the run-folding join kernel keeps a per-warp run list next to the group table
    const size_t run_bytes = 32 * sizeof(gx_runlist);
    // rows through the copy engine (gx_k_runjoin_tma): packed group slots, so at most 4096 of them; 16-byte aligned columns
    if (use_run && gx_runjoin_tma_enabled() && A.s_slots <= 4096 && (A.row0 & 1) == 0 &&
        ((uintptr_t) FA.okey & 15) == 0 && ((uintptr_t) FA.vcol & 15) == 0) {
        const size_t tma_smem = (size_t) A.s_slots * 16 + 32 * sizeof(gx_runlist) + 32 * sizeof(gx_rowstage) + 32 * 8;
        if (tma_smem + 1024 <= ctx->smem_optin) {
            if (A.cslots) return sum ? launch_runjoin_tma_t<true, true>(ctx, A, FA, tma_smem, name) : launch_runjoin_tma_t<false, true>(ctx, A, FA, tma_smem, name);
            return sum ? launch_runjoin_tma_t<true, false>(ctx, A, FA, tma_smem, name) : launch_runjoin_tma_t<false, false>(ctx, A, FA, tma_smem, name);
        }
    }
    // compact table + order-preserving slots: the streamed-table variant (gx_k_runjoin_seg)
    if (use_run && A.cslots && A.sf.mode != 0 && gx_runjoin_seg_enabled()) {
        int nbuf = 2;
        const unsigned int seg_slots = runjoin_seg_slots(ctx, smem, A, &nbuf);
        if (seg_slots >= 512) {
            if (cnt && sum) return launch_runjoin_seg_t<true, true>(ctx, A, FA, smem, seg_slots, nbuf, name);
            if (cnt) return launch_runjoin_seg_t<true, false>(ctx, A, FA, smem, seg_slots, nbuf, name);
            return launch_runjoin_seg_t<false, true>(ctx, A, FA, smem, seg_slots, nbuf, name);
        }
    }
    if (use_run) {
        if (A.cslots) {
            if (cnt && sum) return launch_runjoin_t<true, true, true>(ctx, A, FA, smem + run_bytes, name);
            if (cnt) return launch_runjoin_t<true, false, true>(ctx, A, FA, smem + run_bytes, name);
            return launch_runjoin_t<false, true, true>(ctx, A, FA, smem + run_bytes, name);
        }
        if (cnt && sum) return launch_runjoin_t<true, true, false>(ctx, A, FA, smem + run_bytes, name);
        if (cnt) return launch_runjoin_t<true, false, false>(ctx, A, FA, smem + run_bytes, name);
        return launch_runjoin_t<false, true, false>(ctx, A, FA, smem + run_bytes, name);
    }
    if (join) {
        if (cnt && sum) return launch_fast_t<true, true, true>(ctx, A, FA, smem, name);
        if (cnt) return launch_fast_t<true, true, false>(ctx, A, FA, smem, name);
        return launch_fast_t<true, false, true>(ctx, A, FA, smem, name);
    }
    if (cnt && sum) return launch_fast_t<false, true, true>(ctx, A, FA, smem, name);
    if (cnt) return launch_fast_t<false, true, false>(ctx, A, FA, smem, name);
    return launch_fast_t<false, false, true>(ctx, A, FA, smem, name);
}

static int read_counters(gx_ctx *ctx, long long *c /* 4 */, long long *cursor = nullptr)
{
    GX_CUDA(ctx, cudaMemcpyAsync(ctx->h_scratch + 8, ctx->d_scratch + 8, 5 * sizeof(long long), cudaMemcpyDeviceToHost, ctx->stream));
    GX_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    for (int i = 0; i < 4; i++) c[i] = ctx->h_scratch[8 + i];
    if (cursor) *cursor = ctx->h_scratch[12];                     // d_scratch[12]: the dense-output cursor
    return GX_OK;
}

// global table -> result (dense)
static int table_to_result(gx_ctx *ctx, compiled_plan *cp, const gx_agg_plan *plan, unsigned long long *g_tab, long long g_cap,
                           long long ngroups, gx_result **out)
{
    const int RW = 3 + cp->A.P.nwords;
    gx_result *r; gx_result_alloc(ctx, plan, cp->group_types, ngroups, &r);
    r->nkw = cp->A.P.nkw; r->nwords = cp->A.P.nwords; r->rec_words = RW; r->need_w0 = cp->need_w0;
    for (int a = 0; a < plan->n_aggs; a++) { r->agg_word[a] = cp->agg_word[a]; r->agg_cnt_word[a] = cp->agg_cnt_word[a]; }
    cudaError_t e = gx_tmp_alloc(ctx, (void **) &r->d_recs, (size_t) r->cap * RW * 8);
    if (e != cudaSuccess) { gx_result_free(r); GX_SET_ERR(ctx, "result: %s", cudaGetErrorString(e)); return GX_ERR_NOMEM; }
    GX_CUDA(ctx, cudaMemsetAsync(ctx->d_scratch + 12, 0, sizeof(long long), ctx->stream));
    if (ngroups > 0) {
        gx_launch_scope ls(ctx, "agg_compact");
        gx_k_compact_groups<<<ctx->sm_count * 4, 256, 0, ctx->stream>>>(g_tab, g_cap, cp->A.P.nwords, (unsigned long long *) r->d_recs, ctx->d_scratch + 12);
    }
    GX_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    r->ngroups = ngroups;
    *out = r;
    return GX_OK;
}

// keep the compiled layout around for fetch/combine
struct result_layout { int gword[GX_MAX_GROUP_COLS], gshift[GX_MAX_GROUP_COLS], gbytes[GX_MAX_GROUP_COLS]; int wkind[GX_MAX_WORDS]; long long winit[GX_MAX_WORDS]; };
static std::map<gx_result *, result_layout> *g_layouts;
static void remember_layout(gx_result *r, const compiled_plan *cp)
{
    if (!g_layouts) g_layouts = new std::map<gx_result *, result_layout>();
    result_layout L; memset(&L, 0, sizeof(L));
    for (int c = 0; c < GX_MAX_GROUP_COLS; c++) { L.gword[c] = cp->gword[c]; L.gshift[c] = cp->gshift[c]; L.gbytes[c] = cp->gbytes[c]; }
    for (int i = 0; i < GX_MAX_WORDS; i++) { L.wkind[i] = cp->A.wkind[i]; L.winit[i] = cp->A.winit[i]; }
    (*g_layouts)[r] = L;
}

static int run_radix(gx_ctx *ctx, compiled_plan *cp, const gx_agg_plan *plan, long long nrows_in, gx_result **out);
int gx_result_layout_words(gx_result *r, int *wkind, long long *winit);

extern "C" int gx_hash_agg(gx_ctx *ctx, const gx_table *outer, const gx_hash *h, const gx_agg_plan *plan, gx_result **out)
{
    if (!ctx || !outer || !plan || !out) return GX_ERR_ARG;
    compiled_plan cp;
    int rc = compile_plan(ctx, outer, h, plan, &cp); if (rc) return rc;
    gx_agg_dev &A = cp.A;
    const int nwords = A.P.nwords, RW = 3 + nwords;
    long long est = plan->est_groups > 0 ? plan->est_groups : 1024;
    if (plan->n_group_cols == 0) est = 1;

    // ---- shared-memory plan (strategy 1) -----------------------------------
    // key bytes <= 7 and one key word: the tag word carries the key itself
    int keybytes = 0;
    for (int c = 0; c < plan->n_group_cols; c++) keybytes += cp.gbytes[c];
    const int tagkey = (A.P.nkw == 1 && keybytes <= 7) ? 1 : 0;
    const size_t budget = ctx->smem_optin - 1024;
    auto dense_bytes = [&](long long S) { return (size_t) S * 8 * (1 + (tagkey ? 0 : A.P.nkw) + nwords); };
    long long smax = 16; while (dense_bytes(smax * 2) <= budget) smax *= 2;
    int strategy = plan->strategy;
    if (strategy == 0) strategy = (est * 3 / 2 <= smax) ? 1 : 2;
    GX_CHECK_ARG(ctx, strategy >= 1 && strategy <= 3, "agg plan: unknown strategy %d", strategy);
    A.need_w0 = cp.need_w0;

    // ---- does the plan have the shape the specialised kernel was written for?
    gx_fast_args FA; memset(&FA, 0, sizeof(FA));
    { const char *pf = getenv("GX_RUNJOIN_PF"); FA.pf = pf ? atoi(pf) : 0; }
    bool fast_ok = plan->n_preds == 0 && plan->n_group_cols == 1 && tagkey && outer->nrows > 0;
    if (fast_ok) {
        const gx_dgroupcol &gc = A.P.gcols[0];
        if (A.P.has_join) {
            fast_ok = gc.side == 1 && gc.payload_idx == 0 && gc.bytes == 4 && h->unique && A.P.key_type == GX_INT8 && A.P.okey.nulls == nullptr;
            FA.okey = (const long long *) A.P.okey.data;
        } else {
            fast_ok = gc.side == 0 && gc.bytes == 4 && gc.col.nulls == nullptr;
            FA.gcol = (const int *) gc.col.data;
        }
        int nvalue = 0;
        for (int a = 0; a < plan->n_aggs && fast_ok; a++) {
            const gx_dagg &ga = A.P.aggs[a];
            if (plan->aggs[a].fn == GX_AGG_COUNT_STAR) continue;
            if ((plan->aggs[a].fn == GX_AGG_SUM_F8 || plan->aggs[a].fn == GX_AGG_AVG_F8) && ga.expr.nterms == 1 && ga.expr.t[0].kind == GXT_COL &&
                ga.expr.t[0].col.type == GX_FLOAT8 && ga.expr.t[0].col.nulls == nullptr && nvalue == 0) {
                FA.vcol = (const double *) ga.expr.t[0].col.data; FA.sum_word = ga.word; nvalue++;
            } else fast_ok = false;
        }
    }

    // only gx_k_runjoin reads the compact table form; everything else needs the 16-byte slots
    auto need_wide = [&]() -> int {
        if (!h || A.slots) return GX_OK;
        int wrc = gx_hash_wide(ctx, const_cast<gx_hash *>(h));
        A.slots = h->slots;
        return wrc;
    };
    const size_t run_bytes = 32 * sizeof(gx_runlist);
    const char *norun = getenv("GX_NO_RUNJOIN");
    const bool runjoin_env = !(norun && norun[0] == '1');

    // the tile-at-a-time lane-private kernel: no join, count(*) and float8 sums over NOT-NULL float8 columns
    bool lptile_ok = !A.P.has_join;
    for (int a = 0; a < A.P.nagg && lptile_ok; a++) {
        const gx_dagg &ga = A.P.aggs[a];
        if (ga.kind == GXU_NONE) continue;
        lptile_ok = ga.kind == GXU_ADD_F64 && !ga.is_int && ga.cnt_word == 0 && ga.expr.nterms >= 1;
        for (int t = 0; t < ga.expr.nterms && lptile_ok; t++)
            lptile_ok = ga.expr.t[t].kind == GXT_CONST || (ga.expr.t[t].col.type == GX_FLOAT8 && ga.expr.t[t].col.nulls == nullptr);
    }
    { const char *e = getenv("GX_NO_LPTILE"); if (e && e[0] == '1') lptile_ok = false; }
    // register-accumulator kernels for <= FG_G groups (Q1, config 1): same plan shape as the tiled kernel,
    // key in one word without NULLs
    gx_fewgroups_args FG; memset(&FG, 0, sizeof(FG));
    bool fewgroups_ok = lptile_ok && A.P.nkw == 1 && plan->n_group_cols >= 1 && outer->nrows > 0;
    for (int c = 0; c < plan->n_group_cols && fewgroups_ok; c++) fewgroups_ok = A.P.gcols[c].side == 0 && A.P.gcols[c].col.nulls == nullptr;
    for (int a = 0; a < A.P.nagg && fewgroups_ok; a++) {
        if (A.P.aggs[a].kind == GXU_NONE) continue;
        if (FG.nv >= FG_NV) { fewgroups_ok = false; break; }
        const gx_dexpr &e = A.P.aggs[a].expr;
        for (int t = 0; t < e.nterms && fewgroups_ok; t++) {
            int slot = -1;
            if (e.t[t].kind != GXT_CONST) {
                const double *cp = (const double *) e.t[t].col.data;
                for (int c = 0; c < FG.nc; c++) if (FG.col[c] == cp) slot = c;
                if (slot < 0) { if (FG.nc < FG_NC) { slot = FG.nc; FG.col[FG.nc++] = cp; } else fewgroups_ok = false; }
            }
            FG.tslot[FG.nv][t] = (signed char) slot;
        }
        FG.vagg[FG.nv] = a; FG.vword[FG.nv] = A.P.aggs[a].word; FG.nv++;
    }
    { const char *e = getenv("GX_NO_FEWGROUPS"); if (e && e[0] == '1') fewgroups_ok = false; }
    bool countchar_ok = fewgroups_ok && FG.nv == 0 && plan->n_preds == 0 && plan->n_group_cols == 1 && A.P.gcols[0].type == GX_CHAR;

    // ---- GROUP BY contains the join key of a unique build side and the outer side is in key order:
    // a run of equal keys is a group (gx_k_runagg).  Tried first; a raised "keys descend" flag sends the
    // plan down the general path below.
    {
        gx_runagg_args RA; memset(&RA, 0, sizeof(RA));
        { const char *pf = getenv("GX_RUNAGG_PF"); RA.pf = pf ? atoi(pf) : 1; }     // Q3 chain at SF100: 5.68 ms without, 5.52 with the rows, 5.59 with rows + table lines
        const char *e = getenv("GX_NO_RUNAGG");
        bool ok = !(e && e[0] == '1') && plan->strategy == 0 && A.P.has_join && h->unique && A.P.key_type == GX_INT8 && A.P.okey.nulls == nullptr &&
                  outer->nrows > 0 && plan->n_group_cols >= 1;
        bool has_key = false;
        for (int c = 0; c < plan->n_group_cols && ok; c++) {
            const gx_dgroupcol &gc = A.P.gcols[c];
            if (gc.side == 0) { ok = plan->group_cols[c].col == plan->outer_key_col; RA.gk_from_key[c] = 1; has_key = true; }
            else RA.gk_pbit[c] = gc.payload_idx;
            RA.gk_word[c] = gc.word; RA.gk_shift[c] = gc.shift; RA.gk_bytes[c] = gc.bytes;
        }
        RA.ngk = plan->n_group_cols;
        ok = ok && has_key;
        for (int a = 0; a < A.P.nagg && ok; a++) {
            const gx_dagg &ga = A.P.aggs[a];
            if (ga.kind == GXU_NONE) continue;
            ok = ga.kind == GXU_ADD_F64 && !ga.is_int && ga.cnt_word == 0 && RA.nv < RA_NV && ga.expr.nterms >= 1;
            for (int t = 0; t < ga.expr.nterms && ok; t++)
                ok = ga.expr.t[t].kind == GXT_CONST || (ga.expr.t[t].col.type == GX_FLOAT8 && ga.expr.t[t].col.nulls == nullptr);
            for (int t = 0; t < ga.expr.nterms && ok; t++) {
                int slot = -1;
                if (ga.expr.t[t].kind != GXT_CONST) {
                    const double *cp = (const double *) ga.expr.t[t].col.data;
                    for (int c = 0; c < RA.nc; c++) if (RA.col[c] == cp) slot = c;
                    if (slot < 0) { if (RA.nc < FG_NC) { slot = RA.nc; RA.col[RA.nc++] = cp; } else ok = false; }
                }
                RA.tslot[RA.nv][t] = (signed char) slot;
            }
            if (ok) { RA.vagg[RA.nv] = a; RA.vword[RA.nv] = ga.word; RA.nv++; }
        }
        if (ok) {
            rc = need_wide(); if (rc) return rc;
            static bool attr = false;
            const bool small = RA.nv <= 2 && RA.nc <= 2;           // two CTAs of 384 threads per SM (85 registers each)
            const char *dn = getenv("GX_RUNAGG_DENSE");
            // 2 x 384 threads: 5.03 ms for the Q3 chain's lineitem side at SF100; 2 x 512 (28 bytes of spills): 4.49 ms
            const int dense = (small && RA.nv <= 1) ? (dn ? atoi(dn) != 0 : 1) : 0;      // 2 x 640 (48 registers): 4.80 ms, profiles/r02_occupancy_variants.txt
            const int threads = (small && !dense) ? 384 : 512, nwarps = threads / 32;
            const size_t smem = (size_t) nwarps * ((size_t) RA_LIST * (1 + RA.nv) + RA_LIST / 2) * 8;
            if (!attr) {
                GX_CUDA(ctx, cudaFuncSetAttribute(gx_k_runagg<1, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) ctx->smem_optin));
                GX_CUDA(ctx, cudaFuncSetAttribute(gx_k_runagg<2, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) ctx->smem_optin));
                GX_CUDA(ctx, cudaFuncSetAttribute(gx_k_runagg<1, 2, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) ctx->smem_optin));
                GX_CUDA(ctx, cudaFuncSetAttribute(gx_k_runagg<RA_NV, FG_NC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) ctx->smem_optin));
                attr = true;
            }
            const long long nrows = outer->nrows, total_warps = (long long) ctx->sm_count * (small ? 2 : 1) * nwarps;
            long long rpw = (nrows + total_warps - 1) / total_warps; rpw = (rpw + 31) / 32 * 32; if (rpw < 128) rpw = 128;
            const long long nchunks = (nrows + rpw - 1) / rpw;
            const unsigned grid = (unsigned) ((nchunks + nwarps - 1) / nwarps);
            RA.rows_per_warp = rpw;
            {
                // what a tile reads, for the row prefetch: the key, the argument columns, the qual columns (first four)
                auto list = [&](const void *ptr, int size) {
                    if (RA.pf_n < 4 && ptr) { RA.pf_ptr[RA.pf_n] = (const char *) ptr; RA.pf_size[RA.pf_n] = size; RA.pf_lines[RA.pf_n] = size; RA.pf_n++; }
                };
                list(A.P.okey.data, 8);
                for (int c = 0; c < RA.nc; c++) list(RA.col[c], 8);
                for (int q = 0; q < A.P.npreds; q++) list(A.P.preds[q].col.data, gx_type_size(A.P.preds[q].col.type));
            }
            const long long out_cap = (h->nentries < nrows ? h->nentries : nrows) + 64;
            const long long g_cap = gx_pow2_ceil(8 * nchunks + 1024);
            unsigned long long *g_tab, *d_out;
            GX_CUDA(ctx, gx_tmp_alloc(ctx, (void **) &g_tab, (size_t) g_cap * RW * 8));
            cudaError_t ae = gx_tmp_alloc(ctx, (void **) &d_out, (size_t) out_cap * RW * 8);
            if (ae != cudaSuccess) { gx_tmp_free(ctx, g_tab); GX_SET_ERR(ctx, "hash_agg: %s", cudaGetErrorString(ae)); return GX_ERR_NOMEM; }
            GX_CUDA(ctx, cudaMemsetAsync(g_tab, 0, (size_t) g_cap * RW * 8, ctx->stream));
            GX_CUDA(ctx, cudaMemsetAsync(A.counters, 0, 5 * sizeof(long long), ctx->stream));
            A.g_tab = g_tab; A.g_mask = (unsigned long long) g_cap - 1;
            RA.out = d_out; RA.out_cap = out_cap; RA.cursor = ctx->d_scratch + 12;
            {
                gx_launch_scope ls(ctx, "runagg");
                if (dense) gx_k_runagg<1, 2, 1><<<grid, threads, smem, ctx->stream>>>(A, RA);
                else if (small && RA.nv <= 1) gx_k_runagg<1, 2><<<grid, threads, smem, ctx->stream>>>(A, RA);
                else if (small) gx_k_runagg<2, 2><<<grid, threads, smem, ctx->stream>>>(A, RA);
                else gx_k_runagg<RA_NV, FG_NC><<<grid, threads, smem, ctx->stream>>>(A, RA);
            }
            GX_CUDA(ctx, cudaGetLastError());
            long long c[4], direct = 0;
            rc = read_counters(ctx, c, &direct);
            // an out-of-order outer side (flag 8) may also overrun the output: the general path answers either way
            if (rc == GX_OK && !(c[1] & 8) && (c[1] & 6)) { GX_SET_ERR(ctx, "hash_agg: run-aggregate output overflowed (flags %lld)", c[1]); rc = GX_ERR_STATE; }
            if (rc != GX_OK) { gx_tmp_free(ctx, g_tab); gx_tmp_free(ctx, d_out); return rc; }
            if (!(c[1] & 8)) {
                if (c[0] > 0) {
                    gx_launch_scope ls(ctx, "runagg_merge");
                    gx_k_compact_groups<<<(unsigned) ((g_cap + 255) / 256 < (long long) ctx->sm_count * 4 ? (g_cap + 255) / 256 : (long long) ctx->sm_count * 4), 256, 0, ctx->stream>>>(
                        g_tab, g_cap, nwords, d_out, ctx->d_scratch + 12);
                    GX_CUDA(ctx, cudaGetLastError());
                }
                gx_tmp_free(ctx, g_tab);
                gx_result *r; gx_result_alloc(ctx, plan, cp.group_types, direct + c[0], &r);
                r->nkw = A.P.nkw; r->nwords = nwords; r->rec_words = RW; r->need_w0 = 1;
                for (int a = 0; a < plan->n_aggs; a++) { r->agg_word[a] = cp.agg_word[a]; r->agg_cnt_word[a] = cp.agg_cnt_word[a]; }
                r->d_recs = (long long *) d_out; r->ngroups = direct + c[0]; r->cap = out_cap;
                remember_layout(r, &cp);
                *out = r;
                return GX_OK;
            }
            gx_tmp_free(ctx, g_tab); gx_tmp_free(ctx, d_out);      // keys descend somewhere: general path
            A.g_tab = nullptr;
        }
    }

    for (int attempt = 0; attempt < 8; attempt++) {
        if (strategy == 2) { rc = need_wide(); if (rc) return rc; rc = run_radix(ctx, &cp, plan, outer->nrows, out); if (rc == GX_OK) remember_layout(*out, &cp); return rc; }
        long long S = 16; while (S * 2 < est * 3 && S < smax) S *= 2;     // load factor <= 0.67
        // lane-private mode for a handful of groups: [warp][word][group][lane]
        int gmax = 0, lp_warps = 0; size_t lp_bytes = 0;
        if (strategy == 1 && est <= 16) {
            // 8, 16 or 32 groups per CTA.  Sized to the estimate, not twice it: the accumulators are
            // words x groups x 8 B PER LANE, and a wrong estimate only costs the retry below — while
            // falling back to the CTA-shared table with a handful of groups serialises every atomic
            // (Q1 shape, 11 words: 212 ms instead of single-digit ms).
            gmax = 8; while (gmax < est) gmax *= 2;
            S = 4 * gmax;
            size_t dir = (size_t) S * 8 * (1 + (tagkey ? 0 : A.P.nkw)) + ((S + 2) / 2 + 1) * 8;
            size_t per_warp = (size_t) nwords * gmax * 32 * 8;
            lp_warps = (int) ((budget - dir) / per_warp); if (lp_warps > 32) lp_warps = 32;
            if (lp_warps < 4) { gmax = 0; S = 16; while (S < est * 2 && S < smax) S *= 2; }   // too many words: use the dense table
            else lp_bytes = dir + per_warp * lp_warps;
        }
        long long g_cap = gx_pow2_ceil((strategy == 1 ? S : est) * 4 + 1024);
        unsigned long long *g_tab;
        GX_CUDA(ctx, gx_tmp_alloc(ctx, (void **) &g_tab, (size_t) g_cap * RW * 8));
        GX_CUDA(ctx, cudaMemsetAsync(g_tab, 0, (size_t) g_cap * RW * 8, ctx->stream));
        GX_CUDA(ctx, cudaMemsetAsync(A.counters, 0, 4 * sizeof(long long), ctx->stream));
        A.g_tab = g_tab; A.g_mask = (unsigned long long) g_cap - 1;
        A.s_slots = strategy == 1 ? (int) S : 0; A.s_log2 = ilog2(S); A.s_tagkey = tagkey; A.s_gmax = gmax;
        const char *kname = h ? "probe_agg" : "agg";
        const bool use_fast = strategy == 1 && !gmax && fast_ok;
        const bool use_run = use_fast && A.P.has_join && runjoin_env && dense_bytes(S) + run_bytes <= ctx->smem_optin - 1024;
        if (!use_run) { rc = need_wide(); if (rc) { gx_tmp_free(ctx, g_tab); return rc; } }
        const bool use_few = strategy == 1 && gmax && fewgroups_ok && est <= 2 * FG_G;
        { const char *dbg = getenv("GX_DEBUG_AGG");
          if (dbg && dbg[0] == '1')
              fprintf(stderr, "gpuexec: hash_agg attempt %d strategy %d S %lld gmax %d fast_ok %d use_fast %d use_run %d cslots %d slot mode %d seg %d tma %d rows %lld\n",
                      attempt, strategy, S, gmax, (int) fast_ok, (int) use_fast, (int) use_run, A.cslots != nullptr, A.sf.mode,
                      (int) gx_runjoin_seg_enabled(), (int) gx_runjoin_tma_enabled(), (long long) outer->nrows); }
        if (use_fast) rc = launch_fast(ctx, A, FA, A.P.has_join != 0, cp.need_w0 != 0, FA.vcol != nullptr, dense_bytes(S), kname, use_run);
        else if (use_few && countchar_ok) {
            gx_launch_scope ls(ctx, kname);
            gx_k_count_char<<<ctx->sm_count * 2, 512, 0, ctx->stream>>>(A, (const signed char *) A.P.gcols[0].col.data);
            rc = cudaGetLastError() == cudaSuccess ? GX_OK : GX_ERR_CUDA;
        } else if (use_few) {
            const char *fv = getenv("GX_FG_VARIANT");
            const bool v768 = !(fv && fv[0] == '0');                 // <4, 768> unless GX_FG_VARIANT=0 asks for <8, 512> (profiles/r02_fewgroups_variants.txt)
            const int fg_threads = v768 ? 768 : 512, fg_k = v768 ? 4 : 8, fg_warps = fg_threads / 32;
            const size_t fg_smem = (size_t) fg_warps * (1 + FG.nv) * (FG_G + 1) * 32 * 8;
            bool bytekey = plan->n_group_cols <= 2;
            for (int c = 0; c < plan->n_group_cols; c++) bytekey = bytekey && A.P.gcols[c].type == GX_CHAR && A.P.gcols[c].word == 0;
            static bool fg_attr = false;
            if (!fg_attr) {
                const int lim = (int) ctx->smem_optin - 1024;        // static shared memory counts too
                GX_CUDA(ctx, cudaFuncSetAttribute(gx_k_fewgroups<true, 8, 512>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
                GX_CUDA(ctx, cudaFuncSetAttribute(gx_k_fewgroups<false, 8, 512>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
                GX_CUDA(ctx, cudaFuncSetAttribute(gx_k_fewgroups<true, 4, 768>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
                GX_CUDA(ctx, cudaFuncSetAttribute(gx_k_fewgroups<false, 4, 768>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim));
                fg_attr = true;
            }
            long long nb = (outer->nrows + (long long) fg_warps * 32 * fg_k - 1) / ((long long) fg_warps * 32 * fg_k);
            const unsigned fg_grid = (unsigned) (nb < ctx->sm_count ? nb : ctx->sm_count);
            gx_launch_scope ls(ctx, kname);
            if (v768) { if (bytekey) gx_k_fewgroups<true, 4, 768><<<fg_grid, 768, fg_smem, ctx->stream>>>(A, FG); else gx_k_fewgroups<false, 4, 768><<<fg_grid, 768, fg_smem, ctx->stream>>>(A, FG); }
            else { if (bytekey) gx_k_fewgroups<true, 8, 512><<<fg_grid, 512, fg_smem, ctx->stream>>>(A, FG); else gx_k_fewgroups<false, 8, 512><<<fg_grid, 512, fg_smem, ctx->stream>>>(A, FG); }
            rc = cudaGetLastError() == cudaSuccess ? GX_OK : GX_ERR_CUDA;
        }
        else if (strategy == 1 && gmax && lptile_ok) rc = launch_lptile(ctx, A, lp_bytes, kname, lp_warps * 32);
        else if (strategy == 1 && gmax) rc = launch_agg<SINK_SMEM_LP>(ctx, A, lp_bytes, kname, lp_warps * 32);
        else if (strategy == 1) rc = launch_agg<SINK_SMEM>(ctx, A, dense_bytes(S), kname);
        else rc = launch_agg<SINK_GLOBAL>(ctx, A, 0, kname);
        long long c[4];
        if (rc == GX_OK) rc = read_counters(ctx, c);
        if (rc != GX_OK) { gx_tmp_free(ctx, g_tab); return rc; }
        if (c[1] == 0) {
            rc = table_to_result(ctx, &cp, plan, g_tab, g_cap, c[0], out);
            gx_tmp_free(ctx, g_tab);
            if (rc == GX_OK) remember_layout(*out, &cp);
            return rc;
        }
        gx_tmp_free(ctx, g_tab);
        if (c[1] & 16) {                                          // gx_k_runjoin_seg gave up on a barrier: same plan again with gx_k_runjoin
            fprintf(stderr, "gpuexec: a bounded mbarrier wait of gx_k_runjoin_seg / gx_k_runjoin_tma gave up; continuing with gx_k_runjoin\n");
            g_runjoin_seg_broken = true; continue;
        }
        if (use_few) { fewgroups_ok = false; continue; }          // more than FG_G groups: same estimate, general kernels
        // the planner's estimate was too low: grow, then fall over to radix
        est = est < 8 ? 9 : est < 16 ? 17 : est * 8;
        if (strategy == 1 && est * 3 / 2 > smax) strategy = (plan->strategy == 1) ? 3 : 2;
    }
    GX_SET_ERR(ctx, "hash_agg: group table kept overflowing");
    return GX_ERR_STATE;
}

// single-block exclusive scan (same as gx_table.cu's, kept local to this TU)
__global__ void gx_k_scan_i64(long long *v, long long n, long long *total)
{
    __shared__ long long sm[33];
    long long carry = 0;
    for (long long base = 0; base < n; base += blockDim.x) {
        long long i = base + threadIdx.x;
        long long x = i < n ? v[i] : 0, tot;
        long long ex = gx_block_exscan(x, &tot, sm);
        if (i < n) v[i] = carry + ex;
        carry += tot;
    }
    if (threadIdx.x == 0 && total) *total = carry;
}

// Records (already materialised, nrec of them at d_recs) -> dense groups.
// Used by strategy 2 and by gx_result_combine.
int gx_aggregate_records(gx_ctx *ctx, gx_agg_dev A, unsigned long long *d_recs, long long nrec,
                         unsigned long long **d_out, long long *ngroups_out)
{
    const int nwords = A.P.nwords, RW = 3 + nwords;
    *d_out = nullptr; *ngroups_out = 0;
    if (nrec == 0) return GX_OK;
    // pass-2 table: as large as one CTA's shared memory allows
    size_t budget = ctx->smem_optin - 1024;
    int S2 = 16; while (smem_bytes_for(S2 * 2, 2, nwords) <= budget) S2 *= 2;
    int bits = 0; while (bits < RADIX_MAX_BITS && (nrec >> bits) > S2 / 4) bits++;
    const int P = 1 << bits;
    unsigned nblk = (unsigned) (ctx->sm_count * 2);
    if ((long long) nblk * 512 > nrec) nblk = (unsigned) ((nrec + 511) / 512);
    long long *d_hist; unsigned long long *d_part, *d_groups; int *d_over;
    GX_CUDA(ctx, gx_tmp_alloc(ctx, (void **) &d_hist, (size_t) P * nblk * sizeof(long long)));
    GX_CUDA(ctx, gx_tmp_alloc(ctx, (void **) &d_part, (size_t) nrec * RW * 8));
    GX_CUDA(ctx, gx_tmp_alloc(ctx, (void **) &d_groups, (size_t) nrec * RW * 8));
    GX_CUDA(ctx, gx_tmp_alloc(ctx, (void **) &d_over, (size_t) P * sizeof(int)));
    GX_CUDA(ctx, cudaMemsetAsync(d_over, 0, (size_t) P * sizeof(int), ctx->stream));
    GX_CUDA(ctx, cudaMemsetAsync(ctx->d_scratch + 12, 0, sizeof(long long), ctx->stream));
    static bool attr = false;
    if (!attr) { GX_CUDA(ctx, cudaFuncSetAttribute(gx_k_radix_agg, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) ctx->smem_optin - 512)); attr = true; }
    {
        gx_launch_scope ls(ctx, "radix_partition", 3);
        gx_k_radix_hist<<<nblk, 512, P * sizeof(unsigned), ctx->stream>>>(d_recs, nrec, RW, bits, d_hist);
        gx_k_scan_i64<<<1, 1024, 0, ctx->stream>>>(d_hist, (long long) P * nblk, nullptr);
        gx_k_radix_scatter<<<nblk, 512, P * sizeof(unsigned), ctx->stream>>>(d_recs, nrec, RW, bits, d_hist, d_part);
    }
    A.s_slots = S2; A.s_log2 = ilog2(S2); A.rec_cap = nrec;
    {
        gx_launch_scope ls(ctx, "radix_agg");
        unsigned grid = (unsigned) (P < ctx->sm_count ? P : ctx->sm_count);
        gx_k_radix_agg<<<grid, 512, smem_bytes_for(S2, 2, nwords), ctx->stream>>>(A, d_part, d_hist, P, (int) nblk, d_groups, ctx->d_scratch + 12, d_over);
    }
    GX_CUDA(ctx, cudaGetLastError());
    // partitions that overflowed shared memory go through a global table
    int *h_over = (int *) malloc((size_t) P * sizeof(int));
    long long *h_hist0 = (long long *) malloc((size_t) P * sizeof(long long));
    GX_CUDA(ctx, cudaMemcpyAsync(h_over, d_over, (size_t) P * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    GX_CUDA(ctx, cudaMemcpy2DAsync(h_hist0, sizeof(long long), d_hist, (size_t) nblk * sizeof(long long), sizeof(long long), P, cudaMemcpyDeviceToHost, ctx->stream));
    GX_CUDA(ctx, cudaMemcpyAsync(ctx->h_scratch + 12, ctx->d_scratch + 12, sizeof(long long), cudaMemcpyDeviceToHost, ctx->stream));
    GX_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    long long ngroups = ctx->h_scratch[12];
    long long over_recs = 0; int nover = 0;
    for (int p = 0; p < P; p++) if (h_over[p]) { nover++; over_recs += ((p + 1 < P) ? h_hist0[p + 1] : nrec) - h_hist0[p]; }
    free(h_over); free(h_hist0);
    int rc = GX_OK;
    if (nover) {
        long long g_cap = gx_pow2_ceil(over_recs * 2 + 1024);
        unsigned long long *g_tab;
        GX_CUDA(ctx, gx_tmp_alloc(ctx, (void **) &g_tab, (size_t) g_cap * RW * 8));
        GX_CUDA(ctx, cudaMemsetAsync(g_tab, 0, (size_t) g_cap * RW * 8, ctx->stream));
        GX_CUDA(ctx, cudaMemsetAsync(A.counters, 0, 4 * sizeof(long long), ctx->stream));
        A.g_tab = g_tab; A.g_mask = (unsigned long long) g_cap - 1;
        {
            gx_launch_scope ls(ctx, "radix_overflow", 2);
            gx_k_merge_records<<<ctx->sm_count * 2, 512, 0, ctx->stream>>>(A, d_part, d_hist, (int) nblk, d_over, P, nrec);
            GX_CUDA(ctx, cudaMemcpyAsync(ctx->d_scratch + 12, ctx->h_scratch + 12, sizeof(long long), cudaMemcpyHostToDevice, ctx->stream));
            gx_k_compact_groups<<<ctx->sm_count * 4, 256, 0, ctx->stream>>>(g_tab, g_cap, nwords, d_groups, ctx->d_scratch + 12);
        }
        long long c[4];
        rc = read_counters(ctx, c);
        if (rc == GX_OK && c[1]) { GX_SET_ERR(ctx, "radix overflow table overflowed"); rc = GX_ERR_STATE; }
        if (rc == GX_OK) ngroups += c[0];
        gx_tmp_free(ctx, g_tab);
    }
    gx_tmp_free(ctx, d_hist); gx_tmp_free(ctx, d_part); gx_tmp_free(ctx, d_over);
    if (rc != GX_OK) { gx_tmp_free(ctx, d_groups); return rc; }
    *d_out = d_groups; *ngroups_out = ngroups;
    return GX_OK;
}

// Finalize step of gx_result_combine: merge received partial records by key.
int gx_combine_records(gx_ctx *ctx, gx_result *r, unsigned long long *d_recs, long long nrec,
                       unsigned long long **d_out, long long *ngroups_out)
{
    gx_agg_dev A; memset(&A, 0, sizeof(A));
    A.P.nwords = r->nwords; A.P.nkw = 2;
    int rc = gx_result_layout_words(r, A.wkind, A.winit); if (rc) { GX_SET_ERR(ctx, "combine: unknown result"); return rc; }
    A.counters = ctx->d_scratch + 8;
    return gx_aggregate_records(ctx, A, d_recs, nrec, d_out, ngroups_out);
}

// small-result Finalize: pack this rank's partial records into a fixed-capacity segment
int gx_pack_partial(gx_ctx *ctx, gx_result *r, long long cap, unsigned long long *d_seg)
{
    gx_launch_scope ls(ctx, "combine_pack");
    long long words = r->ngroups * r->rec_words;
    unsigned grid = (unsigned) ((words + 255) / 256); if (grid < 1) grid = 1; if (grid > (unsigned) ctx->sm_count * 4) grid = (unsigned) ctx->sm_count * 4;
    gx_k_pack_partial<<<grid, 256, 0, ctx->stream>>>((const unsigned long long *) r->d_recs, r->ngroups, cap, r->rec_words, d_seg);
    GX_CUDA(ctx, cudaGetLastError());
    return GX_OK;
}
// ... and merge the all-gathered segments; *anybig = some rank did not fit (caller takes the general path)
int gx_combine_gathered(gx_ctx *ctx, gx_result *r, const unsigned long long *d_gather, int nseg, long long cap,
                        unsigned long long **d_out, long long *ngroups_out, int *anybig)
{
    gx_agg_dev A; memset(&A, 0, sizeof(A));
    A.P.nwords = r->nwords; A.P.nkw = 2;
    int rc = gx_result_layout_words(r, A.wkind, A.winit); if (rc) { GX_SET_ERR(ctx, "combine: unknown result"); return rc; }
    A.counters = ctx->d_scratch + 8;
    const int RW = 3 + r->nwords;
    long long g_cap = gx_pow2_ceil(2 * (long long) nseg * cap + 1024);
    unsigned long long *g_tab, *d_groups;
    GX_CUDA(ctx, gx_tmp_alloc(ctx, (void **) &g_tab, (size_t) g_cap * RW * 8));
    GX_CUDA(ctx, cudaMemsetAsync(g_tab, 0, (size_t) g_cap * RW * 8, ctx->stream));
    GX_CUDA(ctx, cudaMemsetAsync(A.counters, 0, 5 * sizeof(long long), ctx->stream));     // [4] = compact cursor
    A.g_tab = g_tab; A.g_mask = (unsigned long long) g_cap - 1;
    // every group of the gathered set may be owned by this rank in the worst case
    GX_CUDA(ctx, gx_tmp_alloc(ctx, (void **) &d_groups, (size_t) nseg * cap * RW * 8 + 64));
    {
        gx_launch_scope ls(ctx, "combine_merge", 2);
        long long total = (long long) nseg * cap;
        unsigned grid = (unsigned) ((total + 255) / 256); if (grid > (unsigned) ctx->sm_count * 8) grid = (unsigned) ctx->sm_count * 8;
        gx_k_merge_gathered<<<grid, 256, 0, ctx->stream>>>(A, d_gather, nseg, cap, ctx->rank, ctx->nranks);
        gx_k_compact_groups<<<ctx->sm_count * 4, 256, 0, ctx->stream>>>(g_tab, g_cap, r->nwords, d_groups, ctx->d_scratch + 12);
    }
    GX_CUDA(ctx, cudaGetLastError());
    long long c[4];
    rc = read_counters(ctx, c);
    gx_tmp_free(ctx, g_tab);
    if (rc == GX_OK && c[1]) { GX_SET_ERR(ctx, "combine: merge table overflowed"); rc = GX_ERR_STATE; }
    if (rc != GX_OK) { gx_tmp_free(ctx, d_groups); return rc; }
    *anybig = c[3] != 0;
    if (*anybig) { gx_tmp_free(ctx, d_groups); *d_out = nullptr; *ngroups_out = 0; return GX_OK; }
    *d_out = d_groups; *ngroups_out = c[0];
    return GX_OK;
}

static int run_radix(gx_ctx *ctx, compiled_plan *cp, const gx_agg_plan *plan, long long nrows_in, gx_result **out)
{
    gx_agg_dev &A = cp->A;
    const int nwords = A.P.nwords, RW = 3 + nwords;
    // stage A: one record per (joined, qualifying) row.  Capacity: rows in for a
    // unique build; otherwise count first with the record sink disabled.
    long long cap = nrows_in;
    unsigned long long *d_recs = nullptr;
    for (int pass = 0; pass < 2; pass++) {
        GX_CUDA(ctx, gx_tmp_alloc(ctx, (void **) &d_recs, (size_t) (cap > 0 ? cap : 1) * RW * 8));
        GX_CUDA(ctx, cudaMemsetAsync(A.counters, 0, 4 * sizeof(long long), ctx->stream));
        A.recs = d_recs; A.rec_cap = cap; A.s_slots = 0;
        int rc = launch_agg<SINK_RECORD>(ctx, A, 0, A.P.has_join ? "probe_records" : "scan_records");
        long long c[4];
        if (rc == GX_OK) rc = read_counters(ctx, c);
        if (rc != GX_OK) { gx_tmp_free(ctx, d_recs); return rc; }
        if (!(c[1] & 4)) { cap = c[2]; break; }
        gx_tmp_free(ctx, d_recs); d_recs = nullptr;
        cap = c[2];                                   // exact need (N:M join fan-out)
        if (pass == 1) { GX_SET_ERR(ctx, "radix: record buffer overflow"); return GX_ERR_STATE; }
    }
    unsigned long long *d_groups; long long ngroups;
    int rc = gx_aggregate_records(ctx, A, d_recs, cap, &d_groups, &ngroups);
    gx_tmp_free(ctx, d_recs);
    if (rc) return rc;
    gx_result *r; gx_result_alloc(ctx, plan, cp->group_types, ngroups, &r);
    r->nkw = A.P.nkw; r->nwords = nwords; r->rec_words = RW; r->need_w0 = cp->need_w0;
    for (int a = 0; a < plan->n_aggs; a++) { r->agg_word[a] = cp->agg_word[a]; r->agg_cnt_word[a] = cp->agg_cnt_word[a]; }
    r->d_recs = (long long *) d_groups; r->ngroups = ngroups; r->cap = ngroups;
    if (!d_groups) { GX_CUDA(ctx, gx_tmp_alloc(ctx, (void **) &r->d_recs, 64)); }
    *out = r;
    return GX_OK;
}

// ------------------------------------------------------------ results
extern "C" int64_t gx_result_ngroups(const gx_result *r)
{
    if (!r) return -1;
    // a plain aggregate over zero rows still returns one row (agg_retrieve_direct)
    if (r->plan.n_group_cols == 0 && r->ngroups == 0) return 1;
    return r->ngroups;
}

extern "C" void gx_result_free(gx_result *r)
{
    if (!r) return;
    if (g_layouts) g_layouts->erase(r);
    gx_tmp_free(r->ctx, r->d_recs);
    gx_tmp_free(r->ctx, r->d_nullmask);
    free(r);
}

// accessors for gx_comm.cu (combine across datanodes)
int gx_result_layout_words(gx_result *r, int *wkind, long long *winit)
{
    if (!g_layouts || !g_layouts->count(r)) return GX_ERR_STATE;
    const result_layout &L = (*g_layouts)[r];
    for (int i = 0; i < GX_MAX_WORDS; i++) { wkind[i] = L.wkind[i]; winit[i] = L.winit[i]; }
    return GX_OK;
}

// finalize_aggregates (nodeAgg.c:1363).  float8_avg = Sx / N, NULL when N == 0 (float.c:2991-3008).
// Small results are finalized on the host from the raw records; large ones (Q3: millions of
// groups) on the device, straight into the caller's column layout, so the host only copies.
struct gx_final_args {
    const unsigned long long *recs; long long ngroups; int RW, ng, na, need_w0;
    int gword[GX_MAX_GROUP_COLS], gshift[GX_MAX_GROUP_COLS], gtype[GX_MAX_GROUP_COLS];
    int fn[GX_MAX_AGGS], word[GX_MAX_AGGS], cw[GX_MAX_AGGS];
    long long *key_out; double *agg_out; unsigned char *null_out; int *overflow;
};
__global__ void gx_k_finalize(const gx_final_args F)
{
    const long long stride = (long long) gridDim.x * blockDim.x;
    for (long long gI = (long long) blockIdx.x * blockDim.x + threadIdx.x; gI < F.ngroups; gI += stride) {
        const unsigned long long *rec = F.recs + (size_t) gI * F.RW, *w = rec + 3;
        const unsigned int nullmask = (unsigned int) rec[0];
        for (int c = 0; c < F.ng; c++) {
            const bool isnull = (nullmask >> c) & 1;
            const unsigned long long v = (F.gword[c] == 0 ? rec[1] : rec[2]) >> F.gshift[c];
            long long sv;
            switch (F.gtype[c]) {
                case GX_INT4: case GX_DATE: sv = (long long) (int) (unsigned int) v; break;
                case GX_CHAR: sv = (long long) (signed char) (unsigned char) v; break;
                default: sv = (long long) v; break;
            }
            F.key_out[gI * F.ng + c] = isnull ? 0 : sv;
            if (F.null_out) F.null_out[gI * (F.ng + F.na) + c] = isnull;
        }
        for (int a = 0; a < F.na; a++) {
            const int fn = F.fn[a], word = F.word[a], cw = F.cw[a];
            const long long cnt = cw ? (long long) w[cw] : (F.need_w0 ? (long long) w[0] : 1);
            bool isnull = false, is_int = false; double res = 0.0; long long ires = 0;
            switch (fn) {
                case GX_AGG_COUNT_STAR: ires = (long long) w[0]; is_int = true; break;
                case GX_AGG_COUNT: ires = (long long) w[word]; is_int = true; break;
                case GX_AGG_SUM_I4: case GX_AGG_SUM_I8: ires = (long long) w[word]; is_int = true; isnull = cnt == 0; break;
                case GX_AGG_AVG_F8: { const double sx = __longlong_as_double((long long) w[word]); if (cnt == 0) isnull = true; else res = sx / (double) cnt; break; }
                default: res = __longlong_as_double((long long) w[word]); isnull = cnt == 0; break;
            }
            if (isnull) { res = 0.0; ires = 0; }
            F.agg_out[gI * F.na + a] = is_int ? __longlong_as_double(ires) : res;
            if (F.null_out) F.null_out[gI * (F.ng + F.na) + F.ng + a] = isnull;
            if (!is_int && !isnull && (fn == GX_AGG_SUM_F8 || fn == GX_AGG_AVG_F8) && isinf(res)) *F.overflow = 1;
        }
    }
}

static int fetch_on_device(gx_result *r, const result_layout &L, int64_t *key_out, double *agg_out, uint8_t *null_out)
{
    gx_ctx *ctx = r->ctx;
    const int ng = r->plan.n_group_cols, na = r->plan.n_aggs;
    const size_t n = (size_t) r->ngroups;
    gx_final_args F; memset(&F, 0, sizeof(F));
    F.recs = (const unsigned long long *) r->d_recs; F.ngroups = r->ngroups; F.RW = r->rec_words; F.ng = ng; F.na = na; F.need_w0 = r->need_w0;
    for (int c = 0; c < ng; c++) { F.gword[c] = L.gword[c]; F.gshift[c] = L.gshift[c]; F.gtype[c] = r->group_types[c]; }
    for (int a = 0; a < na; a++) { F.fn[a] = r->plan.aggs[a].fn; F.word[a] = r->agg_word[a]; F.cw[a] = r->agg_cnt_word[a]; }
    char *d = nullptr;
    const size_t kb = n * (ng > 0 ? ng : 1) * 8, ab = n * (na > 0 ? na : 1) * 8, nb = (n * (ng + na) + 15) & ~(size_t) 15;
    GX_CUDA(ctx, gx_tmp_alloc(ctx, (void **) &d, kb + ab + nb + 16));
    F.key_out = (long long *) d; F.agg_out = (double *) (d + kb); F.null_out = null_out ? (unsigned char *) (d + kb + ab) : nullptr;
    F.overflow = (int *) (d + kb + ab + nb);
    GX_CUDA(ctx, cudaMemsetAsync(F.overflow, 0, sizeof(int), ctx->stream));
    {
        gx_launch_scope ls(ctx, "finalize");
        gx_k_finalize<<<ctx->sm_count * 4, 256, 0, ctx->stream>>>(F);
    }
    cudaError_t e = cudaGetLastError();
    if (e == cudaSuccess && ng) e = cudaMemcpyAsync(key_out, F.key_out, n * ng * 8, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess && na) e = cudaMemcpyAsync(agg_out, F.agg_out, n * na * 8, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess && null_out) e = cudaMemcpyAsync(null_out, F.null_out, n * (ng + na), cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(ctx->h_scratch + 16, F.overflow, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    gx_tmp_free(ctx, d);
    if (e != cudaSuccess) { GX_SET_ERR(ctx, "result_fetch: %s", cudaGetErrorString(e)); return GX_ERR_CUDA; }
    if (*(int *) (ctx->h_scratch + 16)) { GX_SET_ERR(ctx, "value out of range: overflow"); return GX_ERR_OVERFLOW; }
    return GX_OK;
}

extern "C" int gx_result_fetch(gx_result *r, int64_t max_groups, int64_t *key_out, double *agg_out, uint8_t *null_out)
{
    if (!r) return GX_ERR_ARG;
    gx_ctx *ctx = r->ctx;
    const int ng = r->plan.n_group_cols, na = r->plan.n_aggs, RW = r->rec_words;
    if (ng == 0 && r->ngroups == 0) {
        GX_CHECK_ARG(ctx, max_groups >= 1, "result_fetch: buffer too small");
        for (int a = 0; a < na; a++) {
            int fn = r->plan.aggs[a].fn;
            bool is_count = fn == GX_AGG_COUNT_STAR || fn == GX_AGG_COUNT;
            long long zero = 0; memcpy(&agg_out[a], &zero, 8);
            if (null_out) null_out[a] = is_count ? 0 : 1;
        }
        return GX_OK;
    }
    GX_CHECK_ARG(ctx, max_groups >= r->ngroups, "result_fetch: buffer holds %lld groups, result has %lld", (long long) max_groups, (long long) r->ngroups);
    if (r->ngroups == 0) return GX_OK;
    GX_CHECK_ARG(ctx, g_layouts && g_layouts->count(r), "result_fetch: unknown result");
    const result_layout &L = (*g_layouts)[r];
    if (r->ngroups > 8192) return fetch_on_device(r, L, key_out, agg_out, null_out);
    unsigned long long *h = (unsigned long long *) malloc((size_t) r->ngroups * RW * 8);
    cudaError_t e = cudaMemcpyAsync(h, r->d_recs, (size_t) r->ngroups * RW * 8, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) { free(h); GX_SET_ERR(ctx, "result_fetch: %s", cudaGetErrorString(e)); return GX_ERR_CUDA; }
    for (int64_t g = 0; g < r->ngroups; g++) {
        const unsigned long long *rec = h + (size_t) g * RW, *w = rec + 3;
        unsigned int nullmask = (unsigned int) rec[0];
        for (int c = 0; c < ng; c++) {
            bool isnull = (nullmask >> c) & 1;
            unsigned long long v = (L.gword[c] == 0 ? rec[1] : rec[2]) >> L.gshift[c];
            long long sv;
            switch (r->group_types[c]) {
                case GX_INT4: case GX_DATE: sv = (long long) (int32_t) (uint32_t) v; break;
                case GX_CHAR: sv = (long long) (int8_t) (uint8_t) v; break;
                default: sv = (long long) v; break;
            }
            key_out[g * ng + c] = isnull ? 0 : sv;
            if (null_out) null_out[g * (ng + na) + c] = isnull;
        }
        for (int a = 0; a < na; a++) {
            int fn = r->plan.aggs[a].fn, word = r->agg_word[a], cw = r->agg_cnt_word[a];
            // cw == 0: the argument cannot be NULL, so a group that exists has input;
            // w0 (rows per group) is only maintained when count(*)/avg need it
            long long cnt = cw ? (long long) w[cw] : (r->need_w0 ? (long long) w[0] : 1);
            uint8_t isnull = 0; double res = 0.0; long long ires = 0; bool is_int = false;
            switch (fn) {
                case GX_AGG_COUNT_STAR: ires = (long long) w[0]; is_int = true; break;
                case GX_AGG_COUNT: ires = (long long) w[word]; is_int = true; break;
                case GX_AGG_SUM_I4: case GX_AGG_SUM_I8: ires = (long long) w[word]; is_int = true; isnull = cnt == 0; break;
                case GX_AGG_AVG_F8: { double sx; memcpy(&sx, &w[word], 8); if (cnt == 0) isnull = 1; else res = sx / (double) cnt; break; }
                default: { memcpy(&res, &w[word], 8); isnull = cnt == 0; break; }
            }
            if (isnull) { res = 0.0; ires = 0; }
            if (is_int) memcpy(&agg_out[g * na + a], &ires, 8); else agg_out[g * na + a] = res;
            if (null_out) null_out[g * (ng + na) + ng + a] = isnull;
            // float8pl's CHECKFLOATVAL: a finite-input sum that reached infinity is an ERROR in the reference
            if (!is_int && !isnull && (fn == GX_AGG_SUM_F8 || fn == GX_AGG_AVG_F8) && __builtin_isinf(res)) {
                free(h); GX_SET_ERR(ctx, "value out of range: overflow"); return GX_ERR_OVERFLOW;
            }
        }
    }
    free(h);
    return GX_OK;
}

// Partial (transition) states for a two-phase plan: the reference's Finalize Agg above a
// RemoteSubplan combines them with int8pl / float8pl / float8_combine / float8smaller ...
// (AGGSPLIT_INITIAL_SERIAL on this side, planner.c:8743-8749; combine functions
// pg_aggregate.h:178-252).  Per aggregate: cnt_out = N (rows for count(*), non-NULL inputs
// otherwise), val_out = Sx / min / max as float8 or the int8 sum bit-cast; null_out = 1 when the
// transition value is still NULL (no non-NULL input seen; count states are never NULL).
extern "C" int gx_result_fetch_states(gx_result *r, int64_t max_groups, int64_t *key_out, double *val_out, int64_t *cnt_out, uint8_t *null_out)
{
    if (!r || !key_out || !val_out || !cnt_out) return GX_ERR_ARG;
    gx_ctx *ctx = r->ctx;
    const int ng = r->plan.n_group_cols, na = r->plan.n_aggs, RW = r->rec_words;
    if (ng == 0 && r->ngroups == 0) {                           // plain aggregate over zero rows: initial states
        GX_CHECK_ARG(ctx, max_groups >= 1, "result_fetch_states: buffer too small");
        for (int a = 0; a < na; a++) {
            const int fn = r->plan.aggs[a].fn;
            val_out[a] = 0.0; cnt_out[a] = 0;
            if (null_out) null_out[a] = (fn == GX_AGG_COUNT_STAR || fn == GX_AGG_COUNT || fn == GX_AGG_AVG_F8) ? 0 : 1;
        }
        return GX_OK;
    }
    GX_CHECK_ARG(ctx, max_groups >= r->ngroups, "result_fetch_states: buffer holds %lld groups, result has %lld", (long long) max_groups, (long long) r->ngroups);
    if (r->ngroups == 0) return GX_OK;
    GX_CHECK_ARG(ctx, g_layouts && g_layouts->count(r), "result_fetch_states: unknown result");
    const result_layout &L = (*g_layouts)[r];
    unsigned long long *h = (unsigned long long *) malloc((size_t) r->ngroups * RW * 8);
    cudaError_t e = cudaMemcpyAsync(h, r->d_recs, (size_t) r->ngroups * RW * 8, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) { free(h); GX_SET_ERR(ctx, "result_fetch_states: %s", cudaGetErrorString(e)); return GX_ERR_CUDA; }
    for (int64_t gI = 0; gI < r->ngroups; gI++) {
        const unsigned long long *rec = h + (size_t) gI * RW, *w = rec + 3;
        const unsigned int nullmask = (unsigned int) rec[0];
        for (int c = 0; c < ng; c++) {
            const bool isnull = (nullmask >> c) & 1;
            const unsigned long long v = (L.gword[c] == 0 ? rec[1] : rec[2]) >> L.gshift[c];
            long long sv;
            switch (r->group_types[c]) {
                case GX_INT4: case GX_DATE: sv = (long long) (int32_t) (uint32_t) v; break;
                case GX_CHAR: sv = (long long) (int8_t) (uint8_t) v; break;
                default: sv = (long long) v; break;
            }
            key_out[gI * ng + c] = isnull ? 0 : sv;
            if (null_out) null_out[gI * (ng + na) + c] = isnull;
        }
        for (int a = 0; a < na; a++) {
            const int fn = r->plan.aggs[a].fn, word = r->agg_word[a], cw = r->agg_cnt_word[a];
            const long long rows = (long long) w[0];
            const long long cnt = cw ? (long long) w[cw] : (r->need_w0 ? rows : 1);
            double v = 0.0; long long n = cnt; uint8_t isnull = 0;
            switch (fn) {
                case GX_AGG_COUNT_STAR: n = rows; break;
                case GX_AGG_COUNT: n = (long long) w[word]; break;
                case GX_AGG_SUM_I4: case GX_AGG_SUM_I8: memcpy(&v, &w[word], 8); isnull = cnt == 0; break;
                case GX_AGG_AVG_F8: memcpy(&v, &w[word], 8); break;              // {N, Sx}: never NULL (initial state '{0,0,0}')
                default: memcpy(&v, &w[word], 8); isnull = cnt == 0; break;      // sum / min / max: strict, NULL until the first input
            }
            if ((fn == GX_AGG_SUM_F8 || fn == GX_AGG_AVG_F8) && !isnull && __builtin_isinf(v)) {
                free(h); GX_SET_ERR(ctx, "value out of range: overflow"); return GX_ERR_OVERFLOW;
            }
            val_out[gI * na + a] = isnull ? 0.0 : v; cnt_out[gI * na + a] = n;
            if (null_out) null_out[gI * (ng + na) + ng + a] = isnull;
        }
    }
    free(h);
    return GX_OK;
}
