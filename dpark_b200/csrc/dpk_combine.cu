// dpk_combine.cu -- reduce side of the shuffle: DiskHashMerger._merge
// (dpark/shuffle.py:600-608): combined[k] = mergeCombiners(combined[k], v) over
// every row fetched for the reduce partitions this GPU owns.
//
// Three implementations behind dpk_combine (dpk_set_option "reduce_impl"), all bit-identical:
//
//   2 (default)  second-level split + shared-memory merge.  Every first-level bucket of the received
//      rows is split once more by further hash bits (seg_multisplit, dpk_partition.cu) into fine
//      buckets of <= ~2 k rows; k_smem_aggregate (dpk_aggregate.cuh) merges one fine bucket per CTA in
//      a 4096-slot shared-memory table and writes its distinct rows straight into the partition's
//      output range (chained look-back for the offset).  Probes cost ~30 cycles instead of an L2 round
//      trip; DRAM traffic = the algorithmic (K+V) * (rows + distinct) plus the split's 2 * (K+V) * rows.
//   1  one thread-block cluster of 8 CTAs per first-level bucket (k_bucket_reduce): the bucket's
//      table region in HBM is initialised, filled and compacted while it is L2-resident.
//   0  three grid-wide passes over per-bucket table regions in HBM:
//        k_tbl_init    : slots <- {EMPTY, identity(op)}
//        k_tbl_insert  : per row: bucket from the key's hash, claim a slot with atomicCAS on the key
//                        word (linear probing inside the region), then one native atomic on the accumulator
//        k_tbl_compact : per occupied slot: recompute its partition, reserve an output index inside
//                        that partition's range (CTA-aggregated), write.
// Common to all: 16-byte slots {key bits, accumulator}; k_tbl_plan computes per-bucket region offsets
// (1.5 x rows), per-partition output offsets and the first row of every (source, bucket) segment.
// Accumulators: int64 for integer values (exact while |sum| < 2^63, as the reference's big ints),
// float64 for float values (the reference adds Python floats).
#include "dpk_common.cuh"
#include <cooperative_groups.h>
#include <type_traits>

namespace cg = cooperative_groups;

namespace dpk {

constexpr int CB_THREADS = 256;
constexpr int64_t kEmpty = INT64_MIN;  // slot-free marker; a real key with these bits uses the side slot

struct __align__(16) Slot {
    int64_t key;
    int64_t acc;  // int64 or the bits of a double
};

template <typename KeyT> __device__ __forceinline__ int64_t key_bits(KeyT k);
template <> __device__ __forceinline__ int64_t key_bits<int64_t>(int64_t k) { return k; }
template <> __device__ __forceinline__ int64_t key_bits<int32_t>(int32_t k) { return (int64_t)k; }
template <> __device__ __forceinline__ int64_t key_bits<uint64_t>(uint64_t k) { return (int64_t)k; }
template <> __device__ __forceinline__ int64_t key_bits<double>(double k) {
    if (k == 0.0) k = 0.0;  // -0.0 == 0.0 is one dict key in Python
    return __double_as_longlong(k);
}
template <> __device__ __forceinline__ int64_t key_bits<float>(float k) {
    if (k == 0.0f) k = 0.0f;
    return (int64_t)__float_as_int(k);
}
template <typename KeyT> __device__ __forceinline__ KeyT key_from_bits(int64_t b);
template <> __device__ __forceinline__ int64_t key_from_bits<int64_t>(int64_t b) { return b; }
template <> __device__ __forceinline__ int32_t key_from_bits<int32_t>(int64_t b) { return (int32_t)b; }
template <> __device__ __forceinline__ uint64_t key_from_bits<uint64_t>(int64_t b) { return (uint64_t)b; }
template <> __device__ __forceinline__ double key_from_bits<double>(int64_t b) { return __longlong_as_double(b); }
template <> __device__ __forceinline__ float key_from_bits<float>(int64_t b) { return __int_as_float((int)b); }

// Row-id keys (DPK_K_ROWID): the key column holds the index of a representative
// row of a variable-length key (dpk_dict_encode); its portable_hash is looked up
// in `aux` (the per-row hash column) instead of being computed from the id.
struct RowId { int64_t v; };
template <> __device__ __forceinline__ int64_t key_bits<RowId>(RowId k) { return k.v; }
template <> __device__ __forceinline__ RowId key_from_bits<RowId>(int64_t b) { RowId r; r.v = b; return r; }
template <typename KeyT> __device__ __forceinline__ int64_t hash_of(KeyT k, const int64_t *) { return KeyHash<KeyT>::of(k); }
template <> __device__ __forceinline__ int64_t hash_of<RowId>(RowId k, const int64_t *aux) { return __ldg(&aux[k.v]); }

// ---- accumulator ops (op is kernel-uniform, so the switch costs nothing) ------
template <typename AccT> struct Acc;

template <> struct Acc<int64_t> {
    static int64_t identity(int op) {
        switch (op) {
        case DPK_OP_MIN: return INT64_MAX;
        case DPK_OP_MAX: return INT64_MIN;
        case DPK_OP_PROD: return 1;
        case DPK_OP_AND: return -1;
        default: return 0;
        }
    }
    static bool supports(int op) { return op >= DPK_OP_SUM && op <= DPK_OP_XOR; }
    static __device__ __forceinline__ void apply(int op, int64_t *a, int64_t v) {
        switch (op) {
        case DPK_OP_SUM: atomicAdd((unsigned long long *)a, (unsigned long long)v); break;
        case DPK_OP_MIN: atomicMin((long long *)a, (long long)v); break;
        case DPK_OP_MAX: atomicMax((long long *)a, (long long)v); break;
        case DPK_OP_AND: atomicAnd((unsigned long long *)a, (unsigned long long)v); break;
        case DPK_OP_OR: atomicOr((unsigned long long *)a, (unsigned long long)v); break;
        case DPK_OP_XOR: atomicXor((unsigned long long *)a, (unsigned long long)v); break;
        default: {  // PROD (wrapping, like int64 multiply)
            unsigned long long old = *(volatile unsigned long long *)a, assumed;
            do {
                assumed = old;
                old = atomicCAS((unsigned long long *)a, assumed, assumed * (unsigned long long)v);
            } while (old != assumed);
        }
        }
    }
};

template <> struct Acc<double> {
    // SUM starts at -0.0, the IEEE additive identity (-0.0 + x == x for every x, +0.0 + -0.0 == +0.0): a key whose
    // only values are -0.0 keeps -0.0 in the kernels that add every value into a fresh accumulator
    static int64_t identity(int op) {
        double d = -0.0;
        switch (op) {
        case DPK_OP_MIN: d = INFINITY; break;
        case DPK_OP_MAX: d = -INFINITY; break;
        case DPK_OP_PROD: d = 1.0; break;
        default: d = -0.0;
        }
        int64_t b;
        memcpy(&b, &d, 8);
        return b;
    }
    static bool supports(int op) { return op >= DPK_OP_SUM && op <= DPK_OP_PROD; }
    static __device__ __forceinline__ void apply(int op, int64_t *a, double v) {
        if (op == DPK_OP_SUM) {
            atomicAdd((double *)a, v);
            return;
        }
        unsigned long long old = *(volatile unsigned long long *)a, assumed;
        do {
            assumed = old;
            double cur = __longlong_as_double((long long)assumed), nv;
            if (op == DPK_OP_MIN) nv = v < cur ? v : cur;
            else if (op == DPK_OP_MAX) nv = v > cur ? v : cur;
            else nv = cur * v;
            if (__double_as_longlong(nv) == (long long)assumed) break;
            old = atomicCAS((unsigned long long *)a, assumed, (unsigned long long)__double_as_longlong(nv));
        } while (old != assumed);
    }
};

// ---- kernels ---------------------------------------------------------------
// plan (single CTA).  seg_rows[nsrc][F]: rows of local fine bucket b that came
// from source s (the received buffer is source-major, bucket-major inside).
//   tbl_off[F+1]   slot offsets: region b holds 1.5*rows_b + 32 slots, rounded to 8
//   part_off[nparts+1] row offsets of the partitions (= start of their output ranges)
//   seg_start[nsrc][F] first row of segment (s, b) in the received buffer
__global__ void __launch_bounds__(CB_THREADS)
k_tbl_plan(const int64_t *__restrict__ seg_rows, int32_t nsrc, int32_t F, int32_t sub_bits, int32_t nparts,
           int64_t *__restrict__ tbl_off, int64_t *__restrict__ part_off, int64_t *__restrict__ seg_start) {
    __shared__ long long s_slots[CB_THREADS], s_rows[CB_THREADS], s_carry;
    const int E = (F + CB_THREADS - 1) / CB_THREADS;
    const int b0 = threadIdx.x * E, b1 = min(b0 + E, F);
    long long slots = 0, rows = 0;
    for (int b = b0; b < b1; b++) {
        long long r = 0;
        for (int s = 0; s < nsrc; s++) r += seg_rows[(int64_t)s * F + b];
        slots += ((r + (r >> 1) + 32 + 7) >> 3) << 3;
        rows += r;
    }
    s_slots[threadIdx.x] = slots;
    s_rows[threadIdx.x] = rows;
    __syncthreads();
    long long sbase = 0, rbase = 0;
    for (int t = 0; t < (int)threadIdx.x; t++) { sbase += s_slots[t]; rbase += s_rows[t]; }
    const int S = 1 << sub_bits;
    for (int b = b0; b < b1; b++) {
        long long r = 0;
        for (int s = 0; s < nsrc; s++) r += seg_rows[(int64_t)s * F + b];
        tbl_off[b] = sbase;
        if ((b & (S - 1)) == 0) part_off[b >> sub_bits] = rbase;
        sbase += ((r + (r >> 1) + 32 + 7) >> 3) << 3;
        rbase += r;
    }
    if (b0 < F && b1 == F) { tbl_off[F] = sbase; part_off[nparts] = rbase; }
    if (F == 0 && threadIdx.x == 0) { tbl_off[0] = 0; part_off[0] = 0; }
    // seg_start: running row offset, source by source
    if (threadIdx.x == 0) s_carry = 0;
    __syncthreads();
    for (int s = 0; s < nsrc; s++) {
        long long mine = 0;
        for (int b = b0; b < b1; b++) mine += seg_rows[(int64_t)s * F + b];
        s_rows[threadIdx.x] = mine;
        __syncthreads();
        long long base = s_carry;
        for (int t = 0; t < (int)threadIdx.x; t++) base += s_rows[t];
        for (int b = b0; b < b1; b++) {
            seg_start[(int64_t)s * F + b] = base;
            base += seg_rows[(int64_t)s * F + b];
        }
        __syncthreads();
        if (threadIdx.x == CB_THREADS - 1) s_carry = base;   // last thread saw every earlier bucket
        __syncthreads();
    }
}

__device__ __forceinline__ int4 slot_fill(int64_t ident) {
    return make_int4((int)(uint32_t)((uint64_t)kEmpty & 0xffffffffu), (int)(uint32_t)((uint64_t)kEmpty >> 32),
                     (int)(uint32_t)((uint64_t)ident & 0xffffffffu), (int)(uint32_t)((uint64_t)ident >> 32));
}

// claim-or-find the slot of key bits `kb` inside `region` (size slots), linear probing
__device__ __forceinline__ Slot *probe_slot(Slot *region, uint32_t size, int64_t kb) {
    uint32_t h = (uint32_t)(((mix64((uint64_t)kb) & 0xffffffffull) * (uint64_t)size) >> 32);
    for (;;) {
        int64_t cur = __ldcg(&region[h].key);
        if (cur == kb) break;
        if (cur == kEmpty) {
            unsigned long long prev = atomicCAS((unsigned long long *)&region[h].key, (unsigned long long)kEmpty,
                                                (unsigned long long)kb);
            if (prev == (unsigned long long)kEmpty || prev == (unsigned long long)kb) break;
        }
        h = h + 1 == size ? 0 : h + 1;
    }
    return &region[h];
}

// ===== implementation 0: three grid-wide passes over all regions ================
__global__ void __launch_bounds__(CB_THREADS)
k_tbl_init(Slot *__restrict__ table, const int64_t *__restrict__ tbl_total, int64_t ident) {
    const int64_t slots = *tbl_total;
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    const int4 fill = slot_fill(ident);
    for (; i < slots; i += stride) reinterpret_cast<int4 *>(table)[i] = fill;
}

template <typename KeyT, typename ValT, typename AccT>
__global__ void __launch_bounds__(CB_THREADS)
k_tbl_insert(const KeyT *__restrict__ keys, const int64_t *__restrict__ aux, const ValT *__restrict__ vals,
             int64_t n, int op, PartFn f, int32_t bucket_first, int32_t F,
             const int64_t *__restrict__ tbl_off, Slot *__restrict__ table, Slot *__restrict__ side,
             int32_t *__restrict__ side_used) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (; i < n; i += stride) {
        const KeyT key = keys[i];
        const int64_t kb = key_bits<KeyT>(key);
        const AccT v = (AccT)vals[i];
        Slot *s;
        if (kb == kEmpty) {
            s = side;
            *side_used = 1;
        } else {
            int b = f.bucket(hash_of<KeyT>(key, aux)) - bucket_first;
            b = min(max(b, 0), F - 1);
            const int64_t base = __ldg(&tbl_off[b]);
            s = probe_slot(table + base, (uint32_t)(__ldg(&tbl_off[b + 1]) - base), kb);
        }
        Acc<AccT>::apply(op, &s->acc, v);
    }
}

template <typename KeyT>
__global__ void __launch_bounds__(CB_THREADS)
k_tbl_compact(const Slot *__restrict__ table, const int64_t *__restrict__ tbl_total,
              const int64_t *__restrict__ aux, PartFn f, int32_t part_first, int32_t nparts,
              const int64_t *__restrict__ part_offsets, KeyT *__restrict__ out_keys,
              int64_t *__restrict__ out_vals, unsigned long long *__restrict__ out_counts) {
    extern __shared__ __align__(16) int32_t s_mem[];  // [nparts] counts, [nparts] 64-bit bases after
    int32_t *s_cnt = s_mem;
    long long *s_base = reinterpret_cast<long long *>(s_mem + ((nparts + 1) & ~1));
    const int lane = threadIdx.x & 31;
    constexpr int ITEMS = 4;
    const int64_t total = *tbl_total;
    const int64_t tile = (int64_t)CB_THREADS * ITEMS;
    for (int64_t t0 = (int64_t)blockIdx.x * tile; t0 < total; t0 += (int64_t)gridDim.x * tile) {
        for (int p = threadIdx.x; p < nparts; p += CB_THREADS) s_cnt[p] = 0;
        __syncthreads();
        int64_t kb[ITEMS], acc[ITEMS];
        int lp[ITEMS], rk[ITEMS];
#pragma unroll
        for (int j = 0; j < ITEMS; j++) {
            int64_t i = t0 + (int64_t)j * CB_THREADS + threadIdx.x;
            lp[j] = -1;
            if (i < total) {
                int4 raw = __ldcs(reinterpret_cast<const int4 *>(table) + i);
                kb[j] = (int64_t)(((uint64_t)(uint32_t)raw.y << 32) | (uint32_t)raw.x);
                acc[j] = (int64_t)(((uint64_t)(uint32_t)raw.w << 32) | (uint32_t)raw.z);
                if (kb[j] != kEmpty) lp[j] = f(hash_of<KeyT>(key_from_bits<KeyT>(kb[j]), aux)) - part_first;
            }
        }
#pragma unroll
        for (int j = 0; j < ITEMS; j++) {
            unsigned m = __match_any_sync(0xffffffffu, lp[j]);
            int base = 0;
            const bool ok = lp[j] >= 0 && lp[j] < nparts;
            if (ok && lane == __ffs(m) - 1) base = atomicAdd(&s_cnt[lp[j]], __popc(m));
            base = __shfl_sync(0xffffffffu, base, __ffs(m) - 1);
            rk[j] = base + __popc(m & ((1u << lane) - 1u));
        }
        __syncthreads();
        for (int p = threadIdx.x; p < nparts; p += CB_THREADS) {
            int c = s_cnt[p];
            s_base[p] = c ? (long long)atomicAdd(&out_counts[p], (unsigned long long)c) : 0;
        }
        __syncthreads();
#pragma unroll
        for (int j = 0; j < ITEMS; j++) {
            if (lp[j] >= 0 && lp[j] < nparts) {
                int64_t dst = part_offsets[lp[j]] + s_base[lp[j]] + rk[j];
                out_keys[dst] = key_from_bits<KeyT>(kb[j]);
                out_vals[dst] = acc[j];
            }
        }
        __syncthreads();
    }
}

// ===== implementation 1: one thread-block cluster per fine bucket ===============
// A cluster of 8 CTAs (8 SMs, hardware cluster barrier) takes a bucket and runs its
// whole life cycle back to back -- init the region, insert the bucket's rows, compact
// the region into the partition's output range -- so the region is written, probed
// and read while it sits in L2: HBM sees the rows once (read) and the distinct pairs
// once (write), plus the write-back of dirty table lines.  ~16 clusters run at once,
// each on a different bucket (16 x ~5 MB of live tables in the 126 MB L2).
constexpr int BR_THREADS = 1024;
constexpr int BR_CLUSTER = 8;

template <typename KeyT, typename ValT, typename AccT>
__global__ void __cluster_dims__(BR_CLUSTER, 1, 1) __launch_bounds__(BR_THREADS, 1)
k_bucket_reduce(const KeyT *__restrict__ keys, const int64_t *__restrict__ aux, const ValT *__restrict__ vals,
                int op, int64_t ident, int32_t sub_bits, int32_t F, int32_t nsrc,
                const int64_t *__restrict__ seg_start, const int64_t *__restrict__ seg_rows,
                const int64_t *__restrict__ tbl_off, Slot *__restrict__ table, Slot *__restrict__ side,
                int32_t *__restrict__ side_used, const int64_t *__restrict__ part_offsets,
                KeyT *__restrict__ out_keys, int64_t *__restrict__ out_vals,
                unsigned long long *__restrict__ out_counts, int *__restrict__ bucket_counter) {
    cg::cluster_group cluster = cg::this_cluster();
    const unsigned crank = cluster.block_rank();
    __shared__ int s_bucket;
    __shared__ int s_wsum[BR_THREADS / 32];
    __shared__ long long s_base;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t tid_c = (int64_t)crank * BR_THREADS + threadIdx.x;
    const int64_t nth_c = (int64_t)BR_CLUSTER * BR_THREADS;
    const int4 fill = slot_fill(ident);
    for (;;) {
        if (crank == 0 && threadIdx.x == 0) s_bucket = atomicAdd(bucket_counter, 1);
        cluster.sync();
        const int b = *cluster.map_shared_rank(&s_bucket, 0);
        cluster.sync();  // every CTA has read rank 0's shared memory before anyone may exit or overwrite
        if (b >= F) break;
        const int64_t base = tbl_off[b];
        const uint32_t size = (uint32_t)(tbl_off[b + 1] - base);
        Slot *region = table + base;
        // ---- 1. init (full 16 B stores: write-allocate in L2, nothing is fetched from HBM)
        for (int64_t i = tid_c; i < size; i += nth_c) reinterpret_cast<int4 *>(region)[i] = fill;
        cluster.sync();
        // ---- 2. insert the bucket's rows (one segment per source rank)
        for (int s = 0; s < nsrc; s++) {
            const int64_t r0 = seg_start[(int64_t)s * F + b];
            const int64_t rn = seg_rows[(int64_t)s * F + b];
            for (int64_t i = tid_c; i < rn; i += nth_c) {
                const int64_t kb = key_bits<KeyT>(keys[r0 + i]);
                const AccT v = (AccT)vals[r0 + i];
                Slot *sl;
                if (kb == kEmpty) {
                    sl = side;
                    *side_used = 1;
                } else {
                    sl = probe_slot(region, size, kb);
                }
                Acc<AccT>::apply(op, &sl->acc, v);
            }
        }
        cluster.sync();
        // ---- 3. compact the region into the partition's output range
        const int p = b >> sub_bits;
        const int64_t pbase = part_offsets[p];
        constexpr int ITEMS = 4;
        const int64_t tile = (int64_t)BR_THREADS * ITEMS;
        for (int64_t t0 = (int64_t)crank * tile; t0 < size; t0 += (int64_t)BR_CLUSTER * tile) {
            int64_t kb[ITEMS], acc[ITEMS];
            int c = 0;
#pragma unroll
            for (int j = 0; j < ITEMS; j++) {
                const int64_t i = t0 + (int64_t)threadIdx.x * ITEMS + j;
                kb[j] = kEmpty;
                if (i < size) {
                    int4 raw = __ldcg(reinterpret_cast<const int4 *>(region) + i);
                    kb[j] = (int64_t)(((uint64_t)(uint32_t)raw.y << 32) | (uint32_t)raw.x);
                    acc[j] = (int64_t)(((uint64_t)(uint32_t)raw.w << 32) | (uint32_t)raw.z);
                }
                c += kb[j] != kEmpty;
            }
            // block exclusive scan of c
            int inc = c;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                int t = __shfl_up_sync(0xffffffffu, inc, d);
                if (lane >= d) inc += t;
            }
            if (lane == 31) s_wsum[warp] = inc;
            __syncthreads();
            if (warp == 0) {
                int w = s_wsum[lane];
                int winc = w;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) {
                    int t = __shfl_up_sync(0xffffffffu, winc, d);
                    if (lane >= d) winc += t;
                }
                s_wsum[lane] = winc - w;  // exclusive
                if (lane == 31) s_base = winc ? (long long)atomicAdd(&out_counts[p], (unsigned long long)winc) : 0;
            }
            __syncthreads();
            int64_t dst = pbase + s_base + s_wsum[warp] + (inc - c);
#pragma unroll
            for (int j = 0; j < ITEMS; j++) {
                if (kb[j] != kEmpty) {
                    out_keys[dst] = key_from_bits<KeyT>(kb[j]);
                    out_vals[dst] = acc[j];
                    dst++;
                }
            }
            __syncthreads();
        }
    }
}

// ===== implementation 2: second-level split + shared-memory tables (dpk_aggregate.cuh) =====
#include "dpk_aggregate.cuh"
#include "dpk_aggregate2.cuh"
#include "dpk_aggregate3.cuh"

// the key whose bits equal the free-slot marker lives in the side slot: append it
template <typename KeyT>
__global__ void k_side_flush(const Slot *__restrict__ side, const int32_t *__restrict__ side_used,
                             const int64_t *__restrict__ aux, PartFn f, int32_t part_first, int32_t nparts,
                             const int64_t *__restrict__ part_offsets, KeyT *__restrict__ out_keys,
                             int64_t *__restrict__ out_vals, unsigned long long *__restrict__ out_counts) {
    if (threadIdx.x != 0 || blockIdx.x != 0 || *side_used == 0) return;
    const KeyT key = key_from_bits<KeyT>(kEmpty);
    const int p = f(hash_of<KeyT>(key, aux)) - part_first;
    if (p < 0 || p >= nparts) return;
    const int64_t dst = part_offsets[p] + (int64_t)atomicAdd(&out_counts[p], 1ull);
    out_keys[dst] = key;
    out_vals[dst] = side->acc;
}

// host-side upper bound of the slot count for n rows in F buckets
static inline int64_t max_slots_for(int64_t n, int32_t F) { return n + (n >> 1) + (int64_t)F * 40 + 64; }

static inline int grid_cap(int64_t items, int per_cta, int waves) {
    int64_t g = (items + per_cta - 1) / per_cta;
    int64_t cap = (int64_t)sm_count() * waves;
    if (g > cap) g = cap;
    if (g < 1) g = 1;
    return (int)g;
}

int g_reduce_impl = 2;  // dpk_set_option("reduce_impl", 0|1|2)

constexpr int AG_MAX_SB2 = 10;       // at most 1024 fine buckets per first-level bucket
int g_agg_wide = 1;
int g_agg_ctas = 4;                  // measured: 4 resident CTAs (64 registers, some spills) 1.58 ms vs 1.72 ms at 3
int g_agg_timing = 0;
int g_agg_split = 1;
int g_agg_cursor = 1;
int g_agg_pipe = 0;                  // dpk_set_option("agg_pipe"): 1 = k_smem_aggregate3 (rows prefetched into registers), 2 = same, 2 CTAs per SM
int g_agg_batched = 0;               // measured: the four-rows-in-flight insert executes 40 % more instructions (spills) -> 2.22 ms vs 1.72 ms
int g_agg_impl = 1;                  // dpk_set_option("agg_impl"): 1 = k_smem_aggregate2 (row-index tags), 0 = round-1 kernel
int g_agg_target_rows = 2048;        // rows per fine bucket the split aims for (measured on the C4 shape: an average of
                                     // 954 rows at a 1536 target costs more -- 7.4 ms merge + 5.3 ms 1024-way split -- than
                                     // 1907 rows with 29 % of the buckets in the multi-window path: 5.0 + 4.0 ms)

static inline int choose_sb2(int64_t n, int32_t F) {
    int sb2 = 0;
    while (sb2 < AG_MAX_SB2 && n / ((int64_t)F << sb2) > g_agg_target_rows) sb2++;
    return sb2;
}

struct Ctx {
    int key_kind, val_bytes;
    int64_t *fine_off;
    unsigned long long *fb_state;
    int *part_err;
    void *seg_ws;
    int64_t seg_ws_bytes;
    const void *keys, *vals;
    const int64_t *aux;
    int64_t n;
    int op;
    PartFn f;
    int32_t part_first, nparts, F, nsrc;
    const int64_t *seg_rows, *seg_start, *tbl_off, *part_off;
    Slot *table, *side;
    int64_t max_slots;
    int32_t *side_used;
    int *bucket_counter;
    void *out_keys;
    int64_t *out_vals;
    unsigned long long *out_counts;
    cudaStream_t st;
};

template <typename KeyT, typename ValT, typename AccT>
static int dispatch_op(const Ctx &c) {
    if (!Acc<AccT>::supports(c.op)) return fail(DPK_ERR_UNSUPPORTED, "op %d unsupported for this value kind", c.op);
    const int64_t ident = Acc<AccT>::identity(c.op);
    if (g_reduce_impl == 2) {
        // second-level split into the (idle) table region, then shared-memory merge per fine bucket
        const int sb2 = choose_sb2(c.n, c.F);
        const int32_t S2 = 1 << sb2;
        PartFn fine = c.f;
        fine.mode = 5; fine.P = S2; fine.shift = 32 - c.f.sub_bits - sb2; fine.sub_bits = 0; fine.row_hash = c.aux;
        KeyT *rekeys = (KeyT *)c.table;
        ValT *revals = (ValT *)((char *)c.table + (size_t)c.n * 8);
        int rc = seg_multisplit(c.keys, c.key_kind, c.vals, (int32_t)sizeof(ValT), c.n, fine, c.F, c.nsrc, c.seg_start,
                                c.seg_rows, rekeys, revals, c.fine_off, c.seg_ws, c.seg_ws_bytes, c.st);
        if (rc) return rc;
        const int32_t nfine = c.F * S2;
        int grid = sm_count() * 8;
        if (grid > nfine) grid = nfine;
        // dpk_set_option("agg_wide"): 1 = claim a slot and deposit the first value with one 128-bit CAS
        auto agg = g_agg_wide ? k_smem_aggregate<KeyT, ValT, AccT, true> : k_smem_aggregate<KeyT, ValT, AccT, false>;
        const int agg_smem = AG_CAP * 16 + AG_CAP * 2;  // keys | accumulators | claim list
        DPK_CUDA_TRY(cudaFuncSetAttribute(agg, cudaFuncAttributeMaxDynamicSharedMemorySize, agg_smem));
        DPK_CUDA_TRY(cudaMemsetAsync(c.fb_state, 0, (size_t)nfine * 8, c.st));
        if (g_agg_impl == 1) {
            // dpk_set_option("agg_ctas"): resident CTAs per SM the kernel is compiled for (3: 80 registers, 4: 64)
            // dpk_set_option("agg_cursor"): 1 = output ranges reserved with one atomicAdd per fine bucket, 0 = chained look-back
            // dpk_set_option("agg_batched"): 1 = four rows per thread in flight in the insert phase, 0 (default) = probe loop per row
            auto agg2 = k_smem_aggregate2<KeyT, ValT, AccT, 3, true, true>;
            if (g_agg_cursor && g_agg_batched) agg2 = g_agg_ctas == 4 ? k_smem_aggregate2<KeyT, ValT, AccT, 4, true, true> : k_smem_aggregate2<KeyT, ValT, AccT, 3, true, true>;
            else if (g_agg_cursor) agg2 = g_agg_ctas == 4 ? k_smem_aggregate2<KeyT, ValT, AccT, 4, true, false> : k_smem_aggregate2<KeyT, ValT, AccT, 3, true, false>;
            // (the batched variants are compiled for 3 CTAs per SM only when batched: see above)
            else agg2 = k_smem_aggregate2<KeyT, ValT, AccT, 3, false, false>;
            const int smem2 = AG2_TAGS * 4 + AG2_CAP * 16;
            DPK_CUDA_TRY(cudaFuncSetAttribute(agg2, cudaFuncAttributeMaxDynamicSharedMemorySize, smem2));
            DPK_CUDA_TRY(cudaMemsetAsync(c.part_err, 0, (size_t)(c.nparts + 2) * 4, c.st));
            long long *timing = nullptr;
            if (g_agg_timing) {
                static long long *d_timing = nullptr;
                if (!d_timing) DPK_CUDA_TRY(cudaMalloc(&d_timing, 64));
                DPK_CUDA_TRY(cudaMemsetAsync(d_timing, 0, 64, c.st));
                timing = d_timing;
            }
            if (g_agg_pipe && g_agg_cursor) {
                // register-pipelined fast path for the buckets that fit one window; the oversized ones go to a list
                // (two ints behind the per-partition error flags: list length, list-mode work counter) and are merged by
                // the staged kernel in a second launch
                auto agg3 = g_agg_pipe == 2 ? k_smem_aggregate3<KeyT, ValT, AccT, 2, false>
                          : (g_agg_batched ? k_smem_aggregate3<KeyT, ValT, AccT, 3, true> : k_smem_aggregate3<KeyT, ValT, AccT, 3, false>);
                const int smem3 = AG2_TAGS * 4 + AG2_CAP * 8;
                DPK_CUDA_TRY(cudaFuncSetAttribute(agg3, cudaFuncAttributeMaxDynamicSharedMemorySize, smem3));
                int *big_count = c.part_err + c.nparts, *list_counter = c.part_err + c.nparts + 1;
                int *big_list = reinterpret_cast<int *>(c.fb_state);          // nfine * 8 bytes: idle in cursor mode
                int g3 = sm_count() * (g_agg_pipe == 2 ? 2 : 3);
                if (g3 > nfine) g3 = nfine;
                DPK_LAUNCH("smem_aggregate", c.st, agg3<<<g3, AG2_THREADS, smem3, c.st>>>(
                    rekeys, revals, c.op, ident, c.fine_off, nfine, (1 << c.f.sub_bits) * S2, c.part_off,
                    (KeyT *)c.out_keys, c.out_vals, (long long *)c.out_counts, c.bucket_counter, big_list, big_count));
                auto aggb = k_smem_aggregate2<KeyT, ValT, AccT, 3, true, false>;
                DPK_CUDA_TRY(cudaFuncSetAttribute(aggb, cudaFuncAttributeMaxDynamicSharedMemorySize, smem2));
                DPK_LAUNCH("smem_aggregate_big", c.st, aggb<<<sm_count(), AG2_THREADS, smem2, c.st>>>(
                    rekeys, revals, c.op, c.fine_off, nfine, (1 << c.f.sub_bits) * S2, c.part_off,
                    (KeyT *)c.out_keys, c.out_vals, (long long *)c.out_counts, c.fb_state, list_counter, c.part_err,
                    big_list, big_count, nullptr, nullptr, nullptr));
            } else if (g_agg_cursor && !g_agg_batched && g_agg_split) {
                // dpk_set_option("agg_split") 1 (default): the hot launch holds the one-window path only (fewer live
                // registers); oversized buckets are listed and merged by the full kernel in a second, usually empty launch
                auto fast = g_agg_ctas == 4 ? k_smem_aggregate2<KeyT, ValT, AccT, 4, true, false, true>
                                            : k_smem_aggregate2<KeyT, ValT, AccT, 3, true, false, true>;
                DPK_CUDA_TRY(cudaFuncSetAttribute(fast, cudaFuncAttributeMaxDynamicSharedMemorySize, smem2));
                int *big_count = c.part_err + c.nparts, *list_counter = c.part_err + c.nparts + 1;
                int *big_list = reinterpret_cast<int *>(c.fb_state);          // nfine * 8 bytes: idle in cursor mode
                DPK_LAUNCH("smem_aggregate", c.st, fast<<<grid, AG2_THREADS, smem2, c.st>>>(
                    rekeys, revals, c.op, c.fine_off, nfine, (1 << c.f.sub_bits) * S2, c.part_off,
                    (KeyT *)c.out_keys, c.out_vals, (long long *)c.out_counts, c.fb_state, c.bucket_counter, c.part_err,
                    nullptr, nullptr, timing, big_list, big_count));
                auto aggb = k_smem_aggregate2<KeyT, ValT, AccT, 3, true, false>;
                DPK_CUDA_TRY(cudaFuncSetAttribute(aggb, cudaFuncAttributeMaxDynamicSharedMemorySize, smem2));
                DPK_LAUNCH("smem_aggregate_big", c.st, aggb<<<sm_count() * 2, AG2_THREADS, smem2, c.st>>>(
                    rekeys, revals, c.op, c.fine_off, nfine, (1 << c.f.sub_bits) * S2, c.part_off,
                    (KeyT *)c.out_keys, c.out_vals, (long long *)c.out_counts, c.fb_state, list_counter, c.part_err,
                    big_list, big_count, nullptr, nullptr, nullptr));
            } else {
            DPK_LAUNCH("smem_aggregate", c.st, agg2<<<grid, AG2_THREADS, smem2, c.st>>>(
                rekeys, revals, c.op, c.fine_off, nfine, (1 << c.f.sub_bits) * S2, c.part_off,
                (KeyT *)c.out_keys, c.out_vals, (long long *)c.out_counts, c.fb_state, c.bucket_counter, c.part_err,
                nullptr, nullptr, timing, nullptr, nullptr));
            if (timing) {   // debugging aid: synchronises and prints the per-phase averages of this launch
                long long h[8];
                DPK_CUDA_TRY(cudaMemcpyAsync(h, timing, sizeof(h), cudaMemcpyDeviceToHost, c.st));
                DPK_CUDA_TRY(cudaStreamSynchronize(c.st));
                const double nb = h[5] ? (double)h[5] : 1.0;
                fprintf(stderr, "agg_timing: %lld buckets; cycles per bucket: load+stage %.0f | insert %.0f | reserve %.0f | write-out %.0f | "
                        "to next top %.0f | total %.0f\n", h[5], h[0] / nb, h[1] / nb, h[2] / nb, h[3] / nb, h[4] / nb,
                        (h[0] + h[1] + h[2] + h[3] + h[4]) / nb);
            }
            }
            if (g_agg_cursor)
                DPK_LAUNCH("agg_finalize", c.st, k_agg_finalize<<<1, 256, 0, c.st>>>(c.part_err, (long long *)c.out_counts, c.nparts));
            return DPK_OK;
        }
        DPK_LAUNCH("smem_aggregate", c.st, agg<<<grid, AG_THREADS, agg_smem, c.st>>>(
            rekeys, revals, c.op, ident, c.fine_off, nfine, (1 << c.f.sub_bits) * S2, c.part_off,
            (KeyT *)c.out_keys, c.out_vals, c.out_counts, c.fb_state, c.bucket_counter));
        return DPK_OK;
    }
    if (g_reduce_impl == 1) {
        auto kern = k_bucket_reduce<KeyT, ValT, AccT>;
        int nclusters = sm_count() / BR_CLUSTER;
        if (nclusters > c.F) nclusters = c.F;
        if (nclusters < 1) nclusters = 1;
        DPK_LAUNCH("bucket_reduce", c.st, kern<<<nclusters * BR_CLUSTER, BR_THREADS, 0, c.st>>>(
            (const KeyT *)c.keys, c.aux, (const ValT *)c.vals, c.op, ident, c.f.sub_bits, c.F, c.nsrc,
            c.seg_start, c.seg_rows, c.tbl_off, c.table, c.side, c.side_used, c.part_off, (KeyT *)c.out_keys,
            c.out_vals, c.out_counts, c.bucket_counter));
    } else {
        DPK_LAUNCH("tbl_init", c.st, k_tbl_init<<<grid_cap(c.max_slots, CB_THREADS, 16), CB_THREADS, 0, c.st>>>(
            c.table, c.tbl_off + c.F, ident));
        if (c.n > 0) {
            DPK_LAUNCH("tbl_insert", c.st, k_tbl_insert<KeyT, ValT, AccT><<<grid_cap(c.n, CB_THREADS, 16), CB_THREADS, 0, c.st>>>(
                (const KeyT *)c.keys, c.aux, (const ValT *)c.vals, c.n, c.op, c.f, c.part_first << c.f.sub_bits,
                c.F, c.tbl_off, c.table, c.side, c.side_used));
        }
        size_t sh = (size_t)((c.nparts + 1) & ~1) * 4 + (size_t)c.nparts * 8;
        DPK_LAUNCH("tbl_compact", c.st, k_tbl_compact<KeyT><<<grid_cap(c.max_slots, CB_THREADS * 4, 8), CB_THREADS, sh, c.st>>>(
            c.table, c.tbl_off + c.F, c.aux, c.f, c.part_first, c.nparts, c.part_off, (KeyT *)c.out_keys,
            c.out_vals, c.out_counts));
    }
    DPK_LAUNCH("side_flush", c.st, k_side_flush<KeyT><<<1, 32, 0, c.st>>>(
        c.side, c.side_used, c.aux, c.f, c.part_first, c.nparts, c.part_off, (KeyT *)c.out_keys, c.out_vals,
        c.out_counts));
    return DPK_OK;
}

template <typename KeyT>
static int dispatch_valkind(int val_kind, const Ctx &c) {
    switch (val_kind) {
    case DPK_V_I64: return dispatch_op<KeyT, int64_t, int64_t>(c);
    case DPK_V_I32: return dispatch_op<KeyT, int32_t, int64_t>(c);
    case DPK_V_F64: return dispatch_op<KeyT, double, double>(c);
    case DPK_V_F32: return dispatch_op<KeyT, float, double>(c);
    }
    return fail(DPK_ERR_UNSUPPORTED, "value kind %d unsupported", val_kind);
}

template <typename KeyT>
static int run_combine(Ctx &c, int val_kind, int64_t *out_offsets, void *ws) {
    // workspace: Slot table[max_slots] | Slot side | int32 side_used[4] | int64 tbl_off[F+1] | int64 seg_start[nsrc*F]
    c.table = (Slot *)ws;
    c.side = c.table + c.max_slots;
    c.side_used = (int32_t *)(c.side + 1);
    c.bucket_counter = (int *)(c.side_used + 2);
    int64_t *tbl_off = (int64_t *)(c.side_used + 4);
    int64_t *seg_start = tbl_off + c.F + 2;
    c.tbl_off = tbl_off;
    c.seg_start = seg_start;
    c.part_off = out_offsets;
    // implementation 2: fine_off[F * 256 + 1] | segmented-multisplit workspace
    c.fine_off = seg_start + (int64_t)c.nsrc * c.F + 2;
    const int sb2 = choose_sb2(c.n, c.F);
    c.fb_state = (unsigned long long *)(c.fine_off + ((int64_t)c.F << sb2) + 2);
    c.part_err = (int *)(c.fb_state + ((int64_t)c.F << sb2) + 2);
    c.seg_ws = (void *)(((uintptr_t)(c.part_err + c.F + 2) + 255) & ~(uintptr_t)255);
    c.seg_ws_bytes = seg_multisplit_ws_bytes(c.n, c.F, 1 << sb2, c.nsrc);
    // side slot: free marker + identity are written by the init below; flags cleared here
    DPK_CUDA_TRY(cudaMemsetAsync(c.side_used, 0, 16, c.st));
    DPK_CUDA_TRY(cudaMemsetAsync(c.out_counts, 0, (size_t)c.nparts * 8, c.st));
    DPK_LAUNCH("tbl_plan", c.st, k_tbl_plan<<<1, CB_THREADS, 0, c.st>>>(c.seg_rows, c.nsrc, c.F, c.f.sub_bits, c.nparts,
                                                                       tbl_off, out_offsets, seg_start));
    return dispatch_valkind<KeyT>(val_kind, c);
}

__global__ void k_side_init(Slot *side, int64_t ident) {
    if (threadIdx.x == 0 && blockIdx.x == 0) { side->key = kEmpty; side->acc = ident; }
}

}  // namespace dpk

using namespace dpk;

extern "C" {

int dpk_set_option(const char *name, int64_t value) {
    if (!name) return fail(DPK_ERR_INVALID, "name is NULL");
    if (strcmp(name, "reduce_impl") == 0) {
        if (value < 0 || value > 2) return fail(DPK_ERR_INVALID, "reduce_impl must be 0, 1 or 2");
        g_reduce_impl = (int)value;
        return DPK_OK;
    }
    if (strcmp(name, "agg_impl") == 0) {
        if (value != 0 && value != 1) return fail(DPK_ERR_INVALID, "agg_impl must be 0 or 1");
        g_agg_impl = (int)value;
        return DPK_OK;
    }
    if (strcmp(name, "agg_batched") == 0) {
        if (value != 0 && value != 1) return fail(DPK_ERR_INVALID, "agg_batched must be 0 or 1");
        g_agg_batched = (int)value;
        return DPK_OK;
    }
    if (strcmp(name, "agg_split") == 0) {
        g_agg_split = value != 0;
        return DPK_OK;
    }
    if (strcmp(name, "agg_timing") == 0) {
        g_agg_timing = value != 0;
        return DPK_OK;
    }
    if (strcmp(name, "agg_pipe") == 0) {
        if (value < 0 || value > 2) return fail(DPK_ERR_INVALID, "agg_pipe must be 0, 1 or 2");
        g_agg_pipe = (int)value;
        return DPK_OK;
    }
    if (strcmp(name, "agg_cursor") == 0) {
        if (value != 0 && value != 1) return fail(DPK_ERR_INVALID, "agg_cursor must be 0 or 1");
        g_agg_cursor = (int)value;
        return DPK_OK;
    }
    if (strcmp(name, "agg_ctas") == 0) {
        if (value != 3 && value != 4) return fail(DPK_ERR_INVALID, "agg_ctas must be 3 or 4");
        g_agg_ctas = (int)value;
        return DPK_OK;
    }
    if (strcmp(name, "agg_wide") == 0) {
        if (value != 0 && value != 1) return fail(DPK_ERR_INVALID, "agg_wide must be 0 or 1");
        g_agg_wide = (int)value;
        return DPK_OK;
    }
    if (strcmp(name, "scatter_items") == 0) {
        if (value != 8 && value != 16) return fail(DPK_ERR_INVALID, "scatter_items must be 8 or 16");
        g_scatter_items = (int)value;
        return DPK_OK;
    }
    if (strcmp(name, "scatter_threads") == 0) {
        if (value != 256 && value != 512 && value != 1024) return fail(DPK_ERR_INVALID, "scatter_threads must be 256, 512 or 1024");
        g_scatter_threads = (int)value;
        return DPK_OK;
    }
    if (strcmp(name, "scatter_seg_wide") == 0) {
        g_scatter_seg_wide = value != 0;
        return DPK_OK;
    }
    if (strcmp(name, "scatter_wide_from") == 0) {
        if (value < 0 || value > DPK_MAX_PARTITIONS) return fail(DPK_ERR_INVALID, "scatter_wide_from out of range");
        g_scatter_wide_from = (int)value;
        return DPK_OK;
    }
    if (strcmp(name, "copy_tma") == 0) {
        if (value != 0 && value != 1) return fail(DPK_ERR_INVALID, "copy_tma must be 0 or 1");
        g_copy_tma = (int)value;
        return DPK_OK;
    }
    if (strcmp(name, "copy_sms") == 0) {
        if (value < 0 || value > 1024) return fail(DPK_ERR_INVALID, "copy_sms out of range");
        g_copy_sms = (int)value;
        return DPK_OK;
    }
    if (strcmp(name, "scatter_ptr_bulk") == 0) {
        if (value != 0 && value != 1) return fail(DPK_ERR_INVALID, "scatter_ptr_bulk must be 0 or 1");
        g_scatter_ptr_bulk = (int)value;
        return DPK_OK;
    }
    if (strcmp(name, "scatter_ptr_threads") == 0) {
        if (value != 512 && value != 1024) return fail(DPK_ERR_INVALID, "scatter_ptr_threads must be 512 or 1024");
        g_scatter_ptr_threads = (int)value;
        return DPK_OK;
    }
    if (strcmp(name, "scatter_bulk") == 0) {
        if (value != 0 && value != 1) return fail(DPK_ERR_INVALID, "scatter_bulk must be 0 or 1");
        g_scatter_bulk = (int)value;
        return DPK_OK;
    }
    if (strcmp(name, "count_mode") == 0) {
        if (value != 0 && value != 1) return fail(DPK_ERR_INVALID, "count_mode must be 0 or 1");
        g_count_mode = (int)value;
        return DPK_OK;
    }
    if (strcmp(name, "agg_target_rows") == 0) {
        if (value < 64 || value > AG_LIMIT) return fail(DPK_ERR_INVALID, "agg_target_rows must be in [64, %d]", AG_LIMIT);
        g_agg_target_rows = (int)value;
        return DPK_OK;
    }
    return fail(DPK_ERR_INVALID, "unknown option %s", name);
}

int64_t dpk_combine_workspace_bytes(int64_t n, int32_t nbuckets, int32_t nsrc) {
    if (n < 0) n = 0;
    if (nbuckets < 1) nbuckets = 1;
    if (nsrc < 1) nsrc = 1;
    return (max_slots_for(n, nbuckets) + 2) * (int64_t)sizeof(Slot) +
           ((int64_t)nbuckets + 4 + (int64_t)nbuckets * nsrc) * 8 + 64 +
           (((int64_t)nbuckets << choose_sb2(n, nbuckets)) + 4) * 16 + 512 + ((int64_t)nbuckets + 2) * 4 +
           seg_multisplit_ws_bytes(n, nbuckets, 1 << choose_sb2(n, nbuckets), nsrc);
}

int dpk_combine(const void *keys, int key_kind, const int64_t *key_aux, const void *vals, int val_kind, int64_t n,
                int op, int32_t P, const int64_t *thresholds, int32_t nthr, int32_t sub_bits, int32_t part_first,
                int32_t nparts, int32_t nsrc, const int64_t *seg_rows, void *out_keys, void *out_vals,
                int64_t *out_offsets, int64_t *out_counts, void *ws, int64_t ws_bytes, dpk_stream_t stream) {
    if (n < 0 || n >= ((int64_t)1 << 31)) return fail(DPK_ERR_INVALID, "n=%lld out of range [0, 2^31)", (long long)n);
    if (nparts < 1 || part_first < 0 || part_first + nparts > P)
        return fail(DPK_ERR_INVALID, "bad partition range first=%d n=%d P=%d", part_first, nparts, P);
    if (nsrc < 1) return fail(DPK_ERR_INVALID, "nsrc must be >= 1");
    if (!seg_rows || !out_counts || !out_offsets || !ws) return fail(DPK_ERR_INVALID, "NULL pointer");
    if (n > 0 && (!keys || !vals || !out_keys || !out_vals)) return fail(DPK_ERR_INVALID, "NULL pointer");
    Ctx c;
    int rc = make_partfn(P, thresholds, nthr, sub_bits, &c.f);
    if (rc) return rc;
    c.F = nparts << sub_bits;
    if (c.F > DPK_MAX_PARTITIONS)
        return fail(DPK_ERR_UNSUPPORTED, "%d local buckets exceed %d", c.F, DPK_MAX_PARTITIONS);
    if (ws_bytes < dpk_combine_workspace_bytes(n, c.F, nsrc))
        return fail(DPK_ERR_WORKSPACE, "workspace needs %lld B, got %lld", (long long)dpk_combine_workspace_bytes(n, c.F, nsrc), (long long)ws_bytes);
    c.keys = keys; c.vals = vals; c.n = n; c.op = op; c.aux = key_aux; c.key_kind = key_kind; c.val_bytes = 0;
    if (key_kind == DPK_K_ROWID && n > 0 && !key_aux) return fail(DPK_ERR_INVALID, "DPK_K_ROWID needs key_aux (the per-row hash column)");
    c.part_first = part_first; c.nparts = nparts; c.nsrc = nsrc; c.seg_rows = seg_rows;
    c.max_slots = max_slots_for(n, c.F);
    c.out_keys = out_keys; c.out_vals = (int64_t *)out_vals; c.out_counts = (unsigned long long *)out_counts;
    c.st = (cudaStream_t)stream;
    // the side slot must hold {free marker, identity} before any insert
    {
        int64_t ident = (val_kind == DPK_V_F64 || val_kind == DPK_V_F32) ? Acc<double>::identity(op) : Acc<int64_t>::identity(op);
        Slot *side = (Slot *)ws + c.max_slots;
        DPK_LAUNCH("side_init", c.st, k_side_init<<<1, 32, 0, c.st>>>(side, ident));
    }
    switch (key_kind) {
    case DPK_K_I64: return run_combine<int64_t>(c, val_kind, out_offsets, ws);
    case DPK_K_I32: return run_combine<int32_t>(c, val_kind, out_offsets, ws);
    case DPK_K_F64: return run_combine<double>(c, val_kind, out_offsets, ws);
    case DPK_K_U64: return run_combine<uint64_t>(c, val_kind, out_offsets, ws);
    case DPK_K_F32: return run_combine<float>(c, val_kind, out_offsets, ws);
    case DPK_K_ROWID: return run_combine<RowId>(c, val_kind, out_offsets, ws);
    }
    return fail(DPK_ERR_UNSUPPORTED, "key kind %d is unhashable by portable_hash", key_kind);
}

}  // extern "C"
