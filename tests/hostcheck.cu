// tests/hostcheck.cu -- runs the product's __host__ __device__ hash / partition
// functions (dpark_b200/csrc/dpk_common.cuh) on the CPU so that the arithmetic
// can be checked against the oracle without a GPU.  Test-only; not shipped.
#include "dpk_common.cuh"
extern "C" {
void hc_hash_i64(const int64_t *k, int64_t n, int64_t *o) { for (int64_t i = 0; i < n; i++) o[i] = dpk::hash_i64(k[i]); }
void hc_hash_u64(const uint64_t *k, int64_t n, int64_t *o) { for (int64_t i = 0; i < n; i++) o[i] = dpk::hash_u64(k[i]); }
void hc_hash_f64(const double *k, int64_t n, int64_t *o) { for (int64_t i = 0; i < n; i++) o[i] = dpk::hash_f64(k[i]); }
void hc_hash_bytes(const uint8_t *d, const int64_t *off, int64_t n, int mode, int64_t *o) {
    for (int64_t i = 0; i < n; i++)
        o[i] = mode == 0 ? dpk::hash_bytes_signed(d + off[i], off[i + 1] - off[i])
                         : dpk::hash_utf8_codepoints(d + off[i], off[i + 1] - off[i]);
}
void hc_hash_tuple(const int64_t *item_hash, int64_t n, int32_t arity, int64_t *o) {
    for (int64_t i = 0; i < n; i++) o[i] = dpk::hash_tuple_items(item_hash, n, i, arity);
}
int hc_partition(const int64_t *h, int64_t n, int32_t P, const int64_t *thr, int32_t nthr, int32_t *o) {
    dpk::PartFn f;
    int rc = dpk::make_partfn(P, thr, nthr, 0, &f);
    if (rc) return rc;
    for (int64_t i = 0; i < n; i++) o[i] = f(h[i]);
    return 0;
}
// the tokeniser's per-thread arithmetic (dpk_strings.cu k_tok_count / k_tok_emit) walked sequentially: token starts from
// the 16-byte masks, token ends by the forward scan; returns the token count, -1 if a byte >= 0x80 was seen
int64_t hc_tokenize(const uint8_t *data, int64_t n, int64_t *starts, int64_t *lens) {
    int64_t m = 0;
    bool any_hi = false;
    for (int64_t i0 = 0; i0 < n; i0 += dpk::TK_BYTES) {
        bool hi = false;
        uint32_t mask = dpk::tok_starts16(data, n, i0, &hi);
        any_hi |= hi;
        for (int j = 0; j < dpk::TK_BYTES; j++)
            if (mask & (1u << j)) {
                const int64_t b = i0 + j;
                int64_t e = b + 1;
                while (e < n && !dpk::tok_ws(data[e])) e++;
                starts[m] = b;
                lens[m] = e - b;
                m++;
            }
    }
    return any_hi ? -1 : m;
}
int hc_bucket(const int64_t *h, int64_t n, int32_t P, int32_t sub_bits, int32_t *o) {
    dpk::PartFn f;
    int rc = dpk::make_partfn(P, nullptr, 0, sub_bits, &f);
    if (rc) return rc;
    for (int64_t i = 0; i < n; i++) o[i] = f.bucket(h[i]);
    return 0;
}
// slot hash of the shared-memory merge tables (k_smem_aggregate2/3) over 64 key bits
void hc_slot_hash32(const int64_t *kb, int64_t n, uint32_t *o) { for (int64_t i = 0; i < n; i++) o[i] = dpk::slot_hash32((uint64_t)kb[i]); }
// fine bucket of the reduce side's second-level split inside its first-level bucket: the PartFn mode 5 that
// dpk_combine builds for 2^sb2 fine buckets under a first level of sub_bits
void hc_fine_bucket(const int64_t *h, int64_t n, int32_t sub_bits, int32_t sb2, int32_t *o) {
    dpk::PartFn f{};
    f.mode = 5; f.P = 1 << sb2; f.shift = 32 - sub_bits - sb2; f.sub_bits = 0;
    for (int64_t i = 0; i < n; i++) o[i] = f.bucket(h[i]);
}
}
