/* hm_internal.h -- shared by the translation units of libhetmers_b200.so (not installed) */
#ifndef HM_INTERNAL_H
#define HM_INTERNAL_H

#include <stdarg.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* record a message for hm_last_error() and return `code` */
int hm_set_error(int code, const char *fmt, ...);

#ifdef __cplusplus
}
#endif

#ifdef __CUDACC__
/* chunk-wise index construction for the loader (hm_kernels.cu) */
int hm_build_bucket_index_range(const uint64_t *d_keys, int64_t n, int bits, void *d_bucket,
                                int idx64, int64_t i0, int64_t i1, void *stream);
int hm_build_filter_range(const uint64_t *d_keys, int filter_bits, uint32_t *d_filter,
                          int64_t i0, int64_t i1, void *stream);

/* every shard's table arrays of a sharded scan, as addressable from one device (hm_symm.cu) */
typedef struct hm_shard_tabs
  { const uint64_t *keys[HM_MAX_SHARDS], *keys_lo[HM_MAX_SHARDS];
    const uint16_t *cnt[HM_MAX_SHARDS];
    const void     *bucket[HM_MAX_SHARDS];
    int64_t         n[HM_MAX_SHARDS];
  } hm_shard_tabs;
int hm_symm_resolve_sharded(const hm_shard_tabs *tabs, int bits, int idx64, int kmer, void *d_work,
                            const hm_symm_layout *layout, const hm_symm_shards *shards,
                            unsigned long long *d_plot, void *stream);
/* extract_kmer_pairs from the symmetric scan's candidates, one slice at a time (hm_symm.cu) */
int64_t hm_symm_extract_slice(const hm_symm_layout *layout);
int hm_symm_extract(const uint64_t *d_keys, const uint64_t *d_keys_lo, const uint16_t *d_cnt, int64_t n,
                    const void *d_bucket, const hm_shard_tabs *tabs, int bits, int idx64, int kmer,
                    void *d_work, const hm_symm_layout *layout, const hm_symm_shards *shards,
                    const uint16_t *d_pixmap, int64_t c0, int64_t c1, void *stream);
int hm_symm_extract_fetch(const void *d_work, const hm_symm_layout *layout, hm_pair_rec **buf, int64_t *cap,
                          int64_t *at, uint64_t *status, void *stream);

#include <cuda_runtime.h>
/* sharded conditioning (hm_condition.cu) */
int hm_sort_unique_arrays(int kmer, uint64_t *k, uint64_t *l, uint16_t *c, int64_t *pn, cudaStream_t st);
int hm_k_partition(const uint64_t *keys, const uint64_t *keys_lo, const uint16_t *cnt, int64_t n, int kmer,
                   int ethresh, int do_trim, int do_symm, const uint64_t *cut, int n_shards,
                   unsigned long long *d_cursor, uint64_t *okeys, uint64_t *okeys_lo, uint16_t *ocnt,
                   cudaStream_t st);
int hm_cuda_fail(cudaError_t e, const char *what);
#define HM_CUDA(call)                                              \
  do { cudaError_t _e = (call);                                    \
       if (_e != cudaSuccess) return hm_cuda_fail(_e,#call);       \
     } while (0)
#endif

#endif
