/*******************************************************************************************
 * hetmers_b200.h -- C ABI of libhetmers_b200.so, the B200 (sm_100a) implementation of
 * smudgeplot's `hetmers` hot path.
 *
 * The reference has NO in-process API for this path: its boundary is the `hetmers` executable
 * spawned by smudgeplot's CLI (/root/reference/src/smudgeplot/cli.py:57-72,348-361) and the
 * whole computation lives in src/lib/PloidyPlot.c + the Kmer_Stream part of src/lib/libfastk.c.
 * The drop-in therefore is our own `hetmers` executable (smudgeplot_b200/host/hetmers_main.c,
 * plain C); this header is the thin layer between that C host (or any FFI: ctypes, cgo, JNI)
 * and the CUDA kernels.  Plain pointers and sizes only; no torch / C++ types.
 *
 * Every entry point names the reference code it replaces (file:line under /root/reference).
 * All functions return 0 on success and a negative HM_E* code on failure; hm_last_error()
 * gives the message (thread-local).  There is NO CPU fallback anywhere behind this ABI.
 *
 * Layers
 *   A. hm_k_*      kernels on caller-owned DEVICE memory, enqueued on a caller stream
 *                  (used by the torch.distributed plumbing in smudgeplot_b200/dist.py and by B)
 *   B. hm_scan_*   whole path from HOST buffers holding raw FastK part payloads: H2D, unpack,
 *                  bucket index, pass 1, pass 2, D2H of the plot (used by hetmers_main.c,
 *                  by smudgeplot_b200.hetmers() and by bench.py's e2e leg)
 *   C. hm_table_*  FastK stub/part parser on the host (plain C, host/fastk_table.c)
 *******************************************************************************************/
#ifndef HETMERS_B200_H
#define HETMERS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HM_SMAX        1000                 /* max CovA+CovB      (PloidyPlot.c:48) */
#define HM_FMAX         500                 /* max min(CovA,CovB) (PloidyPlot.c:49) */
#define HM_PLOT_W      (HM_FMAX+1)
#define HM_PLOT_CELLS  ((HM_SMAX+1)*(HM_FMAX+1))   /* int64 plot[1001][501] (PloidyPlot.c:1466-1473) */
#define HM_MAX_KMER      64                 /* 1 (k<=32) or 2 (k<=64) 64-bit words per packed k-mer */
#define HM_MAX_SHARDS    16                 /* GPUs one table can be sharded over           */
#define HM_FILTER_MIN_BITS 22               /* prefix-filter width in bits                  */
#define HM_FILTER_MAX_BITS 37

#define HM_OK            0
#define HM_EINVAL       -1                  /* bad argument                                   */
#define HM_ECUDA        -2                  /* CUDA runtime / launch failure                  */
#define HM_ENOMEM       -3                  /* host or device allocation failed               */
#define HM_EIO          -4                  /* cannot open / read a table file                */
#define HM_EFORMAT      -5                  /* malformed FastK table                          */
#define HM_EUNSUPPORTED -6                  /* valid input this build does not handle (k>64)  */

const char *hm_last_error(void);
int         hm_abi_version(void);
/* number of visible CUDA devices (0 if none / no driver) */
int         hm_device_count(void);
/* name, SM count and total memory of device `dev` (for -v / bench provenance) */
int         hm_device_info(int dev, char *name, int name_len, int *sm_count, int64_t *total_mem);

/* ======================= A. kernels on device memory ===================================== *
 * Device table layout (structure of arrays, DESIGN.md §3):
 *   keys  uint64[n]  packed 2-bit k-mer, LEFT aligned (base i in bits 63-2i..62-2i), ascending;
 *                    uint64 order == FastK table order (libfastk.c packing :571-579)
 *   keys_lo uint64[n] bases 32..63 (left aligned) when k > 32, else NULL: order = (keys, keys_lo)
 *   cnt   uint16[n]  k-mer counts
 *   deg   uint8 [n]  incidence array == the reference's `Pair` (PloidyPlot.c:163), allocated
 *                    with size rounded up to a multiple of 4 and 4-byte aligned
 *   bucket           lower-bound offsets of every `bits`-bit key prefix, (1<<bits)+1 entries,
 *                    uint32 if idx64==0 (n < 2^32-1) else uint64
 * `stream` is a cudaStream_t passed as void* (NULL = default stream).                        */

/* FastK part records -> SoA.  Replaces Next_Kmer_Entry/Current_Entry (libfastk.c:1159-1176,
 * :1230-1269): re-attaches the ibyte-byte prefix found from the stub index and splits the
 * unaligned (suffix || uint16 count) record.  d_rec: n records of pbyte=kbyte-ibyte+2 bytes,
 * holding table ordinals [first, first+n); d_stub_index: int64[1<<(8*ibyte)] on the device.   */
int hm_k_unpack_records(const uint8_t *d_rec, int64_t n, int64_t first,
                        const int64_t *d_stub_index, int ibyte, int kmer,
                        uint64_t *d_keys, uint64_t *d_keys_lo, uint16_t *d_cnt, void *stream);

/* Prefix (bucket) index over the sorted keys; takes the place of the stub index + on-disk
 * bisection of GoTo_Kmer_Entry (libfastk.c:1320-1409).                                        */
int hm_k_build_bucket_index(const uint64_t *d_keys, int64_t n, int bits,
                            void *d_bucket, int idx64, void *stream);

/* Prefix presence filter: bit f of d_filter is set iff some key starts with the filter_bits-bit
 * prefix f; hm_filter_words(filter_bits) uint32 words (zeroed here).  It answers "is there any
 * k-mer with this prefix" for pass 1's probes -- the role the 4-way merge's "no list head has
 * this suffix" plays in the reference (PloidyPlot.c:618-643).                                  */
int     hm_k_build_filter(const uint64_t *d_keys, int64_t n, int filter_bits,
                          uint32_t *d_filter, void *stream);
int64_t hm_filter_words(int filter_bits);
int     hm_pick_filter_bits(int64_t n);

/* Sharded incidence array (multi-GPU, DESIGN.md §6).  The table is cut into n_shards contiguous
 * index ranges [off[r], off[r+1]); GPU r owns the incidence bytes of shard r.  deg[r] is GPU r's
 * FULL-LENGTH array as addressable from the calling GPU (peer access in one process, or a CUDA
 * IPC mapping from hm_ipc_open between processes); only its slice r is meaningful.  With such a
 * table pass 1 adds to a foreign partner's byte with a remote atomic over NVLink and pass 2 reads
 * a foreign partner's byte with a remote load, so no collective has to move the array; the caller
 * only orders the phases (all pass 1 kernels done -> pass 2; all pass 2 done -> next zeroing).
 * NULL (or n_shards <= 1) = dense mode: every byte lives in d_deg.                              */
typedef struct hm_shards
  { int32_t  n_shards;
    int32_t  self;                          /* the calling GPU's shard                          */
    int64_t  off[HM_MAX_SHARDS+1];
    uint8_t *deg[HM_MAX_SHARDS];
    void    *scratch;                       /* optional device scratch for pass 2: look-ups of       */
    int64_t  scratch_bytes;                 /*   foreign partners are batched instead of done inline */
  } hm_shards;                              /*   (size: hm_pass2_scratch_bytes)                      */

int64_t hm_pass2_scratch_bytes(int64_t range, int idx64);

/* Pass 1 (PASS1=1 of PloidyPlot.c:1489; analysis_in_core_1 :454-568, analysis_thread_1
 * :168-301, big_window :712-842): for every entry x in [lo,hi) find every one-substitution
 * neighbour y > x in the table; for each such pair with cnt sum <= SMAX add 1 to deg[x] and
 * deg[y] (mod 256, atomically) and remember the pair's upper member in d_up[x-lo]
 * (all-ones = none; d_up is initialised here).  d_deg must be zeroed by the caller before the
 * first call (several ranges / GPUs accumulate into it).                                      */
int hm_k_pass1_degree(const uint64_t *d_keys, const uint64_t *d_keys_lo,
                      const uint16_t *d_cnt, int64_t n,
                      const void *d_bucket, int bits, int idx64,
                      const uint32_t *d_filter, int filter_bits, int kmer,
                      int64_t lo, int64_t hi, uint8_t *d_deg, void *d_up,
                      const hm_shards *shards, void *stream);

/* Pass 2 (PASS1=0; analysis_in_core_2 :570-700, analysis_thread_2 :303-452): for x in [lo,hi)
 * with deg[x]<=1 whose recorded upper partner y has deg[y]<=1: plot[cx+cy][min(cx,cy)] += 1.
 * d_plot: uint64[HM_PLOT_CELLS], accumulated into (caller zeroes it).                        */
int hm_k_pass2_plot(const uint16_t *d_cnt, const uint8_t *d_deg, const void *d_up, int idx64,
                    int64_t lo, int64_t hi, unsigned long long *d_plot,
                    const hm_shards *shards, void *stream);

/* extract_kmer_pairs' pass 2 (src/lib/PloidyList.c:425-450,680-705): every isolated pair whose
 * pixel (sum, min) has a non-zero label in d_pixmap (uint16[HM_PLOT_CELLS], the PLOT array the
 * reference fills from the .sma file, PloidyList.c:1313-1350) is appended to d_out: the k-mer with
 * the higher count, the varying position and the other k-mer's base there.  *d_count (zeroed by
 * the caller) counts all matches, also those beyond `cap`.                                      */
typedef struct hm_pair_rec
  { uint64_t key_hi, key_lo;   /* packed k-mer that print_het prints (left aligned words)       */
    uint32_t smudge;           /* label from the pixmap (index into the .sma smudge list, 1-based) */
    uint8_t  pos, alt;         /* varying base position; base (0..3 = acgt) of the partner there */
    uint16_t pad;
  } hm_pair_rec;

int hm_k_pass2_extract(const uint64_t *d_keys, const uint64_t *d_keys_lo, const uint16_t *d_cnt,
                       const uint8_t *d_deg, const void *d_up, int idx64, int64_t lo, int64_t hi,
                       const uint16_t *d_pixmap, hm_pair_rec *d_out, int64_t cap,
                       unsigned long long *d_count, const hm_shards *shards, void *stream);

/* ---- the strand-symmetric scan (csrc/hm_symm.cu): every entry read once ------------------------
 * On a table that holds rc(x) with count(x) for every x -- what the reference demands before it
 * scans (examine_table, PloidyPlot.c:1199-1229; `Symmex` otherwise, :1401-1414) -- the pairs that
 * differ at a low position are mirror images of the pairs that differ at a high position, and those
 * sit in one short run of neighbouring entries.  hm_k_symm_runscan + hm_k_symm_resolve produce the
 * same plot as hm_k_pass1_degree + hm_k_pass2_plot (= the reference's two passes) on such a table;
 * hm_k_symm_fingerprint decides whether a table is one (keyed multiset fingerprints of {(x,cnt)}
 * and {(rc x,cnt)}: acc[0]==acc[2] && acc[1]==acc[3]); anything else must take the direct passes.
 * Replaces, for such tables: analysis_in_core_1/_2 + analysis_thread_1/_2 and the window / recursion
 * drivers around them (PloidyPlot.c:168-700,:712-1084); the fingerprint extends examine_table's
 * one-k-mer symmetry probe (PloidyPlot.c:1199-1229) to the whole table.
 * Side effect: hm_k_symm_runscan puts an access-policy window (persisting L2 lines) over the Bloom
 * filter on `stream` and hm_k_symm_resolve lifts it again (HETMERS_L2_PERSIST=0 disables it).      */
#define HM_SYMM_MIN_KMER 2

typedef struct hm_symm_layout               /* work area of one scan range (hm_symm_plan fills it in)     */
  { int64_t bytes;                          /* device bytes to allocate (256-byte aligned)                */
    int64_t off_header;                     /* uint64[3]: candidate count, status bits (hm_symm_status), runs */
    int64_t off_bloom;                      /* n_seg segments of seg_words uint32: Bloom filter over the  */
    int64_t seg_words;                      /*   entries with a partner in their upper half, per shard    */
    int64_t off_cand_key, off_cand_lo, off_cand_meta;   /* candidate pair records                         */
    int64_t cand_cap;
    int64_t range;
    int64_t off_runs, runs_cap;             /* heads of the runs of three or more entries (uint64 indices) */
    int32_t n_seg, pad;
  } hm_symm_layout;

typedef struct hm_symm_shards               /* several GPUs: shard r scans [off[r], off[r+1]) and fills   */
  { int32_t  n_seg, self;                   /*   Bloom segment r; the segments are all-gathered between   */
    int64_t  off[HM_MAX_SHARDS+1];          /*   the two kernels.  Cuts lie on run boundaries             */
    uint64_t first_key[HM_MAX_SHARDS];      /*   (hm_symm_align_cut); first_key[r] = keys[off[r]]         */
  } hm_symm_shards;

#define HM_SYMM_ASYMMETRIC 1                /* status bit: some rc(x) was not in the table -> result void */
#define HM_SYMM_OVERFLOW   2                /* status bit: candidate list full (cut not on a run boundary) */

int  hm_symm_plan(int64_t n, int64_t range, int kmer, int n_seg, hm_symm_layout *out);
void hm_symm_seeds(uint64_t seed[2]);       /* per-process random seeds for the fingerprint               */
/* adds the fingerprints of entries [i0,i1) to d_acc (device uint64[4], zeroed by the caller)            */
int  hm_k_symm_fingerprint(const uint64_t *d_keys, const uint64_t *d_keys_lo, const uint16_t *d_cnt,
                           int64_t i0, int64_t i1, int kmer, const uint64_t seed[2],
                           uint64_t *d_acc, void *stream);
/* "pass 1": run scan of [lo,hi): Bloom segment `self` + candidate records (both initialised here), then
 * hm_k_symm_runs for the runs it only listed (call both, in this order, on the same stream).            */
int  hm_k_symm_runscan(const uint64_t *d_keys, const uint64_t *d_keys_lo, const uint16_t *d_cnt, int64_t n,
                       const void *d_bucket, int bits, int idx64, int kmer, int64_t lo, int64_t hi,
                       void *d_work, const hm_symm_layout *layout, const hm_symm_shards *shards, void *stream);
int  hm_k_symm_runs(const uint64_t *d_keys, const uint64_t *d_keys_lo, const uint16_t *d_cnt, int64_t n,
                    const void *d_bucket, int bits, int idx64, int kmer, int64_t lo, int64_t hi,
                    void *d_work, const hm_symm_layout *layout, const hm_symm_shards *shards, void *stream);
/* "pass 2": candidates -> isolated pairs -> d_plot (accumulated into; caller zeroes it)                 */
int  hm_k_symm_resolve(const uint64_t *d_keys, const uint64_t *d_keys_lo, const uint16_t *d_cnt, int64_t n,
                       const void *d_bucket, int bits, int idx64, int kmer,
                       void *d_work, const hm_symm_layout *layout, const hm_symm_shards *shards,
                       unsigned long long *d_plot, void *stream);
int  hm_symm_status(const void *d_work, const hm_symm_layout *layout, uint64_t *n_cand, uint64_t *status,
                    void *stream);
int  hm_symm_align_cut(const uint64_t *d_keys, int64_t n, int kmer, int64_t cut, int64_t *out);

/* Device memory that can be mapped by the other ranks of a one-process-per-GPU job (CUDA IPC):
 * hm_dev_alloc gives a zeroed base allocation on the current device, hm_ipc_export its 64-byte
 * handle (send it to the peers with any host transport), hm_ipc_open maps a peer's allocation.
 * hm_p2p_native_atomics: 1 iff devices a and b can do remote atomics on each other (NVLink).    */
int hm_dev_alloc(int64_t bytes, void **dptr);
int hm_dev_free(void *dptr);
int hm_ipc_export(void *dptr, unsigned char handle[64]);
int hm_ipc_open(const unsigned char handle[64], void **dptr);
int hm_ipc_close(void *dptr);
int hm_p2p_native_atomics(int dev_a, int dev_b);

/* examine_table (PloidyPlot.c:1167-1197): smallest count v>=1 (read as int16) in [frst,last);
 * *d_min (device int) must be preset to 0x8000.                                               */
int hm_k_min_count(const uint16_t *d_cnt, int64_t frst, int64_t last, int *d_min, void *stream);

/* exact-match lookup of nq packed k-mers: d_pos[q] = table index or -1.  Replaces
 * GoTo_Kmer_Entry's "return 1 iff exact hit" use (libfastk.c:1320-1409; PloidyPlot.c:1213). */
int hm_k_find_keys(const uint64_t *d_keys, const uint64_t *d_keys_lo, int64_t n,
                   const void *d_bucket, int bits, int idx64,
                   const uint64_t *d_query, const uint64_t *d_query_lo, int64_t nq,
                   int64_t *d_pos, void *stream);

/* choice of bucket-index width for a table of n entries (DESIGN.md §4) */
int hm_pick_bucket_bits(int64_t n);

/* ======================= B. whole path from host buffers ================================= */

typedef struct hm_host_table
  { int32_t         kmer;        /* k                                                   */
    int32_t         ibyte;       /* prefix bytes folded into the stub index (1..3)      */
    int32_t         nparts;
    int32_t         minval;
    int64_t         nels;        /* sum of part_nels                                    */
    const int64_t  *index;       /* int64[1 << (8*ibyte)] bucket END offsets            */
    const int64_t  *part_nels;   /* [nparts]                                            */
    const uint8_t **part_rec;    /* [nparts] payloads: part_nels[p]*pbyte bytes each    */
    const int32_t  *part_fd;     /* optional [nparts]: open descriptor of the part file (or -1);  */
    const int64_t  *part_fd_off; /*   payload starts at this offset.  When given, the loader       */
                                 /*   pread()s with its host threads instead of touching part_rec  */
  } hm_host_table;

typedef struct hm_scan_stats
  { int64_t nels;
    int32_t n_gpus;
    int32_t bucket_bits;
    int32_t filter_bits;
    int32_t path;                /* HM_PATH_DIRECT or HM_PATH_SYMM: which scan produced the plot */
    double  ms_h2d_unpack;       /* H2D copies + unpack + bucket index (T_load, device part) */
    double  ms_pass1;
    double  ms_pass2;
    double  ms_scan;             /* pass1 + exchange + pass2 + plot reduce (T_scan)          */
    double  ms_total;            /* wall clock of the call                                   */
    int64_t kernel_launches;     /* kernels of ours launched by the call                     */
    double  ms_alloc;            /* of ms_h2d_unpack: context + device allocations           */
    double  ms_records;          /*                   host staging + H2D + unpack            */
    double  ms_index;            /*                   shard exchange + bucket index + filter */
  } hm_scan_stats;

typedef struct hm_scan hm_scan;   /* opaque: device-resident table + work buffers            */

/* Load a table onto `n_gpus` devices (ids dev[0..n_gpus-1]; every device holds a full replica,
 * work is sharded by contiguous index range, DESIGN.md §6).  Replaces Open_Kmer_Stream +
 * Clone_Kmer_Stream + the 4 GiB cache fill (libfastk.c:786-951; PloidyPlot.c:954-964).       */
int  hm_scan_create(const hm_host_table *t, const int *dev, int n_gpus, hm_scan **out);
/* Optional: start CUDA (driver + primary contexts of the first n_gpus visible devices, 0 = all) and
 * the pinned staging buffers on a background thread and return at once; hm_scan_create waits for
 * it.  Lets a short-lived process overlap CUDA start-up with opening its table files.             */
void hm_prewarm(int n_gpus);
/* host threads used to stage pageable (e.g. mmap'ed) part payloads into pinned memory during
 * hm_scan_create; 0 = min(16, cores).  The executable passes its -T here.                      */
void hm_set_io_threads(int n);
void hm_scan_destroy(hm_scan *s);
/* examine_table decisions (PloidyPlot.c:1167-1230) computed on the device */
int  hm_scan_examine(hm_scan *s, int ethresh, int *trim, int *symm);
/* Condition the device-resident table in place: trim = drop entries with count < ethresh (what
 * `Logex '...=A[<L>-]'` does), symm = add the reverse complement of every k-mer with the same
 * count (what `Symmex` does) -- PloidyPlot.c:1381-1426 shells out to those FastK tools; here the
 * table never leaves the GPU.  *nels_out = entries afterwards.                                  */
int  hm_scan_condition(hm_scan *s, int ethresh, int do_trim, int do_symm, int64_t *nels_out);
/* both passes; plot: host int64[HM_PLOT_CELLS]; stats optional.  Tables that hm_scan_create found
 * strand-symmetric (fingerprint over the whole table) take the symmetric scan of csrc/hm_symm.cu,
 * all others the direct passes; both give the reference's plot.  hm_scan_run_path forces one
 * (HM_PATH_SYMM on a table that is not symmetric is an error); HETMERS_PATH=direct|symm overrides
 * HM_PATH_AUTO.                                                                                  */
#define HM_PATH_AUTO   0
#define HM_PATH_DIRECT 1
#define HM_PATH_SYMM   2
int  hm_scan_run(hm_scan *s, int64_t *plot, hm_scan_stats *stats);
int  hm_scan_run_path(hm_scan *s, int path, int64_t *plot, hm_scan_stats *stats);
int  hm_scan_is_symmetric(const hm_scan *s);
/* the pair list of extract_kmer_pairs (runs the direct passes first if the last run did not) for a pixel->smudge map (host
 * uint16[HM_PLOT_CELLS]); *out is malloc'ed (caller frees), sorted by (smudge, k-mer).          */
int  hm_scan_extract(hm_scan *s, const uint16_t *pixmap, hm_pair_rec **out, int64_t *n_out);
/* the same list by either route.  HM_PATH_SYMM judges the candidates the symmetric scan left on the
 * devices again and writes the records of the isolated, labelled ones (running that scan first if
 * there was none since the last conditioning, or it fell back to the direct passes); it works on
 * sharded tables, allocates no device memory and is HM_EINVAL on a table that is not strand-symmetric
 * or has k < HM_SYMM_MIN_KMER.  HM_PATH_DIRECT is hm_scan_extract.  HM_PATH_AUTO takes the path
 * hm_scan_run takes (HETMERS_PATH included).  stats (may be NULL): the path taken, the number of
 * slices the candidates were judged in, the records, and the times of the extraction kernels, of
 * copying the records to the host and of sorting them there.                                      */
typedef struct hm_extract_stats
  { int32_t path, slices;
    int64_t n_records;
    double  ms_kernel, ms_copy, ms_sort;
  } hm_extract_stats;
int  hm_scan_extract_path(hm_scan *s, int path, const uint16_t *pixmap, hm_pair_rec **out, int64_t *n_out,
                          hm_extract_stats *stats);
/* one call: create + run + destroy (what bench.py's e2e leg times) */
int  hm_hetmers_host(const hm_host_table *t, const int *dev, int n_gpus,
                     int64_t *plot, hm_scan_stats *stats);
/* copy device arrays back for tests: any pointer may be NULL.  A sharded scan gives the
 * concatenation of its shards and has no incidence array (deg must be NULL).                     */
int  hm_scan_download(hm_scan *s, uint64_t *keys, uint64_t *keys_lo, uint16_t *cnt, uint8_t *deg);

/* ---- sharded placement (DESIGN.md §6): tables larger than one GPU's memory -------------------
 * Shard r of n_shards holds only the entries of its key range [cut_r, cut_r+1) on device dev[r]; the
 * cuts sit on boundaries of the first k/2 bases, so no run of the table is split.  The same device
 * may carry several logical shards.  Each shard loads 1/n_shards of the part files; the key ranges
 * are established by the first hm_scan_condition (which trims / symmetrises on the way) or, for a
 * table that needs no conditioning, by the first scan.  On a sharded scan hm_scan_examine,
 * hm_scan_condition, hm_scan_run / hm_scan_run_path(HM_PATH_SYMM), hm_scan_extract_path (HM_PATH_AUTO /
 * HM_PATH_SYMM) and hm_scan_download work; hm_scan_extract, HM_PATH_DIRECT and tables that are not
 * strand-symmetric are HM_EUNSUPPORTED.                                                             */
int  hm_scan_create_sharded(const hm_host_table *t, const int *dev, int n_shards, hm_scan **out);
/* shard r: device, index of its first entry in the concatenated table, entries, and the device bytes
 * the library keeps for it (table arrays, bucket index, plot, scan work area).  On a replica scan:
 * device r's full replica.                                                                         */
int  hm_scan_shard_info(const hm_scan *s, int r, int *dev, int64_t *first_index, int64_t *n,
                        int64_t *device_bytes);
/* Shard cuts from a sample of m records (hi / lo key words, lo NULL for k <= 32; cnt NULL = no trim):
 * records with count < min_count are left out, add_rc adds each record's reverse complement; cut[0]
 * = 0 and cut[r] = the first word of the (r/n_shards)-quantile rounded down to its first k/2 bases. */
int  hm_shard_cuts(const uint64_t *hi, const uint64_t *lo, const uint16_t *cnt, int64_t m, int kmer,
                   int min_count, int add_rc, int n_shards, uint64_t *cut);
/* Placement of a table of nels entries (do_symm: it will be symmetrised, up to 2 x nels) on n_gpus
 * devices with free_bytes[g] free: a full replica on every device if one fits (with the peak of
 * conditioning it when do_symm), else one shard per device, else neither.  Pure host arithmetic from
 * the library's own allocation sizes; need_* (optional) = the bytes per device of either choice.   */
int  hm_device_free_bytes(int dev, int64_t *free_bytes);     /* what device `dev` has free now */
#define HM_PLACE_NOFIT   0
#define HM_PLACE_REPLICA 1
#define HM_PLACE_SHARDED 2
int  hm_plan_placement(int kmer, int64_t nels, int do_symm, int n_gpus, const int64_t *free_bytes,
                       int64_t *need_replica, int64_t *need_shard);

/* ======================= C. FastK table files (host, plain C) ============================ */

typedef struct hm_table hm_table;          /* parsed stub + mapped part payloads            */

/* Open <name>[.ktab] + hidden parts; replaces Open_Kmer_Stream (libfastk.c:786-908).
 * HM_EIO if the stub cannot be opened (the reference's "Cannot open k-mer table").          */
int  hm_table_open(const char *name, hm_table **out);
void hm_table_close(hm_table *t);
const hm_host_table *hm_table_view(const hm_table *t);

/* .smu writer: "min\t(sum-min)\tcount\n", sum-major, min < FMAX (PloidyPlot.c:1603-1617) */
int  hm_write_smu(const char *path, const int64_t *plot);

#ifdef __cplusplus
}
#endif
#endif
