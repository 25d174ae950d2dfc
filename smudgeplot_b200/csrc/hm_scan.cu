/*******************************************************************************************
 * hm_scan.cu -- layer B of include/hetmers_b200.h: the whole hetmers path from HOST buffers.
 *
 *   hm_scan_create   H2D of the raw FastK part payloads (double-buffered, copy stream ||
 *                    unpack stream), SoA unpack, bucket index          ("T_load", device part)
 *   hm_scan_examine  trimmed? / symmetric? decisions of examine_table (PloidyPlot.c:1167-1230)
 *   hm_scan_run      pass 1 -> (degree exchange when >1 GPU) -> pass 2 -> plot D2H  ("T_scan")
 *
 * Every device holds a full replica of the table whenever one fits; work is sharded by contiguous
 * index range [lo_g, hi_g).  With one GPU there is no exchange at all.  A table too large for one
 * device is placed SHARDED instead (hm_scan_create_sharded, DESIGN.md §6): device g keeps only the
 * entries [lo_g, hi_g) of its run-aligned key range, at local index 0.
 * With several GPUs in this single process the loader gathers the shards over NVLink peer
 * copies and foreign degree bytes are reached through the owner's array (remote atomics / loads
 * fused into the two kernels; summed by a peer-memory kernel of hm_peer.cu if there are no
 * native NVLink atomics); the
 * one-process-per-GPU variant (torch.distributed / NCCL) lives in smudgeplot_b200/dist.py and
 * uses layer A directly.
 *******************************************************************************************/
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>
#include <pthread.h>
#include <unistd.h>
#include <errno.h>

#include "hetmers_b200.h"
#include "hm_internal.h"

#define HM_MAX_GPUS 16
#define LOAD_CHUNK  (16ll<<20)        /* records per H2D/unpack chunk */

typedef struct
  { int                 dev;
    cudaStream_t        st, st_copy;
    uint64_t           *keys;
    uint64_t           *keys_lo;      /* second key word, k > 32 only */
    uint16_t           *cnt;
    uint8_t            *deg;          /* n rounded up to 4 */
    void               *bucket;
    uint32_t           *filter;       /* prefix presence bitmap */
    void               *up;           /* hi-lo entries */
    void               *p2scratch;    /* pass 2 defer list (multi-GPU peer mode) */
    int64_t             p2scratch_bytes;
    unsigned long long *plot;
    int64_t             lo, hi;       /* this device's work range */
    void               *symm_work;    /* work area of the strand-symmetric scan (hm_symm.cu) */
    hm_symm_layout      symm_layout;
    int64_t             slo, shi;     /* its run-aligned range */
    uint64_t           *fp_acc;       /* device uint64[4]: symmetry fingerprint sums of the entries loaded here */
  } DevTable;

struct hm_scan
  { int      kmer, ibyte, bits, fpos, idx64, ngpu;
    int64_t  n;
    DevTable d[HM_MAX_GPUS];
    double   ms_load, ms_alloc, ms_records, ms_index;
    int      ran, peer_mode;              /* ran: the direct passes have filled deg/up (extract, download) */
    hm_shards sh[HM_MAX_GPUS];
    int64_t  launches;
    int      symmetric;                   /* fingerprint verdict: every rc(x) present with count(x)        */
    int      have_direct;                 /* deg / up / filter allocated and the filter built               */
    int      have_symm;                   /* symmetric-scan work areas allocated, cuts aligned              */
    int      last_path;                   /* HM_PATH_DIRECT / HM_PATH_SYMM of the last run                  */
    int      symm_ran;                    /* the work areas hold the candidates + Bloom segments of a clean  */
                                          /*   symmetric scan of the current table (extraction reads them)   */
    int      invalid;                     /* a failed conditioning left the replicas inconsistent            */
    int      sharded;                     /* d[r] holds only entries [d[r].lo, d[r].hi), at local index 0   */
    int      aligned;                     /* sharded: shard r owns the keys in [cut[r], cut[r+1]) (run-aligned) */
    uint64_t cut[HM_MAX_GPUS];
    hm_symm_shards ssh[HM_MAX_GPUS];
    uint64_t seed[2];
  };

static double now_ms(void)
{ struct timespec ts;
  clock_gettime(CLOCK_MONOTONIC,&ts);
  return ts.tv_sec*1e3 + ts.tv_nsec*1e-6;
}

/* multi-GPU helpers (hm_peer.cu) */
int hm_peer_enable(const int *dev, int n);
int hm_peer_sum_deg(uint8_t **deg, const int64_t *lo, const int64_t *hi, const int *dev,
                    cudaStream_t *st, int n, int64_t nels);
int hm_peer_sum_plot(unsigned long long **plot, const int *dev, cudaStream_t *st, int n);
/* GPU trim / symmetrise (hm_condition.cu) */
int hm_condition_arrays(int kmer, int ethresh, int do_trim, int do_symm,
                        uint64_t **pk, uint64_t **pl, uint16_t **pc, int64_t *pn, cudaStream_t st);

/* Device allocations of a one-GPU scan come from the device's stream-ordered memory pool with a
 * release threshold of "never": a second hm_scan_create in the same process (bench e2e leg, a
 * service handling many tables) reuses the memory instead of paying cudaMalloc / cudaFree of
 * several GB every call (measured: ~20 ms of a 61 ms call).  Multi-GPU scans keep cudaMalloc:
 * their arrays are mapped by the peers.  HETMERS_NO_POOL=1 disables the pool.                  */
#define POOL_MAX 32
typedef struct { void *p[POOL_MAX]; int n, enabled; } PoolReg;
static PoolReg g_pool[64];

static void pool_setup(int dev, int enable)
{ static int configured[64] = {0};
  if (dev < 0 || dev >= 64) return;
  g_pool[dev].enabled = enable && getenv("HETMERS_NO_POOL") == NULL;
  if (g_pool[dev].enabled && !configured[dev])
    { cudaMemPool_t pool;
      unsigned long long never = ~0ull;
      if (cudaDeviceGetDefaultMemPool(&pool,dev) != cudaSuccess ||
          cudaMemPoolSetAttribute(pool,cudaMemPoolAttrReleaseThreshold,&never) != cudaSuccess)
        { cudaGetLastError(); g_pool[dev].enabled = 0; }
      configured[dev] = 1;
    }
}

static cudaError_t dalloc(int dev, cudaStream_t st, void **p, size_t bytes)
{ PoolReg *R = (dev >= 0 && dev < 64) ? g_pool+dev : NULL;
  if (R != NULL && R->enabled && R->n < POOL_MAX)
    { cudaError_t e = cudaMallocAsync(p,bytes,st);
      if (e == cudaSuccess)
        { R->p[R->n++] = *p; return e; }
      cudaGetLastError();
    }
  return cudaMalloc(p,bytes);
}

static void dfree(int dev, cudaStream_t st, void *p)
{ PoolReg *R = (dev >= 0 && dev < 64) ? g_pool+dev : NULL;
  if (p == NULL) return;
  if (R != NULL)
    for (int k = 0; k < R->n; k++)
      if (R->p[k] == p)
        { R->p[k] = R->p[--R->n];
          cudaFreeAsync(p,st);
          return;
        }
  cudaFree(p);
}

static void free_dev(DevTable *D)
{ cudaSetDevice(D->dev);
  dfree(D->dev,D->st,D->keys);  dfree(D->dev,D->st,D->keys_lo); dfree(D->dev,D->st,D->cnt);
  dfree(D->dev,D->st,D->deg);   dfree(D->dev,D->st,D->bucket);  dfree(D->dev,D->st,D->filter);
  dfree(D->dev,D->st,D->up);    dfree(D->dev,D->st,D->plot);
  dfree(D->dev,D->st,D->fp_acc);
  if (D->p2scratch) cudaFree(D->p2scratch);
  dfree(D->dev,D->st,D->symm_work);
  if (D->st) cudaStreamSynchronize(D->st);
  if (D->st)      cudaStreamDestroy(D->st);
  if (D->st_copy) cudaStreamDestroy(D->st_copy);
  memset(D,0,sizeof(*D));
}

extern "C" void hm_scan_destroy(hm_scan *s)
{ if (s == NULL)
    return;
  for (int g = 0; g < s->ngpu; g++)
    { int had_symm = (s->d[g].symm_work != NULL);
      free_dev(s->d+g);
      if (had_symm)                              /* hand the L2 lines the Bloom window made persisting back */
        { cudaCtxResetPersistingL2Cache(); cudaGetLastError(); }
    }
  free(s);
}

/* ---- host-side staging for pageable sources (mmap'ed part files) -------------------------
 * cudaMemcpyAsync from pageable memory is staged by the driver on one thread (~3-6 GB/s).  The
 * executable's table lives in the page cache, so the loader copies each chunk into a pinned
 * buffer with a few host threads (this is what the reference's -T is for on the host side) while
 * the previous chunk is in flight to the GPU.                                                   */
static int g_io_threads = 0;

extern "C" void hm_set_io_threads(int n) { g_io_threads = n; }

typedef struct { uint8_t *dst; const uint8_t *src; size_t bytes; int fd; int64_t off; int err; } CopyJob;

static void *copy_worker(void *arg)
{ CopyJob *j = (CopyJob *) arg;
  j->err = 0;
  if (j->fd < 0)
    memcpy(j->dst,j->src,j->bytes);
  else
    { size_t got = 0;                                   /* page cache -> pinned buffer, no mapping */
      while (got < j->bytes)
        { ssize_t r = pread(j->fd,j->dst+got,j->bytes-got,j->off+(int64_t) got);
          if (r < 0 && errno == EINTR) continue;
          if (r <= 0) { j->err = (r < 0) ? errno : -1; break; }    /* -1: file shorter than its header says */
          got += (size_t) r;
        }
    }
  return NULL;
}

/* fill dst[0,bytes) from memory `src` (fd < 0) or from file `fd` at `off`, with the I/O threads;
 * 0, or the errno (-1 = short file) of the first slice that could not be read                  */
static int parallel_fill(uint8_t *dst, const uint8_t *src, int fd, int64_t foff, size_t bytes)
{ int nt = g_io_threads;
  if (nt <= 0)
    { long c = sysconf(_SC_NPROCESSORS_ONLN);
      nt = c > 16 ? 16 : (c < 1 ? 1 : (int) c);
    }
  if (nt > 64) nt = 64;
  if (bytes < ((size_t) 4<<20)) nt = 1;
  pthread_t th[64];
  CopyJob   job[64];
  int       created[64];
  size_t    per = ((bytes/nt)+4095) & ~(size_t) 4095;
  int       njob = 0, err = 0;
  for (int k = 0; k < nt; k++)
    { size_t off = per*k;
      if (off >= bytes) break;
      job[k].dst = dst+off; job[k].src = src ? src+off : NULL;
      job[k].fd = fd; job[k].off = foff+(int64_t) off;
      job[k].bytes = bytes-off < per ? bytes-off : per;
      created[k] = 0;
      njob = k+1;
      if (k == nt-1 || off+per >= bytes)
        { copy_worker(job+k); break; }                 /* the calling thread takes the last slice */
      if (pthread_create(th+k,NULL,copy_worker,job+k) != 0)
        copy_worker(job+k);                            /* no thread to be had: copy inline */
      else
        created[k] = 1;
    }
  for (int k = 0; k < njob; k++)
    { if (created[k])
        pthread_join(th[k],NULL);
      if (job[k].err != 0 && err == 0)
        err = job[k].err;
    }
  return err;
}

/* ---- background start-up (hm_prewarm) ---- */
#define PIN_CACHE_BYTES ((size_t) (LOAD_CHUNK/2) * 8)
static pthread_t g_warm_th;
static int       g_warm_state = 0;            /* 0 idle, 1 running, 2 joined */
static int       g_warm_ngpu = 1;
static uint8_t  *g_pin_cache[2] = { NULL, NULL };

static void *warm_one(void *arg)
{ int g = (int) (intptr_t) arg;
  if (cudaSetDevice(g) == cudaSuccess)
    cudaFree(0);                              /* creates the primary context */
  return NULL;
}

static void *warm_worker(void *)
{ int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess)
    { cudaGetLastError(); return NULL; }
  int use = (g_warm_ngpu <= 0 || g_warm_ngpu > n) ? n : g_warm_ngpu;
  if (use > HM_MAX_GPUS) use = HM_MAX_GPUS;
  pthread_t th[HM_MAX_GPUS];
  int       made[HM_MAX_GPUS];
  for (int g = 1; g < use; g++)               /* the contexts of several GPUs at once */
    made[g] = (pthread_create(th+g,NULL,warm_one,(void *) (intptr_t) g) == 0);
  warm_one((void *) (intptr_t) 0);
  for (int g = 1; g < use; g++)
    if (made[g]) pthread_join(th[g],NULL);
    else         warm_one((void *) (intptr_t) g);
  cudaSetDevice(0);
  for (int i = 0; i < 2; i++)
    if (cudaHostAlloc(&g_pin_cache[i],PIN_CACHE_BYTES,cudaHostAllocDefault) != cudaSuccess)
      { cudaGetLastError(); g_pin_cache[i] = NULL; }
  return NULL;
}

extern "C" void hm_prewarm(int n_gpus)
{ if (g_warm_state != 0)
    return;
  g_warm_ngpu = n_gpus;
  if (pthread_create(&g_warm_th,NULL,warm_worker,NULL) == 0)
    g_warm_state = 1;
}

static void prewarm_join(void)
{ if (g_warm_state == 1)
    { pthread_join(g_warm_th,NULL);
      g_warm_state = 2;
    }
}

static int is_pageable(const void *p)
{ cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a,p) != cudaSuccess)
    { cudaGetLastError(); return 1; }
  return (a.type == cudaMemoryTypeUnregistered);
}

/* Load ordinals [first, first+count) of the table onto device D (keys/cnt already allocated for
 * the full table).  Walks the parts, copies payload chunks H2D on st_copy into one of two device
 * staging buffers and unpacks them on st (copy of chunk c+1 overlaps the unpack of chunk c);
 * pageable sources additionally go through two pinned host buffers filled by host threads.      */
static int load_range(hm_scan *s, DevTable *D, const hm_host_table *t, const int64_t *d_index,
                      int64_t first, int64_t count, int64_t base)
{ int      kbyte = (t->kmer+3)>>2;
  int      pbyte = kbyte - t->ibyte + 2;
  uint8_t *stage[2] = { NULL, NULL };
  uint8_t *pin[2]   = { NULL, NULL };
  cudaEvent_t copied[2], unpacked[2];
  int64_t  chunk = LOAD_CHUNK;
  int      rc = HM_OK, b = 0, used[2] = {0,0};
  int      staged = 0;

  if (count <= 0)
    return HM_OK;
  for (int p = 0; p < t->nparts && !staged; p++)
    if (t->part_nels[p] > 0 &&
        ((t->part_fd != NULL && t->part_fd[p] >= 0) || is_pageable(t->part_rec[p])))
      staged = 1;
  if (staged)
    chunk = LOAD_CHUNK/2;
  if (chunk > count) chunk = count;
  int pin_cached[2] = {0,0};
  for (int i = 0; i < 2; i++)
    { HM_CUDA(dalloc(D->dev,D->st,(void **) &stage[i],(size_t) chunk*pbyte));
      if (staged)
        { if (s->ngpu == 1 && g_pin_cache[i] != NULL && (size_t) chunk*pbyte <= PIN_CACHE_BYTES)
            { pin[i] = g_pin_cache[i]; g_pin_cache[i] = NULL; pin_cached[i] = 1; }   /* from hm_prewarm */
          else
            HM_CUDA(cudaHostAlloc(&pin[i],(size_t) chunk*pbyte,cudaHostAllocDefault));
        }
      HM_CUDA(cudaEventCreateWithFlags(&copied[i],cudaEventDisableTiming));
      HM_CUDA(cudaEventCreateWithFlags(&unpacked[i],cudaEventDisableTiming));
    }
  /* one GPU: the whole table arrives here in order, so the bucket index is built chunk by chunk
   * right behind the unpack (hidden behind the next chunk's H2D); so is the symmetry fingerprint   */
  const int inc = (!s->sharded && s->ngpu == 1 && first == 0 && count == s->n);
  HM_CUDA(cudaStreamSynchronize(D->st));         /* (pool) allocations are used on both streams */
  int64_t pstart = 0;                               /* ordinal of the part's first record */
  for (int p = 0; p < t->nparts && rc == HM_OK; p++)
    { int64_t pn   = t->part_nels[p];
      int64_t from = first > pstart ? first : pstart;
      int64_t to   = first+count < pstart+pn ? first+count : pstart+pn;
      for (int64_t o = from; o < to && rc == HM_OK; o += chunk)
        { int64_t        m   = to-o < chunk ? to-o : chunk;
          const uint8_t *src = t->part_rec[p] + (o-pstart)*pbyte;
          if (staged)
            { if (used[b])
                cudaEventSynchronize(copied[b]);      /* pin[b] has left for the GPU */
              int ferr;
              if (t->part_fd != NULL && t->part_fd[p] >= 0)
                ferr = parallel_fill(pin[b],NULL,t->part_fd[p],t->part_fd_off[p]+(o-pstart)*pbyte,(size_t) m*pbyte);
              else
                ferr = parallel_fill(pin[b],src,-1,0,(size_t) m*pbyte);
              if (ferr != 0)
                { rc = hm_set_error(HM_EIO,"short read on part %d of the table (%s)",p+1,
                                    ferr > 0 ? strerror(ferr) : "file truncated");
                  break;
                }
              src = pin[b];
            }
          if (used[b])
            cudaStreamWaitEvent(D->st_copy,unpacked[b],0);
          cudaError_t e = cudaMemcpyAsync(stage[b],src,(size_t) m*pbyte,cudaMemcpyHostToDevice,D->st_copy);
          if (e != cudaSuccess) { rc = hm_cuda_fail(e,"cudaMemcpyAsync(H2D records)"); break; }
          cudaEventRecord(copied[b],D->st_copy);
          cudaStreamWaitEvent(D->st,copied[b],0);
          rc = hm_k_unpack_records(stage[b],m,o,d_index,t->ibyte,t->kmer,D->keys+(o-base),
                                   D->keys_lo ? D->keys_lo+(o-base) : NULL,D->cnt+(o-base),D->st);
          __sync_fetch_and_add(&s->launches,1);
          cudaEventRecord(unpacked[b],D->st);
          if (inc && rc == HM_OK)
            { rc = hm_build_bucket_index_range(D->keys,s->n,s->bits,D->bucket,s->idx64,o,o+m,D->st);
              __sync_fetch_and_add(&s->launches,1);
            }
          if (rc == HM_OK && s->kmer >= HM_SYMM_MIN_KMER)       /* symmetry fingerprint of what this device loads */
            { rc = hm_k_symm_fingerprint(D->keys,D->keys_lo,D->cnt,o-base,o-base+m,s->kmer,s->seed,D->fp_acc,D->st);
              __sync_fetch_and_add(&s->launches,1);
            }
          used[b] = 1;
          b ^= 1;
        }
      pstart += pn;
    }
  cudaStreamSynchronize(D->st_copy);
  cudaError_t e = cudaStreamSynchronize(D->st);
  for (int i = 0; i < 2; i++)
    { dfree(D->dev,D->st,stage[i]); cudaEventDestroy(copied[i]); cudaEventDestroy(unpacked[i]);
      if (pin[i] != NULL)
        { if (pin_cached[i]) g_pin_cache[i] = pin[i];        /* back into the cache for the next table */
          else               cudaFreeHost(pin[i]);
        }
    }
  if (rc == HM_OK && e != cudaSuccess)
    rc = hm_cuda_fail(e,"unpack");
  return rc;
}

/* one host thread per device: stub index upload + this device's shard of the records */
typedef struct { hm_scan *s; int g; const hm_host_table *t; int rc; char msg[512]; } LoadJob;

static void *load_worker(void *arg)
{ LoadJob  *J = (LoadJob *) arg;
  hm_scan  *s = J->s;
  DevTable *D = s->d+J->g;
  int64_t  *d_index = NULL;
  int64_t   ixlen = (int64_t) 1 << (8*J->t->ibyte);
  J->rc = HM_OK;
  cudaError_t e = cudaSetDevice(D->dev);
  if (e == cudaSuccess) e = dalloc(D->dev,D->st,(void **) &d_index,sizeof(int64_t)*ixlen);
  if (e == cudaSuccess) e = cudaMemcpyAsync(d_index,J->t->index,sizeof(int64_t)*ixlen,cudaMemcpyHostToDevice,D->st);
  if (e == cudaSuccess) e = cudaMemsetAsync(D->fp_acc,0,4*sizeof(uint64_t),D->st);
  if (e == cudaSuccess) e = cudaStreamSynchronize(D->st);     /* pool memory is about to be used on the copy stream too */
  if (e != cudaSuccess)
    J->rc = hm_cuda_fail(e,"stub index upload");
  else
    J->rc = load_range(s,D,J->t,d_index,D->lo,D->hi-D->lo,s->sharded ? D->lo : 0);
  if (d_index != NULL) dfree(D->dev,D->st,d_index);
  if (J->rc != HM_OK)
    { strncpy(J->msg,hm_last_error(),sizeof(J->msg)-1); J->msg[sizeof(J->msg)-1] = 0; }
  return NULL;
}

/* sum of the per-device fingerprint accumulators -> s->symmetric */
static int fingerprint_verdict(hm_scan *s)
{ uint64_t tot[4] = {0,0,0,0};
  if (s->kmer < HM_SYMM_MIN_KMER)
    { s->symmetric = 0; return HM_OK; }
  for (int g = 0; g < s->ngpu; g++)
    { uint64_t h[4];
      HM_CUDA(cudaSetDevice(s->d[g].dev));
      HM_CUDA(cudaMemcpyAsync(h,s->d[g].fp_acc,sizeof(h),cudaMemcpyDeviceToHost,s->d[g].st));
      HM_CUDA(cudaStreamSynchronize(s->d[g].st));
      for (int k = 0; k < 4; k++) tot[k] += h[k];
    }
  s->symmetric = (tot[0] == tot[2] && tot[1] == tot[3]);
  return HM_OK;
}

static int create_scan(const hm_host_table *t, const int *dev, int n_gpus, int sharded, hm_scan **out)
{ double t0 = now_ms();
  if (t == NULL || out == NULL || n_gpus < 1 || n_gpus > HM_MAX_GPUS)
    return hm_set_error(HM_EINVAL,"hm_scan_create: bad arguments");
  if (t->kmer < 1 || t->kmer > HM_MAX_KMER)
    return hm_set_error(HM_EUNSUPPORTED,"k-mer length %d not supported by this build (1..%d)",
                        t->kmer,HM_MAX_KMER);
  int kbyte = (t->kmer+3)>>2;
  if (t->ibyte < 1 || t->ibyte > 3 || t->ibyte > kbyte)
    return hm_set_error(HM_EFORMAT,"table has ibyte=%d with k=%d",t->ibyte,t->kmer);
  prewarm_join();
  if (hm_device_count() < 1)
    return hm_set_error(HM_ECUDA,"no CUDA device visible (this build has no CPU fallback)");

  hm_scan *s = (hm_scan *) calloc(1,sizeof(hm_scan));
  if (s == NULL)
    return hm_set_error(HM_ENOMEM,"out of host memory");
  s->kmer = t->kmer; s->ibyte = t->ibyte; s->n = t->nels; s->ngpu = n_gpus;
  s->sharded = sharded;
  s->bits  = hm_pick_bucket_bits(s->n);
  s->fpos  = hm_pick_filter_bits(s->n);
  s->idx64 = (s->n >= 0xFFFFFFF0ll);
  if (sharded)                                     /* bucket offsets are local to a shard */
    s->idx64 = ((s->n+n_gpus-1)/n_gpus >= 0xFFFFFFF0ll);
  hm_symm_seeds(s->seed);
  int64_t n  = s->n;
  size_t  ib = s->idx64 ? 8 : 4;
  int     rc = HM_OK;

  if (n_gpus > 1 && (rc = hm_peer_enable(dev,n_gpus)) != HM_OK)
    { free(s); return rc; }

  /* table arrays + bucket index; the work buffers of either scan path are allocated by the path
   * that runs (ensure_direct / ensure_symm)                                                     */
  for (int g = 0; g < n_gpus && rc == HM_OK; g++)
    { DevTable *D = s->d+g;
      D->dev = dev ? dev[g] : g;
      D->lo  = n*g/n_gpus;
      D->hi  = n*(g+1)/n_gpus;
      int64_t na = sharded ? D->hi-D->lo : n;            /* entries held on this device */
      cudaError_t e;
#define TRY(call) if (rc == HM_OK && (e = (call)) != cudaSuccess) rc = hm_cuda_fail(e,#call)
      TRY(cudaSetDevice(D->dev));
      pool_setup(D->dev,n_gpus == 1 && !sharded);
      TRY(cudaStreamCreateWithFlags(&D->st,cudaStreamNonBlocking));
      TRY(cudaStreamCreateWithFlags(&D->st_copy,cudaStreamNonBlocking));
      TRY(dalloc(D->dev,D->st,(void **) &D->keys,sizeof(uint64_t)*(size_t) (na+1)));
      if (t->kmer > 32)
        TRY(dalloc(D->dev,D->st,(void **) &D->keys_lo,sizeof(uint64_t)*(size_t) (na+1)));
      TRY(dalloc(D->dev,D->st,(void **) &D->cnt,sizeof(uint16_t)*(size_t) (na+8)));
      TRY(dalloc(D->dev,D->st,(void **) &D->bucket,ib*(((size_t) 1<<s->bits)+1)));
      TRY(dalloc(D->dev,D->st,(void **) &D->plot,sizeof(unsigned long long)*HM_PLOT_CELLS));
      TRY(dalloc(D->dev,D->st,(void **) &D->fp_acc,4*sizeof(uint64_t)));
#undef TRY
    }

  double t_alloc = now_ms();
  /* each device unpacks its own shard from the host -- all devices at once, one host thread each --
   * then the shards are exchanged over peer copies so that every device ends with the full table */
  if (rc == HM_OK)
    { LoadJob   job[HM_MAX_GPUS];
      pthread_t th[HM_MAX_GPUS];
      int       created[HM_MAX_GPUS];
      for (int g = 0; g < n_gpus; g++)
        { job[g].s = s; job[g].g = g; job[g].t = t; job[g].rc = HM_OK; job[g].msg[0] = 0;
          created[g] = 0;
          if (g == n_gpus-1 || pthread_create(th+g,NULL,load_worker,job+g) != 0)
            load_worker(job+g);                              /* the calling thread takes the last device */
          else
            created[g] = 1;
        }
      for (int g = 0; g < n_gpus; g++)
        { if (created[g]) pthread_join(th[g],NULL);
          if (job[g].rc != HM_OK && rc == HM_OK)
            rc = hm_set_error(job[g].rc,"%s",job[g].msg);
        }
    }
  double t_rec = now_ms();
  if (n_gpus > 1 && rc == HM_OK && !sharded)
    { for (int g = 0; g < n_gpus && rc == HM_OK; g++)        /* all-gather by peer copies */
        for (int h = 0; h < n_gpus && rc == HM_OK; h++)
          if (h != g)
            { DevTable *S = s->d+h, *D = s->d+g;
              int64_t m = S->hi-S->lo;
              if (m <= 0) continue;
              cudaSetDevice(D->dev);
              cudaError_t e = cudaMemcpyPeerAsync(D->keys+S->lo,D->dev,S->keys+S->lo,S->dev,
                                                  sizeof(uint64_t)*(size_t) m,D->st);
              if (e == cudaSuccess && D->keys_lo != NULL)
                e = cudaMemcpyPeerAsync(D->keys_lo+S->lo,D->dev,S->keys_lo+S->lo,S->dev,
                                        sizeof(uint64_t)*(size_t) m,D->st);
              if (e == cudaSuccess)
                e = cudaMemcpyPeerAsync(D->cnt+S->lo,D->dev,S->cnt+S->lo,S->dev,
                                        sizeof(uint16_t)*(size_t) m,D->st);
              if (e != cudaSuccess) rc = hm_cuda_fail(e,"cudaMemcpyPeerAsync(table shard)");
            }
      for (int g = 0; g < n_gpus; g++)
        { cudaSetDevice(s->d[g].dev); cudaStreamSynchronize(s->d[g].st); }
    }
  for (int g = 0; g < n_gpus && rc == HM_OK && (n_gpus > 1 || sharded); g++)     /* (one GPU: done chunk-wise) */
    { DevTable *D = s->d+g;
      cudaSetDevice(D->dev);
      rc = hm_k_build_bucket_index(D->keys,sharded ? D->hi-D->lo : n,s->bits,D->bucket,s->idx64,D->st);
      s->launches += 1;
    }
  for (int g = 0; g < n_gpus; g++)
    { cudaSetDevice(s->d[g].dev);
      cudaError_t e = cudaStreamSynchronize(s->d[g].st);
      if (rc == HM_OK && e != cudaSuccess) rc = hm_cuda_fail(e,"table load");
    }
  if (rc == HM_OK)
    rc = fingerprint_verdict(s);
  if (rc != HM_OK)
    { hm_scan_destroy(s); return rc; }
  s->ms_load = now_ms()-t0;
  s->ms_alloc = t_alloc-t0; s->ms_records = t_rec-t_alloc; s->ms_index = now_ms()-t_rec;
  *out = s;
  return HM_OK;
}

extern "C" int hm_scan_create(const hm_host_table *t, const int *dev, int n_gpus, hm_scan **out)
{ return create_scan(t,dev,n_gpus,0,out); }

extern "C" int hm_scan_create_sharded(const hm_host_table *t, const int *dev, int n_shards, hm_scan **out)
{ if (t != NULL && t->kmer < HM_SYMM_MIN_KMER)
    return hm_set_error(HM_EUNSUPPORTED,"a sharded table needs k >= %d (k=%d)",HM_SYMM_MIN_KMER,t->kmer);
  if (n_shards > HM_MAX_SHARDS)
    return hm_set_error(HM_EINVAL,"hm_scan_create_sharded: at most %d shards",HM_MAX_SHARDS);
  return create_scan(t,dev,n_shards,1,out);
}

/* reverse complement of a left-aligned packed k-mer (k <= 32) */
static uint64_t revcomp64(uint64_t x, int k)
{ x = ~x;
  x = ((x >> 2)  & 0x3333333333333333ull) | ((x & 0x3333333333333333ull) << 2);
  x = ((x >> 4)  & 0x0F0F0F0F0F0F0F0Full) | ((x & 0x0F0F0F0F0F0F0F0Full) << 4);
  x = ((x >> 8)  & 0x00FF00FF00FF00FFull) | ((x & 0x00FF00FF00FF00FFull) << 8);
  x = ((x >> 16) & 0x0000FFFF0000FFFFull) | ((x & 0x0000FFFF0000FFFFull) << 16);
  x = (x >> 32) | (x << 32);
  if (k < 32)
    x = (x & (((uint64_t) 1 << (2*k))-1)) << (64-2*k);
  return x;
}

/* reverse complement of a left-aligned packed k-mer of 33..64 bases held in two words */
static void revcomp128(uint64_t hi, uint64_t lo, int k, uint64_t *rhi, uint64_t *rlo)
{ /* reversing all 64 slots swaps the words; the k real bases end up right-aligned over 128 bits */
  uint64_t a = revcomp64(lo,32), b = revcomp64(hi,32);      /* full-word reverse complements */
  int      sh = 2*(64-k);                                    /* pad slots now sit on top: shift them out */
  if (sh == 0) { *rhi = a; *rlo = b; }
  else         { *rhi = (a << sh) | (b >> (64-sh)); *rlo = b << sh; }
}

/* ---- sharded placement (DESIGN.md §6) --------------------------------------------------------- */

static int cmp_u64(const void *a, const void *b)
{ uint64_t x = *(const uint64_t *) a, y = *(const uint64_t *) b;
  return x < y ? -1 : (x > y);
}

extern "C" int hm_shard_cuts(const uint64_t *hi, const uint64_t *lo, const uint16_t *cnt, int64_t m, int kmer,
                             int min_count, int add_rc, int n_shards, uint64_t *cut)
{ if (hi == NULL || cut == NULL || m < 0 || n_shards < 1 || n_shards > HM_MAX_SHARDS ||
      kmer < HM_SYMM_MIN_KMER || kmer > HM_MAX_KMER || (kmer > 32 && add_rc && lo == NULL))
    return hm_set_error(HM_EINVAL,"hm_shard_cuts: bad arguments");
  const uint64_t pmask = ~(uint64_t) 0 << (64-2*(kmer>>1));      /* the first k/2 bases: one run */
  uint64_t *v = (uint64_t *) malloc(sizeof(uint64_t)*(size_t) (2*m+1));
  if (v == NULL)
    return hm_set_error(HM_ENOMEM,"out of host memory");
  int64_t nv = 0;
  for (int64_t i = 0; i < m; i++)
    { if (cnt != NULL && (int) cnt[i] < min_count)
        continue;
      v[nv++] = hi[i] & pmask;
      if (add_rc)
        { uint64_t r, rl;
          if (kmer > 32) revcomp128(hi[i],lo[i],kmer,&r,&rl);
          else           r = revcomp64(hi[i],kmer);
          v[nv++] = r & pmask;
        }
    }
  qsort(v,(size_t) nv,sizeof(uint64_t),cmp_u64);
  cut[0] = 0;
  for (int r = 1; r < n_shards; r++)
    cut[r] = nv > 0 ? v[nv*r/n_shards] : 0;
  free(v);
  return HM_OK;
}

/* Device bytes one device keeps for the symmetric scan of a table of which it holds `n` entries and
 * scans `range` of them: table arrays, bucket index, plot, fingerprint sums and the scan's work area
 * (candidate records and run heads for `range` entries, Bloom segments sized for n_seg x seg_n).  A
 * replica holds all n entries and scans its run-aligned 1/G of them (ensure_symm); a shard holds
 * and scans its own entries.                                                                      */
static int64_t resident_bytes(int kmer, int64_t n, int64_t range, int bits, int idx64, int n_seg, int64_t seg_n)
{ hm_symm_layout L;
  int64_t b = (int64_t) sizeof(uint64_t)*(n+1)*(kmer > 32 ? 2 : 1) + (int64_t) sizeof(uint16_t)*(n+8)
            + (idx64 ? 8 : 4)*(((int64_t) 1 << bits)+1) + (int64_t) sizeof(unsigned long long)*HM_PLOT_CELLS + 32;
  if (range > seg_n*n_seg) range = seg_n*n_seg;
  if (kmer >= HM_SYMM_MIN_KMER && hm_symm_plan(seg_n*n_seg,range,kmer,n_seg,&L) == HM_OK)
    b += L.bytes;
  return b;
}

/* peak of conditioning m entries into m2 on one device (replica: hm_condition_arrays; shard: raw +
 * outbox, then inbox + its sort buffers + flags + CUB temporary storage, about one more copy)     */
static int64_t condition_peak(int kmer, int64_t m, int64_t m2)
{ int64_t tb = 8*(kmer > 32 ? 2 : 1) + 2;
  int64_t a = tb*(m+m2);
  int64_t b = 3*tb*m2 + (kmer > 32 ? 8*m2 : 0) + m2;
  return a > b ? a : b;
}

/* entries a shard may receive: for k > 32 its sort carries a 32-bit permutation (hm_sort_unique_arrays) */
#define SHARD_SORT_MAX 0xFFFFFFF0ll

extern "C" int hm_plan_placement(int kmer, int64_t nels, int do_symm, int n_gpus, const int64_t *free_bytes,
                                 int64_t *need_replica, int64_t *need_shard)
{ if (kmer < 1 || kmer > HM_MAX_KMER || nels < 0 || n_gpus < 1 || n_gpus > HM_MAX_SHARDS || free_bytes == NULL)
    return hm_set_error(HM_EINVAL,"hm_plan_placement: bad arguments");
  const int     G = n_gpus;
  const int64_t n2 = do_symm ? 2*nels : nels;          /* entries after conditioning (at most) */
  int64_t fmin = free_bytes[0];
  for (int g = 1; g < G; g++)
    if (free_bytes[g] < fmin) fmin = free_bytes[g];
  /* a replica: the whole table on every device, each scanning its run-aligned 1/G (+ slack for the
   * alignment); symmetrising it in place first (hm_condition_arrays) peaks above that               */
  int64_t rng = (n2+G-1)/G;
  rng += rng/20 + 1024;
  int64_t rep = resident_bytes(kmer,n2,rng,hm_pick_bucket_bits(n2),n2 >= 0xFFFFFFF0ll,G,(n2+G-1)/G);
  if (do_symm)
    { int64_t pk = resident_bytes(kmer,nels,0,hm_pick_bucket_bits(nels),nels >= 0xFFFFFFF0ll,1,nels) + condition_peak(kmer,nels,n2);
      if (pk > rep) rep = pk;
      if (kmer > 32 && n2 >= 0xFFFFFFF0ll)             /* beyond hm_condition_arrays' 32-bit sort indices */
        rep = INT64_MAX;
    }
  /* a shard: its 1/S share with 5 % slack for the sampled cuts, the bucket index of the whole table's width */
  int64_t per = (nels+G-1)/G, per2 = (n2+G-1)/G;
  per2 += per2/20 + 1024;
  int     bits = hm_pick_bucket_bits(n2);
  int64_t fix = (per2 >= 0xFFFFFFF0ll ? 8 : 4)*(((int64_t) 1 << bits)+1) + (int64_t) sizeof(unsigned long long)*HM_PLOT_CELLS;
  int64_t shd = resident_bytes(kmer,per2,per2,bits,per2 >= 0xFFFFFFF0ll,G,per2);
  if (fix + condition_peak(kmer,per,per2) > shd)          /* the redistribution, before the scan's work area exists */
    shd = fix + condition_peak(kmer,per,per2);
  if (kmer > 32 && per2 >= SHARD_SORT_MAX)
    shd = INT64_MAX;
  if (need_replica) *need_replica = rep;
  if (need_shard)   *need_shard = shd;
  if (rep <= fmin)  return HM_PLACE_REPLICA;
  if (G > 1 && shd <= fmin) return HM_PLACE_SHARDED;
  return HM_PLACE_NOFIT;
}

extern "C" int hm_device_free_bytes(int dev, int64_t *free_bytes)
{ size_t fr = 0, tot = 0;
  if (free_bytes == NULL)
    return hm_set_error(HM_EINVAL,"hm_device_free_bytes: no output");
  int cur = 0;
  cudaGetDevice(&cur);
  HM_CUDA(cudaSetDevice(dev));
  cudaError_t e = cudaMemGetInfo(&fr,&tot);
  cudaSetDevice(cur);
  if (e != cudaSuccess)
    return hm_cuda_fail(e,"cudaMemGetInfo");
  *free_bytes = (int64_t) fr;
  return HM_OK;
}

/* Give every shard the run-aligned key range [cut[r], cut[r+1]) -- trimming (count >= ethresh) and
 * adding reverse complements on the way when asked: sample -> cuts (host) -> partition_kernel
 * counts, then fills per-owner outboxes -> peer copies into each owner's inbox (originals first) ->
 * sort + first-of-run per owner -> bucket index + fingerprint per shard.                         */
typedef struct { int dev, kmer, rc; cudaStream_t st; uint64_t *k, *l; uint16_t *c; int64_t *n; char msg[512]; } SortJob;

static void *sort_worker(void *arg)
{ SortJob *J = (SortJob *) arg;
  cudaError_t e = cudaSetDevice(J->dev);
  J->rc = (e != cudaSuccess) ? hm_cuda_fail(e,"cudaSetDevice") : hm_sort_unique_arrays(J->kmer,J->k,J->l,J->c,J->n,J->st);
  if (J->rc != HM_OK)
    { strncpy(J->msg,hm_last_error(),sizeof(J->msg)-1); J->msg[sizeof(J->msg)-1] = 0; }
  return NULL;
}

static int shard_partition(hm_scan *s, int ethresh, int do_trim, int do_symm)
{ const int S = s->ngpu, kmer = s->kmer, two = (kmer > 32);
  int       rc = HM_OK;
  /* 1. cuts from an equal-stride sample of all shards */
  const int64_t want = 1 << 15;
  int64_t step = s->n / ((int64_t) S*want);
  if (step < 1) step = 1;
  int64_t ns = 0;
  for (int r = 0; r < S; r++) ns += (s->d[r].hi-s->d[r].lo+step-1)/step;
  uint64_t *sh = (uint64_t *) malloc(sizeof(uint64_t)*(size_t) (ns+1));
  uint64_t *sl = (uint64_t *) malloc(sizeof(uint64_t)*(size_t) (ns+1));
  uint16_t *sc = (uint16_t *) malloc(sizeof(uint16_t)*(size_t) (ns+1));
  if (sh == NULL || sl == NULL || sc == NULL)
    { free(sh); free(sl); free(sc); return hm_set_error(HM_ENOMEM,"out of host memory"); }
  int64_t at = 0;
  for (int r = 0; r < S && rc == HM_OK; r++)
    { DevTable *D = s->d+r;
      int64_t   m = (D->hi-D->lo+step-1)/step;
      if (m <= 0) continue;
      cudaError_t e = cudaSetDevice(D->dev);
      if (e == cudaSuccess) e = cudaMemcpy2D(sh+at,8,D->keys,8*step,8,m,cudaMemcpyDeviceToHost);
      if (e == cudaSuccess && two) e = cudaMemcpy2D(sl+at,8,D->keys_lo,8*step,8,m,cudaMemcpyDeviceToHost);
      if (e == cudaSuccess) e = cudaMemcpy2D(sc+at,2,D->cnt,2*step,2,m,cudaMemcpyDeviceToHost);
      if (e != cudaSuccess) rc = hm_cuda_fail(e,"shard sample");
      at += m;
    }
  uint64_t cut[HM_MAX_SHARDS];
  if (rc == HM_OK)
    rc = hm_shard_cuts(sh,two ? sl : NULL,do_trim ? sc : NULL,at,kmer,ethresh,do_symm,S,cut);
  free(sh); free(sl); free(sc);
  if (rc != HM_OK)
    return rc;

  /* 2. count per (source, owner, kind), then fill each source's outbox */
  typedef unsigned long long ull;
  ull      cnts[HM_MAX_SHARDS][2*HM_MAX_SHARDS];
  int64_t  ooff[HM_MAX_SHARDS][2*HM_MAX_SHARDS+1];        /* slot offsets inside source r's outbox */
  ull     *d_cur[HM_MAX_SHARDS];
  uint64_t *ok[HM_MAX_SHARDS], *ol[HM_MAX_SHARDS];
  uint16_t *oc[HM_MAX_SHARDS];
  memset(d_cur,0,sizeof(d_cur)); memset(ok,0,sizeof(ok)); memset(ol,0,sizeof(ol)); memset(oc,0,sizeof(oc));
  uint64_t *ik[HM_MAX_SHARDS], *il[HM_MAX_SHARDS];
  uint16_t *ic[HM_MAX_SHARDS];
  memset(ik,0,sizeof(ik)); memset(il,0,sizeof(il)); memset(ic,0,sizeof(ic));
  int64_t  inn[HM_MAX_SHARDS];
  ull      fill_end[HM_MAX_SHARDS][2*HM_MAX_SHARDS];
#define TRY(call) do { cudaError_t _e = (call); if (_e != cudaSuccess && rc == HM_OK) rc = hm_cuda_fail(_e,#call); } while (0)
  /* every device works at once: each loop only enqueues, the synchronisation follows in a loop of its own */
  for (int r = 0; r < S && rc == HM_OK; r++)
    { DevTable *D = s->d+r;
      TRY(cudaSetDevice(D->dev));
      TRY(cudaMalloc(&d_cur[r],sizeof(ull)*2*S));
      TRY(cudaMemsetAsync(d_cur[r],0,sizeof(ull)*2*S,D->st));
      if (rc == HM_OK)
        rc = hm_k_partition(D->keys,D->keys_lo,D->cnt,D->hi-D->lo,kmer,ethresh,do_trim,do_symm,cut,S,
                            d_cur[r],NULL,NULL,NULL,D->st);
      TRY(cudaMemcpyAsync(cnts[r],d_cur[r],sizeof(ull)*2*S,cudaMemcpyDeviceToHost,D->st));
      s->launches += 1;
    }
  for (int r = 0; r < S; r++)
    { cudaSetDevice(s->d[r].dev);
      TRY(cudaStreamSynchronize(s->d[r].st));
    }
  for (int o = 0; o < S && rc == HM_OK; o++)               /* what every owner will receive */
    { inn[o] = 0;
      for (int r = 0; r < S; r++) inn[o] += (int64_t) (cnts[r][2*o] + cnts[r][2*o+1]);
      if (two && inn[o] >= SHARD_SORT_MAX)
        rc = hm_set_error(HM_EUNSUPPORTED,"shard %d would receive %lld entries of k=%d, more than its sort handles "
                          "(%lld): use more shards",o,(long long) inn[o],kmer,(long long) SHARD_SORT_MAX);
    }
  if (rc != HM_OK)                                          /* nothing has been touched yet */
    { for (int r = 0; r < S; r++)
        { cudaSetDevice(s->d[r].dev); cudaFree(d_cur[r]); }
      return rc;
    }
  for (int r = 0; r < S && rc == HM_OK; r++)
    { DevTable *D = s->d+r;
      ooff[r][0] = 0;
      for (int j = 0; j < 2*S; j++) ooff[r][j+1] = ooff[r][j] + (int64_t) cnts[r][j];
      int64_t tot = ooff[r][2*S];
      TRY(cudaSetDevice(D->dev));
      TRY(cudaMalloc(&ok[r],sizeof(uint64_t)*(size_t) (tot+1)));
      if (two) TRY(cudaMalloc(&ol[r],sizeof(uint64_t)*(size_t) (tot+1)));
      TRY(cudaMalloc(&oc[r],sizeof(uint16_t)*(size_t) (tot+1)));
      TRY(cudaMemcpyAsync(d_cur[r],ooff[r],sizeof(ull)*2*S,cudaMemcpyHostToDevice,D->st));
      if (rc == HM_OK)
        rc = hm_k_partition(D->keys,D->keys_lo,D->cnt,D->hi-D->lo,kmer,ethresh,do_trim,do_symm,cut,S,
                            d_cur[r],ok[r],ol[r],oc[r],D->st);
      TRY(cudaMemcpyAsync(fill_end[r],d_cur[r],sizeof(ull)*2*S,cudaMemcpyDeviceToHost,D->st));
      s->launches += 1;
    }
  for (int r = 0; r < S; r++)
    { DevTable *D = s->d+r;
      cudaSetDevice(D->dev);
      TRY(cudaStreamSynchronize(D->st));
      for (int j = 0; j < 2*S && rc == HM_OK; j++)           /* a fill that disagrees with its count */
        if ((int64_t) fill_end[r][j] != ooff[r][j+1])
          rc = hm_set_error(HM_ECUDA,"partition of shard %d: slot %d filled to %llu, counted %lld",r,j,
                            fill_end[r][j],(long long) ooff[r][j+1]);
    }
  int raw_gone = (rc == HM_OK);
  for (int r = 0; r < S && rc == HM_OK; r++)                /* the raw shards now live in the outboxes */
    { DevTable *D = s->d+r;
      cudaSetDevice(D->dev);
      cudaFree(D->keys); cudaFree(D->keys_lo); cudaFree(D->cnt);
      D->keys = NULL; D->keys_lo = NULL; D->cnt = NULL;
    }
  /* 3. every owner pulls its slots: originals of all sources first, then their reverse complements */
  for (int o = 0; o < S && rc == HM_OK; o++)
    { DevTable *O = s->d+o;
      int64_t   tot = inn[o];
      TRY(cudaSetDevice(O->dev));
      TRY(cudaMalloc(&ik[o],sizeof(uint64_t)*(size_t) (tot+1)));
      if (two) TRY(cudaMalloc(&il[o],sizeof(uint64_t)*(size_t) (tot+1)));
      TRY(cudaMalloc(&ic[o],sizeof(uint16_t)*(size_t) (tot+8)));
      int64_t dst = 0;
      for (int kind = 0; kind < 2; kind++)
        for (int r = 0; r < S && rc == HM_OK; r++)
          { int64_t c = (int64_t) cnts[r][2*o+kind], src = ooff[r][2*o+kind];
            if (c == 0) continue;
            int sd = s->d[r].dev;
            TRY(cudaMemcpyPeerAsync(ik[o]+dst,O->dev,ok[r]+src,sd,sizeof(uint64_t)*(size_t) c,O->st));
            if (two) TRY(cudaMemcpyPeerAsync(il[o]+dst,O->dev,ol[r]+src,sd,sizeof(uint64_t)*(size_t) c,O->st));
            TRY(cudaMemcpyPeerAsync(ic[o]+dst,O->dev,oc[r]+src,sd,sizeof(uint16_t)*(size_t) c,O->st));
            dst += c;
          }
    }
  for (int o = 0; o < S; o++)
    { cudaSetDevice(s->d[o].dev);
      TRY(cudaStreamSynchronize(s->d[o].st));
    }
  for (int r = 0; r < S; r++)
    { cudaSetDevice(s->d[r].dev);
      cudaFree(ok[r]); cudaFree(ol[r]); cudaFree(oc[r]); cudaFree(d_cur[r]);
    }
  /* 4. sort + first of every run, per owner: one host thread each (the sort synchronises its stream) */
  if (rc == HM_OK)
    { SortJob   job[HM_MAX_SHARDS];
      pthread_t th[HM_MAX_SHARDS];
      int       made[HM_MAX_SHARDS];
      for (int o = 0; o < S; o++)
        { job[o].dev = s->d[o].dev; job[o].st = s->d[o].st; job[o].kmer = kmer;
          job[o].k = ik[o]; job[o].l = il[o]; job[o].c = ic[o]; job[o].n = &inn[o]; job[o].msg[0] = 0;
          made[o] = (o+1 < S) && pthread_create(th+o,NULL,sort_worker,job+o) == 0;
          if (!made[o])
            sort_worker(job+o);
        }
      for (int o = 0; o < S; o++)
        { if (made[o]) pthread_join(th[o],NULL);
          if (job[o].rc != HM_OK && rc == HM_OK)
            rc = hm_set_error(job[o].rc,"%s",job[o].msg);
        }
      s->launches += 6*S;
    }
  if (rc != HM_OK)
    { for (int o = 0; o < S; o++)
        { cudaSetDevice(s->d[o].dev); cudaFree(ik[o]); cudaFree(il[o]); cudaFree(ic[o]); }
      if (raw_gone)
        s->invalid = 1;                      /* the raw shards are gone */
      return rc;
    }
  /* 5. the shards' new ranges, index and fingerprints */
  int64_t pos = 0, nmax = 0;
  for (int o = 0; o < S; o++)
    { DevTable *O = s->d+o;
      O->keys = ik[o]; O->keys_lo = il[o]; O->cnt = ic[o];
      O->lo = pos; O->hi = pos+inn[o]; pos += inn[o];
      if (inn[o] > nmax) nmax = inn[o];
      s->cut[o] = cut[o];
    }
  s->n     = pos;
  s->bits  = hm_pick_bucket_bits(s->n);
  s->fpos  = hm_pick_filter_bits(s->n);
  s->idx64 = (nmax >= 0xFFFFFFF0ll);
  size_t ib = s->idx64 ? 8 : 4;
  for (int o = 0; o < S && rc == HM_OK; o++)
    { DevTable *O = s->d+o;
      TRY(cudaSetDevice(O->dev));
      dfree(O->dev,O->st,O->bucket); O->bucket = NULL;
      TRY(cudaMalloc(&O->bucket,ib*(((size_t) 1<<s->bits)+1)));
      TRY(cudaMemsetAsync(O->fp_acc,0,4*sizeof(uint64_t),O->st));
      if (rc == HM_OK)
        rc = hm_k_build_bucket_index(O->keys,O->hi-O->lo,s->bits,O->bucket,s->idx64,O->st);
      if (rc == HM_OK)
        rc = hm_k_symm_fingerprint(O->keys,O->keys_lo,O->cnt,0,O->hi-O->lo,kmer,s->seed,O->fp_acc,O->st);
      s->launches += 2;
    }
  for (int o = 0; o < S; o++)
    { cudaSetDevice(s->d[o].dev);
      TRY(cudaStreamSynchronize(s->d[o].st));
    }
#undef TRY
  if (rc == HM_OK)
    rc = fingerprint_verdict(s);
  if (rc != HM_OK)
    { s->invalid = 1; return rc; }
  s->aligned = 1;
  return HM_OK;
}

extern "C" int hm_scan_shard_info(const hm_scan *s, int r, int *dev, int64_t *first_index, int64_t *n,
                                  int64_t *device_bytes)
{ if (s == NULL || r < 0 || r >= s->ngpu)
    return hm_set_error(HM_EINVAL,"hm_scan_shard_info: no shard %d",r);
  const DevTable *D = s->d+r;
  int64_t na = s->sharded ? D->hi-D->lo : s->n;
  if (dev)         *dev = D->dev;
  if (first_index) *first_index = s->sharded ? D->lo : 0;
  if (n)           *n = na;
  if (device_bytes)
    { int64_t b = (int64_t) sizeof(uint64_t)*(na+1)*(D->keys_lo ? 2 : 1) + (int64_t) sizeof(uint16_t)*(na+8)
                + (s->idx64 ? 8 : 4)*(((int64_t) 1 << s->bits)+1) + (int64_t) sizeof(unsigned long long)*HM_PLOT_CELLS
                + 4*(int64_t) sizeof(uint64_t);
      if (D->symm_work != NULL) b += D->symm_layout.bytes;
      *device_bytes = b;
    }
  return HM_OK;
}

/* work buffers of the direct passes (hm_kernels.cu): incidence array, recorded partners, prefix filter */
static int ensure_direct(hm_scan *s)
{ if (s->have_direct)
    return HM_OK;
  int64_t n  = s->n;
  size_t  ib = s->idx64 ? 8 : 4;
  int     rc = HM_OK;
  for (int g = 0; g < s->ngpu && rc == HM_OK; g++)
    { DevTable *D = s->d+g;
      cudaError_t e;
#define TRY(call) if (rc == HM_OK && (e = (call)) != cudaSuccess) rc = hm_cuda_fail(e,#call)
      TRY(cudaSetDevice(D->dev));
      if (D->deg == NULL)    TRY(dalloc(D->dev,D->st,(void **) &D->deg,(size_t) ((n+4)&~3ll)));
      if (D->up == NULL)     TRY(dalloc(D->dev,D->st,(void **) &D->up,ib*(size_t) (D->hi-D->lo+1)));
      if (D->filter == NULL) TRY(dalloc(D->dev,D->st,(void **) &D->filter,sizeof(uint32_t)*(size_t) hm_filter_words(s->fpos)));
#undef TRY
      if (rc == HM_OK)
        rc = hm_k_build_filter(D->keys,n,s->fpos,D->filter,D->st);
      s->launches += 1;
    }
  for (int g = 0; g < s->ngpu; g++)
    { cudaSetDevice(s->d[g].dev);
      cudaError_t e = cudaStreamSynchronize(s->d[g].st);
      if (rc == HM_OK && e != cudaSuccess) rc = hm_cuda_fail(e,"prefix filter");
    }
  if (rc == HM_OK)
    s->have_direct = 1;
  return rc;
}

/* sharded table: the key ranges are made run-aligned first (without conditioning, if that has not
 * happened yet); shard r scans its own entries and fills Bloom segment r, segments sized for the
 * largest shard; a key's owner is found by comparing it with the cuts                            */
static int ensure_symm_sharded(hm_scan *s)
{ int G = s->ngpu, rc;
  if (!s->aligned && (rc = shard_partition(s,0,0,0)) != HM_OK)
    return rc;
  int64_t nmax = 1;
  for (int g = 0; g < G; g++)
    if (s->d[g].hi-s->d[g].lo > nmax) nmax = s->d[g].hi-s->d[g].lo;
  for (int g = 0; g < G; g++)
    { DevTable *D = s->d+g;
      hm_symm_shards *sh = s->ssh+g;
      memset(sh,0,sizeof(*sh));
      sh->n_seg = G; sh->self = g;
      for (int r = 0; r < G; r++)
        { sh->off[r] = s->d[r].lo; sh->first_key[r] = r > 0 ? s->cut[r] : 0; }
      sh->off[G] = s->n;
      D->slo = 0; D->shi = D->hi-D->lo;
      if ((rc = hm_symm_plan(nmax*G,D->shi,s->kmer,G,&D->symm_layout)) != HM_OK)
        return rc;
      HM_CUDA(cudaSetDevice(D->dev));
      if (D->symm_work != NULL) { cudaFree(D->symm_work); D->symm_work = NULL; }
      HM_CUDA(cudaMalloc(&D->symm_work,(size_t) D->symm_layout.bytes));
    }
  s->have_symm = 1;
  return HM_OK;
}

/* work areas of the strand-symmetric scan (hm_symm.cu); several GPUs: cuts on run boundaries */
static int ensure_symm(hm_scan *s)
{ if (s->have_symm)
    return HM_OK;
  if (s->sharded)
    return ensure_symm_sharded(s);
  int     G = s->ngpu;
  int64_t n = s->n, cut[HM_MAX_GPUS+1];
  cut[0] = 0; cut[G] = n;
  HM_CUDA(cudaSetDevice(s->d[0].dev));
  for (int g = 1; g < G; g++)
    { int rc = hm_symm_align_cut(s->d[0].keys,n,s->kmer,n*g/G,&cut[g]);
      if (rc != HM_OK) return rc;
      if (cut[g] < cut[g-1]) cut[g] = cut[g-1];
    }
  for (int g = 0; g < G; g++)
    { DevTable *D = s->d+g;
      hm_symm_shards *sh = s->ssh+g;
      memset(sh,0,sizeof(*sh));
      sh->n_seg = G; sh->self = g;
      for (int r = 0; r <= G; r++) sh->off[r] = cut[r];
      HM_CUDA(cudaSetDevice(D->dev));
      for (int r = 1; r < G; r++)
        if (cut[r] < n)
          HM_CUDA(cudaMemcpy(&sh->first_key[r],D->keys+cut[r],sizeof(uint64_t),cudaMemcpyDeviceToHost));
        else
          sh->first_key[r] = ~0ull;
      D->slo = cut[g]; D->shi = cut[g+1];
      int rc = hm_symm_plan(n,D->shi-D->slo,s->kmer,G,&D->symm_layout);
      if (rc != HM_OK) return rc;
      if (D->symm_work != NULL) { dfree(D->dev,D->st,D->symm_work); D->symm_work = NULL; }
      HM_CUDA(dalloc(D->dev,D->st,&D->symm_work,(size_t) D->symm_layout.bytes));
    }
  s->have_symm = 1;
  return HM_OK;
}

/* Trim (count >= ethresh) and / or symmetrise (add reverse complements) the device-resident table
 * in place: what the reference gets from `Logex` and `Symmex` (PloidyPlot.c:1381-1426), without
 * leaving the GPU.  Every device conditions its own replica (deterministic, identical results);
 * the index structures and work buffers are rebuilt for the new size.                          */
extern "C" int hm_scan_condition(hm_scan *s, int ethresh, int do_trim, int do_symm, int64_t *nels_out)
{ int     G = s->ngpu, rc = HM_OK;
  int64_t n_new = -1;
  if (s->invalid)
    return hm_set_error(HM_EINVAL,"this scan was left unusable by an earlier failed conditioning");
  if (!do_trim && !do_symm)
    { if (nels_out) *nels_out = s->n;
      return HM_OK;
    }
  if (s->sharded)
    { for (int g = 0; g < G; g++)
        { DevTable *D = s->d+g;
          HM_CUDA(cudaSetDevice(D->dev));
          HM_CUDA(cudaStreamSynchronize(D->st));
          if (D->symm_work != NULL) { cudaFree(D->symm_work); D->symm_work = NULL; }
        }
      s->have_symm = 0; s->symm_ran = 0;
      rc = shard_partition(s,ethresh,do_trim,do_symm);
      if (nels_out) *nels_out = s->n;
      return rc;
    }
  /* everything derived from the old table goes first: work buffers of both paths, the index */
  s->ran = 0; s->have_direct = 0; s->have_symm = 0; s->symm_ran = 0;
  for (int g = 0; g < G; g++)
    { DevTable *D = s->d+g;
      HM_CUDA(cudaSetDevice(D->dev));
      HM_CUDA(cudaStreamSynchronize(D->st));
      dfree(D->dev,D->st,D->deg);    D->deg = NULL;
      dfree(D->dev,D->st,D->up);     D->up = NULL;
      dfree(D->dev,D->st,D->bucket); D->bucket = NULL;
      dfree(D->dev,D->st,D->filter); D->filter = NULL;
      if (D->symm_work != NULL) { dfree(D->dev,D->st,D->symm_work); D->symm_work = NULL; }
      /* the table arrays are about to be replaced by plain cudaMalloc'ed ones: hand pooled ones back
       * (conditioning frees them with cudaFree, which is legal for pool memory)                    */
      PoolReg *R = g_pool + (D->dev < 64 ? D->dev : 0);
      void *arr[3] = { D->keys, D->keys_lo, D->cnt };
      for (int a = 0; a < 3; a++)
        for (int k = 0; k < R->n; k++)
          if (arr[a] != NULL && R->p[k] == arr[a])
            R->p[k] = R->p[--R->n];
    }
  for (int g = 0; g < G && rc == HM_OK; g++)
    { DevTable *D = s->d+g;
      int64_t   n = s->n;
      HM_CUDA(cudaSetDevice(D->dev));
      rc = hm_condition_arrays(s->kmer,ethresh,do_trim,do_symm,&D->keys,&D->keys_lo,&D->cnt,&n,D->st);
      s->launches += 6;
      if (rc == HM_OK && n_new >= 0 && n != n_new)
        rc = hm_set_error(HM_ECUDA,"conditioning gave %lld entries on GPU %d but %lld on GPU 0",
                          (long long) n,D->dev,(long long) n_new);
      if (rc != HM_OK && g > 0)
        s->invalid = 1;                        /* the replicas no longer agree */
      n_new = n;
    }
  if (rc == HM_OK)
    { s->n     = n_new;
      s->bits  = hm_pick_bucket_bits(s->n);
      s->fpos  = hm_pick_filter_bits(s->n);
      s->idx64 = (s->n >= 0xFFFFFFF0ll);
    }
  /* index (also after a failure on GPU 0: the old table is intact and stays usable) */
  size_t ib = s->idx64 ? 8 : 4;
  int    rc2 = HM_OK;
  for (int g = 0; g < G && rc2 == HM_OK && !s->invalid; g++)
    { DevTable *D = s->d+g;
      int64_t   n = s->n;
      cudaError_t e;
      D->lo = n*g/G;
      D->hi = n*(g+1)/G;
#define TRY(call) if (rc2 == HM_OK && (e = (call)) != cudaSuccess) rc2 = hm_cuda_fail(e,#call)
      TRY(cudaSetDevice(D->dev));
      TRY(dalloc(D->dev,D->st,(void **) &D->bucket,ib*(((size_t) 1<<s->bits)+1)));
      TRY(cudaMemsetAsync(D->fp_acc,0,4*sizeof(uint64_t),D->st));
#undef TRY
      if (rc2 == HM_OK)
        rc2 = hm_k_build_bucket_index(D->keys,n,s->bits,D->bucket,s->idx64,D->st);
      if (rc2 == HM_OK && s->kmer >= HM_SYMM_MIN_KMER)
        rc2 = hm_k_symm_fingerprint(D->keys,D->keys_lo,D->cnt,D->lo,D->hi,s->kmer,s->seed,D->fp_acc,D->st);
      s->launches += 2;
    }
  for (int g = 0; g < G; g++)
    { cudaSetDevice(s->d[g].dev);
      cudaError_t e = cudaStreamSynchronize(s->d[g].st);
      if (rc2 == HM_OK && e != cudaSuccess) rc2 = hm_cuda_fail(e,"re-index after conditioning");
    }
  if (rc2 == HM_OK && !s->invalid)
    rc2 = fingerprint_verdict(s);
  if (rc2 != HM_OK)
    s->invalid = 1;
  if (nels_out) *nels_out = s->n;
  return rc != HM_OK ? rc : rc2;
}

/* examine_table (PloidyPlot.c:1167-1230).  trim: smallest non-zero count among the middle <=1e8
 * entries >= ethresh.  symm: reverse complement of entry 1 (moving on past palindromes, where
 * the reference's loop would never terminate) is present.                                      */
extern "C" int hm_scan_examine(hm_scan *s, int ethresh, int *trim, int *symm)
{ /* the table as views: a replica is one view of the whole table on d[0]; a sharded table has one per
   * shard, view v holding table indices [lo[v], hi[v]) at local index 0                              */
  int       nv = s->sharded ? s->ngpu : 1;
  int64_t   vlo[HM_MAX_GPUS], vhi[HM_MAX_GPUS];
  int64_t   n = s->n, frst, last;
  int       h_min = 0x8000, *d_min = NULL;
  uint64_t *d_q = NULL;
  int64_t  *d_pos = NULL;
  int       two = (s->kmer > 32), rc = HM_OK;
  if (s->invalid && s->sharded)
    return hm_set_error(HM_EINVAL,"this scan was left unusable by a failed conditioning");
  for (int v = 0; v < nv; v++)
    { vlo[v] = s->sharded ? s->d[v].lo : 0; vhi[v] = s->sharded ? s->d[v].hi : n; }

  if (n+3 < 100000000) { frst = 0; last = n; }
  else { frst = n/2-50000000; last = n/2+50000000; }
  for (int v = 0; v < nv && rc == HM_OK; v++)            /* min over the middle entries = min of the views' minima */
    { DevTable *D = s->d+v;
      int64_t   a = frst > vlo[v] ? frst : vlo[v], b = last < vhi[v] ? last : vhi[v];
      int       vmin = 0x8000;
      if (a >= b) continue;
      HM_CUDA(cudaSetDevice(D->dev));
      HM_CUDA(cudaMalloc(&d_min,sizeof(int)));
      HM_CUDA(cudaMemcpyAsync(d_min,&vmin,sizeof(int),cudaMemcpyHostToDevice,D->st));
      rc = hm_k_min_count(D->cnt,a-vlo[v],b-vlo[v],d_min,D->st);
      s->launches += 1;
      if (rc == HM_OK)
        { cudaError_t e = cudaMemcpyAsync(&vmin,d_min,sizeof(int),cudaMemcpyDeviceToHost,D->st);
          if (e == cudaSuccess) e = cudaStreamSynchronize(D->st);
          if (e != cudaSuccess) rc = hm_cuda_fail(e,"min_count");
        }
      cudaFree(d_min);
      if (vmin < h_min) h_min = vmin;
    }
  if (rc != HM_OK)
    return rc;
  *trim = (h_min >= ethresh);

  /* entry sidx from the view that holds it, its reverse complement looked up by key (in whichever
   * view has it: the key ranges of the views do not overlap)                                    */
  *symm = 1;
  for (int64_t sidx = 1; sidx < n && rc == HM_OK; sidx++)
    { uint64_t x, xw = 0, q[2];
      int64_t  pos = -1;
      int      u = 0;
      while (u+1 < nv && sidx >= vhi[u]) u++;
      DevTable *D = s->d+u;
      HM_CUDA(cudaSetDevice(D->dev));
      cudaError_t e = cudaMemcpyAsync(&x,D->keys+(sidx-vlo[u]),sizeof(uint64_t),cudaMemcpyDeviceToHost,D->st);
      if (e == cudaSuccess && two)
        e = cudaMemcpyAsync(&xw,D->keys_lo+(sidx-vlo[u]),sizeof(uint64_t),cudaMemcpyDeviceToHost,D->st);
      if (e == cudaSuccess) e = cudaStreamSynchronize(D->st);
      if (e != cudaSuccess) { rc = hm_cuda_fail(e,"examine: key fetch"); break; }
      if (two) revcomp128(x,xw,s->kmer,q,q+1);
      else     { q[0] = revcomp64(x,s->kmer); q[1] = 0; }
      for (int v = 0; v < nv && rc == HM_OK && pos < 0; v++)
        { DevTable *V = s->d+v;
          int64_t   p = -1;
          if (vhi[v] <= vlo[v]) continue;
          HM_CUDA(cudaSetDevice(V->dev));
          HM_CUDA(cudaMalloc(&d_q,2*sizeof(uint64_t)));
          HM_CUDA(cudaMalloc(&d_pos,sizeof(int64_t)));
          cudaMemcpyAsync(d_q,q,2*sizeof(uint64_t),cudaMemcpyHostToDevice,V->st);
          rc = hm_k_find_keys(V->keys,V->keys_lo,vhi[v]-vlo[v],V->bucket,s->bits,s->idx64,d_q,two ? d_q+1 : NULL,1,d_pos,V->st);
          s->launches += 1;
          if (rc == HM_OK)
            { e = cudaMemcpyAsync(&p,d_pos,sizeof(int64_t),cudaMemcpyDeviceToHost,V->st);
              if (e == cudaSuccess) e = cudaStreamSynchronize(V->st);
              if (e != cudaSuccess) rc = hm_cuda_fail(e,"examine: lookup");
            }
          cudaFree(d_q); cudaFree(d_pos);
          if (p >= 0) pos = vlo[v]+p;
        }
      if (rc != HM_OK) break;
      if (pos < 0) { *symm = 0; break; }
      if (pos != sidx) { *symm = 1; break; }
    }
  return rc;
}

/* the direct passes of hm_kernels.cu: any table */
static int run_direct(hm_scan *s, int64_t *plot, hm_scan_stats *stats)
{ int         G = s->ngpu, rc = HM_OK;
  int64_t     n = s->n, launches0 = s->launches;
  if ((rc = ensure_direct(s)) != HM_OK)
    return rc;
  double      t0 = now_ms();
  cudaEvent_t ev[HM_MAX_GPUS][4];
  float       ms1 = 0, ms2 = 0, msall = 0;

  /* several GPUs: foreign incidence bytes are reached through the owner's array (remote atomics
   * in pass 1, remote loads in pass 2) when every pair of GPUs has native NVLink atomics; otherwise
   * the partial arrays are summed by the peer-memory kernel of hm_peer.cu                        */
  int        peer_mode = (G > 1);
  hm_shards *sh = s->sh;
  for (int a = 0; a < G && peer_mode; a++)
    for (int b = a+1; b < G && peer_mode; b++)
      if (!hm_p2p_native_atomics(s->d[a].dev,s->d[b].dev))
        peer_mode = 0;
  if (getenv("HETMERS_DENSE_EXCHANGE") != NULL)
    peer_mode = 0;
  if (peer_mode)
    for (int g = 0; g < G; g++)
      { memset(&sh[g],0,sizeof(hm_shards));
        sh[g].n_shards = G; sh[g].self = g;
        for (int r = 0; r < G; r++)
          { sh[g].off[r] = s->d[r].lo; sh[g].deg[r] = s->d[r].deg; }
        sh[g].off[G] = n;
        DevTable *D = s->d+g;
        int64_t need = hm_pass2_scratch_bytes(D->hi-D->lo,s->idx64);
        if (D->p2scratch == NULL || D->p2scratch_bytes < need)
          { HM_CUDA(cudaSetDevice(D->dev));
            if (D->p2scratch) cudaFree(D->p2scratch);
            HM_CUDA(cudaMalloc(&D->p2scratch,(size_t) need));
            D->p2scratch_bytes = need;
          }
        sh[g].scratch = D->p2scratch; sh[g].scratch_bytes = D->p2scratch_bytes;
      }

  for (int g = 0; g < G; g++)
    { DevTable *D = s->d+g;
      HM_CUDA(cudaSetDevice(D->dev));
      for (int k = 0; k < 4; k++)
        HM_CUDA(cudaEventCreate(&ev[g][k]));
      HM_CUDA(cudaEventRecord(ev[g][0],D->st));
      HM_CUDA(cudaMemsetAsync(D->deg,0,(size_t) ((n+4)&~3ll),D->st));
      HM_CUDA(cudaMemsetAsync(D->plot,0,sizeof(unsigned long long)*HM_PLOT_CELLS,D->st));
    }
  if (peer_mode)                                /* nobody adds to a peer before it has been zeroed */
    for (int g = 0; g < G; g++)
      { HM_CUDA(cudaSetDevice(s->d[g].dev)); HM_CUDA(cudaStreamSynchronize(s->d[g].st)); }
  for (int g = 0; g < G; g++)
    { DevTable *D = s->d+g;
      HM_CUDA(cudaSetDevice(D->dev));
      rc = hm_k_pass1_degree(D->keys,D->keys_lo,D->cnt,n,D->bucket,s->bits,s->idx64,D->filter,s->fpos,s->kmer,
                             D->lo,D->hi,D->deg,D->up,peer_mode ? &sh[g] : NULL,D->st);
      if (rc != HM_OK) return rc;
      s->launches += (D->hi > D->lo);
      HM_CUDA(cudaEventRecord(ev[g][1],D->st));
    }
  if (G > 1 && !peer_mode)
    { uint8_t *deg[HM_MAX_GPUS]; int64_t lo[HM_MAX_GPUS], hi[HM_MAX_GPUS];
      int dev[HM_MAX_GPUS]; cudaStream_t st[HM_MAX_GPUS];
      for (int g = 0; g < G; g++)
        { deg[g] = s->d[g].deg; lo[g] = s->d[g].lo; hi[g] = s->d[g].hi;
          dev[g] = s->d[g].dev; st[g] = s->d[g].st;
        }
      rc = hm_peer_sum_deg(deg,lo,hi,dev,st,G,n);
      if (rc != HM_OK) return rc;
      s->launches += G;
    }
  if (peer_mode)                                /* every pass 1 (and its remote atomics) has landed */
    for (int g = 0; g < G; g++)
      { HM_CUDA(cudaSetDevice(s->d[g].dev)); HM_CUDA(cudaStreamSynchronize(s->d[g].st)); }
  for (int g = 0; g < G; g++)
    { DevTable *D = s->d+g;
      HM_CUDA(cudaSetDevice(D->dev));
      HM_CUDA(cudaEventRecord(ev[g][2],D->st));
      rc = hm_k_pass2_plot(D->cnt,D->deg,D->up,s->idx64,D->lo,D->hi,D->plot,
                           peer_mode ? &sh[g] : NULL,D->st);
      if (rc != HM_OK) return rc;
      s->launches += (D->hi > D->lo);
      HM_CUDA(cudaEventRecord(ev[g][3],D->st));
    }
  if (G > 1)
    { unsigned long long *pl[HM_MAX_GPUS]; int dev[HM_MAX_GPUS]; cudaStream_t st[HM_MAX_GPUS];
      for (int g = 0; g < G; g++)
        { pl[g] = s->d[g].plot; dev[g] = s->d[g].dev; st[g] = s->d[g].st; }
      rc = hm_peer_sum_plot(pl,dev,st,G);
      if (rc != HM_OK) return rc;
      s->launches += 1;
    }
  HM_CUDA(cudaSetDevice(s->d[0].dev));
  HM_CUDA(cudaMemcpyAsync(plot,s->d[0].plot,sizeof(int64_t)*HM_PLOT_CELLS,
                          cudaMemcpyDeviceToHost,s->d[0].st));
  for (int g = 0; g < G; g++)
    { HM_CUDA(cudaSetDevice(s->d[g].dev));
      HM_CUDA(cudaStreamSynchronize(s->d[g].st));
    }
  double t1 = now_ms();
  for (int g = 0; g < G; g++)
    { float a = 0, b = 0, c = 0;
      cudaSetDevice(s->d[g].dev);
      cudaEventElapsedTime(&a,ev[g][0],ev[g][1]);
      cudaEventElapsedTime(&b,ev[g][2],ev[g][3]);
      cudaEventElapsedTime(&c,ev[g][0],ev[g][3]);
      if (a > ms1) ms1 = a;
      if (b > ms2) ms2 = b;
      if (c > msall) msall = c;
      for (int k = 0; k < 4; k++)
        cudaEventDestroy(ev[g][k]);
    }
  s->ran = 1; s->peer_mode = peer_mode; s->last_path = HM_PATH_DIRECT;
  if (stats != NULL)
    { stats->nels = n; stats->n_gpus = G; stats->bucket_bits = s->bits;
      stats->filter_bits = s->fpos; stats->path = HM_PATH_DIRECT;
      stats->ms_h2d_unpack = s->ms_load;
      stats->ms_pass1 = ms1; stats->ms_pass2 = ms2;
      stats->ms_scan = G > 1 ? (t1-t0) : msall;
      stats->ms_total = s->ms_load + (t1-t0);
      stats->kernel_launches = s->launches;
      stats->ms_alloc = s->ms_alloc; stats->ms_records = s->ms_records; stats->ms_index = s->ms_index;
    }
  (void) launches0;
  return HM_OK;
}

/* the strand-symmetric scan of hm_symm.cu: run scan -> (Bloom segments all-gathered over peer
 * copies when >1 GPU) -> resolve -> plot reduce.  *status = the OR of the devices' status words:
 * non-zero means the table was not symmetric after all and the plot must not be used.           */
static int run_symm(hm_scan *s, int64_t *plot, hm_scan_stats *stats, uint64_t *status)
{ int         G = s->ngpu, rc = HM_OK;
  int64_t     n = s->n;
  cudaEvent_t ev[HM_MAX_GPUS][4];
  float       ms1 = 0, ms2 = 0, msall = 0;
  if ((rc = ensure_symm(s)) != HM_OK)
    return rc;
  s->symm_ran = 0;
  hm_shard_tabs tabs;                           /* sharded: pass 2 settles Bloom hits in the owner's arrays */
  memset(&tabs,0,sizeof(tabs));
  for (int g = 0; g < G && s->sharded; g++)
    { tabs.keys[g] = s->d[g].keys; tabs.keys_lo[g] = s->d[g].keys_lo; tabs.cnt[g] = s->d[g].cnt;
      tabs.bucket[g] = s->d[g].bucket; tabs.n[g] = s->d[g].hi-s->d[g].lo;
    }
  double      t0 = now_ms();
  for (int g = 0; g < G; g++)
    { DevTable *D = s->d+g;
      HM_CUDA(cudaSetDevice(D->dev));
      for (int k = 0; k < 4; k++)
        HM_CUDA(cudaEventCreate(&ev[g][k]));
      HM_CUDA(cudaEventRecord(ev[g][0],D->st));
      HM_CUDA(cudaMemsetAsync(D->plot,0,sizeof(unsigned long long)*HM_PLOT_CELLS,D->st));
      int64_t na = s->sharded ? D->hi-D->lo : n;         /* entries in this device's arrays */
      rc = hm_k_symm_runscan(D->keys,D->keys_lo,D->cnt,na,D->bucket,s->bits,s->idx64,s->kmer,D->slo,D->shi,
                             D->symm_work,&D->symm_layout,G > 1 ? &s->ssh[g] : NULL,D->st);
      if (rc == HM_OK)
        rc = hm_k_symm_runs(D->keys,D->keys_lo,D->cnt,na,D->bucket,s->bits,s->idx64,s->kmer,D->slo,D->shi,
                            D->symm_work,&D->symm_layout,G > 1 ? &s->ssh[g] : NULL,D->st);
      if (rc != HM_OK) return rc;
      s->launches += 2*(D->shi > D->slo);
      HM_CUDA(cudaEventRecord(ev[g][1],D->st));
    }
  if (G > 1)                                    /* every device pulls the other devices' Bloom segments */
    { for (int g = 0; g < G; g++)
        { HM_CUDA(cudaSetDevice(s->d[g].dev)); HM_CUDA(cudaStreamSynchronize(s->d[g].st)); }
      for (int g = 0; g < G; g++)
        { DevTable *D = s->d+g;
          size_t    segb = sizeof(uint32_t)*(size_t) D->symm_layout.seg_words;
          HM_CUDA(cudaSetDevice(D->dev));
          for (int h = 0; h < G; h++)
            if (h != g)
              { DevTable *S = s->d+h;
                HM_CUDA(cudaMemcpyPeerAsync((uint8_t *) D->symm_work + D->symm_layout.off_bloom + segb*h,D->dev,
                                            (uint8_t *) S->symm_work + S->symm_layout.off_bloom + segb*h,S->dev,
                                            segb,D->st));
              }
        }
    }
  for (int g = 0; g < G; g++)
    { DevTable *D = s->d+g;
      HM_CUDA(cudaSetDevice(D->dev));
      HM_CUDA(cudaEventRecord(ev[g][2],D->st));
      if (s->sharded)
        rc = hm_symm_resolve_sharded(&tabs,s->bits,s->idx64,s->kmer,D->symm_work,&D->symm_layout,
                                     G > 1 ? &s->ssh[g] : NULL,D->plot,D->st);
      else
        rc = hm_k_symm_resolve(D->keys,D->keys_lo,D->cnt,n,D->bucket,s->bits,s->idx64,s->kmer,
                               D->symm_work,&D->symm_layout,G > 1 ? &s->ssh[g] : NULL,D->plot,D->st);
      if (rc != HM_OK) return rc;
      s->launches += 1;
      HM_CUDA(cudaEventRecord(ev[g][3],D->st));
    }
  if (G > 1)
    { unsigned long long *pl[HM_MAX_GPUS]; int dev[HM_MAX_GPUS]; cudaStream_t st[HM_MAX_GPUS];
      for (int g = 0; g < G; g++)
        { pl[g] = s->d[g].plot; dev[g] = s->d[g].dev; st[g] = s->d[g].st; }
      rc = hm_peer_sum_plot(pl,dev,st,G);
      if (rc != HM_OK) return rc;
      s->launches += 1;
    }
  uint64_t hdr[HM_MAX_GPUS][2];
  HM_CUDA(cudaSetDevice(s->d[0].dev));
  HM_CUDA(cudaMemcpyAsync(plot,s->d[0].plot,sizeof(int64_t)*HM_PLOT_CELLS,
                          cudaMemcpyDeviceToHost,s->d[0].st));
  for (int g = 0; g < G; g++)
    { DevTable *D = s->d+g;
      HM_CUDA(cudaSetDevice(D->dev));
      HM_CUDA(cudaMemcpyAsync(hdr[g],(uint8_t *) D->symm_work + D->symm_layout.off_header,2*sizeof(uint64_t),
                              cudaMemcpyDeviceToHost,D->st));
    }
  for (int g = 0; g < G; g++)
    { HM_CUDA(cudaSetDevice(s->d[g].dev));
      HM_CUDA(cudaStreamSynchronize(s->d[g].st));
    }
  double t1 = now_ms();
  *status = 0;
  for (int g = 0; g < G; g++)
    { float a = 0, b = 0, c = 0;
      *status |= hdr[g][1];
      cudaSetDevice(s->d[g].dev);
      cudaEventElapsedTime(&a,ev[g][0],ev[g][1]);
      cudaEventElapsedTime(&b,ev[g][2],ev[g][3]);
      cudaEventElapsedTime(&c,ev[g][0],ev[g][3]);
      if (a > ms1) ms1 = a;
      if (b > ms2) ms2 = b;
      if (c > msall) msall = c;
      for (int k = 0; k < 4; k++)
        cudaEventDestroy(ev[g][k]);
    }
  s->last_path = HM_PATH_SYMM;
  s->symm_ran  = (*status == 0);
  if (stats != NULL)
    { stats->nels = n; stats->n_gpus = G; stats->bucket_bits = s->bits;
      stats->filter_bits = 0; stats->path = HM_PATH_SYMM;
      stats->ms_h2d_unpack = s->ms_load;
      stats->ms_pass1 = ms1; stats->ms_pass2 = ms2;
      stats->ms_scan = G > 1 ? (t1-t0) : msall;
      stats->ms_total = s->ms_load + (t1-t0);
      stats->kernel_launches = s->launches;
      stats->ms_alloc = s->ms_alloc; stats->ms_records = s->ms_records; stats->ms_index = s->ms_index;
    }
  return HM_OK;
}

extern "C" int hm_scan_is_symmetric(const hm_scan *s) { return s->symmetric; }

extern "C" int hm_scan_run_path(hm_scan *s, int path, int64_t *plot, hm_scan_stats *stats)
{ if (s->invalid)
    return hm_set_error(HM_EINVAL,"this scan was left unusable by a failed conditioning");
  if (s->sharded)
    { if (path == HM_PATH_DIRECT)
        return hm_set_error(HM_EUNSUPPORTED,"a sharded table has only the strand-symmetric scan (the direct "
                                            "passes need the whole table on every GPU)");
      if (path != HM_PATH_AUTO && path != HM_PATH_SYMM)
        return hm_set_error(HM_EINVAL,"hm_scan_run_path: unknown path %d",path);
      int rc;
      if (!s->aligned && (rc = ensure_symm(s)) != HM_OK)     /* the verdict is taken on the aligned shards */
        return rc;
      if (!s->symmetric)
        return hm_set_error(HM_EUNSUPPORTED,"the table is not strand-symmetric: a sharded table can only be "
                                            "scanned after conditioning (hm_scan_condition)");
      uint64_t status = 0;
      if ((rc = run_symm(s,plot,stats,&status)) != HM_OK)
        return rc;
      if (status != 0)
        return hm_set_error(HM_EUNSUPPORTED,"symmetric scan of a sharded table failed its own checks (status %llu); "
                                            "the direct passes cannot stand in for it",(unsigned long long) status);
      return HM_OK;
    }
  if (path == HM_PATH_AUTO)
    { const char *e = getenv("HETMERS_PATH");
      if (e != NULL && strcmp(e,"direct") == 0) path = HM_PATH_DIRECT;
      if (e != NULL && strcmp(e,"symm") == 0)   path = HM_PATH_SYMM;
    }
  if (path == HM_PATH_DIRECT || (path == HM_PATH_AUTO && !s->symmetric))
    return run_direct(s,plot,stats);
  if (path != HM_PATH_AUTO && path != HM_PATH_SYMM)
    return hm_set_error(HM_EINVAL,"hm_scan_run_path: unknown path %d",path);
  if (s->kmer < HM_SYMM_MIN_KMER || (path == HM_PATH_SYMM && !s->symmetric))
    return hm_set_error(HM_EINVAL,"the table is not strand-symmetric (or k < %d): the symmetric scan "
                                  "would not give the reference's answer",HM_SYMM_MIN_KMER);
  uint64_t status = 0;
  int rc = run_symm(s,plot,stats,&status);
  if (rc != HM_OK)
    return rc;
  if (status == 0)
    return HM_OK;
  /* the fingerprint was fooled (2^-128) or a cut missed a run boundary: the direct passes are
   * always right                                                                                */
  if (path == HM_PATH_SYMM)
    return hm_set_error(HM_EINVAL,"symmetric scan failed its own checks (status %llu)",(unsigned long long) status);
  s->symmetric = 0;
  return run_direct(s,plot,stats);
}

extern "C" int hm_scan_run(hm_scan *s, int64_t *plot, hm_scan_stats *stats)
{ return hm_scan_run_path(s,HM_PATH_AUTO,plot,stats); }

/* extract / download need the incidence array and the recorded partners of the direct passes */
static int need_direct_results(hm_scan *s)
{ if (s->ran)
    return HM_OK;
  int64_t *tmp = (int64_t *) malloc(sizeof(int64_t)*HM_PLOT_CELLS);
  if (tmp == NULL)
    return hm_set_error(HM_ENOMEM,"out of host memory");
  int rc = run_direct(s,tmp,NULL);
  free(tmp);
  return rc;
}

static int rec_cmp(const void *a, const void *b)
{ const hm_pair_rec *x = (const hm_pair_rec *) a, *y = (const hm_pair_rec *) b;
  if (x->smudge != y->smudge) return (x->smudge < y->smudge ? -1 : 1);
  if (x->key_hi != y->key_hi) return (x->key_hi < y->key_hi ? -1 : 1);
  if (x->key_lo != y->key_lo) return (x->key_lo < y->key_lo ? -1 : 1);
  if (x->pos != y->pos)       return (x->pos < y->pos ? -1 : 1);
  return ((int) x->alt - (int) y->alt);
}

/* extract_kmer_pairs' output as a list (PloidyList.c:425-450) from the direct passes: needs the
 * incidence array and the recorded partners (runs the direct passes first if the last run did not).
 * Two launches per GPU: count, then fill.                                                        */
static int extract_direct(hm_scan *s, const uint16_t *pixmap, hm_pair_rec **out, int64_t *n_out,
                          hm_extract_stats *stats)
{ int G = s->ngpu, rc = HM_OK;
  if (s->invalid)
    return hm_set_error(HM_EINVAL,"this scan was left unusable by a failed conditioning");
  if (s->sharded)
    return hm_set_error(HM_EUNSUPPORTED,"extract_kmer_pairs needs the direct passes, which a sharded table does not have");
  if ((rc = need_direct_results(s)) != HM_OK)
    return rc;
  double       t0 = now_ms(), t1, t2;
  int64_t      total = 0, cnts[HM_MAX_GPUS];
  hm_pair_rec *d_out[HM_MAX_GPUS];
  uint16_t    *d_pix[HM_MAX_GPUS];
  unsigned long long *d_cnt[HM_MAX_GPUS];
  memset(d_out,0,sizeof(d_out)); memset(d_pix,0,sizeof(d_pix)); memset(d_cnt,0,sizeof(d_cnt));
  for (int pass = 0; pass < 2 && rc == HM_OK; pass++)
    { for (int g = 0; g < G && rc == HM_OK; g++)
        { DevTable *D = s->d+g;
          HM_CUDA(cudaSetDevice(D->dev));
          if (pass == 0)
            { HM_CUDA(cudaMalloc(&d_pix[g],sizeof(uint16_t)*HM_PLOT_CELLS));
              HM_CUDA(cudaMalloc(&d_cnt[g],sizeof(unsigned long long)));
              HM_CUDA(cudaMemcpyAsync(d_pix[g],pixmap,sizeof(uint16_t)*HM_PLOT_CELLS,cudaMemcpyHostToDevice,D->st));
            }
          else if (cnts[g] > 0)
            HM_CUDA(cudaMalloc(&d_out[g],sizeof(hm_pair_rec)*(size_t) cnts[g]));
          HM_CUDA(cudaMemsetAsync(d_cnt[g],0,sizeof(unsigned long long),D->st));
          rc = hm_k_pass2_extract(D->keys,D->keys_lo,D->cnt,D->deg,D->up,s->idx64,D->lo,D->hi,d_pix[g],
                                  d_out[g],pass == 0 ? 0 : cnts[g],d_cnt[g],s->peer_mode ? &s->sh[g] : NULL,D->st);
          s->launches += (D->hi > D->lo);
        }
      for (int g = 0; g < G && rc == HM_OK; g++)
        { unsigned long long c = 0;
          HM_CUDA(cudaSetDevice(s->d[g].dev));
          HM_CUDA(cudaMemcpyAsync(&c,d_cnt[g],sizeof(c),cudaMemcpyDeviceToHost,s->d[g].st));
          HM_CUDA(cudaStreamSynchronize(s->d[g].st));
          if (pass == 0) { cnts[g] = (int64_t) c; total += cnts[g]; }
        }
    }
  t1 = now_ms();
  hm_pair_rec *host = (hm_pair_rec *) malloc(sizeof(hm_pair_rec)*(size_t) (total > 0 ? total : 1));
  if (host == NULL && rc == HM_OK)
    rc = hm_set_error(HM_ENOMEM,"out of host memory for %lld pair records",(long long) total);
  int64_t at = 0;
  for (int g = 0; g < G; g++)
    { cudaSetDevice(s->d[g].dev);
      if (rc == HM_OK && cnts[g] > 0)
        { cudaError_t e = cudaMemcpy(host+at,d_out[g],sizeof(hm_pair_rec)*(size_t) cnts[g],cudaMemcpyDeviceToHost);
          if (e != cudaSuccess) rc = hm_cuda_fail(e,"cudaMemcpy(pair records)");
          at += cnts[g];
        }
      if (d_out[g]) cudaFree(d_out[g]);
      if (d_pix[g]) cudaFree(d_pix[g]);
      if (d_cnt[g]) cudaFree(d_cnt[g]);
    }
  if (rc != HM_OK)
    { free(host); return rc; }
  t2 = now_ms();
  qsort(host,(size_t) total,sizeof(hm_pair_rec),rec_cmp);      /* deterministic order */
  *out = host; *n_out = total;
  if (stats != NULL)
    { stats->path = HM_PATH_DIRECT; stats->slices = 1; stats->n_records = total;
      stats->ms_kernel = t1-t0; stats->ms_copy = t2-t1; stats->ms_sort = now_ms()-t2;
    }
  return HM_OK;
}

extern "C" int hm_scan_extract(hm_scan *s, const uint16_t *pixmap, hm_pair_rec **out, int64_t *n_out)
{ return extract_direct(s,pixmap,out,n_out,NULL); }

/* extract_kmer_pairs from the candidates and Bloom segments the symmetric scan left in the work areas
 * (scanning first if they are not those of a clean scan of the current table).  Every device judges
 * its own candidates again -- a replica against its replica, a shard with ShardTabs reaching the other
 * shards -- in slices whose records fit the idle run-head region of its work area; each slice is
 * copied to the host as it finishes.  The label map goes into the device's plot buffer (the plot of
 * the last run is on the host already), so nothing is allocated on the device.                      */
static int extract_symm(hm_scan *s, const uint16_t *pixmap, hm_pair_rec **out, int64_t *n_out,
                        hm_extract_stats *stats)
{ int G = s->ngpu, rc = HM_OK;
  if (!s->sharded && (s->kmer < HM_SYMM_MIN_KMER || !s->symmetric))
    return hm_set_error(HM_EINVAL,"the table is not strand-symmetric (or k < %d): extraction from the symmetric "
                                  "scan would not give the reference's pairs",HM_SYMM_MIN_KMER);
  if (!s->symm_ran)
    { int64_t *tmp = (int64_t *) malloc(sizeof(int64_t)*HM_PLOT_CELLS);
      if (tmp == NULL)
        return hm_set_error(HM_ENOMEM,"out of host memory");
      rc = hm_scan_run_path(s,HM_PATH_SYMM,tmp,NULL);
      free(tmp);
      if (rc != HM_OK)
        return rc;
      if (!s->symm_ran)
        return hm_set_error(HM_EINVAL,"the symmetric scan did not leave its candidates for extraction");
    }
  hm_shard_tabs tabs;
  memset(&tabs,0,sizeof(tabs));
  for (int g = 0; g < G && s->sharded; g++)
    { tabs.keys[g] = s->d[g].keys; tabs.keys_lo[g] = s->d[g].keys_lo; tabs.cnt[g] = s->d[g].cnt;
      tabs.bucket[g] = s->d[g].bucket; tabs.n[g] = s->d[g].hi-s->d[g].lo;
    }
  int64_t  nc[HM_MAX_GPUS], cur[HM_MAX_GPUS], slice[HM_MAX_GPUS];
  float    ms_k[HM_MAX_GPUS];
  cudaEvent_t ev[HM_MAX_GPUS][2];
  uint16_t *d_pix[HM_MAX_GPUS];
  for (int g = 0; g < G; g++)
    { DevTable *D = s->d+g;
      uint64_t  n_cand = 0, st = 0;
      HM_CUDA(cudaSetDevice(D->dev));
      HM_CUDA(cudaEventCreate(&ev[g][0]));
      HM_CUDA(cudaEventCreate(&ev[g][1]));
      d_pix[g] = (uint16_t *) D->plot;
      HM_CUDA(cudaMemcpyAsync(d_pix[g],pixmap,sizeof(uint16_t)*HM_PLOT_CELLS,cudaMemcpyHostToDevice,D->st));
      if ((rc = hm_symm_status(D->symm_work,&D->symm_layout,&n_cand,&st,D->st)) != HM_OK)
        return rc;
      nc[g] = (int64_t) n_cand < D->symm_layout.cand_cap ? (int64_t) n_cand : D->symm_layout.cand_cap;
      cur[g] = 0; ms_k[g] = 0;
      slice[g] = hm_symm_extract_slice(&D->symm_layout);
    }
  double       t_copy = 0;
  int64_t      at = 0, cap = 0;
  int          slices = 0;
  uint64_t     status = 0;
  hm_pair_rec *host = NULL;
  for (int more = 1; more && rc == HM_OK; )
    { more = 0;
      for (int g = 0; g < G && rc == HM_OK; g++)           /* one slice on every device that has candidates left */
        { DevTable *D = s->d+g;
          if (cur[g] >= nc[g]) continue;
          int64_t c1 = cur[g]+slice[g] < nc[g] ? cur[g]+slice[g] : nc[g];
          cudaSetDevice(D->dev);
          cudaEventRecord(ev[g][0],D->st);
          rc = hm_symm_extract(D->keys,D->keys_lo,D->cnt,s->sharded ? D->hi-D->lo : s->n,D->bucket,
                               s->sharded ? &tabs : NULL,s->bits,s->idx64,s->kmer,D->symm_work,&D->symm_layout,
                               G > 1 ? &s->ssh[g] : NULL,d_pix[g],cur[g],c1,D->st);
          cudaEventRecord(ev[g][1],D->st);
          s->launches += 1;
          slices += 1;
        }
      for (int g = 0; g < G && rc == HM_OK; g++)           /* ... and its records to the host */
        { DevTable *D = s->d+g;
          if (cur[g] >= nc[g]) continue;
          float    ms = 0;
          uint64_t st = 0;
          cudaSetDevice(D->dev);
          cudaError_t e = cudaEventSynchronize(ev[g][1]);
          if (e != cudaSuccess) { rc = hm_cuda_fail(e,"extract_kernel"); break; }
          cudaEventElapsedTime(&ms,ev[g][0],ev[g][1]);
          ms_k[g] += ms;
          double t = now_ms();
          rc = hm_symm_extract_fetch(D->symm_work,&D->symm_layout,&host,&cap,&at,&st,D->st);
          t_copy += now_ms()-t;
          status |= st;
          cur[g] += slice[g];
          if (cur[g] < nc[g]) more = 1;
        }
    }
  for (int g = 0; g < G; g++)
    { cudaSetDevice(s->d[g].dev);
      cudaEventDestroy(ev[g][0]); cudaEventDestroy(ev[g][1]);
    }
  if (rc == HM_OK && status != 0)
    { s->symm_ran = 0;                    /* judged again, a candidate came out differently: nothing is trusted */
      rc = hm_set_error(HM_EINVAL,"extraction from the symmetric scan failed its own checks (status %llu)",
                        (unsigned long long) status);
    }
  if (rc != HM_OK)
    { free(host); return rc; }
  if (host == NULL && (host = (hm_pair_rec *) malloc(sizeof(hm_pair_rec))) == NULL)
    return hm_set_error(HM_ENOMEM,"out of host memory");
  double t = now_ms();
  qsort(host,(size_t) at,sizeof(hm_pair_rec),rec_cmp);         /* the order of hm_scan_extract */
  *out = host; *n_out = at;
  if (stats != NULL)
    { float mk = 0;
      for (int g = 0; g < G; g++) if (ms_k[g] > mk) mk = ms_k[g];
      stats->path = HM_PATH_SYMM; stats->slices = slices; stats->n_records = at;
      stats->ms_kernel = mk; stats->ms_copy = t_copy; stats->ms_sort = now_ms()-t;
    }
  return HM_OK;
}

extern "C" int hm_scan_extract_path(hm_scan *s, int path, const uint16_t *pixmap, hm_pair_rec **out,
                                    int64_t *n_out, hm_extract_stats *stats)
{ if (s == NULL || pixmap == NULL || out == NULL || n_out == NULL)
    return hm_set_error(HM_EINVAL,"hm_scan_extract_path: bad arguments");
  if (s->invalid)
    return hm_set_error(HM_EINVAL,"this scan was left unusable by a failed conditioning");
  if (path != HM_PATH_AUTO && path != HM_PATH_DIRECT && path != HM_PATH_SYMM)
    return hm_set_error(HM_EINVAL,"hm_scan_extract_path: unknown path %d",path);
  if (stats != NULL)
    memset(stats,0,sizeof(*stats));
  if (path == HM_PATH_AUTO)                       /* the path hm_scan_run takes */
    { const char *e = getenv("HETMERS_PATH");
      if (s->sharded)                             path = HM_PATH_SYMM;
      else if (e != NULL && strcmp(e,"direct") == 0) path = HM_PATH_DIRECT;
      else if (e != NULL && strcmp(e,"symm") == 0)   path = HM_PATH_SYMM;
      else path = (s->symmetric && s->kmer >= HM_SYMM_MIN_KMER) ? HM_PATH_SYMM : HM_PATH_DIRECT;
    }
  if (path == HM_PATH_DIRECT)
    return extract_direct(s,pixmap,out,n_out,stats);
  return extract_symm(s,pixmap,out,n_out,stats);
}

extern "C" int hm_hetmers_host(const hm_host_table *t, const int *dev, int n_gpus,
                               int64_t *plot, hm_scan_stats *stats)
{ hm_scan *s = NULL;
  int rc = hm_scan_create(t,dev,n_gpus,&s);
  if (rc != HM_OK)
    return rc;
  rc = hm_scan_run(s,plot,stats);
  hm_scan_destroy(s);
  return rc;
}

extern "C" int hm_scan_download(hm_scan *s, uint64_t *keys, uint64_t *keys_lo, uint16_t *cnt, uint8_t *deg)
{ if (s->sharded)                       /* the concatenation of the shards */
    { if (deg != NULL)
        return hm_set_error(HM_EUNSUPPORTED,"a sharded table has no incidence array (pass deg = NULL)");
      if (s->invalid)
        return hm_set_error(HM_EINVAL,"this scan was left unusable by a failed conditioning");
      for (int g = 0; g < s->ngpu; g++)
        { DevTable *O = s->d+g;
          size_t    m = (size_t) (O->hi-O->lo);
          if (m == 0) continue;
          HM_CUDA(cudaSetDevice(O->dev));
          HM_CUDA(cudaStreamSynchronize(O->st));
          if (keys != NULL)    HM_CUDA(cudaMemcpy(keys+O->lo,O->keys,sizeof(uint64_t)*m,cudaMemcpyDeviceToHost));
          if (keys_lo != NULL && O->keys_lo != NULL)
                               HM_CUDA(cudaMemcpy(keys_lo+O->lo,O->keys_lo,sizeof(uint64_t)*m,cudaMemcpyDeviceToHost));
          if (cnt != NULL)     HM_CUDA(cudaMemcpy(cnt+O->lo,O->cnt,sizeof(uint16_t)*m,cudaMemcpyDeviceToHost));
        }
      return HM_OK;
    }
  DevTable *D = s->d;
  HM_CUDA(cudaSetDevice(D->dev));
  HM_CUDA(cudaStreamSynchronize(D->st));
  if (keys != NULL)
    HM_CUDA(cudaMemcpy(keys,D->keys,sizeof(uint64_t)*(size_t) s->n,cudaMemcpyDeviceToHost));
  if (keys_lo != NULL && D->keys_lo != NULL)
    HM_CUDA(cudaMemcpy(keys_lo,D->keys_lo,sizeof(uint64_t)*(size_t) s->n,cudaMemcpyDeviceToHost));
  if (cnt != NULL)
    HM_CUDA(cudaMemcpy(cnt,D->cnt,sizeof(uint16_t)*(size_t) s->n,cudaMemcpyDeviceToHost));
  if (deg != NULL)                      /* every owner's slice (identical copies in dense mode) */
    { int rc = need_direct_results(s);  /* (the symmetric scan never materialises the array) */
      if (rc != HM_OK) return rc;
    }
  if (deg != NULL)
    for (int g = 0; g < s->ngpu; g++)
      { DevTable *O = s->d+g;
        HM_CUDA(cudaSetDevice(O->dev));
        HM_CUDA(cudaStreamSynchronize(O->st));
        if (O->hi > O->lo)
          HM_CUDA(cudaMemcpy(deg+O->lo,O->deg+O->lo,(size_t) (O->hi-O->lo),cudaMemcpyDeviceToHost));
      }
  return HM_OK;
}
