/*******************************************************************************************
 * hm_symm.cu -- the strand-symmetric scan: every table entry is read ONCE.
 *
 * The reference insists on a table that holds the reverse complement of each of its k-mers with
 * the same count (examine_table, PloidyPlot.c:1199-1229; it runs `Symmex` otherwise, :1401-1414),
 * but then searches all k positions directly.  On a table that really is symmetric the pairs that
 * differ at a LOW position p < Pr = k/2 are the mirror images (u,v) -> (rc v, rc u) of the pairs
 * that differ at the HIGH position k-1-p, and pairs at high positions sit next to each other in the
 * sorted table: both members share their first Pr bases, i.e. lie in one short *run* of entries.
 * So with N_p(x) = number of partners of x at position p (count sum <= SMAX, PloidyPlot.c:259):
 *
 *     deg(x) = H(x) + U(rc x),   H(x) = sum_{p >= Pr}   N_p(x)     (found inside x's run)
 *                                U(x) = sum_{p >= k-Pr} N_p(x)     (ditto; = H without the middle
 *                                                                   base of an odd k)
 *     deg(rc x) = deg(x), and a pair and its mirror image land in the same plot cell.
 *
 *   symm_fingerprint_kernel   is the table symmetric?  Keyed multiset fingerprints of
 *                             {(x,cnt)} and {(rc x,cnt)} (seeds drawn per process); equal sums
 *                             <=> equal multisets up to a 2^-128 chance.  Tables that fail --
 *                             they may still pass the reference's one-k-mer probe -- take the
 *                             direct search of hm_kernels.cu, so the answer is the reference's
 *                             either way.
 *   runscan_kernel            ("pass 1") tiles of the sorted table are staged into shared memory by
 *                             TMA bulk copies; entries are classified by the adjacency of their
 *                             runs, runs of two are settled by one comparison (H, U, the partner).
 *                             Entries with U > 0 (the set S) are added to a Bloom filter; pairs
 *                             (x < y) with H(x) = H(y) = 1 become candidate records.
 *   runs_kernel               the runs of three or more entries that runscan_kernel only lists
 *   runscan_dense_kernel      pass 1 for crowded tables (many run mates per entry): all pairs of
 *                             every run, counted with shared-memory atomics
 *   resolve_kernel            ("pass 2") a candidate is an isolated pair iff neither rc x nor rc y
 *                             is in S: Bloom look-up (L2 resident), hits confirmed exactly by
 *                             scanning the run of rc x in the table.  Isolated pairs are counted
 *                             into the plot (shared-memory tile + 64-bit atomics), twice when the
 *                             mirror image is a different pair (PloidyPlot.c:401-415 sees both).
 *
 * Replaces analysis_in_core_1/_2 + the recursion around them (PloidyPlot.c:454-700,:851-1084)
 * for symmetric tables.  Traffic: keys + counts once (TBYTE per entry) + ~2 B per entry of
 * candidate records, instead of 2 x k merge levels in the reference.
 *******************************************************************************************/
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <type_traits>

#include "hetmers_b200.h"
#include "hm_internal.h"
#include "hm_device.cuh"

#define RS_THREADS 256
#define RS_EPT     8
#define RS_TILE    (RS_THREADS*RS_EPT)        /* entries per CTA tile                            */
#define RS_HALO    64                          /* entries staged on either side of the tile      */
#define RS_WIN     (RS_TILE+2*RS_HALO)
#define RS_SCANCAP RS_HALO                     /* longest run half scanned linearly               */
#define RS_LONGRUN 32                          /* dense kernel: runs of more entries go to runs_kernel */
#ifndef RS_MINBLOCKS
#define RS_MINBLOCKS 6                         /* resident CTAs per SM the register budget must allow (40 regs;
                                                *   4: 1.18 ms, 5: 1.07, 6 with 30 KB of shared memory: 0.99)     */
#endif
#ifndef RS_STAGE
#define RS_STAGE   384                         /* candidate records staged per CTA before they leave (a 2048-entry
                                                *   tile of a diploid 1 % table holds 184 +- 14)                    */
#endif

#define SY_STATUS_ASYMMETRIC 1ull              /* a reverse complement was not in the table      */
#define SY_STATUS_OVERFLOW   2ull              /* candidate list full                             */

/* device view of the work area (hm_symm_layout) */
struct SymmView
  { unsigned long long *cand_n;
    unsigned long long *status;
    uint32_t *bloom;                            /* n_seg segments of seg_words words               */
    uint32_t  seg_words;
    int       n_seg, self;
    uint64_t  first_key[HM_MAX_SHARDS];         /* word 0 of the first key of segments 1.. (0 unused) */
    uint64_t *cand_key, *cand_lo, *cand_meta;
    unsigned long long cand_cap;
    unsigned long long *runs_n;                 /* heads of runs of three or more entries (table indices) */
    uint64_t *runs;
    unsigned long long runs_cap;
  };

/* Bloom slot of key (hi,lo).  The WORD is chosen by the key's last k/2 bases, the two BITS inside it by
 * the bases before them: rc x and rc y of a candidate pair differ at one base of the front part only, so
 * both of pass 2's look-ups for a pair fall into the same word -- one load (when one shard owns both). */
template <int KW>
__device__ __forceinline__ void bloom_slot(const SymmView &W, int seg, int kmer, uint64_t hi, uint64_t lo,
                                           uint32_t *&word, uint32_t &mask)
{ const int Pr = kmer >> 1, pup = kmer-Pr;
  uint64_t sfx;                                                /* the last Pr bases, right aligned */
  if (KW == 1)
    sfx = hi >> (64-2*kmer);
  else
    { const int sr = 128-2*kmer;                               /* 0..62 */
      sfx = sr == 0 ? lo : ((lo >> sr) | (hi << (64-sr)));
    }
  if (2*Pr < 64)
    sfx &= (((uint64_t) 1 << (2*Pr)) - 1);
  const uint64_t pfx = hi >> (64-2*pup);                       /* the first pup <= 32 bases */
  uint32_t h = ((uint32_t) sfx ^ (uint32_t) (sfx >> 32) * 0x85EBCA6Bu) * 0x9E3779B1u;     /* 32-bit mixing is plenty here */
  uint32_t g = ((uint32_t) pfx ^ (uint32_t) (pfx >> 32) * 0xC2B2AE35u) * 0x27D4EB2Fu;
  h ^= h >> 15;
  word = W.bloom + (size_t) seg * W.seg_words + __umulhi(h * 0x2C1B3C6Du,W.seg_words);
  mask = (1u << (g >> 27)) | (1u << ((g >> 22) & 31));
}

/* L2 residency: the Bloom segments (tens of MB) are what pass 2 hits at random, the candidate records
 * stream through once                                                                             */
__device__ __forceinline__ uint32_t ld_keep(const uint32_t *p)
{ uint32_t v; uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
  asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.u32 %0, [%1], %2;" : "=r"(v) : "l"(p), "l"(pol));
  return v;
}

__device__ __forceinline__ uint64_t ld_stream(const uint64_t *p)
{ uint64_t v, pol;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.u64 %0, [%1], %2;" : "=l"(v) : "l"(p), "l"(pol));
  return v;
}

__device__ __forceinline__ int owner_of(const SymmView &W, uint64_t hi)
{ int r = 0;
  for (int s = 1; s < W.n_seg; s++)
    r += (hi >= W.first_key[s]);
  return r;
}

/* all partners of x at positions >= p0, one bucket look-up per candidate (long runs only) */
template <typename IdxT, int KW>
__device__ __noinline__ void neighbours_slow(const uint64_t *__restrict__ keys, const uint64_t *__restrict__ keys_lo,
                                             const uint16_t *__restrict__ cnt, const IdxT *__restrict__ bucket,
                                             int bshift, int kmer, int p0, int pup,
                                             uint64_t x, uint64_t xl, int cx,
                                             int &H, int &U, int64_t &part, int &ppos)
{ H = 0; U = 0; part = -1; ppos = 0;
  for (int p = p0; p < kmer; p++)
    { int b = base_at<KW>(x,xl,p);
      for (int c = 0; c < 4; c++)
        { if (c == b) continue;
          uint64_t y = x, yl = xl;
          set_base<KW>(y,yl,p,c);
          int64_t j = bucket_find<IdxT,KW>(keys,keys_lo,bucket,bshift,y,yl);
          if (j >= 0 && cx + (int) __ldg(cnt+j) <= HM_SMAX)
            { H += 1;
              if (p >= pup) U += 1;
              part = j; ppos = p;
            }
        }
    }
}

/* ------------------------------------------------------------------- fingerprint -------- */

__device__ __forceinline__ uint64_t fp_mix(uint64_t hi, uint64_t lo, uint32_t c, uint64_t seed)
{ uint64_t v = (hi ^ seed) * 0xBF58476D1CE4E5B9ull;
  v ^= v >> 32;
  v = (v + lo + ((uint64_t) c << 40) + c) * 0x94D049BB133111EBull;
  v ^= v >> 29;
  v *= (seed | 1);
  v ^= v >> 32;
  return v;
}

template <int KW>
__global__ void __launch_bounds__(256)
symm_fingerprint_kernel(const uint64_t *__restrict__ keys, const uint64_t *__restrict__ keys_lo,
                        const uint16_t *__restrict__ cnt, int64_t i0, int64_t i1, int kmer,
                        uint64_t seed0, uint64_t seed1, unsigned long long *__restrict__ acc)
{ uint64_t a0 = 0, a1 = 0, a2 = 0, a3 = 0;
  const int64_t stride = (int64_t) gridDim.x * blockDim.x;
  for (int64_t i = i0 + (int64_t) blockIdx.x * blockDim.x + threadIdx.x; i < i1; i += stride)
    { uint64_t x = keys[i], xl = KW == 2 ? keys_lo[i] : 0, r, rl;
      uint32_t c = cnt[i];
      revcomp_kmer<KW>(x,xl,kmer,r,rl);
      a0 += fp_mix(x,xl,c,seed0);  a1 += fp_mix(x,xl,c,seed1);
      a2 += fp_mix(r,rl,c,seed0);  a3 += fp_mix(r,rl,c,seed1);
    }
  for (int o = 16; o > 0; o >>= 1)
    { a0 += __shfl_xor_sync(0xffffffffu,a0,o); a1 += __shfl_xor_sync(0xffffffffu,a1,o);
      a2 += __shfl_xor_sync(0xffffffffu,a2,o); a3 += __shfl_xor_sync(0xffffffffu,a3,o);
    }
  if ((threadIdx.x & 31) == 0)
    { atomicAdd(acc+0,(unsigned long long) a0); atomicAdd(acc+1,(unsigned long long) a1);
      atomicAdd(acc+2,(unsigned long long) a2); atomicAdd(acc+3,(unsigned long long) a3);
    }
}

extern "C" int hm_k_symm_fingerprint(const uint64_t *d_keys, const uint64_t *d_keys_lo, const uint16_t *d_cnt,
                                     int64_t i0, int64_t i1, int kmer, const uint64_t seed[2],
                                     uint64_t *d_acc, void *stream)
{ if (kmer < 1 || kmer > HM_MAX_KMER || (kmer > 32) != (d_keys_lo != NULL) || seed == NULL || d_acc == NULL)
    return hm_set_error(HM_EINVAL,"symm_fingerprint: bad arguments (k=%d)",kmer);
  if (i1 <= i0)
    return HM_OK;
  int64_t want = (i1-i0+255)/256;
  int     grid = (int) (want < 148*16 ? want : 148*16);
  if (kmer <= 32)
    symm_fingerprint_kernel<1><<<grid,256,0,(cudaStream_t) stream>>>
        (d_keys,NULL,d_cnt,i0,i1,kmer,seed[0],seed[1],(unsigned long long *) d_acc);
  else
    symm_fingerprint_kernel<2><<<grid,256,0,(cudaStream_t) stream>>>
        (d_keys,d_keys_lo,d_cnt,i0,i1,kmer,seed[0],seed[1],(unsigned long long *) d_acc);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess)
    return hm_cuda_fail(e,"symm_fingerprint_kernel");
  return HM_OK;
}

/* per-process seeds of the fingerprint (the table cannot have been chosen against them) */
extern "C" void hm_symm_seeds(uint64_t seed[2])
{ static uint64_t s[2] = {0,0};
  static int have = 0;
  if (!have)
    { FILE *f = fopen("/dev/urandom","rb");
      if (f == NULL || fread(s,sizeof(uint64_t),2,f) != 2)
        { struct timespec ts;
          clock_gettime(CLOCK_REALTIME,&ts);
          s[0] = 0x9E3779B97F4A7C15ull * (uint64_t) ts.tv_nsec ^ (uint64_t) ts.tv_sec;
          s[1] = 0xD1B54A32D192ED03ull * (uint64_t) (uintptr_t) &ts ^ ((uint64_t) ts.tv_nsec << 17);
        }
      if (f != NULL) fclose(f);
      have = 1;
    }
  seed[0] = s[0]; seed[1] = s[1];
}

/* ------------------------------------------------------------------------ layout -------- */

extern "C" int hm_symm_plan(int64_t n, int64_t range, int kmer, int n_seg, hm_symm_layout *out)
{ if (out == NULL || n < 0 || range < 0 || range > n || n_seg < 1 || n_seg > HM_MAX_SHARDS)
    return hm_set_error(HM_EINVAL,"hm_symm_plan: bad arguments");
  int bits = 2;                                  /* Bloom bits per table entry (S is ~1/6 of the table; two bits set per
                                                  *   element): 50 MB at 2e8 entries, kept in L2 by an access-policy
                                                  *   window (bloom_window).  Without the window its inserts miss L2 in
                                                  *   pass 1 (+0.55 ms) and 1 bit per entry is the better choice        */
  if (n_seg > 1)                                 /* several GPUs: all segments together are far beyond L2 and have to
                                                  *   cross NVLink between the kernels (0.95 ms of a 4.6 ms scan at 8
                                                  *   GPUs with 2 bits): half the filter, a few more exact checks      */
    bits = 1;
  const char *e = getenv("HETMERS_BLOOM_BITS");
  if (e != NULL && atoi(e) >= 1 && atoi(e) <= 64)
    bits = atoi(e);
  int64_t per = (n+n_seg-1)/n_seg;               /* every segment the same size on every rank: all-gather friendly */
  int64_t segw = (per*bits+31)/32;
  if (segw < 1024) segw = 1024;
  segw = (segw+63) & ~63ll;
  if (segw > 0x7fffffffll)
    return hm_set_error(HM_EUNSUPPORTED,"Bloom segment of %lld words too large",(long long) segw);
  int64_t cap = range/2 + 1024;
  int64_t at = 0;
  memset(out,0,sizeof(*out));
  out->off_header = at;  at += 256;
  out->off_bloom = at;   at += 4*segw*n_seg;
  out->seg_words = segw;
  at = (at+255) & ~255ll;
  out->off_cand_key = at;   at += 8*cap;
  out->off_cand_lo = at;    at += (kmer > 32) ? 8*cap : 0;
  out->off_cand_meta = at;  at += 8*cap;
  out->cand_cap = cap;
  out->off_runs = at;       out->runs_cap = range/3 + 1024;   at += 8*out->runs_cap;
  out->n_seg = n_seg;
  out->range = range;
  out->bytes = (at+255) & ~255ll;
  return HM_OK;
}

/* L2 residency of the Bloom segments for the kernels launched on `st` from here on: an access-policy window
 * marks the filter "persisting" (its read-modify-writes in pass 1 and its look-ups in pass 2 then hit L2
 * although 2 GB of table stream through next to them).  on = 0 lifts the window again.                   */
static void bloom_window(cudaStream_t st, const void *base, size_t bytes, int on)
{ static int limit_set[64] = {0};
  static size_t max_win[64] = {0}, max_persist[64] = {0};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 64) return;
  if (!limit_set[dev])
    { cudaDeviceProp p;
      limit_set[dev] = 1;
      if (cudaGetDeviceProperties(&p,dev) == cudaSuccess)
        { max_win[dev] = (size_t) p.accessPolicyMaxWindowSize;
          max_persist[dev] = (size_t) p.persistingL2CacheMaxSize;
          if (max_persist[dev] > 0)
            cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize,max_persist[dev]);
        }
      cudaGetLastError();
    }
  if (max_win[dev] == 0 || max_persist[dev] == 0)
    return;
  cudaStreamAttrValue a;
  memset(&a,0,sizeof(a));
  if (on)
    { size_t w = bytes < max_win[dev] ? bytes : max_win[dev];
      a.accessPolicyWindow.base_ptr  = (void *) base;
      a.accessPolicyWindow.num_bytes = w;
      a.accessPolicyWindow.hitRatio  = w <= max_persist[dev] ? 1.0f : (float) max_persist[dev] / (float) w;
      a.accessPolicyWindow.hitProp   = cudaAccessPropertyPersisting;
      a.accessPolicyWindow.missProp  = cudaAccessPropertyStreaming;
    }
  cudaStreamSetAttribute(st,cudaStreamAttributeAccessPolicyWindow,&a);
  cudaGetLastError();
}

static int l2_persist(void)                    /* HETMERS_L2_PERSIST=0 switches the window off */
{ const char *e = getenv("HETMERS_L2_PERSIST");
  return (e == NULL || strcmp(e,"0") != 0);
}

static SymmView make_view(void *d_work, const hm_symm_layout *L, const hm_symm_shards *sh)
{ SymmView W;
  uint8_t *b = (uint8_t *) d_work;
  memset(&W,0,sizeof(W));
  W.cand_n    = (unsigned long long *) (b + L->off_header);
  W.status    = W.cand_n + 1;
  W.bloom     = (uint32_t *) (b + L->off_bloom);
  W.seg_words = (uint32_t) L->seg_words;
  W.n_seg     = L->n_seg;
  W.self      = 0;
  if (sh != NULL && sh->n_seg > 1)
    { W.self = sh->self;
      for (int r = 0; r < sh->n_seg; r++) W.first_key[r] = sh->first_key[r];
    }
  W.cand_key  = (uint64_t *) (b + L->off_cand_key);
  W.cand_lo   = (uint64_t *) (b + L->off_cand_lo);
  W.cand_meta = (uint64_t *) (b + L->off_cand_meta);
  W.cand_cap  = (unsigned long long) L->cand_cap;
  W.runs_n    = W.cand_n + 2;
  W.runs      = (uint64_t *) (b + L->off_runs);
  W.runs_cap  = (unsigned long long) L->runs_cap;
  return W;
}

/* ------------------------------------------------------------------------ pass 1 -------- */

/* shared-memory views of one CTA's window + its staging areas */
template <int KW> struct RsSmem
  { uint64_t *key, *klo;                /* window: RS_WIN slots (+1 spare)                        */
    uint16_t *cnt;
    uint64_t *ckey, *clo, *cmeta;       /* staged candidate records: RS_STAGE                     */
    uint16_t *t1;                       /* per warp: heads of two-entry runs (RS_TILE/2 in all)    */
    uint16_t *t2r;                      /* CTA: heads of longer runs                               */
  };

__device__ __forceinline__ uint64_t pack_meta(int cx, int cy, int pos, int yb)
{ return (uint64_t) cx | ((uint64_t) cy << 16) | ((uint64_t) pos << 32) | ((uint64_t) yb << 40); }

/* candidate records into the CTA's staging area (warp-wide call; `emit` per lane): one shared atomic for
 * all the lanes that emit; lanes that find the staging area full
 * go to the list directly, again with one (global) atomic for all of them                              */
template <int KW>
__device__ __forceinline__ void stage_candidates(const RsSmem<KW> &S, unsigned *s_nc, const SymmView &W,
                                                 bool emit, uint64_t x, uint64_t xl, uint64_t meta,
                                                 int lane, unsigned lt)
{ const unsigned bal = __ballot_sync(0xffffffffu,emit);
  if (bal == 0)
    return;
  unsigned base = 0;
  if (lane == 0)
    base = atomicAdd(s_nc,(unsigned) __popc(bal));
  base = __shfl_sync(0xffffffffu,base,0);
  const unsigned at = base + __popc(bal & lt);
  const bool     over = emit && (at >= RS_STAGE);
  if (emit && !over)
    { S.ckey[at] = x;
      if (KW == 2) S.clo[at] = xl;
      S.cmeta[at] = meta;
    }
  if (base + __popc(bal) <= RS_STAGE)                  /* (warp-uniform) nobody overflowed */
    return;
  const unsigned ob = __ballot_sync(0xffffffffu,over);
  unsigned long long g0 = 0;
  if (lane == 0)
    g0 = atomicAdd(W.cand_n,(unsigned long long) __popc(ob));
  g0 = __shfl_sync(0xffffffffu,g0,0) + (unsigned long long) __popc(ob & lt);
  if (over)
    { if (g0 < W.cand_cap)
        { W.cand_key[g0] = x;
          if (KW == 2) W.cand_lo[g0] = xl;
          W.cand_meta[g0] = meta;
        }
      else
        atomicOr(W.status,SY_STATUS_OVERFLOW);
    }
}

template <int KW>
__device__ __forceinline__ void bloom_insert(const SymmView &W, int kmer, uint64_t x, uint64_t xl)
{ uint32_t *word, mask;
  bloom_slot<KW>(W,W.self,kmer,x,xl,word,mask);
  atomicOr(word,mask);
}

/* Pass 1b: the runs of three or more entries (1-2 % of the entries; collisions of a heterozygous pair
 * with an unrelated k-mer, repeats, low-complexity sequence) are irregular work: runscan_kernel only
 * lists their heads, this kernel takes one run per thread, straight from global memory (the keys of a
 * run are neighbours in the table).
 *   3..8 entries: every pair once, the members' partner counts packed into nibbles
 *   longer:       the warp takes the run together, one member per lane and trip, with one bucket
 *                 look-up per candidate partner (neighbours_slow) -- dense / tiny-k tables live here   */
template <typename IdxT, int KW>
__global__ void __launch_bounds__(256)
runs_kernel(const uint64_t *__restrict__ keys, const uint64_t *__restrict__ keys_lo,
            const uint16_t *__restrict__ cnt, int64_t n, const IdxT *__restrict__ bucket, int bshift,
            int kmer, int64_t lo, int64_t hi, const SymmView W)
{ const int      Pr = kmer >> 1, pup = kmer-Pr, psh = 64-2*Pr;
  const uint64_t pmask = ~(uint64_t) 0 << psh;
  const unsigned FULL = 0xffffffffu;
  const int      lane = threadIdx.x & 31;
  const unsigned lt   = (1u << lane) - 1;
  unsigned long long nrl = *W.runs_n;
  if (nrl > W.runs_cap) nrl = W.runs_cap;
  const int64_t nr     = (int64_t) nrl;
  const int64_t stride = (int64_t) gridDim.x * blockDim.x;
  for (int64_t r0 = (int64_t) blockIdx.x * blockDim.x + threadIdx.x - lane; r0 < nr; r0 += stride)
    { const int64_t r = r0+lane;
      const bool    valid = (r < nr);
      int64_t  h = 0;
      uint64_t x0 = 0;
      int      L = 1;
      if (valid)
        { h  = (int64_t) W.runs[r];
          x0 = __ldg(keys+h);
          while (L <= 8 && h+L < n && ((__ldg(keys+h+L) ^ x0) & pmask) == 0)
            L += 1;
        }
      const bool islong = valid && (L > 8);
      /* ---- short run: all pairs ---- */
      uint32_t H = 0, U = 0, PT = 0;
      uint64_t PP = 0;
      int      nrec = 0;
      if (valid && !islong)
        { for (int i = 0; i+1 < L; i++)
            { const uint64_t xi = __ldg(keys+h+i), xil = KW == 2 ? __ldg(keys_lo+h+i) : 0;
              const int      ci = __ldg(cnt+h+i);
              for (int j = i+1; j < L; j++)
                { int pos;
                  if (one_base_apart<KW>(xi,xil,__ldg(keys+h+j),KW == 2 ? __ldg(keys_lo+h+j) : 0,pos) &&
                      ci + (int) __ldg(cnt+h+j) <= HM_SMAX)
                    { H += (1u << (4*i)) + (1u << (4*j));
                      if (pos >= pup) U += (1u << (4*i)) + (1u << (4*j));
                      PT = (PT & ~((7u << (3*i)) | (7u << (3*j)))) | ((uint32_t) j << (3*i)) | ((uint32_t) i << (3*j));
                      PP = (PP & ~(((uint64_t) 255 << (8*i)) | ((uint64_t) 255 << (8*j)))) |
                           ((uint64_t) pos << (8*i)) | ((uint64_t) pos << (8*j));
                    }
                }
            }
          for (int i = 0; i < L; i++)
            { const int64_t g = h+i;
              if (g < lo || g >= hi) continue;
              if (((U >> (4*i)) & 15) != 0)
                bloom_insert<KW>(W,kmer,__ldg(keys+g),KW == 2 ? __ldg(keys_lo+g) : 0);
              const int j = (int) ((PT >> (3*i)) & 7);
              if (((H >> (4*i)) & 15) == 1 && j > i && ((H >> (4*j)) & 15) == 1)
                nrec += 1;
            }
        }
      /* candidate records of the short runs: one global atomic per warp */
      { int pre = nrec;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1)
          { int v = __shfl_up_sync(FULL,pre,o);
            if (lane >= o) pre += v;
          }
        const int tot = __shfl_sync(FULL,pre,31);
        if (tot > 0)
          { unsigned long long base = 0;
            if (lane == 0)
              base = atomicAdd(W.cand_n,(unsigned long long) tot);
            base = __shfl_sync(FULL,base,0) + (unsigned long long) (pre-nrec);
            if (nrec > 0)
              for (int i = 0; i < L; i++)
                { const int64_t g = h+i;
                  if (g < lo || g >= hi) continue;
                  const int j = (int) ((PT >> (3*i)) & 7);
                  if (((H >> (4*i)) & 15) == 1 && j > i && ((H >> (4*j)) & 15) == 1)
                    { const int      pos = (int) ((PP >> (8*i)) & 255);
                      const uint64_t y = __ldg(keys+h+j), yl = KW == 2 ? __ldg(keys_lo+h+j) : 0;
                      if (base < W.cand_cap)
                        { W.cand_key[base] = __ldg(keys+g);
                          if (KW == 2) W.cand_lo[base] = __ldg(keys_lo+g);
                          W.cand_meta[base] = pack_meta(__ldg(cnt+g),__ldg(cnt+h+j),pos,base_at<KW>(y,yl,pos));
                        }
                      else
                        atomicOr(W.status,SY_STATUS_OVERFLOW);
                      base += 1;
                    }
                }
          }
      }
      /* ---- long runs: the whole warp, one after the other ---- */
      unsigned lb = __ballot_sync(FULL,islong);
      while (lb != 0)
        { const int     src = __ffs(lb)-1;
          lb &= lb-1;
          const int64_t hh = __shfl_sync(FULL,h,src);
          const uint64_t xx = __shfl_sync(FULL,x0,src);
          int64_t end = hh+9;                          /* entries hh .. hh+8 are known to be in the run */
          while (true)
            { const int64_t t = end+lane;
              const bool same = (t < n) && (((__ldg(keys+t) ^ xx) & pmask) == 0);
              const unsigned sb = __ballot_sync(FULL,same);
              if (sb == FULL) { end += 32; continue; }
              end += __ffs(~sb)-1;
              break;
            }
          for (int64_t g0 = hh; g0 < end; g0 += 32)
            { const int64_t g = g0+lane;
              bool     emit = false;
              uint64_t x = 0, xl = 0, meta = 0;
              if (g < end && g >= lo && g < hi)
                { x = __ldg(keys+g);
                  if (KW == 2) xl = __ldg(keys_lo+g);
                  const int cx = __ldg(cnt+g);
                  int Hn, Un, ppos; int64_t part;
                  neighbours_slow<IdxT,KW>(keys,keys_lo,cnt,bucket,bshift,kmer,Pr,pup,x,xl,cx,Hn,Un,part,ppos);
                  if (Un > 0)
                    bloom_insert<KW>(W,kmer,x,xl);
                  if (Hn == 1 && part > g)
                    { const uint64_t y = __ldg(keys+part), yl = KW == 2 ? __ldg(keys_lo+part) : 0;
                      const int cy = __ldg(cnt+part);
                      int Hy, Uy, py; int64_t party;
                      neighbours_slow<IdxT,KW>(keys,keys_lo,cnt,bucket,bshift,kmer,Pr,pup,y,yl,cy,Hy,Uy,party,py);
                      if (Hy == 1)
                        { emit = true;
                          meta = pack_meta(cx,cy,ppos,base_at<KW>(y,yl,ppos));
                        }
                    }
                }
              const unsigned eb = __ballot_sync(FULL,emit);
              if (eb != 0)
                { unsigned long long base = 0;
                  if (lane == 0)
                    base = atomicAdd(W.cand_n,(unsigned long long) __popc(eb));
                  base = __shfl_sync(FULL,base,0) + (unsigned long long) __popc(eb & lt);
                  if (emit)
                    { if (base < W.cand_cap)
                        { W.cand_key[base] = x;
                          if (KW == 2) W.cand_lo[base] = xl;
                          W.cand_meta[base] = meta;
                        }
                      else
                        atomicOr(W.status,SY_STATUS_OVERFLOW);
                    }
                }
            }
        }
    }
}

/* Pass 1.  83 % of the entries of a genome-sized table are alone in their run (no other entry shares
 * their first k/2 bases) and 15 % sit in a run of exactly two -- almost always the two alleles of one
 * heterozygous site.  The kernel is bound by instruction issue and by the latency of its few serial
 * phases, not by bytes (55 warp instructions per 32 entries is all a B200 can issue while HBM delivers
 * them), so the common cases are loop-free and, once the tile has landed, every WARP works on its own
 * 256 entries without any CTA barrier:
 *   1. adjacency bits: eq[i] = slots i, i+1 belong to one run (one ballot per 32 slots; a warp computes
 *      the ten words it needs itself and keeps them one per lane)
 *   2. classification of 8 x 32 entries with bit operations, one WORD PER LANE:
 *      head of a two-entry run / head of a longer run / nothing
 *   3. two-entry runs: one comparison settles both members (per-warp task list, every lane busy)
 *   4. heads of longer runs are only LISTED (1-2 % of the entries, irregular work): runs_kernel
 *      takes them one per thread afterwards
 *   5. candidate records and run heads are staged in shared memory; the LAST warp to finish moves
 *      them out with one global atomic per CTA and list (one per record, or per warp, on the one
 *      list counter serialises in L2: 9.2 ms for 1.8e7 records)
 * (Scanning every entry's run in place cost 436 warp instructions per 32 entries at 34 % lane
 * utilisation; per-entry classification with predicated list writes 163; CTA-wide task lists with a
 * barrier per phase 117, but 57 % of the stall samples at those barriers; longer runs handled by
 * single lanes of every warp in place: slower again.)                                               */
template <typename IdxT, int KW>
__global__ void __launch_bounds__(RS_THREADS,RS_MINBLOCKS)
runscan_kernel(const uint64_t *__restrict__ keys, const uint64_t *__restrict__ keys_lo,
               const uint16_t *__restrict__ cnt, int64_t n, const IdxT *__restrict__ bucket, int bshift,
               int kmer, int64_t lo, int64_t hi, int64_t tile0, int use_tma, const SymmView W)
{ extern __shared__ __align__(128) uint8_t smem[];
  __shared__ __align__(8) uint64_t s_bar;
  __shared__ unsigned s_nc, s_nr, s_done;
  RsSmem<KW> S;
  S.key   = (uint64_t *) smem;
  S.klo   = S.key + (KW == 2 ? RS_WIN : 0);
  S.ckey  = S.key + KW*RS_WIN;
  S.clo   = S.ckey + (KW == 2 ? RS_STAGE : 0);
  S.cmeta = S.ckey + KW*RS_STAGE;
  S.cnt   = (uint16_t *) (S.cmeta + RS_STAGE);
  S.t1    = S.cnt + RS_WIN;                          /* per warp: RS_TILE/2/8 heads of two-entry runs        */
  S.t2r   = S.t1 + RS_TILE/2;                        /* CTA: heads of longer runs (at most RS_TILE/3)        */

  const int      Pr   = kmer >> 1;                 /* run = entries sharing their first Pr bases     */
  const int      pup  = kmer - Pr;                 /* positions >= pup have a mirror position < Pr   */
  const int      psh  = 64-2*Pr;
  const uint64_t pmask = ~(uint64_t) 0 << psh;
  const unsigned FULL = 0xffffffffu;
  const int      lane = threadIdx.x & 31;
  const int      warp = threadIdx.x >> 5;
  const unsigned lt   = (1u << lane) - 1;

  const int64_t T0 = (tile0 + blockIdx.x) * RS_TILE;
  const int64_t ws = T0 - RS_HALO;
  const int64_t e0 = ws > 0 ? ws : 0;
  const int64_t e1 = T0+RS_TILE+RS_HALO < n ? T0+RS_TILE+RS_HALO : n;
  const int     v0 = (int) (e0-ws), v1 = (int) (e1-ws);          /* valid window slots [v0,v1)   */

  /* ---- stage the window: TMA bulk copies for the 16-byte multiple, plain loads for the rest ---- */
  const int m   = v1-v0;
  const int mt  = use_tma ? (m & ~7) : 0;
  if (threadIdx.x == 0)
    { s_nc = 0; s_nr = 0; s_done = 0;
      if (mt > 0)
        { mbar_init(&s_bar,1);
          fence_proxy_async_smem();
        }
    }
  __syncthreads();
  if (threadIdx.x == 0 && mt > 0)
    { mbar_arrive_expect_tx(&s_bar,(unsigned) (mt*(8*KW+2)));
      bulk_copy_g2s(S.key+v0,keys+e0,(unsigned) (8*mt),&s_bar);
      if (KW == 2)
        bulk_copy_g2s(S.klo+v0,keys_lo+e0,(unsigned) (8*mt),&s_bar);
      bulk_copy_g2s(S.cnt+v0,cnt+e0,(unsigned) (2*mt),&s_bar);
    }
  if (mt < m || v0 > 0 || v1 < RS_WIN)                /* boundary tiles / unaligned tables only (CTA-uniform) */
    { for (int j = mt + threadIdx.x; j < m; j += RS_THREADS)
        { S.key[v0+j] = keys[e0+j];
          if (KW == 2) S.klo[v0+j] = keys_lo[e0+j];
          S.cnt[v0+j] = cnt[e0+j];
        }
      if (mt > 0)
        mbar_wait(&s_bar,0);
      __syncthreads();
      /* slots outside the table: a key no neighbour can share a run with */
      const uint64_t sa = ~S.key[v0], sb = ~S.key[v1-1];
      __syncthreads();
      for (int j = threadIdx.x; j < RS_WIN; j += RS_THREADS)
        if (j < v0)       S.key[j] = sa;
        else if (j >= v1) S.key[j] = sb;
      __syncthreads();
    }
  else
    mbar_wait(&s_bar,0);

  /* ---- 1. adjacency bits of this warp's words wd0-1 .. wd0+RS_EPT, word t in lane t ---- */
  const int wd0 = RS_HALO/32 + warp*RS_EPT;            /* first word (32 slots) of this warp's part of the tile */
  unsigned  eqw = 0;
#pragma unroll
  for (int t = 0; t < RS_EPT+2; t++)
    { const int i = (wd0-1+t)*32 + lane;
      bool eq;
      if (psh >= 32)                                   /* k <= 33: the first Pr bases sit in the upper word */
        { const uint32_t a = (uint32_t) (S.key[i] >> 32);
          uint32_t       b = __shfl_down_sync(FULL,a,1);
          if (lane == 31) b = (uint32_t) (S.key[i+1] >> 32);
          eq = (((a ^ b) >> (psh-32)) == 0);
        }
      else
        eq = (((S.key[i] ^ S.key[i+1]) & pmask) == 0);
      const unsigned bal = __ballot_sync(FULL,eq);
      if (lane == t) eqw = bal;
    }

  /* ---- 2. classify: lane t in 1..RS_EPT takes word wd0-1+t ---- */
  const int a0 = RS_HALO + (lo > T0 ? (int) (lo-T0 < RS_TILE ? lo-T0 : RS_TILE) : 0);   /* slots this CTA answers for */
  const int a1 = RS_HALO + (hi-T0 < RS_TILE ? (int) (hi-T0) : RS_TILE);
  uint16_t *my1  = S.t1  + warp*(RS_TILE/2/(RS_THREADS/32));
  int n1;
  { const unsigned P = __shfl_up_sync(FULL,eqw,1), N = __shfl_down_sync(FULL,eqw,1);
    unsigned m2 = 0, m3 = 0;
    const int wd = wd0-1+lane;
    if (lane >= 1 && lane <= RS_EPT)
      { const unsigned E = eqw;
        const unsigned em1 = (E << 1) | (P >> 31);                     /* eq[w-1] */
        const unsigned em2 = (E << 2) | (P >> 30);                     /* eq[w-2] */
        const unsigned ep1 = (E >> 1) | (N << 31);                     /* eq[w+1] */
        const int      s0  = wd*32;                                    /* slot of bit 0 */
        unsigned act = 0xffffffffu;
        if (s0 < a0)      act &= (a0-s0 >= 32) ? 0u : (0xffffffffu << (a0-s0));
        if (s0+32 > a1)   act &= (a1-s0 <= 0)  ? 0u : (0xffffffffu >> (s0+32-a1));
        const unsigned more = (em1 & E) | (E & ep1) | (em1 & em2);
        m2 = (E & ~em1 & ~ep1) & act;                                  /* head of a run of exactly two */
        m3 = more & act & ~em1;                                        /* head of a longer run: listed for runs_kernel */
      }
    /* per-warp task lists: inclusive scans of the counts over the lanes */
    const int c2 = __popc(m2), c3 = __popc(m3);
    int pre2 = c2, pre3 = c3;
#pragma unroll
    for (int o = 1; o <= RS_EPT; o <<= 1)
      { int v2 = __shfl_up_sync(FULL,pre2,o), v3 = __shfl_up_sync(FULL,pre3,o);
        if (lane >= o) { pre2 += v2; pre3 += v3; }
      }
    n1 = __shfl_sync(FULL,pre2,RS_EPT);
    const int n3 = __shfl_sync(FULL,pre3,RS_EPT);
    int at = pre2-c2;
    while (m2 != 0)
      { my1[at++] = (uint16_t) (wd*32 + __ffs(m2)-1);
        m2 &= m2-1;
      }
    if (n3 > 0)                                          /* (warp-uniform) heads of longer runs: CTA list */
      { unsigned b3 = 0;
        if (lane == 0)
          b3 = atomicAdd(&s_nr,(unsigned) n3);
        at = (int) __shfl_sync(FULL,b3,0) + pre3-c3;
        while (m3 != 0)
          { S.t2r[at++] = (uint16_t) (wd*32 + __ffs(m3)-1);
            m3 &= m3-1;
          }
      }
  }
  __syncwarp();

  /* ---- 3. runs of two: one comparison settles both members ---- */
  for (int i0 = 0; i0 < n1; i0 += 32)
    { const int i = i0+lane;
      bool     emit = false;
      uint64_t x = 0, xl = 0, meta = 0;
      if (i < n1)
        { const int w = my1[i];
          x = S.key[w];
          const uint64_t y = S.key[w+1];
          uint64_t yl = 0;
          if (KW == 2) { xl = S.klo[w]; yl = S.klo[w+1]; }
          const int cx = S.cnt[w], cy = S.cnt[w+1];
          int pos;
          if (one_base_apart<KW>(x,xl,y,yl,pos) && cx+cy <= HM_SMAX)      /* H(x) = H(y) = 1 */
            { emit = true;
              meta = pack_meta(cx,cy,pos,base_at<KW>(y,yl,pos));
              if (pos >= pup)                                              /* U(x) = U(y) = 1: both are in S */
                { bloom_insert<KW>(W,kmer,x,xl);
                  bloom_insert<KW>(W,kmer,y,yl);
                }
            }
        }
      stage_candidates<KW>(S,&s_nc,W,emit,x,xl,meta,lane,lt);
    }

  /* ---- 5. the last warp to get here moves the staged records out ---- */
  __syncwarp();
  unsigned last = 0;
  if (lane == 0)
    { __threadfence_block();
      last = (atomicAdd(&s_done,1u) == RS_THREADS/32-1);
    }
  last = __shfl_sync(FULL,last,0);
  if (!last)
    return;
  __threadfence_block();
  const unsigned nr = s_nr;
  if (nr > 0)
    { unsigned long long rb = 0;
      if (lane == 0)
        rb = atomicAdd(W.runs_n,(unsigned long long) nr);
      rb = __shfl_sync(FULL,rb,0);
      for (unsigned i = lane; i < nr; i += 32)
        if (rb+i < W.runs_cap)
          W.runs[rb+i] = (uint64_t) (T0 + ((int) S.t2r[i] - RS_HALO));
        else
          atomicOr(W.status,SY_STATUS_OVERFLOW);
    }
  const unsigned nc = s_nc < RS_STAGE ? s_nc : RS_STAGE;
  if (nc == 0)
    return;
  unsigned long long base = 0;
  if (lane == 0)
    base = atomicAdd(W.cand_n,(unsigned long long) nc);
  base = __shfl_sync(FULL,base,0);
  for (unsigned i = lane; i < nc; i += 32)
    { unsigned long long at = base + i;
      if (at < W.cand_cap)
        { W.cand_key[at] = S.ckey[i];
          if (KW == 2) W.cand_lo[at] = S.clo[i];
          W.cand_meta[at] = S.cmeta[i];
        }
      else
        atomicOr(W.status,SY_STATUS_OVERFLOW);
    }
}

/* Pass 1, crowded tables.  A run is the set of entries sharing their first k/2 bases, so an entry has
 * n / 4^(k/2) run mates on average whatever the sequence: 0.19 at 2e8 k-mers of k = 31 (where "alone" and
 * "a run of two" are all there is and runscan_kernel's classification pays), but 1.9 at 2e9 and 4.7 at
 * 5e9, where nearly every entry sits in a run of several unrelated k-mers.  Here every window slot
 * compares itself with the slots AFTER it in its run (the run's extent comes from the adjacency bits),
 * a pair found adds to both members' partner counts (byte-packed shared-memory atomics) and records the
 * partner; after a barrier every entry of the tile reads its own counts: Bloom insert if it has an
 * upper partner, candidate record if it and its single partner have one partner each.  All pairs of a
 * run are compared exactly once, the comparisons are spread evenly over the lanes, and the cost grows
 * with the run length instead of falling off a cliff (the one-thread-per-run kernel took 9.2 ms per
 * 2.5e8 entries at 2e9 k-mers, 377 ms per 6.25e8 at 5e9).  Runs of more than RS_LONGRUN entries are
 * listed for runs_kernel as before.                                                                   */
template <typename IdxT, int KW>
__global__ void __launch_bounds__(RS_THREADS,RS_MINBLOCKS)
runscan_dense_kernel(const uint64_t *__restrict__ keys, const uint64_t *__restrict__ keys_lo,
                     const uint16_t *__restrict__ cnt, int64_t n, int kmer, int64_t lo, int64_t hi,
                     int64_t tile0, int use_tma, const SymmView W)
{ extern __shared__ __align__(128) uint8_t smem[];
  __shared__ __align__(8) uint64_t s_bar;
  __shared__ unsigned s_nc, s_nl, s_done;
  __shared__ unsigned s_eq[RS_WIN/32+1];
  RsSmem<KW> S;
  S.key   = (uint64_t *) smem;
  S.klo   = S.key + (KW == 2 ? RS_WIN : 0);
  S.ckey  = S.key + KW*RS_WIN;
  S.clo   = S.ckey + (KW == 2 ? RS_STAGE : 0);
  S.cmeta = S.ckey + KW*RS_STAGE;
  S.cnt   = (uint16_t *) (S.cmeta + RS_STAGE);
  S.t1    = S.cnt + RS_WIN;                          /* here: a mark per window slot (RS_WIN)                */
  S.t2r   = S.t1 + RS_WIN;                           /* here: heads of runs of more than RS_LONGRUN entries  */
  uint16_t *s_part = S.t2r + RS_TILE/8;               /* partner slot of every window slot (RS_WIN)           */
  unsigned *hu = (unsigned *) (s_part + RS_WIN);      /* partner counts: per slot H (low byte) | U (high byte) */
  uint32_t *rem = hu + RS_WIN/2;                      /* k <= 32: the bases after the run prefix, 32 bits per slot */

  const int      Pr   = kmer >> 1, pup = kmer - Pr, psh = 64-2*Pr;
  const uint64_t pmask = ~(uint64_t) 0 << psh;
  const unsigned FULL = 0xffffffffu;
  const int      lane = threadIdx.x & 31;
  const int      warp = threadIdx.x >> 5;
  const unsigned lt   = (1u << lane) - 1;

  const int64_t T0 = (tile0 + blockIdx.x) * RS_TILE;
  const int64_t ws = T0 - RS_HALO;
  const int64_t e0 = ws > 0 ? ws : 0;
  const int64_t e1 = T0+RS_TILE+RS_HALO < n ? T0+RS_TILE+RS_HALO : n;
  const int     v0 = (int) (e0-ws), v1 = (int) (e1-ws);

  const int m   = v1-v0;
  const int mt  = use_tma ? (m & ~7) : 0;
  if (threadIdx.x == 0)
    { s_nc = 0; s_nl = 0; s_done = 0;
      if (mt > 0)
        { mbar_init(&s_bar,1);
          fence_proxy_async_smem();
        }
    }
  for (int j = threadIdx.x; j < RS_WIN/2; j += RS_THREADS)
    hu[j] = 0;
  __syncthreads();
  if (threadIdx.x == 0 && mt > 0)
    { mbar_arrive_expect_tx(&s_bar,(unsigned) (mt*(8*KW+2)));
      bulk_copy_g2s(S.key+v0,keys+e0,(unsigned) (8*mt),&s_bar);
      if (KW == 2)
        bulk_copy_g2s(S.klo+v0,keys_lo+e0,(unsigned) (8*mt),&s_bar);
      bulk_copy_g2s(S.cnt+v0,cnt+e0,(unsigned) (2*mt),&s_bar);
    }
  if (mt < m || v0 > 0 || v1 < RS_WIN)                /* boundary tiles / unaligned tables only (CTA-uniform) */
    { for (int j = mt + threadIdx.x; j < m; j += RS_THREADS)
        { S.key[v0+j] = keys[e0+j];
          if (KW == 2) S.klo[v0+j] = keys_lo[e0+j];
          S.cnt[v0+j] = cnt[e0+j];
        }
      if (mt > 0)
        mbar_wait(&s_bar,0);
      __syncthreads();
      const uint64_t sa = ~S.key[v0], sb = ~S.key[v1-1];
      __syncthreads();
      for (int j = threadIdx.x; j < RS_WIN; j += RS_THREADS)
        if (j < v0)       S.key[j] = sa;
        else if (j >= v1) S.key[j] = sb;
      __syncthreads();
    }
  else
    mbar_wait(&s_bar,0);

  /* ---- adjacency bits of the whole window; k <= 32: the bases after the run prefix as one 32-bit word ---- */
  const bool narrow = (KW == 1) && (kmer-Pr <= 16);      /* CTA-uniform: pair tests in 32-bit arithmetic */
  for (int wd = warp; wd < RS_WIN/32; wd += RS_THREADS/32)
    { const int i = wd*32 + lane;
      bool eq = false;
      const uint64_t ki = S.key[i];
      if (i+1 < RS_WIN)
        eq = (((ki ^ S.key[i+1]) & pmask) == 0);
      if (narrow)
        rem[i] = (uint32_t) ((ki << (2*Pr)) >> 32);
      const unsigned bal = __ballot_sync(FULL,eq);
      if (lane == 0)
        s_eq[wd] = bal;
    }
  if (threadIdx.x == 0)
    s_eq[RS_WIN/32] = 0;
  __syncthreads();

  /* ---- run mates after / before every slot = consecutive ones in the adjacency bits (32 are in view) ---- */
  const int a0 = RS_HALO + (lo > T0 ? (int) (lo-T0 < RS_TILE ? lo-T0 : RS_TILE) : 0);   /* slots this CTA answers for */
  const int a1 = RS_HALO + (hi-T0 < RS_TILE ? (int) (hi-T0) : RS_TILE);
  for (int i = threadIdx.x; i < RS_WIN; i += RS_THREADS)
    { const int      w = i >> 5, b = i & 31;
      const unsigned up = __funnelshift_r(s_eq[w],s_eq[w+1],b);                 /* eq[i], eq[i+1], ... */
      const int      fwd = (~up == 0) ? 32 : __ffs((int) ~up)-1;
      int back = 0;
      if (i > 0)
        { const int      wq = (i-1) >> 5, bq = (i-1) & 31;
          const unsigned dn = __funnelshift_l(wq > 0 ? s_eq[wq-1] : 0u,s_eq[wq],31-bq);   /* eq[i-1], eq[i-2], ... from the top */
          back = (~dn == 0) ? 32 : __clz((int) ~dn);
        }
      uint16_t mark = (uint16_t) fwd;                                            /* 0..31 run mates after this slot */
      if (back+fwd+1 > RS_LONGRUN)
        { mark = 0xffff;                                                         /* member of a long run: not ours */
          if (back == 0 && i >= a0 && i < a1)                                    /* its head, in our range: runs_kernel */
            S.t2r[atomicAdd(&s_nl,1u)] = (uint16_t) i;
        }
      S.t1[i] = mark;
      s_part[i] = (uint16_t) i;
    }
  __syncthreads();

  /* ---- every slot against the slots after it in its run ---- */
  for (int i = threadIdx.x; i < RS_WIN; i += RS_THREADS)
    { const int fwd = S.t1[i];
      if (fwd == 0 || fwd == 0xffff)
        continue;
      const int cx = S.cnt[i];
      if (narrow)
        { const uint32_t rx = rem[i];
          for (int j = i+1; j <= i+fwd; j++)
            { const uint32_t d = rx ^ rem[j];
              const uint32_t u = (d | (d>>1)) & 0x55555555u;
              if ((u & (u-1)) == 0 && cx + (int) S.cnt[j] <= HM_SMAX)
                { const int      pos = Pr + (__clz((int) d) >> 1);
                  const unsigned inc = 1u | (pos >= pup ? 0x100u : 0u);
                  atomicAdd(hu + (i>>1), inc << (16*(i&1)));
                  atomicAdd(hu + (j>>1), inc << (16*(j&1)));
                  s_part[i] = (uint16_t) j;                /* any partner: only read when there is exactly one */
                  s_part[j] = (uint16_t) i;
                }
            }
        }
      else
        { const uint64_t x = S.key[i], xl = KW == 2 ? S.klo[i] : 0;
          for (int j = i+1; j <= i+fwd; j++)
            { int pos;
              if (one_base_apart<KW>(x,xl,S.key[j],KW == 2 ? S.klo[j] : 0,pos) && cx + (int) S.cnt[j] <= HM_SMAX)
                { const unsigned inc = 1u | (pos >= pup ? 0x100u : 0u);
                  atomicAdd(hu + (i>>1), inc << (16*(i&1)));
                  atomicAdd(hu + (j>>1), inc << (16*(j&1)));
                  s_part[i] = (uint16_t) j;
                  s_part[j] = (uint16_t) i;
                }
            }
        }
    }
  __syncthreads();

  /* ---- every entry of the tile: its counts -> Bloom insert, candidate record ---- */
  for (int i0 = RS_HALO + (threadIdx.x & ~31); i0 < RS_HALO+RS_TILE; i0 += RS_THREADS)
    { const int i = i0+lane;
      bool     emit = false;
      uint64_t x = 0, xl = 0, meta = 0;
      if (i >= a0 && i < a1 && S.t1[i] != 0xffff)
        { const unsigned c = (hu[i>>1] >> (16*(i&1))) & 0xffffu;
          const int H = (int) (c & 0xff), U = (int) (c >> 8);
          if (H > 0)
            { x = S.key[i];
              if (KW == 2) xl = S.klo[i];
              if (U > 0)
                bloom_insert<KW>(W,kmer,x,xl);
              const int j = s_part[i];
              if (H == 1 && j > i && ((hu[j>>1] >> (16*(j&1))) & 0xffu) == 1)
                { const uint64_t y = S.key[j], yl = KW == 2 ? S.klo[j] : 0;
                  int pos;
                  one_base_apart<KW>(x,xl,y,yl,pos);
                  emit = true;
                  meta = pack_meta(S.cnt[i],S.cnt[j],pos,base_at<KW>(y,yl,pos));
                }
            }
        }
      stage_candidates<KW>(S,&s_nc,W,emit,x,xl,meta,lane,lt);
    }

  /* ---- the last warp to get here moves the staged records and the long-run heads out ---- */
  __syncwarp();
  unsigned last = 0;
  if (lane == 0)
    { __threadfence_block();
      last = (atomicAdd(&s_done,1u) == RS_THREADS/32-1);
    }
  last = __shfl_sync(FULL,last,0);
  if (!last)
    return;
  __threadfence_block();
  const unsigned nr = s_nl;
  if (nr > 0)
    { unsigned long long rb = 0;
      if (lane == 0)
        rb = atomicAdd(W.runs_n,(unsigned long long) nr);
      rb = __shfl_sync(FULL,rb,0);
      for (unsigned i = lane; i < nr; i += 32)
        if (rb+i < W.runs_cap)
          W.runs[rb+i] = (uint64_t) (T0 + ((int) S.t2r[i] - RS_HALO));
        else
          atomicOr(W.status,SY_STATUS_OVERFLOW);
    }
  const unsigned nc = s_nc < RS_STAGE ? s_nc : RS_STAGE;
  if (nc == 0)
    return;
  unsigned long long base = 0;
  if (lane == 0)
    base = atomicAdd(W.cand_n,(unsigned long long) nc);
  base = __shfl_sync(FULL,base,0);
  for (unsigned i = lane; i < nc; i += 32)
    { unsigned long long at = base + i;
      if (at < W.cand_cap)
        { W.cand_key[at] = S.ckey[i];
          if (KW == 2) W.cand_lo[at] = S.clo[i];
          W.cand_meta[at] = S.cmeta[i];
        }
      else
        atomicOr(W.status,SY_STATUS_OVERFLOW);
    }
}

template <typename IdxT, int KW>
static cudaError_t launch_runscan(const uint64_t *keys, const uint64_t *keys_lo, const uint16_t *cnt, int64_t n,
                                  const void *bucket, int bits, int kmer, int64_t lo, int64_t hi,
                                  const SymmView &W, cudaStream_t st)
{ static int configured[64] = {0};                            /* per instantiation */
  int dev = 0;
  cudaGetDevice(&dev);
  int64_t tile0 = lo/RS_TILE, tile1 = (hi+RS_TILE-1)/RS_TILE;
  int     tma   = ((((uintptr_t) keys) | ((uintptr_t) cnt) | ((uintptr_t) (keys_lo ? keys_lo : keys))) & 15) == 0;
  /* mean number of run mates of an entry = n / 4^(k/2): sparse tables take the classifying kernel, crowded
   * ones the all-pairs-in-the-run kernel (HETMERS_RUNSCAN=sparse|dense forces one)                       */
  const int   Pr  = kmer >> 1;
  double      lam = (2*Pr >= 62) ? 0.0 : (double) n / (double) ((uint64_t) 1 << (2*Pr));
  bool        dense = (lam > 0.6);
  const char *force = getenv("HETMERS_RUNSCAN");
  if (force != NULL && strcmp(force,"dense") == 0)  dense = true;
  if (force != NULL && strcmp(force,"sparse") == 0) dense = false;
  cudaError_t e;
  if (dense)
    { size_t smem = (size_t) RS_WIN*(8*KW+2) + (size_t) RS_STAGE*8*(KW+1) +
                    2*(size_t) (RS_WIN+RS_TILE/8+RS_WIN) + 4*(size_t) (RS_WIN/2+RS_WIN);   /* 52 KB (k <= 32) / 74 KB */
      if (smem > 48*1024 && (dev >= 64 || !(configured[dev] & 2)))
        { e = cudaFuncSetAttribute(runscan_dense_kernel<IdxT,KW>,cudaFuncAttributeMaxDynamicSharedMemorySize,(int) smem);
          if (e != cudaSuccess) return e;
          if (dev < 64) configured[dev] |= 2;
        }
      runscan_dense_kernel<IdxT,KW><<<(unsigned) (tile1-tile0),RS_THREADS,smem,st>>>
          (keys,keys_lo,cnt,n,kmer,lo,hi,tile0,tma,W);
    }
  else
    { size_t smem = (size_t) RS_WIN*(8*KW+2) + (size_t) RS_STAGE*8*(KW+1) +
                    2*(size_t) (RS_TILE/2+RS_TILE/2);                                /* 34 KB (k <= 32) / 55 KB */
      if (smem > 48*1024 && (dev >= 64 || !(configured[dev] & 1)))
        { e = cudaFuncSetAttribute(runscan_kernel<IdxT,KW>,cudaFuncAttributeMaxDynamicSharedMemorySize,(int) smem);
          if (e != cudaSuccess) return e;
          if (dev < 64) configured[dev] |= 1;
        }
      runscan_kernel<IdxT,KW><<<(unsigned) (tile1-tile0),RS_THREADS,smem,st>>>
          (keys,keys_lo,cnt,n,(const IdxT *) bucket,64-bits,kmer,lo,hi,tile0,tma,W);
    }
  return cudaGetLastError();
}

template <typename IdxT, int KW>
static cudaError_t launch_runs(const uint64_t *keys, const uint64_t *keys_lo, const uint16_t *cnt, int64_t n,
                               const void *bucket, int bits, int kmer, int64_t lo, int64_t hi,
                               const SymmView &W, cudaStream_t st)
{ /* (building the Bloom filter from the record list in a kernel of its own instead of inside runscan_kernel
   *  was measured slower: +0.15 ms)                                                                        */
  int64_t want = ((hi-lo)/64+255)/256;                        /* ~1 run of three or more per 60 entries: a thread each */
  int     grid = (int) (want < 0x7fffffff ? (want > 0 ? want : 1) : 0x7fffffff);
  runs_kernel<IdxT,KW><<<grid,256,0,st>>>(keys,keys_lo,cnt,n,(const IdxT *) bucket,64-bits,kmer,lo,hi,W);
  return cudaGetLastError();
}

extern "C" int hm_k_symm_runscan(const uint64_t *d_keys, const uint64_t *d_keys_lo, const uint16_t *d_cnt, int64_t n,
                                 const void *d_bucket, int bits, int idx64, int kmer, int64_t lo, int64_t hi,
                                 void *d_work, const hm_symm_layout *layout, const hm_symm_shards *shards,
                                 void *stream)
{ if (kmer < HM_SYMM_MIN_KMER || kmer > HM_MAX_KMER)
    return hm_set_error(HM_EUNSUPPORTED,"symmetric scan needs %d <= k <= %d (k=%d)",HM_SYMM_MIN_KMER,HM_MAX_KMER,kmer);
  if (lo < 0 || hi > n || lo > hi || bits < 1 || bits > 30 || d_work == NULL || layout == NULL)
    return hm_set_error(HM_EINVAL,"symm_runscan: bad range [%lld,%lld) of %lld or bits %d",
                        (long long) lo,(long long) hi,(long long) n,bits);
  if ((kmer > 32) != (d_keys_lo != NULL))
    return hm_set_error(HM_EINVAL,"symm_runscan: second key word array %s for k=%d",
                        d_keys_lo ? "given" : "missing",kmer);
  if ((shards != NULL && shards->n_seg > 1) != (layout->n_seg > 1) ||
      (shards != NULL && shards->n_seg > 1 && (shards->n_seg != layout->n_seg || shards->self < 0 ||
                                               shards->self >= shards->n_seg)))
    return hm_set_error(HM_EINVAL,"symm_runscan: shard table does not match the work-area layout");
  cudaStream_t st = (cudaStream_t) stream;
  SymmView W = make_view(d_work,layout,shards);
  HM_CUDA(cudaMemsetAsync(W.cand_n,0,256,st));
  HM_CUDA(cudaMemsetAsync(W.bloom + (size_t) W.self*W.seg_words,0,sizeof(uint32_t)*(size_t) W.seg_words,st));
  if (l2_persist())
    bloom_window(st,W.bloom,sizeof(uint32_t)*(size_t) W.seg_words*(size_t) W.n_seg,1);
  if (hi == lo)
    return HM_OK;
  cudaError_t e;
  if (kmer <= 32)
    e = idx64 ? launch_runscan<uint64_t,1>(d_keys,NULL,d_cnt,n,d_bucket,bits,kmer,lo,hi,W,st)
              : launch_runscan<uint32_t,1>(d_keys,NULL,d_cnt,n,d_bucket,bits,kmer,lo,hi,W,st);
  else
    e = idx64 ? launch_runscan<uint64_t,2>(d_keys,d_keys_lo,d_cnt,n,d_bucket,bits,kmer,lo,hi,W,st)
              : launch_runscan<uint32_t,2>(d_keys,d_keys_lo,d_cnt,n,d_bucket,bits,kmer,lo,hi,W,st);
  if (e != cudaSuccess)
    return hm_cuda_fail(e,"runscan_kernel");
  return HM_OK;
}

/* the runs runscan listed (three or more entries on sparse tables, more than RS_LONGRUN on crowded ones):
 * second half of "pass 1", a launch of its own so that callers can time the dominant kernel alone      */
extern "C" int hm_k_symm_runs(const uint64_t *d_keys, const uint64_t *d_keys_lo, const uint16_t *d_cnt, int64_t n,
                              const void *d_bucket, int bits, int idx64, int kmer, int64_t lo, int64_t hi,
                              void *d_work, const hm_symm_layout *layout, const hm_symm_shards *shards,
                              void *stream)
{ if (kmer < HM_SYMM_MIN_KMER || kmer > HM_MAX_KMER || d_work == NULL || layout == NULL ||
      (kmer > 32) != (d_keys_lo != NULL) || lo < 0 || hi > n || lo > hi)
    return hm_set_error(HM_EINVAL,"symm_runs: bad arguments");
  if (hi == lo)
    return HM_OK;
  cudaStream_t st = (cudaStream_t) stream;
  SymmView W = make_view(d_work,layout,shards);
  cudaError_t e;
  if (kmer <= 32)
    e = idx64 ? launch_runs<uint64_t,1>(d_keys,NULL,d_cnt,n,d_bucket,bits,kmer,lo,hi,W,st)
              : launch_runs<uint32_t,1>(d_keys,NULL,d_cnt,n,d_bucket,bits,kmer,lo,hi,W,st);
  else
    e = idx64 ? launch_runs<uint64_t,2>(d_keys,d_keys_lo,d_cnt,n,d_bucket,bits,kmer,lo,hi,W,st)
              : launch_runs<uint32_t,2>(d_keys,d_keys_lo,d_cnt,n,d_bucket,bits,kmer,lo,hi,W,st);
  if (e != cudaSuccess)
    return hm_cuda_fail(e,"runs_kernel");
  return HM_OK;
}

/* ------------------------------------------------------------------------ pass 2 -------- */

#define RV_TS 192      /* shared-memory plot tile: sums < 192, mins < 96 (72 KB) */
#define RV_TM 96
#define RV_THREADS 512
#define RV_CTAS_PER_SM 2
#define RV_ILP 4

/* does table entry q (count cq: the table is symmetric, so it is the count of the candidate member
 * whose reverse complement q is) have a partner at a position >= pup?  Exact.  The bucket index is at
 * most as fine as a run (bits <= 2*Pr), so q's bucket holds q's whole run: one pass over those few keys
 * finds q itself and its partners -- bucket offsets -> keys -> counts, three dependent accesses.        */
template <typename IdxT, int KW>
__device__ __noinline__ bool has_upper_partner(const uint64_t *__restrict__ keys, const uint64_t *__restrict__ keys_lo,
                                               const uint16_t *__restrict__ cnt, int64_t n,
                                               const IdxT *__restrict__ bucket, int bshift, int kmer,
                                               uint64_t q, uint64_t ql, int cq, unsigned long long *status)
{ const int Pr = kmer >> 1, pup = kmer-Pr, psh = 64-2*Pr;
  if (bshift >= psh)                                            /* bucket prefix no longer than the run prefix */
    { const uint64_t bk = q >> bshift;
      const int64_t  l = (int64_t) bucket[bk], r = (int64_t) bucket[bk+1];
      if (r-l <= 48)
        { bool found = false, hit = false;
          for (int64_t i = l; i < r; i++)
            { const uint64_t z = __ldg(keys+i), zl = KW == 2 ? __ldg(keys_lo+i) : 0;
              if (z == q && (KW == 1 || zl == ql))
                { found = true; continue; }
              if (((z ^ q) >> psh) != 0)
                continue;
              int pos;
              if (one_base_apart<KW>(q,ql,z,zl,pos) && pos >= pup && cq + (int) __ldg(cnt+i) <= HM_SMAX)
                hit = true;
            }
          if (!found)
            atomicOr(status,SY_STATUS_ASYMMETRIC);
          return hit;
        }
    }
  int64_t j = bucket_find<IdxT,KW>(keys,keys_lo,bucket,bshift,q,ql);
  if (j < 0)
    { atomicOr(status,SY_STATUS_ASYMMETRIC);
      return true;
    }
  bool capped = false;
  for (int dir = -1; dir <= 1; dir += 2)
    { int steps = 0;
      for (int64_t i = j+dir; i >= 0 && i < n; i += dir)
        { uint64_t z = __ldg(keys+i);
          if (((z ^ q) >> psh) != 0) break;
          if (++steps > RS_SCANCAP) { capped = true; break; }
          int pos;
          if (one_base_apart<KW>(q,ql,z,KW == 2 ? __ldg(keys_lo+i) : 0,pos) && pos >= pup &&
              cq + (int) __ldg(cnt+i) <= HM_SMAX)
            return true;
        }
    }
  if (!capped)
    return false;
  int H, U, ppos; int64_t part;
  neighbours_slow<IdxT,KW>(keys,keys_lo,cnt,bucket,bshift,kmer,pup,pup,q,ql,cq,H,U,part,ppos);
  return (U > 0);
}

/* per-shard tables of a sharded scan (every shard holds only its own key range, DESIGN.md §6): the exact
 * check of a Bloom hit reads rc x's run in the arrays of the shard that owns it, as peer memory       */
typedef hm_shard_tabs ShardTabs;
struct NoTabs {};                                           /* a replica: the table is local */

template <typename IdxT, int KW, typename Tabs>
__device__ __forceinline__ bool exact_upper_partner(const uint64_t *__restrict__ keys, const uint64_t *__restrict__ keys_lo,
                                                    const uint16_t *__restrict__ cnt, int64_t n,
                                                    const IdxT *__restrict__ bucket, int bshift, int kmer,
                                                    const SymmView &W, const Tabs &T, uint64_t q, uint64_t ql, int cq)
{ if constexpr (std::is_same<Tabs,ShardTabs>::value)
    { const int o = W.n_seg > 1 ? owner_of(W,q) : 0;
      return has_upper_partner<IdxT,KW>(T.keys[o],T.keys_lo[o],T.cnt[o],T.n[o],(const IdxT *) T.bucket[o],
                                        bshift,kmer,q,ql,cq,W.status);
    }
  else
    return has_upper_partner<IdxT,KW>(keys,keys_lo,cnt,n,bucket,bshift,kmer,q,ql,cq,W.status);
}

/* one candidate: are rc x / rc y in S?  Bloom bits first; EXACT = also settle the hits.
 * -> 0 isolated pair, 1 not isolated, 2 undecided (a Bloom hit, EXACT == false)                  */
template <typename IdxT, int KW, bool EXACT, typename Tabs>
__device__ __forceinline__ int judge_candidate(const uint64_t *__restrict__ keys, const uint64_t *__restrict__ keys_lo,
                                               const uint16_t *__restrict__ cnt, int64_t n,
                                               const IdxT *__restrict__ bucket, int bshift, int kmer,
                                               const SymmView &W, const Tabs &T, uint64_t x, uint64_t xl, uint64_t meta)
{ const int cx = (int) (meta & 0xffff), cy = (int) ((meta >> 16) & 0xffff);
  const int p  = (int) ((meta >> 32) & 0xff), yb = (int) ((meta >> 40) & 3);
  uint64_t rx, rxl, ry, ryl;
  revcomp_kmer<KW>(x,xl,kmer,rx,rxl);
  ry = rx; ryl = rxl;
  set_base<KW>(ry,ryl,kmer-1-p,3-yb);                      /* rc y = rc x with the mirrored base swapped */
  uint32_t *wa, *wb, ba, bb;
  bloom_slot<KW>(W,W.n_seg > 1 ? owner_of(W,rx) : 0,kmer,rx,rxl,wa,ba);
  bloom_slot<KW>(W,W.n_seg > 1 ? owner_of(W,ry) : 0,kmer,ry,ryl,wb,bb);
  const uint32_t va = ld_keep(wa);
  const uint32_t vb = (wb == wa) ? va : ld_keep(wb);       /* one shard owns both: the same word */
  const bool ha = (va & ba) == ba, hb = (vb & bb) == bb;
  if (!ha && !hb)
    return 0;
  if (!EXACT)
    return 2;
  if (ha && exact_upper_partner<IdxT,KW>(keys,keys_lo,cnt,n,bucket,bshift,kmer,W,T,rx,rxl,cx))
    return 1;
  if (hb && exact_upper_partner<IdxT,KW>(keys,keys_lo,cnt,n,bucket,bshift,kmer,W,T,ry,ryl,cy))
    return 1;
  return 0;
}

__device__ __forceinline__ void count_pair(uint32_t *tile, unsigned long long *__restrict__ plot,
                                           uint64_t meta, int kmer)
{ const int cx = (int) (meta & 0xffff), cy = (int) ((meta >> 16) & 0xffff);
  const int p  = (int) ((meta >> 32) & 0xff);
  const unsigned wgt = (2*p == kmer-1) ? 1u : 2u;          /* middle base: the mirror pair is found itself */
  const int s = cx+cy;
  const int m = cx < cy ? cx : cy;
  if (s < RV_TS && m < RV_TM)
    atomicAdd(tile + s*RV_TM + m, wgt);
  else
    atomicAdd(plot + s*HM_PLOT_W + m, (unsigned long long) wgt);
}

/* What pass 2 does with a candidate judged to be an isolated pair (take() is called by the lanes that
 * hold one):
 *   PlotSink    counts it into the plot (resolve_kernel, resolve_sharded_kernel)
 *   RecordSink  writes extract_kmer_pairs' records of it (extract_kernel, extract_sharded_kernel)
 * first() / last() pick the candidates [first, min(count, last)) the kernel judges.                   */
struct PlotSink
  { unsigned long long *plot;
    int kmer;
    __device__ __forceinline__ int64_t first() const { return 0; }
    __device__ __forceinline__ int64_t last(int64_t nc) const { return nc; }
    __device__ __forceinline__ void begin() const
    { extern __shared__ uint32_t tile[];
      for (int t = threadIdx.x; t < RV_TS*RV_TM; t += blockDim.x)
        tile[t] = 0;
      __syncthreads();
    }
    __device__ __forceinline__ void take(uint64_t, uint64_t, uint64_t meta) const
    { extern __shared__ uint32_t tile[];
      count_pair(tile,plot,meta,kmer);
    }
    __device__ __forceinline__ void end() const
    { extern __shared__ uint32_t tile[];
      __syncthreads();
      for (int t = threadIdx.x; t < RV_TS*RV_TM; t += blockDim.x)
        { uint32_t v = tile[t];
          if (v != 0)
            atomicAdd(plot + (t/RV_TM)*HM_PLOT_W + (t%RV_TM), (unsigned long long) v);
        }
    }
  };

/* extract_kmer_pairs' records of one isolated candidate x < y (differing at p >= k/2, x's base bx <
 * y's base by), when its pixel carries a label -- what the reference prints for the pair and for its
 * mirror image (PloidyList.c:432-447), which the direct passes find as a pair of its own:
 *   the pair         cx < cy: y with alt bx, else (a tie too) x with alt by;             pos p
 *   the mirror       (rc y, rc x): rc y is the lower member (3-by < 3-bx at k-1-p) and has count cy,
 *                    so cy < cx: rc x with alt 3-by, else (a tie too) rc y with alt 3-bx; pos k-1-p
 * The mirror is left out at the middle base of an odd k (2p == k-1), where it is found as a candidate
 * itself -- count_pair's weight of 1 -- so n records == plot[pixmap > 0].sum().  Records are appended
 * with one global atomic per warp and call (ballot + prefix over the lanes that hold an isolated pair:
 * the active mask).  A slice of the candidates yields at most 2 records each, so `cap` is never reached.          */
template <int KW>
struct RecordSink
  { const uint16_t *pixmap;
    hm_pair_rec *out;
    unsigned long long *out_n, *status, cap;
    int64_t c0, c1;
    int kmer;
    __device__ __forceinline__ int64_t first() const { return c0; }
    __device__ __forceinline__ int64_t last(int64_t nc) const { return nc < c1 ? nc : c1; }
    __device__ __forceinline__ void begin() const {}
    __device__ __forceinline__ void end() const {}
    __device__ __forceinline__ void put(unsigned long long at, uint64_t h, uint64_t l, uint32_t lab, int pos, int alt) const
    { if (at >= cap)
        { atomicOr(status,SY_STATUS_OVERFLOW); return; }
      hm_pair_rec r;
      r.key_hi = h; r.key_lo = l; r.smudge = lab; r.pos = (uint8_t) pos; r.alt = (uint8_t) alt; r.pad = 0;
      out[at] = r;
    }
    __device__ __forceinline__ void take(uint64_t x, uint64_t xl, uint64_t meta) const
    { const int cx = (int) (meta & 0xffff), cy = (int) ((meta >> 16) & 0xffff);
      const int p  = (int) ((meta >> 32) & 0xff), by = (int) ((meta >> 40) & 3);
      const uint32_t lab = __ldg(pixmap + (cx+cy)*HM_PLOT_W + (cx < cy ? cx : cy));
      const bool     one = (lab != 0), two = one && (2*p != kmer-1);
      const unsigned m  = __activemask();
      const unsigned b1 = __ballot_sync(m,one), b2 = __ballot_sync(m,two);
      if (b1 == 0)
        return;
      const int      lane = threadIdx.x & 31, lead = __ffs((int) m)-1;
      const unsigned lt   = (1u << lane) - 1;
      unsigned long long at = 0;
      if (lane == lead)
        at = atomicAdd(out_n,(unsigned long long) (__popc(b1)+__popc(b2)));
      at = __shfl_sync(m,at,lead) + (unsigned long long) (__popc(b1 & lt) + __popc(b2 & lt));
      if (!one)
        return;
      const int bx = base_at<KW>(x,xl,p);
      uint64_t  y = x, yl = xl;
      set_base<KW>(y,yl,p,by);
      if (cx < cy) put(at,y,yl,lab,p,bx);
      else         put(at,x,xl,lab,p,by);
      if (!two)
        return;
      uint64_t rx, rxl, ry, ryl;
      revcomp_kmer<KW>(x,xl,kmer,rx,rxl);
      ry = rx; ryl = rxl;
      set_base<KW>(ry,ryl,kmer-1-p,3-by);
      if (cy < cx) put(at+1,rx,rxl,lab,kmer-1-p,3-by);
      else         put(at+1,ry,ryl,lab,kmer-1-p,3-bx);
    }
  };

/* Candidates whose Bloom look-up misses (~95 %) are settled at once.  The others need the exact
 * answer -- bucket offsets, keys, counts: three dependent random accesses -- and a warp in which one
 * lane does that stalls all 32: they are parked in a per-warp queue and settled 32 at a time, every
 * lane busy.  RV_ILP candidates per thread and trip keep that many record / Bloom loads in flight
 * (the kernel is bound by the latency of record -> Bloom word, not by bytes or instructions).         */
template <typename IdxT, int KW, typename Tabs, typename Sink>
__device__ __forceinline__ void resolve_body(const uint64_t *__restrict__ keys, const uint64_t *__restrict__ keys_lo,
                                             const uint16_t *__restrict__ cnt, int64_t n, const IdxT *__restrict__ bucket,
                                             int bshift, int kmer, const SymmView &W, const Tabs &T, const Sink &sink)
{ __shared__ uint32_t s_q[RV_THREADS/32][32*(RV_ILP+1)];
  const unsigned FULL = 0xffffffffu;
  const int      lane = threadIdx.x & 31;
  const unsigned lt   = (1u << lane) - 1;
  uint32_t *q  = s_q[threadIdx.x >> 5];
  int       qn = 0;
  sink.begin();
  unsigned long long ncl = *W.cand_n;
  if (ncl > W.cand_cap) ncl = W.cand_cap;
  const int64_t c0     = sink.first();
  const int64_t nc     = sink.last((int64_t) ncl) - c0;
  const uint64_t *ckey = W.cand_key + c0, *clo = W.cand_lo + c0, *cmeta = W.cand_meta + c0;
  const int64_t stride = (int64_t) gridDim.x * blockDim.x;
  const int64_t first  = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
  for (uint32_t it = 0; first-lane + (int64_t) it*RV_ILP*stride < nc; it++)
    { uint64_t x[RV_ILP], xl[RV_ILP], meta[RV_ILP];
      uint32_t *wa[RV_ILP], *wb[RV_ILP], ba[RV_ILP], bb[RV_ILP], va[RV_ILP], vb[RV_ILP];
      bool     ok[RV_ILP];
#pragma unroll
      for (int u = 0; u < RV_ILP; u++)
        { const int64_t i = first + ((int64_t) it*RV_ILP+u)*stride;
          ok[u] = (i < nc);
          x[u] = 0; xl[u] = 0; meta[u] = 0;
          if (ok[u])
            { x[u] = ld_stream(ckey+i);
              if (KW == 2) xl[u] = ld_stream(clo+i);
              meta[u] = ld_stream(cmeta+i);
            }
        }
#pragma unroll
      for (int u = 0; u < RV_ILP; u++)
        { const int p  = (int) ((meta[u] >> 32) & 0xff), yb = (int) ((meta[u] >> 40) & 3);
          uint64_t rx, rxl, ry, ryl;
          revcomp_kmer<KW>(x[u],xl[u],kmer,rx,rxl);
          ry = rx; ryl = rxl;
          set_base<KW>(ry,ryl,kmer-1-p,3-yb);
          bloom_slot<KW>(W,W.n_seg > 1 ? owner_of(W,rx) : 0,kmer,rx,rxl,wa[u],ba[u]);
          bloom_slot<KW>(W,W.n_seg > 1 ? owner_of(W,ry) : 0,kmer,ry,ryl,wb[u],bb[u]);
        }
#pragma unroll
      for (int u = 0; u < RV_ILP; u++)
        { va[u] = 0; vb[u] = 0;
          if (ok[u])
            { va[u] = ld_keep(wa[u]);
              vb[u] = (wb[u] == wa[u]) ? va[u] : ld_keep(wb[u]);
            }
        }
#pragma unroll
      for (int u = 0; u < RV_ILP; u++)
        { const bool hit = ok[u] && ((va[u] & ba[u]) == ba[u] || (vb[u] & bb[u]) == bb[u]);
          if (ok[u] && !hit)
            sink.take(x[u],xl[u],meta[u]);
          const unsigned bal = __ballot_sync(FULL,hit);
          if (hit)
            q[qn + __popc(bal & lt)] = ((it*RV_ILP+u) << 5) | (uint32_t) lane;
          qn += __popc(bal);
        }
      __syncwarp();
      while (qn >= 32)
        { qn -= 32;
          const uint32_t e = q[qn+lane];
          __syncwarp();
          const int64_t j = first-lane + (int64_t) (e & 31) + (int64_t) (e >> 5)*stride;
          const uint64_t xx = ckey[j], xxl = KW == 2 ? clo[j] : 0, mm = cmeta[j];
          if (judge_candidate<IdxT,KW,true>(keys,keys_lo,cnt,n,bucket,bshift,kmer,W,T,xx,xxl,mm) == 0)
            sink.take(xx,xxl,mm);
        }
    }
  if (lane < qn)
    { const uint32_t e = q[lane];
      const int64_t j = first-lane + (int64_t) (e & 31) + (int64_t) (e >> 5)*stride;
      const uint64_t xx = ckey[j], xxl = KW == 2 ? clo[j] : 0, mm = cmeta[j];
      if (judge_candidate<IdxT,KW,true>(keys,keys_lo,cnt,n,bucket,bshift,kmer,W,T,xx,xxl,mm) == 0)
        sink.take(xx,xxl,mm);
    }
  sink.end();
}

template <typename IdxT, int KW>
__global__ void __launch_bounds__(RV_THREADS,RV_CTAS_PER_SM)
resolve_kernel(const uint64_t *__restrict__ keys, const uint64_t *__restrict__ keys_lo,
               const uint16_t *__restrict__ cnt, int64_t n, const IdxT *__restrict__ bucket, int bshift,
               int kmer, const SymmView W, unsigned long long *__restrict__ plot)
{ resolve_body<IdxT,KW>(keys,keys_lo,cnt,n,bucket,bshift,kmer,W,NoTabs(),PlotSink{plot,kmer}); }

/* pass 2 of a sharded scan: the same, with every Bloom hit settled in the owner's arrays */
template <typename IdxT, int KW>
__global__ void __launch_bounds__(RV_THREADS,RV_CTAS_PER_SM)
resolve_sharded_kernel(int bshift, int kmer, const SymmView W, const ShardTabs T, unsigned long long *__restrict__ plot)
{ resolve_body<IdxT,KW>((const uint64_t *) NULL,(const uint64_t *) NULL,(const uint16_t *) NULL,(int64_t) 0,
                        (const IdxT *) NULL,bshift,kmer,W,T,PlotSink{plot,kmer});
}

/* extract_kmer_pairs from the symmetric scan: pass 2 over the candidates [c0, c1) of the last run
 * scan, isolated pairs written as records (RecordSink) instead of counted.  The record sink keeps the
 * candidates' keys live across the loop, which does not fit the 64 registers of two CTAs per SM
 * without spilling: one CTA per SM (the kernel runs once per extraction, not once per scan).       */
template <typename IdxT, int KW>
__global__ void __launch_bounds__(RV_THREADS,1)
extract_kernel(const uint64_t *__restrict__ keys, const uint64_t *__restrict__ keys_lo,
               const uint16_t *__restrict__ cnt, int64_t n, const IdxT *__restrict__ bucket, int bshift,
               int kmer, const SymmView W, const RecordSink<KW> R)
{ resolve_body<IdxT,KW>(keys,keys_lo,cnt,n,bucket,bshift,kmer,W,NoTabs(),R); }

template <typename IdxT, int KW>
__global__ void __launch_bounds__(RV_THREADS,1)
extract_sharded_kernel(int bshift, int kmer, const SymmView W, const ShardTabs T, const RecordSink<KW> R)
{ resolve_body<IdxT,KW>((const uint64_t *) NULL,(const uint64_t *) NULL,(const uint16_t *) NULL,(int64_t) 0,
                        (const IdxT *) NULL,bshift,kmer,W,T,R);
}

template <typename IdxT, int KW>
static cudaError_t launch_resolve(const uint64_t *keys, const uint64_t *keys_lo, const uint16_t *cnt, int64_t n,
                                  const void *bucket, int bits, int kmer, const SymmView &W,
                                  unsigned long long *plot, int64_t range, cudaStream_t st)
{ static int configured[64] = {0};                            /* per instantiation */
  size_t smem = (size_t) RV_TS*RV_TM*sizeof(uint32_t);
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  if (dev >= 64 || !configured[dev])
    { cudaError_t e = cudaFuncSetAttribute(resolve_kernel<IdxT,KW>,cudaFuncAttributeMaxDynamicSharedMemorySize,(int) smem);
      if (e != cudaSuccess) return e;
      if (dev < 64) configured[dev] = 1;
    }
  cudaDeviceGetAttribute(&sms,cudaDevAttrMultiProcessorCount,dev);
  int64_t want = (range/8+RV_THREADS-1)/RV_THREADS;            /* ~1 candidate per 10 entries */
  int     grid = (int) (want < sms*RV_CTAS_PER_SM ? (want > 0 ? want : 1) : sms*RV_CTAS_PER_SM);
  resolve_kernel<IdxT,KW><<<grid,RV_THREADS,smem,st>>>(keys,keys_lo,cnt,n,(const IdxT *) bucket,64-bits,kmer,W,plot);
  return cudaGetLastError();
}

extern "C" int hm_k_symm_resolve(const uint64_t *d_keys, const uint64_t *d_keys_lo, const uint16_t *d_cnt, int64_t n,
                                 const void *d_bucket, int bits, int idx64, int kmer,
                                 void *d_work, const hm_symm_layout *layout, const hm_symm_shards *shards,
                                 unsigned long long *d_plot, void *stream)
{ if (kmer < HM_SYMM_MIN_KMER || kmer > HM_MAX_KMER || d_work == NULL || layout == NULL || d_plot == NULL)
    return hm_set_error(HM_EINVAL,"symm_resolve: bad arguments");
  if ((kmer > 32) != (d_keys_lo != NULL))
    return hm_set_error(HM_EINVAL,"symm_resolve: second key word array %s for k=%d",
                        d_keys_lo ? "given" : "missing",kmer);
  cudaStream_t st = (cudaStream_t) stream;
  SymmView W = make_view(d_work,layout,shards);
  int64_t range = layout->range;
  cudaError_t e;
  if (kmer <= 32)
    e = idx64 ? launch_resolve<uint64_t,1>(d_keys,NULL,d_cnt,n,d_bucket,bits,kmer,W,d_plot,range,st)
              : launch_resolve<uint32_t,1>(d_keys,NULL,d_cnt,n,d_bucket,bits,kmer,W,d_plot,range,st);
  else
    e = idx64 ? launch_resolve<uint64_t,2>(d_keys,d_keys_lo,d_cnt,n,d_bucket,bits,kmer,W,d_plot,range,st)
              : launch_resolve<uint32_t,2>(d_keys,d_keys_lo,d_cnt,n,d_bucket,bits,kmer,W,d_plot,range,st);
  if (l2_persist())
    bloom_window(st,NULL,0,0);
  if (e != cudaSuccess)
    return hm_cuda_fail(e,"resolve_kernel");
  return HM_OK;
}

template <typename IdxT, int KW>
static cudaError_t launch_resolve_sharded(int bits, int kmer, const SymmView &W, const ShardTabs &T,
                                          unsigned long long *plot, int64_t range, cudaStream_t st)
{ static int configured[64] = {0};
  size_t smem = (size_t) RV_TS*RV_TM*sizeof(uint32_t);
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  if (dev >= 64 || !configured[dev])
    { cudaError_t e = cudaFuncSetAttribute(resolve_sharded_kernel<IdxT,KW>,cudaFuncAttributeMaxDynamicSharedMemorySize,(int) smem);
      if (e != cudaSuccess) return e;
      if (dev < 64) configured[dev] = 1;
    }
  cudaDeviceGetAttribute(&sms,cudaDevAttrMultiProcessorCount,dev);
  int64_t want = (range/8+RV_THREADS-1)/RV_THREADS;
  int     grid = (int) (want < sms*RV_CTAS_PER_SM ? (want > 0 ? want : 1) : sms*RV_CTAS_PER_SM);
  resolve_sharded_kernel<IdxT,KW><<<grid,RV_THREADS,smem,st>>>(64-bits,kmer,W,T,plot);
  return cudaGetLastError();
}

/* pass 2 of a sharded table: tabs holds every shard's arrays as addressable from the calling device */
int hm_symm_resolve_sharded(const hm_shard_tabs *tabs, int bits, int idx64, int kmer, void *d_work,
                            const hm_symm_layout *layout, const hm_symm_shards *shards,
                            unsigned long long *d_plot, void *stream)
{ if (kmer < HM_SYMM_MIN_KMER || kmer > HM_MAX_KMER || tabs == NULL || d_work == NULL || layout == NULL || d_plot == NULL)
    return hm_set_error(HM_EINVAL,"symm_resolve_sharded: bad arguments");
  cudaStream_t st = (cudaStream_t) stream;
  SymmView W = make_view(d_work,layout,shards);
  cudaError_t e;
  if (kmer <= 32)
    e = idx64 ? launch_resolve_sharded<uint64_t,1>(bits,kmer,W,*tabs,d_plot,layout->range,st)
              : launch_resolve_sharded<uint32_t,1>(bits,kmer,W,*tabs,d_plot,layout->range,st);
  else
    e = idx64 ? launch_resolve_sharded<uint64_t,2>(bits,kmer,W,*tabs,d_plot,layout->range,st)
              : launch_resolve_sharded<uint32_t,2>(bits,kmer,W,*tabs,d_plot,layout->range,st);
  if (l2_persist())
    bloom_window(st,NULL,0,0);
  if (e != cudaSuccess)
    return hm_cuda_fail(e,"resolve_sharded_kernel");
  return HM_OK;
}

/* ----------------------------------------------------------- pass 2, extract variant -- */

/* The records of an extraction are staged in the run-head region of the work area (idle once pass 1 is
 * done; the next run scan starts it afresh) and counted in header word 3: 8*runs_cap bytes hold cap =
 * 8*runs_cap/24 records, enough for the records of cap/2 candidates -- one slice.                    */
#define SY_HDR_RECORDS 3

int64_t hm_symm_extract_slice(const hm_symm_layout *layout)
{ return (8*layout->runs_cap / (int64_t) sizeof(hm_pair_rec)) / 2; }

template <typename IdxT, int KW>
static cudaError_t launch_extract(const uint64_t *keys, const uint64_t *keys_lo, const uint16_t *cnt, int64_t n,
                                  const void *bucket, const hm_shard_tabs *tabs, int bits, int kmer,
                                  const SymmView &W, const RecordSink<KW> &R, cudaStream_t st)
{ int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms,cudaDevAttrMultiProcessorCount,dev);
  int64_t want = (R.c1-R.c0+RV_THREADS-1)/RV_THREADS;
  int     grid = (int) (want < sms ? (want > 0 ? want : 1) : sms);
  if (tabs != NULL)
    extract_sharded_kernel<IdxT,KW><<<grid,RV_THREADS,0,st>>>(64-bits,kmer,W,*tabs,R);
  else
    extract_kernel<IdxT,KW><<<grid,RV_THREADS,0,st>>>(keys,keys_lo,cnt,n,(const IdxT *) bucket,64-bits,kmer,W,R);
  return cudaGetLastError();
}

/* extract_kmer_pairs' records of the candidates [c0, c1) (c1-c0 <= hm_symm_extract_slice) of the last
 * symmetric scan on this work area, labelled by d_pixmap (uint16[HM_PLOT_CELLS] on the device): into the
 * run-head region, count in header word 3 (both read back with hm_symm_extract_fetch).  tabs != NULL: a
 * sharded table (keys .. bucket unused), Bloom hits are settled in the owning shard's arrays.          */
int hm_symm_extract(const uint64_t *d_keys, const uint64_t *d_keys_lo, const uint16_t *d_cnt, int64_t n,
                    const void *d_bucket, const hm_shard_tabs *tabs, int bits, int idx64, int kmer,
                    void *d_work, const hm_symm_layout *layout, const hm_symm_shards *shards,
                    const uint16_t *d_pixmap, int64_t c0, int64_t c1, void *stream)
{ if (kmer < HM_SYMM_MIN_KMER || kmer > HM_MAX_KMER || d_work == NULL || layout == NULL || d_pixmap == NULL ||
      c0 < 0 || c1 < c0 || c1-c0 > hm_symm_extract_slice(layout))
    return hm_set_error(HM_EINVAL,"symm_extract: bad arguments");
  if (tabs == NULL && (kmer > 32) != (d_keys_lo != NULL))
    return hm_set_error(HM_EINVAL,"symm_extract: second key word array %s for k=%d",d_keys_lo ? "given" : "missing",kmer);
  cudaStream_t st = (cudaStream_t) stream;
  SymmView W = make_view(d_work,layout,shards);
  uint8_t *b = (uint8_t *) d_work;
  unsigned long long *recs_n = W.cand_n + SY_HDR_RECORDS;
  HM_CUDA(cudaMemsetAsync(recs_n,0,sizeof(unsigned long long),st));
  if (l2_persist())
    bloom_window(st,W.bloom,sizeof(uint32_t)*(size_t) W.seg_words*(size_t) W.n_seg,1);
  cudaError_t e;
  if (kmer <= 32)
    { RecordSink<1> R = { d_pixmap,(hm_pair_rec *) (b + layout->off_runs),recs_n,W.status,
                          (unsigned long long) (2*hm_symm_extract_slice(layout)),c0,c1,kmer };
      e = idx64 ? launch_extract<uint64_t,1>(d_keys,NULL,d_cnt,n,d_bucket,tabs,bits,kmer,W,R,st)
                : launch_extract<uint32_t,1>(d_keys,NULL,d_cnt,n,d_bucket,tabs,bits,kmer,W,R,st);
    }
  else
    { RecordSink<2> R = { d_pixmap,(hm_pair_rec *) (b + layout->off_runs),recs_n,W.status,
                          (unsigned long long) (2*hm_symm_extract_slice(layout)),c0,c1,kmer };
      e = idx64 ? launch_extract<uint64_t,2>(d_keys,d_keys_lo,d_cnt,n,d_bucket,tabs,bits,kmer,W,R,st)
                : launch_extract<uint32_t,2>(d_keys,d_keys_lo,d_cnt,n,d_bucket,tabs,bits,kmer,W,R,st);
    }
  if (l2_persist())
    bloom_window(st,NULL,0,0);
  if (e != cudaSuccess)
    return hm_cuda_fail(e,tabs != NULL ? "extract_sharded_kernel" : "extract_kernel");
  return HM_OK;
}

/* after hm_symm_extract on `stream`: appends its records to the host array *buf (malloc'ed; *cap
 * records, *at in use; grown as needed) and ORs the work area's status word into *status (synchronises) */
int hm_symm_extract_fetch(const void *d_work, const hm_symm_layout *layout, hm_pair_rec **buf, int64_t *cap,
                          int64_t *at, uint64_t *status, void *stream)
{ uint64_t h[4] = {0,0,0,0};
  cudaStream_t st = (cudaStream_t) stream;
  HM_CUDA(cudaMemcpyAsync(h,(const uint8_t *) d_work + layout->off_header,sizeof(h),cudaMemcpyDeviceToHost,st));
  HM_CUDA(cudaStreamSynchronize(st));
  const int64_t room = 2*hm_symm_extract_slice(layout);
  const int64_t m    = (int64_t) h[SY_HDR_RECORDS] < room ? (int64_t) h[SY_HDR_RECORDS] : room;
  *status |= h[1];
  if (m <= 0)
    return HM_OK;
  if (*at + m > *cap)
    { int64_t nc = *cap*2 > *at+m ? *cap*2 : *at+m;
      hm_pair_rec *nb = (hm_pair_rec *) realloc(*buf,sizeof(hm_pair_rec)*(size_t) nc);
      if (nb == NULL)
        return hm_set_error(HM_ENOMEM,"out of host memory for %lld pair records",(long long) nc);
      *buf = nb; *cap = nc;
    }
  HM_CUDA(cudaMemcpyAsync(*buf + *at,(const uint8_t *) d_work + layout->off_runs,sizeof(hm_pair_rec)*(size_t) m,
                          cudaMemcpyDeviceToHost,st));
  HM_CUDA(cudaStreamSynchronize(st));
  *at += m;
  return HM_OK;
}

/* candidate count + status word of the last runscan/resolve on this work area (synchronises) */
extern "C" int hm_symm_status(const void *d_work, const hm_symm_layout *layout, uint64_t *n_cand,
                              uint64_t *status, void *stream)
{ uint64_t h[2] = {0,0};
  HM_CUDA(cudaMemcpyAsync(h,(const uint8_t *) d_work + layout->off_header,sizeof(h),cudaMemcpyDeviceToHost,
                          (cudaStream_t) stream));
  HM_CUDA(cudaStreamSynchronize((cudaStream_t) stream));
  if (n_cand != NULL) *n_cand = h[0];
  if (status != NULL) *status = h[1];
  return HM_OK;
}

/* Move a proposed shard cut to the next run boundary at or after it (a run = entries sharing their
 * first k/2 bases): pairs found by the run scan then never straddle two shards.                 */
extern "C" int hm_symm_align_cut(const uint64_t *d_keys, int64_t n, int kmer, int64_t cut, int64_t *out)
{ if (d_keys == NULL || out == NULL || cut < 0 || cut > n || kmer < HM_SYMM_MIN_KMER)
    return hm_set_error(HM_EINVAL,"hm_symm_align_cut: bad arguments");
  const int psh = 64-2*(kmer>>1);
  if (cut == 0 || cut == n)
    { *out = cut; return HM_OK; }
  uint64_t prev, buf[4096];
  HM_CUDA(cudaMemcpy(&prev,d_keys+cut-1,sizeof(uint64_t),cudaMemcpyDeviceToHost));
  while (cut < n)
    { int64_t m = n-cut < 4096 ? n-cut : 4096;
      HM_CUDA(cudaMemcpy(buf,d_keys+cut,sizeof(uint64_t)*(size_t) m,cudaMemcpyDeviceToHost));
      for (int64_t i = 0; i < m; i++)
        if (((buf[i] ^ prev) >> psh) != 0)
          { *out = cut+i; return HM_OK; }
      cut += m;
    }
  *out = n;
  return HM_OK;
}
