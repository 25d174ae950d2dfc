/*******************************************************************************************
 * hm_condition.cu -- table conditioning on the GPU: the two things the reference delegates to
 * external FastK executables before it scans (PloidyPlot.c:1381-1426):
 *
 *   trim        `Logex -T<t> '<tmp>.trim=A[<L>-]' <table>`   keep entries with count >= L
 *   symmetrise  `Symmex -T<t> -P<dir> <table> <tmp>.symx`     add the reverse complement of every
 *                                                             k-mer (same count), keep the table sorted
 *
 * FastK's tools are not part of the reference tree and are not pinned to a version (SURVEY.md
 * §8c), so this restates their documented effect, not their code: parity for THIS step is pinned
 * only against a numpy restatement in tests/ ("parity unpinned" against the real tools).  The
 * executable uses it by default and falls back to the reference's shell-outs with
 * HETMERS_EXTERNAL_CONDITIONING=1.
 *
 * Not a hot path (it runs once, before the scan): selection and sorting use CUB's device-wide
 * primitives (library code); the reverse-complement / duplicate-flag kernels are ours.
 * Duplicates (palindromes for even k, or an input that already held both strands) keep the
 * ORIGINAL entry: the concatenation puts originals first and the radix sort is stable.
 *******************************************************************************************/
#include <cub/cub.cuh>
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>

#include "hetmers_b200.h"
#include "hm_internal.h"
#include "hm_device.cuh"

__device__ __forceinline__ uint64_t rev2_64(uint64_t x)       /* reverse the 32 2-bit fields */
{ x = ((x >> 2)  & 0x3333333333333333ull) | ((x & 0x3333333333333333ull) << 2);
  x = ((x >> 4)  & 0x0F0F0F0F0F0F0F0Full) | ((x & 0x0F0F0F0F0F0F0F0Full) << 4);
  x = ((x >> 8)  & 0x00FF00FF00FF00FFull) | ((x & 0x00FF00FF00FF00FFull) << 8);
  x = ((x >> 16) & 0x0000FFFF0000FFFFull) | ((x & 0x0000FFFF0000FFFFull) << 16);
  return (x >> 32) | (x << 32);
}

__global__ void __launch_bounds__(256)
trim_flag_kernel(const uint16_t *__restrict__ cnt, int64_t n, int ethresh, uint8_t *__restrict__ flag)
{ int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n)
    flag[i] = (cnt[i] >= ethresh);
}

/* out[0,n) = table, out[n,2n) = reverse complements with the same counts */
__global__ void __launch_bounds__(256)
append_revcomp_kernel(const uint64_t *__restrict__ hi, const uint64_t *__restrict__ lo,
                      const uint16_t *__restrict__ cnt, int64_t n, int kmer,
                      uint64_t *__restrict__ ohi, uint64_t *__restrict__ olo, uint16_t *__restrict__ ocnt)
{ int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n)
    return;
  uint64_t x = hi[i];
  uint16_t c = cnt[i];
  ohi[i] = x; ocnt[i] = c; ocnt[n+i] = c;
  if (lo == NULL)
    { uint64_t r = rev2_64(~x);
      if (kmer < 32)
        r = (r & (((uint64_t) 1 << (2*kmer))-1)) << (64-2*kmer);
      ohi[n+i] = r;
    }
  else
    { uint64_t w = lo[i];
      uint64_t a = rev2_64(~w), b = rev2_64(~x);          /* the two words swap */
      int      sh = 2*(64-kmer);
      olo[i] = w;
      if (sh == 0) { ohi[n+i] = a; olo[n+i] = b; }
      else         { ohi[n+i] = (a << sh) | (b >> (64-sh)); olo[n+i] = b << sh; }
    }
}

__global__ void __launch_bounds__(256)
iota_kernel(uint32_t *__restrict__ idx, int64_t n)
{ int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) idx[i] = (uint32_t) i;
}

template <typename T>
__global__ void __launch_bounds__(256)
gather_kernel(const T *__restrict__ src, const uint32_t *__restrict__ idx, int64_t n, T *__restrict__ dst)
{ int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = src[idx[i]];
}

__global__ void __launch_bounds__(256)
first_of_run_kernel(const uint64_t *__restrict__ hi, const uint64_t *__restrict__ lo, int64_t n,
                    uint8_t *__restrict__ flag)
{ int64_t i = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n)
    flag[i] = (i == 0) || hi[i] != hi[i-1] || (lo != NULL && lo[i] != lo[i-1]);
}

#define GRID(n) ((unsigned) (((n)+255)/256))

template <typename T>
static int select_flagged(const T *in, const uint8_t *flag, T *out, int64_t n, int64_t *d_nsel,
                          void **tmp, size_t *tmp_bytes, cudaStream_t st)
{ size_t need = 0;
  HM_CUDA(cub::DeviceSelect::Flagged(NULL,need,in,flag,out,d_nsel,n,st));
  if (need > *tmp_bytes)
    { if (*tmp) cudaFree(*tmp);
      *tmp = NULL; *tmp_bytes = 0;
      HM_CUDA(cudaMalloc(tmp,need));
      *tmp_bytes = need;
    }
  HM_CUDA(cub::DeviceSelect::Flagged(*tmp,need,in,flag,out,d_nsel,n,st));
  return HM_OK;
}

template <typename K, typename V>
static int sort_pairs(const K *kin, K *kout, const V *vin, V *vout, int64_t n, int begin_bit, int end_bit,
                      void **tmp, size_t *tmp_bytes, cudaStream_t st)
{ size_t need = 0;
  HM_CUDA(cub::DeviceRadixSort::SortPairs(NULL,need,kin,kout,vin,vout,n,begin_bit,end_bit,st));
  if (need > *tmp_bytes)
    { if (*tmp) cudaFree(*tmp);
      *tmp = NULL; *tmp_bytes = 0;
      HM_CUDA(cudaMalloc(tmp,need));
      *tmp_bytes = need;
    }
  HM_CUDA(cub::DeviceRadixSort::SortPairs(*tmp,need,kin,kout,vin,vout,n,begin_bit,end_bit,st));
  return HM_OK;
}

/* device allocations of one conditioning call: everything still registered is freed on return */
struct Scratch
  { void *p[32];
    int   n;
    Scratch() : n(0) {}
    ~Scratch() { for (int k = 0; k < n; k++) cudaFree(p[k]); }
    template <typename T> cudaError_t alloc(T **q, size_t bytes)
    { cudaError_t e = cudaMalloc((void **) q,bytes);
      if (e == cudaSuccess && n < 32) p[n++] = (void *) *q;
      return e;
    }
    void release(void *q)                      /* hand q to the caller (or it was freed by hand) */
    { for (int k = 0; k < n; k++)
        if (p[k] == q) { p[k] = p[--n]; return; }
    }
    void free_now(void *q) { if (q != NULL) { release(q); cudaFree(q); } }
  };

/* Sort (h0, l0, c0)[0,m) by key (stable: of equal keys the one nearer the front wins) and keep the
 * first entry of every run of equal keys, back in h0 / l0 / c0; *nsel = entries kept.  l0 is NULL for
 * k <= 32.  The second buffers come from S and are released before returning.                     */
static int sort_unique(int kmer, uint64_t *h0, uint64_t *l0, uint16_t *c0, int64_t m, Scratch &S,
                       int64_t *d_nsel, int64_t *nsel, void **tmp, size_t *tmp_bytes, cudaStream_t st)
{ const int two = (l0 != NULL);
  uint64_t *h1 = NULL, *l1 = NULL;
  uint16_t *c1 = NULL;
  uint8_t  *flag = NULL;
  int       rc;
  HM_CUDA(S.alloc(&h1,sizeof(uint64_t)*(size_t) (m+1)));
  HM_CUDA(S.alloc(&c1,sizeof(uint16_t)*(size_t) (m+1)));
  if (two)
    HM_CUDA(S.alloc(&l1,sizeof(uint64_t)*(size_t) (m+1)));
  if (!two)
    { int bb = kmer < 32 ? 64-2*kmer : 0;
      if ((rc = sort_pairs(h0,h1,c0,c1,m,bb,64,tmp,tmp_bytes,st)) != HM_OK) return rc;
    }
  else
    { uint32_t *i0 = NULL, *i1 = NULL;
      HM_CUDA(S.alloc(&i0,sizeof(uint32_t)*(size_t) m));
      HM_CUDA(S.alloc(&i1,sizeof(uint32_t)*(size_t) m));
      iota_kernel<<<GRID(m),256,0,st>>>(i0,m);
      int bb = kmer < 64 ? 128-2*kmer : 0;
      /* least significant word first, then a stable sort on the most significant word */
      if ((rc = sort_pairs(l0,l1,i0,i1,m,bb,64,tmp,tmp_bytes,st)) != HM_OK) return rc;
      gather_kernel<uint64_t><<<GRID(m),256,0,st>>>(h0,i1,m,h1);          /* hi in lo-order   */
      if ((rc = sort_pairs(h1,l1,i1,i0,m,0,64,tmp,tmp_bytes,st)) != HM_OK) return rc;
      /* l1 = sorted hi, i0 = final permutation */
      gather_kernel<uint64_t><<<GRID(m),256,0,st>>>(l0,i0,m,h1);          /* h1 := lo sorted  */
      gather_kernel<uint16_t><<<GRID(m),256,0,st>>>(c0,i0,m,c1);
      /* arrange as (h1 = hi, l1 = lo) */
      uint64_t *t = h1; h1 = l1; l1 = t;
      HM_CUDA(cudaStreamSynchronize(st));
      S.free_now(i0); S.free_now(i1);
    }
  /* unique (first of every run of equal keys wins) back into h0/l0/c0 */
  HM_CUDA(S.alloc(&flag,(size_t) m));
  first_of_run_kernel<<<GRID(m),256,0,st>>>(h1,two ? l1 : NULL,m,flag);
  if ((rc = select_flagged(h1,flag,h0,m,d_nsel,tmp,tmp_bytes,st)) != HM_OK) return rc;
  if (two && (rc = select_flagged(l1,flag,l0,m,d_nsel,tmp,tmp_bytes,st)) != HM_OK) return rc;
  if ((rc = select_flagged(c1,flag,c0,m,d_nsel,tmp,tmp_bytes,st)) != HM_OK) return rc;
  HM_CUDA(cudaMemcpyAsync(nsel,d_nsel,sizeof(int64_t),cudaMemcpyDeviceToHost,st));
  HM_CUDA(cudaStreamSynchronize(st));
  S.free_now(flag); S.free_now(h1); S.free_now(l1); S.free_now(c1);
  return HM_OK;
}

/* Replace (*pk, *pl, *pc, *pn) by the conditioned table (new cudaMalloc'ed arrays with one spare
 * element).  *pl is NULL for k <= 32.  The caller's arrays are freed and replaced only when the whole
 * call has succeeded; on any failure they are untouched and every temporary is released.        */
int hm_condition_arrays(int kmer, int ethresh, int do_trim, int do_symm,
                        uint64_t **pk, uint64_t **pl, uint16_t **pc, int64_t *pn, cudaStream_t st)
{ int64_t   n = *pn;
  const int two = (*pl != NULL);
  Scratch   S;
  void     *tmp = NULL;                        /* CUB temporary storage (grown on demand) */
  size_t    tmp_bytes = 0;
  uint8_t  *flag = NULL;
  int64_t  *d_nsel = NULL, nsel = 0;
  int       rc = HM_OK;
  /* current table: the caller's arrays, or ours once a stage has produced new ones */
  uint64_t *ck = *pk, *cl = *pl;
  uint16_t *cc = *pc;
  int       own = 0;

  if (do_symm && two && 2*n >= 0xFFFFFFF0ll)   /* before anything is allocated or touched */
    return hm_set_error(HM_EUNSUPPORTED,"symmetrising %lld entries of k=%d needs 64-bit sort indices",
                        (long long) n,kmer);
#define CK(call) do { cudaError_t _e = (call); if (_e != cudaSuccess) { if (tmp) cudaFree(tmp); return hm_cuda_fail(_e,#call); } } while (0)
#define RC(call) do { if ((rc = (call)) != HM_OK) { if (tmp) cudaFree(tmp); return rc; } } while (0)
  CK(S.alloc(&d_nsel,sizeof(int64_t)));

  if (do_trim && n > 0)
    { uint64_t *k2 = NULL, *l2 = NULL; uint16_t *c2 = NULL;
      CK(S.alloc(&flag,(size_t) n));
      CK(S.alloc(&k2,sizeof(uint64_t)*(size_t) (n+1)));
      CK(S.alloc(&c2,sizeof(uint16_t)*(size_t) (n+1)));
      if (two) CK(S.alloc(&l2,sizeof(uint64_t)*(size_t) (n+1)));
      trim_flag_kernel<<<GRID(n),256,0,st>>>(cc,n,ethresh,flag);
      RC(select_flagged(ck,flag,k2,n,d_nsel,&tmp,&tmp_bytes,st));
      if (two) RC(select_flagged(cl,flag,l2,n,d_nsel,&tmp,&tmp_bytes,st));
      RC(select_flagged(cc,flag,c2,n,d_nsel,&tmp,&tmp_bytes,st));
      CK(cudaMemcpyAsync(&nsel,d_nsel,sizeof(int64_t),cudaMemcpyDeviceToHost,st));
      CK(cudaStreamSynchronize(st));
      S.free_now(flag); flag = NULL;
      ck = k2; cc = c2; cl = l2; n = nsel; own = 1;
    }

  if (do_symm && n > 0)
    { int64_t   m = 2*n;
      uint64_t *h0 = NULL, *l0 = NULL;
      uint16_t *c0 = NULL;
      CK(S.alloc(&h0,sizeof(uint64_t)*(size_t) (m+1)));
      CK(S.alloc(&c0,sizeof(uint16_t)*(size_t) (m+1)));
      if (two)
        CK(S.alloc(&l0,sizeof(uint64_t)*(size_t) (m+1)));
      append_revcomp_kernel<<<GRID(n),256,0,st>>>(ck,cl,cc,n,kmer,h0,l0,c0);
      if (own)                                       /* the trimmed intermediate is ours: drop it now */
        { CK(cudaStreamSynchronize(st));
          S.free_now(ck); S.free_now(cc); S.free_now(cl);
          ck = NULL; cc = NULL; cl = NULL; own = 0;
        }
      RC(sort_unique(kmer,h0,l0,c0,m,S,d_nsel,&nsel,&tmp,&tmp_bytes,st));
      ck = h0; cc = c0; cl = l0; n = nsel; own = 1;
    }

  CK(cudaStreamSynchronize(st));
#undef CK
#undef RC
  if (tmp) cudaFree(tmp);
  if (own)                                           /* success: swap the new table in */
    { S.release(ck); S.release(cc); if (cl) S.release(cl);
      cudaFree(*pk); cudaFree(*pc); if (*pl) cudaFree(*pl);
      *pk = ck; *pc = cc; *pl = cl;
    }
  *pn = n;
  return HM_OK;
}

/* Sort + deduplicate a table held in (k, l, c)[0,*pn) (cudaMalloc'ed; l NULL for k <= 32) in place:
 * what each shard of a sharded table does with the entries it received (originals ahead of reverse
 * complements, so that of two equal keys the original survives, as in hm_condition_arrays).        */
int hm_sort_unique_arrays(int kmer, uint64_t *k, uint64_t *l, uint16_t *c, int64_t *pn, cudaStream_t st)
{ int64_t m = *pn, nsel = 0, *d_nsel = NULL;
  void   *tmp = NULL;
  size_t  tmp_bytes = 0;
  if (m <= 0)
    return HM_OK;
  if (l != NULL && m >= 0xFFFFFFF0ll)
    return hm_set_error(HM_EUNSUPPORTED,"a shard of %lld entries of k=%d needs 64-bit sort indices",(long long) m,kmer);
  Scratch S;
  HM_CUDA(S.alloc(&d_nsel,sizeof(int64_t)));
  int rc = sort_unique(kmer,k,l,c,m,S,d_nsel,&nsel,&tmp,&tmp_bytes,st);
  if (tmp) cudaFree(tmp);
  if (rc == HM_OK)
    *pn = nsel;
  return rc;
}

/* ---- sharded placement: every entry to the shard that owns its key range ----------------------
 * Shard r owns the keys whose first word is in [cut[r], cut[r+1]) (cut[0] = 0, ties to the higher
 * shard, the rule owner_of() of hm_symm.cu applies); the cuts sit on boundaries of the first k/2
 * bases, so no run of the table is split.  One thread per entry: trim by count, the entry and (when
 * symmetrising) its reverse complement go to slot 2*owner + (0 original | 1 reverse complement).
 * d_cursor[2*S]: count mode (okeys == NULL) adds the number of entries per slot; fill mode starts
 * from each slot's offset in the outbox and writes the entries there (order inside a slot is free:
 * the owner sorts).  One atomic per warp and slot.                                                */
struct PartCuts { uint64_t c[HM_MAX_SHARDS]; };

template <int KW>
__global__ void __launch_bounds__(256)
partition_kernel(const uint64_t *__restrict__ keys, const uint64_t *__restrict__ keys_lo,
                 const uint16_t *__restrict__ cnt, int64_t n, int kmer, int ethresh, int do_trim, int do_symm,
                 const PartCuts C, int S, unsigned long long *__restrict__ cursor,
                 uint64_t *__restrict__ okeys, uint64_t *__restrict__ okeys_lo, uint16_t *__restrict__ ocnt)
{ const unsigned FULL = 0xffffffffu;
  const int      lane = threadIdx.x & 31;
  const unsigned lt   = (1u << lane) - 1;
  const int64_t  i    = (int64_t) blockIdx.x * blockDim.x + threadIdx.x;
  uint64_t x = 0, xl = 0;
  uint16_t c = 0;
  bool keep = false;
  if (i < n)
    { x = keys[i]; c = cnt[i];
      if (KW == 2) xl = keys_lo[i];
      keep = !do_trim || (int) c >= ethresh;
    }
  for (int kind = 0; kind < 2; kind++)
    { uint64_t y = x, yl = xl;
      if (kind == 1)
        revcomp_kmer<KW>(x,xl,kmer,y,yl);
      const bool act = keep && (kind == 0 || do_symm);
      int slot = -1;
      if (act)
        { int o = 0;
#pragma unroll
          for (int r = 1; r < HM_MAX_SHARDS; r++)            /* (a fixed trip count keeps C in the parameter bank) */
            if (r < S)
              o += (y >= C.c[r]);
          slot = 2*o + kind;
        }
      const unsigned peers  = __match_any_sync(FULL,slot);
      const int      leader = __ffs(peers)-1;
      unsigned long long base = 0;
      if (act && lane == leader)
        base = atomicAdd(cursor+slot,(unsigned long long) __popc(peers));
      base = __shfl_sync(FULL,base,leader);
      if (act && okeys != NULL)
        { const unsigned long long at = base + __popc(peers & lt);
          okeys[at] = y; ocnt[at] = c;
          if (KW == 2) okeys_lo[at] = yl;
        }
    }
}

int hm_k_partition(const uint64_t *keys, const uint64_t *keys_lo, const uint16_t *cnt, int64_t n, int kmer,
                   int ethresh, int do_trim, int do_symm, const uint64_t *cut, int n_shards,
                   unsigned long long *d_cursor, uint64_t *okeys, uint64_t *okeys_lo, uint16_t *ocnt,
                   cudaStream_t st)
{ if (n_shards < 1 || n_shards > HM_MAX_SHARDS || kmer < 1 || kmer > HM_MAX_KMER || (kmer > 32) != (keys_lo != NULL))
    return hm_set_error(HM_EINVAL,"partition: bad arguments");
  if (n <= 0)
    return HM_OK;
  PartCuts C;
  memset(&C,0,sizeof(C));
  for (int r = 0; r < n_shards; r++) C.c[r] = cut[r];
  if (kmer <= 32)
    partition_kernel<1><<<GRID(n),256,0,st>>>(keys,NULL,cnt,n,kmer,ethresh,do_trim,do_symm,C,n_shards,d_cursor,okeys,NULL,ocnt);
  else
    partition_kernel<2><<<GRID(n),256,0,st>>>(keys,keys_lo,cnt,n,kmer,ethresh,do_trim,do_symm,C,n_shards,d_cursor,okeys,okeys_lo,ocnt);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess)
    return hm_cuda_fail(e,"partition_kernel");
  return HM_OK;
}
