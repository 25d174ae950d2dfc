/*******************************************************************************************
 * hetmers_main.c -- the drop-in `hetmers` executable (plain C host; all compute is CUDA behind
 * include/hetmers_b200.h).  Same process boundary as the reference binary that smudgeplot's CLI
 * spawns (/root/reference/src/smudgeplot/cli.py:57-72,348-361):
 *
 *     hetmers [-v] [-T<int(4)>] [-P<dir(/tmp)>] [-o<output>] [-e<int(4)>] <source>[.ktab]
 *
 * mirrors main() of /root/reference/src/lib/PloidyPlot.c:1232-1630: argv grammar and messages
 * (gene_core.h:32-56 ARG_* macros), default output root, the "Found het-table" prompt, the
 * trimmed/symmetric examination (un-conditioned tables are trimmed / symmetrised on the GPU;
 * HETMERS_EXTERNAL_CONDITIONING=1 restores the reference's shell-outs to FastK's Logex/Symmex/Fastrm), the verbose
 * lines, the .smu format and the exit codes.  -T is accepted (and clamped to 64 with the same
 * warning) but the GPU count comes from HETMERS_GPUS (default 1; "all" = every visible GPU).
 * There is no CPU fallback: without a CUDA device the program fails with exit 1.
 *******************************************************************************************/
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <stdarg.h>
#include <unistd.h>
#include <strings.h>

#include <time.h>

#include "hetmers_b200.h"

static double wall_ms(void)
{ struct timespec ts;
  clock_gettime(CLOCK_MONOTONIC,&ts);
  return ts.tv_sec*1e3 + ts.tv_nsec*1e-6;
}

/* Compiled twice: plain -> `hetmers` (PloidyPlot.c), with -DEXTRACT_PAIRS -> `extract_kmer_pairs`
 * (src/lib/PloidyList.c:1207-1583: same search, but the isolated pairs whose (covB,covA) pixel is
 * labelled in <smudges>.sma are written as sequences to <out>.<a>A<b>B.txt instead of counted). */
#ifdef EXTRACT_PAIRS
static const char *Prog_Name = "extract_kmer_pairs";

static const char *Usage[] = { " [-v] [-T<int(4)>] [-P<dir(/tmp)>]",
                               " [-o<output>] [-e<int(4)>] <source>[.ktab] <smudges>[.sma]" };
#define NPOSITIONAL 3

typedef struct { int a, b; FILE *f; } Smudge;
#else
static const char *Prog_Name = "hetmers";

static const char *Usage[] = { " [-v] [-T<int(4)>] [-P<dir(/tmp)>]",
                               " [-o<output>] [-e<int(4)>] <source>[.ktab]" };
#define NPOSITIONAL 2
#endif

static int positive_arg(const char *arg, const char *what)      /* ARG_POSITIVE, gene_core.h:46-56 */
{ char *eptr;
  long  v = strtol(arg+2,&eptr,10);
  if (*eptr != '\0' || arg[2] == '\0')
    { fprintf(stderr,"%s: -%c '%s' argument is not an integer\n",Prog_Name,arg[1],arg+2);
      exit (1);
    }
  if (v <= 0)
    { fprintf(stderr,"%s: %s must be positive (%d)\n",Prog_Name,what,(int) v);
      exit (1);
    }
  return ((int) v);
}

static void systemx(const char *command)                         /* SystemX, gene_core.c:19-24 */
{ if (system(command) != 0)
    { fprintf(stderr,"%s: Command '%s' failed\n",Prog_Name,command);
      exit (1);
    }
}

/* format a command line into `buf` (sized by the caller for the longest one) and run it */
static void run_tool(char *buf, const char *fmt, ...)
{ va_list ap;
  va_start(ap,fmt);
  vsprintf(buf,fmt,ap);
  va_end(ap);
  systemx(buf);
}

/* the reference's -v progress line for a conditioning step: 't' = trim, 's' = symmetrise */
static void announce_step(int verbose, int step, int was_trimmed, int ethresh)
{ if (!verbose)
    return;
  if (step == 't')
    fprintf(stderr,"\n  Trimming k-mers in table with count < %d\n",ethresh);
  else
    fprintf(stderr,was_trimmed ? "\n  Making table symmetric\n" : "\n  Making trimmed table symmetric\n");
  fflush(stderr);
}

static void die_hm(void)
{ fprintf(stderr,"%s: %s\n",Prog_Name,hm_last_error());
  exit (1);
}

#ifdef EXTRACT_PAIRS

/* The smudges named in the .sma file, in order of first appearance; label s+1 in the pixel map
 * refers to set->v[s] (the reference keeps the same numbering in its PLOT array,
 * PloidyList.c:1313-1350).                                                                    */
typedef struct { Smudge *v; int n, cap; } SmudgeSet;

static int smudge_label(SmudgeSet *set, int a, int b, const char *out_root)
{ int s;
  for (s = 0; s < set->n; s++)
    if (set->v[s].a == a && set->v[s].b == b)
      return (s+1);
  if (set->n == set->cap)
    { set->cap += 100;
      set->v = realloc(set->v,set->cap*sizeof(Smudge));
      if (set->v == NULL)
        exit (1);
    }
  { char *name = malloc(strlen(out_root)+64);
    sprintf(name,"%s.%dA%dB.txt",out_root,a,b);
    set->v[s].a = a;
    set->v[s].b = b;
    set->v[s].f = fopen(name,"w");                  /* created even if no pair ends up in it */
    free(name);
  }
  if (set->v[s].f == NULL)
    { fprintf(stderr,"%s: Cannot open smudge file %s.%dA%dB.txt\n",Prog_Name,out_root,a,b);
      exit (1);
    }
  set->n += 1;
  return (s+1);
}

/* <arg>[.sma]: a header line, then "covB covA freq <a>A<b>B" per annotated pixel (written by
 * `smudgeplot all`, cli.py:451-456).  Same acceptance rules and messages as PloidyList.c:1300-1335. */
static void read_sma(const char *arg, const char *out_root, uint16_t *pixmap, SmudgeSet *set)
{ size_t n = strlen(arg);
  char  *root = strdup(arg), *name, line[1000];
  FILE  *f;
  int    covb, cova, a, b;

  if (n > 4 && strcasecmp(root+n-4,".sma") == 0)
    root[n-4] = '\0';
  name = malloc(strlen(root)+8);
  sprintf(name,"%s.sma",root);
  f = fopen(name,"r");
  if (f == NULL)
    { fprintf(stderr,"\n%s: Could not open smudge file %s.sma",Prog_Name,root);
      exit (1);
    }
  if (fgets(line,sizeof(line),f) != NULL)              /* the header is skipped unseen */
    while (fgets(line,sizeof(line),f) != NULL)
      { if (sscanf(line," %d %d %*d %dA%dB",&covb,&cova,&a,&b) != 4)
          { fprintf(stderr,"%s: Cannot parse line '%s'\n",Prog_Name,line);
            exit (1);
          }
        if (a <= 0 || b <= 0 || a < b)
          { fprintf(stderr,"%s: %dA%dB is not a valid smudge label'\n",Prog_Name,a,b);
            exit (1);
          }
        if (covb < 0 || covb > HM_FMAX || cova < covb || covb+cova > HM_SMAX)
          { fprintf(stderr,"%s: (%d,%d) is not a valid pixel coordinate\n",Prog_Name,covb,cova);
            exit (1);
          }
        pixmap[(covb+cova)*HM_PLOT_W+covb] = (uint16_t) smudge_label(set,a,b,out_root);
      }
  fclose(f);
  free(name);
  free(root);
}

#endif

/* How many GPUs HETMERS_GPUS asks for (0 = "all").  Called before the first CUDA call: a process
 * that will use g GPUs of an 8-GPU box need not pay for the driver initialising the other 8-g, so
 * CUDA_VISIBLE_DEVICES is narrowed to the first g visible devices, and CUDA start-up (driver +
 * context creation, ~0.5 s) then runs on a background thread while the table files are opened.  */
static int wanted_gpus(void)
{ const char *g = getenv("HETMERS_GPUS");
  int n = 1;
  if (g != NULL && *g != '\0')
    { if (strcasecmp(g,"all") == 0)
        return 0;
      n = atoi(g);
      if (n < 1) n = 1;
      if (n > 16) n = 16;
    }
  return n;
}

static void start_cuda_early(void)
{ int   want = wanted_gpus(), i;
  const char *vis = getenv("CUDA_VISIBLE_DEVICES");
  if (want > 0)
    { char buf[512];
      if (vis == NULL || *vis == '\0')
        { char *o = buf;
          for (i = 0; i < want; i++)
            o += sprintf(o,i ? ",%d" : "%d",i);
          setenv("CUDA_VISIBLE_DEVICES",buf,1);
        }
      else if (strlen(vis) < sizeof(buf))
        { int commas = 0;
          strcpy(buf,vis);
          for (i = 0; buf[i] != '\0'; i++)
            if (buf[i] == ',' && ++commas == want)
              { buf[i] = '\0'; break; }
          setenv("CUDA_VISIBLE_DEVICES",buf,1);
        }
    }
  hm_prewarm(want);
}

static int pick_gpus(int *devs)
{ int ngpu = 1, navail = hm_device_count(), i;
  const char *g = getenv("HETMERS_GPUS");

  if (navail < 1)
    { fprintf(stderr,"%s: no CUDA device is visible (this hetmers is GPU-only)\n",Prog_Name);
      exit (1);
    }
  if (g != NULL && *g != '\0')
    { if (strcasecmp(g,"all") == 0)
        ngpu = navail;
      else
        ngpu = atoi(g);
      if (ngpu < 1) ngpu = 1;
      if (ngpu > navail)
        { fprintf(stderr,"%s: Warning, only %d GPUs are visible\n",Prog_Name,navail);
          ngpu = navail;
        }
    }
  if (ngpu > 16) ngpu = 16;
  for (i = 0; i < ngpu; i++)
    devs[i] = i;
  return (ngpu);
}

/* Placement of the table on the ngpu devices (hm_plan_placement, from what each device has free):
 * a full replica on every GPU whenever one fits, else one shard per GPU, else neither.           */
static int plan_placement(const hm_host_table *t, const int *devs, int ngpu, int do_symm, hm_scan *held)
{ int64_t fr[16];
  for (int g = 0; g < ngpu; g++)
    { if (hm_device_free_bytes(devs[g],&fr[g]) != HM_OK)
        die_hm();
      if (held != NULL)               /* what the loaded table takes is free again if it is re-placed */
        { int64_t b = 0;
          if (hm_scan_shard_info(held,g,NULL,NULL,NULL,&b) != HM_OK)
            die_hm();
          fr[g] += b;
        }
    }
  int r = hm_plan_placement(t->kmer,t->nels,do_symm,ngpu,fr,NULL,NULL);
  if (r < 0)
    die_hm();
  return r;
}

static void does_not_fit(const hm_host_table *t, int ngpu)
{ fprintf(stderr,"%s: a table of %lld k-mers does not fit on %d GPUs, not even sharded over them; "
                 "set HETMERS_GPUS to use more GPUs\n",Prog_Name,(long long) t->nels,ngpu);
  exit (1);
}

int main(int argc, char *argv[])
{ int    VERBOSE = 0, NTHREADS = 4, ETHRESH = 4;
  const char *SORT_PATH = "/tmp";
  char  *OUT = NULL, *SRC;
  const char *troot = "";      /* the reference's mktemp("._SPAIR.XXXX") fails on glibc and
                                  leaves an empty root (PloidyPlot.c:1093,1313; SURVEY App. C7) */
  int    i, j, k;
  int    flags[128];

  for (i = 0; i < 128; i++)
    flags[i] = 0;

  j = 1;
  for (i = 1; i < argc; i++)
    if (argv[i][0] == '-')
      switch (argv[i][1])
      { default:                                                  /* ARG_FLAGS("vklfs") */
          for (k = 1; argv[i][k] != '\0'; k++)
            { if (strchr("vklfs",argv[i][k]) == NULL)
                { fprintf(stderr,"%s: -%c is an illegal option\n",Prog_Name,argv[i][k]);
                  exit (1);
                }
              flags[(int) argv[i][k]] = 1;
            }
          break;
        case 'e':
          ETHRESH = positive_arg(argv[i],"Error-mer threshold");
          break;
        case 'o':
          free(OUT);
          OUT = strdup(argv[i]+2);
          if (OUT == NULL)
            exit (1);
          break;
        case 'P':
          SORT_PATH = argv[i]+2;
          break;
        case 'T':
          NTHREADS = positive_arg(argv[i],"Number of threads");
          if (NTHREADS > 64)
            { fprintf(stderr,"%s: Warning, only 64 threads will be used\n",Prog_Name);
              NTHREADS = 64;
            }
          break;
      }
    else
      argv[j++] = argv[i];
  argc = j;

  VERBOSE = flags['v'];

  if (argc != NPOSITIONAL)
    { fprintf(stderr,"\nUsage: %s %s\n",Prog_Name,Usage[0]);
      fprintf(stderr,"       %*s %s\n",(int) strlen(Prog_Name),"",Usage[1]);
      fprintf(stderr,"\n");
      fprintf(stderr,"      -o: root name for output table\n");
      fprintf(stderr,"            default is root of <source> argument\n");
      fprintf(stderr,"\n");
      fprintf(stderr,"      -e: count threshold below which k-mers are considered erroneous\n");
      fprintf(stderr,"      -v: verbose mode\n");
      fprintf(stderr,"      -T: number of threads to use\n");
      fprintf(stderr,"      -P: Place all temporary files in directory -P.\n");
      exit (1);
    }

  SRC = argv[1];
  if (OUT == NULL)                                   /* PathnRoot(src,".ktab"), gene_core.c:116-135 */
    { size_t n = strlen(SRC);
      OUT = strdup(SRC);
      if (OUT == NULL)
        exit (1);
      if (n > 5 && strcasecmp(SRC+n-5,".ktab") == 0)
        OUT[n-5] = '\0';
    }

#ifdef EXTRACT_PAIRS
  //  The annotated smudge file: pixel -> label map and one output file per label

  uint16_t *PIXMAP = calloc(HM_PLOT_CELLS,sizeof(uint16_t));
  SmudgeSet SM = { NULL, 0, 0 };
  if (PIXMAP == NULL)
    exit (1);
  read_sma(argv[2],OUT,PIXMAP,&SM);
#else
  //  If appropriately named het-mer table found then ask if reuse (PloidyPlot.c:1318-1337)

  { char *smu = malloc(strlen(OUT)+8);
    FILE *f;
    int   a;

    sprintf(smu,"%s.smu",OUT);
    f = fopen(smu,"r");
    free(smu);
    if (f != NULL)
      { int bypass = 0;
        fprintf(stdout,"\n  Found het-table %s.smu, use it? ",OUT);
        fflush(stdout);
        while ((a = getc(stdin)) != '\n')
          { if (a == EOF)       /* the reference spins for ever here; we treat EOF as "no" */
              break;
            if (a == 'y' || a == 'Y')
              bypass = 1;
          }
        if (bypass)
          { fprintf(stderr,"\n  Using the found het-table, done\n");
            fclose(f);
            exit (0);
          }
        fclose(f);
      }
  }

#endif

  //  Open input table and see if it needs conditioning (PloidyPlot.c:1341-1426)

  hm_table *T;
  hm_scan  *S;
  char     *input = NULL;
  int       ngpu, devs[16], place = HM_PLACE_REPLICA;
  double    t_start = wall_ms(), t_open, t_load, t_exam, t_scan;

  start_cuda_early();            /* background: nothing below waits for it before hm_device_count() */

  { char *command, *tname;
    int   symm, trim;

    tname   = malloc(strlen(SRC) + strlen(troot) + 10);
    command = malloc(strlen(SRC) + strlen(troot) + strlen(SORT_PATH) + 100);
    if (tname == NULL || command == NULL)
      exit (1);

    if (hm_table_open(SRC,&T) != HM_OK)
      { if (strncmp(hm_last_error(),"Cannot open",11) == 0)
          fprintf(stderr,"%s: Cannot open k-mer table %s\n",Prog_Name,SRC);
        else
          fprintf(stderr,"%s: %s\n",Prog_Name,hm_last_error());
        exit (1);
      }
    t_open = wall_ms();
    ngpu = pick_gpus(devs);        /* after the table is known to exist: same first error as the reference */
    hm_set_io_threads(NTHREADS);   /* -T = host threads staging the part files towards the GPU */
    if (hm_table_view(T)->nels < 2)
      { fprintf(stderr,"%s: k-mer table %s has fewer than 2 entries\n",Prog_Name,SRC);
        exit (1);
      }
    place = plan_placement(hm_table_view(T),devs,ngpu,0,NULL);
    if (place == HM_PLACE_NOFIT && ngpu > 1)
      does_not_fit(hm_table_view(T),ngpu);
    if (place == HM_PLACE_SHARDED)
      { if (hm_scan_create_sharded(hm_table_view(T),devs,ngpu,&S) != HM_OK)
          die_hm();
      }
    else if (hm_scan_create(hm_table_view(T),devs,ngpu,&S) != HM_OK)
      die_hm();
    t_load = wall_ms();
    if (hm_scan_examine(S,ETHRESH,&trim,&symm) != HM_OK)
      die_hm();
    t_exam = wall_ms();

    if (VERBOSE)
      { fprintf(stderr,"\n  The input table is");
        if (trim)
          if (symm)
            fprintf(stderr," trimmed and symmetric\n");
          else
            fprintf(stderr," trimmed but not symmetric\n");
        else
          if (symm)
            fprintf(stderr," untrimmed yet symmetric\n");
          else
            fprintf(stderr," untrimmed and not symmetric\n");
      }

    sprintf(tname,"%s",SRC);

    if (trim && symm)
      { free(command);                 //  nothing to do: the table is scanned as it is
        free(tname);
      }
    else if (getenv("HETMERS_EXTERNAL_CONDITIONING") == NULL)
      { //  Condition the table where it already is -- on the GPU -- instead of shelling out to
        //  FastK's Logex / Symmex and re-reading their output (same progress lines with -v)
        int64_t nn;
        if (!trim) announce_step(VERBOSE,'t',trim,ETHRESH);
        if (!symm) announce_step(VERBOSE,'s',trim,ETHRESH);
        if (!symm)                      /* symmetrising doubles the table: placed again for that */
          { int p2 = plan_placement(hm_table_view(T),devs,ngpu,1,S);
            if (p2 == HM_PLACE_NOFIT && ngpu > 1)
              does_not_fit(hm_table_view(T),ngpu);
            if (p2 == HM_PLACE_SHARDED && place == HM_PLACE_REPLICA)
              { hm_scan_destroy(S);
                place = HM_PLACE_SHARDED;
                if (hm_scan_create_sharded(hm_table_view(T),devs,ngpu,&S) != HM_OK)
                  die_hm();
              }
          }
        if (hm_scan_condition(S,ETHRESH,!trim,!symm,&nn) != HM_OK)
          die_hm();
        if (nn < 2)
          { fprintf(stderr,"%s: fewer than 2 k-mers are left after conditioning\n",Prog_Name);
            exit (1);
          }
        free(command);
        free(tname);
      }
    else
      { //  Compatibility shim (HETMERS_EXTERNAL_CONDITIONING=1): hand the table to FastK's own tools as the
        //  reference does (PloidyPlot.c:1381-1426) -- same command lines, so the same files appear -- and load
        //  whatever they leave behind.
        const char *made = NULL;
        if (!trim)
          { announce_step(VERBOSE,'t',trim,ETHRESH);
            run_tool(command,"Logex -T%d '%s.trim=A[%d-]' %s",NTHREADS,troot,ETHRESH,tname);
            made = ".trim";
          }
        if (!symm)
          { char *from = malloc(strlen(tname)+strlen(troot)+10);
            announce_step(VERBOSE,'s',trim,ETHRESH);
            if (from == NULL)
              exit (1);
            if (made != NULL) sprintf(from,"%s%s",troot,made);
            else              strcpy(from,tname);
            run_tool(command,"Symmex -T%d -P%s %s %s.symx",NTHREADS,SORT_PATH,from,troot);
            if (made != NULL)
              run_tool(command,"Fastrm %s.trim",troot);
            free(from);
            made = ".symx";
          }
        free(command);
        sprintf(tname,"%s%s",troot,made);
        input = tname;
        hm_scan_destroy(S);
        hm_table_close(T);
        if (hm_table_open(input,&T) != HM_OK)
          { fprintf(stderr,"%s: Cannot open k-mer table %s\n",Prog_Name,input);
            exit (1);
          }
        place = plan_placement(hm_table_view(T),devs,ngpu,0,NULL);
        if (place == HM_PLACE_SHARDED)
          { if (hm_scan_create_sharded(hm_table_view(T),devs,ngpu,&S) != HM_OK)
              die_hm();
          }
        else if (hm_scan_create(hm_table_view(T),devs,ngpu,&S) != HM_OK)
          die_hm();
      }
  }

  if (VERBOSE)
    { fprintf(stderr,"\n  Starting to count covariant pairs\n");
      fflush(stderr);
    }

  int64_t      *PLOT = malloc(sizeof(int64_t)*HM_PLOT_CELLS);
  hm_scan_stats stats;
  if (PLOT == NULL)
    { fprintf(stderr,"%s: Out of memory (Allocating plot)\n",Prog_Name);
      exit (1);
    }
  if (hm_scan_run(S,PLOT,&stats) != HM_OK)
    die_hm();
  t_scan = wall_ms();
#ifdef EXTRACT_PAIRS
  //  The isolated pairs of the labelled pixels, by the route the scan took: from the symmetric scan's
  //  candidates (any placement, sharded included) or from the direct passes
  hm_pair_rec     *REC = NULL;
  int64_t          NREC = 0;
  int              KMER = hm_table_view(T)->kmer;
  hm_extract_stats XST;
  double           t_extract = wall_ms();
  if (hm_scan_extract_path(S,HM_PATH_AUTO,PIXMAP,&REC,&NREC,&XST) != HM_OK)
    die_hm();
  t_extract = wall_ms()-t_extract;
#endif
  //  (the device-resident table is not torn down: the process is about to end, and destroying the CUDA
  //   context by hand costs ~0.1 s of wall clock for nothing)

  if (getenv("HETMERS_STATS") != NULL)
    { fprintf(stderr,"{\"placement\": \"%s\", \"device_bytes\": [",place == HM_PLACE_SHARDED ? "sharded" : "replica");
      for (i = 0; i < ngpu; i++)
        { int64_t b = 0;
          hm_scan_shard_info(S,i,NULL,NULL,NULL,&b);
          fprintf(stderr,"%s%lld",i ? ", " : "",(long long) b);
        }
      fprintf(stderr,"], ");
    }
#ifdef EXTRACT_PAIRS
  if (getenv("HETMERS_STATS") != NULL)
    fprintf(stderr,"\"extract\": {\"path\": \"%s\", \"pairs\": %lld, \"slices\": %d, \"ms_kernel\": %.3f, "
                   "\"ms_copy\": %.3f, \"ms_sort\": %.3f, \"wall_ms\": %.1f}, ",
            XST.path == HM_PATH_SYMM ? "symmetric" : "direct",(long long) XST.n_records,XST.slices,
            XST.ms_kernel,XST.ms_copy,XST.ms_sort,t_extract);
#endif
  if (getenv("HETMERS_STATS") != NULL)
    fprintf(stderr,"\"nels\": %lld, \"n_gpus\": %d, \"path\": \"%s\", \"bucket_bits\": %d, \"ms_load\": %.3f, "
                   "\"ms_pass1\": %.3f, \"ms_pass2\": %.3f, \"ms_scan\": %.3f, \"kernel_launches\": %lld, "
                   "\"wall_ms\": {\"open\": %.1f, \"cuda_init_load\": %.1f, \"examine\": %.1f, \"scan\": %.1f}, "
                   "\"load_ms\": {\"alloc\": %.1f, \"records\": %.1f, \"index\": %.1f}}\n",
            (long long) stats.nels,stats.n_gpus,stats.path == HM_PATH_SYMM ? "symmetric" : "direct",
            stats.bucket_bits,stats.ms_h2d_unpack,
            stats.ms_pass1,stats.ms_pass2,stats.ms_scan,(long long) stats.kernel_launches,
            t_open-t_start,t_load-t_open,t_exam-t_load,t_scan-t_exam,
            stats.ms_alloc,stats.ms_records,stats.ms_index);

  if (input != NULL)                                              /* PloidyPlot.c:1584-1592 */
    { char *command = malloc(strlen(input)+100);
      if (command == NULL)
        exit (1);
      sprintf(command,"Fastrm %s",input);
      systemx(command);
      free(command);
      free(input);
    }

#ifdef EXTRACT_PAIRS
  //  The pair list comes back sorted by (smudge, k-mer); one line per pair in print_het's format
  //  (PloidyList.c:128-165): lower-case bases with "(x/y)" at the varying position
  { static const char dna[4] = { 'a', 'c', 'g', 't' };
    char   line[160];
    int64_t r;
    for (r = 0; r < NREC; r++)
      { const hm_pair_rec *q = REC+r;
        char *o = line;
        int   p;
        for (p = 0; p < KMER; p++)
          { int bse = (int) (((p < 32 ? q->key_hi : q->key_lo) >> (62-2*(p&31))) & 3);
            if (p == q->pos)
              { *o++ = '('; *o++ = dna[bse]; *o++ = '/'; *o++ = dna[q->alt & 3]; *o++ = ')'; }
            else
              *o++ = dna[bse];
          }
        *o++ = '\n'; *o = '\0';
        fputs(line,SM.v[q->smudge-1].f);
      }
    for (i = 0; i < SM.n; i++)
      fclose(SM.v[i].f);
    free(REC);
  }
#else
  if (VERBOSE)
    { fprintf(stderr,"\n  Count complete, outputting table\n");
      fflush(stderr);
    }

  { char *smu = malloc(strlen(OUT)+8);
    sprintf(smu,"%s.smu",OUT);
    if (hm_write_smu(smu,PLOT) != HM_OK)
      { fprintf(stderr,"Could not open %s.smu\n",OUT);
        exit (1);
      }
    free(smu);
  }

#endif

  free(PLOT);
  free(OUT);
  fflush(NULL);
  _exit (0);                     /* exit(0) without the CUDA runtime's atexit teardown */
}
