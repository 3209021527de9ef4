/* kbench.c -- kernel sweep tool: every CSR/HLL kernel variant on one matrix.
 *
 *   kbench <matrix> [--reps N] [--warmup N] [--flush] [--peak GBs] [--quick]
 *                   [--only csr|hll]
 *   <matrix>: c1 | c2 | c3 | c4 | poisson:NX:NY | stencil:NX:NY:NZ |
 *             uniform:N:K | rmat:SCALE:EF | ragged:N:W | mtx:<path>
 *
 * Prints one line per (kernel, warps/block, knob) with min / median kernel
 * time (CUDA events, matrix resident in HBM), GFLOP/s = 2 nnz / t, achieved
 * GB/s on the minimum-traffic byte count B_min = 12 nnz + 4 (M+1) + 8 M + 8 N,
 * its fraction of --peak, and the largest |dy| / sum|a x| against the host
 * serial CSR loop of libspmv_host (a sanity check; the parity gate proper is
 * tests/ with the oracle).  Plain C over the public C ABI: this is also the
 * usage example of include/spmv_b200.h.
 */
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "csr.h"
#include "cuda_timer.h"
#include "hll.h"
#include "spmv_b200.h"
#include "spmv_gen.h"

static int g_reps = 20, g_warmup = 3, g_flush = 0, g_quick = 0, g_profile = 0, g_cfg_from = -1;
static int g_sell = 0, g_spmm = 0;
static int g_panels[16] = {1, 2, 3, 4, 6, 8, 16}, g_n_panels = 7;
static int g_chunks[16], g_n_chunks = 0, g_auto = 0;
static double g_peak = 6559.7; /* MEASURED_PEAKS.json hbm_gbs of this pool */
static const char *g_only = "";

static int cmp_d(const void *a, const void *b) {
      double x = *(const double *)a, y = *(const double *)b;
      return (x > y) - (x < y);
}

static sparse_csr *make_matrix(const char *spec) {
      int a, b, c;
      if (!strcmp(spec, "c1"))
            return gen_poisson2d(1000, 1000);
      if (!strcmp(spec, "c2"))
            return gen_stencil27(128, 128, 128);
      if (!strcmp(spec, "c3"))
            return gen_uniform_random(16000000, 32, 42);
      if (!strcmp(spec, "c4"))
            return gen_rmat(24, 16, 0.57, 0.19, 0.19, 42);
      if (sscanf(spec, "poisson:%d:%d", &a, &b) == 2)
            return gen_poisson2d(a, b);
      if (sscanf(spec, "stencil:%d:%d:%d", &a, &b, &c) == 3)
            return gen_stencil27(a, b, c);
      if (sscanf(spec, "uniform:%d:%d", &a, &b) == 2)
            return gen_uniform_random(a, b, 42);
      if (sscanf(spec, "rmat:%d:%d", &a, &b) == 2)
            return gen_rmat(a, b, 0.57, 0.19, 0.19, 42);
      if (sscanf(spec, "ragged:%d:%d", &a, &b) == 2)
            return gen_ragged(a, b, 7);
      if (!strncmp(spec, "mtx:", 4)) {
            sparse_csr *A = io_load_csr(spec + 4);
            return (uintptr_t)A > (uintptr_t)-4096 ? NULL : A;
      }
      return NULL;
}

struct ctx {
      const sparse_csr *A;
      double *d_x, *d_y;
      double *y_host, *y_ref, *scale;
      double bmin;
};

static double check(struct ctx *c) {
      const int M = c->A->M;
      spmv_b200_d2h(c->y_host, c->d_y, (size_t)M * 8, NULL);
      spmv_b200_stream_sync(NULL);
      double worst = 0.0;
      for (int r = 0; r < M; ++r) {
            const double err = fabs(c->y_host[r] - c->y_ref[r]);
            const double rel = c->scale[r] > 0 ? err / c->scale[r] : (err > 0 ? INFINITY : 0);
            if (rel > worst)
                  worst = rel;
      }
      return worst;
}

static void report(struct ctx *c, const char *fmt, const char *kname, int wpb, const char *knob,
                   double *ms, int launches) {
      qsort(ms, (size_t)g_reps, sizeof *ms, cmp_d);
      const double tmin = ms[0], tmed = ms[g_reps / 2];
      const double gf = 2.0 * c->A->NZ / (tmed * 1e6);
      const double gbs = c->bmin / (tmed * 1e6);
      const double err = check(c);
      printf("%-4s %-14s wpb=%-2d %-18s launches=%d  min %8.4f ms  med %8.4f ms  %8.1f GFLOP/s  "
             "%7.1f GB/s  %5.1f%% of %.0f  maxrel %.2e %s\n",
             fmt, kname, wpb, knob, launches, tmin, tmed, gf, gbs, 100.0 * gbs / g_peak, g_peak, err,
             err <= 1e-12 ? "ok" : "PARITY-FAIL");
      fflush(stdout);
}

static void poison_y(struct ctx *c) { spmv_b200_dmemset(c->d_y, 0xff, (size_t)c->A->M * 8, NULL); }

static const char *k_csr_names[] = {"thread_row", "warp_row", "adaptive", "block_row", "stream_tma"};
static const char *k_hll_names[] = {"thread_row_rm", "thread_row", "warp_hack_vec", "stream_tma"};

static void run_csr(struct ctx *c, spmv_b200_csr *h, int kernel, int wpb, const char *knob) {
      double *ms = malloc(sizeof(double) * (size_t)g_reps);
      poison_y(c);
      if (spmv_b200_csr_time(h, kernel, wpb, c->d_x, c->d_y, g_warmup, g_reps, g_flush, ms, NULL)) {
            printf("CSR  %-14s wpb=%-2d %-18s FAILED: %s\n", k_csr_names[kernel], wpb, knob,
                   spmv_b200_last_error());
      } else {
            report(c, "CSR", k_csr_names[kernel], wpb, knob, ms, spmv_b200_csr_launches(h, kernel));
      }
      free(ms);
}

static void run_hll(struct ctx *c, spmv_b200_hll *h, int kernel, int wpb, const char *knob) {
      double *ms = malloc(sizeof(double) * (size_t)g_reps);
      poison_y(c);
      if (spmv_b200_hll_time(h, kernel, wpb, c->d_x, c->d_y, g_warmup, g_reps, g_flush, ms, NULL)) {
            printf("HLL  %-14s wpb=%-2d %-18s FAILED: %s\n", k_hll_names[kernel], wpb, knob,
                   spmv_b200_last_error());
      } else {
            report(c, "HLL", k_hll_names[kernel], wpb, knob, ms, 1);
      }
      free(ms);
}

int main(int argc, char **argv) {
      if (argc < 2) {
            fprintf(stderr, "usage: kbench <matrix> [--reps N] [--warmup N] [--flush] [--peak GBs] "
                            "[--quick] [--only csr|hll]\n");
            return 2;
      }
      for (int i = 2; i < argc; ++i) {
            if (!strcmp(argv[i], "--reps") && i + 1 < argc)
                  g_reps = atoi(argv[++i]);
            else if (!strcmp(argv[i], "--warmup") && i + 1 < argc)
                  g_warmup = atoi(argv[++i]);
            else if (!strcmp(argv[i], "--peak") && i + 1 < argc)
                  g_peak = atof(argv[++i]);
            else if (!strcmp(argv[i], "--only") && i + 1 < argc)
                  g_only = argv[++i];
            else if (!strcmp(argv[i], "--flush"))
                  g_flush = 1;
            else if (!strcmp(argv[i], "--quick"))
                  g_quick = 1;
            else if (!strcmp(argv[i], "--cfg-from") && i + 1 < argc)
                  g_cfg_from = atoi(argv[++i]);
            else if (!strcmp(argv[i], "--knob") && i + 1 < argc) {
                  char key[64];
                  int val = 0;
                  if (sscanf(argv[++i], "%63[^=]=%d", key, &val) == 2)
                        spmv_b200_set_knob(key, val);
            } else if (!strcmp(argv[i], "--profile"))
                  g_profile = 1; /* only the headline kernels: for ncu captures */
            else if (!strcmp(argv[i], "--sell"))
                  g_sell = 1; /* SELL-P sweep: panels x sigma x warps/block, CSR and HLL source */
            else if (!strcmp(argv[i], "--spmm"))
                  g_spmm = 1; /* SpMM: 1 (id 2), 2 and 4 right-hand sides in one pass */
            else if (!strcmp(argv[i], "--auto"))
                  g_auto = 1; /* only what the library picks on its own: CSR id 2, HLL id 2 (ncu captures) */
            else if (!strcmp(argv[i], "--chunks") && i + 1 < argc) {
                  for (char *tok = strtok(argv[++i], ","); tok && g_n_chunks < 16; tok = strtok(NULL, ","))
                        g_chunks[g_n_chunks++] = atoi(tok);
            } else if (!strcmp(argv[i], "--panels") && i + 1 < argc) {
                  g_n_panels = 0;
                  for (char *tok = strtok(argv[++i], ","); tok && g_n_panels < 16; tok = strtok(NULL, ","))
                        g_panels[g_n_panels++] = atoi(tok);
            }
      }
      spmv_b200_devinfo info;
      if (spmv_b200_device_info(&info)) {
            fprintf(stderr, "kbench: %s\n", spmv_b200_last_error());
            return 1;
      }
      printf("# device %s sm_%d%d, %d SMs, L2 %d MB, HBM %.1f GB\n", info.name, info.cc_major,
             info.cc_minor, info.sm_count, info.l2_bytes_mb, info.hbm_bytes / 1e9);

      sparse_csr *A = make_matrix(argv[1]);
      if (!A) {
            fprintf(stderr, "kbench: cannot build matrix '%s'\n", argv[1]);
            return 1;
      }
      struct ctx c = {.A = A};
      c.bmin = 12.0 * A->NZ + 4.0 * (A->M + 1) + 8.0 * A->M + 8.0 * A->N;
      printf("# matrix %s M=%d N=%d NZ=%d  B_min=%.0f bytes  reps=%d warmup=%d flush_l2=%d\n", A->name,
             A->M, A->N, A->NZ, c.bmin, g_reps, g_warmup, g_flush);

      /* x in [0,1) from a fixed LCG; reference y and per-row tolerance scale */
      double *x = malloc(sizeof(double) * (size_t)A->N);
      c.y_host = malloc(sizeof(double) * (size_t)A->M);
      c.y_ref = malloc(sizeof(double) * (size_t)A->M);
      c.scale = malloc(sizeof(double) * (size_t)A->M);
      unsigned long long s = 88172645463325252ull;
      for (int i = 0; i < A->N; ++i) {
            s ^= s << 13, s ^= s >> 7, s ^= s << 17;
            x[i] = (double)(s >> 11) / 9007199254740992.0;
      }
#pragma omp parallel for schedule(static, 1024)
      for (int r = 0; r < A->M; ++r) {
            double acc = 0, sc = 0;
            for (int k = A->IRP[r]; k < A->IRP[r + 1]; ++k) {
                  const double p = A->AS[k] * x[A->JA[k]];
                  acc += p, sc += fabs(p);
            }
            c.y_ref[r] = acc, c.scale[r] = sc;
      }
      c.d_x = spmv_b200_dmalloc((size_t)A->N * 8 + 256);
      c.d_y = spmv_b200_dmalloc((size_t)A->M * 8 + 256);
      if (!c.d_x || !c.d_y)
            return 1;
      spmv_b200_h2d(c.d_x, x, (size_t)A->N * 8, NULL);
      spmv_b200_stream_sync(NULL);

      static const int wpbs[] = {2, 4, 8, 16};
      char knob[64];

      if (g_auto) {
            spmv_b200_csr *h = spmv_b200_csr_create(A);
            if (!h) {
                  fprintf(stderr, "kbench: %s\n", spmv_b200_last_error());
                  return 1;
            }
            run_csr(&c, h, 2, 4, "auto");
            if (strcmp(g_only, "csr")) {
                  spmv_b200_hll *hh = spmv_b200_hll_from_csr(h);
                  if (hh) {
                        run_hll(&c, hh, 2, 4, "auto");
                        spmv_b200_hll_destroy(hh);
                  }
            }
            spmv_b200_csr_destroy(h);
            return 0;
      }

      if (g_spmm) {
            /* k right-hand sides in one pass: time per pass, GFLOP/s = 2 nnz k / t, and the gain over
             * k single-vector products */
            spmv_b200_csr *h = spmv_b200_csr_create(A);
            if (!h) {
                  fprintf(stderr, "kbench: %s\n", spmv_b200_last_error());
                  return 1;
            }
            run_csr(&c, h, 2, 4, "k=1 (SpMV)");
            double ms1[64];
            spmv_b200_csr_time(h, 2, 4, c.d_x, c.d_y, g_warmup, g_reps > 64 ? 64 : g_reps, g_flush, ms1, NULL);
            qsort(ms1, g_reps > 64 ? 64 : g_reps, sizeof(double), cmp_d);
            const double t1 = ms1[(g_reps > 64 ? 64 : g_reps) / 2];
            for (int k = 2; k <= 4; k += 2) {
                  double *dX = spmv_b200_dmalloc((size_t)A->N * k * 8), *dY = spmv_b200_dmalloc((size_t)A->M * k * 8);
                  double *X = malloc((size_t)A->N * k * 8), *Y = malloc((size_t)A->M * k * 8);
                  if (!dX || !dY || !X || !Y)
                        return 1;
                  for (long long i = 0; i < (long long)A->N * k; ++i)
                        X[i] = (double)((i * 2654435761u) % 2001) / 1000.0 - 1.0;
                  spmv_b200_h2d(dX, X, (size_t)A->N * k * 8, NULL);
                  double ms[64];
                  const int reps = g_reps > 64 ? 64 : g_reps;
                  for (int r = -g_warmup; r < reps; ++r) {
                        cuda_timer t;
                        timer_init(&t);
                        timer_start(&t, NULL);
                        if (spmv_b200_csr_spmm(h, k, dX, dY, NULL)) {
                              fprintf(stderr, "kbench: %s\n", spmv_b200_last_error());
                              return 1;
                        }
                        const double m = timer_stop(&t, NULL);
                        timer_destroy(&t);
                        if (r >= 0)
                              ms[r] = m;
                  }
                  qsort(ms, reps, sizeof(double), cmp_d);
                  /* check column 0 and column k-1 against the host serial loop */
                  spmv_b200_d2h(Y, dY, (size_t)A->M * k * 8, NULL);
                  spmv_b200_stream_sync(NULL);
                  double worst = 0.0;
                  for (int col = 0; col < k; col += k - 1)
                        for (int r = 0; r < A->M; ++r) {
                              double ref = 0.0, sc = 0.0;
                              for (int q = A->IRP[r]; q < A->IRP[r + 1]; ++q) {
                                    const double p = A->AS[q] * X[(size_t)A->JA[q] * k + col];
                                    ref += p, sc += fabs(p);
                              }
                              const double err = fabs(Y[(size_t)r * k + col] - ref);
                              if (sc > 0 && err / sc > worst)
                                    worst = err / sc;
                        }
                  const double med = ms[reps / 2];
                  printf("CSR  spmm           k=%d  launches=-  min %8.4f ms  med %8.4f ms  %8.1f GFLOP/s  %.2fx the rate of %d "
                         "SpMV passes  maxrel %.2e %s\n", k, ms[0], med, 2.0 * A->NZ * k / (med * 1e6), k * t1 / med, k,
                         worst, worst <= 1e-12 ? "ok" : "MISMATCH");
                  fflush(stdout);
                  spmv_b200_dfree(dX), spmv_b200_dfree(dY), free(X), free(Y);
            }
            spmv_b200_csr_destroy(h);
            return 0;
      }

      if (g_n_chunks) {
            /* ragged matrices: virtual-row chunk size x warps/block */
            int64_t info[11];
            for (int ic = 0; ic < g_n_chunks; ++ic) {
                  spmv_b200_set_knob("sell_chunk", g_chunks[ic]);
                  spmv_b200_csr *h = spmv_b200_csr_create(A);
                  if (!h || spmv_b200_csr_sell_info(h, 1, info, 11) || info[0] != 1) {
                        printf("CSR  sell chunk=%d BUILD FAILED: %s\n", g_chunks[ic], spmv_b200_last_error());
                        spmv_b200_csr_destroy(h);
                        continue;
                  }
                  snprintf(knob, sizeof knob, "C=%d pad=%.1f%%", g_chunks[ic],
                           info[5] ? 100.0 * (info[4] - (double)info[5]) / info[5] : 0.0);
                  for (int w = 1; w < 4; ++w)
                        run_csr(&c, h, 2, wpbs[w], knob);
                  spmv_b200_csr_destroy(h);
            }
            spmv_b200_set_knob("sell_chunk", 256);
            return 0;
      }

      if (g_sell) {
            const int *panels = g_panels;
            static const int sigmas[] = {1024, 16384, 262144};
            int64_t info[8];
            /* what the library picks on its own, then the old paths, then the sweep */
            spmv_b200_csr *h = spmv_b200_csr_create(A);
            if (!h) {
                  fprintf(stderr, "kbench: %s\n", spmv_b200_last_error());
                  return 1;
            }
            for (int w = 1; w < 4; ++w)
                  run_csr(&c, h, 2, wpbs[w], "auto");
            spmv_b200_csr_sell_info(h, 0, info, 8);
            printf("# auto: sell state=%lld panels=%lld sigma=%lld slots=%lld (padding %.2f%%) long_rows=%lld "
                   "gather_span=%.3f\n", (long long)info[0], (long long)info[1], (long long)info[2],
                   (long long)info[4], info[5] ? 100.0 * (info[4] - (double)info[5]) / info[5] : 0.0,
                   (long long)info[6], info[7] * 1e-6);
            run_csr(&c, h, 4, 4, "auto");
            spmv_b200_set_knob("sell", 0);
            run_csr(&c, h, 2, 8, "sell=0");
            run_csr(&c, h, 4, 4, "sell=0");
            spmv_b200_csr_destroy(h);
            spmv_b200_set_knob("sell", 1);
            for (int ip = 0; ip < g_n_panels; ++ip) {
                  for (int is = 0; is < 3; ++is) {
                        if (is != 1 && !(panels[ip] == 1 || panels[ip] == 4))
                              continue; /* sigma only matters for padding: sweep it at two panel counts */
                        spmv_b200_set_knob("sell_panels", panels[ip]);
                        spmv_b200_set_knob("sell_sigma", sigmas[is]);
                        h = spmv_b200_csr_create(A);
                        if (!h || spmv_b200_csr_sell_info(h, 1, info, 8) || info[0] != 1) {
                              printf("CSR  sell panels=%d sigma=%d BUILD FAILED: %s\n", panels[ip],
                                     sigmas[is], spmv_b200_last_error());
                              spmv_b200_csr_destroy(h);
                              continue;
                        }
                        snprintf(knob, sizeof knob, "K=%d s=%d pad=%.1f%%", panels[ip], sigmas[is],
                                 info[5] ? 100.0 * (info[4] - (double)info[5]) / info[5] : 0.0);
                        for (int w = 1; w < 4; ++w)
                              if (is == 1 || w == 2)
                                    run_csr(&c, h, 2, wpbs[w], knob);
                        spmv_b200_csr_destroy(h);
                  }
            }
            if (strcmp(g_only, "csr")) {
                  spmv_b200_set_knob("sell_sigma", 16384);
                  spmv_b200_csr *hc = spmv_b200_csr_create(A);
                  for (int ip = -1; ip < g_n_panels; ++ip) {
                        spmv_b200_set_knob("sell", ip < 0 ? 0 : 1);
                        spmv_b200_set_knob("sell_panels", ip < 0 ? 0 : panels[ip]);
                        spmv_b200_hll *hh = hc ? spmv_b200_hll_from_csr(hc) : NULL;
                        if (!hh) {
                              printf("HLL  build failed: %s\n", spmv_b200_last_error());
                              break;
                        }
                        if (ip < 0)
                              snprintf(knob, sizeof knob, "sell=0");
                        else
                              snprintf(knob, sizeof knob, "K=%d", panels[ip]);
                        run_hll(&c, hh, 2, 8, knob);
                        spmv_b200_hll_destroy(hh);
                  }
                  spmv_b200_csr_destroy(hc);
            }
            spmv_b200_set_knob("sell", -1);
            spmv_b200_set_knob("sell_panels", 0);
            return 0;
      }

      if (g_profile) {
            spmv_b200_csr *h = spmv_b200_csr_create(A);
            if (!h) {
                  fprintf(stderr, "kbench: %s\n", spmv_b200_last_error());
                  return 1;
            }
            run_csr(&c, h, 4, 4, "auto");
            if (strcmp(g_only, "csr")) {
                  spmv_b200_hll *hh = spmv_b200_hll_from_csr(h);
                  if (!hh) {
                        fprintf(stderr, "kbench: %s\n", spmv_b200_last_error());
                        return 1;
                  }
                  run_hll(&c, hh, 2, 16, "auto");
                  run_hll(&c, hh, 3, 8, "auto");
                  spmv_b200_hll_destroy(hh);
            }
            spmv_b200_csr_destroy(h);
            return 0;
      }

      if (strcmp(g_only, "hll")) {
            spmv_b200_csr *h = spmv_b200_csr_create(A);
            if (!h) {
                  fprintf(stderr, "kbench: %s\n", spmv_b200_last_error());
                  return 1;
            }
            int64_t plan[10];
            spmv_b200_csr_plan_info(h, plan, 10);
            printf("# csr bins rows: <=4:%lld <=8:%lld <=16:%lld <=32:%lld <=64:%lld warp:%lld "
                   "block:%lld split:%lld regular=%lld base_kind=%lld\n",
                   (long long)plan[0], (long long)plan[1], (long long)plan[2], (long long)plan[3],
                   (long long)plan[4], (long long)plan[5], (long long)plan[6], (long long)plan[7],
                   (long long)plan[8], (long long)plan[9]);
            for (int w = 0; w < 3; ++w) {
                  run_csr(&c, h, 0, wpbs[w], "-");
                  run_csr(&c, h, 1, wpbs[w], "-");
                  if (!g_quick && A->M <= 4000000)
                        run_csr(&c, h, 3, wpbs[w], "-");
            }
            for (int w = 0; w < 4; ++w)
                  run_csr(&c, h, 2, wpbs[w], "auto");
            spmv_b200_set_knob("csr_pipe", 0); /* short regular rows: without the per-warp rings */
            run_csr(&c, h, 2, 4, "pipe=0");
            spmv_b200_set_knob("csr_pipe", 1);
            run_csr(&c, h, 2, 4, "pipe=1");
            spmv_b200_set_knob("csr_pipe", -1);
            for (int w = 0; w < 3; ++w)
                  run_csr(&c, h, 4, wpbs[w], "auto");
            static const int cfgs[] = {10, 12, 13, 24, 25, 26, 33};
            spmv_b200_set_knob("sell", 0); /* the staged kernel itself, whatever the matrix */
            for (int i = 0; i < 7; ++i) {
                  if (cfgs[i] < g_cfg_from)
                        continue;
                  spmv_b200_set_knob("csr_stream_cfg", cfgs[i]);
                  snprintf(knob, sizeof knob, "cfg=%d", cfgs[i]);
                  run_csr(&c, h, 4, 4, knob);
            }
            spmv_b200_set_knob("sell", -1);
            spmv_b200_set_knob("csr_stream_cfg", -1);
            spmv_b200_csr_destroy(h);
      }

      if (strcmp(g_only, "csr")) {
            /* HLL built on the device from the resident CSR */
            spmv_b200_csr *h = spmv_b200_csr_create(A);
            spmv_b200_hll *hh = h ? spmv_b200_hll_from_csr(h) : NULL;
            if (!hh) {
                  fprintf(stderr, "kbench: %s\n", spmv_b200_last_error());
                  return 1;
            }
            spmv_b200_csr_destroy(h);
            printf("# hll hacks=%lld slots=%lld (padding %.2f%%)\n",
                   (long long)spmv_b200_hll_num_hacks(hh), (long long)spmv_b200_hll_slots(hh),
                   100.0 * (spmv_b200_hll_slots(hh) - (double)A->NZ) / (A->NZ ? A->NZ : 1));
            for (int w = 0; w < 4; ++w)
                  run_hll(&c, hh, 1, wpbs[w], "-");
            spmv_b200_set_knob("hll_pipe", 0); /* warp per hack, whatever the width */
            for (int w = 0; w < 4; ++w)
                  run_hll(&c, hh, 2, wpbs[w], "pipe=0");
            /* narrow hacks: persistent warps with private bulk-copy rings (what id 2 picks for them) */
            spmv_b200_set_knob("hll_pipe", -1);
            run_hll(&c, hh, 2, 4, "pipe=auto");
            spmv_b200_set_knob("hll_pipe", 1);
            run_hll(&c, hh, 2, 4, "pipe=1");
            spmv_b200_set_knob("hll_pipe", -1);
            for (int cfg = 0; cfg < 3; ++cfg) {
                  spmv_b200_set_knob("hll_stream_cfg", cfg);
                  snprintf(knob, sizeof knob, "cfg=%d", cfg);
                  run_hll(&c, hh, 3, 4, knob);
            }
            spmv_b200_set_knob("hll_stream_cfg", -1);
            spmv_b200_hll_destroy(hh);
      }

      spmv_b200_dfree(c.d_x);
      spmv_b200_dfree(c.d_y);
      csr_free(A);
      return 0;
}
