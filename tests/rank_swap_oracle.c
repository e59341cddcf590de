/*
 * rank_swap_oracle.c -- the even/odd temperature swaps inside every virtual rank (DESIGN.md 7c) on top of the C restatement
 * of the reference (oracle/rfinv_oracle.c, included unchanged: its PT state and static helpers are used as they are).
 *
 * TEST INFRASTRUCTURE ONLY, built by tests/rank_swap_oracle.py with the restatement's compiler flags.
 *
 *   rso_philox4x64   Philox4x64-10 (Salmon, Moraes, Dror & Shaw, SC 2011), restated with unsigned __int128
 *   rso_pt_run       orc_pt_run with the rank sweep between the counters / record_chain and the global swap; mode 0 is
 *                    orc_pt_run line for line
 */
#include "../oracle/rfinv_oracle.c"

/* the 4 output words of counter ctr (word 0 least significant) under key `key` */
void rso_philox4x64(const uint64_t ctr_in[4], const uint64_t key_in[2], uint64_t out[4]) {
  uint64_t c0 = ctr_in[0], c1 = ctr_in[1], c2 = ctr_in[2], c3 = ctr_in[3], k0 = key_in[0], k1 = key_in[1];
  for (int round = 0; round < 10; ++round) {
    if (round) { k0 += 0x9E3779B97F4A7C15ULL; k1 += 0xBB67AE8584CAA73BULL; }
    const unsigned __int128 p0 = (unsigned __int128)0xD2E7470EE14C6C93ULL * c0;
    const unsigned __int128 p1 = (unsigned __int128)0xCA5A826395121157ULL * c2;
    const uint64_t hi0 = (uint64_t)(p0 >> 64), lo0 = (uint64_t)p0, hi1 = (uint64_t)(p1 >> 64), lo1 = (uint64_t)p1;
    c0 = hi1 ^ c1 ^ k0; c1 = lo1; c2 = hi0 ^ c3 ^ k1; c3 = lo0;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

/* The rank sweep of iteration i (0-based): in every virtual rank, the chains sorted by (temperature, chain) are levels
 * 0..nc-1; level l = i (mod 2) and level l + 1 swap temperatures with judge_pt's test and a Philox uniform.
 * n_prop / n_acc [nc - 1] are summed over the ranks. */
static void rank_sweep(orc_pt* p, int64_t i, int64_t* n_prop, int64_t* n_acc) {
  const int nc = p->c.nchains;
  int* at = (int*)malloc(sizeof(int) * (size_t)nc); /* at[level] = chain of the rank */
  const uint64_t key[2] = {(uint64_t)(uint32_t)p->c.iseed, 0};
  for (int r = 0; r < p->nproc; ++r) {
    double* t = p->temps + (size_t)r * nc;
    const double* e = p->logl + (size_t)r * nc;
    for (int a = 0; a < nc; ++a) {
      int lvl = 0;
      for (int b = 0; b < nc; ++b) lvl += t[b] < t[a] || (t[b] == t[a] && b < a);
      at[lvl] = a;
    }
    for (int l = (int)(i & 1); l + 1 < nc; l += 2) {
      const int a = at[l], b = at[l + 1];
      const uint64_t ctr[4] = {(uint64_t)i, (uint64_t)r, (uint64_t)l, 0};
      uint64_t w[4];
      rso_philox4x64(ctr, key, w);
      const double u = (double)(w[0] >> 11) * 0x1p-53;
      const double del_s = (e[b] - e[a]) * (1.0 / t[a] - 1.0 / t[b]);
      const int yn = log(u) <= del_s;
      n_prop[l]++;
      n_acc[l] += yn;
      if (yn) { const double ta = t[a]; t[a] = t[b]; t[b] = ta; }
    }
  }
  free(at);
}

/* orc_pt_run (pt_control, pt_mcmc.f90:468-576) with the rank sweep when mode == 1; arguments as there. */
int32_t rso_pt_run(orc_pt* p, int32_t mode, int64_t* n_prop, int64_t* n_acc, int32_t n_iter, int8_t* flags, int8_t* itypes,
                   int32_t* swaps, int32_t record) {
  const rfinv_config* c = &p->c;
  int nc = c->nchains, n = c->nfft, T = c->ntrc;
  size_t G = (size_t)p->nproc * nc;
  int new_cap = p->it_done + n_iter;
  if (new_cap > p->cap_hist) {
    p->likelihood_hist = (double*)realloc(p->likelihood_hist, sizeof(double) * (size_t)new_cap);
    for (int i = p->cap_hist; i < new_cap; ++i) p->likelihood_hist[i] = 0.0;
    p->cap_hist = new_cap;
  }
  int8_t* fl = (int8_t*)malloc(G);
  int8_t* ty = (int8_t*)malloc(G);
  int64_t n_eval_tot = 0;
#pragma omp parallel num_threads(p->nthreads) reduction(+ : n_eval_tot)
  {
    rf_ws* w = ws_create(n);
    double* mis = (double*)malloc(sizeof(double) * (size_t)c->nsmp);
    double* prop_rft = (double*)malloc(sizeof(double) * (size_t)n * T);
    for (int step = 0; step < n_iter; ++step) {
      int it = p->it_done + step + 1; /* 1-based iteration number */
#pragma omp for schedule(dynamic, 1)
      for (int r = 0; r < p->nproc; ++r)
        for (int ic = 0; ic < nc; ++ic) {
          size_t g = (size_t)r * nc + ic;
          int itype;
          fl[g] = (int8_t)mcmc_step(p, w, mis, prop_rft, r, ic, p->temps[g], &itype, &n_eval_tot);
          ty[g] = (int8_t)itype;
        }
#pragma omp single
      {
        for (size_t g = 0; g < G; ++g) { /* counters, pt_mcmc.f90:196-201, in chain order */
          if (p->temps[g] <= 1.0 + COLD_EPS) {
            p->nprop[ty[g] - 1]++;
            if (fl[g] == 1) p->naccept[ty[g] - 1]++;
            p->likelihood_hist[it - 1] += p->logl[g];
            if (record && it > c->nburn && it % c->ncorr == 0) record_chain(p, g);
          }
        }
        if (flags) memcpy(flags + (size_t)step * G, fl, G);
        if (itypes) memcpy(itypes + (size_t)step * G, ty, G);
        if (mode == 1 && nc >= 2) rank_sweep(p, it - 1, n_prop, n_acc);
        if (nc >= 2) { /* pt_mcmc.f90:498-571 */
          int n_all = (int)G;
          mt_state* s0 = &p->rng[0];
          int itarget1 = (int)(orc_grnd(s0) * n_all), itarget2;
          do { itarget2 = (int)(orc_grnd(s0) * n_all); } while (itarget2 == itarget1);
          int rank1 = itarget1 / nc;
          double temp1 = p->temps[itarget1], temp2 = p->temps[itarget2];
          double e1 = p->logl[itarget1], e2 = p->logl[itarget2];
          double del_s = (e2 - e1) * (1.0 / temp1 - 1.0 / temp2); /* judge_pt, pt_mcmc.f90:580-595 */
          int yn = log(orc_grnd(&p->rng[rank1])) <= del_s;
          if (yn) { p->temps[itarget2] = temp1; p->temps[itarget1] = temp2; }
          if (swaps) { swaps[(size_t)step * 3] = itarget1; swaps[(size_t)step * 3 + 1] = itarget2; swaps[(size_t)step * 3 + 2] = yn; }
        }
      }
    }
    free(prop_rft); free(mis); ws_destroy(w);
  }
  p->it_done += n_iter;
  p->n_eval += n_eval_tot;
  free(fl); free(ty);
  return 0;
}
