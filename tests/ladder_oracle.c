/*
 * ladder_oracle.c -- the ladder tuning during the burn-in (DESIGN.md 7d) on top of the rank sweep of rank_swap_oracle.c,
 * which is included unchanged (and with it the C restatement oracle/rfinv_oracle.c).
 *
 * TEST INFRASTRUCTURE ONLY, built by tests/ladder_oracle.py with the restatement's compiler flags.
 *
 *   lo_tune_rank   the ladder tuning of one virtual rank at a tuning point
 *   lo_pt_run      rso_pt_run with per-rank acceptance rows and the tuning after the sweep of the tuning points' iterations
 */
#include "rank_swap_oracle.c"

/* rank_sweep of rank_swap_oracle.c, line for line, that also counts the accepted swaps of every rank: rows [nproc][nc - 1]
 * (the tuning needs each rank's acceptances; rank_sweep sums them over the ranks). */
static void rank_sweep_rows(orc_pt* p, int64_t i, int64_t* n_prop, int64_t* n_acc, int64_t* rows) {
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
      rows[(size_t)r * (nc - 1) + l] += yn;
      if (yn) { const double ta = t[a]; t[a] = t[b]; t[b] = ta; }
    }
  }
  free(at);
}

/* The ladder tuning of one virtual rank at tuning point e (DESIGN.md 7d): t[nc] the temperatures of its chains, acc[nc - 1]
 * its accepted sweep swaps per level pair so far, base[nc - 1] those at the previous tuning point (set to acc on return).
 * The levels above the cold anchor take the inverse temperatures that split the barrier -- the running sum of the rejection
 * rates of the round [s, e) -- into equal parts, interpolated linearly in beta; the rank keeps its ladder if the new one is
 * not strictly increasing or would make a chain cold.  Returns 1 if the ladder changed. */
int32_t lo_tune_rank(int32_t nc, double* t, const int64_t* acc, int64_t* base, int64_t e) {
  int changed = 0;
  int* at = (int*)malloc(sizeof(int) * (size_t)nc);
  for (int a = 0; a < nc; ++a) {
    int lvl = 0;
    for (int b = 0; b < nc; ++b) lvl += t[b] < t[a] || (t[b] == t[a] && b < a);
    at[lvl] = a;
  }
  int c = 0;
  for (int a = 0; a < nc; ++a) c += t[a] <= 1.0 + COLD_EPS;
  const int a0 = c > 0 ? c - 1 : 0, h = nc - 1, K = h - a0;
  if (K >= 2) {
    const int64_t s = e == 64 ? 0 : e / 2;
    const double P = (double)((e - s) / 2);
    double* lam_ = (double*)malloc(sizeof(double) * (size_t)(K + 1)); /* Lambda_0 .. Lambda_K */
    double* beta = (double*)malloc(sizeof(double) * (size_t)(K + 1));
    double* tn = (double*)malloc(sizeof(double) * (size_t)(K + 1));
    lam_[0] = 0.0;
    for (int m = 0; m < K; ++m) {
      const double q = (double)(acc[a0 + m] - base[a0 + m]) / P;
      double rho = 1.0 - q;
      if (rho < 0x1p-10) rho = 0x1p-10;
      lam_[m + 1] = lam_[m] + rho;
    }
    for (int m = 0; m <= K; ++m) beta[m] = 1.0 / t[at[a0 + m]];
    tn[0] = t[at[a0]];
    tn[K] = t[at[h]];
    for (int k = 1; k < K; ++k) {
      const double lam = (lam_[K] * (double)k) / (double)K;
      int m = 0;
      while (m < K - 1 && !(lam < lam_[m + 1])) ++m;
      const double f = (lam - lam_[m]) / (lam_[m + 1] - lam_[m]);
      tn[k] = 1.0 / (beta[m] + (f * (beta[m + 1] - beta[m])));
    }
    int ok = 1;
    for (int k = 1; k <= K; ++k) ok = ok && tn[k] > tn[k - 1];
    for (int k = 1; k < K; ++k) ok = ok && tn[k] > 1.0 + COLD_EPS;
    if (ok)
      for (int k = 1; k < K; ++k) {
        changed = changed || t[at[a0 + k]] != tn[k];
        t[at[a0 + k]] = tn[k];
      }
    free(lam_); free(beta); free(tn);
  }
  for (int l = 0; l + 1 < nc; ++l) base[l] = acc[l];
  free(at);
  return changed;
}

/* the iteration count e after iteration e - 1 is a tuning point: 2^j, j >= 6, e <= nburn */
static int tuning_point(int64_t e, int32_t nburn) { return e >= 64 && e <= nburn && (e & (e - 1)) == 0; }

/* rso_pt_run (rank_swap_oracle.c) with the ladder tuning: the same loop, whose rank sweep also counts the accepted swaps per
 * rank (rows), and, with tune, the tuning of every rank after the sweep of the tuning points' iterations (before the global
 * swap).  rows / base [nproc][nc - 1]: the per-rank acceptances and their snapshot at the last tuning point, kept by the
 * caller; *n_points counts the tuning points passed.  With tune = 0 this is rso_pt_run. */
int32_t lo_pt_run(orc_pt* p, int32_t mode, int32_t tune, int64_t* n_prop, int64_t* n_acc, int64_t* rows, int64_t* base,
                  int32_t* n_points, int32_t n_iter, int8_t* flags, int8_t* itypes, int32_t* swaps, int32_t record) {
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
        if (mode == 1 && nc >= 2) rank_sweep_rows(p, it - 1, n_prop, n_acc, rows);
        if (tune && tuning_point(it, c->nburn)) {
          if (mode == 1 && nc >= 2)
            for (int r = 0; r < p->nproc; ++r)
              lo_tune_rank(nc, p->temps + (size_t)r * nc, rows + (size_t)r * (nc - 1), base + (size_t)r * (nc - 1), it);
          ++*n_points;
        }
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
