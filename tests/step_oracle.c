/*
 * step_oracle.c -- the random-walk width tuning during the burn-in (DESIGN.md 7e) on top of the ladder tuning of
 * ladder_oracle.c, which is included unchanged (and with it rank_swap_oracle.c and the C restatement oracle/rfinv_oracle.c).
 *
 * TEST INFRASTRUCTURE ONLY, built by tests/step_oracle.py with the restatement's compiler flags (-ffp-contract=off: the
 * width dev * scale and the step gauss * width are two products, each rounded on its own, as on the device).
 *
 *   so_mcmc_step   mcmc_step of the restatement with the four widths as an argument instead of c->dev_*
 *   so_step        one chain step through mcmc_step or so_mcmc_step (the test compares them)
 *   so_levels      each chain's level in its rank, (temperature, chain index) order
 *   so_tune_rank   the width tuning of one virtual rank at a tuning point
 *   so_pt_run      lo_pt_run with the levels, the global-pair rule, the per-(rank, level, type) counters and the tuning
 */
#include "ladder_oracle.c"

/* one chain step, pt_mcmc.f90:54-192, with the widths w[4] of the moves z, dVs, dVp, sigma.  Returns flag: -1 null proposal,
 * 0 rejected, 1 accepted.  mcmc_step line for line otherwise. */
static int so_mcmc_step(orc_pt* p, rf_ws* w, double* mis, double* prop_rft, int rank, int ic, double temp, const double wd[4],
                        int* itype_out, int64_t* n_eval) {
  const rfinv_config* c = &p->c;
  mt_state* s = &p->rng[rank];
  int km = c->k_max, T = c->ntrc, n = c->nfft;
  size_t g = (size_t)rank * c->nchains + ic;
  double *cz = p->z + g * (km - 1), *cdvp = p->dvp + g * km, *cdvs = p->dvs + g * km, *csig = p->sig + g * T;
  double prop_dvp[256], prop_dvs[256], prop_z[256], prop_sig[64];
  double log_prior12 = 0.0;
  int prop_k = p->k[g], null_flag = 0, itarget;
  memcpy(prop_dvp, cdvp, sizeof(double) * (size_t)km);
  memcpy(prop_dvs, cdvs, sizeof(double) * (size_t)km);
  memcpy(prop_z, cz, sizeof(double) * (size_t)(km - 1));
  prop_z[km - 1] = 0.0;
  memcpy(prop_sig, csig, sizeof(double) * (size_t)T);
  int itype = (int)(orc_grnd(s) * p->ntype) + 1;
  *itype_out = itype;
  if (itype == p->it_birth) {
    prop_k = prop_k + 1;
    if (prop_k < km) {
      if (c->prior_mode == 1) { prop_dvp[prop_k - 1] = laplace(s) * c->dvp_prior; prop_dvs[prop_k - 1] = laplace(s) * c->dvs_prior; }
      else if (c->prior_mode == 2) { prop_dvp[prop_k - 1] = gauss(s) * c->dvp_prior; prop_dvs[prop_k - 1] = gauss(s) * c->dvs_prior; }
      prop_z[prop_k - 1] = c->z_min + orc_grnd(s) * (c->z_max - c->z_min);
    } else null_flag = 1;
  } else if (itype == p->it_death) {
    prop_k = prop_k - 1;
    if (prop_k >= c->k_min) {
      itarget = (int)(orc_grnd(s) * (prop_k + 1)) + 1;
      for (int il = itarget; il <= prop_k; ++il) {
        prop_dvp[il - 1] = cdvp[il]; prop_dvs[il - 1] = cdvs[il]; prop_z[il - 1] = cz[il];
      }
      prop_dvp[prop_k] = 0.0; prop_dvs[prop_k] = 0.0; prop_z[prop_k] = 0.0;
    } else null_flag = 1;
  } else if (itype == p->it_z) {
    itarget = (int)(orc_grnd(s) * prop_k) + 1;
    prop_z[itarget - 1] = prop_z[itarget - 1] + gauss(s) * wd[0];
    if (prop_z[itarget - 1] < c->z_min || prop_z[itarget - 1] > c->z_max) null_flag = 1;
  } else if (itype == p->it_dvs) {
    itarget = (int)(orc_grnd(s) * (prop_k + 1)) + 1;
    if (itarget == prop_k + 1) itarget = km;
    prop_dvs[itarget - 1] = prop_dvs[itarget - 1] + gauss(s) * wd[1];
    log_prior12 = log_prior_ratio(prop_dvs[itarget - 1], cdvs[itarget - 1], c->dvs_prior, c->prior_mode);
  } else if (itype == p->it_dvp) {
    itarget = (int)(orc_grnd(s) * (prop_k + 1)) + 1;
    if (itarget == prop_k + 1) itarget = km;
    prop_dvp[itarget - 1] = prop_dvp[itarget - 1] + gauss(s) * wd[2];
    log_prior12 = log_prior_ratio(prop_dvp[itarget - 1], cdvp[itarget - 1], c->dvp_prior, c->prior_mode);
  } else if (itype == p->it_sig) {
    itarget = p->isig_trc[(int)(orc_grnd(s) * p->nsig_trc)];
    prop_sig[itarget] = prop_sig[itarget] + gauss(s) * wd[3];
    if (prop_sig[itarget] < c->sig_min[itarget] || prop_sig[itarget] > c->sig_max[itarget]) null_flag = 1;
  }
  if (!null_flag) {
    double alpha[258], beta[258], rho[258], h[258];
    int nlay;
    if (!orc_format_model(c, prop_k, prop_z, prop_dvp, prop_dvs, &nlay, alpha, beta, rho, h)) null_flag = 1;
  }
  if (null_flag) return -1;
  int fwd = itype != p->it_sig;
  double ll2;
  eval_chain(p, w, mis, prop_k, prop_z, prop_dvp, prop_dvs, prop_sig, fwd, p->rft + g * (size_t)n * T, &ll2, prop_rft);
  if (fwd) (*n_eval)++;
  /* judge_mcmc, pt_mcmc.f90:600-621 */
  double del_s = (ll2 - p->logl[g]) / temp + log_prior12, r;
  do { r = orc_grnd(s); } while (!(r >= 2.220446049250313e-16));
  int yn = log(r) <= del_s;
  if (yn) {
    p->logl[g] = ll2;
    p->k[g] = prop_k;
    memcpy(cdvp, prop_dvp, sizeof(double) * (size_t)km);
    memcpy(cdvs, prop_dvs, sizeof(double) * (size_t)km);
    memcpy(cz, prop_z, sizeof(double) * (size_t)(km - 1));
    memcpy(csig, prop_sig, sizeof(double) * (size_t)T);
    memcpy(p->rft + g * (size_t)n * T, prop_rft, sizeof(double) * (size_t)n * T);
  }
  return yn;
}

/* one step of chain (rank, ic) at its temperature: use_copy 0 through mcmc_step (the params.in widths), 1 through so_mcmc_step
 * with the widths wd[4].  Returns the flag; *itype the proposal type. */
int32_t so_step(orc_pt* p, int32_t rank, int32_t ic, const double* wd, int32_t use_copy, int32_t* itype) {
  rf_ws* w = ws_create(p->c.nfft);
  double* mis = (double*)malloc(sizeof(double) * (size_t)p->c.nsmp);
  double* prop_rft = (double*)malloc(sizeof(double) * (size_t)p->c.nfft * p->c.ntrc);
  int64_t n_eval = 0;
  int t = 0;
  const size_t g = (size_t)rank * p->c.nchains + ic;
  const int fl = use_copy ? so_mcmc_step(p, w, mis, prop_rft, rank, ic, p->temps[g], wd, &t, &n_eval)
                          : mcmc_step(p, w, mis, prop_rft, rank, ic, p->temps[g], &t, &n_eval);
  p->n_eval += n_eval;
  *itype = t;
  free(prop_rft); free(mis); ws_destroy(w);
  return fl;
}

/* lvl[G]: each chain's level in its rank, the chains sorted by (temperature, chain index) */
void so_levels(const orc_pt* p, int32_t* lvl) {
  const int nc = p->c.nchains;
  for (int r = 0; r < p->nproc; ++r) {
    const double* t = p->temps + (size_t)r * nc;
    for (int a = 0; a < nc; ++a) {
      int l = 0;
      for (int b = 0; b < nc; ++b) l += t[b] < t[a] || (t[b] == t[a] && b < a);
      lvl[(size_t)r * nc + a] = l;
    }
  }
}

/* row of proposal type itype: 0 move z, 1 dVs, 2 dVp, 3 sigma; -1 birth and death */
static int so_type(const orc_pt* p, int itype) {
  return itype == p->it_z ? 0 : itype == p->it_dvs ? 1 : itype == p->it_dvp ? 2 : itype == p->it_sig ? 3 : -1;
}

/* The width tuning of one virtual rank at a tuning point (DESIGN.md 7e): scale / nprop / nacc [nc][4], proposed[4] 1 for the
 * types the run proposes.  An entry with at least 16 proposals in the round multiplies its scale by (nacc / nprop) / target
 * clamped to [1/2, 2], the scale then clamped to [2^-8, 2^8]; every counter restarts at zero.  Returns the entries changed. */
int32_t so_tune_rank(int32_t nc, double* scale, int64_t* nprop, int64_t* nacc, const int32_t* proposed, double target) {
  int changed = 0;
  for (int j = 0; j < 4 * nc; ++j) {
    if (proposed[j & 3] && nprop[j] >= 16) {
      double f = ((double)nacc[j] / (double)nprop[j]) / target;
      f = f < 0.5 ? 0.5 : (f > 2.0 ? 2.0 : f);
      double s = scale[j] * f;
      s = s < 0x1p-8 ? 0x1p-8 : (s > 0x1p8 ? 0x1p8 : s);
      changed += s != scale[j];
      scale[j] = s;
    }
    nprop[j] = 0;
    nacc[j] = 0;
  }
  return changed;
}

/* lo_pt_run (ladder_oracle.c) with the width tuning when steps = 1: the chain at level lvl[g] of rank r proposes with
 * dev_tau * scale[r][lvl[g]][tau], except the two chains of the previous global swap (pair[2], -1: none), which propose with
 * dev_tau; its proposals then count in st_nprop / st_nacc [nproc][nc][4] (null ones too).  After the sweep (and the ladder
 * tuning) lvl is set to the post-sweep levels; at the tuning points every rank is tuned (so_tune_rank) and *st_points counts
 * them; the global swap records its pair.  pairlog [n_iter][G], optional: 1 for the chains that proposed under the pair rule.
 * Arguments otherwise as in lo_pt_run; with steps = 0 this is lo_pt_run. */
int32_t so_pt_run(orc_pt* p, int32_t mode, int32_t tune, int32_t steps, double target, int64_t* n_prop, int64_t* n_acc,
                  int64_t* rows, int64_t* base, int32_t* n_points, double* scale, int64_t* st_nprop, int64_t* st_nacc,
                  int32_t* lvl, int32_t* pair, int32_t* st_points, int32_t n_iter, int8_t* flags, int8_t* itypes,
                  int32_t* swaps, int8_t* pairlog, int32_t record) {
  const rfinv_config* c = &p->c;
  int nc = c->nchains, n = c->nfft, T = c->ntrc;
  size_t G = (size_t)p->nproc * nc;
  int new_cap = p->it_done + n_iter;
  if (new_cap > p->cap_hist) {
    p->likelihood_hist = (double*)realloc(p->likelihood_hist, sizeof(double) * (size_t)new_cap);
    for (int i = p->cap_hist; i < new_cap; ++i) p->likelihood_hist[i] = 0.0;
    p->cap_hist = new_cap;
  }
  const double dev[4] = {c->dev_z, c->dev_dvs, c->dev_dvp, c->dev_sig};
  const int32_t proposed[4] = {1, 1, p->it_dvp > 0, p->it_sig > 0};
  int8_t* fl = (int8_t*)malloc(G);
  int8_t* ty = (int8_t*)malloc(G);
  int8_t* pr = (int8_t*)malloc(G);
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
          double wd[4] = {dev[0], dev[1], dev[2], dev[3]};
          pr[g] = (int8_t)(steps && ((int)g == pair[0] || (int)g == pair[1]));
          if (steps && !pr[g])
            for (int t = 0; t < 4; ++t) wd[t] = dev[t] * scale[((size_t)r * nc + lvl[g]) * 4 + t];
          fl[g] = (int8_t)(steps ? so_mcmc_step(p, w, mis, prop_rft, r, ic, p->temps[g], wd, &itype, &n_eval_tot)
                                 : mcmc_step(p, w, mis, prop_rft, r, ic, p->temps[g], &itype, &n_eval_tot));
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
        if (steps)
          for (size_t g = 0; g < G; ++g) {
            const int tau = so_type(p, ty[g]);
            if (tau < 0 || pr[g]) continue;
            const size_t row = ((g / nc) * nc + lvl[g]) * 4 + tau;
            st_nprop[row]++;
            st_nacc[row] += fl[g] == 1;
          }
        if (flags) memcpy(flags + (size_t)step * G, fl, G);
        if (itypes) memcpy(itypes + (size_t)step * G, ty, G);
        if (pairlog) memcpy(pairlog + (size_t)step * G, pr, G);
        if (mode == 1 && nc >= 2) rank_sweep_rows(p, it - 1, n_prop, n_acc, rows);
        if (tune && tuning_point(it, c->nburn)) {
          if (mode == 1 && nc >= 2)
            for (int r = 0; r < p->nproc; ++r)
              lo_tune_rank(nc, p->temps + (size_t)r * nc, rows + (size_t)r * (nc - 1), base + (size_t)r * (nc - 1), it);
          ++*n_points;
        }
        if (steps) {
          so_levels(p, lvl);
          if (tuning_point(it, c->nburn)) {
            for (int r = 0; r < p->nproc; ++r)
              so_tune_rank(nc, scale + (size_t)r * nc * 4, st_nprop + (size_t)r * nc * 4, st_nacc + (size_t)r * nc * 4, proposed,
                           target);
            ++*st_points;
          }
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
          if (steps) { pair[0] = itarget1; pair[1] = itarget2; }
        }
      }
    }
    free(prop_rft); free(mis); ws_destroy(w);
  }
  p->it_done += n_iter;
  p->n_eval += n_eval_tot;
  free(fl); free(ty); free(pr);
  return 0;
}
