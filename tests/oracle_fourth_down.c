/*
 * TEST INFRASTRUCTURE ONLY: the C oracle's games with a forced fourth-down choice at the start state (include/fmc.h
 * FMC_4TH_POLICY) -- the reference the GPU's decision kernels are compared with.  Iteration 0 takes the chosen branch,
 * written from the branches of the oracle's handle_fourth (oracle/fmc_oracle.c, compiled in unchanged, as are
 * tests/oracle_live.c and tests/oracle_overtime.c).  From iteration 1 the oracle's own loop plays on: regulation as
 * simulate_game_from plays it, then, with overtime, the period loop of overtime_game through ot_possession.  Loaded by
 * tests/oracle_fourth_down.py.
 */
#include "oracle_overtime.c"

enum { FO_4TH_POLICY = 0, FO_4TH_GO, FO_4TH_FG, FO_4TH_PUNT };

/* handle_fourth with the branch `choice` instead of the go / kick draws; FO_4TH_POLICY is handle_fourth itself.  Each
 * branch reads the draw slots handle_fourth's branch reads.  Returns 1 when no play follows. */
static int forced_fourth(FoGame *G, FoState *s, FoRng *rng, int choice) {
    if (choice == FO_4TH_POLICY) return handle_fourth(G, s, rng);
    const int team = s->offense;
    const double ytg = s->ytg;
    if (choice == FO_4TH_GO) { s->going = 1; G->n_go++; return 0; }
    if (choice == FO_4TH_FG) {
        G->n_fga++;
        double p = field_goal_prob(ytg + 17);
        int good = draw(rng, S_U_FG, 0) < p;
        tick_clock(s, 12);
        if (good) { G->n_fg++; s->score[team] += 3; change_possession(s, 1, 75.0); }
        else change_possession(s, 1, 100.0 - ytg);
        return 1;
    }
    G->n_punt++;
    double gross = pymax(30.0, 43.0 + 6.0 * draw(rng, S_Z_GROSS, 1));
    double ret = pymax(0.0, 6.0 + 3.0 * draw(rng, S_Z_RET, 1));
    double net = gross - ret;
    if (ytg <= 60) {
        double tb = softclip((60.0 - ytg) / 60.0, 0.10, 0.55);
        if (draw(rng, S_U_TB, 0) < tb) net = ytg - 25.0;
    }
    net = softclip(net, 15.0, ytg - 1.0);
    int inet = (int)net;
    tick_clock(s, 16);
    double spot = softclip(100.0 - (ytg - inet), 1, 99);
    change_possession(s, 1, spot);
    return 1;
}

/* One game from `start` with `choice` at iteration 0; max_periods 0: regulation only. */
static void fourth_down_game(FoGame *G, FoRng *rng, int first, const FoStart *start, int choice, int max_periods,
                             int snap_clock, int score_out[2], int *iters_out, int *periods_out, double *trace,
                             double *box_save) {
    FoState s;
    s.offense = start->offense < 0 ? first : start->offense;
    s.sec = start->sec; s.down = start->down; s.dist = start->dist; s.ytg = start->ytg;
    s.period = s.sec > 0 ? 4 - ((s.sec - 1) / 900) : 4;
    s.going = 0;
    s.score[0] = start->score[0]; s.score[1] = start->score[1];
    int it = 0;
    while (s.sec > 0) {                                 /* simulate_game_from's loop */
        rng->iter = it;
        rng->have[0] = rng->have[1] = rng->have[2] = rng->have[3] = 0;
        if (trace && it < FO_MAX_ITERS) {
            double *t = trace + (size_t)it * FO_TRACE_COLS;
            t[0] = (s.offense == first) ? 1.0 : 0.0; t[1] = s.down; t[2] = s.sec;
            t[3] = s.score[first]; t[4] = s.score[first ^ 1]; t[5] = s.dist; t[6] = s.ytg; t[7] = s.going;
        }
        ++it;
        if (forced_fourth(G, &s, rng, it == 1 ? choice : FO_4TH_POLICY)) continue;
        simulate_play(G, &s, rng);
    }
    G->iters += it;
    int k = 0;
    if (max_periods > 0 && s.score[0] == s.score[1]) {   /* overtime_game's period loop */
        FoOt o;
        o.G = G; o.rng = rng; o.first = first; o.it = it; o.snap_clock = snap_clock; o.trace = trace;
        o.box_save = box_save;
        o.s.period = 4;
        o.s.score[0] = s.score[0]; o.s.score[1] = s.score[1];
        for (k = 1;; ++k) {
            const int a = first ^ ((k - 1) & 1);
            if (!ot_possession(&o, k, a, 0)) break;
            if (!ot_possession(&o, k, a ^ 1, 1)) break;
            if (o.s.score[0] != o.s.score[1] || k == max_periods) break;
        }
        s.score[0] = o.s.score[0]; s.score[1] = o.s.score[1];
        it = o.it;
    }
    score_out[0] = s.score[0]; score_out[1] = s.score[1];
    *iters_out = it;
    *periods_out = k;
}

/*
 * fo_overtime_simulate with a forced choice per start: choices[n_starts] (FO_4TH_*; a non-zero choice needs down 4 and
 * sec > 0), and max_periods 0 for regulation only.  Same outputs.
 */
int fo_fourth_down_simulate(const FoConfig *cfg, const FoTeamUsage *usage, int n_slots, double *players,
                            const FoStart *starts, long n_starts, long n, long game0, int matchup, int rng_mode,
                            const double *stream, uint64_t seed, int max_periods, int snap_clock, const int *choices,
                            int *scores, int *iters, int *periods, double *trace, long *counters, int n_threads) {
    if (!starts || !choices || (n_starts != 1 && n_starts != n)) return -3;
    if (max_periods < 0 || max_periods > FO_OT_MAX_PERIODS || snap_clock < 1 || snap_clock > 900) return -3;
    for (long i = 0; i < n_starts; ++i) {
        if (choices[i] < FO_4TH_POLICY || choices[i] > FO_4TH_PUNT) return -3;
        if (choices[i] != FO_4TH_POLICY && (starts[i].down != 4 || starts[i].sec <= 0)) return -3;
    }
    for (int m = FO_PASS_STAGE1; m <= FO_SACK_YARDS; ++m) {
        if (m == FO_PASS_STAGE2 && cfg->stage2_mode == 0) continue;
        if (!g_forest[m].loaded) return -2;
    }
    if (cfg->policy == 1 && !g_forest[FO_PLAY_MODEL].loaded) return -2;
    if (usage && n_slots < 0) return -3;
    long tot[16];
    memset(tot, 0, sizeof(tot));
#ifdef _OPENMP
    if (n_threads > 0) omp_set_num_threads(n_threads);
#endif
#pragma omp parallel
    {
        FoGame G;
        game_constants(&G, cfg);
        double *box_save = NULL;
        if (usage) {
            G.usage = usage;
            G.n_slots = n_slots;
            for (int t = 0; t < 2; ++t)
                for (int r = 0; r < 3; ++r) {
                    const FoUsage *u = &usage[t].role[r];
                    double acc = 0.0;
                    for (int i = 0; i < u->n; ++i) { acc += u->share[i]; G.cdf[t][r][i] = acc; }   /* np.cumsum */
                    for (int i = 0; i < u->n; ++i) G.cdf[t][r][i] /= acc;                           /* cdf /= cdf[-1] */
                }
            box_save = (double *)malloc((size_t)2 * (n_slots > 0 ? n_slots : 1) * FO_PLAYER_FIELDS * sizeof(double));
        }
#pragma omp for schedule(dynamic, 16)
        for (long i = 0; i < n; ++i) {
            long g = game0 + i;
            FoRng rng;
            memset(&rng, 0, sizeof(rng));
            rng.mode = rng_mode;
            rng.rec = stream ? stream + (size_t)i * FO_MAX_ITERS * FO_N_SLOTS : NULL;
            rng.key[0] = (uint32_t)seed; rng.key[1] = (uint32_t)(seed >> 32);
            rng.ctr_game[0] = (uint32_t)((uint64_t)g); rng.ctr_game[1] = (uint32_t)((uint64_t)g >> 32);
            rng.ctr_game[2] = (uint32_t)matchup;
            int it = 0, k = 0;
            const long si = n_starts == 1 ? 0 : i;
            G.box = (usage && players) ? players + (size_t)i * 2 * n_slots * FO_PLAYER_FIELDS : NULL;
            G.cur[0] = G.cur[1] = G.cur[2] = 0;
            fourth_down_game(&G, &rng, (int)(g & 1), starts + si, choices[si], max_periods, snap_clock, scores + 2 * i,
                             &it, &k, trace ? trace + (size_t)i * FO_MAX_ITERS * FO_TRACE_COLS : NULL, box_save);
            if (iters) iters[i] = it;
            if (periods) periods[i] = k;
        }
        free(box_save);
#pragma omp critical
        {
            tot[0] += G.plays; tot[1] += G.iters; tot[2] += G.n_pass; tot[3] += G.n_comp; tot[4] += G.n_inc;
            tot[5] += G.n_int; tot[6] += G.n_sack; tot[7] += G.n_run; tot[8] += G.n_td; tot[9] += G.n_fga;
            tot[10] += G.n_fg; tot[11] += G.n_punt; tot[12] += G.n_go;
        }
    }
    if (counters) memcpy(counters, tot, sizeof(tot));
    return 0;
}
