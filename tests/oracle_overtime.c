/*
 * TEST INFRASTRUCTURE ONLY: the C oracle's games played to a result under college overtime rules (include/fmc.h
 * FMC_OT_MAX_PERIODS) -- the reference the GPU's overtime (fmc_simulate_overtime) is compared with.  Regulation is
 * tests/oracle_live.c's simulate_game_from, unchanged (oracle/fmc_oracle.c is compiled in unchanged too).  A game level
 * after it goes on in periods of one possession per team, each snap played by the oracle's own handle_fourth /
 * simulate_play with the clock set to snap_clock first (simulate_play does nothing at 0 s, which is why the clock is
 * never 0 in overtime).  The loop is written as periods and possessions, not as the kernel's iteration-start state
 * machine, so that the two state the rules independently.  Loaded by tests/oracle_overtime.py.
 */
#include "oracle_live.c"

#define FO_OT_MAX_PERIODS 16

typedef struct {
    FoGame *G;
    FoRng *rng;
    FoState s;
    int first;        /* the opening-kickoff receiver, g & 1 */
    int it;           /* iterations so far, regulation included */
    int snap_clock;
    double *trace;
    double *box_save; /* [2][n_slots][FO_PLAYER_FIELDS] scratch for tries */
} FoOt;

/* One overtime snap (one iteration).  Returns 0 when the iteration cap ends the game first. */
static int ot_snap(FoOt *o) {
    if (o->it >= FO_MAX_ITERS) return 0;
    FoState *s = &o->s;
    s->sec = o->snap_clock;
    o->rng->iter = o->it;
    o->rng->have[0] = o->rng->have[1] = o->rng->have[2] = o->rng->have[3] = 0;
    if (o->trace) {
        double *t = o->trace + (size_t)o->it * FO_TRACE_COLS;
        t[0] = (s->offense == o->first) ? 1.0 : 0.0; t[1] = s->down; t[2] = s->sec;
        t[3] = s->score[o->first]; t[4] = s->score[o->first ^ 1]; t[5] = s->dist; t[6] = s->ytg; t[7] = s->going;
    }
    ++o->it;
    ++o->G->iters;
    if (!handle_fourth(o->G, s, o->rng)) simulate_play(o->G, s, o->rng);
    return 1;
}

/* A two-point try by `team`: 2 points iff its one snap is a touchdown; nothing else of it counts, box lines included.
 * Returns 0 when the iteration cap ends the game first. */
static int ot_try(FoOt *o, int team) {
    FoState *s = &o->s;
    s->offense = team; s->down = 1; s->dist = 3.0; s->ytg = 3.0; s->going = 0;
    const size_t box_n = o->G->box ? (size_t)2 * o->G->n_slots * FO_PLAYER_FIELDS : 0;
    if (box_n) memcpy(o->box_save, o->G->box, box_n * sizeof(double));
    const int before = s->score[team];
    if (!ot_snap(o)) return 0;
    if (box_n) memcpy(o->G->box, o->box_save, box_n * sizeof(double));
    s->score[team] = before + (s->score[team] - before == 7 ? 2 : 0);
    return 1;
}

/* The possession of `team` in period k, second = it is the period's second possession.  Returns 0 when the game
 * ends during it (the iteration cap, or a period-2 touchdown that wins). */
static int ot_possession(FoOt *o, int k, int team, int second) {
    if (k >= 3) return ot_try(o, team);
    FoState *s = &o->s;
    s->offense = team; s->down = 1; s->dist = 10.0; s->ytg = 25.0; s->going = 0;
    const int before = s->score[team];
    while (s->offense == team)
        if (!ot_snap(o)) return 0;
    if (k == 2 && s->score[team] - before == 7) {       /* a touchdown is worth 6 in period 2, then the try */
        s->score[team] -= 1;
        if (second && s->score[team] > s->score[team ^ 1]) return 0;
        return ot_try(o, team);
    }
    return 1;
}

/* simulate_game_from, then overtime while the score is level.  *periods_out = overtime periods begun. */
static void overtime_game(FoGame *G, FoRng *rng, int first, const FoStart *start, int max_periods, int snap_clock,
                          int score_out[2], int *iters_out, int *periods_out, double *trace, double *box_save) {
    int it = 0;
    simulate_game_from(G, rng, first, start, score_out, &it, trace);
    int k = 0;
    if (score_out[0] == score_out[1]) {
        FoOt o;
        o.G = G; o.rng = rng; o.first = first; o.it = it; o.snap_clock = snap_clock; o.trace = trace;
        o.box_save = box_save;
        o.s.period = 4;
        o.s.score[0] = score_out[0]; o.s.score[1] = score_out[1];
        for (k = 1;; ++k) {
            const int a = first ^ ((k - 1) & 1);            /* first possession of period k */
            if (!ot_possession(&o, k, a, 0)) break;
            if (!ot_possession(&o, k, a ^ 1, 1)) break;
            if (o.s.score[0] != o.s.score[1] || k == max_periods) break;
        }
        score_out[0] = o.s.score[0]; score_out[1] = o.s.score[1];
        it = o.it;
    }
    *iters_out = it;
    *periods_out = k;
}

/*
 * fo_live_simulate with overtime: same arguments and outputs, plus max_periods (1..16), snap_clock (1..900) and
 * periods[n] (overtime periods of each game, 0 = decided in regulation).
 */
int fo_overtime_simulate(const FoConfig *cfg, const FoTeamUsage *usage, int n_slots, double *players,
                         const FoStart *starts, long n_starts, long n, long game0, int matchup, int rng_mode,
                         const double *stream, uint64_t seed, int max_periods, int snap_clock, int *scores, int *iters,
                         int *periods, double *trace, long *counters, int n_threads) {
    if (!starts || (n_starts != 1 && n_starts != n)) return -3;
    if (max_periods < 1 || max_periods > FO_OT_MAX_PERIODS || snap_clock < 1 || snap_clock > 900) return -3;
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
            G.box = (usage && players) ? players + (size_t)i * 2 * n_slots * FO_PLAYER_FIELDS : NULL;
            G.cur[0] = G.cur[1] = G.cur[2] = 0;
            overtime_game(&G, &rng, (int)(g & 1), starts + (n_starts == 1 ? 0 : i), max_periods, snap_clock,
                          scores + 2 * i, &it, &k, trace ? trace + (size_t)i * FO_MAX_ITERS * FO_TRACE_COLS : NULL,
                          box_save);
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
