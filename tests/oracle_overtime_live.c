/*
 * TEST INFRASTRUCTURE ONLY: the C oracle's games started inside overtime (include/fmc.h fmc_overtime_state) -- the
 * reference the GPU's overtime start states (fmc_set_start_states_overtime) are compared with -- and the overtime games of
 * tests/oracle_overtime.c with the overtime state of every iteration recorded, which gives the start states of the resume
 * tests.  oracle/fmc_oracle.c, tests/oracle_live.c, tests/oracle_overtime.c and tests/oracle_fourth_down.c are compiled
 * in unchanged.  As in oracle_overtime.c the loop is written as periods and possessions (the rest of the possession in
 * progress, then whole possessions), not as the kernel's iteration-start state machine.  Loaded by
 * tests/oracle_overtime_live.py.
 */
#include "oracle_fourth_down.c"

/* include/fmc.h fmc_overtime_state */
typedef struct {
    int period, possession, two_point_try, reserved;
} FoOtStart;

/* oracle_overtime.c's FoOt plus the overtime state of the snap being played, the forced choice of the game's first snap
 * and the optional per-iteration record of the state */
typedef struct {
    FoOt o;
    int k, second, is_try;
    int choice;     /* FO_4TH_*: the first snap's branch; FO_4TH_POLICY afterwards */
    int *states;    /* optional [FO_MAX_ITERS][3]: period, possession (1, 2), try of each overtime iteration */
} FoOtLive;

/* ot_snap with the forced choice and the state record */
static int ol_snap(FoOtLive *l) {
    FoOt *o = &l->o;
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
    if (l->states) {
        int *r = l->states + (size_t)o->it * 3;
        r[0] = l->k; r[1] = l->second + 1; r[2] = l->is_try;
    }
    ++o->it;
    ++o->G->iters;
    const int c = l->choice;
    l->choice = FO_4TH_POLICY;
    if (!forced_fourth(o->G, s, o->rng, c)) simulate_play(o->G, s, o->rng);
    return 1;
}

/* ot_try: a two-point try by `team`, 2 points iff its one snap is a touchdown, no box line credited */
static int ol_try(FoOtLive *l, int team) {
    FoOt *o = &l->o;
    FoState *s = &o->s;
    s->offense = team; s->down = 1; s->dist = 3.0; s->ytg = 3.0; s->going = 0;
    const size_t box_n = o->G->box ? (size_t)2 * o->G->n_slots * FO_PLAYER_FIELDS : 0;
    if (box_n) memcpy(o->box_save, o->G->box, box_n * sizeof(double));
    const int before = s->score[team];
    l->is_try = 1;
    const int alive = ol_snap(l);
    l->is_try = 0;
    if (!alive) return 0;
    if (box_n) memcpy(o->G->box, o->box_save, box_n * sizeof(double));
    s->score[team] = before + (s->score[team] - before == 7 ? 2 : 0);
    return 1;
}

/* The rest of the possession of `team` in period l->k from the current state: its snaps while it has the ball, then
 * the try of a period-2 touchdown unless the touchdown won.  Returns 0 when the game ends during it. */
static int ol_rest_of_possession(FoOtLive *l, int team) {
    FoState *s = &l->o.s;
    const int before = s->score[team];
    while (s->offense == team)
        if (!ol_snap(l)) return 0;
    if (l->k == 2 && s->score[team] - before == 7) {
        s->score[team] -= 1;
        if (l->second && s->score[team] > s->score[team ^ 1]) return 0;
        return ol_try(l, team);
    }
    return 1;
}

/* ot_possession: the whole possession of `team` in period l->k */
static int ol_possession(FoOtLive *l, int team) {
    if (l->k >= 3) return ol_try(l, team);
    FoState *s = &l->o.s;
    s->offense = team; s->down = 1; s->dist = 10.0; s->ytg = 25.0; s->going = 0;
    return ol_rest_of_possession(l, team);
}

/* overtime_game's period loop from the start of period k, team a with its first possession; returns the last period
 * played */
static int ol_periods(FoOtLive *l, int k, int a, int max_periods) {
    FoState *s = &l->o.s;
    for (;; ++k, a ^= 1) {
        l->k = k; l->second = 0;
        if (!ol_possession(l, a)) return k;
        l->second = 1;
        if (!ol_possession(l, a ^ 1)) return k;
        if (s->score[0] != s->score[1] || k == max_periods) return k;
    }
}

static void ol_init(FoOtLive *l, FoGame *G, FoRng *rng, int first, int snap_clock, double *trace, double *box_save,
                    int *states) {
    memset(l, 0, sizeof(*l));
    l->o.G = G; l->o.rng = rng; l->o.first = first; l->o.snap_clock = snap_clock; l->o.trace = trace;
    l->o.box_save = box_save;
    l->o.s.period = 4;
    l->choice = FO_4TH_POLICY;
    l->states = states;
}

/* overtime_game with the state record: regulation as simulate_game_from plays it, then the period loop */
static void overtime_game_states(FoGame *G, FoRng *rng, int first, const FoStart *start, int max_periods, int snap_clock,
                                 int score_out[2], int *iters_out, int *periods_out, double *trace, double *box_save,
                                 int *states) {
    int it = 0, k = 0;
    simulate_game_from(G, rng, first, start, score_out, &it, trace);
    if (score_out[0] == score_out[1]) {
        FoOtLive l;
        ol_init(&l, G, rng, first, snap_clock, trace, box_save, states);
        l.o.it = it;
        l.o.s.score[0] = score_out[0]; l.o.s.score[1] = score_out[1];
        k = ol_periods(&l, 1, first, max_periods);
        score_out[0] = l.o.s.score[0]; score_out[1] = l.o.s.score[1];
        it = l.o.it;
    }
    *iters_out = it;
    *periods_out = k;
}

/* A game from a snap inside overtime: the rest of the possession in progress (or the try), with `choice` at its first
 * snap, the other possession of the period if it is still to come, then the period loop while the score is level. */
static void overtime_start_game(FoGame *G, FoRng *rng, int first, const FoStart *start, const FoOtStart *ot, int choice,
                                int max_periods, int snap_clock, int score_out[2], int *iters_out, int *periods_out,
                                double *trace, double *box_save, int *states) {
    FoOtLive l;
    ol_init(&l, G, rng, first, snap_clock, trace, box_save, states);
    FoState *s = &l.o.s;
    const int team = start->offense;
    s->offense = team; s->down = start->down; s->dist = start->dist; s->ytg = start->ytg; s->going = 0;
    s->score[0] = start->score[0]; s->score[1] = start->score[1];
    int k = ot->period;
    const int second = ot->possession == 2;
    const int a = second ? team ^ 1 : team;            /* first possession of period k */
    l.k = k; l.second = second; l.choice = choice;
    int alive = ot->two_point_try ? ol_try(&l, team) : ol_rest_of_possession(&l, team);
    if (alive && !second) {
        l.second = 1;
        alive = ol_possession(&l, a ^ 1);
    }
    if (alive && s->score[0] == s->score[1] && k < max_periods) k = ol_periods(&l, k + 1, a ^ 1, max_periods);
    score_out[0] = s->score[0]; score_out[1] = s->score[1];
    *iters_out = l.o.it;
    *periods_out = k;
}

static int ol_check(const FoConfig *cfg, const FoTeamUsage *usage, int n_slots, int max_periods, int snap_clock) {
    if (max_periods < 1 || max_periods > FO_OT_MAX_PERIODS || snap_clock < 1 || snap_clock > 900) return -3;
    for (int m = FO_PASS_STAGE1; m <= FO_SACK_YARDS; ++m) {
        if (m == FO_PASS_STAGE2 && cfg->stage2_mode == 0) continue;
        if (!g_forest[m].loaded) return -2;
    }
    if (cfg->policy == 1 && !g_forest[FO_PLAY_MODEL].loaded) return -2;
    if (usage && n_slots < 0) return -3;
    return 0;
}

/* The per-launch plumbing of oracle_overtime.c's entries; ot == NULL: overtime_game_states from starts, else
 * overtime_start_game from (starts, ot, choices). */
static int ol_run(const FoConfig *cfg, const FoTeamUsage *usage, int n_slots, double *players, const FoStart *starts,
                  const FoOtStart *ot, const int *choices, long n_starts, long n, long game0, int matchup, int rng_mode,
                  const double *stream, uint64_t seed, int max_periods, int snap_clock, int *scores, int *iters,
                  int *periods, double *trace, int *states, long *counters, int n_threads) {
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
            double *tr = trace ? trace + (size_t)i * FO_MAX_ITERS * FO_TRACE_COLS : NULL;
            int *sr = states ? states + (size_t)i * FO_MAX_ITERS * 3 : NULL;
            if (ot)
                overtime_start_game(&G, &rng, (int)(g & 1), starts + si, ot + si, choices ? choices[si] : FO_4TH_POLICY,
                                    max_periods, snap_clock, scores + 2 * i, &it, &k, tr, box_save, sr);
            else
                overtime_game_states(&G, &rng, (int)(g & 1), starts + si, max_periods, snap_clock, scores + 2 * i, &it,
                                     &k, tr, box_save, sr);
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

/*
 * fo_overtime_simulate plus states[n][FO_MAX_ITERS][3] (optional): period, possession (1, 2) and try (0, 1) of every
 * overtime iteration; regulation iterations are left as they are.
 */
int fo_overtime_states_simulate(const FoConfig *cfg, const FoTeamUsage *usage, int n_slots, double *players,
                                const FoStart *starts, long n_starts, long n, long game0, int matchup, int rng_mode,
                                const double *stream, uint64_t seed, int max_periods, int snap_clock, int *scores,
                                int *iters, int *periods, double *trace, int *states, long *counters, int n_threads) {
    if (!starts || (n_starts != 1 && n_starts != n)) return -3;
    const int rc = ol_check(cfg, usage, n_slots, max_periods, snap_clock);
    if (rc) return rc;
    return ol_run(cfg, usage, n_slots, players, starts, NULL, NULL, n_starts, n, game0, matchup, rng_mode, stream, seed,
                  max_periods, snap_clock, scores, iters, periods, trace, states, counters, n_threads);
}

/*
 * Games started inside overtime: starts[i] (offense 0 / 1, down, distance, yards to goal, score; sec is not read) with
 * ot[i] (period 1..max_periods, possession 1 / 2, try) and choices[i] (FO_4TH_*, NULL = all policy) at the first
 * snap.  The state is taken as given: the library's validation is tested against the library, not here.  Outputs as
 * fo_overtime_states_simulate's; periods[i] = the last period played.
 */
int fo_overtime_start_simulate(const FoConfig *cfg, const FoTeamUsage *usage, int n_slots, double *players,
                               const FoStart *starts, const FoOtStart *ot, const int *choices, long n_starts, long n,
                               long game0, int matchup, int rng_mode, const double *stream, uint64_t seed,
                               int max_periods, int snap_clock, int *scores, int *iters, int *periods, double *trace,
                               int *states, long *counters, int n_threads) {
    if (!starts || !ot || (n_starts != 1 && n_starts != n)) return -3;
    const int rc = ol_check(cfg, usage, n_slots, max_periods, snap_clock);
    if (rc) return rc;
    for (long i = 0; i < n_starts; ++i) {
        if (starts[i].offense < 0 || starts[i].offense > 1) return -3;
        if (ot[i].period < 1 || ot[i].period > max_periods || (ot[i].possession != 1 && ot[i].possession != 2)) return -3;
        if (choices && (choices[i] < FO_4TH_POLICY || choices[i] > FO_4TH_PUNT)) return -3;
        if (choices && choices[i] != FO_4TH_POLICY && (starts[i].down != 4 || ot[i].two_point_try)) return -3;
    }
    return ol_run(cfg, usage, n_slots, players, starts, ot, choices, n_starts, n, game0, matchup, rng_mode, stream, seed,
                  max_periods, snap_clock, scores, iters, periods, trace, states, counters, n_threads);
}
