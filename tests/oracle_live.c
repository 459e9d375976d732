/*
 * TEST INFRASTRUCTURE ONLY: the C oracle (oracle/fmc_oracle.c, compiled into this unit unchanged) with a start record
 * per game -- the reference the GPU's start states (fmc_set_start_states) are compared with.  The reference itself has
 * no in-game entry point: simulate_game always starts at the opening kickoff.  From a start record the oracle's own
 * rules apply unchanged (handle_fourth, simulate_play); the period follows from the clock exactly as tick_clock derives
 * it, and timeouts stay unspent as always.  Loaded by tests/oracle_live.py; build flags are oracle/Makefile's.
 */
#include "fmc_oracle.c"

/* The state a game starts from (include/fmc.h fmc_game_state). */
typedef struct {
    int offense;              /* 0 / 1, or -1: the team that receives the opening kickoff (game id parity) */
    int sec, down;
    int score[2];
    double dist, ytg;
} FoStart;

/* simulate_game (FMC:1428-1464) from `start` instead of the kickoff; first = the kickoff receiver (g & 1). */
static void simulate_game_from(FoGame *G, FoRng *rng, int first, const FoStart *start, int score_out[2], int *iters_out,
                               double *trace) {
    FoState s;
    s.offense = start->offense < 0 ? first : start->offense;
    s.sec = start->sec; s.down = start->down; s.dist = start->dist; s.ytg = start->ytg;
    s.period = s.sec > 0 ? 4 - ((s.sec - 1) / 900) : 4;
    s.going = 0;
    s.score[0] = start->score[0]; s.score[1] = start->score[1];
    int it = 0;
    while (s.sec > 0) {
        rng->iter = it;
        rng->have[0] = rng->have[1] = rng->have[2] = rng->have[3] = 0;
        if (trace && it < FO_MAX_ITERS) {
            double *t = trace + (size_t)it * FO_TRACE_COLS;
            t[0] = (s.offense == first) ? 1.0 : 0.0; t[1] = s.down; t[2] = s.sec;
            t[3] = s.score[first]; t[4] = s.score[first ^ 1]; t[5] = s.dist; t[6] = s.ytg; t[7] = s.going;
        }
        ++it;
        if (handle_fourth(G, &s, rng)) continue;
        simulate_play(G, &s, rng);
    }
    score_out[0] = s.score[0]; score_out[1] = s.score[1];
    *iters_out = it;
    G->iters += it;
}

/*
 * fo_simulate / fo_simulate_players (usage == NULL: no player box) with game i of [game0, game0 + n) starting from
 * starts[i] (n_starts == n) or starts[0] (n_starts == 1).  Arguments and outputs as simulate_range's.
 */
int fo_live_simulate(const FoConfig *cfg, const FoTeamUsage *usage, int n_slots, double *players,
                     const FoStart *starts, long n_starts, long n, long game0, int matchup, int rng_mode,
                     const double *stream, uint64_t seed, int *scores, int *iters, double *trace, long *counters,
                     int n_threads) {
    if (!starts || (n_starts != 1 && n_starts != n)) return -3;
    for (int m = FO_PASS_STAGE1; m <= FO_SACK_YARDS; ++m) {
        if (m == FO_PASS_STAGE2 && cfg->stage2_mode == 0) continue;
        if (!g_forest[m].loaded) return -2;
    }
    if (cfg->policy == 1 && !g_forest[FO_PLAY_MODEL].loaded) return -2;
    if (usage) {
        if (n_slots < 0) return -3;
        for (int t = 0; t < 2; ++t)
            for (int r = 0; r < 3; ++r) {
                const FoUsage *u = &usage[t].role[r];
                if (u->n < 1 || u->n > FO_MAX_USAGE) return -3;
                for (int i = 0; i < u->n; ++i)
                    if (u->slot[i] >= n_slots) return -3;
            }
    }
    long tot[16];
    memset(tot, 0, sizeof(tot));
#ifdef _OPENMP
    if (n_threads > 0) omp_set_num_threads(n_threads);
#endif
#pragma omp parallel
    {
        FoGame G;
        game_constants(&G, cfg);
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
            int it = 0;
            G.box = (usage && players) ? players + (size_t)i * 2 * n_slots * FO_PLAYER_FIELDS : NULL;
            G.cur[0] = G.cur[1] = G.cur[2] = 0;
            simulate_game_from(&G, &rng, (int)(g & 1), starts + (n_starts == 1 ? 0 : i), scores + 2 * i, &it,
                               trace ? trace + (size_t)i * FO_MAX_ITERS * FO_TRACE_COLS : NULL);
            if (iters) iters[i] = it;
        }
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
