/*
 * TEST INFRASTRUCTURE ONLY: the scoring sequence of the C oracle's games (next score, drive result, race to N), the
 * reference the GPU's sequence outputs (fmc_simulate_markets) are compared with.  It compiles tests/oracle_live.c, and
 * with it oracle/fmc_oracle.c, unchanged into itself and plays the oracle's own game loop from a start record.  Nothing
 * of the rules is restated: after every iteration the outcome is read from the deltas of the oracle's own counters
 * (n_td, n_fg, n_fga, n_punt, n_int), the scores, the team on offense and the period.  Loaded by
 * tests/oracle_sequence.py; build flags are oracle/Makefile's.
 */
#include "oracle_live.c"

/* include/fmc.h's layout of the sequence words and codes, restated for a build without the library's header */
enum { SEQ_TD = 0, SEQ_FG = 1 };
enum { DR_TD = 0, DR_FG, DR_MISSED_FG, DR_PUNT, DR_INT, DR_DOWNS, DR_HALF, DR_GAME };
#define SEQ_NONE 0xFFFFFFFFu
#define N_RACE 5
static const int kTargets[N_RACE] = {10, 15, 20, 25, 30};
enum { RACE_A = 0, RACE_B = 1, RACE_NEITHER = 2, RACE_SETTLED = -1, RACE_OPEN = -2 };

/* One game from `start` (first = the kickoff receiver, g & 1): the oracle's loop of simulate_game_from (oracle_live.c),
 * observed after every iteration.  seq[0] = next score team | kind << 1 | clock << 2 or SEQ_NONE, seq[1] = drive result
 * | clock << 8, race[t] = RACE_A / RACE_B / RACE_NEITHER / RACE_SETTLED. */
static void sequence_game(FoGame *G, FoRng *rng, int first, const FoStart *start, int score_out[2], int *iters_out,
                          uint32_t seq[2], signed char race[N_RACE]) {
    FoState s;
    s.offense = start->offense < 0 ? first : start->offense;
    s.sec = start->sec; s.down = start->down; s.dist = start->dist; s.ytg = start->ytg;
    s.period = s.sec > 0 ? 4 - ((s.sec - 1) / 900) : 4;
    s.going = 0;
    s.score[0] = start->score[0]; s.score[1] = start->score[1];
    seq[0] = SEQ_NONE;
    int drive_open = 1;
    for (int t = 0; t < N_RACE; ++t)
        race[t] = (s.score[0] >= kTargets[t] || s.score[1] >= kTargets[t]) ? RACE_SETTLED : RACE_OPEN;
    int it = 0;
    while (s.sec > 0) {
        rng->iter = it;
        rng->have[0] = rng->have[1] = rng->have[2] = rng->have[3] = 0;
        ++it;
        const long td0 = G->n_td, fg0 = G->n_fg, fga0 = G->n_fga, punt0 = G->n_punt, int0 = G->n_int;
        const int off0 = s.offense, per0 = s.period, snap = s.sec, a0 = s.score[0], b0 = s.score[1];
        if (!handle_fourth(G, &s, rng)) simulate_play(G, &s, rng);
        const int td = G->n_td > td0, fg = G->n_fg > fg0, fga = G->n_fga > fga0, punt = G->n_punt > punt0,
                  ic = G->n_int > int0;
        if (td || fg) {
            const int team = s.score[0] != a0 ? 0 : 1;
            const int before = team == 0 ? a0 : b0;
            if (seq[0] == SEQ_NONE) seq[0] = (uint32_t)team | ((uint32_t)(td ? SEQ_TD : SEQ_FG) << 1) | ((uint32_t)snap << 2);
            for (int t = 0; t < N_RACE; ++t)
                if (race[t] == RACE_OPEN && before < kTargets[t] && s.score[team] >= kTargets[t] && s.score[team ^ 1] < kTargets[t])
                    race[t] = (signed char)team;
        }
        if (drive_open) {
            /* the halftime change of possession flips the offense once more after a turnover on downs in the same play */
            const int half = per0 <= 2 && s.period >= 3;
            const int flipped = (s.offense != off0) != half;
            int code = -1;
            if (td) code = DR_TD;
            else if (fg) code = DR_FG;
            else if (fga) code = DR_MISSED_FG;
            else if (punt) code = DR_PUNT;
            else if (ic) code = DR_INT;
            else if (flipped) code = DR_DOWNS;
            else if (half) code = DR_HALF;
            if (code >= 0) { seq[1] = (uint32_t)code | ((uint32_t)snap << 8); drive_open = 0; }
        }
    }
    if (drive_open) seq[1] = DR_GAME;
    for (int t = 0; t < N_RACE; ++t)
        if (race[t] == RACE_OPEN) race[t] = RACE_NEITHER;      /* both teams are still below the target */
    score_out[0] = s.score[0]; score_out[1] = s.score[1];
    *iters_out = it;
    G->iters += it;
}

/* Games [game0, game0 + n) of one matchup from starts[i] (n_starts == n) or starts[0]: scores, iterations, sequence
 * words [n][2] and race results [n][N_RACE].  usage (or NULL), rng_mode / stream / seed as fo_live_simulate's; the
 * player box is not kept. */
int fo_sequence_simulate(const FoConfig *cfg, const FoTeamUsage *usage, const FoStart *starts, long n_starts, long n, long game0, int matchup,
                         int rng_mode, const double *stream, uint64_t seed, int *scores, int *iters, uint32_t *seq,
                         signed char *race, int n_threads) {
    if (!starts || (n_starts != 1 && n_starts != n)) return -3;
    for (int m = FO_PASS_STAGE1; m <= FO_SACK_YARDS; ++m) {
        if (m == FO_PASS_STAGE2 && cfg->stage2_mode == 0) continue;
        if (!g_forest[m].loaded) return -2;
    }
    if (cfg->policy == 1 && !g_forest[FO_PLAY_MODEL].loaded) return -2;
#ifdef _OPENMP
    if (n_threads > 0) omp_set_num_threads(n_threads);
#endif
#pragma omp parallel
    {
        FoGame G;
        game_constants(&G, cfg);
        if (usage) {
            G.usage = usage;
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
            G.box = NULL;
            G.cur[0] = G.cur[1] = G.cur[2] = 0;
            int it = 0;
            sequence_game(&G, &rng, (int)(g & 1), starts + (n_starts == 1 ? 0 : i), scores + 2 * i, &it, seq + 2 * i,
                          race + (size_t)N_RACE * i);
            if (iters) iters[i] = it;
        }
    }
    return 0;
}
