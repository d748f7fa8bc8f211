/*
 * tests/alphabeta_oracle.c -- TEST INFRASTRUCTURE ONLY: the CPU reference of oth_alphabeta.
 *
 * The search of include/othello_b200.h restated on the CPU oracle's mailbox boards and rules (oracle/othello_oracle.c,
 * pinned against the reference's goldens), which this file includes unchanged: plain negamax and fail-hard alpha-beta
 * in natural ascending action order (deliberately not the kernel's ordering).  tests/alphabeta_oracle.py compiles it
 * into a temporary directory with the oracle's flags.
 */
#include "../oracle/othello_oracle.c"


/* The search of oth_alphabeta (include/othello_b200.h) restated on mailbox boards: plain negamax and fail-hard
 * alpha-beta in natural ascending action order (deliberately not the kernel's ordering).  Values are from the
 * side to move; every ply, a forced pass included, costs one depth level. */
#define AB_NONE INT32_MIN
#define AB_WIN 10000
#define AB_INF (1 << 30)
#define AB_UNLIMITED (1 << 20)

static const int AB_W[NSQ] = {
    100, -20, 10, 5, 5, 10, -20, 100, -20, -50, -2, -2, -2, -2, -50, -20, 10, -2, -1, -1, -1, -1, -2, 10,
    5,   -2,  -1, -1, -1, -1, -2, 5,  5,   -2,  -1, -1, -1, -1, -2,  5,   10, -2, -1, -1, -1, -1, -2, 10,
    -20, -50, -2, -2, -2, -2, -50, -20, 100, -20, 10, 5, 5, 10, -20, 100};

static int ab_value(const int8_t *s, int player, int depth, int alpha, int beta, int prune, long *nodes)
{
    uint8_t m[NACT], m2[NACT];
    (*nodes)++;
    int n = orc_valid_moves(s, player, m);
    int n2 = orc_valid_moves(s, -player, m2);
    if (n == 0 && n2 == 0) return AB_WIN * orc_score(s, player);
    if (depth == 0) {
        int h = 10 * (n - n2);
        for (int i = 0; i < NSQ; i++) h += AB_W[i] * ((s[i] == player) - (s[i] == -player));
        return h;
    }
    int best = -AB_INF;
    int8_t ns[NSQ];
    for (int a = 0; a < NACT; a++) {
        if (!m[a]) continue;
        orc_next_state(s, a, player, ns);
        int v = -ab_value(ns, -player, depth - 1, -beta, -alpha, prune, nodes);
        if (prune) {
            if (v >= beta) return beta;
            if (v > alpha) alpha = v;
        } else if (v > best) {
            best = v;
        }
    }
    return prune ? alpha : best;
}

static int ab_root(const int8_t *s, int player, int depth, int exact_empties, int prune, int32_t *values, long *nodes)
{
    uint8_t m[NACT];
    int8_t ns[NSQ];
    int empties = 0, best = -1;
    for (int i = 0; i < NSQ; i++) empties += s[i] == 0;
    for (int a = 0; a < NACT; a++) values[a] = AB_NONE;
    int n = orc_valid_moves(s, player, m);
    uint8_t m2[NACT];
    if (n == 0 && orc_valid_moves(s, -player, m2) == 0) return -1;
    int d = empties <= exact_empties ? AB_UNLIMITED : depth;
    for (int a = 0; a < NACT; a++) {
        if (!m[a]) continue;
        orc_next_state(s, a, player, ns);
        values[a] = -ab_value(ns, -player, d - 1, -AB_INF, AB_INF, prune, nodes);
        if (best < 0 || values[a] > values[best]) best = a;
    }
    return best;
}

/* Per-root-action values [65] (AB_NONE where not legal); returns the lowest best action, -1 at a terminal root.
 * *nodes (may be NULL) = positions visited below the root. */
int orc_negamax(const int8_t *s, int player, int depth, int exact_empties, int32_t *values, long *nodes)
{
    long c = 0;
    int b = ab_root(s, player, depth, exact_empties, 0, values, &c);
    if (nodes) *nodes = c;
    return b;
}

int orc_alphabeta(const int8_t *s, int player, int depth, int exact_empties, int32_t *values, long *nodes)
{
    long c = 0;
    int b = ab_root(s, player, depth, exact_empties, 1, values, &c);
    if (nodes) *nodes = c;
    return b;
}
