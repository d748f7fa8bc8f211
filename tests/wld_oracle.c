/*
 * tests/wld_oracle.c -- TEST INFRASTRUCTURE ONLY: the CPU reference of oth_solve_wld.
 *
 * The alpha-beta of tests/alphabeta_oracle.c (included unchanged) run to the end of the game with the window (-1, 1),
 * in ascending action order on the CPU oracle's mailbox boards (deliberately not the kernel's ordering).
 * tests/wld_oracle.py compiles it into a temporary directory with the oracle's flags.
 */
#include "alphabeta_oracle.c"

/* +1 / 0 / -1: the result of (s, player to move) under perfect play.  The sign is taken because ab_value returns a
 * terminal position's score (10 000 x disc difference) without clamping it to the window.  *nodes (may be NULL) =
 * positions visited, the root included. */
int orc_wld(const int8_t *s, int player, long *nodes)
{
    long c = 0;
    int v = ab_value(s, player, AB_UNLIMITED, -1, 1, 1, &c);
    if (nodes) *nodes = c;
    return (v > 0) - (v < 0);
}
