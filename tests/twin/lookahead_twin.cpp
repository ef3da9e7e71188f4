// Host twin of the one-step lookahead's per-cell terms (test infrastructure): lookahead1_rule from cgl_bits.cuh, the
// very expression env_lookahead_fused_kernel and env_lookahead_generic_kernel run, against its definition through the
// scalar stability rule stable_update1_rule.  tests/test_action_rewards_cpu.py compiles it into a temporary directory.
#include <stdint.h>

#include "../../ecen743-project-cgol_b200/csrc/cgl_bits.cuh"

using namespace cgl;

static bool next_of(bool alive, int n) { return n == 3 || (n == 2 && alive); }

// Mismatches over every (state, count 0..8, stability) for one rule and set of constants.
extern "C" uint64_t twin_lookahead_mismatches(int rule, int spawn, int stable_max, int empty, int empty_min, int masked)
{
    const int8_t sp = (int8_t)spawn, mx = (int8_t)stable_max, em = (int8_t)empty, mn = (int8_t)empty_min;
    uint64_t bad = 0;
    for (int alive = 0; alive < 2; ++alive)
        for (int n = 0; n <= 8; ++n)
            for (int s = -128; s <= 127; ++s) {
                const Look1 L = lookahead1_rule(rule, (int8_t)s, alive, n, sp, mx, em, mn, masked != 0);
                const int plain = stable_update1_rule(rule, (int8_t)s, alive, next_of(alive, n), sp, mx, em, mn);
                const int up = stable_update1_rule(rule, (int8_t)s, alive, next_of(alive, n + 1), sp, mx, em, mn);
                const int down = stable_update1_rule(rule, (int8_t)s, alive, next_of(alive, n - 1), sp, mx, em, mn);
                const int8_t put = (masked && alive) ? (int8_t)0 : sp;          // the toggled cell is dead if it was alive
                const int self = stable_update1_rule(rule, put, !alive, next_of(!alive, n), sp, mx, em, mn);
                bad += L.plain != plain;
                bad += L.gp != up - plain;
                bad += L.gm != down - plain;
                bad += L.h != self - plain;
            }
    return bad;
}
