// env_run_actions_twin.cpp -- TEST INFRASTRUCTURE: the traced bit-sliced env run (cgl_env_run_ex) restated on the
// host with the product's bit logic (ecen743-project-cgol_b200/csrc/cgl_bits.cuh, the very expressions the sm_100a
// kernel runs).  tests/test_env_run_actions_cpu.py compiles it with g++ into a temporary directory and checks it
// against the oracle; it is not shipped.
#include <stdint.h>
#include <string.h>
#include <vector>

#include "../../ecen743-project-cgol_b200/csrc/cgl_bits.cuh"

using namespace cgl;

extern "C" {

// mirrors env_run_sliced_kernel<S, RULE, TR = true> (csrc/cgl_env_run.cu) for ONE env, side % 32 == 0, any dead rule:
// before step t the action actions[t] (side*side: no-op, other out-of-range values: ignored, counted in the return's
// bits 16+) flips the bit and writes the cell's planes; after the step reward_trace[t] is the per-32-cell plane reward
// (sliced_reward32, the base rule's wrap term only when the kernel takes it) summed over the env and alive_trace[t]
// the live count.  actions / traces may be NULL.  Returns the steps executed | (ignored actions << 16).
int twin_env_run_sliced_actions(uint32_t *world, int8_t *stable, uint32_t side, uint32_t max_steps, int stop_when_fixed,
                                int spawn, int stable_max, int rule, int empty, int empty_min, int masked,
                                const int32_t *actions, int32_t *reward_trace, uint32_t *alive_trace)
{
    if (side % 32) return -1;
    const int S = (int)side, W = S / 32, SIZE = S * S;
    const bool sat = rule == CGL_DEAD_SAT, decay = rule == CGL_DEAD_DECAY;
    std::vector<uint32_t> cw(world, world + S * W), pl((size_t)S * W * 8), h0(S * W), h1(S * W);
    const uint32_t *sb = reinterpret_cast<const uint32_t *>(stable);
    const int max_rel = (stable_max - spawn) & 0xff, min_rel = (empty_min - spawn) & 0xff;
    uint32_t odd = 0;
    for (int r = 0; r < S; ++r)
        for (int w = 0; w < W; ++w) {
            uint32_t by[8], p[8];
            memcpy(by, sb + ((size_t)r * S + w * 32) / 4, 32);
            bytes_to_planes32(by, p);
            if (!sat) add_const_sliced(p, -spawn);
            if (!sat && !decay) odd |= gt_const_sliced(p, max_rel) & cw[r * W + w];
            memcpy(&pl[((size_t)r * W + w) * 8], p, 32);
        }
    const bool wraps = decay || max_rel > 127 - spawn || odd != 0;
    uint32_t steps = 0, changed = 1, bad = 0;
    while (steps < max_steps) {
        const int a = actions ? actions[steps] : SIZE;
        if (a >= 0 && a < SIZE) {
            const uint32_t bit = 1u << (a & 31);
            uint32_t &c = cw[a >> 5];
            c ^= bit;
            const int v = (masked && !(c & bit)) ? 0 : spawn;
            uint32_t p[8];
            memcpy(p, &pl[(size_t)(a >> 5) * 8], 32);
            set_cells_sliced(p, bit, sat ? v : v - spawn);
            memcpy(&pl[(size_t)(a >> 5) * 8], p, 32);
        } else if (a != SIZE) {
            ++bad;
        }
        std::vector<HSum> hs(S * W);
        for (int r = 0; r < S; ++r)
            for (int w = 0; w < W; ++w) {
                const uint32_t c = cw[r * W + w];
                hs[r * W + w] = hsum(west_plane(cw[r * W + (w + W - 1) % W], c), c, east_plane(c, cw[r * W + (w + 1) % W]));
                h0[r * W + w] = hs[r * W + w].s0;
                h1[r * W + w] = hs[r * W + w].s1;
            }
        if (stop_when_fixed && !changed) break;
        changed = 0;
        int racc = 0;
        uint32_t pacc = 0;
        std::vector<uint32_t> nw(S * W);
        for (int r = 0; r < S; ++r)
            for (int w = 0; w < W; ++w) {
                const int ru = (r == 0 ? S - 1 : r - 1), rd = (r == S - 1 ? 0 : r + 1);
                const HSum up = {h0[ru * W + w], h1[ru * W + w], 0, 0}, dn = {h0[rd * W + w], h1[rd * W + w], 0, 0};
                const uint32_t c = cw[r * W + w];
                const uint32_t n = life_rule(up, hs[r * W + w], dn, c);
                changed |= n ^ c;
                uint32_t p[8];
                memcpy(p, &pl[((size_t)r * W + w) * 8], 32);
                if (sat) stable_update_sliced_sat(p, n & c, n & ~c, spawn, stable_max, empty, empty_min);
                else if (decay) stable_update_sliced_decay(p, n & c, n & ~c, max_rel, min_rel);
                else stable_update_sliced_rel(p, n & c, max_rel);
                racc += sliced_reward32(rule, p, n, spawn, wraps);
                pacc += popc32(n);
                memcpy(&pl[((size_t)r * W + w) * 8], p, 32);
                nw[r * W + w] = n;
            }
        if (reward_trace) reward_trace[steps] = racc;
        if (alive_trace) alive_trace[steps] = pacc;
        cw = nw;
        ++steps;
    }
    uint32_t *so = reinterpret_cast<uint32_t *>(stable);
    for (int r = 0; r < S; ++r)
        for (int w = 0; w < W; ++w) {
            uint32_t p[8], by[8];
            memcpy(p, &pl[((size_t)r * W + w) * 8], 32);
            if (!sat) add_const_sliced(p, spawn);
            if (!sat && !decay)
                for (int b = 0; b < 8; ++b) p[b] &= cw[r * W + w];
            planes_to_bytes32(p, by);
            memcpy(so + ((size_t)r * S + w * 32) / 4, by, 32);
            world[r * W + w] = cw[r * W + w];
        }
    return (int)(steps | (bad << 16));
}

}  // extern "C"
