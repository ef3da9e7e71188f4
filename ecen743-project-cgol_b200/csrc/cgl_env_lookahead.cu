// cgl_env_lookahead.cu -- one-step lookahead: the reward every action would give, and the greedy action per env.
//
// For env e and action a in 0 .. side*side, rewards[e][a] is the reward cgl_env_step_rule returns with actions[e] = a
// (toggle_state(a), step(), reward(): CGL/main.py:66-71); a = side*side is the no-op.  Computed without stepping:
// a toggle at cell c only changes c itself and the neighbour count of its 8 neighbours, so
//   R(c) = R_noop + h(c) + sum_{x in N8(c)} (c alive ? gm(x) : gp(x))        (mod 2^32)
// with the per-cell terms of lookahead1_rule (cgl_bits.cuh).  That needs a torus of side >= 3 (otherwise a cell can be
// its own neighbour, or the same neighbour several times): sides 1 and 2 are computed by definition.
//
//   fused sides (multiples of 32 up to 256)  env_lookahead_fused_kernel: one CTA per env (four per CTA at side <= 64),
//       world bits and the stability plane in shared memory (the plane is read from HBM once).  Lane l of a warp owns
//       the cells at columns 32k + l of a row, so its count comes from bit-sliced adders on whole words (warp-uniform)
//       and the map stores are coalesced.  Each warp walks a band of rows with a rolling window of horizontal sums
//       (two int16 halves of one int32: gp and gm), horizontal neighbours by shuffles.  The argmax is reduced per warp
//       and then per env; the map is written only in map mode.
//   every other side  three small kernels: the plain reward per env, then one thread per (env, action) evaluating the
//       9-cell formula straight from the packed world and the plane (by definition on sides 1 and 2), then the argmax.
#include <utility>

#include "cgl_internal.cuh"

namespace cgl {

template <int S>
struct LookCfg {
    static constexpr int W = S / 32;                       // words per row == cells per lane and row
    static constexpr int SIZE = S * S;
    static constexpr int BR = S <= 64 ? S : 32;             // rows per warp band
    static constexpr int WPE_WARPS = S / BR;                // warps per env
    static constexpr int TPE = 32 * WPE_WARPS;              // threads per env
    static constexpr int EPC = S <= 64 ? 4 : 1;             // envs per CTA
    static constexpr int THREADS = TPE * EPC;
    static constexpr int SLOT = SIZE + S * W * 4;           // shared bytes per env: plane, then world words
    static constexpr int SMEM = EPC * SLOT;
    static_assert(S % 32 == 0 && S >= 32 && S <= 256 && SIZE % 16 == 0, "unsupported side");
};

struct LookArgs {
    const uint32_t *world;
    const int8_t *stable;
    int32_t *rewards, *best_action, *best_reward;
    uint32_t n_envs;
    int8_t spawn, stable_max, empty, empty_min;
    int masked;
};

// The cells of row r at columns 32k + lane: count planes from the row's words (warp-uniform), then the per-cell terms.
// pk[k] = (gp + 256) | (gm + 256) << 16 (both halves stay positive through the 3 x 3 sums).
template <int S, int RULE>
__device__ __forceinline__ void lookahead_row(const uint32_t *wsm, const int8_t *ssm, int r, int lane, const LookArgs &a,
                                              uint32_t (&pk)[LookCfg<S>::W], int (&h)[LookCfg<S>::W],
                                              uint32_t &alive_bits, int &plain_sum)
{
    constexpr int W = LookCfg<S>::W;
    const int ru = r == 0 ? S - 1 : r - 1, rd = r == S - 1 ? 0 : r + 1;
    alive_bits = 0;
#pragma unroll
    for (int k = 0; k < W; ++k) {
        const int kw = (k + W - 1) % W, ke = (k + 1) % W;
        const uint32_t u = wsm[ru * W + k], c = wsm[r * W + k], d = wsm[rd * W + k];
        const HSum up = hsum(west_plane(wsm[ru * W + kw], u), u, east_plane(u, wsm[ru * W + ke]));
        const HSum mid = hsum(west_plane(wsm[r * W + kw], c), c, east_plane(c, wsm[r * W + ke]));
        const HSum dn = hsum(west_plane(wsm[rd * W + kw], d), d, east_plane(d, wsm[rd * W + ke]));
        // n = up.s + mid.t + dn.s as 4 bit planes: x0 + 2 * (up.s1 + dn.s1 + mid.t1 + carry0)
        const uint32_t x0 = up.s0 ^ dn.s0 ^ mid.t0, c0 = maj3(up.s0, dn.s0, mid.t0);
        const uint32_t p = up.s1 ^ dn.s1, q = mid.t1 ^ c0;
        const uint32_t x1 = p ^ q, ca = up.s1 & dn.s1, cb = mid.t1 & c0, cy = p & q;
        const uint32_t x2 = ca ^ cb ^ cy, x3 = ca & cb;
        const int n = (int)((x0 >> lane) & 1u) | (int)(((x1 >> lane) & 1u) << 1) | (int)(((x2 >> lane) & 1u) << 2) |
                      (int)(((x3 >> lane) & 1u) << 3);
        const bool alive = (c >> lane) & 1u;
        alive_bits |= (uint32_t)alive << k;
        const Look1 L = lookahead1_rule(RULE, ssm[r * S + 32 * k + lane], alive, n, a.spawn, a.stable_max, a.empty,
                                        a.empty_min, a.masked != 0);
        pk[k] = (uint32_t)(L.gp + 256) | ((uint32_t)(L.gm + 256) << 16);
        h[k] = L.h;
        plain_sum += L.plain;
    }
}

// Horizontal 3-sums of pk along the torus row: column 32k + lane - 1 is lane - 1's cell k, or lane 31's cell k - 1.
template <int W>
__device__ __forceinline__ void hsum_row(const uint32_t (&pk)[W], int lane, uint32_t (&hs)[W])
{
    uint32_t lf[W], rt[W];
#pragma unroll
    for (int k = 0; k < W; ++k) {
        lf[k] = __shfl_sync(0xffffffffu, pk[k], (lane + 31) & 31);
        rt[k] = __shfl_sync(0xffffffffu, pk[k], (lane + 1) & 31);
    }
#pragma unroll
    for (int k = 0; k < W; ++k) {
        const uint32_t l = lane == 0 ? lf[(k + W - 1) % W] : lf[k];
        const uint32_t r = lane == 31 ? rt[(k + 1) % W] : rt[k];
        hs[k] = l + pk[k] + r;
    }
}

// MAP: write rewards[e][0 .. size]; BEST: write best_action / best_reward.  RULE: the dead-cell rule (compile-time,
// as in the fused step).
template <int S, int RULE, bool MAP, bool BEST>
__global__ void __launch_bounds__(LookCfg<S>::THREADS)
env_lookahead_fused_kernel(LookArgs a)
{
    using C = LookCfg<S>;
    constexpr int W = C::W;
    extern __shared__ __align__(16) unsigned char smem_dyn[];
    __shared__ int red_sum[C::EPC];
    __shared__ unsigned long long red_best[C::EPC];
    const int g = threadIdx.x / C::TPE, t = threadIdx.x % C::TPE;
    const int lane = threadIdx.x & 31, band = t >> 5;
    const uint32_t e = blockIdx.x * C::EPC + g;
    const bool active = e < a.n_envs;
    int8_t *ssm = reinterpret_cast<int8_t *>(smem_dyn + g * C::SLOT);
    uint32_t *wsm = reinterpret_cast<uint32_t *>(smem_dyn + g * C::SLOT + C::SIZE);

    if (t == 0) { red_sum[g] = 0; red_best[g] = 0ull; }
    if (active) {
        const int8_t *sp = a.stable + (size_t)e * C::SIZE;
        if ((reinterpret_cast<uintptr_t>(sp) & 15u) == 0) {
            const uint4 *s4 = reinterpret_cast<const uint4 *>(sp);
            for (int i = t; i < C::SIZE / 16; i += C::TPE) reinterpret_cast<uint4 *>(ssm)[i] = __ldg(s4 + i);
        } else {
            for (int i = t; i < C::SIZE; i += C::TPE) ssm[i] = sp[i];
        }
        const uint32_t *wp = a.world + (size_t)e * (S * W);
        for (int i = t; i < S * W; i += C::TPE) wsm[i] = __ldg(wp + i);
    }
    __syncthreads();

    const int y0 = band * C::BR;
    int plain_sum = 0;
    // Map mode needs R_noop before the first store: one cheaper pass over the band (next state from whole words).
    if (MAP && active) {
#pragma unroll 1
        for (int y = y0; y < y0 + C::BR; ++y) {
            const int ru = y == 0 ? S - 1 : y - 1, rd = y == S - 1 ? 0 : y + 1;
#pragma unroll
            for (int k = 0; k < W; ++k) {
                const int kw = (k + W - 1) % W, ke = (k + 1) % W;
                const uint32_t u = wsm[ru * W + k], c = wsm[y * W + k], d = wsm[rd * W + k];
                const uint32_t nxt = life_rule(hsum(west_plane(wsm[ru * W + kw], u), u, east_plane(u, wsm[ru * W + ke])),
                                               hsum(west_plane(wsm[y * W + kw], c), c, east_plane(c, wsm[y * W + ke])),
                                               hsum(west_plane(wsm[rd * W + kw], d), d, east_plane(d, wsm[rd * W + ke])), c);
                plain_sum += stable_update1_rule(RULE, ssm[y * S + 32 * k + lane], (c >> lane) & 1u, (nxt >> lane) & 1u,
                                                 a.spawn, a.stable_max, a.empty, a.empty_min);
            }
        }
        plain_sum = __reduce_add_sync(0xffffffffu, plain_sum);
        if (lane == 0) atomicAdd(&red_sum[g], plain_sum);
    }
    if (MAP) __syncthreads();
    const int r_noop = MAP ? red_sum[g] : 0;

    int best_v = 0x80000000, best_i = 0;          // over the deltas R(a) - R_noop (no int32 wrap at these sides)
    if (active) {
        int32_t *out = MAP ? a.rewards + (size_t)e * (C::SIZE + 1) : nullptr;
        uint32_t pk[W], hsA[W], hsB[W], hsC[W];
        int hB[W], hC[W], dummy = 0;
        uint32_t wB, wC;
        lookahead_row<S, RULE>(wsm, ssm, (y0 + S - 1) % S, lane, a, pk, hC, wC, dummy);
        hsum_row<W>(pk, lane, hsA);
        int psum = 0;
        uint32_t pkB[W];
        lookahead_row<S, RULE>(wsm, ssm, y0, lane, a, pkB, hB, wB, psum);
        hsum_row<W>(pkB, lane, hsB);
#pragma unroll 1
        for (int y = y0; y < y0 + C::BR; ++y) {
            int pnext = 0;
            lookahead_row<S, RULE>(wsm, ssm, y + 1 == S ? 0 : y + 1, lane, a, pk, hC, wC, pnext);
            hsum_row<W>(pk, lane, hsC);
#pragma unroll
            for (int k = 0; k < W; ++k) {
                const uint32_t box = hsA[k] + hsB[k] + hsC[k] - pkB[k];          // 8 neighbours, each biased by 256
                const int bp = (int)(box & 0xffffu) - 2048, bm = (int)(box >> 16) - 2048;
                const int delta = hB[k] + (((wB >> k) & 1u) ? bm : bp);
                const int idx = y * S + 32 * k + lane;
                if (MAP) out[idx] = (int32_t)((uint32_t)r_noop + (uint32_t)delta);
                if (BEST && delta > best_v) { best_v = delta; best_i = idx; }     // indices ascend: first maximum kept
            }
            plain_sum += psum;
            psum = pnext;
#pragma unroll
            for (int k = 0; k < W; ++k) { hsA[k] = hsB[k]; hsB[k] = hsC[k]; pkB[k] = pk[k]; hB[k] = hC[k]; }
            wB = wC;
        }
        (void)dummy;
        if (MAP && t == 0) out[C::SIZE] = r_noop;
    }
    if (BEST) {
        // key: larger delta first, then the smaller index
        unsigned long long key = active ? ((unsigned long long)((uint32_t)best_v ^ 0x80000000u) << 32) |
                                              (0xffffffffu - (uint32_t)best_i)
                                        : 0ull;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const unsigned long long k2 = __shfl_xor_sync(0xffffffffu, key, o);
            key = k2 > key ? k2 : key;
        }
        if (!MAP) plain_sum = __reduce_add_sync(0xffffffffu, plain_sum);
        if (lane == 0 && active) {
            atomicMax(&red_best[g], key);
            if (!MAP) atomicAdd(&red_sum[g], plain_sum);
        }
        __syncthreads();
        if (active && t == 0) {
            // the no-op: delta 0 at index size, the largest index, so it wins only if every toggle loses reward
            unsigned long long k = red_best[g];
            const unsigned long long noop = (0x80000000ull << 32) | (0xffffffffu - (uint32_t)C::SIZE);
            k = noop > k ? noop : k;
            const int delta = (int)((uint32_t)(k >> 32) ^ 0x80000000u);
            if (a.best_action) a.best_action[e] = (int32_t)(0xffffffffu - (uint32_t)k);
            if (a.best_reward) a.best_reward[e] = (int32_t)((uint32_t)red_sum[g] + (uint32_t)delta);
        }
    }
}

// ---- every other side -------------------------------------------------------------------------------------------
__device__ __forceinline__ bool cell_at(const uint32_t *w, uint32_t side, uint32_t W, uint64_t cell)
{
    const uint32_t r = (uint32_t)(cell / side), c = (uint32_t)(cell - (uint64_t)r * side);
    return (w[(uint64_t)r * W + (c >> 5)] >> (c & 31)) & 1u;
}

// The neighbour count exactly as the reference forms it (CGL/CGL.py:214-225): on sides 1 and 2 a cell can be its own
// neighbour or count one neighbour twice.
__device__ __forceinline__ int count_ref(const uint32_t *w, uint32_t side, uint32_t W, uint64_t size, uint64_t cell,
                                        uint32_t flip_bits, bool small)
{
    const uint64_t x = cell % side, y = cell - x;
    const uint64_t l = (x + side - 1) % side, rr = (x + 1) % side, up = (y + size - side) % size, dn = (y + side) % size;
    const uint64_t nb[8] = {l + up, x + up, rr + up, l + y, rr + y, l + dn, x + dn, rr + dn};
    int n = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) n += (int)cell_at(w, side, W, nb[i]) ^ (small ? (int)((flip_bits >> nb[i]) & 1u) : 0);
    return n;
}

struct LookGenArgs {
    const uint32_t *world;
    const int8_t *stable;
    int32_t *rewards;
    int32_t *r_noop;
    unsigned long long *best_key;
    uint64_t n_envs;
    uint32_t side, W;
    int rule;
    int8_t spawn, stable_max, empty, empty_min;
    int masked;
};

// r_noop[e] = the plain step's reward (zeroed before).  One thread per cell.
__global__ void env_lookahead_noop_kernel(LookGenArgs a)
{
    const uint64_t size = (uint64_t)a.side * a.side, total = a.n_envs * size;
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < total; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t e = i / size, cell = i - e * size;
        const uint32_t *w = a.world + e * a.side * a.W;
        const bool alive = cell_at(w, a.side, a.W, cell);
        const int n = count_ref(w, a.side, a.W, size, cell, 0u, false);
        const int v = stable_update1_rule(a.rule, a.stable[i], alive, n == 3 || (n == 2 && alive), a.spawn, a.stable_max,
                                          a.empty, a.empty_min);
        const unsigned peers = __match_any_sync(__activemask(), e);
        const int sum = __reduce_add_sync(peers, v);
        if ((threadIdx.x & 31) == (unsigned)(__ffs(peers) - 1)) atomicAdd(a.r_noop + e, sum);
    }
}

// One thread per (env, action).
__global__ void env_lookahead_generic_kernel(LookGenArgs a)
{
    const uint64_t size = (uint64_t)a.side * a.side, total = a.n_envs * (size + 1);
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < total; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t e = i / (size + 1), act = i - e * (size + 1);
        const uint32_t *w = a.world + e * a.side * a.W;
        const int8_t *s = a.stable + e * size;
        uint32_t v = (uint32_t)a.r_noop[e];
        if (act < size && a.side <= 2) {
            // by definition: toggle, step, reward over at most 4 cells
            const bool now = cell_at(w, a.side, a.W, act);
            const int8_t put = (a.masked && now) ? (int8_t)0 : a.spawn;
            v = 0;
            for (uint64_t c = 0; c < size; ++c) {
                const bool alive = cell_at(w, a.side, a.W, c) ^ (c == act);
                const int n = count_ref(w, a.side, a.W, size, c, 1u << act, true);
                v += (uint32_t)(int)stable_update1_rule(a.rule, c == act ? put : s[c], alive, n == 3 || (n == 2 && alive),
                                                        a.spawn, a.stable_max, a.empty, a.empty_min);
            }
        } else if (act < size) {
            const uint32_t side = a.side;
            const uint32_t r = (uint32_t)(act / side), c = (uint32_t)(act - (uint64_t)r * side);
            const bool alive_c = cell_at(w, side, a.W, act);
            int delta = 0;
            for (int dy = -1; dy <= 1; ++dy)
                for (int dx = -1; dx <= 1; ++dx) {
                    const uint32_t yy = (r + side + dy) % side, xx = (c + side + dx) % side;
                    const uint64_t x = (uint64_t)yy * side + xx;
                    const bool alive = cell_at(w, side, a.W, x);
                    const int n = count_ref(w, side, a.W, size, x, 0u, false);
                    const Look1 L = lookahead1_rule(a.rule, s[x], alive, n, a.spawn, a.stable_max, a.empty, a.empty_min,
                                                    a.masked != 0);
                    delta += (dy == 0 && dx == 0) ? L.h : (alive_c ? L.gm : L.gp);
                }
            v += (uint32_t)delta;
        }
        if (a.rewards != nullptr) a.rewards[i] = (int32_t)v;
        if (a.best_key != nullptr) {
            const unsigned long long key = ((unsigned long long)(v ^ 0x80000000u) << 32) | (0xffffffffu - (uint32_t)act);
            atomicMax(a.best_key + e, key);
        }
    }
}

__global__ void env_lookahead_best_kernel(const unsigned long long *key, uint64_t n_envs, int32_t *best_action,
                                          int32_t *best_reward)
{
    for (uint64_t e = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; e < n_envs; e += (uint64_t)gridDim.x * blockDim.x) {
        const unsigned long long k = key[e];
        if (best_action) best_action[e] = (int32_t)(0xffffffffu - (uint32_t)k);
        if (best_reward) best_reward[e] = (int32_t)((uint32_t)(k >> 32) ^ 0x80000000u);
    }
}

template <int S, int RULE>
static int launch_lookahead_rule(const LookArgs &la, bool map, bool best, cudaStream_t st)
{
    using C = LookCfg<S>;
    static PerDeviceOnce once;
    if (once.first()) {
        CGL_CUDA(cudaFuncSetAttribute(env_lookahead_fused_kernel<S, RULE, true, false>,
                                      cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM));
        CGL_CUDA(cudaFuncSetAttribute(env_lookahead_fused_kernel<S, RULE, false, true>,
                                      cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM));
        CGL_CUDA(cudaFuncSetAttribute(env_lookahead_fused_kernel<S, RULE, true, true>,
                                      cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM));
    }
    const unsigned grid = (unsigned)((la.n_envs + C::EPC - 1) / C::EPC);
    if (map && best) env_lookahead_fused_kernel<S, RULE, true, true><<<grid, C::THREADS, C::SMEM, st>>>(la);
    else if (map) env_lookahead_fused_kernel<S, RULE, true, false><<<grid, C::THREADS, C::SMEM, st>>>(la);
    else env_lookahead_fused_kernel<S, RULE, false, true><<<grid, C::THREADS, C::SMEM, st>>>(la);
    CGL_LAUNCH_CHECK();
    return 0;
}

template <int S>
static int launch_lookahead_fused(const LookArgs &la, int rule, bool map, bool best, cudaStream_t st)
{
    if (rule == CGL_DEAD_DECAY) return launch_lookahead_rule<S, CGL_DEAD_DECAY>(la, map, best, st);
    if (rule == CGL_DEAD_SAT) return launch_lookahead_rule<S, CGL_DEAD_SAT>(la, map, best, st);
    return launch_lookahead_rule<S, CGL_DEAD_ZERO>(la, map, best, st);
}

}  // namespace cgl

using namespace cgl;

// Do the byte ranges [p, p + np) and [q, q + nq) share a byte?
static bool ranges_overlap(const void *p, unsigned __int128 np, const void *q, unsigned __int128 nq)
{
    if (p == nullptr || q == nullptr || np == 0 || nq == 0) return false;
    const unsigned __int128 a = (uintptr_t)p, b = (uintptr_t)q;
    return a < b + nq && b < a + np;
}

extern "C" int cgl_env_action_rewards(const cgl_env_action_rewards_args_t *args, cgl_stream_t stream)
{
    CGL_REQUIRE(args, CGL_E_BADARG, "cgl_env_action_rewards: null");
    const cgl_env_action_rewards_args_t a = *args;
    CGL_REQUIRE(a.world_dev && a.stable_dev && a.side, CGL_E_BADARG, "cgl_env_action_rewards: bad argument");
    CGL_REQUIRE(a.rewards_out_dev || a.best_action_out_dev || a.best_reward_out_dev, CGL_E_BADARG,
                "cgl_env_action_rewards: no output requested");
    CGL_REQUIRE(a.n_envs > 0 && a.n_envs < (1ull << 31), CGL_E_BADARG, "cgl_env_action_rewards: n_envs must be 1 .. 2^31-1");
    CGL_REQUIRE(a.side <= 46340, CGL_E_BADARG, "cgl_env_action_rewards: side*side + 1 actions must fit int32 (side <= 46340)");
    CGL_REQUIRE(a.dead_rule >= CGL_DEAD_ZERO && a.dead_rule <= CGL_DEAD_SAT, CGL_E_BADARG,
                "cgl_env_action_rewards: dead_rule must be 0 (zero), 1 (decay) or 2 (saturate)");
    CGL_REQUIRE(a.empty >= -128 && a.empty <= 127 && a.empty_min >= -128 && a.empty_min <= 127, CGL_E_BADARG,
                "cgl_env_action_rewards: empty / empty_min must fit int8");
    CGL_REQUIRE(a.masked_toggle == 0 || a.masked_toggle == 1, CGL_E_BADARG,
                "cgl_env_action_rewards: masked_toggle must be 0 or 1");
    const uint64_t size = (uint64_t)a.side * a.side, W = cgl_words_per_row(a.side);
    const unsigned __int128 n = a.n_envs;
    const std::pair<const void *, unsigned __int128> in[2] = {{a.world_dev, n * a.side * W * 4}, {a.stable_dev, n * size}};
    const std::pair<const void *, unsigned __int128> out[3] = {
        {a.rewards_out_dev, n * (size + 1) * 4}, {a.best_action_out_dev, n * 4}, {a.best_reward_out_dev, n * 4}};
    for (int i = 0; i < 3; ++i) {
        for (const auto &p : in)
            CGL_REQUIRE(!ranges_overlap(out[i].first, out[i].second, p.first, p.second), CGL_E_BADARG,
                        "cgl_env_action_rewards: an output overlaps the world or the stability plane");
        for (int k = i + 1; k < 3; ++k)
            CGL_REQUIRE(!ranges_overlap(out[i].first, out[i].second, out[k].first, out[k].second), CGL_E_BADARG,
                        "cgl_env_action_rewards: two outputs overlap");
    }

    cudaStream_t st = as_stream(stream);
    const bool map = a.rewards_out_dev != nullptr, best = a.best_action_out_dev || a.best_reward_out_dev;
    if (cgl_env_step_is_fused(a.side)) {
        LookArgs la;
        la.world = a.world_dev; la.stable = a.stable_dev;
        la.rewards = a.rewards_out_dev; la.best_action = a.best_action_out_dev; la.best_reward = a.best_reward_out_dev;
        la.n_envs = (uint32_t)a.n_envs;
        la.spawn = (int8_t)a.spawn; la.stable_max = (int8_t)a.stable_max;
        la.empty = (int8_t)a.empty; la.empty_min = (int8_t)a.empty_min; la.masked = a.masked_toggle;
        switch (a.side) {
        case 32: return launch_lookahead_fused<32>(la, a.dead_rule, map, best, st);
        case 64: return launch_lookahead_fused<64>(la, a.dead_rule, map, best, st);
        case 96: return launch_lookahead_fused<96>(la, a.dead_rule, map, best, st);
        case 128: return launch_lookahead_fused<128>(la, a.dead_rule, map, best, st);
        case 160: return launch_lookahead_fused<160>(la, a.dead_rule, map, best, st);
        case 192: return launch_lookahead_fused<192>(la, a.dead_rule, map, best, st);
        case 224: return launch_lookahead_fused<224>(la, a.dead_rule, map, best, st);
        case 256: return launch_lookahead_fused<256>(la, a.dead_rule, map, best, st);
        }
    }
    // other sides: plain reward, then every action, then the argmax (stream-ordered scratch)
    LookGenArgs g;
    g.world = a.world_dev; g.stable = a.stable_dev; g.rewards = a.rewards_out_dev;
    g.n_envs = a.n_envs; g.side = a.side; g.W = (uint32_t)W; g.rule = a.dead_rule;
    g.spawn = (int8_t)a.spawn; g.stable_max = (int8_t)a.stable_max; g.empty = (int8_t)a.empty;
    g.empty_min = (int8_t)a.empty_min; g.masked = a.masked_toggle;
    void *scratch = nullptr;
    const size_t bytes = (size_t)a.n_envs * (sizeof(unsigned long long) + sizeof(int32_t));
    CGL_CUDA(cudaMallocAsync(&scratch, bytes, st));
    g.best_key = best ? static_cast<unsigned long long *>(scratch) : nullptr;
    g.r_noop = reinterpret_cast<int32_t *>(static_cast<unsigned long long *>(scratch) + a.n_envs);
    int rc = 0;
    cudaError_t err = cudaMemsetAsync(scratch, 0, bytes, st);
    if (err == cudaSuccess) {
        env_lookahead_noop_kernel<<<grid_for(a.n_envs * size, 256), 256, 0, st>>>(g);
        env_lookahead_generic_kernel<<<grid_for(a.n_envs * (size + 1), 256), 256, 0, st>>>(g);
        if (best)
            env_lookahead_best_kernel<<<grid_for(a.n_envs, 256), 256, 0, st>>>(g.best_key, a.n_envs, a.best_action_out_dev,
                                                                                a.best_reward_out_dev);
        err = cudaGetLastError();
    }
    if (err != cudaSuccess) {
        set_error("cgl_env_action_rewards: %s", cudaGetErrorString(err));
        rc = (int)err;
    }
    CGL_CUDA(cudaFreeAsync(scratch, st));
    return rc;
}
