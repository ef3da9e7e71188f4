// cgl_env_run.cu -- many plain env steps per launch with the environment resident in shared memory,
// optional stop at the first generation that leaves the world unchanged, and the value-count
// "breakdown" of the stability plane (SURVEY.md section 8 row f3).
//
// Reference behaviour restated here:
//   * the plain step loop of CGL/bench.py:39-40 (`for _ in range(iters): env.step()`): kernel `run`
//     CGL/CGL.py:147-181 applied max_steps times;
//   * the convergence loop of CGL/CGL_action+/validate.py:133-139 (`old = get_state(); step();
//     while not match(old) and count_down: ...`): step until a step does not change the world or the
//     budget is spent -- on the reference one D2H copy + host compare per step;
//   * breakdown_stable / breakdown_state (CGL/CGL_action+/CGL.py:294-303): np.unique value counts.
//
// One CTA (or one warp for side <= 64) owns an environment for the whole call: world (two bit planes)
// and the int8 stability plane live in shared memory, HBM is touched once on the way in and once on the
// way out, so k steps cost 2.25/k bytes per cell-update instead of 2.25 and the loop is bound by the
// integer pipe.  The per-step logic is the fused env kernel's (cgl_env.cu): bit-sliced rows, (born,
// surv) nibbles through the lane-private mask tables, byte-SIMD stability update.
//
// cgl_env_run_ex adds an action schedule (toggle_state before every step, as in cgl_env_step_rule) and per-step
// reward / live-count traces to all three kernels, through their TR instantiations (DESIGN.md section 8 f3.1).
// cgl_env_run_obs adds the observation (the stability plane) after every step, through the OBS instantiations of the
// byte and generic kernels (DESIGN.md section 8 f3.2).
// cgl_env_run_cycle stops an env when its world repeats one of its last max_period worlds, through the CYC
// instantiations of the bit-sliced and generic kernels (DESIGN.md section 8 f3.3).
// cgl_env_run_settle stops an env at its first repeated world of any period: world-only finder kernels give each env's
// step count, which the SETTLE instantiations of the same two kernels then run (DESIGN.md section 8 f3.4).
#include <stdlib.h>

#include <utility>

#include "cgl_internal.cuh"

namespace cgl {

template <int S>
struct RunCfg {
    static constexpr int W = S / 32;
    static constexpr int WPE = S * W;
    static constexpr int SIZE = S * S;
    static constexpr int NCHUNK = SIZE / 16;
    static constexpr int TPE = (S <= 64) ? 32 : S;
    static constexpr int EPC = (TPE >= 96) ? 1 : (128 / TPE);
    static constexpr int THREADS = TPE * EPC;
    static constexpr int CPT = NCHUNK / TPE;
    static constexpr int RPB = S / TPE;
    // per env: cur | nxt (WPE words each) | mix (2*WPE words) | stability plane (SIZE bytes)
    static constexpr int ENV_BYTES = WPE * 16 + SIZE;
    // [<= 4 KB align slack][mask tables 4 KB][envs][2 ints per env]
    static constexpr int SMEM = 4096 + 4096 + EPC * ENV_BYTES + EPC * 8;
    static_assert(S % 32 == 0 && NCHUNK % TPE == 0 && WPE % 4 == 0, "unsupported side");
};

template <int N>
__device__ __forceinline__ void lds_words(const uint32_t *p, uint32_t (&x)[N])
{
    if constexpr (N % 4 == 0) {
#pragma unroll
        for (int i = 0; i < N / 4; ++i) {
            const uint4 v = reinterpret_cast<const uint4 *>(p)[i];
            x[4 * i] = v.x; x[4 * i + 1] = v.y; x[4 * i + 2] = v.z; x[4 * i + 3] = v.w;
        }
    } else if constexpr (N % 2 == 0) {
#pragma unroll
        for (int i = 0; i < N / 2; ++i) {
            const uint2 v = reinterpret_cast<const uint2 *>(p)[i];
            x[2 * i] = v.x; x[2 * i + 1] = v.y;
        }
    } else {
#pragma unroll
        for (int i = 0; i < N; ++i) x[i] = p[i];
    }
}

template <int N>
__device__ __forceinline__ void sts_words(uint32_t *p, const uint32_t (&x)[N])
{
    if constexpr (N % 4 == 0) {
#pragma unroll
        for (int i = 0; i < N / 4; ++i)
            reinterpret_cast<uint4 *>(p)[i] = make_uint4(x[4 * i], x[4 * i + 1], x[4 * i + 2], x[4 * i + 3]);
    } else if constexpr (N % 2 == 0) {
#pragma unroll
        for (int i = 0; i < N / 2; ++i) reinterpret_cast<uint2 *>(p)[i] = make_uint2(x[2 * i], x[2 * i + 1]);
    } else {
#pragma unroll
        for (int i = 0; i < N; ++i) p[i] = x[i];
    }
}

__device__ __forceinline__ uint32_t lds32(uint32_t shared_addr)
{
    uint32_t v;
    asm("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(shared_addr));
    return v;
}

// Action schedules and per-step traces (cgl_env_run_ex) for every kernel of this file: TR = true adds the trailing
// arguments' work, TR = false compiles to the kernel without them.  Inside, which of actions / reward trace / alive
// trace are present are uniform run-time tests.  An action is applied as in cgl_env_step_rule: `size` is the no-op,
// any other index outside [0, size) is ignored and reported; the toggled cell's stability becomes SPAWN (0 under the
// masked toggle when the cell is dead after it), and the step sees the toggled world.
struct RunTrace {
    const int32_t *actions;         // int32 [max_steps][n_envs] or NULL
    int32_t *reward;                // int32 [max_steps][n_envs] or NULL
    uint32_t *alive;                // uint32 [max_steps][n_envs] or NULL
    int *err_flag;
    int masked;
};

// OBS (implies TR): every updated 16-byte chunk of the stability plane is also stored to row (step, e) of `obs`
// (int8 [max_steps][n_envs][SIZE]), and the plane is not written back: the run is out of place, the last row holds
// the final plane.  `obs` is a kernel argument of its own because growing RunTrace reschedules the sliced kernels.
template <int S, bool TR, bool OBS = false>
__global__ void __launch_bounds__(RunCfg<S>::THREADS)
env_run_kernel(const uint32_t *world_in, uint32_t *world_out, int8_t *stable, uint32_t n_envs,
               uint32_t max_steps, int stop_when_fixed, uint32_t spawn4, uint32_t max4,
               int32_t *__restrict__ steps_out, int32_t *__restrict__ reward_out, uint32_t *__restrict__ alive_out,
               int rule, uint32_t min4, uint32_t empty4, RunTrace tr, int8_t *obs)
{
    using C = RunCfg<S>;
    extern __shared__ __align__(16) unsigned char smem_dyn[];
    const uint32_t sbase = (uint32_t)__cvta_generic_to_shared(smem_dyn);
    const uint32_t tb = (sbase + 4095u) & ~4095u;            // 4 KB-aligned table base: lookup address = one PRMT
    unsigned char *smem_raw = smem_dyn + (tb - sbase);
    uint32_t *tables = reinterpret_cast<uint32_t *>(smem_raw);
    const int g = threadIdx.x / C::TPE;
    const int t = threadIdx.x % C::TPE;
    unsigned char *env_base = smem_raw + 4096 + g * C::ENV_BYTES;
    uint32_t *cur = reinterpret_cast<uint32_t *>(env_base);
    uint32_t *nxt = cur + C::WPE;
    uint32_t *mix = nxt + C::WPE;
    uint4 *sst = reinterpret_cast<uint4 *>(mix + 2 * C::WPE);
    int *red = reinterpret_cast<int *>(smem_raw + 4096 + C::EPC * C::ENV_BYTES) + g * 2;
    // TR, one env per CTA: per-step (reward, alive) sums of the warps, double-buffered by step parity
    int *slot = reinterpret_cast<int *>(smem_raw + 4096 + C::EPC * C::ENV_BYTES) + 2 * C::EPC;

    const uint32_t e = blockIdx.x * C::EPC + g;
    const bool active = e < n_envs;
    if constexpr (TR && C::EPC == 1)
        if (t == 0) { slot[0] = 0; slot[1] = 0; slot[2] = 0; slot[3] = 0; }

    for (int i = threadIdx.x; i < 1024; i += C::THREADS) {
        const uint32_t m = nibble_to_bytemask((uint32_t)i >> 6);
        tables[i] = (i & 32) ? (m & spawn4) : m;
    }
    if (t == 0) { red[0] = 0; red[1] = 0; }
    if (active) {
        const uint4 *wp = reinterpret_cast<const uint4 *>(world_in + (size_t)e * C::WPE);
        for (int i = t; i < C::WPE / 4; i += C::TPE) reinterpret_cast<uint4 *>(cur)[i] = wp[i];
        const uint4 *sp = reinterpret_cast<const uint4 *>(stable + (size_t)e * C::SIZE);
#pragma unroll 4
        for (int j = 0; j < C::CPT; ++j) sst[j * C::TPE + t] = sp[j * C::TPE + t];
    }
    __syncthreads();

    // One env per CTA synchronises with the CTA barrier; several envs per CTA (one warp each) run
    // their own number of steps and synchronise per warp.
    auto env_vote = [&](bool p) -> bool {
        if constexpr (C::EPC == 1) return __syncthreads_or(p) != 0;
        const bool r = __any_sync(0xffffffffu, p);
        __syncwarp();
        return r;
    };
    auto env_sync = [&]() {
        if constexpr (C::EPC == 1) __syncthreads(); else __syncwarp();
    };

    const uint32_t tbn = ((tb >> 8) & 0xffu) * 0x01010101u;
    const uint32_t lane_s = (threadIdx.x & 31) * 4, lane_b = lane_s + 128;
    uint32_t steps = 0;
    bool done = !active || max_steps == 0;
    const bool want_trace = TR && (tr.reward != nullptr || tr.alive != nullptr);
    int next_act = C::SIZE;                          // the no-op
    if constexpr (TR)
        if (!done && tr.actions != nullptr) next_act = tr.actions[e];
    while (!done) {
        int act = -1;                                // TR: the cell toggled before this step, or -1
        int racc = 0;
        uint32_t pacc = 0;
        uint4 *orow = nullptr;
        if constexpr (OBS) orow = reinterpret_cast<uint4 *>(obs + ((size_t)steps * n_envs + e) * C::SIZE);
        if constexpr (TR) {
            const int a = next_act;
            if (tr.actions != nullptr && steps + 1 < max_steps) next_act = tr.actions[(size_t)(steps + 1) * n_envs + e];
            if (a >= 0 && a < C::SIZE) act = a;
            else if (a != C::SIZE && t == 0) {
                if (tr.err_flag != nullptr) atomicOr(tr.err_flag, 1);
                raise_alarm(ALARM_BAD_ACTION);
            }
        }
        // ---- next generation: smem plane `cur` -> smem plane `nxt`, (born, surv) nibbles -> mix ----
        uint32_t changed = 0;
        {
            HSum hs[C::RPB + 2][C::W];
            uint32_t cw[C::RPB + 2][C::W];
#pragma unroll
            for (int j = 0; j < C::RPB + 2; ++j) {
                int r = t * C::RPB + j - 1;
                r = r < 0 ? S - 1 : (r >= S ? 0 : r);
                lds_words<C::W>(cur + r * C::W, cw[j]);
                if constexpr (TR) {
                    // the toggle goes into every loaded copy of its row; `cur` itself stays as it was
#pragma unroll
                    for (int w = 0; w < C::W; ++w)
                        if (act >= 0 && (act >> 5) == r * C::W + w) cw[j][w] ^= 1u << (act & 31);
                }
#pragma unroll
                for (int w = 0; w < C::W; ++w)
                    hs[j][w] = hsum(west_plane(cw[j][(w + C::W - 1) % C::W], cw[j][w]), cw[j][w],
                                    east_plane(cw[j][w], cw[j][(w + 1) % C::W]));
            }
#pragma unroll
            for (int j = 0; j < C::RPB; ++j) {
                const int r = t * C::RPB + j;
                uint32_t nx[C::W], mx[2 * C::W];
#pragma unroll
                for (int w = 0; w < C::W; ++w) {
                    const uint32_t c = cw[j + 1][w];
                    const uint32_t n = life_rule(hs[j][w], hs[j + 1][w], hs[j + 2][w], c);
                    nx[w] = n;
                    changed |= n ^ c;
                    if constexpr (TR) pacc += __popc(n);
                    mix_nibbles(n & ~c, n & c, mx[2 * w], mx[2 * w + 1]);
                }
                sts_words<C::W>(nxt + r * C::W, nx);
                sts_words<2 * C::W>(mix + 2 * r * C::W, mx);
            }
        }
        const bool any_changed = env_vote(changed != 0);
        if constexpr (TR) {
            // stable[act] = SPAWN (masked: 0 if the toggled cell is dead), written by the thread that updates its chunk
            if (act >= 0 && t == (act >> 4) % C::TPE) {
                const bool live = ((cur[act >> 5] >> (act & 31)) & 1u) == 0u;      // cur holds the untoggled plane
                reinterpret_cast<int8_t *>(sst)[act] = (tr.masked && !live) ? (int8_t)0 : (int8_t)spawn4;
            }
        }
        // ---- stability plane in shared memory -------------------------------------------------------
#pragma unroll 2
        for (int j = 0; j < C::CPT; ++j) {
            const int c = j * C::TPE + t;
            const uint4 v = sst[c];
            uint32_t s[4] = {v.x, v.y, v.z, v.w};
            const uint32_t m = mix[c];
            const uint32_t sv = (m & 0x0f0f0f0fu) | tbn;
            const uint32_t bn = ((m >> 4) & 0x0f0f0f0fu) | tbn;
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const uint32_t surv_mask = lds32(__byte_perm(sv, lane_s, 0x5504 + 16 * k));
                if (rule == CGL_DEAD_ZERO) {
                    const uint32_t born_spawn = lds32(__byte_perm(bn, lane_b, 0x5504 + 16 * k));
                    s[k] = stable_update4(s[k], surv_mask, born_spawn, max4);
                } else {                    // the CGL_action+ fork's dead-cell rules (cgl_bits.cuh)
                    const uint32_t born_mask = lds32(__byte_perm(bn, lane_s, 0x5504 + 16 * k));
                    s[k] = stable_update4_rule(rule, s[k], surv_mask, born_mask, spawn4, max4, min4, empty4);
                }
                if constexpr (TR) racc = __dp4a((int)s[k], 0x01010101, racc);
            }
            sst[c] = make_uint4(s[0], s[1], s[2], s[3]);
            if constexpr (OBS) orow[c] = make_uint4(s[0], s[1], s[2], s[3]);     // (evict-first stores: no faster)
        }
        if (TR && want_trace) {
            racc = __reduce_add_sync(0xffffffffu, racc);
            pacc = __reduce_add_sync(0xffffffffu, pacc);
            if ((threadIdx.x & 31) == 0) {
                if constexpr (C::EPC == 1) {
                    atomicAdd(&slot[2 * (steps & 1)], racc);
                    atomicAdd(reinterpret_cast<unsigned *>(&slot[2 * (steps & 1) + 1]), pacc);
                } else {
                    if (tr.reward != nullptr) tr.reward[(size_t)steps * n_envs + e] = racc;
                    if (tr.alive != nullptr) tr.alive[(size_t)steps * n_envs + e] = pacc;
                }
            }
        }
        uint32_t *tmp = cur; cur = nxt; nxt = tmp;
        ++steps;
        done = steps >= max_steps || (stop_when_fixed && !any_changed);
        env_sync();                                  // mix and the old plane are free again
        if constexpr (TR && C::EPC == 1) {
            if (want_trace && t == 0) {              // the barrier above completed this step's sums
                int *sl = slot + 2 * ((steps - 1) & 1);
                if (tr.reward != nullptr) tr.reward[(size_t)(steps - 1) * n_envs + e] = sl[0];
                if (tr.alive != nullptr) tr.alive[(size_t)(steps - 1) * n_envs + e] = (uint32_t)sl[1];
                sl[0] = 0; sl[1] = 0;
            }
        }
    }

    // ---- write back: world, stability, reward, alive, steps ----------------------------------------
    int acc = 0;
    uint32_t pop = 0;
    if (active) {
        uint4 *wo = reinterpret_cast<uint4 *>(world_out + (size_t)e * C::WPE);
        for (int i = t; i < C::WPE / 4; i += C::TPE) {
            const uint4 v = reinterpret_cast<const uint4 *>(cur)[i];
            pop += __popc(v.x) + __popc(v.y) + __popc(v.z) + __popc(v.w);
            wo[i] = v;
        }
        uint4 *sp = reinterpret_cast<uint4 *>(stable + (size_t)e * C::SIZE);
#pragma unroll 4
        for (int j = 0; j < C::CPT; ++j) {
            const uint4 v = sst[j * C::TPE + t];
            acc = __dp4a((int)v.x, 0x01010101, acc); acc = __dp4a((int)v.y, 0x01010101, acc);
            acc = __dp4a((int)v.z, 0x01010101, acc); acc = __dp4a((int)v.w, 0x01010101, acc);
            if constexpr (!OBS) sp[j * C::TPE + t] = v;
        }
    }
    acc = __reduce_add_sync(0xffffffffu, acc);
    pop = __reduce_add_sync(0xffffffffu, pop);
    if constexpr (C::EPC == 1) {
        if ((threadIdx.x & 31) == 0) {
            atomicAdd(&red[0], acc);
            atomicAdd(reinterpret_cast<unsigned *>(&red[1]), pop);
        }
        __syncthreads();
        acc = red[0];
        pop = (uint32_t)red[1];
    }
    if (active && t == 0) {
        if (reward_out != nullptr) reward_out[e] = acc;
        if (alive_out != nullptr) alive_out[e] = pop;
        if (steps_out != nullptr) steps_out[e] = (int32_t)steps;
    }
}

// CYC (cgl_env_run_cycle): world_j is kept in history slot j % P.  `differs` has bit s set when world_t differs from
// slot s; the slots filled before step t are those of world_max(0, t-P) .. world_{t-1}.  Returns the lag p in
// 1..min(P, t) at which world_t repeats, or 0.  At most one filled slot can match (include/cgl_b200.h).
__device__ __forceinline__ uint32_t cycle_lag(uint32_t differs, uint32_t t, uint32_t P)
{
    const uint32_t filled = (1u << (t < P ? t : P)) - 1u;
    const uint32_t hit = ~differs & filled;
    if (hit == 0) return 0;
    const uint32_t p = (t - (uint32_t)(__ffs(hit) - 1)) % P;
    return p == 0 ? P : p;
}

// =========================================================================================
// Bit-sliced variant for longer runs.  Everything a thread owns stays in REGISTERS for the whole call: its
// rows of the world (bit plane) and their stability as 8 bit planes per 32 cells (cgl_bits.cuh).  The rule
// is ~33 logic ops per 32 cells instead of ~100 with bytes.  The only thing threads exchange per step are
// the horizontal neighbour sums (s0, s1) of their rows, through a double-buffered shared-memory plane -- each
// row's sums are computed once, by its owner -- and the barrier that publishes them also carries the
// "did the previous step change anything" vote: one barrier per step.  The byte <-> bit-plane transposes on
// the way in and out cost about five steps' worth of work, so cgl_env_run takes this kernel from
// max_steps >= 4.
// =========================================================================================
template <int S>
struct SlicedCfg {
    static constexpr int W = S / 32;
    static constexpr int WPE = S * W;
    static constexpr int SIZE = S * S;
    static constexpr int TPE = (S <= 64) ? 32 : S;
    static constexpr int EPC = (TPE >= 96) ? 1 : (128 / TPE);
    static constexpr int THREADS = TPE * EPC;
    static constexpr int RPB = S / TPE;
    // per env: two buffers x two planes (s0, s1) x WPE words
    static constexpr int SMEM = EPC * (4 * WPE * 4) + EPC * 8;
};

// RULE = CGL_DEAD_ZERO: the base env (dead cells are 0; "don't care" planes, spawn-relative).  CGL_DEAD_DECAY: the
// CGL_action+ fork's CUDA-kernel rule (dead cells fall by one per step to EMPTY_MIN), all cells carried
// spawn-relative.  CGL_DEAD_SAT: the fork's CPU rule (dead cells become min(s + EMPTY, EMPTY_MIN)) on absolute planes.
//
// TR (cgl_env_run_ex): the owner of the toggled cell's row flips the bit in its registers before it computes the
// row's sums -- the neighbours see the toggle through the published sums -- and writes the cell's planes.  Each step's
// reward comes from the planes (sliced_reward32), its live count from popc of the new rows.  One env per CTA: every
// warp adds its sums to a shared slot of the step's parity; thread 0 stores step t's after the barrier of step t+1
// (the one that publishes the sums) and clears the slot; the last step's values are the final reward and live count.
// Several envs per CTA (one warp each): lane 0 stores every step's sums.
//
// CYC (cgl_env_run_cycle, stop_when_fixed == 0, no actions): every thread keeps its own rows of the last max_period
// worlds in a ring in shared memory (world_0 written at load time); no other thread reads them, so no barrier is
// added.  Each new word is compared with every slot (one LOP3 per slot into a per-slot accumulator) before it
// replaces the oldest.  The per-slot "differs" bits are OR-reduced over the warp; one env per CTA: warps atomicOr them
// into a shared slot indexed by step & 3, read after the next step's barrier (the one that carries the vote) and
// cleared two steps later, and the last step's slot is read after the final barrier.  Several envs per CTA: the warp
// reduction is the whole env.
//
// SETTLE (cgl_env_run_settle, phase C): env e runs steps_out[e] steps, as set by the settle finder, instead of max_steps.
// One env per CTA: the bound is uniform over the CTA; several envs per CTA: each warp leaves at its own.
template <int S, int RULE, bool TR, bool CYC = false, bool SETTLE = false>
__global__ void __launch_bounds__(SlicedCfg<S>::THREADS)
env_run_sliced_kernel(const uint32_t *world_in, uint32_t *world_out, int8_t *stable, uint32_t n_envs,
                      uint32_t max_steps, int stop_when_fixed, int spawn, int stable_max, int empty_min,
                      int32_t *__restrict__ steps_out, int32_t *__restrict__ reward_out,
                      uint32_t *__restrict__ alive_out, int empty, RunTrace tr, uint32_t max_period,
                      int32_t *__restrict__ period_out)
{
    constexpr bool DECAY = RULE == CGL_DEAD_DECAY, SAT = RULE == CGL_DEAD_SAT;
    using C = SlicedCfg<S>;
    extern __shared__ __align__(16) unsigned char smem_dyn[];
    const int g = threadIdx.x / C::TPE;
    const int t = threadIdx.x % C::TPE;
    uint32_t *hbuf = reinterpret_cast<uint32_t *>(smem_dyn) + g * (4 * C::WPE);     // [buffer][plane][row][w]
    int *red = reinterpret_cast<int *>(smem_dyn + C::EPC * (4 * C::WPE * 4)) + g * 2;
    int *slot = reinterpret_cast<int *>(smem_dyn + C::EPC * (4 * C::WPE * 4)) + 2 * C::EPC;   // TR, EPC == 1
    // CYC: [after the TR slots] 4 "differs" slots (EPC == 1) | ring [env][max_period][word (j, w)][thread]
    unsigned *cyc = reinterpret_cast<unsigned *>(slot + 4);
    uint32_t *ring = reinterpret_cast<uint32_t *>(cyc + 4) + g * max_period * C::WPE + t;
    const uint32_t e = blockIdx.x * C::EPC + g;
    const bool active = e < n_envs;
    if constexpr (SETTLE)
        if (active) max_steps = (uint32_t)steps_out[e];

    uint32_t cw[C::RPB][C::W];                      // this thread's rows of the world
    uint32_t pl[C::RPB][C::W][8];                   // and their stability: 8 bit planes per word
    if (t == 0) { red[0] = 0; red[1] = 0; }
    if constexpr (TR && C::EPC == 1)
        if (t == 0) { slot[0] = 0; slot[1] = 0; slot[2] = 0; slot[3] = 0; }
    if constexpr (CYC && C::EPC == 1)
        if (t == 0) { cyc[0] = 0; cyc[1] = 0; cyc[2] = 0; cyc[3] = 0; }
    uint32_t odd = 0;                               // TR, base rule: live cells loaded with u > STABLE - SPAWN
    if (active) {
        const uint32_t *wp = world_in + (size_t)e * C::WPE;
        const uint4 *sp = reinterpret_cast<const uint4 *>(stable + (size_t)e * C::SIZE);
#pragma unroll
        for (int j = 0; j < C::RPB; ++j) {
            lds_words<C::W>(wp + (t * C::RPB + j) * C::W, cw[j]);       // (plain loads: the helper is address-space agnostic)
            if constexpr (CYC) {
#pragma unroll
                for (int w = 0; w < C::W; ++w) ring[(j * C::W + w) * C::TPE] = cw[j][w];       // world_0 -> slot 0
            }
#pragma unroll
            for (int w = 0; w < C::W; ++w) {
                const uint4 a = sp[((t * C::RPB + j) * S + w * 32) / 16];
                const uint4 b = sp[((t * C::RPB + j) * S + w * 32) / 16 + 1];
                const uint32_t by[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
                bytes_to_planes32(by, pl[j][w]);
                if constexpr (!SAT) add_const_sliced(pl[j][w], -spawn);     // spawn-relative planes (cgl_bits.cuh)
                if constexpr (TR && !SAT && !DECAY) odd |= gt_const_sliced(pl[j][w], (stable_max - spawn) & 0xff) & cw[j][w];
            }
        }
    }
    bool odd_env = false;
    if constexpr (TR) {
        if constexpr (C::EPC == 1) odd_env = __syncthreads_or(odd != 0) != 0;
        else { __syncthreads(); odd_env = __any_sync(0xffffffffu, odd != 0); }
    } else {
        __syncthreads();
    }
    const int max_rel = (stable_max - spawn) & 0xff, min_rel = (empty_min - spawn) & 0xff;

    auto env_vote = [&](bool p) -> bool {
        if constexpr (C::EPC == 1) return __syncthreads_or(p) != 0;
        const bool r = __any_sync(0xffffffffu, p);
        __syncwarp();
        return r;
    };

    // rows above this thread's first row and below its last one (torus)
    const int r_first = t * C::RPB, r_last = t * C::RPB + C::RPB - 1;
    const int r_up = r_first == 0 ? S - 1 : r_first - 1;
    const int r_dn = r_last == S - 1 ? 0 : r_last + 1;

    uint32_t steps = 0, changed = 1u, buf = 0;
    uint32_t period = 0, wslot = CYC ? 1u % max_period : 0u;        // CYC: the ring slot of the next world
    const bool want_trace = TR && (tr.reward != nullptr || tr.alive != nullptr);
    // The base rule's live cells hold u in [0, STABLE - SPAWN] (a toggle or a birth sets 0, survivors count up to it)
    // unless the loaded plane had others; u > 127 - SPAWN then needs SPAWN..MAX to wrap int8.
    const bool wraps = DECAY || max_rel > 127 - spawn || odd_env;
    if (active) {
        int next_act = C::SIZE;                     // the no-op
        if constexpr (TR)
            if (tr.actions != nullptr && max_steps > 0) next_act = tr.actions[e];
        while (steps < max_steps) {
            if constexpr (TR) {
                const int a = next_act;             // all threads of the env load the same word: a broadcast
                if (tr.actions != nullptr && steps + 1 < max_steps) next_act = tr.actions[(size_t)(steps + 1) * n_envs + e];
                if (a >= 0 && a < C::SIZE) {
                    if (a / (S * C::RPB) == t) {    // the owner of the cell's row
                        const int j = (a / S) % C::RPB, w = (a % S) >> 5;
                        const uint32_t bit = 1u << (a & 31);
#pragma unroll
                        for (int jj = 0; jj < C::RPB; ++jj)
#pragma unroll
                            for (int ww = 0; ww < C::W; ++ww)
                                if (jj == j && ww == w) {
                                    cw[jj][ww] ^= bit;
                                    const int v = (tr.masked && !(cw[jj][ww] & bit)) ? 0 : spawn;
                                    set_cells_sliced(pl[jj][ww], bit, SAT ? v : v - spawn);
                                }
                    }
                } else if (a != C::SIZE && t == 0) {
                    if (tr.err_flag != nullptr) atomicOr(tr.err_flag, 1);
                    raise_alarm(ALARM_BAD_ACTION);
                }
            }
            // horizontal sums of my rows; (s0, s1) go to the shared plane for the rows above and below
            HSum hs[C::RPB][C::W];
            uint32_t *h0 = hbuf + buf * (2 * C::WPE), *h1 = h0 + C::WPE;
#pragma unroll
            for (int j = 0; j < C::RPB; ++j) {
                uint32_t s0[C::W], s1[C::W];
#pragma unroll
                for (int w = 0; w < C::W; ++w) {
                    hs[j][w] = hsum(west_plane(cw[j][(w + C::W - 1) % C::W], cw[j][w]), cw[j][w],
                                    east_plane(cw[j][w], cw[j][(w + 1) % C::W]));
                    s0[w] = hs[j][w].s0; s1[w] = hs[j][w].s1;
                }
                if (j == 0 || j == C::RPB - 1) {                // only edge rows are read by other threads
                    sts_words<C::W>(h0 + (t * C::RPB + j) * C::W, s0);
                    sts_words<C::W>(h1 + (t * C::RPB + j) * C::W, s1);
                }
            }
            // one barrier: publishes the sums and votes on whether the PREVIOUS step changed the world
            const bool any_changed = env_vote(changed != 0);
            if (stop_when_fixed && !any_changed) break;
            if constexpr (CYC && C::EPC == 1) {
                if (steps > 0) {                    // the barrier above completed the previous step's "differs" bits
                    period = cycle_lag(cyc[(steps - 1) & 3], steps, max_period);
                    if (period != 0) break;
                }
                if (t == 0) cyc[(steps + 2) & 3] = 0;       // last read in the previous step, next written two on
            }
            if constexpr (TR && C::EPC == 1) {
                if (want_trace && t == 0 && steps > 0) {
                    int *sl = slot + 2 * ((steps - 1) & 1);
                    if (tr.reward != nullptr) tr.reward[(size_t)(steps - 1) * n_envs + e] = sl[0];
                    if (tr.alive != nullptr) tr.alive[(size_t)(steps - 1) * n_envs + e] = (uint32_t)sl[1];
                    sl[0] = 0; sl[1] = 0;
                }
            }
            int racc = 0;
            uint32_t pacc = 0;
            uint32_t up0[C::W], up1[C::W], dn0[C::W], dn1[C::W];
            lds_words<C::W>(h0 + r_up * C::W, up0);
            lds_words<C::W>(h1 + r_up * C::W, up1);
            lds_words<C::W>(h0 + r_dn * C::W, dn0);
            lds_words<C::W>(h1 + r_dn * C::W, dn1);
            changed = 0;
            uint32_t dacc[CGL_RUN_MAX_PERIOD] = {};         // CYC: OR of (new ^ slot s) over my words
#pragma unroll
            for (int j = 0; j < C::RPB; ++j) {
#pragma unroll
                for (int w = 0; w < C::W; ++w) {
                    const HSum up = {j == 0 ? up0[w] : hs[j > 0 ? j - 1 : 0][w].s0,
                                     j == 0 ? up1[w] : hs[j > 0 ? j - 1 : 0][w].s1, 0, 0};
                    const HSum dn = {j == C::RPB - 1 ? dn0[w] : hs[j < C::RPB - 1 ? j + 1 : 0][w].s0,
                                     j == C::RPB - 1 ? dn1[w] : hs[j < C::RPB - 1 ? j + 1 : 0][w].s1, 0, 0};
                    const uint32_t c = cw[j][w];
                    const uint32_t n = life_rule(up, hs[j][w], dn, c);
                    changed |= n ^ c;
                    if constexpr (SAT) stable_update_sliced_sat(pl[j][w], n & c, n & ~c, spawn, stable_max, empty, empty_min);
                    else if constexpr (DECAY) stable_update_sliced_decay(pl[j][w], n & c, n & ~c, max_rel, min_rel);
                    else stable_update_sliced_rel(pl[j][w], n & c, max_rel);
                    if constexpr (TR) {
                        racc += sliced_reward32(RULE, pl[j][w], n, spawn, wraps);
                        pacc += __popc(n);
                    }
                    if constexpr (CYC) {
                        uint32_t *rw = ring + (j * C::W + w) * C::TPE;
#pragma unroll
                        for (int s = 0; s < CGL_RUN_MAX_PERIOD; ++s)
                            if (s < (int)max_period) dacc[s] |= n ^ rw[s * C::WPE];
                        rw[wslot * C::WPE] = n;
                    }
                    cw[j][w] = n;
                }
            }
            if (TR && want_trace) {
                racc = __reduce_add_sync(0xffffffffu, racc);
                pacc = __reduce_add_sync(0xffffffffu, pacc);
                if ((threadIdx.x & 31) == 0) {
                    if constexpr (C::EPC == 1) {
                        atomicAdd(&slot[2 * (steps & 1)], racc);
                        atomicAdd(reinterpret_cast<unsigned *>(&slot[2 * (steps & 1) + 1]), pacc);
                    } else {
                        if (tr.reward != nullptr) tr.reward[(size_t)steps * n_envs + e] = racc;
                        if (tr.alive != nullptr) tr.alive[(size_t)steps * n_envs + e] = pacc;
                    }
                }
            }
            uint32_t differs = 0;
            if constexpr (CYC) {
#pragma unroll
                for (int s = 0; s < CGL_RUN_MAX_PERIOD; ++s) differs |= (dacc[s] != 0 ? 1u : 0u) << s;
                differs = __reduce_or_sync(0xffffffffu, differs);
                if (C::EPC == 1 && (threadIdx.x & 31) == 0 && differs != 0) atomicOr(&cyc[steps & 3], differs);
                wslot = wslot + 1 == max_period ? 0 : wslot + 1;
            }
            ++steps;
            buf ^= 1u;                              // the next step writes the other buffer: no reader is overtaken
            if constexpr (CYC && C::EPC > 1) {
                period = cycle_lag(differs, steps, max_period);
                if (period != 0) break;
            }
        }
    }

    int acc = 0;
    uint32_t pop = 0;
    if (active) {
        uint32_t *wo = world_out + (size_t)e * C::WPE;
        uint4 *sp = reinterpret_cast<uint4 *>(stable + (size_t)e * C::SIZE);
#pragma unroll
        for (int j = 0; j < C::RPB; ++j) {
            sts_words<C::W>(wo + (t * C::RPB + j) * C::W, cw[j]);
#pragma unroll
            for (int w = 0; w < C::W; ++w) {
                pop += __popc(cw[j][w]);
                if constexpr (!SAT) add_const_sliced(pl[j][w], spawn);      // back to absolute values; dead cells are 0
                if constexpr (!DECAY && !SAT) {
#pragma unroll
                    for (int b = 0; b < 8; ++b) pl[j][w][b] &= cw[j][w];
                }
                // reward = sum of int8 values = sum_b 2^b popc(plane b), the sign plane weighing -128
#pragma unroll
                for (int b = 0; b < 7; ++b) acc += __popc(pl[j][w][b]) << b;
                acc -= __popc(pl[j][w][7]) << 7;
                uint32_t by[8];
                planes_to_bytes32(pl[j][w], by);
                sp[((t * C::RPB + j) * S + w * 32) / 16] = make_uint4(by[0], by[1], by[2], by[3]);
                sp[((t * C::RPB + j) * S + w * 32) / 16 + 1] = make_uint4(by[4], by[5], by[6], by[7]);
            }
        }
    }
    acc = __reduce_add_sync(0xffffffffu, acc);
    pop = __reduce_add_sync(0xffffffffu, pop);
    if constexpr (C::EPC == 1) {
        if ((threadIdx.x & 31) == 0) {
            atomicAdd(&red[0], acc);
            atomicAdd(reinterpret_cast<unsigned *>(&red[1]), pop);
        }
        __syncthreads();
        acc = red[0];
        pop = (uint32_t)red[1];
        // a run that used its whole budget: the barrier above completed the last step's "differs" bits
        if constexpr (CYC)
            if (period == 0 && steps > 0) period = cycle_lag(cyc[(steps - 1) & 3], steps, max_period);
    }
    if (active && t == 0) {
        if (reward_out != nullptr) reward_out[e] = acc;
        if (alive_out != nullptr) alive_out[e] = pop;
        if (steps_out != nullptr) steps_out[e] = (int32_t)steps;
        if constexpr (CYC)
            if (period_out != nullptr) period_out[e] = (int32_t)period;
        if constexpr (TR && C::EPC == 1) {
            if (steps > 0) {                        // the last step: its sums are the final reward and live count
                if (tr.reward != nullptr) tr.reward[(size_t)(steps - 1) * n_envs + e] = acc;
                if (tr.alive != nullptr) tr.alive[(size_t)(steps - 1) * n_envs + e] = pop;
            }
        }
    }
}

// Any side whose three byte planes fit in 220 KiB of shared memory (side <= 274): one CTA per env, one byte per cell.
// TR: thread 0 applies the step's toggle before a barrier; the per-step sums ride on the loop over the cells and are
// stored by thread 0 after the step's vote.  OBS (implies TR): every cell's new stability byte is also stored to row
// (step, e) of `obs` (rows need not be 16-byte aligned), and the plane is not written back.
// CYC (cgl_env_run_cycle): the last max_period worlds are kept as flat bit vectors of ceil(size/32) words after the
// three planes.  The cell loop runs over whole warps; each warp packs its 32 new cells with one ballot (i is
// warp-contiguous; the bit order does not matter for equality) and its lane 0 compares the word with every slot and
// stores it.  Lane 0s atomicOr their "differs" bits into a shared slot indexed by step & 3, read after the vote.
// SETTLE (cgl_env_run_settle, phase C): the env runs steps_out[e] steps, as set by the settle finder, not max_steps.
template <bool TR, bool OBS = false, bool CYC = false, bool SETTLE = false>
__global__ void __launch_bounds__(256)
env_run_generic_kernel(const uint32_t *world_in, uint32_t *world_out, int8_t *stable, uint32_t side, uint32_t W,
                       uint32_t max_steps, int stop_when_fixed, int8_t spawn, int8_t stable_max,
                       int32_t *__restrict__ steps_out, int32_t *__restrict__ reward_out,
                       uint32_t *__restrict__ alive_out, int rule, int8_t empty, int8_t empty_min, RunTrace tr,
                       int8_t *obs, uint32_t max_period, int32_t *__restrict__ period_out)
{
    extern __shared__ __align__(16) unsigned char smem_dyn[];
    const uint32_t size = side * side;
    uint8_t *a = smem_dyn, *b = a + size;
    int8_t *st = reinterpret_cast<int8_t *>(b + size);
    const uint32_t nw = (size + 31) / 32;           // CYC: words per world in the history
    uint32_t *hist = reinterpret_cast<uint32_t *>(smem_dyn + ((3 * size + 3) & ~3u));
    __shared__ int red[(TR ? 6 : 2) + (CYC ? 4 : 0)];   // TR: red[2 + 2 * (step & 1)] = the step's (reward, alive)
    unsigned *cyc = reinterpret_cast<unsigned *>(red + (TR ? 6 : 2));      // CYC: "differs" bits by step & 3
    const uint64_t e = blockIdx.x;
    const uint32_t *wi = world_in + e * side * W;
    uint32_t *wo = world_out + e * side * W;
    int8_t *sg = stable + e * size;
    if constexpr (SETTLE) max_steps = (uint32_t)steps_out[e];
    if (threadIdx.x == 0) { red[0] = 0; red[1] = 0; }
    if constexpr (TR)
        if (threadIdx.x == 0) { red[2] = 0; red[3] = 0; red[4] = 0; red[5] = 0; }
    if constexpr (CYC)
        if (threadIdx.x == 0) { cyc[0] = 0; cyc[1] = 0; cyc[2] = 0; cyc[3] = 0; }
    for (uint32_t i = threadIdx.x; i < size; i += blockDim.x) {
        const uint32_t y = i / side, x = i - y * side;
        a[i] = (wi[y * W + (x >> 5)] >> (x & 31)) & 1u;
        st[i] = sg[i];
    }
    __syncthreads();
    if constexpr (CYC) {                            // world_0 -> slot 0, in the bit order of the step's ballots
        for (uint32_t w = threadIdx.x; w < nw; w += blockDim.x) {
            uint32_t word = 0;
            for (uint32_t j = 0; j < 32 && 32 * w + j < size; ++j) word |= (uint32_t)a[32 * w + j] << j;
            hist[w] = word;
        }
        __syncthreads();
    }
    uint32_t steps = 0, period = 0, wslot = CYC ? 1u % max_period : 0u;
    bool done = max_steps == 0;
    while (!done) {
        int changed = 0;
        int racc = 0;
        uint32_t pacc = 0;
        int8_t *orow = nullptr;
        if constexpr (OBS) orow = obs + ((size_t)steps * gridDim.x + e) * size;
        if constexpr (TR) {
            if (tr.actions != nullptr) {
                if (threadIdx.x == 0) {
                    const int act = tr.actions[(size_t)steps * gridDim.x + e];
                    if (act >= 0 && (uint32_t)act < size) {
                        a[act] ^= 1u;
                        st[act] = (tr.masked && !a[act]) ? (int8_t)0 : spawn;
                    } else if ((uint32_t)act != size) {
                        if (tr.err_flag != nullptr) atomicOr(tr.err_flag, 1);
                        raise_alarm(ALARM_BAD_ACTION);
                    }
                }
                __syncthreads();
            }
        }
        uint32_t differs = 0;                        // CYC, lane 0: bit s = a word of mine differs from slot s
        const uint32_t lim = CYC ? nw * 32 : size;
        for (uint32_t i = threadIdx.x; i < lim; i += blockDim.x) {
            bool live = false;
            if (!CYC || i < size) {
                const uint32_t y = i / side, x = i - y * side;
                const uint32_t yu = (y == 0 ? side : y) - 1, yd = (y + 1 == side) ? 0 : y + 1;
                const uint32_t xl = (x == 0 ? side : x) - 1, xr = (x + 1 == side) ? 0 : x + 1;
                const uint32_t n = a[yu * side + xl] + a[yu * side + x] + a[yu * side + xr] + a[y * side + xl] +
                                   a[y * side + xr] + a[yd * side + xl] + a[yd * side + x] + a[yd * side + xr];
                const uint8_t p = a[i];
                const uint8_t q = (n == 3u) || (n == 2u && p);
                b[i] = q;
                changed |= (p != q);
                st[i] = stable_update1_rule(rule, st[i], p != 0, q != 0, spawn, stable_max, empty, empty_min);
                if constexpr (OBS) orow[i] = st[i];
                if constexpr (TR) { racc += st[i]; pacc += q; }
                live = q != 0;
            }
            if constexpr (CYC) {
                const uint32_t word = __ballot_sync(0xffffffffu, live);
                if ((threadIdx.x & 31) == 0) {
                    uint32_t *hw = hist + (i >> 5);
                    for (uint32_t s = 0; s < max_period; ++s) differs |= (hw[s * nw] != word ? 1u : 0u) << s;
                    hw[wslot * nw] = word;
                }
            }
        }
        if constexpr (CYC)
            if ((threadIdx.x & 31) == 0 && differs != 0) atomicOr(&cyc[steps & 3], differs);
        if constexpr (TR) {
            racc = __reduce_add_sync(0xffffffffu, racc);
            pacc = __reduce_add_sync(0xffffffffu, pacc);
            if ((threadIdx.x & 31) == 0) {
                atomicAdd(&red[2 + 2 * (steps & 1)], racc);
                atomicAdd(reinterpret_cast<unsigned *>(&red[3 + 2 * (steps & 1)]), pacc);
            }
        }
        const bool any_changed = __syncthreads_or(changed) != 0;
        if constexpr (TR) {
            // the vote's barrier completed the sums; the slot is added to again two steps later, after the next vote
            if (threadIdx.x == 0) {
                int *sl = red + 2 + 2 * (steps & 1);
                if (tr.reward != nullptr) tr.reward[(size_t)steps * gridDim.x + e] = sl[0];
                if (tr.alive != nullptr) tr.alive[(size_t)steps * gridDim.x + e] = (uint32_t)sl[1];
                sl[0] = 0; sl[1] = 0;
            }
        }
        if constexpr (CYC) {
            // the vote's barrier completed this step's bits; the slot two steps on was last read a step ago
            period = cycle_lag(cyc[steps & 3], steps + 1, max_period);
            if (threadIdx.x == 0) cyc[(steps + 2) & 3] = 0;
            wslot = wslot + 1 == max_period ? 0 : wslot + 1;
        }
        uint8_t *tmp = a; a = b; b = tmp;
        ++steps;
        done = steps >= max_steps || (stop_when_fixed && !any_changed) || period != 0;
    }
    int acc = 0;
    uint32_t pop = 0;
    for (uint32_t i = threadIdx.x; i < size; i += blockDim.x) {
        if constexpr (!OBS) sg[i] = st[i];
        acc += st[i];
    }
    for (uint32_t wdx = threadIdx.x; wdx < side * W; wdx += blockDim.x) {
        const uint32_t y = wdx / W, x0 = (wdx - y * W) * 32;
        uint32_t word = 0;
        for (uint32_t j = 0; j < 32 && x0 + j < side; ++j) word |= (uint32_t)a[y * side + x0 + j] << j;
        pop += __popc(word);
        wo[wdx] = word;
    }
    acc = __reduce_add_sync(0xffffffffu, acc);
    pop = __reduce_add_sync(0xffffffffu, pop);
    if ((threadIdx.x & 31) == 0) {
        atomicAdd(&red[0], acc);
        atomicAdd(reinterpret_cast<unsigned *>(&red[1]), pop);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        if (reward_out != nullptr) reward_out[e] = red[0];
        if (alive_out != nullptr) alive_out[e] = (uint32_t)red[1];
        if (steps_out != nullptr) steps_out[e] = (int32_t)steps;
        if constexpr (CYC)
            if (period_out != nullptr) period_out[e] = (int32_t)period;
    }
}

// =========================================================================================
// cgl_env_run_settle, phases A and B: each env's first repeated world, of any period, from world-only generations.
// A settle run takes no actions, so the world evolves without reference to the stability plane.  With M = max_steps:
//   A: advance world_t and compare it with one checkpoint world_c, c the largest member of {0} u {2^k < M} u {M}
//      below t.  The first match gives lambda = t - c: a match implies c >= mu, and the first match after c is at
//      c + lambda.  No match by t = 2M means mu + lambda > M, since world_{M+lambda} == world_M would have matched.
//   B: runners from world_0 and world_lambda in lockstep; the first equal pair is world_mu.  Given up once
//      mu + lambda > M.
// steps_out[e] = mu + lambda and period_out[e] = lambda, or (M, 0).  Phase C (the SETTLE instantiations above) then
// runs exactly steps_out[e] full steps from the untouched inputs.  The counters are 64-bit: 2M passes 2^32.
// =========================================================================================
__device__ __forceinline__ bool settle_checkpoint(uint64_t t, uint64_t M)
{
    return t == M || (t < M && (t & (t - 1)) == 0);
}

// Fused sides: the bit-sliced kernel's layout and its one barrier per generation, without the stability planes.
// Each thread holds its rows of the world and the checkpoint (phase A) or of both runners (phase B) in registers;
// the barrier that publishes a generation's sums also carries the vote on the previous comparison.
template <int S>
__global__ void __launch_bounds__(SlicedCfg<S>::THREADS)
env_settle_find_kernel(const uint32_t *world_in, uint32_t n_envs, uint32_t max_steps, int32_t *__restrict__ steps_out,
                       int32_t *__restrict__ period_out)
{
    using C = SlicedCfg<S>;
    extern __shared__ __align__(16) unsigned char smem_dyn[];
    const int g = threadIdx.x / C::TPE;
    const int t = threadIdx.x % C::TPE;
    uint32_t *hbuf = reinterpret_cast<uint32_t *>(smem_dyn) + g * (4 * C::WPE);     // [buffer][plane][row][w]
    const uint32_t e = blockIdx.x * C::EPC + g;
    if (e >= n_envs) return;                        // a whole CTA (one env per CTA) or a whole warp (one per env)
    const uint32_t *wp = world_in + (size_t)e * C::WPE;
    const int r_first = t * C::RPB, r_last = t * C::RPB + C::RPB - 1;
    const int r_up = r_first == 0 ? S - 1 : r_first - 1;
    const int r_dn = r_last == S - 1 ? 0 : r_last + 1;
    uint32_t buf = 0;

    auto env_vote = [&](bool p) -> bool {
        if constexpr (C::EPC == 1) return __syncthreads_or(p) != 0;
        const bool r = __any_sync(0xffffffffu, p);
        __syncwarp();
        return r;
    };
    auto load = [&](uint32_t (&x)[C::RPB][C::W]) {
#pragma unroll
        for (int j = 0; j < C::RPB; ++j) lds_words<C::W>(wp + (t * C::RPB + j) * C::W, x[j]);
    };
    // One generation of x in two halves around the barrier: sums() publishes the edge rows' sums, next() reads the
    // neighbours' sums and replaces x, calling visit(j, w, old word, new word) for every word.
    auto sums = [&](const uint32_t (&x)[C::RPB][C::W], HSum (&hs)[C::RPB][C::W]) {
        uint32_t *h0 = hbuf + buf * (2 * C::WPE), *h1 = h0 + C::WPE;
#pragma unroll
        for (int j = 0; j < C::RPB; ++j) {
            uint32_t s0[C::W], s1[C::W];
#pragma unroll
            for (int w = 0; w < C::W; ++w) {
                hs[j][w] = hsum(west_plane(x[j][(w + C::W - 1) % C::W], x[j][w]), x[j][w],
                                east_plane(x[j][w], x[j][(w + 1) % C::W]));
                s0[w] = hs[j][w].s0; s1[w] = hs[j][w].s1;
            }
            if (j == 0 || j == C::RPB - 1) {
                sts_words<C::W>(h0 + (t * C::RPB + j) * C::W, s0);
                sts_words<C::W>(h1 + (t * C::RPB + j) * C::W, s1);
            }
        }
    };
    auto next = [&](uint32_t (&x)[C::RPB][C::W], const HSum (&hs)[C::RPB][C::W], auto &&visit) {
        const uint32_t *h0 = hbuf + buf * (2 * C::WPE), *h1 = h0 + C::WPE;
        uint32_t up0[C::W], up1[C::W], dn0[C::W], dn1[C::W];
        lds_words<C::W>(h0 + r_up * C::W, up0);
        lds_words<C::W>(h1 + r_up * C::W, up1);
        lds_words<C::W>(h0 + r_dn * C::W, dn0);
        lds_words<C::W>(h1 + r_dn * C::W, dn1);
#pragma unroll
        for (int j = 0; j < C::RPB; ++j) {
#pragma unroll
            for (int w = 0; w < C::W; ++w) {
                const HSum up = {j == 0 ? up0[w] : hs[j > 0 ? j - 1 : 0][w].s0,
                                 j == 0 ? up1[w] : hs[j > 0 ? j - 1 : 0][w].s1, 0, 0};
                const HSum dn = {j == C::RPB - 1 ? dn0[w] : hs[j < C::RPB - 1 ? j + 1 : 0][w].s0,
                                 j == C::RPB - 1 ? dn1[w] : hs[j < C::RPB - 1 ? j + 1 : 0][w].s1, 0, 0};
                const uint32_t n = life_rule(up, hs[j][w], dn, x[j][w]);
                visit(j, w, x[j][w], n);
                x[j][w] = n;
            }
        }
        buf ^= 1u;                                  // the next generation writes the other buffer
    };
    auto nop = [](int, int, uint32_t, uint32_t) {};

    // ---- phase A: lambda ------------------------------------------------------------------------------
    const uint64_t M = max_steps;
    uint32_t x[C::RPB][C::W], y[C::RPB][C::W];      // A: the world and the checkpoint; B: the two runners
    load(x);
    load(y);
    uint64_t c = 0, lam = 0;
    uint32_t diff = 0;                              // OR of world_i ^ world_c over my words
    for (uint64_t i = 0;; ++i) {
        HSum hs[C::RPB][C::W];
        sums(x, hs);
        const bool differs = env_vote(diff != 0);
        if (i > 0 && !differs) { lam = i - c; break; }
        if (i == 2 * M) break;
        const bool keep = settle_checkpoint(i, M);  // world_i becomes the checkpoint
        if (keep) c = i;
        diff = 0;
        next(x, hs, [&](int j, int w, uint32_t o, uint32_t n) {
            if (keep) y[j][w] = o;
            diff |= n ^ y[j][w];
        });
    }

    // ---- phase B: mu ----------------------------------------------------------------------------------
    uint64_t steps = M;
    uint32_t period = 0;
    if (lam != 0 && lam <= M) {
        load(x);
        load(y);
        for (uint64_t i = 0; i < lam; ++i) {       // y = world_lambda
            HSum hs[C::RPB][C::W];
            sums(y, hs);
            env_vote(false);
            next(y, hs, nop);
        }
        diff = 0;
#pragma unroll
        for (int j = 0; j < C::RPB; ++j)
#pragma unroll
            for (int w = 0; w < C::W; ++w) diff |= x[j][w] ^ y[j][w];
        for (uint64_t mu = 0;; ++mu) {             // x = world_mu, y = world_{mu + lambda}
            HSum hs[C::RPB][C::W];
            sums(x, hs);
            if (!env_vote(diff != 0)) { steps = mu + lam; period = (uint32_t)lam; break; }
            if (mu + lam == M) break;
            next(x, hs, nop);
            sums(y, hs);
            env_vote(false);
            diff = 0;
            next(y, hs, [&](int j, int w, uint32_t, uint32_t n) { diff |= n ^ x[j][w]; });
        }
    }
    if (t == 0) {
        steps_out[e] = (int32_t)(uint32_t)steps;
        if (period_out != nullptr) period_out[e] = (int32_t)period;
    }
}

// Other sides: one CTA per env.  Worlds are flat bit vectors of ceil(side^2/32) words in shared memory (bit i = cell
// i), four of them: phase A uses three (the world, the next one and the checkpoint, which is the world's own buffer
// until the world moves on), phase B two per runner.  A generation packs each warp's 32 new cells with one ballot;
// lane 0 stores the word and compares it with the reference world's, and one barrier carries the vote.
__global__ void __launch_bounds__(256)
env_settle_find_generic_kernel(const uint32_t *world_in, uint32_t side, uint32_t W, uint32_t max_steps,
                               int32_t *__restrict__ steps_out, int32_t *__restrict__ period_out)
{
    extern __shared__ __align__(16) unsigned char smem_dyn[];
    const uint32_t size = side * side, nw = (size + 31) / 32;
    uint32_t *bits = reinterpret_cast<uint32_t *>(smem_dyn);
    auto world = [&](int k) { return bits + k * nw; };
    const uint32_t *wi = world_in + (uint64_t)blockIdx.x * side * W;
    auto load = [&](uint32_t *dst) {
        for (uint32_t w = threadIdx.x; w < nw; w += blockDim.x) {
            uint32_t word = 0;
            for (uint32_t j = 0; j < 32 && 32 * w + j < size; ++j) {
                const uint32_t i = 32 * w + j, y = i / side, x = i - y * side;
                word |= ((wi[y * W + (x >> 5)] >> (x & 31)) & 1u) << j;
            }
            dst[w] = word;
        }
    };
    // src -> dst; returns whether any new word differs from ref's (ref may be NULL: no comparison)
    auto gen = [&](const uint32_t *src, uint32_t *dst, const uint32_t *ref) -> bool {
        auto cell = [&](uint32_t y, uint32_t x) { const uint32_t k = y * side + x; return (src[k >> 5] >> (k & 31)) & 1u; };
        uint32_t d = 0;
        for (uint32_t i = threadIdx.x; i < nw * 32; i += blockDim.x) {       // whole warps: nw * 32 cells
            bool live = false;
            if (i < size) {
                const uint32_t y = i / side, x = i - y * side;
                const uint32_t yu = (y == 0 ? side : y) - 1, yd = (y + 1 == side) ? 0 : y + 1;
                const uint32_t xl = (x == 0 ? side : x) - 1, xr = (x + 1 == side) ? 0 : x + 1;
                const uint32_t n = cell(yu, xl) + cell(yu, x) + cell(yu, xr) + cell(y, xl) + cell(y, xr) +
                                   cell(yd, xl) + cell(yd, x) + cell(yd, xr);
                live = n == 3u || (n == 2u && cell(y, x));
            }
            const uint32_t word = __ballot_sync(0xffffffffu, live);
            if ((threadIdx.x & 31) == 0) {
                dst[i >> 5] = word;
                if (ref != nullptr) d |= word ^ ref[i >> 5];
            }
        }
        return __syncthreads_or(d != 0) != 0;
    };

    // ---- phase A: lambda ------------------------------------------------------------------------------
    const uint64_t M = max_steps;
    load(world(0));
    __syncthreads();
    int cur = 0, ck = 0;
    uint64_t c = 0, lam = 0;
    for (uint64_t i = 0; i < 2 * M; ++i) {
        if (settle_checkpoint(i, M)) { ck = cur; c = i; }
        const int nxt = cur != ck ? 3 - cur - ck : (cur + 1) % 3;
        const bool differs = gen(world(cur), world(nxt), world(ck));
        cur = nxt;
        if (!differs) { lam = i + 1 - c; break; }
    }

    // ---- phase B: mu ----------------------------------------------------------------------------------
    uint64_t steps = M;
    uint32_t period = 0;
    if (lam != 0 && lam <= M) {
        int x = 0, y = 2;                           // x in buffers 0 / 1, y in 2 / 3
        load(world(x));
        load(world(y));
        __syncthreads();
        for (uint64_t i = 0; i < lam; ++i) { gen(world(y), world(y ^ 1), nullptr); y ^= 1; }
        uint32_t d = 0;
        for (uint32_t w = threadIdx.x; w < nw; w += blockDim.x) d |= world(x)[w] ^ world(y)[w];
        bool differs = __syncthreads_or(d != 0) != 0;
        uint64_t mu = 0;
        for (; differs && mu + lam < M; ++mu) {
            gen(world(x), world(x ^ 1), nullptr); x ^= 1;
            differs = gen(world(y), world(y ^ 1), world(x)); y ^= 1;
        }
        if (!differs) { steps = mu + lam; period = (uint32_t)lam; }
    }
    if (threadIdx.x == 0) {
        steps_out[blockIdx.x] = (int32_t)(uint32_t)steps;
        if (period_out != nullptr) period_out[blockIdx.x] = (int32_t)period;
    }
}

// Shared memory of the generic settle finder: four bit-vector worlds.
static uint64_t settle_find_smem(uint32_t side)
{
    return 4 * 4 * (((uint64_t)side * side + 31) / 32);
}

// CGL_RUN_IMPL=bytes | sliced forces one kernel (tests, tuning); default: sliced from 4 steps on
// (measured on B200 at 4096 x 128^2: a launch costs ~50 us + 5.3 us per step sliced, ~25 us + 14 us per step bytes).
static bool run_use_sliced(uint32_t max_steps)
{
    static int forced = -1;
    if (forced < 0) {
        const char *v = getenv("CGL_RUN_IMPL");
        forced = (v && v[0] == 'b') ? 1 : (v && v[0] == 's') ? 2 : 0;
    }
    if (forced == 1) return false;
    if (forced == 2) return true;
    return max_steps >= 4;
}

// OBS runs take the byte kernel at every step count: the bit-sliced kernel would need a planes -> bytes transpose
// per 32 cells in every step to store the observation (DESIGN.md section 8 f3.2).
template <int S, bool TR, bool OBS>
static void launch_env_run_as(const cgl_env_run_args_t &a, const RunTrace &tr, int8_t *obs, cudaStream_t st)
{
    using C = RunCfg<S>;
    const unsigned grid = (unsigned)((a.n_envs + C::EPC - 1) / C::EPC);
    if (!OBS && run_use_sliced(a.max_steps)) {
        using D = SlicedCfg<S>;
        constexpr int smem = D::SMEM + (TR ? 16 : 0);             // TR: the step sums' slots
#define CGL_RUN_SLICED(RULE)                                                                                          \
    env_run_sliced_kernel<S, RULE, TR><<<grid, D::THREADS, smem, st>>>(                                                \
        a.world_in_dev, a.world_out_dev, a.stable_dev, (uint32_t)a.n_envs, a.max_steps, a.stop_when_fixed, a.spawn,   \
        a.stable_max, a.empty_min, a.steps_out_dev, a.reward_out_dev, a.alive_out_dev, a.empty, tr, 0u, nullptr)
        if (a.dead_rule == CGL_DEAD_DECAY) CGL_RUN_SLICED(CGL_DEAD_DECAY);
        else if (a.dead_rule == CGL_DEAD_SAT) CGL_RUN_SLICED(CGL_DEAD_SAT);
        else CGL_RUN_SLICED(CGL_DEAD_ZERO);
#undef CGL_RUN_SLICED
    } else {
        env_run_kernel<S, TR, OBS><<<grid, C::THREADS, C::SMEM + (TR ? 16 : 0), st>>>(
            a.world_in_dev, a.world_out_dev, a.stable_dev, (uint32_t)a.n_envs, a.max_steps, a.stop_when_fixed,
            rep4(a.spawn), rep4(a.stable_max), a.steps_out_dev, a.reward_out_dev, a.alive_out_dev, a.dead_rule,
            rep4(a.empty_min), rep4(a.empty), tr, obs);
    }
}

template <int S>
static int launch_env_run(const cgl_env_run_args_t &a, bool traced, const RunTrace &tr, int8_t *obs, cudaStream_t st)
{
    using C = RunCfg<S>;
    static PerDeviceOnce once;
    if (once.first()) {
        CGL_CUDA(cudaFuncSetAttribute(env_run_kernel<S, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM));
        CGL_CUDA(cudaFuncSetAttribute(env_run_kernel<S, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM + 16));
        CGL_CUDA(cudaFuncSetAttribute(env_run_kernel<S, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      C::SMEM + 16));
    }
    if (obs != nullptr) launch_env_run_as<S, true, true>(a, tr, obs, st);
    else if (traced) launch_env_run_as<S, true, false>(a, tr, obs, st);
    else launch_env_run_as<S, false, false>(a, tr, obs, st);
    CGL_LAUNCH_CHECK();
    return 0;
}

// CYC runs take the bit-sliced kernel at every step count: the byte kernel has no CYC instantiation.
template <int S, bool TR>
static void launch_env_run_cycle_as(const cgl_env_run_args_t &a, const RunTrace &tr, uint32_t max_period,
                                    int32_t *period_out, cudaStream_t st)
{
    using D = SlicedCfg<S>;
    const unsigned grid = (unsigned)((a.n_envs + D::EPC - 1) / D::EPC);
    const size_t smem = D::SMEM + 32 + (size_t)D::EPC * max_period * D::WPE * 4;     // TR slots, cyc slots, ring
#define CGL_RUN_SLICED(RULE)                                                                                          \
    env_run_sliced_kernel<S, RULE, TR, true><<<grid, D::THREADS, smem, st>>>(                                          \
        a.world_in_dev, a.world_out_dev, a.stable_dev, (uint32_t)a.n_envs, a.max_steps, 0, a.spawn, a.stable_max,      \
        a.empty_min, a.steps_out_dev, a.reward_out_dev, a.alive_out_dev, a.empty, tr, max_period, period_out)
    if (a.dead_rule == CGL_DEAD_DECAY) CGL_RUN_SLICED(CGL_DEAD_DECAY);
    else if (a.dead_rule == CGL_DEAD_SAT) CGL_RUN_SLICED(CGL_DEAD_SAT);
    else CGL_RUN_SLICED(CGL_DEAD_ZERO);
#undef CGL_RUN_SLICED
}

template <int S>
static int launch_env_run_cycle(const cgl_env_run_args_t &a, bool traced, const RunTrace &tr, uint32_t max_period,
                                int32_t *period_out, cudaStream_t st)
{
    using D = SlicedCfg<S>;
    constexpr size_t smem_max = D::SMEM + 32 + (size_t)D::EPC * CGL_RUN_MAX_PERIOD * D::WPE * 4;
    static PerDeviceOnce once;
    if (smem_max > 48 * 1024 && once.first()) {       // 256^2 at max_period 8: 96 KB
#define CGL_OPT_IN(RULE, TR) \
    CGL_CUDA(cudaFuncSetAttribute(env_run_sliced_kernel<S, RULE, TR, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max))
        CGL_OPT_IN(CGL_DEAD_ZERO, false); CGL_OPT_IN(CGL_DEAD_DECAY, false); CGL_OPT_IN(CGL_DEAD_SAT, false);
        CGL_OPT_IN(CGL_DEAD_ZERO, true); CGL_OPT_IN(CGL_DEAD_DECAY, true); CGL_OPT_IN(CGL_DEAD_SAT, true);
#undef CGL_OPT_IN
    }
    if (traced) launch_env_run_cycle_as<S, true>(a, tr, max_period, period_out, st);
    else launch_env_run_cycle_as<S, false>(a, tr, max_period, period_out, st);
    CGL_LAUNCH_CHECK();
    return 0;
}

// Shared memory of the generic kernel: three byte planes, and for CYC runs max_period bit-vector worlds after them.
static uint64_t generic_smem(uint32_t side, uint32_t max_period)
{
    const uint64_t size = (uint64_t)side * side;
    return max_period == 0 ? 3 * size : ((3 * size + 3) & ~3ull) + (uint64_t)max_period * 4 * ((size + 31) / 32);
}

// Settle runs on the fused sides: the finder, then phase C on the bit-sliced kernel at every step count (CGL_RUN_IMPL
// does not apply).  Both kernels read the untouched inputs; only phase C writes.
template <int S, bool TR>
static void launch_env_run_settle_as(const cgl_env_run_args_t &a, const RunTrace &tr, cudaStream_t st)
{
    using D = SlicedCfg<S>;
    const unsigned grid = (unsigned)((a.n_envs + D::EPC - 1) / D::EPC);
    constexpr int smem = D::SMEM + (TR ? 16 : 0);                 // TR: the step sums' slots
#define CGL_RUN_SLICED(RULE)                                                                                          \
    env_run_sliced_kernel<S, RULE, TR, false, true><<<grid, D::THREADS, smem, st>>>(                                   \
        a.world_in_dev, a.world_out_dev, a.stable_dev, (uint32_t)a.n_envs, a.max_steps, 0, a.spawn, a.stable_max,      \
        a.empty_min, a.steps_out_dev, a.reward_out_dev, a.alive_out_dev, a.empty, tr, 0u, nullptr)
    if (a.dead_rule == CGL_DEAD_DECAY) CGL_RUN_SLICED(CGL_DEAD_DECAY);
    else if (a.dead_rule == CGL_DEAD_SAT) CGL_RUN_SLICED(CGL_DEAD_SAT);
    else CGL_RUN_SLICED(CGL_DEAD_ZERO);
#undef CGL_RUN_SLICED
}

template <int S>
static int launch_env_run_settle(const cgl_env_run_args_t &a, bool traced, const RunTrace &tr, int32_t *period_out,
                                 cudaStream_t st)
{
    using D = SlicedCfg<S>;
    const unsigned grid = (unsigned)((a.n_envs + D::EPC - 1) / D::EPC);
    env_settle_find_kernel<S><<<grid, D::THREADS, D::EPC * 4 * D::WPE * 4, st>>>(
        a.world_in_dev, (uint32_t)a.n_envs, a.max_steps, a.steps_out_dev, period_out);
    if (traced) launch_env_run_settle_as<S, true>(a, tr, st);
    else launch_env_run_settle_as<S, false>(a, tr, st);
    CGL_LAUNCH_CHECK();
    return 0;
}

// Settle runs on the other sides: the generic finder, then phase C on the generic kernel.
static int launch_env_run_settle_generic(const cgl_env_run_args_t &a, bool traced, const RunTrace &tr,
                                         int32_t *period_out, cudaStream_t st)
{
    static PerDeviceOnce once;
    if (once.first()) {
        CGL_CUDA(cudaFuncSetAttribute(env_run_generic_kernel<false, false, false, true>,
                                      cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
        CGL_CUDA(cudaFuncSetAttribute(env_run_generic_kernel<true, false, false, true>,
                                      cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
    }
    const uint32_t W = cgl_words_per_row(a.side);
    env_settle_find_generic_kernel<<<(unsigned)a.n_envs, 256, settle_find_smem(a.side), st>>>(
        a.world_in_dev, a.side, W, a.max_steps, a.steps_out_dev, period_out);
#define CGL_RUN_GENERIC(TR)                                                                                            \
    env_run_generic_kernel<TR, false, false, true><<<(unsigned)a.n_envs, 256, generic_smem(a.side, 0), st>>>(         \
        a.world_in_dev, a.world_out_dev, a.stable_dev, a.side, W, a.max_steps, 0, (int8_t)a.spawn,                     \
        (int8_t)a.stable_max, a.steps_out_dev, a.reward_out_dev, a.alive_out_dev, a.dead_rule, (int8_t)a.empty,        \
        (int8_t)a.empty_min, tr, nullptr, 0u, nullptr)
    if (traced) CGL_RUN_GENERIC(true);
    else CGL_RUN_GENERIC(false);
#undef CGL_RUN_GENERIC
    CGL_LAUNCH_CHECK();
    return 0;
}

// Value counts of int8 planes: hist[e][v + 128] = #{i : stable[e][i] == v}.  One CTA per env; equal
// values inside a warp are merged with MATCH before the shared-memory atomic (planes hold few values).
__global__ void __launch_bounds__(256)
breakdown_kernel(const int8_t *__restrict__ stable, uint64_t size, uint32_t *__restrict__ hist_out)
{
    __shared__ uint32_t hist[256];
    hist[threadIdx.x] = 0;
    __syncthreads();
    const int8_t *s = stable + (uint64_t)blockIdx.x * size;
    const uint64_t padded = (size + blockDim.x - 1) / blockDim.x * blockDim.x;
    for (uint64_t i = threadIdx.x; i < padded; i += blockDim.x) {
        const bool in = i < size;
        const uint32_t v = in ? (uint32_t)(s[i] + 128) : 256u;
        const uint32_t peers = __match_any_sync(0xffffffffu, v);
        if (in && (threadIdx.x & 31) == (uint32_t)(__ffs(peers) - 1)) atomicAdd(&hist[v], __popc(peers));
    }
    __syncthreads();
    hist_out[(uint64_t)blockIdx.x * 256 + threadIdx.x] = hist[threadIdx.x];
}

}  // namespace cgl

using namespace cgl;

// Do the byte ranges [p, p + np) and [q, q + nq) share a byte?  (Lengths up to 2^96: no wrap-around.)
static bool ranges_overlap(const void *p, unsigned __int128 np, const void *q, unsigned __int128 nq)
{
    if (p == nullptr || q == nullptr || np == 0 || nq == 0) return false;
    const unsigned __int128 a = (uintptr_t)p, b = (uintptr_t)q;
    return a < b + nq && b < a + np;
}

// The argument checks of cgl_env_run_obs (obs may be NULL) and cgl_env_run_cycle: 0 or CGL_E_BADARG.
static int check_env_run_args(const cgl_env_run_args_t &a, const int8_t *obs)
{
    CGL_REQUIRE(a.world_in_dev && a.world_out_dev && a.stable_dev && a.n_envs && a.side, CGL_E_BADARG,
                "cgl_env_run: bad argument");
    CGL_REQUIRE(a.n_envs < (1ull << 31), CGL_E_BADARG, "cgl_env_run: n_envs too large");
    CGL_REQUIRE(a.dead_rule >= CGL_DEAD_ZERO && a.dead_rule <= CGL_DEAD_SAT && a.empty >= -128 && a.empty <= 127 &&
                    a.empty_min >= -128 && a.empty_min <= 127,
                CGL_E_BADARG, "cgl_env_run_rule: dead_rule must be 0..2, empty / empty_min must fit int8");
    CGL_REQUIRE(a.masked_toggle == 0 || a.masked_toggle == 1, CGL_E_BADARG, "cgl_env_run_ex: masked_toggle must be 0 or 1");
    CGL_REQUIRE(!(a.stop_when_fixed && a.actions_dev), CGL_E_BADARG,
                "cgl_env_run_ex: stop_when_fixed cannot take an action schedule (a fixed point is not defined under actions)");
    const void *bufs[3] = {a.actions_dev, a.reward_trace_dev, a.alive_trace_dev};
    for (int i = 0; i < 3; ++i)
        for (int k = i + 1; k < 3; ++k)
            CGL_REQUIRE(bufs[i] == nullptr || bufs[i] != bufs[k], CGL_E_BADARG,
                        "cgl_env_run_ex: the action schedule and the traces must be separate buffers");
    if (obs != nullptr) {
        CGL_REQUIRE(!a.stop_when_fixed, CGL_E_BADARG,
                    "cgl_env_run_obs: stop_when_fixed cannot take an obs trace (its rows would end at different steps)");
        CGL_REQUIRE(a.side <= 274, CGL_E_BADARG,
                    "cgl_env_run: side must be a fused side or small enough for shared memory (side <= 274)");
        const uint64_t size = (uint64_t)a.side * a.side;
        const unsigned __int128 rows = (unsigned __int128)a.max_steps * a.n_envs;
        const unsigned __int128 obs_bytes = rows * size;
        const unsigned __int128 plane = (unsigned __int128)a.n_envs * size;
        const unsigned __int128 world = (unsigned __int128)a.n_envs * a.side * cgl_words_per_row(a.side) * 4;
        const std::pair<const void *, unsigned __int128> other[6] = {
            {a.stable_dev, plane}, {a.actions_dev, rows * 4}, {a.reward_trace_dev, rows * 4},
            {a.alive_trace_dev, rows * 4}, {a.world_in_dev, world}, {a.world_out_dev, world}};
        for (const auto &o : other)
            CGL_REQUIRE(!ranges_overlap(obs, obs_bytes, o.first, o.second), CGL_E_BADARG,
                        "cgl_env_run_obs: the obs trace overlaps the stability plane, a world, the action schedule or a "
                        "trace");
        CGL_REQUIRE(!cgl_env_step_is_fused(a.side) || ((uintptr_t)obs & 15) == 0, CGL_E_BADARG,
                    "cgl_env_run_obs: the obs trace must be 16-byte aligned on the fused sides");
    }
    CGL_REQUIRE(cgl_env_step_is_fused(a.side) || generic_smem(a.side, 0) <= 220 * 1024, CGL_E_BADARG,
                "cgl_env_run: side must be a fused side or small enough for shared memory (side <= 274)");
    return 0;
}

// The one implementation behind cgl_env_run_ex, cgl_env_run and cgl_env_run_rule (see include/cgl_b200.h).
extern "C" int cgl_env_run_obs(const cgl_env_run_obs_args_t *args, cgl_stream_t stream)
{
    CGL_REQUIRE(args, CGL_E_BADARG, "cgl_env_run_obs: null");
    const cgl_env_run_args_t &a = args->run;
    int8_t *const obs = args->obs_trace_dev;
    if (const int rc = check_env_run_args(a, obs)) return rc;
    const bool traced = a.actions_dev || a.reward_trace_dev || a.alive_trace_dev || obs;
    const RunTrace tr = {a.actions_dev, a.reward_trace_dev, a.alive_trace_dev, a.err_flag_dev, a.masked_toggle};
    cudaStream_t st = as_stream(stream);
    if (cgl_env_step_is_fused(a.side)) {
#define CGL_CASE(S) \
    case S: return launch_env_run<S>(a, traced, tr, obs, st)
        switch (a.side) {
            CGL_CASE(32); CGL_CASE(64); CGL_CASE(96); CGL_CASE(128);
            CGL_CASE(160); CGL_CASE(192); CGL_CASE(224); CGL_CASE(256);
        }
#undef CGL_CASE
    }
    const size_t smem = generic_smem(a.side, 0);
    static PerDeviceOnce once;                   // opt in to the largest size once per device
    if (once.first()) {
        CGL_CUDA(cudaFuncSetAttribute(env_run_generic_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
        CGL_CUDA(cudaFuncSetAttribute(env_run_generic_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
        CGL_CUDA(cudaFuncSetAttribute(env_run_generic_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      220 * 1024));
    }
#define CGL_RUN_GENERIC(TR, OBS)                                                                                       \
    env_run_generic_kernel<TR, OBS><<<(unsigned)a.n_envs, 256, smem, st>>>(                                            \
        a.world_in_dev, a.world_out_dev, a.stable_dev, a.side, cgl_words_per_row(a.side), a.max_steps,                \
        a.stop_when_fixed, (int8_t)a.spawn, (int8_t)a.stable_max, a.steps_out_dev, a.reward_out_dev, a.alive_out_dev, \
        a.dead_rule, (int8_t)a.empty, (int8_t)a.empty_min, tr, obs, 0u, nullptr)
    if (obs != nullptr) CGL_RUN_GENERIC(true, true);
    else if (traced) CGL_RUN_GENERIC(true, false);
    else CGL_RUN_GENERIC(false, false);
#undef CGL_RUN_GENERIC
    CGL_LAUNCH_CHECK();
    return 0;
}

extern "C" int cgl_env_run_cycle(const cgl_env_run_args_t *args, uint32_t max_period, int32_t *period_out,
                                 cgl_stream_t stream)
{
    CGL_REQUIRE(args, CGL_E_BADARG, "cgl_env_run_cycle: null");
    const cgl_env_run_args_t &a = *args;
    if (const int rc = check_env_run_args(a, nullptr)) return rc;
    CGL_REQUIRE(!a.stop_when_fixed, CGL_E_BADARG, "cgl_env_run_cycle: stop_when_fixed must be 0 (max_period replaces it)");
    CGL_REQUIRE(!a.actions_dev, CGL_E_BADARG,
                "cgl_env_run_cycle: no action schedule (a cycle is not defined under actions)");
    CGL_REQUIRE(max_period >= 1 && max_period <= CGL_RUN_MAX_PERIOD, CGL_E_BADARG,
                "cgl_env_run_cycle: max_period must be in 1..%d", CGL_RUN_MAX_PERIOD);
    const bool traced = a.reward_trace_dev || a.alive_trace_dev;
    const RunTrace tr = {nullptr, a.reward_trace_dev, a.alive_trace_dev, a.err_flag_dev, a.masked_toggle};
    cudaStream_t st = as_stream(stream);
    if (cgl_env_step_is_fused(a.side)) {
#define CGL_CASE(S) \
    case S: return launch_env_run_cycle<S>(a, traced, tr, max_period, period_out, st)
        switch (a.side) {
            CGL_CASE(32); CGL_CASE(64); CGL_CASE(96); CGL_CASE(128);
            CGL_CASE(160); CGL_CASE(192); CGL_CASE(224); CGL_CASE(256);
        }
#undef CGL_CASE
    }
    const uint64_t smem = generic_smem(a.side, max_period);
    CGL_REQUIRE(smem <= 220 * 1024, CGL_E_BADARG,
                "cgl_env_run_cycle: a side that is not fused needs 3*side^2 + max_period*4*ceil(side^2/32) bytes <= "
                "220 KiB of shared memory (side <= 268 at max_period 1, <= 237 at 8); side %u at max_period %u needs %llu",
                a.side, max_period, (unsigned long long)smem);
    static PerDeviceOnce once;
    if (once.first()) {
        CGL_CUDA(cudaFuncSetAttribute(env_run_generic_kernel<false, false, true>,
                                      cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
        CGL_CUDA(cudaFuncSetAttribute(env_run_generic_kernel<true, false, true>,
                                      cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
    }
#define CGL_RUN_GENERIC(TR)                                                                                            \
    env_run_generic_kernel<TR, false, true><<<(unsigned)a.n_envs, 256, smem, st>>>(                                    \
        a.world_in_dev, a.world_out_dev, a.stable_dev, a.side, cgl_words_per_row(a.side), a.max_steps, 0,             \
        (int8_t)a.spawn, (int8_t)a.stable_max, a.steps_out_dev, a.reward_out_dev, a.alive_out_dev, a.dead_rule,        \
        (int8_t)a.empty, (int8_t)a.empty_min, tr, nullptr, max_period, period_out)
    if (traced) CGL_RUN_GENERIC(true);
    else CGL_RUN_GENERIC(false);
#undef CGL_RUN_GENERIC
    CGL_LAUNCH_CHECK();
    return 0;
}

extern "C" int cgl_env_run_settle(const cgl_env_run_args_t *args, int32_t *period_out, cgl_stream_t stream)
{
    CGL_REQUIRE(args, CGL_E_BADARG, "cgl_env_run_settle: null");
    cgl_env_run_args_t a = *args;
    // the side bound of check_env_run_args is the settle bound too: phase C needs 3*side^2 bytes of shared memory,
    // the generic finder 16*ceil(side^2/32)
    if (const int rc = check_env_run_args(a, nullptr)) return rc;
    CGL_REQUIRE(!a.stop_when_fixed, CGL_E_BADARG,
                "cgl_env_run_settle: stop_when_fixed must be 0 (the first repeat of any period replaces it)");
    CGL_REQUIRE(!a.actions_dev, CGL_E_BADARG,
                "cgl_env_run_settle: no action schedule (a cycle is not defined under actions)");
    const bool traced = a.reward_trace_dev || a.alive_trace_dev;
    const RunTrace tr = {nullptr, a.reward_trace_dev, a.alive_trace_dev, a.err_flag_dev, a.masked_toggle};
    cudaStream_t st = as_stream(stream);
    void *scratch = nullptr;                     // the per-env step counts hand phase C its bounds
    if (a.steps_out_dev == nullptr) {
        CGL_CUDA(cudaMallocAsync(&scratch, (size_t)a.n_envs * sizeof(int32_t), st));
        a.steps_out_dev = static_cast<int32_t *>(scratch);
    }
    int rc = 0;
    if (cgl_env_step_is_fused(a.side)) {
#define CGL_CASE(S) \
    case S: rc = launch_env_run_settle<S>(a, traced, tr, period_out, st); break
        switch (a.side) {
            CGL_CASE(32); CGL_CASE(64); CGL_CASE(96); CGL_CASE(128);
            CGL_CASE(160); CGL_CASE(192); CGL_CASE(224); CGL_CASE(256);
        }
#undef CGL_CASE
    } else {
        rc = launch_env_run_settle_generic(a, traced, tr, period_out, st);
    }
    if (scratch != nullptr) CGL_CUDA(cudaFreeAsync(scratch, st));
    return rc;
}

extern "C" int cgl_env_run_ex(const cgl_env_run_args_t *args, cgl_stream_t stream)
{
    CGL_REQUIRE(args, CGL_E_BADARG, "cgl_env_run_ex: null");
    const cgl_env_run_obs_args_t o = {*args, nullptr};
    return cgl_env_run_obs(&o, stream);
}

extern "C" int cgl_env_run_rule(const uint32_t *win, uint32_t *wout, int8_t *stable, uint64_t n_envs, uint32_t side,
                                uint32_t max_steps, int stop_when_fixed, int spawn, int stable_max, int dead_rule,
                                int empty, int empty_min, int32_t *steps, int32_t *reward, uint32_t *alive,
                                cgl_stream_t stream)
{
    cgl_env_run_args_t a = {};
    a.world_in_dev = win; a.world_out_dev = wout; a.stable_dev = stable; a.n_envs = n_envs; a.side = side;
    a.max_steps = max_steps; a.stop_when_fixed = stop_when_fixed; a.spawn = spawn; a.stable_max = stable_max;
    a.dead_rule = dead_rule; a.empty = empty; a.empty_min = empty_min;
    a.steps_out_dev = steps; a.reward_out_dev = reward; a.alive_out_dev = alive;
    return cgl_env_run_ex(&a, stream);
}

extern "C" int cgl_env_run(const uint32_t *win, uint32_t *wout, int8_t *stable, uint64_t n_envs, uint32_t side,
                           uint32_t max_steps, int stop_when_fixed, int spawn, int stable_max, int32_t *steps,
                           int32_t *reward, uint32_t *alive, cgl_stream_t stream)
{
    return cgl_env_run_rule(win, wout, stable, n_envs, side, max_steps, stop_when_fixed, spawn, stable_max,
                            CGL_DEAD_ZERO, 0, 0, steps, reward, alive, stream);
}

extern "C" int cgl_breakdown_stable(const int8_t *stable, uint64_t n_envs, uint64_t size, uint32_t *hist_out,
                                    cgl_stream_t stream)
{
    CGL_REQUIRE(stable && n_envs && size && hist_out && n_envs < (1ull << 31), CGL_E_BADARG,
                "cgl_breakdown_stable: bad argument");
    breakdown_kernel<<<(unsigned)n_envs, 256, 0, as_stream(stream)>>>(stable, size, hist_out);
    CGL_LAUNCH_CHECK();
    return 0;
}
