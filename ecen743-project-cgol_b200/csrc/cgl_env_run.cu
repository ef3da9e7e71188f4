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
#include <stdlib.h>

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

template <int S>
__global__ void __launch_bounds__(RunCfg<S>::THREADS)
env_run_kernel(const uint32_t *world_in, uint32_t *world_out, int8_t *stable, uint32_t n_envs,
               uint32_t max_steps, int stop_when_fixed, uint32_t spawn4, uint32_t max4,
               int32_t *__restrict__ steps_out, int32_t *__restrict__ reward_out, uint32_t *__restrict__ alive_out,
               int rule, uint32_t min4, uint32_t empty4)
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

    const uint32_t e = blockIdx.x * C::EPC + g;
    const bool active = e < n_envs;

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
    while (!done) {
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
                    mix_nibbles(n & ~c, n & c, mx[2 * w], mx[2 * w + 1]);
                }
                sts_words<C::W>(nxt + r * C::W, nx);
                sts_words<2 * C::W>(mix + 2 * r * C::W, mx);
            }
        }
        const bool any_changed = env_vote(changed != 0);
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
            }
            sst[c] = make_uint4(s[0], s[1], s[2], s[3]);
        }
        uint32_t *tmp = cur; cur = nxt; nxt = tmp;
        ++steps;
        done = steps >= max_steps || (stop_when_fixed && !any_changed);
        env_sync();                                  // mix and the old plane are free again
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
            sp[j * C::TPE + t] = v;
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
template <int S, int RULE>
__global__ void __launch_bounds__(SlicedCfg<S>::THREADS)
env_run_sliced_kernel(const uint32_t *world_in, uint32_t *world_out, int8_t *stable, uint32_t n_envs,
                      uint32_t max_steps, int stop_when_fixed, int spawn, int stable_max, int empty_min,
                      int32_t *__restrict__ steps_out, int32_t *__restrict__ reward_out,
                      uint32_t *__restrict__ alive_out, int empty)
{
    constexpr bool DECAY = RULE == CGL_DEAD_DECAY, SAT = RULE == CGL_DEAD_SAT;
    using C = SlicedCfg<S>;
    extern __shared__ __align__(16) unsigned char smem_dyn[];
    const int g = threadIdx.x / C::TPE;
    const int t = threadIdx.x % C::TPE;
    uint32_t *hbuf = reinterpret_cast<uint32_t *>(smem_dyn) + g * (4 * C::WPE);     // [buffer][plane][row][w]
    int *red = reinterpret_cast<int *>(smem_dyn + C::EPC * (4 * C::WPE * 4)) + g * 2;
    const uint32_t e = blockIdx.x * C::EPC + g;
    const bool active = e < n_envs;

    uint32_t cw[C::RPB][C::W];                      // this thread's rows of the world
    uint32_t pl[C::RPB][C::W][8];                   // and their stability: 8 bit planes per word
    if (t == 0) { red[0] = 0; red[1] = 0; }
    if (active) {
        const uint32_t *wp = world_in + (size_t)e * C::WPE;
        const uint4 *sp = reinterpret_cast<const uint4 *>(stable + (size_t)e * C::SIZE);
#pragma unroll
        for (int j = 0; j < C::RPB; ++j) {
            lds_words<C::W>(wp + (t * C::RPB + j) * C::W, cw[j]);       // (plain loads: the helper is address-space agnostic)
#pragma unroll
            for (int w = 0; w < C::W; ++w) {
                const uint4 a = sp[((t * C::RPB + j) * S + w * 32) / 16];
                const uint4 b = sp[((t * C::RPB + j) * S + w * 32) / 16 + 1];
                const uint32_t by[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
                bytes_to_planes32(by, pl[j][w]);
                if constexpr (!SAT) add_const_sliced(pl[j][w], -spawn);     // spawn-relative planes (cgl_bits.cuh)
            }
        }
    }
    __syncthreads();
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
    if (active) {
        while (steps < max_steps) {
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
            uint32_t up0[C::W], up1[C::W], dn0[C::W], dn1[C::W];
            lds_words<C::W>(h0 + r_up * C::W, up0);
            lds_words<C::W>(h1 + r_up * C::W, up1);
            lds_words<C::W>(h0 + r_dn * C::W, dn0);
            lds_words<C::W>(h1 + r_dn * C::W, dn1);
            changed = 0;
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
                    cw[j][w] = n;
                }
            }
            ++steps;
            buf ^= 1u;                              // the next step writes the other buffer: no reader is overtaken
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
    }
    if (active && t == 0) {
        if (reward_out != nullptr) reward_out[e] = acc;
        if (alive_out != nullptr) alive_out[e] = pop;
        if (steps_out != nullptr) steps_out[e] = (int32_t)steps;
    }
}

// Any side whose three byte planes fit in 220 KiB of shared memory (side <= 274): one CTA per env, one byte per cell.
__global__ void __launch_bounds__(256)
env_run_generic_kernel(const uint32_t *world_in, uint32_t *world_out, int8_t *stable, uint32_t side, uint32_t W,
                       uint32_t max_steps, int stop_when_fixed, int8_t spawn, int8_t stable_max,
                       int32_t *__restrict__ steps_out, int32_t *__restrict__ reward_out,
                       uint32_t *__restrict__ alive_out, int rule, int8_t empty, int8_t empty_min)
{
    extern __shared__ __align__(16) unsigned char smem_dyn[];
    const uint32_t size = side * side;
    uint8_t *a = smem_dyn, *b = a + size;
    int8_t *st = reinterpret_cast<int8_t *>(b + size);
    __shared__ int red[2];
    const uint64_t e = blockIdx.x;
    const uint32_t *wi = world_in + e * side * W;
    uint32_t *wo = world_out + e * side * W;
    int8_t *sg = stable + e * size;
    if (threadIdx.x == 0) { red[0] = 0; red[1] = 0; }
    for (uint32_t i = threadIdx.x; i < size; i += blockDim.x) {
        const uint32_t y = i / side, x = i - y * side;
        a[i] = (wi[y * W + (x >> 5)] >> (x & 31)) & 1u;
        st[i] = sg[i];
    }
    __syncthreads();
    uint32_t steps = 0;
    bool done = max_steps == 0;
    while (!done) {
        int changed = 0;
        for (uint32_t i = threadIdx.x; i < size; i += blockDim.x) {
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
        }
        const bool any_changed = __syncthreads_or(changed) != 0;
        uint8_t *tmp = a; a = b; b = tmp;
        ++steps;
        done = steps >= max_steps || (stop_when_fixed && !any_changed);
    }
    int acc = 0;
    uint32_t pop = 0;
    for (uint32_t i = threadIdx.x; i < size; i += blockDim.x) {
        sg[i] = st[i];
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
    }
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

template <int S>
static int launch_env_run(const uint32_t *win, uint32_t *wout, int8_t *stable, uint64_t n_envs, uint32_t max_steps,
                          int stop, int spawn, int stable_max, int32_t *steps, int32_t *reward, uint32_t *alive,
                          cudaStream_t st, int rule, int empty, int empty_min)
{
    using C = RunCfg<S>;
    static PerDeviceOnce once;
    if (once.first())
        CGL_CUDA(cudaFuncSetAttribute(env_run_kernel<S>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM));
    const unsigned grid = (unsigned)((n_envs + C::EPC - 1) / C::EPC);
    if (run_use_sliced(max_steps)) {
        using D = SlicedCfg<S>;
#define CGL_RUN_SLICED(RULE)                                                                                          \
    env_run_sliced_kernel<S, RULE><<<grid, D::THREADS, D::SMEM, st>>>(win, wout, stable, (uint32_t)n_envs, max_steps, \
                                                                       stop, spawn, stable_max, empty_min, steps,      \
                                                                       reward, alive, empty)
        if (rule == CGL_DEAD_DECAY) CGL_RUN_SLICED(CGL_DEAD_DECAY);
        else if (rule == CGL_DEAD_SAT) CGL_RUN_SLICED(CGL_DEAD_SAT);
        else CGL_RUN_SLICED(CGL_DEAD_ZERO);
#undef CGL_RUN_SLICED
    } else {
        env_run_kernel<S><<<grid, C::THREADS, C::SMEM, st>>>(win, wout, stable, (uint32_t)n_envs, max_steps, stop,
                                                            rep4(spawn), rep4(stable_max), steps, reward, alive, rule,
                                                            rep4(empty_min), rep4(empty));
    }
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

extern "C" int cgl_env_run_rule(const uint32_t *win, uint32_t *wout, int8_t *stable, uint64_t n_envs, uint32_t side,
                                uint32_t max_steps, int stop_when_fixed, int spawn, int stable_max, int dead_rule,
                                int empty, int empty_min, int32_t *steps, int32_t *reward, uint32_t *alive,
                                cgl_stream_t stream)
{
    CGL_REQUIRE(win && wout && stable && n_envs && side, CGL_E_BADARG, "cgl_env_run: bad argument");
    CGL_REQUIRE(n_envs < (1ull << 31), CGL_E_BADARG, "cgl_env_run: n_envs too large");
    CGL_REQUIRE(dead_rule >= CGL_DEAD_ZERO && dead_rule <= CGL_DEAD_SAT && empty >= -128 && empty <= 127 &&
                    empty_min >= -128 && empty_min <= 127,
                CGL_E_BADARG, "cgl_env_run_rule: dead_rule must be 0..2, empty / empty_min must fit int8");
    cudaStream_t st = as_stream(stream);
    if (cgl_env_step_is_fused(side)) {
#define CGL_CASE(S)                                                                                       \
    case S:                                                                                               \
        return launch_env_run<S>(win, wout, stable, n_envs, max_steps, stop_when_fixed, spawn, stable_max, \
                                 steps, reward, alive, st, dead_rule, empty, empty_min)
        switch (side) {
            CGL_CASE(32); CGL_CASE(64); CGL_CASE(96); CGL_CASE(128);
            CGL_CASE(160); CGL_CASE(192); CGL_CASE(224); CGL_CASE(256);
        }
#undef CGL_CASE
    }
    const size_t smem = 3ull * side * side;
    CGL_REQUIRE(smem <= 220 * 1024, CGL_E_BADARG,
                "cgl_env_run: side must be a fused side or small enough for shared memory (side <= 274)");
    static PerDeviceOnce once;                   // opt in to the largest size once per device
    if (once.first())
        CGL_CUDA(cudaFuncSetAttribute(env_run_generic_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024));
    env_run_generic_kernel<<<(unsigned)n_envs, 256, smem, st>>>(win, wout, stable, side, cgl_words_per_row(side),
                                                               max_steps, stop_when_fixed, (int8_t)spawn,
                                                               (int8_t)stable_max, steps, reward, alive, dead_rule,
                                                               (int8_t)empty, (int8_t)empty_min);
    CGL_LAUNCH_CHECK();
    return 0;
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
