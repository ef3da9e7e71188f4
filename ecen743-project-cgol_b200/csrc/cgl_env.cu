// cgl_env.cu -- the env step (toggle -> generation -> int8 stability -> reward) for sm_100a.
//
// Reference semantics: kernel `run` /root/reference/CGL/CGL.py:147-181, its driver
// `__step_state_gpu` :203-208, toggle_state :322-328, reward :255-256, alive :259-260.
// Nothing here is translated from that kernel (one thread per byte cell, 10 byte loads, 4 integer
// modulos): state is 1 bit per cell + 1 int8 per cell, the generation is bit-sliced LOP3 logic on
// 32 cells per instruction, and the stability plane is streamed once with 128-bit accesses and
// updated 4 cells per instruction.
#include <stdlib.h>

#include "cgl_internal.cuh"

namespace cgl {

// =========================================================================================
// Fused fast path: side % 32 == 0, side <= 256.  One CTA handles EPC environments, TPE threads
// each.  HBM traffic per env: world 2 * side^2/8 B, stability 2 * side^2 B  (2.25 B / cell).
//
//   phase 0  the first batch of stability uint4 loads is issued (independent of the bits)
//   phase A  world words -> shared memory (uint4, coalesced), action bit flipped on the way
//   phase B  next generation from shared memory: a thread owns whole rows (vector LDS, in-register
//            horizontal neighbours, ~22 LOP3/SHF per 32 cells), vector store to HBM; (born,surv)
//            nibbles interleaved into one table-index byte per 4 cells
//   phase C  stability stream: LDG.128 -> 4 x {2 conflict-free mask LDS, byte-SIMD update, IDP.4A}
//            -> STG.128; reward reduced with REDUX + one shared atomic per warp
// =========================================================================================
template <int S>
struct EnvCfg {
    static constexpr int W = S / 32;              // words per row
    static constexpr int WPE = S * W;             // words per env
    static constexpr int SIZE = S * S;            // cells per env
    static constexpr int NCHUNK = SIZE / 16;      // 16-cell (uint4) stability chunks per env
    static constexpr int TPE = (S <= 64) ? 32 : S;          // threads per env
    static constexpr int EPC = (TPE >= 128) ? 1 : (128 / TPE);  // envs per CTA
    static constexpr int THREADS = TPE * EPC;
    static constexpr int CPT = NCHUNK / TPE;      // chunks per thread
    static constexpr int UNR = CPT < 8 ? CPT : 8; // chunks in flight per thread
    // [<= 4 KB align slack][mask tables 4 KB][per env: cur WPE*4 | mix WPE*8][per env: 4 ints]
    static constexpr int SMEM = 4096 + 4096 + EPC * (WPE * 4 + WPE * 8) + EPC * 16;
    static_assert(S % 32 == 0 && NCHUNK % TPE == 0 && WPE % 4 == 0, "unsupported side");
};

// N consecutive words (N*4-byte aligned base) with the widest vector accesses available.
template <int N>
__device__ __forceinline__ void load_words(const uint32_t *p, uint32_t (&x)[N])
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
__device__ __forceinline__ void store_words(uint32_t *p, const uint32_t (&x)[N])
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

__device__ __forceinline__ uint32_t lds_u32(uint32_t shared_addr)
{
    uint32_t v;
    asm("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(shared_addr));
    return v;
}

struct RuleArgs { int rule, empty, empty_min, masked; };

// nibble -> byte mask (bit i -> byte i = 0xFF), the 16 values of nibble_to_bytemask()
__constant__ uint32_t c_bytemask16[16] = {
    0x00000000u, 0x000000ffu, 0x0000ff00u, 0x0000ffffu, 0x00ff0000u, 0x00ff00ffu, 0x00ffff00u, 0x00ffffffu,
    0xff000000u, 0xff0000ffu, 0xff00ff00u, 0xff00ffffu, 0xffff0000u, 0xffff00ffu, 0xffffff00u, 0xffffffffu};

// Fill the lane-private mask tables: word (nib*64 + which*32 + lane) = mask(nib) [& SPAWN if which].  Every CTA does
// this once, so it is kept short: with a thread count that is a multiple of 64 a thread's `which` and its nibble
// sequence are fixed, and an entry is one constant-bank load (warp-uniform index), one AND and one store.
template <int THREADS>
__device__ __forceinline__ void fill_mask_tables(uint32_t *tables, uint32_t spawn4)
{
    if constexpr (THREADS % 64 == 0) {
        const uint32_t andm = (threadIdx.x & 32u) ? spawn4 : 0xffffffffu;
        const uint32_t nb0 = threadIdx.x >> 6;
#pragma unroll
        for (int k = 0; k < (1024 + THREADS - 1) / THREADS; ++k)
            if (k * THREADS + THREADS <= 1024 || threadIdx.x + k * THREADS < 1024)
                tables[threadIdx.x + k * THREADS] = c_bytemask16[nb0 + k * (THREADS / 64)] & andm;
    } else {
        for (int i = threadIdx.x; i < 1024; i += THREADS) {
            const uint32_t m = c_bytemask16[(uint32_t)i >> 6];
            tables[i] = (i & 32) ? (m & spawn4) : m;
        }
    }
}

// IO = false: the stability plane is updated in place.  IO = true: it is read from `stable` and the
// new values go to `stable_out` (another buffer of the same shape) -- the replay ring of the batched
// DQN loop hands the env its next observation slot, so "adding to the replay buffer" costs no copy.
// RULE >= 0: the CGL_action+ fork's variants (cgl_bits.cuh): the rule for cells that are dead after the step
// (CGL_DEAD_ZERO / DECAY / SAT; min4 / empty4 = EMPTY_MIN / EMPTY replicated) and `masked` toggles (a cell
// toggled to dead gets 0, not SPAWN: CGL_action+/CGL.py:382-384).  RULE = -1 is the base env and compiles to
// exactly the code it had before these parameters existed.  The rule is a template parameter on purpose: as a
// run-time switch inside the unrolled stability loop it tripled the branch count and cost ~15 %.
template <int S, bool IO, int RULE>
__global__ void __launch_bounds__(EnvCfg<S>::THREADS)
env_step_fused_kernel(const uint32_t *__restrict__ world_in, uint32_t *__restrict__ world_out,
                      int8_t *stable, int8_t *stable_out, uint32_t n_envs,
                      const int32_t *__restrict__ actions, uint32_t spawn4, uint32_t max4,
                      int32_t *__restrict__ reward_out, uint32_t *__restrict__ alive_out,
                      int *__restrict__ err_flag, uint32_t *__restrict__ epoch, uint32_t want, uint32_t publish,
                      uint32_t min4, uint32_t empty4, int masked, int seq_tokens)
{
    constexpr bool EXT = RULE >= 0;
    using C = EnvCfg<S>;
    extern __shared__ __align__(16) unsigned char smem_dyn[];
    // Mask tables, one copy per lane so that a lookup never bank-conflicts:
    //   word (nib*64 + which*32 + lane): which 0 = byte mask of `nib`, which 1 = that mask & SPAWN.
    // The table base is aligned to 4 KB so that a lookup address is ONE byte-permute:
    //   addr = TB | nib << 8 | which << 7 | lane << 2.
    const uint32_t sbase = (uint32_t)__cvta_generic_to_shared(smem_dyn);
    const uint32_t tb = (sbase + 4095u) & ~4095u;
    unsigned char *smem_raw = smem_dyn + (tb - sbase);
    uint32_t *tables = reinterpret_cast<uint32_t *>(smem_raw);
    const int g = threadIdx.x / C::TPE;           // env slot in this CTA
    const int t = threadIdx.x % C::TPE;
    uint32_t *cur = reinterpret_cast<uint32_t *>(smem_raw + 4096) + g * (C::WPE * 3);
    uint32_t *mix = cur + C::WPE;                 // 2 words per world word
    int *red = reinterpret_cast<int *>(smem_raw + 4096 + C::EPC * C::WPE * 12) + g * 4;   // reward, alive, token ok

    const uint32_t e = blockIdx.x * C::EPC + g;
    bool active = e < n_envs;

    // Programmatic dependent launch: the NEXT launch's CTAs may take the SM slots this grid frees in
    // its tail (hides the launch latency between back-to-back steps).  The stability loads stay the first
    // thing a CTA does after its wait -- a CTA's life is latency-bound, and the mask-table fill overlaps
    // with them.
    if (epoch == nullptr) {
        cudaTriggerProgrammaticLaunchCompletion();
        cudaGridDependencySynchronize();            // plain form: wait for the whole previous grid
    } else {
        // Chained steps: env e of this launch depends only on env e of the previous launch, which
        // published epoch[e] = want (the id of the plane this launch reads) when it was done.  The
        // next launch's first CTAs therefore start while the previous launch's last CTAs are still
        // running (ramp-up overlaps the tail); the spin almost never iterates because CTAs are
        // dispatched in env order.  The token load is issued first and the mask tables are filled in
        // its shadow.
        //
        // Token values.  seq_tokens: want / publish are consecutive per-env SEQUENCE NUMBERS (32 bits, compared
        // for equality): a token value then names exactly one launch, any number of launches may be in flight,
        // and the CTA triggers its dependents at entry.  Otherwise they are two PLANE IDS that alternate (a
        // captured CUDA graph replays, which baked-in sequence numbers cannot): two ids are enough ONLY IF a CTA
        // allows its dependents to launch once it has SEEN its token -- launch n+2 can then start only when
        // every CTA of launch n+1 has seen the token of launch n, i.e. when launch n has completely finished,
        // so at most two consecutive launches are in flight and an id cannot be mistaken for the same id two
        // launches back (with the trigger at entry and small batches three grids fit on the GPU at once: the
        // round-1 bug).  The trigger sits on the launch-to-launch critical path (the dependent grid fills the
        // slots this grid's last, partial wave leaves free; measured per C2 step: trigger behind the barrier
        // 26.5 us, decided per thread from a relaxed load of the token 25.7 us, at entry 24.9 us).  A CTA counts
        // as triggered as soon as ANY of its threads has executed the trigger (measured: letting the idle warps
        // of a partly filled CTA trigger early brings the hazard back), so in id mode CTAs that hold several
        // envs (side <= 64: one warp each) trigger behind the barrier that collects all their tokens.
        //
        // The wait is bounded (g_wait_ns, cgl_set_wait_timeout_ms).  A token that never arrives (caller bug,
        // a predecessor that was never launched) sets bit 1 of the error flag, raises the alarm word and
        // SKIPS the env: no plane is written and no token published, so nothing is computed from stale
        // planes and every later chained step of that env fails the same way (fast: see wait_expired).
        if (seq_tokens) cudaTriggerProgrammaticLaunchCompletion();
        uint32_t v = want, v_seen = want;
        if (C::EPC == 1 && active && !seq_tokens)
            asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v_seen) : "l"(epoch + e) : "memory");
        if (t == 0 && active) asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(epoch + e) : "memory");
        fill_mask_tables<C::THREADS>(tables, spawn4);
        const bool seen = seq_tokens || (C::EPC == 1 && v_seen == want);     // seen: already triggered
        if (seen && !seq_tokens) cudaTriggerProgrammaticLaunchCompletion();
        if (t == 0) {
            if (active && v != want) {
                const unsigned long long t0 = globaltimer_ns();
                uint32_t spins = 0;
                do {
                    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(epoch + e) : "memory");
                } while (v != want && ((++spins & 255u) != 0 || !wait_expired(t0, ALARM_ENV_TOKEN)));
                if (v != want) {
                    if (err_flag != nullptr) atomicOr(err_flag, 2);
                    raise_alarm(ALARM_ENV_TOKEN);
                }
            }
            red[2] = (v == want);
        }
        __syncthreads();
        if (!seen) cudaTriggerProgrammaticLaunchCompletion();
        active = active && red[2] != 0;
    }

    // ---- phase 0: stability loads in flight before anything else --------------------------
    uint4 *sp = reinterpret_cast<uint4 *>(stable + (size_t)e * C::SIZE);
    uint4 sreg[C::UNR];
    if (active) {
#pragma unroll
        for (int u = 0; u < C::UNR; ++u) sreg[u] = (sp + t)[u * C::TPE];
    }

    if (epoch == nullptr) fill_mask_tables<C::THREADS>(tables, spawn4);
    if (t == 0) { red[0] = 0; red[1] = 0; }

    // ---- action decode (toggle_state before step, CGL/main.py:66-67) ----------------------
    int act = -1;                                 // -1: nothing to toggle
    if (active && actions != nullptr) {
        int a = actions[e];
        if (a >= 0 && a < C::SIZE) act = a;
        else if (a != C::SIZE && t == 0) {
            if (err_flag != nullptr) atomicOr(err_flag, 1);
            raise_alarm(ALARM_BAD_ACTION);
        }
    }
    // cell index == bit index because a row is exactly W full words
    const int act_word = act >> 5;
    const uint32_t act_bit = 1u << (act & 31);

    // ---- phase A: world -> smem ------------------------------------------------------------
    if (active) {
        const uint4 *wp = reinterpret_cast<const uint4 *>(world_in + (size_t)e * C::WPE);
        for (int i = t; i < C::WPE / 4; i += C::TPE) {
            uint4 v = __ldg(wp + i);
            if (act >= 0 && (act_word >> 2) == i) {
                int k = act_word & 3;
                if (k == 0) v.x ^= act_bit; else if (k == 1) v.y ^= act_bit;
                else if (k == 2) v.z ^= act_bit; else v.w ^= act_bit;
            }
            reinterpret_cast<uint4 *>(cur)[i] = v;
        }
    }
    __syncthreads();

    // ---- phase B: next generation ------------------------------------------------------------
    // A thread owns RPB consecutive rows at full width (W words): vector LDS of whole rows,
    // horizontal neighbours (incl. the torus wrap) stay in registers, one vector store per row.
    uint32_t pop = 0;
    if (active) {
        uint32_t *wo = world_out + (size_t)e * C::WPE;
        constexpr int RPB = S / C::TPE;            // rows per thread (1 or 2)
        HSum hs[RPB + 2][C::W];
        uint32_t cw[RPB + 2][C::W];
#pragma unroll
        for (int j = 0; j < RPB + 2; ++j) {
            int r = t * RPB + j - 1;
            r = r < 0 ? S - 1 : (r >= S ? 0 : r);
            load_words<C::W>(cur + r * C::W, cw[j]);
#pragma unroll
            for (int w = 0; w < C::W; ++w)
                hs[j][w] = hsum(west_plane(cw[j][(w + C::W - 1) % C::W], cw[j][w]), cw[j][w],
                                east_plane(cw[j][w], cw[j][(w + 1) % C::W]));
        }
#pragma unroll
        for (int j = 0; j < RPB; ++j) {
            const int r = t * RPB + j;
            uint32_t nx[C::W], mx[2 * C::W];
#pragma unroll
            for (int w = 0; w < C::W; ++w) {
                const uint32_t c = cw[j + 1][w];
                const uint32_t nxt = life_rule(hs[j][w], hs[j + 1][w], hs[j + 2][w], c);
                nx[w] = nxt;
                pop += __popc(nxt);
                // byte per 4 cells: born nibble << 4 | surv nibble
                mix_nibbles(nxt & ~c, nxt & c, mx[2 * w], mx[2 * w + 1]);
            }
            store_words<C::W>(wo + r * C::W, nx);
            store_words<2 * C::W>(mix + 2 * r * C::W, mx);
        }
    }
    __syncthreads();

    // ---- phase C: stability stream + reward -------------------------------------------------
    int acc = 0;
    if (active) {
        // stable[action] = spawn before the update (CGL.py:326): chunk act>>4 is chunk number
        // act_u of thread act_t -- an env-uniform test per chunk, the patch itself runs once.
        const int act_u = act >= 0 ? (act >> 4) / C::TPE : -1;
        const int act_t = (act >> 4) % C::TPE;
        const int act_sub = (act >> 2) & 3;
        const uint32_t act_mask = 0xffu << ((act & 3) * 8);
        const uint32_t tbn = ((tb >> 8) & 0xffu) * 0x01010101u;   // table-base byte under every nibble
        const uint32_t lane_s = (threadIdx.x & 31) * 4, lane_b = lane_s + 128;
        uint4 *spt = sp + t;                          // this thread's chunks: spt[u * TPE] (immediate offsets)
        uint4 *spo = IO ? reinterpret_cast<uint4 *>(stable_out + (size_t)e * C::SIZE) + t : spt;
        const uint32_t *mixt = mix + t;
        uint32_t put = spawn4 & act_mask;
        if constexpr (EXT) {
            // masked toggle: the cell's state AFTER the toggle decides (cur holds the toggled plane)
            if (masked && act >= 0 && !((cur[act_word] >> (act & 31)) & 1u)) put = 0u;
        }
        const uint32_t keep = ~act_mask;
        // the thread that owns the action's chunk patches it once, outside the unrolled chunk loop
        auto patch = [&](uint4 &v) {
            if (act_sub == 0) v.x = (v.x & keep) | put;
            else if (act_sub == 1) v.y = (v.y & keep) | put;
            else if (act_sub == 2) v.z = (v.z & keep) | put;
            else v.w = (v.w & keep) | put;
        };
        if (t == act_t && act_u >= 0 && act_u < C::UNR) {
#pragma unroll
            for (int u = 0; u < C::UNR; ++u)
                if (act_u == u) patch(sreg[u]);
        }
#pragma unroll
        for (int b0 = 0; b0 < C::CPT; b0 += C::UNR) {
            if (b0 > 0) {
#pragma unroll
                for (int u = 0; u < C::UNR; ++u)
                    if (b0 + u < C::CPT) {
                        sreg[u] = spt[(b0 + u) * C::TPE];
                        if (act_u == b0 + u && t == act_t) patch(sreg[u]);
                    }
            }
#pragma unroll
            for (int u = 0; u < C::UNR; ++u) {
                if (b0 + u >= C::CPT) continue;
                uint32_t s[4] = {sreg[u].x, sreg[u].y, sreg[u].z, sreg[u].w};
                const uint32_t m = mixt[(b0 + u) * C::TPE];
                const uint32_t sv = (m & 0x0f0f0f0fu) | tbn;
                const uint32_t bn = ((m >> 4) & 0x0f0f0f0fu) | tbn;
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    // address bytes: [lane*4 (+128 for the born table), TBhi | nibble, 0, 0]
                    const uint32_t surv_mask = lds_u32(__byte_perm(sv, lane_s, 0x5504 + 16 * k));
                    if constexpr (EXT) {
                        const uint32_t born_mask = lds_u32(__byte_perm(bn, lane_s, 0x5504 + 16 * k));
                        s[k] = stable_update4_rule(RULE, s[k], surv_mask, born_mask, spawn4, max4, min4, empty4);
                    } else {
                        const uint32_t born_spawn = lds_u32(__byte_perm(bn, lane_b, 0x5504 + 16 * k));
                        s[k] = stable_update4(s[k], surv_mask, born_spawn, max4);
                    }
                    acc = __dp4a((int)s[k], 0x01010101, acc);
                }
                spo[(b0 + u) * C::TPE] = make_uint4(s[0], s[1], s[2], s[3]);
            }
        }
    }
    // ---- reward / alive, then the token --------------------------------------------------------
    // Order matters: the env's thread 0 stores reward and alive BEFORE it publishes the token, so the next
    // launch's CTA of this env (which may already be spinning on it) can never be overtaken by these stores.
    const bool want_red = reward_out != nullptr || alive_out != nullptr;
    if (want_red) {
        acc = __reduce_add_sync(0xffffffffu, acc);
        pop = __reduce_add_sync(0xffffffffu, pop);
        if ((threadIdx.x & 31) == 0) {
            atomicAdd(&red[0], acc);
            atomicAdd(reinterpret_cast<unsigned *>(&red[1]), pop);
        }
    }
    if (want_red || epoch != nullptr) __syncthreads();      // all stores of this env issued, sums complete
    if (active && t == 0) {
        if (reward_out != nullptr) reward_out[e] = red[0];
        if (alive_out != nullptr) alive_out[e] = (uint32_t)red[1];
        // ONE release store: release is cumulative over what the barrier ordered before it (the grid-sync idiom)
        if (epoch != nullptr) asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(epoch + e), "r"(publish) : "memory");
    }
}

CGL_DEFINE_TU_HOOKS(env)

// CGL_ENV_PDL=0 turns programmatic dependent launch off (tuning / debugging); cgl_rollout.cu suppresses it while
// it captures its copy -> step graphs.
int g_pdl_suppress = 0;
static bool pdl_enabled()
{
    static int v = -1;
    if (v < 0) {
        const char *e = getenv("CGL_ENV_PDL");
        v = (e && e[0] == '0') ? 0 : 1;
    }
    return v != 0 && !g_pdl_suppress;
}

// CGL_ENV_BYTES=0 sends the sides the fused kernel does not take through the three generic kernels again (tests
// force both paths; tuning).
static bool env_bytes_enabled()
{
    static int v = -1;
    if (v < 0) {
        const char *e = getenv("CGL_ENV_BYTES");
        v = (e && e[0] == '0') ? 0 : 1;
    }
    return v != 0;
}

// Sides the one-launch byte-plane kernel (env_step_bytes_kernel, below) takes.  CGL_ENV_BYTES=2 forces it for every
// side up to 256 (tests).
static bool env_bytes_takes(uint32_t side)
{
    if (!env_bytes_enabled() || side > 256) return false;
    static int force = -1;
    if (force < 0) {
        const char *e = getenv("CGL_ENV_BYTES");
        force = (e && e[0] == '2') ? 1 : 0;
    }
    return force || side >= 32;
}

template <int S>
static int launch_env_fused(const cgl_env_step_args_t &a, cudaStream_t st)
{
    using C = EnvCfg<S>;
    const unsigned grid = (unsigned)((a.n_envs + C::EPC - 1) / C::EPC);
    static int pad = -1;                        // tuning knob: extra dynamic smem limits CTAs/SM
    static PerDeviceOnce once;
    if (pad < 0) {
        const char *v = getenv("CGL_ENV_SMEM_PAD");
        pad = v ? atoi(v) : 0;
    }
    if (once.first()) {
        CGL_CUDA(cudaFuncSetAttribute(env_step_fused_kernel<S, false, -1>,
                                      cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM + pad));
        CGL_CUDA(cudaFuncSetAttribute(env_step_fused_kernel<S, true, -1>,
                                      cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM + pad));
        CGL_CUDA(cudaFuncSetAttribute(env_step_fused_kernel<S, true, CGL_DEAD_ZERO>,
                                      cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM + pad));
        CGL_CUDA(cudaFuncSetAttribute(env_step_fused_kernel<S, true, CGL_DEAD_DECAY>,
                                      cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM + pad));
        CGL_CUDA(cudaFuncSetAttribute(env_step_fused_kernel<S, true, CGL_DEAD_SAT>,
                                      cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM + pad));
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid);
    cfg.blockDim = dim3(C::THREADS);
    cfg.dynamicSmemBytes = C::SMEM + pad;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl_enabled() ? 1 : 0;
    const uint32_t n32 = (uint32_t)a.n_envs, sp4 = rep4(a.spawn), mx4 = rep4(a.stable_max);
    const uint32_t mn4 = rep4(a.empty_min), em4 = rep4(a.empty);
    const uint32_t *win = a.world_in_dev;
    uint32_t *wout = a.world_out_dev;
    int8_t *sin = const_cast<int8_t *>(a.stable_in_dev), *sout = a.stable_out_dev;
    uint32_t *tok = a.chain_mode != CGL_CHAIN_NONE ? a.token_dev : nullptr;
    const int seq = a.chain_mode == CGL_CHAIN_SEQ, masked = a.masked_toggle != 0;
#define CGL_LAUNCH(IO, RULE)                                                                                        \
    CGL_CUDA(cudaLaunchKernelEx(&cfg, env_step_fused_kernel<S, IO, RULE>, win, wout, sin, sout, n32, a.actions_dev, \
                                sp4, mx4, a.reward_out_dev, a.alive_out_dev, a.err_flag_dev, tok, a.want, a.publish, \
                                mn4, em4, masked, seq))
    if (a.dead_rule != CGL_DEAD_ZERO || masked) {   // fork variants: one kernel per rule, in/out planes may alias
        if (a.dead_rule == CGL_DEAD_DECAY) CGL_LAUNCH(true, CGL_DEAD_DECAY);
        else if (a.dead_rule == CGL_DEAD_SAT) CGL_LAUNCH(true, CGL_DEAD_SAT);
        else CGL_LAUNCH(true, CGL_DEAD_ZERO);
    } else if (sout != sin) {
        CGL_LAUNCH(true, -1);
    } else {
        CGL_LAUNCH(false, -1);
    }
#undef CGL_LAUNCH
    return 0;
}

// =========================================================================================
// Generic path: any side >= 1, any batch.  Three small kernels (toggle, generation, stability).
// =========================================================================================

// One thread per env; indices of one env are handled sequentially so that a duplicated index
// toggles once (numpy gather-then-scatter, CGL/CGL.py:325).
__global__ void toggle_kernel(uint32_t *__restrict__ world, int8_t *__restrict__ stable,
                              uint64_t n_envs, uint32_t side, uint32_t W,
                              const int32_t *__restrict__ idx, uint32_t k, int8_t spawn,
                              int *__restrict__ err_flag, int masked)
{
    const uint64_t size = (uint64_t)side * side;
    for (uint64_t e = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; e < n_envs;
         e += (uint64_t)gridDim.x * blockDim.x) {
        const int32_t *my = idx + e * k;
        for (uint32_t j = 0; j < k; ++j) {
            const int64_t a = my[j];
            if (a < 0 || (uint64_t)a > size) {
                if (err_flag != nullptr) atomicOr(err_flag, 1);
                raise_alarm(ALARM_BAD_ACTION);
                continue;
            }
            if ((uint64_t)a == size) continue;               // "do nothing" action
            bool dup = false;
            for (uint32_t j2 = 0; j2 < j; ++j2) dup |= (my[j2] == my[j]);
            if (dup) continue;
            const uint32_t r = (uint32_t)((uint64_t)a / side), c = (uint32_t)((uint64_t)a % side);
            const uint32_t word = world[(e * side + r) * W + (c >> 5)] ^ (1u << (c & 31));
            world[(e * side + r) * W + (c >> 5)] = word;
            // base env: SPAWN even when toggled to dead (N2); fork: SPAWN * new state (CGL_action+/CGL.py:382-384)
            stable[e * size + a] = (masked && !((word >> (c & 31)) & 1u)) ? (int8_t)0 : spawn;
        }
    }
}

// One thread per packed word.  wrap_rows: torus rows (reference) or dead rows outside (bands).
__global__ void life_generic_kernel(const uint32_t *__restrict__ in, uint32_t *__restrict__ out,
                                    uint64_t n_envs, uint32_t rows, uint32_t cols, uint32_t W,
                                    int wrap_rows, uint32_t *__restrict__ alive_out)
{
    const uint64_t wpe = (uint64_t)rows * W;
    const uint64_t total = n_envs * wpe;
    const uint32_t rbits = cols - 32 * (W - 1);
    const uint32_t last_mask = rbits == 32 ? 0xffffffffu : ((1u << rbits) - 1u);
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < total;
         i += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t e = i / wpe;
        const uint32_t rem = (uint32_t)(i - e * wpe);
        const uint32_t r = rem / W, w = rem - r * W;
        const uint32_t *base = in + e * wpe;
        const RowPlanes pc = load_row_planes(base + (uint64_t)r * W, w, W, rbits);
        RowPlanes pa = {0, 0, 0}, pb = {0, 0, 0};
        if (r > 0) pa = load_row_planes(base + (uint64_t)(r - 1) * W, w, W, rbits);
        else if (wrap_rows) pa = load_row_planes(base + (uint64_t)(rows - 1) * W, w, W, rbits);
        if (r + 1 < rows) pb = load_row_planes(base + (uint64_t)(r + 1) * W, w, W, rbits);
        else if (wrap_rows) pb = load_row_planes(base, w, W, rbits);
        uint32_t nxt = life_rule(hsum(pa.west, pa.c, pa.east), hsum(pc.west, pc.c, pc.east),
                                 hsum(pb.west, pb.c, pb.east), pc.c);
        if (w == W - 1) nxt &= last_mask;
        out[i] = nxt;
        if (alive_out != nullptr) {
            // envs are contiguous: reduce over the lanes that share this env, one atomic each
            const unsigned peers = __match_any_sync(__activemask(), e);
            const unsigned total_pop = __reduce_add_sync(peers, (unsigned)__popc(nxt));
            if ((threadIdx.x & 31) == (unsigned)(__ffs(peers) - 1)) atomicAdd(alive_out + e, total_pop);
        }
    }
}

// One thread per cell: scalar form of the stability rule (CGL/CGL.py:236-242).
__global__ void stable_generic_kernel(const uint32_t *__restrict__ prev, const uint32_t *__restrict__ next,
                                      int8_t *__restrict__ stable, uint64_t n_envs, uint32_t side,
                                      uint32_t W, int8_t spawn, int8_t stable_max,
                                      int32_t *__restrict__ reward_out, int rule, int8_t empty, int8_t empty_min)
{
    const uint64_t size = (uint64_t)side * side;
    const uint64_t total = n_envs * size;
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < total;
         i += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t e = i / size;
        const uint64_t cell = i - e * size;
        const uint32_t r = (uint32_t)(cell / side), c = (uint32_t)(cell - (uint64_t)r * side);
        const uint64_t widx = (e * side + r) * W + (c >> 5);
        const bool p = (prev[widx] >> (c & 31)) & 1u;
        const bool n = (next[widx] >> (c & 31)) & 1u;
        const int8_t s = stable_update1_rule(rule, stable[i], p, n, spawn, stable_max, empty, empty_min);
        stable[i] = s;
        if (reward_out != nullptr) {
            const unsigned peers = __match_any_sync(__activemask(), e);
            const int sum = __reduce_add_sync(peers, (int)s);
            if ((threadIdx.x & 31) == (unsigned)(__ffs(peers) - 1)) atomicAdd(reward_out + e, sum);
        }
    }
}

// =========================================================================================
// Any side up to ENV_BYTES_MAX_SIDE in ONE launch: one CTA per env, the world as one byte per cell in shared memory
// with torus halos (rows of `stride` bytes: left halo at byte 3, cell x at byte 4 + x, right halo at byte 4 + side,
// every other byte 0; halo rows above and below), so that a thread's four cells and their neighbours are three
// aligned words plus six bytes whatever the side is, the generation is packed-byte arithmetic (life_next4_bytes)
// and the stability update is the 4-cells-per-word rule of the fused kernel.  ~50 instructions per 4 cells against
// ~20 in the fused kernel (which needs side % 32 == 0), but one pass over HBM instead of three kernels with a scalar
// rule per cell.  Measured against the three-kernel path, us per step: 1024 x 200^2 63 vs 306, 4096 x 100^2 66 vs 253,
// 2048 x 130^2 109 vs 230, 16384 x 50^2 158 vs 251 (sides that are not multiples of 4 pay byte accesses to the
// stability plane); instruction-bound (181 thread instructions per 4 cells, issue slots 71 % busy), so sides below 32
// -- several envs per CTA, little work per thread -- stay on the small kernels.
// =========================================================================================
constexpr uint32_t ENV_BYTES_MAX_SIDE = 256;
constexpr uint32_t ENV_BYTES_MIN_SIDE = 32;      // below that the three small kernels win (measured: side 10, 65536 envs: 55 vs 68 us)
constexpr int ENV_BYTES_THREADS = 256;

__host__ __device__ __forceinline__ uint32_t env_bytes_stride(uint32_t side) { return (side + 5u + 3u) & ~3u; }

// VEC: side % 4 == 0 (then side^2 % 16 == 0: every row of every env's stability plane is word-aligned); RULE: the
// dead-cell rule, compile-time like in the fused kernel.
template <bool VEC, int RULE>
__global__ void __launch_bounds__(ENV_BYTES_THREADS)
env_step_bytes_kernel(const uint32_t *__restrict__ world_in, uint32_t *__restrict__ world_out, const int8_t *stable_in,
                      int8_t *stable_out, uint32_t side, uint32_t W, const int32_t *__restrict__ actions, int8_t spawn,
                      uint32_t max4, uint32_t min4, uint32_t empty4, int masked,
                      int32_t *__restrict__ reward_out, uint32_t *__restrict__ alive_out, int *__restrict__ err_flag,
                      uint32_t tpr, uint32_t rows_per_pass, uint32_t n_envs, uint32_t slot_threads, uint32_t slots,
                      uint32_t slot_bytes)
{
    // Small sides: several envs per CTA, one SLOT of slot_threads (a multiple of 32) threads each, its own piece of
    // shared memory; every slot runs the same trip counts, so the barriers stay CTA-wide.
    extern __shared__ __align__(16) unsigned char smem_dyn[];
    const uint32_t size = side * side, n_words = side * W, S = env_bytes_stride(side);
    const uint32_t slot = threadIdx.x / slot_threads, tid = threadIdx.x - slot * slot_threads;
    const uint32_t e_raw = blockIdx.x * slots + slot;
    const bool env_ok = slot < slots && e_raw < n_envs;
    const uint32_t e = env_ok ? e_raw : 0u;
    uint8_t *plane = smem_dyn + (slot < slots ? slot : 0u) * slot_bytes;
    uint32_t *nw = reinterpret_cast<uint32_t *>(plane + (((side + 2) * S + 15u) & ~15u));         // next world, packed
    __shared__ int red_all[2 * (ENV_BYTES_THREADS / 32)];
    int *red = red_all + 2 * (slot < slots ? slot : 0u);
    const uint32_t *win = world_in + (size_t)e * n_words;
    const size_t sbase = (size_t)e * size;

    // toggle_state before the step (CGL/main.py:66-67): applied to the packed words as they are loaded
    int act = -1;
    if (actions != nullptr && env_ok) {
        const int a = actions[e];
        if (a >= 0 && (uint32_t)a < size) act = a;
        else if ((uint32_t)a != size && tid == 0) {
            if (err_flag != nullptr) atomicOr(err_flag, 1);
            raise_alarm(ALARM_BAD_ACTION);
        }
    }
    const uint32_t act_y = act >= 0 ? (uint32_t)act / side : 0xffffffffu;
    const uint32_t act_x = act >= 0 ? (uint32_t)act - act_y * side : 0u;
    auto load_word = [&](uint32_t y, uint32_t w) {
        uint32_t v = __ldg(win + y * W + w);
        if (y == act_y && w == (act_x >> 5)) v ^= 1u << (act_x & 31);
        return v;
    };

    if (tid == 0 && env_ok) { red[0] = 0; red[1] = 0; }
    // world bits -> byte plane; the thread that handles a row's first / last word also writes the row's halos, and
    // the first / last row is written a second time as the halo row below / above the grid
    for (uint32_t i = tid; i < n_words && env_ok; i += slot_threads) {
        nw[i] = 0;
        const uint32_t y = i / W, w = i - y * W;
        const uint32_t bits = load_word(y, w);
        const uint32_t cells_here = side - 32 * w < 32 ? side - 32 * w : 32;
        const uint32_t groups = (cells_here + 3) >> 2;
        // the row's halos: cell side-1 left of cell 0 (written with word 0), cell 0 right of cell side-1 (last word)
        const uint32_t last_bit = w == 0 ? (load_word(y, W - 1) >> ((side - 1) & 31)) & 1u : 0u;
        const uint32_t first_bit = w == W - 1 ? load_word(y, 0) & 1u : 0u;
        for (int image = 0; image < 3; ++image) {
            if (image == 1 && y != 0) continue;                   // row 0 again as the halo row below the grid
            if (image == 2 && y != side - 1) continue;            // row side-1 again as the halo row above it
            uint8_t *row = plane + (image == 0 ? y + 1 : (image == 1 ? side + 1 : 0)) * S;
            for (uint32_t g = 0; g < groups; ++g)
                *reinterpret_cast<uint32_t *>(row + 4 + 32 * w + 4 * g) = (((bits >> (4 * g)) & 0xfu) * 0x00204081u) & 0x01010101u;
            if (w == 0) *reinterpret_cast<uint32_t *>(row) = last_bit << 24;                  // pads 0..2 and the left halo
            if (w == W - 1) {                                                                 // right halo, then pads
                row[4 + side] = (uint8_t)first_bit;
                for (uint32_t b = 4 + side + 1; b < S; ++b) row[b] = 0;
            }
        }
    }
    __syncthreads();

    const uint32_t ty = tid / tpr, x0 = (tid - ty * tpr) * 4;
    const bool lane_ok = ty < rows_per_pass && env_ok;
    const uint32_t nx = side - x0 < 4 ? side - x0 : 4;
    const uint32_t valid = nx == 4 ? 0xffffffffu : ((1u << (8 * nx)) - 1u);
    constexpr bool vec = VEC;
    const uint32_t spawn4 = rep4(spawn);
    int acc = 0;
    uint32_t pop = 0;
    auto load_sv = [&](uint32_t y) {
        const uint32_t base = y * side + x0;
        uint32_t sv = 0;
        if (vec) sv = *reinterpret_cast<const uint32_t *>(stable_in + sbase + base);
        else for (uint32_t k = 0; k < nx; ++k) sv |= (uint32_t)(uint8_t)stable_in[sbase + base + k] << (8 * k);
        return sv;
    };
    auto step_row = [&](uint32_t y, uint32_t sv) {
        const uint8_t *rm = plane + (y + 1) * S + 4 + x0;                                     // 4-byte aligned
        const uint32_t u = *reinterpret_cast<const uint32_t *>(rm - S);
        const uint32_t m = *reinterpret_cast<const uint32_t *>(rm);
        const uint32_t d = *reinterpret_cast<const uint32_t *>(rm + S);
        const uint32_t lc = (uint32_t)rm[-(int)S - 1] + rm[-1] + rm[S - 1];
        const uint32_t rc = (uint32_t)rm[4 - (int)S] + rm[4] + rm[S + 4];
        const uint32_t q = life_next4_bytes(u, m, d, lc, rc) & valid;                           // alive next, 0/1 per byte
        const uint32_t mv = m & valid;
        const uint32_t base = y * side + x0;
        if (y == act_y && act_x - x0 < nx) {                      // stable[action] = spawn (fork: 0 if toggled to dead)
            const uint32_t k = act_x - x0;
            const uint32_t alive_now = (mv >> (8 * k)) & 1u;
            const uint32_t put = (masked && !alive_now) ? 0u : (uint32_t)(uint8_t)spawn;
            sv = (sv & ~(0xffu << (8 * k))) | (put << (8 * k));
        }
        const uint32_t out = stable_update4_rule(RULE, sv, (q & mv) * 255u, (q & ~mv) * 255u, spawn4, max4, min4,
                                                 empty4) & valid;
        acc = __dp4a((int)out, 0x01010101, acc);
        pop += __popc(q);
        const uint32_t nib = (q * 0x10204080u) >> 28;             // byte j -> bit j
        if (nib) atomicOr(&nw[y * W + (x0 >> 5)], nib << (x0 & 31));
        if (vec) *reinterpret_cast<uint32_t *>(stable_out + sbase + base) = out;
        else for (uint32_t k = 0; k < nx; ++k) stable_out[sbase + base + k] = (int8_t)(out >> (8 * k));
    };
    // a thread's rows are ty, ty + rows_per_pass, ...: the stability words of FOUR of them are requested before the
    // first is used (a CTA's life is latency: one dependent HBM access per row otherwise)
    constexpr int U = 4;
    if (lane_ok)
        for (uint32_t y0 = ty; y0 < side; y0 += U * rows_per_pass) {
            uint32_t svs[U];
#pragma unroll
            for (int k = 0; k < U; ++k)
                if (y0 + k * rows_per_pass < side) svs[k] = load_sv(y0 + k * rows_per_pass);
#pragma unroll
            for (int k = 0; k < U; ++k)
                if (y0 + k * rows_per_pass < side) step_row(y0 + k * rows_per_pass, svs[k]);
        }
    acc = __reduce_add_sync(0xffffffffu, acc);
    pop = __reduce_add_sync(0xffffffffu, pop);
    if ((threadIdx.x & 31) == 0 && env_ok) {
        atomicAdd(&red[0], acc);
        atomicAdd(reinterpret_cast<unsigned *>(&red[1]), pop);
    }
    __syncthreads();
    uint32_t *wout = world_out + (size_t)e * n_words;
    for (uint32_t i = tid; i < n_words && env_ok; i += slot_threads) wout[i] = nw[i];
    if (tid == 0 && env_ok) {
        if (reward_out != nullptr) reward_out[e] = red[0];
        if (alive_out != nullptr) alive_out[e] = (uint32_t)red[1];
    }
}

static size_t env_bytes_smem(uint32_t side)
{
    const size_t b = ((((size_t)side + 2) * env_bytes_stride(side) + 15u) & ~(size_t)15u) + 4 * (size_t)side * cgl_words_per_row(side);
    return (b + 15u) & ~(size_t)15u;
}

static int launch_env_bytes(const cgl_env_step_args_t &a, cudaStream_t st)
{
    static PerDeviceOnce once;
    if (once.first()) {
        const int cap = (int)env_bytes_smem(ENV_BYTES_MAX_SIDE);
#define CGL_ATTR(V, R) CGL_CUDA(cudaFuncSetAttribute(env_step_bytes_kernel<V, R>, cudaFuncAttributeMaxDynamicSharedMemorySize, cap))
        CGL_ATTR(true, CGL_DEAD_ZERO); CGL_ATTR(true, CGL_DEAD_DECAY); CGL_ATTR(true, CGL_DEAD_SAT);
        CGL_ATTR(false, CGL_DEAD_ZERO); CGL_ATTR(false, CGL_DEAD_DECAY); CGL_ATTR(false, CGL_DEAD_SAT);
#undef CGL_ATTR
    }
    const uint32_t side = a.side, W = cgl_words_per_row(side), tpr = (side + 3) / 4;
    uint32_t rows_per_pass = ENV_BYTES_THREADS / tpr;             // tpr <= 64
    if (rows_per_pass > side) rows_per_pass = side;
    const uint32_t slot_threads = (tpr * rows_per_pass + 31) / 32 * 32;       // threads of one env, warp-aligned
    const uint32_t slots = ENV_BYTES_THREADS / slot_threads;                  // envs per CTA (1 for side >= 23)
    const uint32_t slot_bytes = (uint32_t)env_bytes_smem(side);
    const unsigned grid = (unsigned)((a.n_envs + slots - 1) / slots);
#define CGL_BYTES(V, R)                                                                                              \
    env_step_bytes_kernel<V, R><<<grid, ENV_BYTES_THREADS, (size_t)slots * slot_bytes, st>>>(                          \
        a.world_in_dev, a.world_out_dev, a.stable_in_dev, a.stable_out_dev, side, W, a.actions_dev, (int8_t)a.spawn,   \
        rep4(a.stable_max), rep4(a.empty_min), rep4(a.empty), a.masked_toggle != 0, a.reward_out_dev, a.alive_out_dev, \
        a.err_flag_dev, tpr, rows_per_pass, (uint32_t)a.n_envs, slot_threads, slots, slot_bytes)
    const bool vec = side % 4 == 0;
    if (a.dead_rule == CGL_DEAD_DECAY) { if (vec) CGL_BYTES(true, CGL_DEAD_DECAY); else CGL_BYTES(false, CGL_DEAD_DECAY); }
    else if (a.dead_rule == CGL_DEAD_SAT) { if (vec) CGL_BYTES(true, CGL_DEAD_SAT); else CGL_BYTES(false, CGL_DEAD_SAT); }
    else { if (vec) CGL_BYTES(true, CGL_DEAD_ZERO); else CGL_BYTES(false, CGL_DEAD_ZERO); }
#undef CGL_BYTES
    CGL_LAUNCH_CHECK();
    return 0;
}

// =========================================================================================
// Layout conversion and reductions
// =========================================================================================

// One warp builds 32 consecutive packed words; lane j reads the j-th cell of each word
// (coalesced 32-byte reads), __ballot_sync assembles the word, lane k keeps word k.
__global__ void pack_kernel(const uint8_t *__restrict__ cells, uint32_t *__restrict__ world,
                            uint64_t n_envs, uint32_t rows, uint32_t cols, uint32_t W)
{
    const uint64_t total_words = n_envs * rows * W;
    const uint32_t lane = threadIdx.x & 31;
    const uint64_t warp = (blockIdx.x * (uint64_t)blockDim.x + threadIdx.x) >> 5;
    const uint64_t n_warps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    for (uint64_t base = warp * 32; base < total_words; base += n_warps * 32) {
        uint32_t mine = 0;
        for (uint32_t k = 0; k < 32; ++k) {
            const uint64_t widx = base + k;
            uint32_t bit = 0;
            if (widx < total_words) {
                const uint64_t row = widx / W;               // global row index (e * rows + r)
                const uint32_t w = (uint32_t)(widx - row * W);
                const uint32_t col = w * 32 + lane;
                if (col < cols) bit = cells[row * cols + col] != 0;
            }
            const uint32_t word = __ballot_sync(0xffffffffu, bit);
            if (lane == k) mine = word;
        }
        if (base + lane < total_words) world[base + lane] = mine;
    }
}

// Rows of whole words (cols % 32 == 0: every fused side, every large grid): the cell index IS the bit index, so the
// conversions are flat streams.  pack: a thread turns 32 cell bytes (two 16-byte loads) into one word -- "byte != 0"
// lands in bit 7 of each byte, a multiply gathers the four bits of a word into a nibble.  HBM-bound: 1 + 1/8 bytes
// per cell instead of one 32-byte request and one ballot per 32 cells.
__global__ void __launch_bounds__(256)
pack_words_kernel(const uint4 *__restrict__ cells16, uint32_t *__restrict__ world, uint64_t total_words)
{
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < total_words;
         i += (uint64_t)gridDim.x * blockDim.x) {
        const uint4 a = __ldg(cells16 + 2 * i), b = __ldg(cells16 + 2 * i + 1);
        const uint32_t in[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
        uint32_t word = 0;
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const uint32_t x = in[k];
            const uint32_t nz = ((((x & 0x7f7f7f7fu) + 0x7f7f7f7fu) | x) & 0x80808080u) >> 7;      // 0/1 per byte
            word |= ((nz * 0x10204080u) >> 28) << (4 * k);           // byte j of the group -> bit j of the nibble
        }
        world[i] = word;
    }
}

// unpack / init_stable for rows of whole words: a thread expands 16 bits into one 16-byte store.
// mode 0: cells = bit.  mode 1: stable = bit ? spawn : 0, zeros then replaced by `empty`.
__global__ void __launch_bounds__(256)
unpack_words_kernel(const uint32_t *__restrict__ world, uint4 *__restrict__ cells16, uint64_t total16, int mode,
                    uint32_t spawn4, uint32_t empty4)
{
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < total16;
         i += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t half = (__ldg(world + (i >> 1)) >> ((i & 1) * 16)) & 0xffffu;
        uint32_t out[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const uint32_t ones = (((half >> (4 * k)) & 0xfu) * 0x00204081u) & 0x01010101u;        // 0/1 per byte
            if (mode == 0) {
                out[k] = ones;
            } else {
                const uint32_t m = ones * 0xffu;
                const uint32_t v = m & spawn4;                         // alive ? spawn : 0 ...
                // ... and every byte that is 0 now (dead cells, or alive with spawn == 0) becomes `empty`
                const uint32_t nz = (((v & 0x7f7f7f7fu) + 0x7f7f7f7fu) | v) & 0x80808080u;
                out[k] = v | (empty4 & ~((nz >> 7) * 0xffu));
            }
        }
        cells16[i] = make_uint4(out[0], out[1], out[2], out[3]);
    }
}

// One thread per cell.  mode 0: cells = bit.  mode 1: stable = bit ? spawn : 0, zeros then replaced by
// `empty` (CGL/CGL.py:111-112; the fork's `stable[stable == 0] = empty`, CGL_action+/CGL.py:124-126).
__global__ void unpack_kernel(const uint32_t *__restrict__ world, uint8_t *__restrict__ cells,
                              uint64_t n_envs, uint32_t rows, uint32_t cols, uint32_t W,
                              int mode, uint8_t spawn, uint8_t empty = 0)
{
    const uint64_t total = n_envs * rows * cols;
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < total;
         i += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t row = i / cols;
        const uint32_t c = (uint32_t)(i - row * cols);
        const uint32_t bit = (world[row * W + (c >> 5)] >> (c & 31)) & 1u;
        const uint8_t v = bit ? spawn : (uint8_t)0;
        cells[i] = mode == 0 ? (uint8_t)bit : (v ? v : empty);
    }
}

// blockIdx.y = env; blocks along x stride over the env's bytes; one atomic per block.
__global__ void reward_kernel(const int8_t *__restrict__ stable, uint64_t size,
                              int32_t *__restrict__ reward_out)
{
    const int8_t *s = stable + (uint64_t)blockIdx.y * size;
    int acc = 0;
    const uint64_t tid = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    const uint64_t nthr = (uint64_t)gridDim.x * blockDim.x;
    if ((reinterpret_cast<uintptr_t>(s) & 15) == 0) {
        const uint4 *v = reinterpret_cast<const uint4 *>(s);
        const uint64_t nvec = size / 16;
        for (uint64_t i = tid; i < nvec; i += nthr) {
            const uint4 x = __ldg(v + i);
            acc = __dp4a((int)x.x, 0x01010101, acc);
            acc = __dp4a((int)x.y, 0x01010101, acc);
            acc = __dp4a((int)x.z, 0x01010101, acc);
            acc = __dp4a((int)x.w, 0x01010101, acc);
        }
        for (uint64_t i = nvec * 16 + tid; i < size; i += nthr) acc += s[i];
    } else {
        for (uint64_t i = tid; i < size; i += nthr) acc += s[i];
    }
    acc = __reduce_add_sync(0xffffffffu, acc);
    __shared__ int block_acc;
    if (threadIdx.x == 0) block_acc = 0;
    __syncthreads();
    if ((threadIdx.x & 31) == 0 && acc != 0) atomicAdd(&block_acc, acc);
    __syncthreads();
    if (threadIdx.x == 0 && block_acc != 0) atomicAdd(reward_out + blockIdx.y, block_acc);
}

__global__ void alive_kernel(const uint32_t *__restrict__ world, uint64_t wpe,
                             uint32_t *__restrict__ alive_out)
{
    const uint32_t *w = world + (uint64_t)blockIdx.y * wpe;
    unsigned acc = 0;
    const uint64_t tid = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x;
    const uint64_t nthr = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = tid; i < wpe; i += nthr) acc += __popc(__ldg(w + i));
    acc = __reduce_add_sync(0xffffffffu, acc);
    __shared__ unsigned block_acc;
    if (threadIdx.x == 0) block_acc = 0;
    __syncthreads();
    if ((threadIdx.x & 31) == 0 && acc != 0) atomicAdd(&block_acc, acc);
    __syncthreads();
    if (threadIdx.x == 0 && block_acc != 0) atomicAdd(alive_out + blockIdx.y, block_acc);
}

__global__ void set_int_kernel(int *p, int v) { *p = v; }

__global__ void match_kernel(const uint32_t *__restrict__ a, const uint32_t *__restrict__ b,
                             uint64_t n_words, int *__restrict__ equal_out)
{
    bool diff = false;
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n_words;
         i += (uint64_t)gridDim.x * blockDim.x)
        diff |= (a[i] != b[i]);
    if (__any_sync(0xffffffffu, diff) && (threadIdx.x & 31) == 0) atomicAnd(equal_out, 0);
}

}  // namespace cgl

// =========================================================================================
// C ABI
// =========================================================================================
using namespace cgl;

extern "C" uint32_t cgl_words_per_row(uint32_t cols) { return (cols + 31) / 32; }

extern "C" int cgl_env_step_is_fused(uint32_t side) { return side % 32 == 0 && side >= 32 && side <= 256; }

extern "C" int cgl_env_step_launches(uint32_t side, int has_actions)
{
    if (cgl_env_step_is_fused(side) || env_bytes_takes(side)) return 1;
    return 2 + (has_actions ? 1 : 0);
}

extern "C" int cgl_pack(const uint8_t *cells, uint32_t *world, uint64_t n_envs, uint32_t rows,
                        uint32_t cols, cgl_stream_t stream)
{
    CGL_REQUIRE(cells && world && n_envs && rows && cols, CGL_E_BADARG, "cgl_pack: bad argument");
    const uint32_t W = cgl_words_per_row(cols);
    const uint64_t words = n_envs * rows * W;
    if (cols % 32 == 0 && (reinterpret_cast<uintptr_t>(cells) & 15u) == 0)
        pack_words_kernel<<<grid_for(words, 256), 256, 0, as_stream(stream)>>>(reinterpret_cast<const uint4 *>(cells),
                                                                                world, words);
    else
        pack_kernel<<<grid_for(words, 256), 256, 0, as_stream(stream)>>>(cells, world, n_envs, rows, cols, W);
    CGL_LAUNCH_CHECK();
    return 0;
}

extern "C" int cgl_unpack(const uint32_t *world, uint8_t *cells, uint64_t n_envs, uint32_t rows,
                          uint32_t cols, cgl_stream_t stream)
{
    CGL_REQUIRE(cells && world && n_envs && rows && cols, CGL_E_BADARG, "cgl_unpack: bad argument");
    const uint64_t total = n_envs * rows * cols;
    if (cols % 32 == 0 && (reinterpret_cast<uintptr_t>(cells) & 15u) == 0)
        unpack_words_kernel<<<grid_for(total / 16, 256), 256, 0, as_stream(stream)>>>(
            world, reinterpret_cast<uint4 *>(cells), total / 16, 0, 0u, 0u);
    else
        unpack_kernel<<<grid_for(total, 256), 256, 0, as_stream(stream)>>>(
            world, cells, n_envs, rows, cols, cgl_words_per_row(cols), 0, 0);
    CGL_LAUNCH_CHECK();
    return 0;
}

extern "C" int cgl_init_stable(const uint32_t *world, int8_t *stable, uint64_t n_envs, uint32_t side,
                               int spawn, cgl_stream_t stream)
{
    CGL_REQUIRE(stable && world && n_envs && side, CGL_E_BADARG, "cgl_init_stable: bad argument");
    const uint64_t total = n_envs * side * side;
    if (side % 32 == 0 && (reinterpret_cast<uintptr_t>(stable) & 15u) == 0)
        unpack_words_kernel<<<grid_for(total / 16, 256), 256, 0, as_stream(stream)>>>(
            world, reinterpret_cast<uint4 *>(stable), total / 16, 1, rep4(spawn), 0u);
    else
        unpack_kernel<<<grid_for(total, 256), 256, 0, as_stream(stream)>>>(
            world, reinterpret_cast<uint8_t *>(stable), n_envs, side, side, cgl_words_per_row(side), 1,
            (uint8_t)(int8_t)spawn);
    CGL_LAUNCH_CHECK();
    return 0;
}

extern "C" int cgl_toggle(uint32_t *world, int8_t *stable, uint64_t n_envs, uint32_t side,
                          const int32_t *idx, uint32_t k, int spawn, int *err_flag,
                          cgl_stream_t stream)
{
    CGL_REQUIRE(world && stable && n_envs && side && idx, CGL_E_BADARG, "cgl_toggle: bad argument");
    if (k == 0) return 0;
    toggle_kernel<<<grid_for(n_envs, 128), 128, 0, as_stream(stream)>>>(
        world, stable, n_envs, side, cgl_words_per_row(side), idx, k, (int8_t)spawn, err_flag, 0);
    CGL_LAUNCH_CHECK();
    return 0;
}

extern "C" int cgl_toggle_rule(uint32_t *world, int8_t *stable, uint64_t n_envs, uint32_t side,
                               const int32_t *idx, uint32_t k, int spawn, int masked, int *err_flag,
                               cgl_stream_t stream)
{
    CGL_REQUIRE(world && stable && n_envs && side && idx, CGL_E_BADARG, "cgl_toggle_rule: bad argument");
    if (k == 0) return 0;
    toggle_kernel<<<grid_for(n_envs, 128), 128, 0, as_stream(stream)>>>(
        world, stable, n_envs, side, cgl_words_per_row(side), idx, k, (int8_t)spawn, err_flag, masked);
    CGL_LAUNCH_CHECK();
    return 0;
}

extern "C" int cgl_init_stable_rule(const uint32_t *world, int8_t *stable, uint64_t n_envs, uint32_t side,
                                    int spawn, int empty, cgl_stream_t stream)
{
    CGL_REQUIRE(stable && world && n_envs && side, CGL_E_BADARG, "cgl_init_stable_rule: bad argument");
    const uint64_t total = n_envs * side * side;
    if (side % 32 == 0 && (reinterpret_cast<uintptr_t>(stable) & 15u) == 0)
        unpack_words_kernel<<<grid_for(total / 16, 256), 256, 0, as_stream(stream)>>>(
            world, reinterpret_cast<uint4 *>(stable), total / 16, 1, rep4(spawn), rep4(empty));
    else
        unpack_kernel<<<grid_for(total, 256), 256, 0, as_stream(stream)>>>(
            world, reinterpret_cast<uint8_t *>(stable), n_envs, side, side, cgl_words_per_row(side), 1,
            (uint8_t)(int8_t)spawn, (uint8_t)(int8_t)empty);
    CGL_LAUNCH_CHECK();
    return 0;
}

extern "C" int cgl_life_step(const uint32_t *in, uint32_t *out, uint64_t n_envs, uint32_t rows,
                             uint32_t cols, int wrap_rows, uint32_t *alive_out, cgl_stream_t stream);

// The one implementation behind every env-step entry point (see include/cgl_b200.h, cgl_env_step_ex).
extern "C" int cgl_env_step_ex(const cgl_env_step_args_t *args, cgl_stream_t stream)
{
    CGL_REQUIRE(args, CGL_E_BADARG, "cgl_env_step_ex: null");
    cgl_env_step_args_t a = *args;
    CGL_REQUIRE(a.world_in_dev && a.world_out_dev && a.stable_in_dev && a.n_envs && a.side, CGL_E_BADARG,
                "cgl_env_step: bad argument");
    CGL_REQUIRE(a.world_in_dev != a.world_out_dev, CGL_E_BADARG, "cgl_env_step: world_in and world_out must not alias");
    CGL_REQUIRE(a.n_envs < (1ull << 31), CGL_E_BADARG, "cgl_env_step: n_envs too large");
    CGL_REQUIRE(a.dead_rule >= CGL_DEAD_ZERO && a.dead_rule <= CGL_DEAD_SAT, CGL_E_BADARG,
                "cgl_env_step: dead_rule must be 0 (zero), 1 (decay) or 2 (saturate)");
    CGL_REQUIRE(a.empty >= -128 && a.empty <= 127 && a.empty_min >= -128 && a.empty_min <= 127, CGL_E_BADARG,
                "cgl_env_step: empty / empty_min must fit int8");
    CGL_REQUIRE(a.chain_mode <= CGL_CHAIN_SEQ && (a.chain_mode == CGL_CHAIN_NONE || a.token_dev), CGL_E_BADARG,
                "cgl_env_step: chain_mode must be 0..2 and needs token_dev");
    if (a.stable_out_dev == nullptr) a.stable_out_dev = const_cast<int8_t *>(a.stable_in_dev);
    if (a.chain_mode == CGL_CHAIN_NONE) a.token_dev = nullptr;
    const bool fused = cgl_env_step_is_fused(a.side);
    CGL_REQUIRE(fused || a.chain_mode == CGL_CHAIN_NONE, CGL_E_BADARG,
                "cgl_env_step: chained steps need a fused side (multiple of 32, 32..256)");
    if (a.chain_mode == CGL_CHAIN_SEQ && a.seq_counter_host != nullptr) {
        a.want = *a.seq_counter_host;               // consecutive sequence numbers, kept by the caller's counter
        a.publish = a.want + 1;
    }
    cudaStream_t st = as_stream(stream);
    int rc = -100;
    if (fused) {
        switch (a.side) {
        case 32: rc = launch_env_fused<32>(a, st); break;
        case 64: rc = launch_env_fused<64>(a, st); break;
        case 96: rc = launch_env_fused<96>(a, st); break;
        case 128: rc = launch_env_fused<128>(a, st); break;
        case 160: rc = launch_env_fused<160>(a, st); break;
        case 192: rc = launch_env_fused<192>(a, st); break;
        case 224: rc = launch_env_fused<224>(a, st); break;
        case 256: rc = launch_env_fused<256>(a, st); break;
        }
    }
    if (rc == -100 && env_bytes_takes(a.side))
        rc = launch_env_bytes(a, st);                // any side up to 256: one launch, one CTA per env
    if (rc == -100) {
        // larger sides: (plane copy) -> toggle -> generation -> stability, all in place on stable_out
        const uint32_t W = cgl_words_per_row(a.side);
        const uint64_t cells = a.n_envs * a.side * a.side;
        if (a.stable_in_dev != a.stable_out_dev)
            CGL_CUDA(cudaMemcpyAsync(a.stable_out_dev, a.stable_in_dev, cells, cudaMemcpyDeviceToDevice, st));
        if (a.actions_dev != nullptr &&
            (rc = cgl_toggle_rule(a.world_in_dev, a.stable_out_dev, a.n_envs, a.side, a.actions_dev, 1, a.spawn,
                                  a.masked_toggle, a.err_flag_dev, stream)))
            return rc;
        if ((rc = cgl_life_step(a.world_in_dev, a.world_out_dev, a.n_envs, a.side, a.side, 1, a.alive_out_dev, stream)))
            return rc;
        if (a.reward_out_dev != nullptr) CGL_CUDA(cudaMemsetAsync(a.reward_out_dev, 0, a.n_envs * sizeof(int32_t), st));
        stable_generic_kernel<<<grid_for(cells, 256), 256, 0, st>>>(
            a.world_in_dev, a.world_out_dev, a.stable_out_dev, a.n_envs, a.side, W, (int8_t)a.spawn, (int8_t)a.stable_max,
            a.reward_out_dev, a.dead_rule, (int8_t)a.empty, (int8_t)a.empty_min);
        CGL_LAUNCH_CHECK();
        rc = 0;
    }
    if (rc == 0 && a.chain_mode == CGL_CHAIN_SEQ && a.seq_counter_host != nullptr) ++*a.seq_counter_host;
    return rc;
}

static cgl_env_step_args_t base_args(uint32_t *win, uint32_t *wout, const int8_t *sin, int8_t *sout, uint64_t n_envs,
                                     uint32_t side, const int32_t *actions, int spawn, int stable_max, int32_t *reward,
                                     uint32_t *alive, int *err)
{
    cgl_env_step_args_t a = {};
    a.world_in_dev = win; a.world_out_dev = wout; a.stable_in_dev = sin; a.stable_out_dev = sout;
    a.n_envs = n_envs; a.side = side; a.actions_dev = actions; a.spawn = spawn; a.stable_max = stable_max;
    a.reward_out_dev = reward; a.alive_out_dev = alive; a.err_flag_dev = err;
    return a;
}

extern "C" int cgl_env_step(uint32_t *win, uint32_t *wout, int8_t *stable, uint64_t n_envs,
                            uint32_t side, const int32_t *actions, int spawn, int stable_max,
                            int32_t *reward, uint32_t *alive, int *err, cgl_stream_t stream)
{
    const cgl_env_step_args_t a = base_args(win, wout, stable, stable, n_envs, side, actions, spawn, stable_max, reward,
                                            alive, err);
    return cgl_env_step_ex(&a, stream);
}

// Chained form of cgl_env_step for the fused sides (plane ids: replayable): see include/cgl_b200.h.
extern "C" int cgl_env_step_chained(uint32_t *win, uint32_t *wout, int8_t *stable, uint64_t n_envs, uint32_t side,
                                    const int32_t *actions, int spawn, int stable_max, int32_t *reward,
                                    uint32_t *alive, int *err, uint32_t *epoch_flags, uint32_t want,
                                    uint32_t publish, cgl_stream_t stream)
{
    CGL_REQUIRE(epoch_flags, CGL_E_BADARG, "cgl_env_step_chained: bad argument");
    cgl_env_step_args_t a = base_args(win, wout, stable, stable, n_envs, side, actions, spawn, stable_max, reward, alive, err);
    a.token_dev = epoch_flags; a.want = want; a.publish = publish; a.chain_mode = CGL_CHAIN_IDS;
    return cgl_env_step_ex(&a, stream);
}

// A whole sequence of env steps enqueued by ONE call (see include/cgl_b200.h): the launch loop runs in C, so the
// host side of a step is one cudaLaunchKernelEx (~2 us) instead of a trip through the binding per step.
extern "C" int cgl_env_step_seq(const cgl_env_step_args_t *steps, uint32_t n_descs, uint64_t n_steps, uint64_t first,
                                cgl_stream_t stream)
{
    CGL_REQUIRE(steps && n_descs, CGL_E_BADARG, "cgl_env_step_seq: bad argument");
    for (uint64_t i = 0; i < n_steps; ++i) {
        const int rc = cgl_env_step_ex(&steps[(first + i) % n_descs], stream);
        if (rc) return rc;
    }
    return 0;
}

// The same with the caller's two CUDA events recorded on `stream` right before the first and right after the last
// launch: a timed region then starts with the first launch instead of with the binding's call overhead.
extern "C" int cgl_env_step_seq_timed(const cgl_env_step_args_t *steps, uint32_t n_descs, uint64_t n_steps, uint64_t first,
                                      cgl_stream_t stream, void *start_event, void *stop_event)
{
    CGL_REQUIRE(steps && n_descs, CGL_E_BADARG, "cgl_env_step_seq_timed: bad argument");
    if (start_event) CGL_CUDA(cudaEventRecord(static_cast<cudaEvent_t>(start_event), as_stream(stream)));
    for (uint64_t i = 0; i < n_steps; ++i) {
        const int rc = cgl_env_step_ex(&steps[(first + i) % n_descs], stream);
        if (rc) return rc;
    }
    if (stop_event) CGL_CUDA(cudaEventRecord(static_cast<cudaEvent_t>(stop_event), as_stream(stream)));
    return 0;
}

// Out-of-place form: the new stability plane goes to `stable_out` (see include/cgl_b200.h).
extern "C" int cgl_env_step_io(uint32_t *win, uint32_t *wout, const int8_t *stable_in, int8_t *stable_out,
                               uint64_t n_envs, uint32_t side, const int32_t *actions, int spawn, int stable_max,
                               int32_t *reward, uint32_t *alive, int *err, uint32_t *epoch_flags, uint32_t want,
                               uint32_t publish, cgl_stream_t stream)
{
    CGL_REQUIRE(stable_out, CGL_E_BADARG, "cgl_env_step_io: bad argument");
    cgl_env_step_args_t a = base_args(win, wout, stable_in, stable_out, n_envs, side, actions, spawn, stable_max, reward,
                                      alive, err);
    a.token_dev = epoch_flags; a.want = want; a.publish = publish;
    a.chain_mode = epoch_flags ? CGL_CHAIN_IDS : CGL_CHAIN_NONE;
    return cgl_env_step_ex(&a, stream);
}

// The CGL_action+ fork's env step: see include/cgl_b200.h.
extern "C" int cgl_env_step_rule(uint32_t *win, uint32_t *wout, const int8_t *stable_in, int8_t *stable_out,
                                 uint64_t n_envs, uint32_t side, const int32_t *actions, int spawn, int stable_max,
                                 int dead_rule, int empty, int empty_min, int masked_toggle, int32_t *reward,
                                 uint32_t *alive, int *err, uint32_t *epoch_flags, uint32_t want, uint32_t publish,
                                 cgl_stream_t stream)
{
    CGL_REQUIRE(stable_out, CGL_E_BADARG, "cgl_env_step_rule: bad argument");
    cgl_env_step_args_t a = base_args(win, wout, stable_in, stable_out, n_envs, side, actions, spawn, stable_max, reward,
                                      alive, err);
    a.dead_rule = dead_rule; a.empty = empty; a.empty_min = empty_min; a.masked_toggle = masked_toggle != 0;
    a.token_dev = epoch_flags; a.want = want; a.publish = publish;
    a.chain_mode = epoch_flags ? CGL_CHAIN_IDS : CGL_CHAIN_NONE;
    return cgl_env_step_ex(&a, stream);
}

extern "C" int cgl_life_step_generic(const uint32_t *in, uint32_t *out, uint64_t n_envs, uint32_t rows,
                                     uint32_t cols, int wrap_rows, uint32_t *alive_out,
                                     cgl_stream_t stream)
{
    CGL_REQUIRE(in && out && n_envs && rows && cols && in != out, CGL_E_BADARG,
                "cgl_life_step: bad argument");
    cudaStream_t st = as_stream(stream);
    const uint32_t W = cgl_words_per_row(cols);
    if (alive_out != nullptr) CGL_CUDA(cudaMemsetAsync(alive_out, 0, n_envs * sizeof(uint32_t), st));
    const uint64_t words = n_envs * rows * W;
    life_generic_kernel<<<grid_for(words, 256), 256, 0, st>>>(in, out, n_envs, rows, cols, W,
                                                             wrap_rows, alive_out);
    CGL_LAUNCH_CHECK();
    return 0;
}

extern "C" int cgl_reward(const int8_t *stable, uint64_t n_envs, uint64_t size, int32_t *reward_out,
                          cgl_stream_t stream)
{
    CGL_REQUIRE(stable && n_envs && size && reward_out && n_envs <= 65535 * 1024ull, CGL_E_BADARG,
                "cgl_reward: bad argument");
    cudaStream_t st = as_stream(stream);
    CGL_CUDA(cudaMemsetAsync(reward_out, 0, n_envs * sizeof(int32_t), st));
    const unsigned threads = 256;
    uint64_t bx = (size / 16 + threads * 4 - 1) / (threads * 4);
    const uint64_t cap = (uint64_t)sm_count() * 8;
    bx = bx < 1 ? 1 : (bx > cap ? cap : bx);
    for (uint64_t e0 = 0; e0 < n_envs; e0 += 65535) {        // gridDim.y limit
        const unsigned ny = (unsigned)((n_envs - e0) < 65535 ? (n_envs - e0) : 65535);
        reward_kernel<<<dim3((unsigned)bx, ny), threads, 0, st>>>(stable + e0 * size, size, reward_out + e0);
        CGL_LAUNCH_CHECK();
    }
    return 0;
}

extern "C" int cgl_alive(const uint32_t *world, uint64_t n_envs, uint64_t wpe, uint32_t *alive_out,
                         cgl_stream_t stream)
{
    CGL_REQUIRE(world && n_envs && wpe && alive_out, CGL_E_BADARG, "cgl_alive: bad argument");
    cudaStream_t st = as_stream(stream);
    CGL_CUDA(cudaMemsetAsync(alive_out, 0, n_envs * sizeof(uint32_t), st));
    const unsigned threads = 256;
    uint64_t bx = (wpe + threads * 4 - 1) / (threads * 4);
    const uint64_t cap = (uint64_t)sm_count() * 8;
    bx = bx < 1 ? 1 : (bx > cap ? cap : bx);
    for (uint64_t e0 = 0; e0 < n_envs; e0 += 65535) {
        const unsigned ny = (unsigned)((n_envs - e0) < 65535 ? (n_envs - e0) : 65535);
        alive_kernel<<<dim3((unsigned)bx, ny), threads, 0, st>>>(world + e0 * wpe, wpe, alive_out + e0);
        CGL_LAUNCH_CHECK();
    }
    return 0;
}

extern "C" int cgl_match(const uint32_t *a, const uint32_t *b, uint64_t n_words, int *equal_out,
                         cgl_stream_t stream)
{
    CGL_REQUIRE(a && b && n_words && equal_out, CGL_E_BADARG, "cgl_match: bad argument");
    cudaStream_t st = as_stream(stream);
    set_int_kernel<<<1, 1, 0, st>>>(equal_out, 1);
    match_kernel<<<grid_for(n_words, 256), 256, 0, st>>>(a, b, n_words, equal_out);
    CGL_LAUNCH_CHECK();
    return 0;
}
