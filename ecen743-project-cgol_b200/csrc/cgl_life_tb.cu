// cgl_life_tb.cu -- temporal blocking for life mode: K generations per launch, one HBM pass.
//
// Reference semantics: K applications of the world half of kernel `run`
// (/root/reference/CGL/CGL.py:154-170).  BASELINE.json configs[4].
//
// Time-skewed register pipeline (no shared memory, no re-reads):
//   * a warp owns a strip of 30 packed word-columns (+1 halo word-column on each side, lanes 0 and
//     31) and streams down the rows; lane l holds word-column 30*cg + l - 1.  The halo words go
//     stale by one bit-column per generation, so lanes 1..30 stay exact for K <= 32.
//   * level g (1..K) keeps a 2-row window of horizontal partial sums of generation g-1; when row
//     rho of generation g-1 arrives it emits row rho-1 of generation g, which feeds level g+1 on
//     the NEXT row step (one step of skew makes the K levels independent within a step: ILP = K).
//   * per 32 cells and generation: 2 SHFL + 2 SHF + 10 LOP3 -- the k = 1 kernel's ALU work -- while
//     HBM traffic drops to (32/30 read + 1 write) bits per cell per K generations.
// Row r of generation K leaves the pipeline 3K-1 row steps after gen-0 row r-K entered it, so a
// strip of L rows costs L + 3K - 1 steps.
#include <stdlib.h>

#include "cgl_internal.cuh"

namespace cgl {

struct Win {            // window of one level: rows (a-1, a) of the level's input generation
    uint32_t us0, us1;                  // row a-1: west+centre+east sum bits
    uint32_t ms0, ms1, mt0, mt1, mc;    // row a: sums with / without the centre, and the centre word
};

// Tried and measured on B200 (profiles/r01_sweeps.md): moving the two funnel shifts to the FMA pipe
// (IMAD / IMAD.HI with opaque multipliers) is 6 % SLOWER although the kernel is ALU-pipe bound, and
// one-warp CTAs are 12 % slower than 4-warp CTAs, and mapping a whole CTA to one row block (loop
// bounds in uniform registers) is 7 % slower than the warp-linear mapping below; all removed again.

// Chained launches of one cgl_life_run: strip (cg, rb) of launch j needs the outputs of -- and must
// not overwrite the inputs of -- the 3 x 3 neighbouring strips of launch j-1.  Each strip publishes
// tokens[rb * n_cgroups + cg] = j + 1 when it is done and launch j waits for the nine neighbours to
// reach j; with programmatic dependent launch the first strips of launch j+1 then run while the
// last strips of launch j finish, which removes the cost of a partly filled last wave.
struct ChainCtx { uint32_t *tokens; uint32_t want; uint32_t cap; };

// Predicated store: `if (ok && a < b) *p = v` as ONE predicated STG.  Written in PTX on purpose: the
// row-range test is CTA-uniform, and for a uniform condition the compiler emits a branch around the
// store, which splits the 6-step unrolled body into basic blocks and costs ~8 % (measured) because
// independent levels of neighbouring steps can no longer be interleaved.
__device__ __forceinline__ void st_if_lt(uint32_t *p, uint32_t v, bool ok, uint32_t a, uint32_t b)
{
    asm volatile(
        "{\n\t.reg .pred p, q;\n\t"
        "setp.lt.u32 p, %2, %3;\n\t"
        "setp.ne.u32 q, %4, 0;\n\t"
        "and.pred p, p, q;\n\t"
        "@p st.global.u32 [%0], %1;\n\t}"
        ::"l"(p), "r"(v), "r"(a), "r"(b), "r"((uint32_t)ok) : "memory");
}

constexpr int TB_UNROLL = 6;            // row steps per loop trip (loads issued up front)
constexpr int TB_COLS = 30;             // valid word-columns per warp

constexpr int TB_THREADS = 128;

// Population trace of a counted launch (cgl_life_run_pop): pop[g] += live cells of generation g + 1 of the launch in
// the rows of [row0, row1) that the strip owns, counted by the lanes that store.  A thread keeps two levels' counts
// per register as 16-bit halves (K/2 registers instead of K), so a counted launch keeps its strips at most
// TB_POP_MAX_ROWS rows long: at most 2047 x 32 < 2^16 cells per thread and level.
struct PopCtx { unsigned long long *pop; uint32_t row0, row1; };
constexpr uint32_t TB_POP_MAX_ROWS = 2047;

// Add the popcount of level g's output row y to the thread's count if the row lies in the strip's part of the count
// window: t = row - max(r0, row0) < cn.  CNT 0: no count (the uncounted kernels).
// Measured alternatives, none kept (ptxas -v, life_tb2_kernel<8>): a separate steady-state loop without the row test
// for strips inside the window takes 142-148 registers (three loop nests), shared-memory counters 163, and a
// __launch_bounds__ minimum of 5 CTAs spills; the row test in every step costs 108 registers (4 CTAs per SM).
template <int CNT, int K>
__device__ __forceinline__ void tally(uint32_t (&acc)[(K + 1) / 2], int g, uint32_t y, uint32_t t, uint32_t cn)
{
    if constexpr (CNT == 1) acc[g >> 1] += (t < cn ? (uint32_t)__popc(y) : 0u) << (16 * (g & 1));
}

// Strip-uniform set-up of a counted launch: the row test of level g at step s is (uint32_t)(s - m g + cbase) < cn,
// where level g emits row r0 - K + s - m g - 1 (m = 1 direct, 2 skewed).  Every count of a padding warp or of a strip
// whose token wait expired is dropped by pop_flush (store_ok).
struct PopWin { int cbase; uint32_t cn; };
__device__ __forceinline__ PopWin pop_window(const PopCtx &pc, int r0, int r1, int K)
{
    const int lo = r0 > (int)pc.row0 ? r0 : (int)pc.row0;
    const int hi = r1 < (int)pc.row1 ? r1 : (int)pc.row1;
    return PopWin{r0 - K - 1 - lo, hi > lo ? (uint32_t)(hi - lo) : 0u};
}

// End of a counted strip: the storing lanes' counts of each level, summed over the warp, go to pop[g].
template <int K>
__device__ __forceinline__ void pop_flush(const uint32_t (&acc)[(K + 1) / 2], const PopCtx &pc, bool store_ok, uint32_t lane)
{
#pragma unroll
    for (int g = 0; g < K; ++g) {
        uint32_t v = store_ok ? (acc[g >> 1] >> (16 * (g & 1))) & 0xffffu : 0u;
        v = __reduce_add_sync(0xffffffffu, v);
        if (lane == 0 && v != 0) atomicAdd(pc.pop + g, (unsigned long long)v);
    }
}

template <int K, bool POP>
__global__ void __launch_bounds__(TB_THREADS)
life_tb_kernel(const uint32_t *__restrict__ in, uint32_t *__restrict__ out, uint32_t rows, uint32_t W,
               uint32_t rpt, int wrap_rows, uint32_t n_cgroups, uint32_t n_rblocks, const ChainCtx chain,
               const PopCtx popc)
{
    // Warps are numbered along the row first (column group fastest).  No early exit: padding warps
    // redo the last strip with stores off and the loop trip count is the same for every warp, so
    // every shuffle below is provably convergent (plain SHFL; a divergence fallback path costs ~8 %).
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t warp = blockIdx.x * (TB_THREADS / 32) + (threadIdx.x >> 5);
    const uint32_t cg = warp % n_cgroups;
    uint32_t rb = warp / n_cgroups;
    const bool warp_ok = rb < n_rblocks;
    rb = warp_ok ? rb : n_rblocks - 1;
    bool wait_ok = true;                                       // warp-uniform: false once a bounded wait expired

    if (chain.tokens != nullptr) {                             // kernel-uniform branch
        cudaTriggerProgrammaticLaunchCompletion();
        // lanes 0..8 watch one neighbour strip each (columns always wrap, rows wrap on the torus)
        const int dj = (int)(lane % 3) - 1, di = (int)(lane / 3) - 1;
        const uint32_t ncg = (cg + n_cgroups + (uint32_t)dj) % n_cgroups;
        int nrb = (int)rb + di;
        bool need = lane < 9;
        if (nrb < 0 || nrb >= (int)n_rblocks) {
            if (wrap_rows) nrb = nrb < 0 ? nrb + (int)n_rblocks : nrb - (int)n_rblocks;
            else need = false;
        }
        const uint32_t *tp = chain.tokens + (need ? (uint32_t)nrb * n_cgroups + ncg : 0u);
        uint32_t v, spins = 0;
        unsigned long long t0 = 0;
        while (true) {                                         // every exit is a warp vote (see above)
            asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(tp) : "memory");
            if (__all_sync(0xffffffffu, !need || (int32_t)(v - chain.want) >= 0)) break;
            if (spins == 0) t0 = globaltimer_ns();
            if ((++spins & 255u) == 0 && __any_sync(0xffffffffu, wait_expired(t0, ALARM_LIFE_TOKEN))) {
                // a neighbour strip of the previous launch never finished: store nothing, publish nothing
                // (later launches of the chain then fail the same way) and tell the host
                wait_ok = false;
                if (lane == 0) raise_alarm(ALARM_LIFE_TOKEN);
                break;
            }
        }
    }

    const int wi = (int)(cg * TB_COLS + lane) - 1;             // word column of this lane (may be -1 or >= W)
    const uint32_t wcol = wi < 0 ? (uint32_t)(wi + (int)W) : ((uint32_t)wi >= W ? (uint32_t)wi - W : (uint32_t)wi);
    const bool store_ok = warp_ok && wait_ok && lane >= 1 && lane <= TB_COLS && (uint32_t)wi < W;

    const int r0 = (int)(rb * rpt);
    const int r1 = (r0 + (int)rpt < (int)rows) ? r0 + (int)rpt : (int)rows;
    const int irows = (int)rows;
    const int rstart = r0 - K;                                  // first gen-0 row fed to level 1 (>= -K)
    const int n_steps = (int)rpt + 3 * K - 1;                   // same trip count for every warp (uniform loop)
    // Step s loads gen-0 row rstart + s.  It is needed (and inside the grid, for open rows) iff
    // s_lo <= s < s_hi; rows from r1 + K on can no longer reach an output row of this strip.
    const int s_lo = wrap_rows ? 0 : (rstart < 0 ? -rstart : 0);
    const int last = (wrap_rows || r1 + K < irows) ? r1 + K : irows;
    const uint32_t span = (uint32_t)(last - rstart - s_lo);
    const uint32_t out_rows = (uint32_t)(r1 - r0);
    // Row index modulo rows, in [0, rows): the row loop wraps it with one subtraction per trip.  A true modulo,
    // because a torus with fewer rows than K starts more than one lap above row 0.
    int rw = (rstart % irows + irows) % irows;
    const uint32_t *ip = in + wcol;
    uint32_t *op = out + (store_ok ? (uint32_t)wi : 0u);

    Win win[K];
    uint32_t pend[K];                   // pend[g] = output of level g+1 at the previous step
#pragma unroll
    for (int g = 0; g < K; ++g) {
        win[g] = Win{0, 0, 0, 0, 0, 0, 0};
        pend[g] = 0;
    }
    uint32_t acc[(K + 1) / 2] = {};
    const PopWin pw = POP ? pop_window(popc, r0, r1, K) : PopWin{0, 0};
    constexpr int CNT = POP ? 1 : 0;

    for (int s0 = 0; s0 < n_steps; s0 += TB_UNROLL) {
        uint32_t raw[TB_UNROLL];
#pragma unroll
        for (int u = 0; u < TB_UNROLL; ++u) {
            const uint32_t ru = umin((uint32_t)rw + u, (uint32_t)rw + u - rows);      // (rw + u) mod rows
            raw[u] = 0;
            if ((uint32_t)(s0 + u - s_lo) < span)                                       // rows * W < 2^32
                raw[u] = __ldg(ip + ru * W);
        }
        rw += TB_UNROLL;
        rw = rw >= irows ? rw - irows : rw;
#pragma unroll
        for (int u = 0; u < TB_UNROLL; ++u) {
            // levels in descending order: level g+1 reads pend[g-1] before level g overwrites it
#pragma unroll
            for (int g = K - 1; g >= 0; --g) {
                const uint32_t x = (g == 0) ? raw[u] : pend[g - 1];
                const uint32_t left = __shfl_up_sync(0xffffffffu, x, 1);
                const uint32_t right = __shfl_down_sync(0xffffffffu, x, 1);
                const HSum d = hsum(west_plane(left, x), x, east_plane(x, right));
                const HSum up = {win[g].us0, win[g].us1, 0, 0};
                const HSum mid = {0, 0, win[g].mt0, win[g].mt1};
                pend[g] = life_rule(up, mid, d, win[g].mc);
                win[g].us0 = win[g].ms0; win[g].us1 = win[g].ms1;
                win[g].ms0 = d.s0; win[g].ms1 = d.s1; win[g].mt0 = d.t0; win[g].mt1 = d.t1; win[g].mc = x;
                tally<CNT, K>(acc, g, pend[g], (uint32_t)(s0 + u - 2 * g + pw.cbase), pw.cn);     // row r0 - K + s - 2g - 1
            }
            // row r0 + so of generation K has just left level K
            const uint32_t so = (uint32_t)(s0 + u - (3 * K - 1));
            const uint32_t ro = (uint32_t)r0 + so;
            st_if_lt(op + ro * W, pend[K - 1], store_ok, so, out_rows);
        }
    }
    if constexpr (POP) pop_flush<K>(acc, popc, store_ok, lane);
    if (chain.tokens != nullptr) {
        __threadfence();                             // this strip's rows are visible device-wide ...
        __syncwarp();
        if (lane == 0 && warp_ok && wait_ok)         // ... before its token is published
            asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(chain.tokens + rb * n_cgroups + cg),
                         "r"(chain.want + 1) : "memory");
    }
}

// ---------------------------------------------------------------------------------------------------------
// Direct pipeline (no skew) with a triangular start-up.  Level g+1 consumes level g's row in the SAME row step, so
// a strip of L rows costs L + 2K steps instead of L + 3K - 1, and during the first 2K steps level g is skipped
// until step 2g (nothing it could produce before is needed): the start-up costs K(K+1) level-steps = (K+1)/2 full
// steps' worth of work on top of the K dead rows -- 9 instead of 23 step equivalents for K = 8.  That matters where
// strips are short: the 8192-row bands of the 8-GPU C4 run (~200-row strips) spend 10 % of every launch in the
// fill of the skewed pipeline.  Parallelism inside a warp now comes from the wavefront over the unrolled row steps
// (step u+1 of level g and step u of level g+1 are independent) instead of from K independent levels.
// Same strip geometry, chaining and ghost-zone contract as life_tb_kernel.
// Row steps per block and software prefetch of the next block's rows.  Measured on B200 (8320 x 65536 band /
// 65536^2 torus, us per generation): 6 steps no prefetch 16.18 / 116.5, 8 steps 15.97 / 115.1, 4 steps with the
// next block's rows requested before the current block is computed 15.76 / 114.1 (96 registers: still 5 CTAs per
// SM), 3 steps with prefetch 15.88 / 115.2, 4 steps without 21.2 / 151.
constexpr int TB2_UNROLL = 4;

template <int K, bool PRO, int CNT>
__device__ __forceinline__ void tb2_block(const uint32_t (&raw)[TB2_UNROLL], Win (&win)[K], int s0, uint32_t *op, uint32_t r0W,
                                          uint32_t W, bool store_ok, uint32_t out_rows, uint32_t (&acc)[(K + 1) / 2],
                                          const PopWin &pw)
{
#pragma unroll
    for (int u = 0; u < TB2_UNROLL; ++u) {
        uint32_t x = raw[u];
#pragma unroll
        for (int g = 0; g < K; ++g) {
            if (PRO && s0 + u < 2 * g) {             // warp-uniform: this level has nothing to do yet
                x = 0;
                continue;
            }
            const uint32_t left = __shfl_up_sync(0xffffffffu, x, 1);
            const uint32_t right = __shfl_down_sync(0xffffffffu, x, 1);
            const HSum d = hsum(west_plane(left, x), x, east_plane(x, right));
            const HSum up = {win[g].us0, win[g].us1, 0, 0};
            const HSum mid = {0, 0, win[g].mt0, win[g].mt1};
            const uint32_t y = life_rule(up, mid, d, win[g].mc);
            win[g].us0 = win[g].ms0; win[g].us1 = win[g].ms1;
            win[g].ms0 = d.s0; win[g].ms1 = d.s1; win[g].mt0 = d.t0; win[g].mt1 = d.t1; win[g].mc = x;
            x = y;
            tally<CNT, K>(acc, g, y, (uint32_t)(s0 + u - g + pw.cbase), pw.cn);     // row r0 - K + s0 + u - g - 1
        }
        // row r0 + so of generation K has just left level K
        const uint32_t so = (uint32_t)(s0 + u - 2 * K);
        st_if_lt(op + r0W + so * W, x, store_ok, so, out_rows);
    }
}

template <int K, bool POP>
__global__ void __launch_bounds__(TB_THREADS)
life_tb2_kernel(const uint32_t *__restrict__ in, uint32_t *__restrict__ out, uint32_t rows, uint32_t W, uint32_t rpt,
                int wrap_rows, uint32_t n_cgroups, uint32_t n_rblocks, const ChainCtx chain, const PopCtx popc)
{
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t warp = blockIdx.x * (TB_THREADS / 32) + (threadIdx.x >> 5);
    const uint32_t cg = warp % n_cgroups;
    uint32_t rb = warp / n_cgroups;
    const bool warp_ok = rb < n_rblocks;
    rb = warp_ok ? rb : n_rblocks - 1;
    bool wait_ok = true;

    if (chain.tokens != nullptr) {                             // kernel-uniform branch (see life_tb_kernel)
        cudaTriggerProgrammaticLaunchCompletion();
        const int dj = (int)(lane % 3) - 1, di = (int)(lane / 3) - 1;
        const uint32_t ncg = (cg + n_cgroups + (uint32_t)dj) % n_cgroups;
        int nrb = (int)rb + di;
        bool need = lane < 9;
        if (nrb < 0 || nrb >= (int)n_rblocks) {
            if (wrap_rows) nrb = nrb < 0 ? nrb + (int)n_rblocks : nrb - (int)n_rblocks;
            else need = false;
        }
        const uint32_t *tp = chain.tokens + (need ? (uint32_t)nrb * n_cgroups + ncg : 0u);
        uint32_t v, spins = 0;
        unsigned long long t0 = 0;
        while (true) {
            asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(tp) : "memory");
            if (__all_sync(0xffffffffu, !need || (int32_t)(v - chain.want) >= 0)) break;
            if (spins == 0) t0 = globaltimer_ns();
            if ((++spins & 255u) == 0 && __any_sync(0xffffffffu, wait_expired(t0, ALARM_LIFE_TOKEN))) {
                wait_ok = false;
                if (lane == 0) raise_alarm(ALARM_LIFE_TOKEN);
                break;
            }
        }
    }

    const int wi = (int)(cg * TB_COLS + lane) - 1;
    const uint32_t wcol = wi < 0 ? (uint32_t)(wi + (int)W) : ((uint32_t)wi >= W ? (uint32_t)wi - W : (uint32_t)wi);
    const bool store_ok = warp_ok && wait_ok && lane >= 1 && lane <= TB_COLS && (uint32_t)wi < W;
    const int r0 = (int)(rb * rpt);
    const int r1 = (r0 + (int)rpt < (int)rows) ? r0 + (int)rpt : (int)rows;
    const int irows = (int)rows;
    const int rstart = r0 - K;
    const int n_steps = (int)rpt + 2 * K;                       // same trip count for every warp
    const int s_lo = wrap_rows ? 0 : (rstart < 0 ? -rstart : 0);
    const int last = (wrap_rows || r1 + K < irows) ? r1 + K : irows;
    const uint32_t span = (uint32_t)(last - rstart - s_lo);
    const uint32_t out_rows = (uint32_t)(r1 - r0);
    int rw = (rstart % irows + irows) % irows;                  // in [0, rows) also when rows < K (see life_tb_kernel)
    const uint32_t *ip = in + wcol;
    uint32_t *op = out + (store_ok ? (uint32_t)wi : 0u);
    const uint32_t r0W = (uint32_t)r0 * W;

    Win win[K];
#pragma unroll
    for (int g = 0; g < K; ++g) win[g] = Win{0, 0, 0, 0, 0, 0, 0};

    auto load = [&](uint32_t (&raw)[TB2_UNROLL], int s0) {
#pragma unroll
        for (int u = 0; u < TB2_UNROLL; ++u) {
            const uint32_t ru = umin((uint32_t)rw + u, (uint32_t)rw + u - rows);
            raw[u] = 0;
            if ((uint32_t)(s0 + u - s_lo) < span) raw[u] = __ldg(ip + ru * W);
        }
        rw += TB2_UNROLL;
        rw = rw >= irows ? rw - irows : rw;
    };
    uint32_t acc[(K + 1) / 2] = {};
    const PopWin pw = POP ? pop_window(popc, r0, r1, K) : PopWin{0, 0};

    constexpr int PRO_STEPS = (2 * K + TB2_UNROLL - 1) / TB2_UNROLL * TB2_UNROLL;   // start-up: levels come in one by one
    constexpr int CNT = POP ? 1 : 0;
    int s0 = 0;
    // software pipeline: the rows of block i + 1 are requested before block i is computed (two row buffers)
    uint32_t ra[TB2_UNROLL], rbuf[TB2_UNROLL];
    load(ra, 0);
    for (; s0 < PRO_STEPS && s0 < n_steps; s0 += 2 * TB2_UNROLL) {
        load(rbuf, s0 + TB2_UNROLL);
        tb2_block<K, true, CNT>(ra, win, s0, op, r0W, W, store_ok, out_rows, acc, pw);
        load(ra, s0 + 2 * TB2_UNROLL);
        tb2_block<K, true, CNT>(rbuf, win, s0 + TB2_UNROLL, op, r0W, W, store_ok, out_rows, acc, pw);
    }
    for (; s0 < n_steps; s0 += 2 * TB2_UNROLL) {
        load(rbuf, s0 + TB2_UNROLL);
        tb2_block<K, false, CNT>(ra, win, s0, op, r0W, W, store_ok, out_rows, acc, pw);
        load(ra, s0 + 2 * TB2_UNROLL);
        tb2_block<K, false, CNT>(rbuf, win, s0 + TB2_UNROLL, op, r0W, W, store_ok, out_rows, acc, pw);
    }
    if constexpr (POP) pop_flush<K>(acc, popc, store_ok, lane);
    if (chain.tokens != nullptr) {
        __threadfence();
        __syncwarp();
        if (lane == 0 && warp_ok && wait_ok)
            asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(chain.tokens + rb * n_cgroups + cg),
                         "r"(chain.want + 1) : "memory");
    }
}

// Which pipeline a K-generation launch uses: true = direct (life_tb2_kernel), false = skewed (life_tb_kernel).  Measured on
// B200 (profiles/r02_sweeps.md), us per generation direct vs skewed -- one 8-GPU band of C4 (8320 x 65536): K = 2
// 28.8 / 34.8, 4: 17.8 / 23.7, 6: 17.5 / 23.6, 8: 16.2 / 16.8, 12: 16.8 / 18.2, 16: 18.8 / 18.1; 32768^2: K = 2
// 41.0 / 65.1, 4: 33.4 / 45.4, 8: 30.5 / 31.2, 16: 34.1 / 35.1.  The direct pipeline wins wherever the K levels fit
// the register file with room to overlap row steps; at K = 16 (164 registers, 3 CTAs per SM) it is a tie and the
// skewed one stays.
constexpr bool tb_direct(int K) { return K <= 12; }

// Strip length for a (rows x cols) grid.  A strip costs rpt + 3K - 1 row steps (pipeline fill), and
// the grid runs in ceil(CTAs / resident CTAs) waves of equally long CTAs; pick the candidate that
// minimises waves x steps (measured on B200, profiles/r01_sweeps.md: both effects are real, and
// fewer than ~3 waves balance badly, which the 0.97 factor for >= 3 waves encodes).
static uint32_t tb_pick_rows(uint32_t rows, uint32_t n_cgroups, int K, uint64_t slot_ctas)
{
    // candidates: a ladder of lengths plus the lengths that fill exactly one, two or three waves of resident CTAs
    uint32_t cand[16] = {96, 128, 160, 192, 224, 256, 320, 384, 448, 512, 640, 768, 1024};
    int n_cand = 13;
    for (uint64_t w = 1; w <= 3; ++w) {
        const uint64_t rb = (w * slot_ctas * (TB_THREADS / 32)) / n_cgroups;
        if (rb >= 1) cand[n_cand++] = (uint32_t)((rows + rb - 1) / rb);
    }
    uint32_t best = 256;
    double best_t = 1e30;
    for (int ci = 0; ci < n_cand; ++ci) {
        const uint32_t rpt = cand[ci];
        if (rpt < 8u * K) continue;
        const uint32_t eff = rpt < rows ? rpt : rows;
        const uint64_t warps = (uint64_t)n_cgroups * ((rows + eff - 1) / eff);
        const uint64_t ctas = (warps + TB_THREADS / 32 - 1) / (TB_THREADS / 32);
        const uint64_t waves = (ctas + slot_ctas - 1) / slot_ctas;
        double t = (double)waves * (eff + 2 * K + 2);
        if (waves >= 3) t *= 0.97;
        if (t < best_t) { best_t = t; best = eff; }
    }
    return best;
}

// Strip lengths measured by cgl_life_tune for a (rows, words per row, K) shape.
struct TunedRows { uint32_t rows, W; int K; uint32_t rpt; };
static TunedRows g_tuned[64];
static int g_n_tuned = 0;

static uint32_t tuned_rows(uint32_t rows, uint32_t W, int K)
{
    for (int i = 0; i < g_n_tuned; ++i)
        if (g_tuned[i].rows == rows && g_tuned[i].W == W && g_tuned[i].K == K) return g_tuned[i].rpt;
    return 0;
}

template <int K, bool POP>
static int launch_tb(const uint32_t *in, uint32_t *out, uint32_t rows, uint32_t cols, int wrap_rows,
                     cudaStream_t st, ChainCtx chain, PopCtx popc)
{
    static int rpt_knob = -1, occ = 0;   // per (K, POP): CGL_TB_ROWS overrides the strip length (tuning)
    if (rpt_knob < 0) {
        const char *e = getenv("CGL_TB_ROWS");
        rpt_knob = e ? atoi(e) : 0;
        int n = 0;
        if constexpr (tb_direct(K))
            CGL_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, life_tb2_kernel<K, POP>, TB_THREADS, 0));
        else
            CGL_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, life_tb_kernel<K, POP>, TB_THREADS, 0));
        occ = n > 0 ? n : 1;
    }
    const uint32_t W = cols / 32;
    const uint32_t n_cgroups = (W + TB_COLS - 1) / TB_COLS;
    uint32_t rpt = rpt_knob > 0 ? (uint32_t)rpt_knob : tuned_rows(rows, W, K);
    if (rpt == 0) rpt = tb_pick_rows(rows, n_cgroups, K, (uint64_t)sm_count() * occ);
    if (POP && rpt > TB_POP_MAX_ROWS) rpt = TB_POP_MAX_ROWS;     // 16-bit counts per thread (see PopCtx)
    if (rpt > rows) rpt = rows;
    const uint32_t n_rblocks = (rows + rpt - 1) / rpt;
    const uint64_t blocks = ((uint64_t)n_cgroups * n_rblocks + TB_THREADS / 32 - 1) / (TB_THREADS / 32);
    CGL_REQUIRE(blocks < (1ull << 31) && rows < (1u << 30) && (uint64_t)rows * W < (1ull << 32), CGL_E_BADARG,
                "cgl_life_run: grid too large for the k-blocked kernel (rows * cols/32 must be < 2^32)");
    // chaining needs the nine-neighbour footprint (strips at least K rows long) and a large enough token buffer
    if (chain.tokens != nullptr && (rpt < (uint32_t)K || (uint64_t)n_cgroups * n_rblocks > chain.cap)) chain.tokens = nullptr;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)blocks);
    cfg.blockDim = dim3(TB_THREADS);
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = (chain.tokens != nullptr && chain.want > 0) ? 1 : 0;        // the first launch of a run waits normally
    if constexpr (tb_direct(K))
        CGL_CUDA(cudaLaunchKernelEx(&cfg, life_tb2_kernel<K, POP>, in, out, rows, W, rpt, wrap_rows, n_cgroups, n_rblocks, chain,
                                    popc));
    else
        CGL_CUDA(cudaLaunchKernelEx(&cfg, life_tb_kernel<K, POP>, in, out, rows, W, rpt, wrap_rows, n_cgroups, n_rblocks, chain,
                                    popc));
    return 0;
}

// popc.pop == nullptr: the uncounted kernels.
static int tb_dispatch(int k, const uint32_t *in, uint32_t *out, uint32_t rows, uint32_t cols, int wrap_rows,
                       cudaStream_t st, ChainCtx chain, PopCtx popc)
{
#define CGL_TB_CASE(KK)                                                                     \
    case KK: return popc.pop ? launch_tb<KK, true>(in, out, rows, cols, wrap_rows, st, chain, popc) \
                             : launch_tb<KK, false>(in, out, rows, cols, wrap_rows, st, chain, popc)
    switch (k) {
        CGL_TB_CASE(2); CGL_TB_CASE(3); CGL_TB_CASE(4);
        CGL_TB_CASE(6); CGL_TB_CASE(8); CGL_TB_CASE(12); CGL_TB_CASE(16);
    }
#undef CGL_TB_CASE
    set_error("cgl_life_run: no temporal-blocking kernel for k=%d", k);
    return CGL_E_BADARG;
}

// Token buffers of the chained launches, one per (device, stream) so that concurrent streams do not
// share tokens.  Returns nullptr when chaining is off (CGL_TB_CHAIN=0) or no buffer can be had.
static uint32_t *chain_tokens(cudaStream_t st, uint32_t rows, uint32_t cols, uint32_t *cap_out)
{
    struct TokenBuf { int dev; cudaStream_t st; uint32_t *p; uint32_t cap; };
    static TokenBuf bufs[16] = {};
    static int n_bufs = 0, chain_on = -1;
    if (chain_on < 0) {
        const char *e = getenv("CGL_TB_CHAIN");
        chain_on = (e && e[0] == '0') ? 0 : 1;
    }
    int dev = 0;
    if (!chain_on || cudaGetDevice(&dev) != cudaSuccess) return nullptr;
    const uint32_t max_strips = ((cols / 32 + TB_COLS - 1) / TB_COLS) * ((rows + 95) / 96 + 1);
    TokenBuf *tb = nullptr;
    for (int i = 0; i < n_bufs; ++i)
        if (bufs[i].dev == dev && bufs[i].st == st) tb = &bufs[i];
    if (tb == nullptr && n_bufs < 16) {
        tb = &bufs[n_bufs++];
        *tb = TokenBuf{dev, st, nullptr, 0};
    }
    if (tb == nullptr) return nullptr;
    if (tb->cap < max_strips) {
        if (tb->p) cudaFree(tb->p);
        tb->p = nullptr;
        tb->cap = 0;
        if (cudaMalloc(&tb->p, (size_t)max_strips * 4) == cudaSuccess) tb->cap = max_strips;
        else cudaGetLastError();
    }
    *cap_out = tb->cap;
    return tb->p;
}

// pop += live cells of the n_words words starting at w (rows of W words; the last word of a row keeps the bits of
// tail_mask): the population of a count window after a generation that ran outside the k-blocked kernels.
__global__ void window_pop_kernel(const uint32_t *__restrict__ w, uint64_t n_words, uint32_t W, uint32_t tail_mask,
                                  unsigned long long *__restrict__ pop)
{
    unsigned acc = 0;
    const uint64_t nthr = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n_words; i += nthr) {
        uint32_t v = __ldg(w + i);
        if (i % W == W - 1) v &= tail_mask;
        acc += __popc(v);
    }
    acc = __reduce_add_sync(0xffffffffu, acc);
    if ((threadIdx.x & 31) == 0 && acc != 0) atomicAdd(pop, (unsigned long long)acc);
}

static int window_pop(const uint32_t *grid, uint32_t cols, uint32_t row0, uint32_t n_rows, unsigned long long *pop,
                      cudaStream_t st)
{
    const uint32_t W = (cols + 31) / 32;
    const uint64_t n_words = (uint64_t)n_rows * W;
    const uint32_t tail_mask = cols % 32 ? (1u << (cols % 32)) - 1u : 0xffffffffu;
    const unsigned threads = 256;
    uint64_t bx = (n_words + threads * 4 - 1) / (threads * 4);
    const uint64_t cap = (uint64_t)sm_count() * 8;
    bx = bx < 1 ? 1 : (bx > cap ? cap : bx);
    window_pop_kernel<<<(unsigned)bx, threads, 0, st>>>(grid + (uint64_t)row0 * W, n_words, W, tail_mask, pop);
    CGL_LAUNCH_CHECK();
    return 0;
}

CGL_DEFINE_TU_HOOKS(life_tb)

}  // namespace cgl

using namespace cgl;

extern "C" int cgl_life_step(const uint32_t *in, uint32_t *out, uint64_t n_envs, uint32_t rows,
                             uint32_t cols, int wrap_rows, uint32_t *alive_out, cgl_stream_t stream);

// Test hook (tests/test_gpu_waits.py): which = 1 makes the next chained cgl_life_run wait for strip tokens that
// are never published, so that the bounded wait, the alarm word and the "store nothing" path can be exercised.
static int g_fault_next_chain = 0;
extern "C" int cgl_test_fault(int which)
{
    CGL_REQUIRE(which == 1, CGL_E_BADARG, "cgl_test_fault: unknown fault %d", which);
    g_fault_next_chain = 1;
    return 0;
}

// k generations per launch where a kernel exists for the block size, else smaller blocks.
// With wrap_rows = 0 the k rows next to each open edge are a ghost zone: their contents after a
// k-blocked launch are unspecified (they differ from k single steps); every row at least k rows
// away from an open edge is exact.
// pop != nullptr (cgl_life_run_pop): pop[i] += live cells of rows [row0, row0 + n_rows) after generation i + 1.
static int life_run(uint32_t *buf_a, uint32_t *buf_b, uint32_t rows, uint32_t cols, int wrap_rows, uint32_t gens,
                    uint32_t k, int *result_in_a_out, cgl_stream_t stream, unsigned long long *pop, uint32_t row0,
                    uint32_t n_rows)
{
    CGL_REQUIRE(buf_a && buf_b && rows && cols && buf_a != buf_b, CGL_E_BADARG, "cgl_life_run: bad argument");
    CGL_REQUIRE(k >= 1 && k <= 16, CGL_E_BADARG, "cgl_life_run: k must be in 1..16");
    cudaStream_t st = as_stream(stream);
    if (pop != nullptr && gens > 0) CGL_CUDA(cudaMemsetAsync(pop, 0, (size_t)gens * sizeof(*pop), st));
    static const int sizes[] = {16, 12, 8, 6, 4, 3, 2, 1};
    uint32_t *src = buf_a, *dst = buf_b;
    uint32_t left = gens;
    const bool tiled = cols % 32 == 0 && cols >= 32 * TB_COLS && rows >= 8;
    uint32_t token_cap = 0;
    uint32_t *token_buf = (tiled && k > 1) ? chain_tokens(st, rows, cols, &token_cap) : nullptr;
    const bool chain_ok = token_buf != nullptr;
    int prev_step = 0;
    uint32_t chained = 0;                 // launches of the current chain so far
    while (left > 0) {
        int step = 1;
        if (tiled && k > 1) {
            for (int s : sizes)
                if ((uint32_t)s <= k && (uint32_t)s <= left) { step = s; break; }
        }
        int rc;
        if (step == 1) {
            rc = cgl_life_step(src, dst, 1, rows, cols, wrap_rows, nullptr, stream);
            if (rc == 0 && pop != nullptr) rc = window_pop(dst, cols, row0, n_rows, pop + (gens - left), st);
            prev_step = 0;
        } else {
            ChainCtx chain{nullptr, 0, 0};
            if (chain_ok) {
                if (step != prev_step) {   // new geometry: start a new chain behind everything queued so far
                    CGL_CUDA(cudaMemsetAsync(token_buf, 0, (size_t)token_cap * 4, st));
                    chained = g_fault_next_chain ? 1000u : 0u;      // test hook: tokens that can never arrive
                    g_fault_next_chain = 0;
                }
                chain = ChainCtx{token_buf, chained, token_cap};
            }
            const PopCtx popc{pop != nullptr ? pop + (gens - left) : nullptr, row0, row0 + n_rows};
            rc = tb_dispatch(step, src, dst, rows, cols, wrap_rows, st, chain, popc);
            prev_step = step;
            ++chained;
        }
        if (rc) return rc;
        uint32_t *t = src; src = dst; dst = t;
        left -= (uint32_t)step;
    }
    if (result_in_a_out) *result_in_a_out = (src == buf_a) ? 1 : 0;
    return 0;
}

extern "C" int cgl_life_run(uint32_t *buf_a, uint32_t *buf_b, uint32_t rows, uint32_t cols,
                            int wrap_rows, uint32_t gens, uint32_t k, int *result_in_a_out,
                            cgl_stream_t stream)
{
    return life_run(buf_a, buf_b, rows, cols, wrap_rows, gens, k, result_in_a_out, stream, nullptr, 0, 0);
}

extern "C" int cgl_life_run_pop(uint32_t *buf_a, uint32_t *buf_b, uint32_t rows, uint32_t cols, int wrap_rows,
                                uint32_t gens, uint32_t k, uint32_t count_row0, uint32_t count_rows, uint64_t *pop_out,
                                int *result_in_a_out, cgl_stream_t stream)
{
    CGL_REQUIRE(pop_out != nullptr, CGL_E_BADARG, "cgl_life_run_pop: pop_out_dev is NULL");
    CGL_REQUIRE(count_rows > 0, CGL_E_BADARG, "cgl_life_run_pop: count_rows must be at least 1");
    CGL_REQUIRE((uint64_t)count_row0 + count_rows <= rows, CGL_E_BADARG,
                "cgl_life_run_pop: count window [%u, %u + %u) is not inside the %u rows", count_row0, count_row0,
                count_rows, rows);
    static_assert(sizeof(unsigned long long) == sizeof(uint64_t), "pop_out is uint64");
    return life_run(buf_a, buf_b, rows, cols, wrap_rows, gens, k, result_in_a_out, stream,
                    reinterpret_cast<unsigned long long *>(pop_out), count_row0, count_rows);
}

// Measure the strip length for this shape on the caller's buffers (buf_b is clobbered) and remember
// the fastest; later cgl_life_run calls with the same (rows, cols, k) use it.  Synchronises the
// stream; call it once at set-up, never inside a capture.
extern "C" int cgl_life_tune(uint32_t *buf_a, uint32_t *buf_b, uint32_t rows, uint32_t cols, int wrap_rows,
                             uint32_t k, cgl_stream_t stream)
{
    CGL_REQUIRE(buf_a && buf_b && buf_a != buf_b && rows && cols, CGL_E_BADARG, "cgl_life_tune: bad argument");
    if (!(cols % 32 == 0 && cols >= 32 * TB_COLS && rows >= 8) || k < 2) return 0;    // nothing to tune
    int kk = 1;
    for (int sz : {16, 12, 8, 6, 4, 3, 2})
        if ((uint32_t)sz <= k) { kk = sz; break; }
    const uint32_t W = cols / 32;
    if (tuned_rows(rows, W, kk) != 0 || g_n_tuned >= 64) return 0;
    cudaStream_t st = as_stream(stream);
    cudaEvent_t e0, e1;
    CGL_CUDA(cudaEventCreate(&e0));
    CGL_CUDA(cudaEventCreate(&e1));
    uint32_t cand[16] = {96, 128, 160, 192, 224, 256, 320, 384, 512, 640, 768};
    int n_cand = 11;
    {
        int occ = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, life_tb2_kernel<8, false>, TB_THREADS, 0) != cudaSuccess || occ <= 0) {
            cudaGetLastError();
            occ = 5;
        }
        const uint32_t n_cg = (W + TB_COLS - 1) / TB_COLS;
        for (uint64_t w = 1; w <= 3; ++w) {              // exactly w waves of resident CTAs
            const uint64_t rb = (w * (uint64_t)sm_count() * occ * (TB_THREADS / 32)) / n_cg;
            if (rb >= 1) cand[n_cand++] = (uint32_t)((rows + rb - 1) / rb);
        }
    }
    float best_ms = 1e30f;
    uint32_t best = 0;
    TunedRows &slot = g_tuned[g_n_tuned];
    slot = TunedRows{rows, W, kk, 0};
    ++g_n_tuned;                                   // visible to launch_tb through tuned_rows()
    uint32_t token_cap = 0;
    uint32_t *token_buf = chain_tokens(st, rows, cols, &token_cap);
    for (int ci = 0; ci < n_cand; ++ci) {
        const uint32_t rpt = cand[ci];
        if (rpt < 8u * kk || rpt > rows) continue;
        slot.rpt = rpt;
        // time 4 launches chained like cgl_life_run chains them (all a -> b: every launch writes the same
        // values, so re-running a strip early is harmless); the first one doubles as warm-up
        if (token_buf) CGL_CUDA(cudaMemsetAsync(token_buf, 0, (size_t)token_cap * 4, st));
        int rc = tb_dispatch(kk, buf_a, buf_b, rows, cols, wrap_rows, st, ChainCtx{token_buf, 0, token_cap}, PopCtx{});
        if (rc) return rc;
        CGL_CUDA(cudaEventRecord(e0, st));
        for (uint32_t rep = 1; rep <= 4; ++rep)
            if ((rc = tb_dispatch(kk, buf_a, buf_b, rows, cols, wrap_rows, st, ChainCtx{token_buf, rep, token_cap}, PopCtx{})))
                return rc;
        CGL_CUDA(cudaEventRecord(e1, st));
        CGL_CUDA(cudaEventSynchronize(e1));
        float ms = 0;
        CGL_CUDA(cudaEventElapsedTime(&ms, e0, e1));
        if (ms < best_ms) { best_ms = ms; best = rpt; }
    }
    slot.rpt = best;
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    if (best == 0) --g_n_tuned;
    return 0;
}
