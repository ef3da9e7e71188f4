// cgl_life_persist.cu -- life mode, many k-generation sub-steps in ONE cooperative launch.
//
// Reference semantics: repeated application of the world half of kernel `run`
// (/root/reference/CGL/CGL.py:154-170) on a torus the reference cannot even index (BASELINE.json configs[3], [4]).
//
// cgl_life_tb.cu runs K generations per launch (time-skewed register pipeline, one HBM pass) and chains the
// launches strip by strip.  What that leaves on the table shows where a GPU's share of the grid is small (the
// 8-GPU row bands of C4: 8192 + 128 rows = ONE wave of strips per launch): every launch boundary is a ramp, every
// halo exchange a kernel of its own on the compute stream.  Here a strip is owned by ONE WARP FOR THE WHOLE CALL:
//   * the grid is sized to what is co-resident (cooperative launch: the runtime refuses anything else), a warp
//     loops over the sub-steps of K generations each, ping-ponging between the two band buffers;
//   * sub-step s of strip (cg, rb) waits for sub-step s-1 of its 3 x 3 neighbour strips (their outputs are its
//     inputs, and it overwrites what they read) through per-strip tokens -- neighbours only, never the whole grid;
//   * HALO (row bands over NVLink, one process per GPU): every `sub_per_block` sub-steps the strips that own the
//     first / last `ghost` owned rows store them into the ring neighbours' LANDING ZONES (CUDA-IPC mapped peer
//     memory, two slots alternating by block) and bump an arrival counter (system-scope release); a strip whose
//     read footprint touches ghost rows waits for the counter and copies what it is about to read from its own
//     landing zone into the band buffer.  No exchange launch, no host round trip: interior strips never wait for
//     a neighbour GPU, so the exchange overlaps the interior by construction.  The hot row loop is the same in
//     both variants (the exchange happens between sub-steps), so HALO costs no registers.
// The pipeline fill (3K - 1 row steps per strip and sub-step) is still paid; longer strips make it small on one
// GPU (65536 rows / 42 strips), on an 8192-row band it is what remains (DESIGN.md section 4.6).
#include <cooperative_groups.h>
#include <stdlib.h>

#include "cgl_internal.cuh"

namespace cgl {

struct PWin {           // window of one level: rows (a-1, a) of the level's input generation (see cgl_life_tb.cu)
    uint32_t us0, us1;
    uint32_t ms0, ms1, mt0, mt1, mc;
};

constexpr int PB_UNROLL = 6;
constexpr int PB_COLS = 30;
constexpr int PB_THREADS = 128;

__device__ __forceinline__ void pst_if_lt(uint32_t *p, uint32_t v, bool ok, uint32_t a, uint32_t b)
{
    asm volatile(
        "{\n\t.reg .pred p, q;\n\t"
        "setp.lt.u32 p, %2, %3;\n\t"
        "setp.ne.u32 q, %4, 0;\n\t"
        "and.pred p, p, q;\n\t"
        "@p st.global.u32 [%0], %1;\n\t}"
        ::"l"(p), "r"(v), "r"(a), "r"(b), "r"((uint32_t)ok) : "memory");
}

struct PersistHalo {
    uint32_t ghost;                       // ghost depth; owned rows are [ghost, rows - ghost)
    uint32_t sub_per_block;               // sub-steps between exchanges (ghost / K)
    uint32_t blk0;                        // global index of the first block of this call (= pushes consumed so far)
    uint32_t n_top, n_bot;                // strips (all column groups) that own rows of the top / bottom edge range
    uint32_t initial_push;                // push the INPUT's edge rows before the first sub-step (fresh grid)
    uint32_t *peer_up_landing[2], *peer_dn_landing[2];       // per slot: where my first / last owned rows land
    uint32_t *peer_up_ctr, *peer_dn_ctr;                     // the neighbours' arrival counters
    const uint32_t *my_landing_up[2], *my_landing_dn[2];     // per slot: rows for my top / bottom ghost rows
    const uint32_t *my_ctr_up, *my_ctr_dn;                   // my arrival counters (bumped by the neighbours)
};

// Every exit of a wait is a warp vote, so the warp stays convergent for the shuffles of the row loop.
// Returns false if the wait was abandoned (deadline, or another warp already gave up).
__device__ __forceinline__ bool pwait(const uint32_t *p, uint32_t target, bool need, bool sys, uint32_t *abort_flag,
                                      int alarm_word)
{
    uint32_t v, spins = 0;
    unsigned long long t0 = 0;
    while (true) {
        if (sys) asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
        else asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
        if (__all_sync(0xffffffffu, !need || (int32_t)(v - target) >= 0)) return true;
        if (spins == 0) t0 = globaltimer_ns();
        if ((++spins & 127u) == 0) {
            const bool give_up = wait_expired(t0, alarm_word) || *reinterpret_cast<volatile uint32_t *>(abort_flag) != 0;
            if (__any_sync(0xffffffffu, give_up)) return false;
        }
    }
}

// Everything a warp needs to know about its strip, derived from its warp index and the kernel parameters.  The
// persistent kernel RECOMPUTES this before and after every pass (from an "opaque" copy of the warp index, so that
// the compiler cannot hoist it out of the pass loop): the row loop's pipeline state fills the register file, and
// whatever else lived across it was spilled inside the loop (measured: 43 instead of 31 us per generation at 32768^2).
struct StripGeom {
    uint32_t lane, cg, rb, wcol;
    int wi, r0, r1;
    bool warp_ok, store_lane;
};

__device__ __forceinline__ StripGeom strip_geom(uint32_t W, uint32_t rows, uint32_t rpt, uint32_t n_cgroups, uint32_t n_rblocks)
{
    uint32_t warp;
    asm volatile("{\n\t.reg .u32 c, t;\n\tmov.u32 c, %%ctaid.x;\n\tmov.u32 t, %%tid.x;\n\tshr.u32 t, t, 5;\n\t"
                 "mad.lo.u32 %0, c, %1, t;\n\t}" : "=r"(warp) : "r"((uint32_t)(PB_THREADS / 32)));
    StripGeom g;
    g.lane = threadIdx.x & 31;
    g.cg = warp % n_cgroups;
    uint32_t rb = warp / n_cgroups;
    g.warp_ok = rb < n_rblocks;                            // padding warps shadow the last strip with stores off
    g.rb = g.warp_ok ? rb : n_rblocks - 1;
    g.wi = (int)(g.cg * PB_COLS + g.lane) - 1;             // word column of this lane (may be -1 or >= W)
    g.wcol = g.wi < 0 ? (uint32_t)(g.wi + (int)W) : ((uint32_t)g.wi >= W ? (uint32_t)g.wi - W : (uint32_t)g.wi);
    g.store_lane = g.warp_ok && g.lane >= 1 && g.lane <= PB_COLS && (uint32_t)g.wi < W;
    g.r0 = (int)(g.rb * rpt);
    g.r1 = (g.r0 + (int)rpt < (int)rows) ? g.r0 + (int)rpt : (int)rows;
    return g;
}

// 5 CTAs (20 warps) per SM like the launch-per-pass kernel (K <= 8).
template <int K, bool HALO>
__global__ void __launch_bounds__(PB_THREADS, K <= 8 ? 5 : 3)
life_persist_kernel(uint32_t *buf_a, uint32_t *buf_b, uint32_t rows, uint32_t W, uint32_t rpt, int wrap_rows,
                    uint32_t n_cgroups, uint32_t n_rblocks, uint32_t n_sub, uint32_t *tokens, uint32_t token_base,
                    uint32_t *abort_flag, const PersistHalo h)
{
    const int irows = (int)rows;
    const uint32_t own_lo = HALO ? h.ghost : 0u, own_hi = HALO ? rows - h.ghost : rows;

    // my first owned rows -> the upper neighbour's bottom ghost rows; my last owned rows -> the lower one's top
    auto push_edges = [&](const StripGeom &g, const uint32_t *src, uint32_t slot) {
        const int pu0 = max(g.r0, (int)own_lo), pu1 = min(g.r1, (int)(own_lo + h.ghost));
        const int pd0 = max(g.r0, (int)(own_hi - h.ghost)), pd1 = min(g.r1, (int)own_hi);
        const bool push_up = g.warp_ok && pu0 < pu1, push_dn = g.warp_ok && pd0 < pd1;
        if (!(push_up || push_dn)) return;                 // warp-uniform
        uint32_t *lu = slot ? h.peer_up_landing[1] : h.peer_up_landing[0];
        uint32_t *ld = slot ? h.peer_dn_landing[1] : h.peer_dn_landing[0];
        if (push_up && g.store_lane)
            for (int r = pu0; r < pu1; ++r)
                lu[(uint32_t)(r - (int)own_lo) * W + (uint32_t)g.wi] = __ldcg(src + (uint32_t)r * W + (uint32_t)g.wi);
        if (push_dn && g.store_lane)
            for (int r = pd0; r < pd1; ++r)
                ld[(uint32_t)(r - (int)(own_hi - h.ghost)) * W + (uint32_t)g.wi] = __ldcg(src + (uint32_t)r * W + (uint32_t)g.wi);
        __threadfence_system();                      // my peer stores are visible system-wide ...
        __syncwarp();
        if (g.lane == 0) {                           // ... before the arrival is published
            if (push_up) asm volatile("red.release.sys.global.add.u32 [%0], 1;" ::"l"(h.peer_up_ctr) : "memory");
            if (push_dn) asm volatile("red.release.sys.global.add.u32 [%0], 1;" ::"l"(h.peer_dn_ctr) : "memory");
        }
    };

    bool alive = true;                               // warp-uniform: false once a wait was abandoned
    if (HALO && h.initial_push) push_edges(strip_geom(W, rows, rpt, n_cgroups, n_rblocks), buf_a, h.blk0 & 1u);

    for (uint32_t s = 0; s < n_sub; ++s) {
        uint32_t *in = (s & 1u) ? buf_b : buf_a, *out = (s & 1u) ? buf_a : buf_b;
        const uint32_t *ip;
        uint32_t *op;
        uint32_t span, out_rows, ro0;
        int n_steps, s_lo, rw;
        bool store_ok;
        {
            // ---- cold prologue: dependencies, halo copy-in, row-loop operands --------------------------------
            const StripGeom g = strip_geom(W, rows, rpt, n_cgroups, n_rblocks);
            // the 3 x 3 neighbour strips have finished pass s - 1: lanes 0..8 watch one each
            const int dj = (int)(g.lane % 3) - 1, di = (int)(g.lane / 3) - 1;
            const uint32_t ncg = (g.cg + n_cgroups + (uint32_t)dj) % n_cgroups;
            int nrb = (int)g.rb + di;
            bool need = g.lane < 9;
            if (nrb < 0 || nrb >= (int)n_rblocks) {
                if (wrap_rows) nrb = nrb < 0 ? nrb + (int)n_rblocks : nrb - (int)n_rblocks;
                else need = false;
            }
            const uint32_t *tp = tokens + (need ? (uint32_t)nrb * n_cgroups + ncg : 0u);
            if (alive && !pwait(tp, token_base + s, need, false, abort_flag, ALARM_LIFE_TOKEN)) {
                alive = false;
                if (g.lane == 0) { *reinterpret_cast<volatile uint32_t *>(abort_flag) = 1u; raise_alarm(ALARM_LIFE_TOKEN); }
            }
            const int f0 = g.r0 - K < 0 ? 0 : g.r0 - K, f1 = g.r1 + K > irows ? irows : g.r1 + K;   // read footprint
            const bool reads_up = HALO && f0 < (int)own_lo, reads_dn = HALO && f1 > (int)own_hi;
            if (HALO && alive && s % h.sub_per_block == 0 && (reads_up || reads_dn)) {
                // block start: the neighbours' edge rows have arrived; copy what I am about to read
                const uint32_t blk = h.blk0 + s / h.sub_per_block, slot = blk & 1u;
                bool ok = true;
                if (reads_up) ok = pwait(h.my_ctr_up, (blk + 1u) * h.n_bot, g.lane == 0, true, abort_flag, ALARM_HALO);
                if (ok && reads_dn) ok = pwait(h.my_ctr_dn, (blk + 1u) * h.n_top, g.lane == 0, true, abort_flag, ALARM_HALO);
                if (!ok) {
                    alive = false;
                    if (g.lane == 0) { *reinterpret_cast<volatile uint32_t *>(abort_flag) = 1u; raise_alarm(ALARM_HALO); }
                } else {
                    const uint32_t *lu = slot ? h.my_landing_up[1] : h.my_landing_up[0];
                    const uint32_t *ld = slot ? h.my_landing_dn[1] : h.my_landing_dn[0];
                    if (reads_up)
                        for (int r = f0; r < (int)own_lo; ++r) in[(uint32_t)r * W + g.wcol] = __ldcg(lu + (uint32_t)r * W + g.wcol);
                    if (reads_dn)
                        for (int r = max(f0, (int)own_hi); r < f1; ++r)
                            in[(uint32_t)r * W + g.wcol] = __ldcg(ld + (uint32_t)(r - (int)own_hi) * W + g.wcol);
                    __syncwarp();
                }
            }
            const int rstart = g.r0 - K;
            n_steps = (int)rpt + 3 * K - 1;
            s_lo = wrap_rows ? 0 : (rstart < 0 ? -rstart : 0);
            const int last = (wrap_rows || g.r1 + K < irows) ? g.r1 + K : irows;
            span = (uint32_t)(last - rstart - s_lo);
            out_rows = (uint32_t)(g.r1 - g.r0);
            ro0 = (uint32_t)g.r0;
            rw = (rstart % irows + irows) % irows;   // in [0, rows) also when rows < K (see life_tb_kernel)
            ip = in + g.wcol;
            op = out + (g.store_lane ? (uint32_t)g.wi : 0u);
            store_ok = g.store_lane && alive;
        }

        // ---- K generations: the time-skewed register pipeline of cgl_life_tb.cu ----------------------------
        {
            PWin win[K];
            uint32_t pend[K];
#pragma unroll
            for (int g = 0; g < K; ++g) {
                win[g] = PWin{0, 0, 0, 0, 0, 0, 0};
                pend[g] = 0;
            }
            for (int s0 = 0; s0 < n_steps; s0 += PB_UNROLL) {
                uint32_t raw[PB_UNROLL];
#pragma unroll
                for (int u = 0; u < PB_UNROLL; ++u) {
                    const uint32_t ru = umin((uint32_t)rw + u, (uint32_t)rw + u - rows);      // (rw + u) mod rows
                    raw[u] = 0;
                    if ((uint32_t)(s0 + u - s_lo) < span) raw[u] = __ldcg(ip + ru * W);         // written by other SMs: L2
                }
                rw += PB_UNROLL;
                rw = rw >= irows ? rw - irows : rw;
#pragma unroll
                for (int u = 0; u < PB_UNROLL; ++u) {
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
                    }
                    const uint32_t so = (uint32_t)(s0 + u - (3 * K - 1));
                    pst_if_lt(op + (ro0 + so) * W, pend[K - 1], store_ok, so, out_rows);
                }
            }
        }

        // ---- cold epilogue: publish, exchange ----------------------------------------------------------------
        {
            const StripGeom g = strip_geom(W, rows, rpt, n_cgroups, n_rblocks);
            __threadfence();                             // this strip's rows are visible device-wide ...
            __syncwarp();
            if (g.lane == 0 && g.warp_ok && alive)       // ... before its token is published
                asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(tokens + g.rb * n_cgroups + g.cg),
                             "r"(token_base + s + 1u) : "memory");
            if (HALO && alive && ((s + 1u) % h.sub_per_block == 0 || s + 1u == n_sub))
                push_edges(g, out, (h.blk0 + s / h.sub_per_block + 1u) & 1u);
        }
    }
}

CGL_DEFINE_TU_HOOKS(life_persist)

// Token / abort storage per (device, stream), grown on demand.
struct PersistScratch { int dev; cudaStream_t st; uint32_t *p; uint32_t cap; };
static PersistScratch g_scratch[16] = {};
static int g_n_scratch = 0;

static uint32_t *persist_scratch(cudaStream_t st, uint32_t n_tokens)
{
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return nullptr;
    PersistScratch *sc = nullptr;
    for (int i = 0; i < g_n_scratch; ++i)
        if (g_scratch[i].dev == dev && g_scratch[i].st == st) sc = &g_scratch[i];
    if (sc == nullptr && g_n_scratch < 16) {
        sc = &g_scratch[g_n_scratch++];
        *sc = PersistScratch{dev, st, nullptr, 0};
    }
    if (sc == nullptr) return nullptr;
    if (sc->cap < n_tokens + 1) {
        if (sc->p) cudaFree(sc->p);
        sc->p = nullptr;
        sc->cap = 0;
        if (cudaMalloc(&sc->p, (size_t)(n_tokens + 1) * 4) == cudaSuccess) sc->cap = n_tokens + 1;
        else cudaGetLastError();
    }
    return sc->p;
}

// Opt-in (CGL_LIFE_PERSIST=1) for plain cgl_life_run: measured on B200 the persistent kernel is SLOWER than one
// launch per pass (32768^2, K = 8: 42.9 vs 30.8 us per generation; one 8-GPU band of C4 as a ring of one: 22.2 vs
// 16.2) -- keeping the strip bookkeeping alive across the row loop costs registers the pipeline needs (96 are all
// taken), and a single wave of strips in lock step exposes every load latency.  The in-kernel exchange
// (cgl_life_band_run, RowBandLife(exchange="persist")) stays available and tested; it is not the default.
static int persist_enabled()
{
    static int v = -1;
    if (v < 0) {
        const char *e = getenv("CGL_LIFE_PERSIST");
        v = (e && e[0] == '1') ? 1 : 0;
    }
    return v;
}

// Geometry of a persistent run: as many row blocks as stay co-resident.  Returns 0 if the shape does not fit.
template <int K, bool HALO>
static int persist_geometry(uint32_t rows, uint32_t W, uint32_t *rpt_out, uint32_t *n_cg_out, uint32_t *n_rb_out,
                            unsigned *blocks_out)
{
    static int occ = 0;
    if (occ == 0) {
        int n = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, life_persist_kernel<K, HALO>, PB_THREADS, 0) != cudaSuccess || n <= 0) {
            cudaGetLastError();
            return 0;
        }
        occ = n;
    }
    static int rb_knob = -1;                    // CGL_PERSIST_RBLOCKS overrides the number of row blocks (tuning)
    if (rb_knob < 0) {
        const char *e = getenv("CGL_PERSIST_RBLOCKS");
        rb_knob = e ? atoi(e) : 0;
    }
    const uint32_t n_cg = (W + PB_COLS - 1) / PB_COLS;
    const uint64_t cap_warps = (uint64_t)sm_count() * occ * (PB_THREADS / 32);
    uint32_t n_rb = (uint32_t)(cap_warps / n_cg);
    if (rb_knob > 0 && (uint32_t)rb_knob < n_rb) n_rb = (uint32_t)rb_knob;
    if (n_rb == 0) return 0;
    uint32_t rpt = (rows + n_rb - 1) / n_rb;
    if (rpt < (uint32_t)(2 * K)) rpt = 2 * K;   // the nine-neighbour footprint needs strips of at least K rows
    if (rpt > rows) rpt = rows;
    n_rb = (rows + rpt - 1) / rpt;
    if ((uint64_t)rows * W >= (1ull << 32) || rows >= (1u << 30)) return 0;
    *rpt_out = rpt; *n_cg_out = n_cg; *n_rb_out = n_rb;
    *blocks_out = (unsigned)(((uint64_t)n_cg * n_rb + PB_THREADS / 32 - 1) / (PB_THREADS / 32));
    return 1;
}

template <int K, bool HALO>
static int launch_persist(uint32_t *a, uint32_t *b, uint32_t rows, uint32_t cols, int wrap_rows, uint32_t n_sub,
                          PersistHalo h, cudaStream_t st)
{
    uint32_t rpt, n_cg, n_rb;
    unsigned blocks;
    if (!persist_geometry<K, HALO>(rows, cols / 32, &rpt, &n_cg, &n_rb, &blocks)) return -100;
    uint32_t *scratch = persist_scratch(st, n_cg * n_rb);
    if (scratch == nullptr) return -100;
    if (HALO) {
        // strips (per column group) that own rows of the top / bottom edge range -- the same on every rank
        auto touching = [&](uint32_t lo, uint32_t hi) { return (hi - 1) / rpt - lo / rpt + 1; };
        h.n_top = touching(h.ghost, 2 * h.ghost) * n_cg;
        h.n_bot = touching(rows - 2 * h.ghost, rows - h.ghost) * n_cg;
    }
    CGL_CUDA(cudaMemsetAsync(scratch, 0, (size_t)(n_cg * n_rb + 1) * 4, st));
    uint32_t *tokens = scratch, *abort_flag = scratch + n_cg * n_rb;
    uint32_t W = cols / 32, token_base = 0;
    void *args[] = {&a, &b, &rows, &W, &rpt, &wrap_rows, &n_cg, &n_rb, &n_sub, &tokens, &token_base, &abort_flag, &h};
    // cooperative launch: the runtime guarantees that all CTAs are co-resident (the strips wait for each other)
    cudaError_t e = cudaLaunchCooperativeKernel((const void *)life_persist_kernel<K, HALO>, dim3(blocks), dim3(PB_THREADS),
                                                args, 0, st);
    if (e == cudaErrorCooperativeLaunchTooLarge || e == cudaErrorNotSupported) {
        cudaGetLastError();
        return -100;
    }
    CGL_CUDA(e);
    return 0;
}

// Persistent torus / open-row run: n_sub sub-steps of k generations each, a -> b -> a ...; -100 = not applicable
// (shape, k, or CGL_LIFE_PERSIST=0): the caller falls back to one launch per sub-step.
int life_persist_run(uint32_t *a, uint32_t *b, uint32_t rows, uint32_t cols, int wrap_rows, uint32_t n_sub, int k,
                     cudaStream_t st)
{
    if (!persist_enabled() || cols % 32 != 0 || cols < 32 * PB_COLS || rows < 8 || n_sub < 2) return -100;
    PersistHalo h = {};
    switch (k) {
    case 4: return launch_persist<4, false>(a, b, rows, cols, wrap_rows, n_sub, h, st);
    case 8: return launch_persist<8, false>(a, b, rows, cols, wrap_rows, n_sub, h, st);
    case 16: return launch_persist<16, false>(a, b, rows, cols, wrap_rows, n_sub, h, st);
    }
    return -100;
}

}  // namespace cgl

using namespace cgl;

// Row-band run with the halo exchange inside the kernel: see include/cgl_b200.h.
extern "C" int cgl_life_band_run(uint32_t *buf_a, uint32_t *buf_b, uint32_t buf_rows, uint32_t cols, uint32_t ghost,
                                 uint32_t k, uint32_t n_sub, uint32_t block_index, int initial_push,
                                 uint32_t *const peer_up_landing[2], uint32_t *const peer_dn_landing[2],
                                 uint32_t *peer_up_ctr, uint32_t *peer_dn_ctr, const uint32_t *const my_landing_up[2],
                                 const uint32_t *const my_landing_dn[2], const uint32_t *my_ctr_up,
                                 const uint32_t *my_ctr_dn, cgl_stream_t stream)
{
    CGL_REQUIRE(buf_a && buf_b && buf_a != buf_b && peer_up_landing && peer_dn_landing && peer_up_ctr && peer_dn_ctr &&
                    my_landing_up && my_landing_dn && my_ctr_up && my_ctr_dn,
                CGL_E_BADARG, "cgl_life_band_run: null pointer");
    CGL_REQUIRE(cols % 32 == 0 && cols >= 32 * PB_COLS && (k == 4 || k == 8 || k == 16) && ghost >= k && ghost % k == 0 &&
                    buf_rows > 4 * ghost,
                CGL_E_BADARG, "cgl_life_band_run: bad shape (k in {4, 8, 16}, ghost a multiple of k, buf_rows > 4 ghost)");
    if (n_sub == 0 && !initial_push) return 0;
    PersistHalo h = {};
    h.ghost = ghost;
    h.sub_per_block = ghost / k;
    h.blk0 = block_index;
    h.initial_push = initial_push != 0;
    for (int s = 0; s < 2; ++s) {
        h.peer_up_landing[s] = peer_up_landing[s]; h.peer_dn_landing[s] = peer_dn_landing[s];
        h.my_landing_up[s] = my_landing_up[s]; h.my_landing_dn[s] = my_landing_dn[s];
    }
    h.peer_up_ctr = peer_up_ctr; h.peer_dn_ctr = peer_dn_ctr; h.my_ctr_up = my_ctr_up; h.my_ctr_dn = my_ctr_dn;
    cudaStream_t st = as_stream(stream);
    int rc = -100;
    switch (k) {
    case 4: rc = launch_persist<4, true>(buf_a, buf_b, buf_rows, cols, 0, n_sub, h, st); break;
    case 8: rc = launch_persist<8, true>(buf_a, buf_b, buf_rows, cols, 0, n_sub, h, st); break;
    case 16: rc = launch_persist<16, true>(buf_a, buf_b, buf_rows, cols, 0, n_sub, h, st); break;
    }
    CGL_REQUIRE(rc != -100, CGL_E_BADARG, "cgl_life_band_run: the band does not fit a cooperative launch on this device");
    return rc;
}

extern "C" int cgl_life_band_run_supported(uint32_t buf_rows, uint32_t cols, uint32_t k)
{
    uint32_t rpt, n_cg, n_rb;
    unsigned blocks;
    if (cols % 32 != 0 || cols < 32 * PB_COLS) return 0;
    switch (k) {
    case 4: return persist_geometry<4, true>(buf_rows, cols / 32, &rpt, &n_cg, &n_rb, &blocks);
    case 8: return persist_geometry<8, true>(buf_rows, cols / 32, &rpt, &n_cg, &n_rb, &blocks);
    case 16: return persist_geometry<16, true>(buf_rows, cols / 32, &rpt, &n_cg, &n_rb, &blocks);
    }
    return 0;
}
