// cgl_life.cu -- world-only generations ("life mode") of large bit-packed grids for sm_100a.
//
// Reference semantics: the world half of kernel `run`, /root/reference/CGL/CGL.py:154-170
// (torus neighbour count + B3/S23).  The reference cannot even express these sizes (its
// `unsigned int` index math overflows above side 46340, SURVEY.md section 5).
//
// life_rows_kernel (k = 1 streaming):  HBM traffic = 1 bit read + 1 bit written per cell
// (0.25 B / cell-update).  A thread owns a 128-cell-wide column (one uint4 per row) and walks
// down RPT rows keeping a 3-row window of horizontal partial sums in registers; horizontal
// neighbours come from the adjacent lanes by warp shuffle, the two warp-edge lanes load one halo
// word.  Per 32 cells: 2 SHF + 4 LOP3 (row sums, reused by 3 output rows) + 6 LOP3 (rule).
#include <stdlib.h>

#include "cgl_internal.cuh"

namespace cgl {

struct RowRaw { uint4 v; uint32_t halo; };
struct RowSums { HSum h[4]; uint4 c; };

// Per-lane constants of a strip walk.
struct Lane {
    const uint32_t *gin;      // grid base of this env
    uint32_t rows, W;
    int wrap_rows;
    uint32_t c4, hidx;        // uint4 column of this lane, halo word index (edge lanes)
    bool valid, store, edge, edge_l, edge_r;
};

// Load this lane's segment of row r (any integer; rows outside [0, rows) wrap or are dead).
// Straight-line code: the row index is fixed up with selects and the loads are predicated.
__device__ __forceinline__ RowRaw load_row_raw(const Lane &L, int r)
{
    const int rows = (int)L.rows;
    const bool outside = (r < 0) | (r >= rows);
    const int rw = r < 0 ? r + rows : (r >= rows ? r - rows : r);
    const bool live = !outside | (L.wrap_rows != 0);
    const uint32_t *row = L.gin + (uint64_t)(uint32_t)rw * L.W;
    RowRaw o;
    o.v = make_uint4(0, 0, 0, 0);
    o.halo = 0;
    if (L.valid && live) o.v = __ldg(reinterpret_cast<const uint4 *>(row) + L.c4);
    if (L.edge && live) o.halo = __ldg(row + L.hidx);
    return o;
}

__device__ __forceinline__ void row_sums(RowSums &s, const RowRaw &raw, const Lane &L)
{
    uint32_t left = __shfl_up_sync(0xffffffffu, raw.v.w, 1);
    uint32_t right = __shfl_down_sync(0xffffffffu, raw.v.x, 1);
    left = L.edge_l ? raw.halo : left;
    right = L.edge_r ? raw.halo : right;
    s.c = raw.v;
    s.h[0] = hsum(west_plane(left, raw.v.x), raw.v.x, east_plane(raw.v.x, raw.v.y));
    s.h[1] = hsum(west_plane(raw.v.x, raw.v.y), raw.v.y, east_plane(raw.v.y, raw.v.z));
    s.h[2] = hsum(west_plane(raw.v.y, raw.v.z), raw.v.z, east_plane(raw.v.z, raw.v.w));
    s.h[3] = hsum(west_plane(raw.v.z, raw.v.w), raw.v.w, east_plane(raw.v.w, right));
}

template <bool COUNT>
__device__ __forceinline__ void emit_row(const RowSums &up, const RowSums &mid, const RowSums &dn,
                                         uint32_t *__restrict__ gout, const Lane &L, int r, unsigned &pop)
{
    uint4 o;
    o.x = life_rule(up.h[0], mid.h[0], dn.h[0], mid.c.x);
    o.y = life_rule(up.h[1], mid.h[1], dn.h[1], mid.c.y);
    o.z = life_rule(up.h[2], mid.h[2], dn.h[2], mid.c.z);
    o.w = life_rule(up.h[3], mid.h[3], dn.h[3], mid.c.w);
    if (L.store && r < (int)L.rows)
        reinterpret_cast<uint4 *>(gout + (uint64_t)(uint32_t)r * L.W)[L.c4] = o;
    if (COUNT && r < (int)L.rows) pop += __popc(o.x) + __popc(o.y) + __popc(o.z) + __popc(o.w);
}

// The general strip walk: any row index (rows outside [0, rows) wrap or are dead), stores predicated per row.
template <bool COUNT, int PF>
__device__ __forceinline__ void walk_general(const Lane &L, uint32_t *__restrict__ gout, const int r0, const int rpt,
                                             unsigned &pop)
{
    RowSums A, B, C;
    row_sums(A, load_row_raw(L, r0 - 1), L);
    row_sums(B, load_row_raw(L, r0), L);

    RowRaw nxt[PF];
#pragma unroll
    for (int u = 0; u < PF; ++u) nxt[u] = load_row_raw(L, r0 + u + 1);

    for (int i = 0; i < rpt; i += PF) {                        // uniform trip count
        const int r = r0 + i;
        RowRaw cur[PF];
#pragma unroll
        for (int u = 0; u < PF; ++u) cur[u] = nxt[u];
        if (i + PF < rpt) {                                    // uniform: prefetch the next trip's rows
#pragma unroll
            for (int u = 0; u < PF; ++u) nxt[u] = load_row_raw(L, r + PF + u + 1);
        }
#pragma unroll
        for (int u = 0; u < PF; u += 3) {
            row_sums(C, cur[u], L);     emit_row<COUNT>(A, B, C, gout, L, r + u, pop);
            row_sums(A, cur[u + 1], L); emit_row<COUNT>(B, C, A, gout, L, r + u + 1, pop);
            row_sums(B, cur[u + 2], L); emit_row<COUNT>(C, A, B, gout, L, r + u + 2, pop);
        }
    }
}

// The interior strip walk: every row touched is a real row of the grid, so a row is `pointer += W`.
template <bool COUNT>
__device__ __forceinline__ void emit_row_at(const RowSums &up, const RowSums &mid, const RowSums &dn, uint32_t *po,
                                            const Lane &L, unsigned &pop)
{
    uint4 o;
    o.x = life_rule(up.h[0], mid.h[0], dn.h[0], mid.c.x);
    o.y = life_rule(up.h[1], mid.h[1], dn.h[1], mid.c.y);
    o.z = life_rule(up.h[2], mid.h[2], dn.h[2], mid.c.z);
    o.w = life_rule(up.h[3], mid.h[3], dn.h[3], mid.c.w);
    if (L.store) *reinterpret_cast<uint4 *>(po) = o;
    if (COUNT) pop += __popc(o.x) + __popc(o.y) + __popc(o.z) + __popc(o.w);
}

template <bool COUNT, int PF>
__device__ __forceinline__ void walk_interior(const Lane &L, uint32_t *__restrict__ gout, const int r0, const int rpt,
                                              unsigned &pop)
{
    const uint32_t W = L.W;
    const uint32_t *pm = L.gin + (uint64_t)(uint32_t)(r0 - 1) * W + 4 * L.c4;      // this lane's uint4 of row r0 - 1
    const int hoff = (int)L.hidx - 4 * (int)L.c4;                                  // halo word relative to it
    uint32_t *po = gout + (uint64_t)(uint32_t)r0 * W + 4 * L.c4;
    auto load = [&](const uint32_t *p) {
        RowRaw o;
        o.v = make_uint4(0, 0, 0, 0);
        o.halo = 0;
        if (L.valid) o.v = __ldg(reinterpret_cast<const uint4 *>(p));
        if (L.edge) o.halo = __ldg(p + hoff);
        return o;
    };
    RowSums A, B, C;
    row_sums(A, load(pm), L); pm += W;
    row_sums(B, load(pm), L); pm += W;
    RowRaw nxt[PF];
#pragma unroll
    for (int u = 0; u < PF; ++u) { nxt[u] = load(pm); pm += W; }

    for (int i = 0; i < rpt; i += PF) {                        // uniform trip count
        RowRaw cur[PF];
#pragma unroll
        for (int u = 0; u < PF; ++u) cur[u] = nxt[u];
        if (i + PF < rpt) {
#pragma unroll
            for (int u = 0; u < PF; ++u) { nxt[u] = load(pm); pm += W; }
        }
#pragma unroll
        for (int u = 0; u < PF; u += 3) {
            row_sums(C, cur[u], L);     emit_row_at<COUNT>(A, B, C, po, L, pop); po += W;
            row_sums(A, cur[u + 1], L); emit_row_at<COUNT>(B, C, A, po, L, pop); po += W;
            row_sums(B, cur[u + 2], L); emit_row_at<COUNT>(C, A, B, po, L, pop); po += W;
        }
    }
}

constexpr int LIFE_ROWS_THREADS = 128;   // 4 warps = 4 horizontally adjacent column groups

// rpt must be a multiple of PF (PF a multiple of 3); strips may run past `rows` (loads wrap / are
// dead, stores are predicated), so the loop body is branch-free and the 3-row window of partial
// sums rotates through three register sets A, B, C without moves.  The rows of trip i+1 are loaded
// (software pipelining) before trip i is computed, which keeps PF 16-byte loads per thread in
// flight whatever the instruction scheduler does inside a trip.
template <bool COUNT, int PF, int MINB>
__global__ void __launch_bounds__(LIFE_ROWS_THREADS, MINB)
life_rows_kernel(const uint32_t *__restrict__ in, uint32_t *__restrict__ out, uint32_t n_envs,
                 uint32_t rows, uint32_t W, uint32_t rpt, int wrap_rows, uint32_t n_cgroups,
                 uint32_t n_rblocks, uint32_t *__restrict__ alive_out)
{
    // Programmatic dependent launch: the next generation's CTAs may be placed while this grid's last wave drains;
    // they (like this CTA) wait for the whole previous grid before touching memory -- consecutive generations
    // ping-pong the two buffers, so a generation may neither read its input nor overwrite its output earlier.
    cudaTriggerProgrammaticLaunchCompletion();
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t warp = blockIdx.x * (LIFE_ROWS_THREADS / 32) + (threadIdx.x >> 5);
    const uint32_t cg = warp % n_cgroups;
    const uint32_t tmp = warp / n_cgroups;
    const uint32_t rb = tmp % n_rblocks;
    uint32_t e = tmp / n_rblocks;
    // no early exit (keeps the shuffles provably convergent): padding warps redo the last env, stores off
    const bool warp_ok = e < n_envs;
    e = warp_ok ? e : n_envs - 1;

    Lane L;
    const uint32_t W4 = W >> 2;
    L.rows = rows; L.W = W; L.wrap_rows = wrap_rows;
    L.c4 = cg * 32 + lane;
    L.valid = L.c4 < W4;
    L.store = L.valid && warp_ok;
    L.edge_l = lane == 0;
    L.edge_r = L.valid && (lane == 31 || L.c4 == W4 - 1);
    L.hidx = L.edge_l ? (L.c4 == 0 ? W - 1 : 4 * L.c4 - 1) : (L.c4 == W4 - 1 ? 0 : 4 * L.c4 + 4);
    L.edge = L.valid && (L.edge_l || L.edge_r);
    L.gin = in + (uint64_t)e * rows * W;
    uint32_t *gout = out + (uint64_t)e * rows * W;

    const int r0 = (int)(rb * rpt);
    unsigned pop = 0;
    cudaGridDependencySynchronize();
    // Strips whose rows r0 - 1 .. r0 + rpt all lie inside the grid (all but the first and last of an env) take the
    // lean walk: running pointers, no wrap / dead-row selects, unpredicated row tests.
    // (decided per CTA from blockIdx and kernel parameters only, so that the compiler can prove it uniform)
    bool cta_interior = true;
#pragma unroll
    for (uint32_t k = 0; k < LIFE_ROWS_THREADS / 32; ++k) {
        const uint32_t tk = (blockIdx.x * (LIFE_ROWS_THREADS / 32) + k) / n_cgroups;
        const uint32_t rk = (tk % n_rblocks) * rpt;
        cta_interior = cta_interior && rk >= 1 && rk + rpt + 1 <= rows && tk / n_rblocks < n_envs;
    }
    if (cta_interior)
        walk_interior<COUNT, PF>(L, gout, r0, (int)rpt, pop);
    else
        walk_general<COUNT, PF>(L, gout, r0, (int)rpt, pop);
    if (COUNT) {
        if (!L.store) pop = 0;
        pop = __reduce_add_sync(0xffffffffu, pop);
        if (lane == 0 && pop) atomicAdd(alive_out + e, pop);
    }
}

static uint32_t pick_rows_per_strip(uint64_t n_envs, uint32_t rows, uint32_t n_cgroups)
{
    // aim for >= 8 strips per resident warp slot (148 SMs x 16 warps) to keep the tail small,
    // but never fewer than 12 rows per strip (2 halo rows are re-read per strip).
    const uint64_t want = (uint64_t)sm_count() * 16 * 8;
    uint64_t rpt = 96;                                   // multiples of LIFE_ROWS_PF
    while (rpt > 12 && n_envs * n_cgroups * ((rows + rpt - 1) / rpt) < want) rpt >>= 1;
    return (uint32_t)rpt;
}

}  // namespace cgl

using namespace cgl;

extern "C" int cgl_life_step_generic(const uint32_t *in, uint32_t *out, uint64_t n_envs, uint32_t rows,
                                     uint32_t cols, int wrap_rows, uint32_t *alive_out,
                                     cgl_stream_t stream);

extern "C" int cgl_life_step(const uint32_t *in, uint32_t *out, uint64_t n_envs, uint32_t rows,
                             uint32_t cols, int wrap_rows, uint32_t *alive_out, cgl_stream_t stream)
{
    CGL_REQUIRE(in && out && n_envs && rows && cols && in != out, CGL_E_BADARG,
                "cgl_life_step: bad argument");
    if (cols % 128 != 0 || cols < 2048 || (cols / 128) % 32 == 1 || n_envs >= (1ull << 31))
        return cgl_life_step_generic(in, out, n_envs, rows, cols, wrap_rows, alive_out, stream);
    cudaStream_t st = as_stream(stream);
    const uint32_t W = cols / 32, W4 = W / 4;
    const uint32_t n_cgroups = (W4 + 31) / 32;
    static int rows_knob = -1;                   // CGL_LIFE_ROWS overrides the strip length (tuning; multiple of 6)
    if (rows_knob < 0) {
        const char *v = getenv("CGL_LIFE_ROWS");
        rows_knob = v ? atoi(v) : 0;
    }
    const uint32_t rpt = rows_knob > 0 ? (uint32_t)rows_knob : pick_rows_per_strip(n_envs, rows, n_cgroups);
    // A strip reads rows r0 - 1 .. r0 + rpt and load_row_raw wraps a row index once: on a torus with 2 * rows <= rpt
    // that would read past the env.  Such tiny tori take the generic kernel.
    if (wrap_rows && 2ull * rows <= rpt)
        return cgl_life_step_generic(in, out, n_envs, rows, cols, wrap_rows, alive_out, stream);
    const uint32_t n_rblocks = (rows + rpt - 1) / rpt;
    const uint64_t warps = n_envs * n_cgroups * n_rblocks;
    const uint64_t blocks = (warps + (LIFE_ROWS_THREADS / 32) - 1) / (LIFE_ROWS_THREADS / 32);
    CGL_REQUIRE(blocks < (1ull << 31) && warps < (1ull << 32) && rows < (1u << 30), CGL_E_BADARG, "cgl_life_step: grid too large");
    static int pf = 0;                           // tuning knob: rows prefetched per thread (3 or 6)
    if (pf == 0) {
        const char *v = getenv("CGL_LIFE_PF");
        pf = (v && atoi(v) == 6) ? 6 : 3;
    }
    static int minb = 0;                         // tuning knob: resident CTAs per SM the register allocation aims for (5 or 6)
    if (minb == 0) {
        const char *v = getenv("CGL_LIFE_MINB");
        minb = (v && atoi(v) == 5) ? 5 : 6;
    }
    static int pdl = -1;                         // CGL_LIFE_PDL=0: plain stream order (tuning / debugging)
    if (pdl < 0) {
        const char *v = getenv("CGL_LIFE_PDL");
        pdl = (v && v[0] == '0') ? 0 : 1;
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)blocks);
    cfg.blockDim = dim3(LIFE_ROWS_THREADS);
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl ? 1 : 0;
    const uint32_t n32 = (uint32_t)n_envs;
#define CGL_LIFE_ROWS(COUNT, PF, MINB, AL)                                                                        \
    CGL_CUDA(cudaLaunchKernelEx(&cfg, life_rows_kernel<COUNT, PF, MINB>, in, out, n32, rows, W, rpt, wrap_rows,    \
                                n_cgroups, n_rblocks, (uint32_t *)(AL)))
    if (alive_out != nullptr) {
        CGL_CUDA(cudaMemsetAsync(alive_out, 0, n_envs * sizeof(uint32_t), st));
        CGL_LIFE_ROWS(true, 3, 5, alive_out);
    } else if (pf == 6) {
        CGL_LIFE_ROWS(false, 6, 4, nullptr);
    } else if (minb == 5) {
        CGL_LIFE_ROWS(false, 3, 5, nullptr);
    } else {
        CGL_LIFE_ROWS(false, 3, 6, nullptr);
    }
#undef CGL_LIFE_ROWS
    CGL_LAUNCH_CHECK();
    return 0;
}
