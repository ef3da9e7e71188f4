// cgl_bits.cuh -- bit-sliced B3/S23 logic and the SIMD-in-register int8 stability rule.
//
// Everything here is `__host__ __device__` so the exact expressions the sm_100a kernels
// execute are also compiled by g++ into tests/twin/ (CPU-box unit tests of the bit logic).
//
// Layout convention (whole repo): a world row is ceil(cols/32) uint32 words; bit j of word w is
// the cell at column 32*w + j; padding bits above `cols` in the last word are ZERO.
//
// Semantics restated from the reference kernel `run`, /root/reference/CGL/CGL.py:147-181
// (CPU twin :211-243):
//   n    = sum of the 8 torus neighbours                         (:162-165)
//   next = (n == 3) || (n == 2 && prev)                          (:168-170)
//   stable' = surv ? (s == STABLE ? s : int8(s + 1)) : born ? SPAWN : 0      (:177-179)
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define CGL_HD __host__ __device__ __forceinline__
#else
#define CGL_HD inline
#endif

namespace cgl {

// ---- horizontal neighbour planes ------------------------------------------------------
// west(c)[j] = cell at column-1, east(c)[j] = cell at column+1, for an interior word.
CGL_HD uint32_t west_plane(uint32_t prev_word, uint32_t c) { return (c << 1) | (prev_word >> 31); }
CGL_HD uint32_t east_plane(uint32_t c, uint32_t next_word) { return (c >> 1) | (next_word << 31); }

// Horizontal partial sums of one row (2 bit-planes each):
//   t = west + east           (centre excluded; used for the cell's own row)
//   s = west + centre + east  (used for the rows above and below)
struct HSum { uint32_t s0, s1, t0, t1; };

CGL_HD HSum hsum(uint32_t w, uint32_t c, uint32_t e)
{
    HSum h;
    h.t0 = w ^ e;
    h.t1 = w & e;
    h.s0 = h.t0 ^ c;
    h.s1 = h.t1 | (h.t0 & c);
    return h;
}

CGL_HD uint32_t maj3(uint32_t a, uint32_t b, uint32_t c) { return (a & b) | (c & (a | b)); }

// n = up.s + mid.t + dn.s  in 0..8;   n = x0 + 2*(up.s1 + dn.s1 + mid.t1 + carry0)
// next = (#weight-2 terms == 1) & (x0 | centre)         [n==3 -> x0=1 ; n==2 -> needs centre]
CGL_HD uint32_t life_rule(const HSum &up, const HSum &mid, const HSum &dn, uint32_t centre)
{
    uint32_t x0 = up.s0 ^ dn.s0 ^ mid.t0;
    uint32_t c0 = maj3(up.s0, dn.s0, mid.t0);
    uint32_t f1 = up.s1 ^ dn.s1 ^ mid.t1;           // low bit of (up.s1 + dn.s1 + mid.t1)
    uint32_t f2 = maj3(up.s1, dn.s1, mid.t1);       // high bit
    uint32_t one = ~f2 & (f1 ^ c0);                 // (that sum + carry0) == 1
    return one & (x0 | centre);
}

// Full 3x3 evaluation from 9 already-shifted-independent words (generic path).
//   rows: a = above, c = current, b = below; each with its west/east adjacent WORDS.
CGL_HD uint32_t life_word(uint32_t aw, uint32_t a, uint32_t ae,
                          uint32_t cw, uint32_t c, uint32_t ce,
                          uint32_t bw, uint32_t b, uint32_t be)
{
    return life_rule(hsum(aw, a, ae), hsum(cw, c, ce), hsum(bw, b, be), c);
}

// ---- generic row access: torus columns for an arbitrary `cols` -----------------------------
// The last word of a row holds `rbits` valid bits (1..32); the column left of column 0 is
// column cols-1 and vice versa (CGL/CGL.py:156-157).  W == 1 makes prev == next == the word itself.
struct RowPlanes { uint32_t west, c, east; };

CGL_HD RowPlanes load_row_planes(const uint32_t *row, uint32_t w, uint32_t W, uint32_t rbits)
{
    RowPlanes p;
    p.c = row[w];
    uint32_t prev = row[w == 0 ? W - 1 : w - 1];
    const uint32_t next = row[w == W - 1 ? 0 : w + 1];
    if (w == 0) prev <<= (32 - rbits);                      // last valid column -> bit 31
    p.west = west_plane(prev, p.c);
    p.east = (w == W - 1) ? ((p.c >> 1) | ((next & 1u) << (rbits - 1))) : east_plane(p.c, next);
    return p;
}

// ---- SIMD-in-register int8 stability rule (4 cells per 32-bit word) --------------------
// Per byte: (x != MAX) ? x + 1 : x, with int8 wrap-around and no carry between bytes.
//   max4 = stable_max replicated into the 4 bytes.
CGL_HD uint32_t inc_unless_max4(uint32_t s, uint32_t max4)
{
    uint32_t x = s ^ max4;                                           // byte == 0  <=>  s == MAX
    uint32_t ne7 = (((x & 0x7f7f7f7fu) + 0x7f7f7f7fu) | x) & 0x80808080u;   // bit7 = (byte != 0)
#if defined(__CUDA_ARCH__)
    // (ne7 >> 7) + (s & 0x7f..) as ONE multiply-add on the FMA pipe: hi32(ne7 * 2^25) + addend
    uint32_t lo = __umulhi(ne7, 1u << 25) + (s & 0x7f7f7f7fu);
#else
    uint32_t lo = (s & 0x7f7f7f7fu) + (ne7 >> 7);                    // carry stops at bit 7
#endif
    return lo ^ (s & 0x80808080u);
}

// stable' for 4 cells given byte masks: surv_mask (0xFF where alive->alive) and
// born_spawn (SPAWN byte where dead->alive, 0 elsewhere); everything else becomes 0.
CGL_HD uint32_t stable_update4(uint32_t s, uint32_t surv_mask, uint32_t born_spawn, uint32_t max4)
{
    return (inc_unless_max4(s, max4) & surv_mask) | born_spawn;
}

// ---- the CGL_action+ fork's rule for cells that are dead after the step ------------------
// The base env zeroes them (CGL/CGL.py:179,242).  The fork lets them decay; its CUDA kernel and its CPU
// step disagree, so both are here (SURVEY.md section 8 row f2):
//   CGL_DEAD_ZERO  (0)  s' = 0
//   CGL_DEAD_DECAY (1)  s' = (s == EMPTY_MIN) ? s : int8(s - 1)     CGL_action+/CGL.py:190-193 (kernel `run`)
//   CGL_DEAD_SAT   (2)  s' = min(int8(s + EMPTY), EMPTY_MIN)        CGL_action+/CGL.py:256 (__step_state_cpu)
enum { CGL_DEAD_ZERO = 0, CGL_DEAD_DECAY = 1, CGL_DEAD_SAT = 2 };

// Per byte: (x != MIN) ? x - 1 : x, int8 wrap-around, no borrow between bytes.
CGL_HD uint32_t dec_unless_min4(uint32_t s, uint32_t min4)
{
    const uint32_t H = 0x80808080u;
    uint32_t x = s ^ min4;
    uint32_t ne1 = ((((x & 0x7f7f7f7fu) + 0x7f7f7f7fu) | x) & H) >> 7;      // 1 where byte != MIN
    return ((s | H) - ne1) ^ (s & H) ^ H;                                    // bytewise s - ne1
}

// Per byte int8(a + b) with wrap-around.
CGL_HD uint32_t add_wrap4(uint32_t a, uint32_t b)
{
    return ((a & 0x7f7f7f7fu) + (b & 0x7f7f7f7fu)) ^ ((a ^ b) & 0x80808080u);
}

// Per byte signed minimum.
CGL_HD uint32_t min_s8x4(uint32_t a, uint32_t b)
{
#if defined(__CUDA_ARCH__)
    return __vmins4(a, b);
#else
    uint32_t r = 0;
    for (int i = 0; i < 4; ++i) {
        const int8_t x = (int8_t)(a >> (8 * i)), y = (int8_t)(b >> (8 * i));
        r |= (uint32_t)(uint8_t)(x < y ? x : y) << (8 * i);
    }
    return r;
#endif
}

CGL_HD uint32_t dead_value4(int rule, uint32_t s, uint32_t min4, uint32_t empty4)
{
    if (rule == CGL_DEAD_DECAY) return dec_unless_min4(s, min4);
    if (rule == CGL_DEAD_SAT) return min_s8x4(add_wrap4(s, empty4), min4);
    return 0u;
}

// The decay rule for 4 cells as ONE equality test and ONE bytewise INCREMENT.  A cell is a survivor, dead or born;
// survivors compare against MAX and add 1, dead cells compare against MIN and subtract 1, born cells are overwritten
// with SPAWN at the end (whatever was computed for them).  The constant a byte is compared with is SELECTED per byte
// (one LOP3); "byte != constant" leaves a 0/1 per byte (bit 7 -> bit 0 on the FMA pipe); and because
// s - 1 == ~(~s + 1), the dead bytes are complemented on the way in and on the way out (folded into the masking
// LOP3s), so that every byte that moves is incremented by that 0/1.  11 operations per 4 cells (the form with a
// general bytewise addition of a +1 / -1 delta took 14, the two-test form 16); the kernel's time follows its
// instruction count.
CGL_HD uint32_t stable_update4_decay(uint32_t s, uint32_t surv_mask, uint32_t born_mask, uint32_t spawn4,
                                     uint32_t max4, uint32_t min4)
{
    const uint32_t H = 0x80808080u, L = 0x7f7f7f7fu;
    const uint32_t cmp = (max4 & surv_mask) | (min4 & ~surv_mask);                  // per byte: MAX or MIN
    const uint32_t x = s ^ cmp;
    const uint32_t ne7 = (((x & L) + L) | x) & H;                                   // bit 7: s != its constant
#if defined(__CUDA_ARCH__)
    const uint32_t e = __umulhi(ne7, 1u << 25);                                     // 0/1 per byte: the byte moves
#else
    const uint32_t e = ne7 >> 7;
#endif
    const uint32_t t = ((s ^ ~surv_mask) & L) + e;                                  // low 7 bits of (dead ? ~s : s) + e
    // (dead ? ~s : s) + e, complemented back for dead bytes:  t ^ ((s ^ ~surv) & H) ^ ~surv  ==  t ^ (s & H) ^ (~surv & L)
    const uint32_t r = (t ^ (s & H)) ^ (~surv_mask & L);
    return (r & ~born_mask) | (spawn4 & born_mask);
}

// stable' for 4 cells with a dead-cell rule: surv_mask / born_mask are byte masks (0xFF) of the cells that
// stayed alive / were born.
CGL_HD uint32_t stable_update4_rule(int rule, uint32_t s, uint32_t surv_mask, uint32_t born_mask, uint32_t spawn4,
                                    uint32_t max4, uint32_t min4, uint32_t empty4)
{
    if (rule == CGL_DEAD_DECAY) return stable_update4_decay(s, surv_mask, born_mask, spawn4, max4, min4);
    // (the saturating rule as one merged addition + minimum was measured SLOWER than the two separate updates: 29.7 vs 28.8 us)
    const uint32_t live = (inc_unless_max4(s, max4) & surv_mask) | (spawn4 & born_mask);
    return live | (dead_value4(rule, s, min4, empty4) & ~(surv_mask | born_mask));
}

CGL_HD int8_t stable_update1_rule(int rule, int8_t s, bool prev, bool next, int8_t spawn, int8_t stable_max,
                                  int8_t empty, int8_t empty_min)
{
    if (next && prev) return (s != stable_max) ? (int8_t)(s + 1) : s;
    if (next) return spawn;
    if (rule == CGL_DEAD_DECAY) return (s != empty_min) ? (int8_t)(s - 1) : s;
    if (rule == CGL_DEAD_SAT) {
        const int8_t t = (int8_t)(s + empty);
        return t < empty_min ? t : empty_min;
    }
    return 0;
}

// ---- one-step lookahead: every action's next-step reward (cgl_env_lookahead.cu) -------------------------------------
// A toggle at cell c changes only c's state and stability and, by the same +-1, the neighbour count of the 8 cells
// around c (on a torus of side >= 3 those 9 cells are distinct).  So with the plain step's reward R_noop,
//   R(c) = R_noop + h(c) + sum_{x in N8(c)} (c alive ? gm(x) : gp(x))        (mod 2^32)
// where, for a cell with state `alive`, neighbour count n and stability s:
//   plain  its stability after the plain step;
//   gp/gm  how that changes if n becomes n + 1 / n - 1 (state and stability kept);
//   h      its stability after the step if the cell itself is toggled first (state flipped, stability set by the
//          toggle: SPAWN, or with the masked toggle 0 for a cell toggled to dead), minus plain.
// Closed forms: with live = (alive ? s incremented unless MAX : SPAWN) the value a live-next cell gets and D the
// dead-cell rule's value, the stability only moves where `next` changes, by +-(live - D):
//   gp = +V at n == 2 - alive, -V at n == 3;   gm = +V at n == 4, -V at n == 3 - alive;   V = live - D.
struct Look1 { int plain, gp, gm, h; };

CGL_HD int8_t dead_value1(int rule, int8_t s, int8_t empty, int8_t empty_min)
{
    if (rule == CGL_DEAD_DECAY) return (s != empty_min) ? (int8_t)(s - 1) : s;
    if (rule == CGL_DEAD_SAT) {
        const int8_t t = (int8_t)(s + empty);
        return t < empty_min ? t : empty_min;
    }
    return 0;
}

CGL_HD Look1 lookahead1_rule(int rule, int8_t s, bool alive, int n, int8_t spawn, int8_t stable_max, int8_t empty,
                             int8_t empty_min, bool masked)
{
    const int8_t inc = (s != stable_max) ? (int8_t)(s + 1) : s;
    const int d = dead_value1(rule, s, empty, empty_min);
    const int live = alive ? (int)inc : (int)spawn;
    const bool next = n == 3 || (n == 2 && alive);
    const int v = live - d;
    Look1 r;
    r.plain = next ? live : d;
    r.gp = n == 2 - (int)alive ? v : (n == 3 ? -v : 0);
    r.gm = n == 4 ? v : (n == 3 - (int)alive ? -v : 0);
    // the toggled cell: a dead cell becomes alive with SPAWN and survives at n = 2, 3; a live one becomes dead (SPAWN,
    // or 0 with the masked toggle) and is born at n = 3
    const int8_t put = (masked && alive) ? (int8_t)0 : spawn;
    int t;
    if (alive) t = n == 3 ? (int)spawn : (int)dead_value1(rule, put, empty, empty_min);
    else t = (n == 2 || n == 3) ? (int)((put != stable_max) ? (int8_t)(put + 1) : put)
                                : (int)dead_value1(rule, put, empty, empty_min);
    r.h = t - r.plain;
    return r;
}

// ---- bit-sliced int8 stability (32 cells per operation) -----------------------------------
// For kernels that keep an env on chip for many steps the int8 plane is held as 8 bit planes per 32 cells
// (plane b, bit j = bit b of cell j's byte): the rule then costs ~33 logic ops per 32 cells instead of ~100
// with 4-cells-per-word bytes.  The price is a bit-matrix transpose on the way in and out.

// 8x8 bit-matrix transpose (Hacker's Delight 7-3): byte r of x = row r  ->  byte c of the result = column c.
CGL_HD uint64_t transpose8x8(uint64_t x)
{
    uint64_t t;
    t = (x ^ (x >> 7)) & 0x00AA00AA00AA00AAull;  x = x ^ t ^ (t << 7);
    t = (x ^ (x >> 14)) & 0x0000CCCC0000CCCCull; x = x ^ t ^ (t << 14);
    t = (x ^ (x >> 28)) & 0x00000000F0F0F0F0ull; x = x ^ t ^ (t << 28);
    return x;
}

// 4x4 byte transpose: out[i] byte k = in[k] byte i.
CGL_HD void transpose4x4_bytes(const uint32_t (&a)[4], uint32_t (&o)[4])
{
#if defined(__CUDA_ARCH__)
    const uint32_t t0 = __byte_perm(a[0], a[1], 0x5140), t1 = __byte_perm(a[2], a[3], 0x5140);
    const uint32_t t2 = __byte_perm(a[0], a[1], 0x7362), t3 = __byte_perm(a[2], a[3], 0x7362);
    o[0] = __byte_perm(t0, t1, 0x5410); o[1] = __byte_perm(t0, t1, 0x7632);
    o[2] = __byte_perm(t2, t3, 0x5410); o[3] = __byte_perm(t2, t3, 0x7632);
#else
    for (int i = 0; i < 4; ++i) {
        o[i] = 0;
        for (int k = 0; k < 4; ++k) o[i] |= ((a[k] >> (8 * i)) & 0xffu) << (8 * k);
    }
#endif
}

// 32 int8 cells (8 words, cell j = byte j % 4 of word j / 4)  ->  8 bit planes.
CGL_HD void bytes_to_planes32(const uint32_t (&w)[8], uint32_t (&p)[8])
{
    uint32_t lo[4], hi[4], pl[4], ph[4];
    for (int k = 0; k < 4; ++k) {              // cells 8k..8k+7: byte b of the result = plane b of those cells
        const uint64_t x = transpose8x8((uint64_t)w[2 * k] | ((uint64_t)w[2 * k + 1] << 32));
        lo[k] = (uint32_t)x; hi[k] = (uint32_t)(x >> 32);
    }
    transpose4x4_bytes(lo, pl);
    transpose4x4_bytes(hi, ph);
    for (int b = 0; b < 4; ++b) { p[b] = pl[b]; p[4 + b] = ph[b]; }
}

CGL_HD void planes_to_bytes32(const uint32_t (&p)[8], uint32_t (&w)[8])
{
    const uint32_t pl[4] = {p[0], p[1], p[2], p[3]}, ph[4] = {p[4], p[5], p[6], p[7]};
    uint32_t lo[4], hi[4];
    transpose4x4_bytes(pl, lo);
    transpose4x4_bytes(ph, hi);
    for (int k = 0; k < 4; ++k) {
        const uint64_t x = transpose8x8((uint64_t)lo[k] | ((uint64_t)hi[k] << 32));
        w[2 * k] = (uint32_t)x; w[2 * k + 1] = (uint32_t)(x >> 32);
    }
}

// p += k (mod 256) for all 32 cells, k a constant: ripple-carry addition of a uniform operand.
CGL_HD void add_const_sliced(uint32_t (&p)[8], int k)
{
    uint32_t c = 0;
    for (int b = 0; b < 8; ++b) {
        const uint32_t kb = ((k >> b) & 1) ? 0xffffffffu : 0u;
        const uint32_t pb = p[b];
        p[b] = pb ^ kb ^ c;
        c = (pb & kb) | (c & (pb | kb));
    }
}

// The base env's stability rule on bit planes in SPAWN-RELATIVE form: the planes hold u = s - SPAWN (mod 256)
// for live cells and anything for dead ones (a dead cell's value is never read: a birth overwrites it and the
// caller masks the planes with the world when it converts back).  Then a born cell is u = 0, exactly like a
// dead one, and the whole rule is: survivors increment unless u == max_rel (= STABLE - SPAWN mod 256),
// everything else becomes 0.  25 logic ops per 32 cells plus the 8 compares.
CGL_HD void stable_update_sliced_rel(uint32_t (&p)[8], uint32_t surv, int max_rel)
{
    uint32_t diff = 0;
    for (int b = 0; b < 8; ++b) diff |= p[b] ^ (((max_rel >> b) & 1) ? 0xffffffffu : 0u);
    uint32_t c = surv & diff;                                  // cells that increment
    for (int b = 0; b < 8; ++b) {
        const uint32_t pb = p[b];
        const uint32_t n = pb ^ c;
        c &= pb;
        p[b] = surv & n;
    }
}

// The CGL_action+ fork's decay rule (CGL_DEAD_DECAY) on spawn-relative bit planes.  Here dead cells DO carry a
// value (they fall by one per step down to EMPTY_MIN), so all cells are kept relative to SPAWN: survivors
// add 1 unless u == max_rel, dead cells subtract 1 unless u == min_rel (= EMPTY_MIN - SPAWN mod 256), born
// cells become 0.  One ripple pass adds the per-cell operand D (bit 0 = inc | dec, bits 1..7 = dec).
CGL_HD void stable_update_sliced_decay(uint32_t (&p)[8], uint32_t surv, uint32_t born, int max_rel, int min_rel)
{
    uint32_t dmax = 0, dmin = 0;
    for (int b = 0; b < 8; ++b) {
        dmax |= p[b] ^ (((max_rel >> b) & 1) ? 0xffffffffu : 0u);
        dmin |= p[b] ^ (((min_rel >> b) & 1) ? 0xffffffffu : 0u);
    }
    const uint32_t dec = ~(surv | born) & dmin;                // dead cells above the floor
    const uint32_t d0 = (surv & dmax) | dec;
    const uint32_t keep = ~born;
    uint32_t c = 0;
    for (int b = 0; b < 8; ++b) {
        const uint32_t pb = p[b], db = b == 0 ? d0 : dec;
        p[b] = (pb ^ db ^ c) & keep;
        c = (pb & db) | (c & (pb | db));
    }
}

// B3/S23 for FOUR cells held one per byte (values 0/1): u, m, d are the words of the row above, the cells' own row
// and the row below; lc / rc the sums (0..3) of the three cells in the column left of byte 0 / right of byte 3.
// Packed-byte arithmetic: column sums, then the 3x3 sum INCLUDING the cell (<= 9, no carry between bytes), then
// alive next <=> sum == 3, or sum == 4 and alive now.  Returns 0/1 per byte.  (The single-env server, cgl_sim1.cu.)
CGL_HD uint32_t life_next4_bytes(uint32_t u, uint32_t m, uint32_t d, uint32_t lc, uint32_t rc)
{
    const uint32_t col = u + m + d;
    const uint32_t t = col + ((col << 8) | lc) + ((col >> 8) | (rc << 24));
    const uint32_t ne3 = ((t ^ 0x03030303u) + 0x7f7f7f7fu) & 0x80808080u;           // bit 7 set: sum != 3
    const uint32_t ne4 = ((t ^ 0x04040404u) + 0x7f7f7f7fu) & 0x80808080u;
    return ((~ne3 >> 7) | ((~ne4 >> 7) & m)) & 0x01010101u;
}

// The CGL_action+ fork's SATURATING rule (CGL_DEAD_SAT, its CPU step) on ABSOLUTE bit planes: survivors add 1 unless
// s == MAX, born cells become SPAWN, dead cells become min(int8(s + EMPTY), EMPTY_MIN) (signed).  The addition is a
// ripple pass with a constant operand, the signed comparison runs MSB first with the sign planes inverted, every
// constant enters as an all-ones / all-zeros word.  ~90 logic operations per 32 cells (the byte form needs ~22 per 4).
CGL_HD uint32_t bit_mask_of(int v, int b) { return ((v >> b) & 1) ? 0xffffffffu : 0u; }

CGL_HD void stable_update_sliced_sat(uint32_t (&p)[8], uint32_t surv, uint32_t born, int spawn, int stable_max, int empty,
                                     int empty_min)
{
    uint32_t diff = 0;
    for (int b = 0; b < 8; ++b) diff |= p[b] ^ bit_mask_of(stable_max, b);
    uint32_t t[8], cy = 0;                                       // t = s + EMPTY (mod 256)
    for (int b = 0; b < 8; ++b) {
        const uint32_t kb = bit_mask_of(empty, b), pb = p[b];
        t[b] = pb ^ kb ^ cy;
        cy = (pb & kb) | (cy & (pb | kb));
    }
    uint32_t lt = 0, eq = 0xffffffffu;                            // lt: t < EMPTY_MIN as signed bytes
    for (int b = 7; b >= 0; --b) {
        uint32_t tb = t[b], mb = bit_mask_of(empty_min, b);
        if (b == 7) { tb = ~tb; mb = ~mb; }                       // sign bit: 1 sorts BELOW 0
        lt |= eq & ~tb & mb;
        eq &= ~(tb ^ mb);
    }
    const uint32_t dead = ~(surv | born);
    uint32_t c = surv & diff;                                    // survivors that increment
    for (int b = 0; b < 8; ++b) {
        const uint32_t pb = p[b];
        const uint32_t inc = pb ^ c;
        c &= pb;
        const uint32_t dv = (t[b] & lt) | (bit_mask_of(empty_min, b) & ~lt);
        p[b] = (surv & inc) | (born & bit_mask_of(spawn, b)) | (dead & dv);
    }
}

// ---- per-step reward straight from the bit planes (cgl_env_run_ex) -------------------------------------------------
CGL_HD int popc32(uint32_t x)
{
#if defined(__CUDA_ARCH__)
    return __popc(x);
#else
    return __builtin_popcount(x);
#endif
}

// The cells of `bit` take the byte value v in every plane (a toggle's stability write).
CGL_HD void set_cells_sliced(uint32_t (&p)[8], uint32_t bit, int v)
{
    for (int b = 0; b < 8; ++b) p[b] = (p[b] & ~bit) | (bit_mask_of(v, b) & bit);
}

// Cells whose byte, read unsigned, exceeds the constant k (0..255): an MSB-first compare against a uniform operand.
CGL_HD uint32_t gt_const_sliced(const uint32_t (&p)[8], int k)
{
    uint32_t gt = 0, eq = 0xffffffffu;
    for (int b = 7; b >= 0; --b) {
        const uint32_t kb = bit_mask_of(k, b);
        gt |= eq & p[b] & ~kb;
        eq &= ~(p[b] ^ kb);
    }
    return gt;
}

// The int8 sum of 32 cells after a step of the run kernel, from the planes it carries (cgl_env_run.cu):
//   CGL_DEAD_SAT    absolute planes: sum_b 2^b popc(plane b) with the sign plane weighing -128;
//   CGL_DEAD_DECAY  every cell spawn-relative, s = int8(u + SPAWN) = u + SPAWN - 256 [u > 127 - SPAWN];
//   CGL_DEAD_ZERO   the same over the live cells (`live`): after stable_update_sliced_rel every other cell is u = 0.
// `wraps` may be false when no reachable u exceeds 127 - SPAWN (the base rule with SPAWN..MAX inside int8): the
// compare is then skipped.
CGL_HD int sliced_reward32(int rule, const uint32_t (&p)[8], uint32_t live, int spawn, bool wraps)
{
    int s = 0;
    for (int b = 0; b < 8; ++b) s += popc32(p[b]) << b;
    if (rule == CGL_DEAD_SAT) return s - (popc32(p[7]) << 8);
    s += spawn * (rule == CGL_DEAD_DECAY ? 32 : popc32(live));
    if (wraps) s -= popc32(gt_const_sliced(p, 127 - spawn)) << 8;
    return s;
}

// Expand a 4-bit nibble to 4 byte masks (bit i -> byte i = 0xFF).
CGL_HD uint32_t nibble_to_bytemask(uint32_t nib)
{
    uint32_t spread = (nib * 0x00204081u) & 0x01010101u;             // bit i -> bit 8*i
    return spread * 0xFFu;
}

// Scalar form of the rule (generic per-cell path); identical to CGL/CGL.py:236-242.
CGL_HD int8_t stable_update1(int8_t s, bool prev, bool next, int8_t spawn, int8_t stable_max)
{
    if (next && prev) return (s != stable_max) ? (int8_t)(s + 1) : s;
    if (next) return spawn;
    return 0;
}

// Interleave the nibbles of two 32-cell planes `cur` and `nxt` into 8 bytes
// ((cur_nibble << 4) | nxt_nibble), ordered so that out[0] serves cells 0..15 and out[1]
// serves cells 16..31, byte k of out[h] <-> cells 16h + 4k .. 16h + 4k + 3.
CGL_HD void mix_nibbles(uint32_t cur, uint32_t nxt, uint32_t &out_lo, uint32_t &out_hi)
{
    uint32_t even = (nxt & 0x0f0f0f0fu) | ((cur & 0x0f0f0f0fu) << 4);   // byte m <-> nibble 2m
    uint32_t odd = ((nxt >> 4) & 0x0f0f0f0fu) | (cur & 0xf0f0f0f0u);    // byte m <-> nibble 2m+1
#if defined(__CUDA_ARCH__)
    out_lo = __byte_perm(even, odd, 0x5140);     // e0 o0 e1 o1
    out_hi = __byte_perm(even, odd, 0x7362);     // e2 o2 e3 o3
#else
    out_lo = (even & 0xffu) | ((odd & 0xffu) << 8) | ((even & 0xff00u) << 8) | ((odd & 0xff00u) << 16);
    out_hi = ((even >> 16) & 0xffu) | (((odd >> 16) & 0xffu) << 8) | (((even >> 24) & 0xffu) << 16) |
             (((odd >> 24) & 0xffu) << 24);
#endif
}

CGL_HD uint32_t rep4(int v) { return (uint32_t)(uint8_t)v * 0x01010101u; }

}  // namespace cgl
