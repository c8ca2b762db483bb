// Host-side plan of one TC-ELBO evaluation: padded sizes, work split and workspace layout.
// Shared by tcelbo_workspace_bytes / tcelbo_forward / tcelbo_backward so the three always agree.
#pragma once
#include <cstddef>
#include <cstdint>

namespace tcelbo {

constexpr int kTileFloats = 4096;     // floats of column data per pipeline stage (16 KiB)
constexpr int kStages     = 3;        // bulk-copy pipeline depth
constexpr int kRowPad     = 128;      // column-variance sweeps: b_loc / b_glob are padded to a multiple of this
constexpr int kColPad     = 32;       // row-variance sweeps: columns pad to this (one forward tile, two backward tiles)
constexpr int kSmallTile  = 4;        // forward column tile of the small-problem instantiation
constexpr int kFwdWarps   = 4;
constexpr int kBwdWarps   = 8;
constexpr int kFinWarps   = 8;        // rows (one warp each) per CTA of the forward finalize kernel
constexpr int kFinRedSlots = 5;       // batch means the forward finalize kernel reduces: (loss, kl | mi, -| tc, -| dimkl, exp-ELBO)

inline int64_t round_up(int64_t x, int64_t m) { return (x + m - 1) / m * m; }

constexpr int kMaxSplits = 16;        // upper bound on the partial-sum slots per row block (bounds the scratch)

// Balanced segments: a sweep's work is n_blocks row blocks x tiles_per_block column tiles.  Linearised block-major
// and cut into n_ctas contiguous segments whose lengths differ by at most one tile (one CTA each, n_ctas a whole number
// of waves of resident CTA slots), every CTA carries the same load for any batch shape -- a uniform (row block x
// column split) grid loses up to a full wave when n_blocks * n_splits lands just above a multiple of the slots (15 %
// of the backward sweep at 1024 rows per GPU).  A segment that crosses a block boundary writes one partial slot per
// block it touches; at most kMaxSplits segments touch a block.
#ifdef __CUDACC__
#define TCELBO_HD __host__ __device__
#else
#define TCELBO_HD
#endif
struct Segments {
    int n_ctas, base, rem;            // segments 0..rem-1 hold base+1 tiles, the others base tiles
};
TCELBO_HD inline int64_t seg_begin(const Segments& s, int c) { return (int64_t)c * s.base + (c < s.rem ? c : s.rem); }
TCELBO_HD inline int seg_len(const Segments& s, int c) { return s.base + (c < s.rem ? 1 : 0); }
TCELBO_HD inline int seg_of(const Segments& s, int64_t g) {           // the segment that holds tile g
    const int64_t cut = (int64_t)s.rem * (s.base + 1);
    if (g < cut) return g <= 0x7fffffff ? (int)((uint32_t)g / (uint32_t)(s.base + 1)) : (int)(g / (s.base + 1));
    const int64_t h = g - cut;
    return s.rem + (h <= 0x7fffffff ? (int)((uint32_t)h / (uint32_t)s.base) : (int)(h / s.base));
}
// number of segments that touch block q (tiles [q*T, (q+1)*T))
TCELBO_HD inline int seg_slots(const Segments& s, int64_t q, int tiles_per_block) {
    return seg_of(s, (q + 1) * tiles_per_block - 1) - seg_of(s, q * tiles_per_block) + 1;
}

// Shipped configurations of the backward row-variance sweep, tc_bwd_ds_kernel<RP, CH, NW, MINB, JT> (tc_bwd_ds.cu): RP row
// pairs per warp, CH warps per 32*CH-dim slice, NW warps per CTA, MINB resident CTAs per SM (the launch bounds, and the wave
// size the segment plan assumes), JT columns per tile.  The measured alternatives they beat are in profiles/r2_bwd_ds_sweep.md.
struct BwdDsConfig { int rp, ch, nw, minb, jt; };
constexpr BwdDsConfig kBwdDsConfigs[6] = {
    {8, 4, 12, 1, 16}, {8, 2, 12, 1, 16}, {8, 1, 12, 1, 16},   // 16 rows per warp, 12 warps per SM (168 registers); dp >= 128 / 64 / 32
    {2, 4, 8, 2, 16},  {2, 2, 8, 2, 16},  {2, 1, 8, 2, 16},    // small problems: 4 rows per warp, so that row blocks x tiles covers more SMs
};
// Column-variance sweeps (tc_colvar.cu), DPT = dp / 32: resident CTAs per SM (the kernels' launch bounds) and, backward, rows per warp
constexpr int kColvarFwdRes = 3;
constexpr int colvar_bwd_rows_per_warp(int dpt) { return dpt <= 4 ? 4 : 16 / dpt; }
constexpr int colvar_bwd_res(int dpt) { return dpt <= 2 ? 2 : 1; }

struct Plan {
    // padded problem
    int d, dp, dpt;            // dp = power of two >= max(d, 32); dpt = dp / 32 (floats per lane / lanes per row)
    int b_loc, b_glob, bl_pad, bg_pad;
    int jt;                    // column-tile height (rows of mu per stage) = kTileFloats / dp
    // forward sweep: grid (n_rb_fwd, n_js_fwd)
    int fwd_rows, n_rb_fwd, n_js_fwd, js_len_fwd;            // uniform split (column-variance sweep)
    Segments seg_fwd; int tiles_fwd, slots_fwd;               // balanced segments (row-variance sweep)
    int n_part_fwd;                                           // partial-sum slots the scratch holds
    // backward sweep: n_rb_bwd row blocks of bwd_rows rows
    int bwd_rows, n_rb_bwd;
    int n_js_bwd, js_len_bwd;                                 // uniform split: grid (n_rb_bwd, n_js_bwd) (column-variance sweep)
    int bwd_cfg, slice_bwd, n_slices_bwd;                     // kBwdDsConfigs entry, dims per slice (row-variance sweep) ...
    Segments seg_bwd; int tiles_bwd;                          // ... balanced segments over blocks q = slice * n_rb_bwd + row block
    // workspace (byte offsets)
    size_t off_mu, off_zs, off_ns, off_qmax, off_shift, off_vr;   // [bg_pad|bl_pad][dp]
    size_t off_S, off_J2;                                         // persistent forward results
    size_t off_red; int n_fin_ctas;                               // per-CTA partials + ticket of the finalize kernel's batch means
    size_t off_s2; int64_t ld_s2;                                 // joint exponents [bl_pad][bg_pad]
    size_t off_scratch;                                           // forward split partials (S, J)
    size_t total_bytes;                                           // forward workspace (read-only in backward)
    // backward scratch (its own buffer, so the forward workspace stays immutable and backward can be re-run)
    size_t boff_gps, boff_gj, boff_gk, boff_A, boff_CR, boff_G, boff_gpz, bwd_bytes;
    bool save, var_col;
    int fwd_lpr, fwd_kch, fwd_warps;   // forward sweep mapping: lanes per row, 16-byte chunks (4 dims) per lane, warps per CTA
    bool small;                // fewer work units than SMs with the standard tiles: small-tile / few-rows instantiations
};

inline size_t align256(size_t x) { return (x + 255) & ~size_t(255); }


// Pick how many ranges to cut `len` (a multiple of `quantum`) into so that n_blocks * n_splits CTAs fill
// `slots` resident CTA slots in whole waves: minimises ceil(ctas / slots) / n_splits, i.e. the time of
// the sweep in units of one full-length CTA.  Ties go to fewer splits (less partial-sum traffic).
inline void choose_splits(int n_blocks, int slots, int len, int quantum, int min_quanta, int& n_splits, int& split_len) {
    int max_splits = len / (quantum * min_quanta);
    if (max_splits < 1) max_splits = 1;
    if (max_splits > kMaxSplits) max_splits = kMaxSplits;
    double best = 1e30; int best_n = 1;
    for (int n = 1; n <= max_splits; ++n) {
        const int sl = (int)round_up((len + n - 1) / n, quantum);
        const int n_eff = (len + sl - 1) / sl;
        const long long ctas = (long long)n_blocks * n_eff;
        const double waves = (double)((ctas + slots - 1) / slots);
        const double cost = waves * (double)sl;               // time ~ waves x columns per CTA
        if (cost < best * 0.999) { best = cost; best_n = n_eff; }
    }
    split_len = (int)round_up((len + best_n - 1) / best_n, quantum);
    n_splits = (len + split_len - 1) / split_len;
}

inline Segments plan_segments(int64_t n_blocks, int tiles_per_block, int slots, int target_tiles) {
    const int64_t total = n_blocks * tiles_per_block;
    int64_t min_seg = (tiles_per_block - 1 + (kMaxSplits - 3)) / (kMaxSplits - 2);   // (T-1)/base + 2 <= kMaxSplits
    if (min_seg < 1) min_seg = 1;                 // small problems: down to one tile per CTA, so that they still spread over the SMs
    const int64_t want = target_tiles > min_seg ? target_tiles : min_seg;
    int64_t waves = (total + (int64_t)slots * want / 2) / ((int64_t)slots * want);    // nearest whole number of waves
    if (waves < 1) waves = 1;
    int64_t n = (int64_t)slots * waves;
    while (waves > 1 && total / n < min_seg) { --waves; n = (int64_t)slots * waves; }
    if (total / n < min_seg) n = total / min_seg;                                     // small problems: fewer, full-length CTAs
    if (n < 1) n = 1;
    Segments s;
    s.n_ctas = (int)n; s.base = (int)(total / n); s.rem = (int)(total % n);
    return s;
}

// `sms` = multiprocessor count of the current device (148 on B200).
inline bool make_plan(Plan& p, int b_loc, int b_glob, int d, uint32_t flags, int sms) {
    if (b_loc < 1 || b_glob < 1 || d < 1 || d > 512) return false;
    p = Plan();
    p.d = d;
    int dp = 32; while (dp < d) dp <<= 1;
    p.dp = dp; p.dpt = dp / 32;
    p.b_loc = b_loc; p.b_glob = b_glob;
    p.save = (flags & 4u) != 0;
    p.var_col = (flags & 2u) != 0;
    // ---- forward: a CTA owns fwd_rows rows and a contiguous range of columns
    // forward mapping: lanes per row x 16-byte chunks per lane.  Shipped: 16 dims per lane (dp/16 lanes per row, 128 registers,
    // 16 warps per SM) -- 4 warps per CTA for D <= 128, 8 warps per CTA for wider latents, so that a CTA still owns 16 (D = 256) /
    // 8 (D = 512) rows and the L2 -> SM traffic of the column tiles does not grow.  Small problems (BASELINE cfg 1 / 2: B = 3 / 64)
    // and the column-variance sweeps keep round 1's 32 dims per lane (dp/32 lanes per row, 3 CTAs of 4 warps per SM); the small
    // ones with 4-column tiles, so that row blocks x tiles still gives every SM a CTA.
    // Rows pad to whole forward row blocks, columns to whole 32-column tiles; the column-variance sweeps keep the 128-row padding
    // their uniform grids were written for.
    auto set_map = [&](int lpr, int kch, int warps) {
        p.fwd_lpr = lpr; p.fwd_kch = kch; p.fwd_warps = warps;
        p.fwd_rows = warps * (32 / lpr);
        const int row_pad = p.var_col ? kRowPad : (p.fwd_rows > kColPad ? p.fwd_rows : kColPad);
        p.bl_pad = (int)round_up(b_loc, row_pad);
        p.n_rb_fwd = p.bl_pad / p.fwd_rows;
    };
    set_map(p.dpt, 8, kFwdWarps);
    p.bg_pad = (int)round_up(b_glob, p.var_col ? kRowPad : kColPad);
    p.jt = kTileFloats / dp;                                   // 128 .. 8
    if (p.jt > 32) p.jt = 32;
    p.small = !p.var_col && (int64_t)p.n_rb_fwd * (p.bg_pad / p.jt) < sms;
    if (p.small) p.jt = kSmallTile;
    else if (!p.var_col) set_map(dp / 16, 4, dp <= 128 ? kFwdWarps : 8);
    const int fwd_res = p.fwd_kch == 4 ? 16 / p.fwd_warps : 3;   // resident CTAs per SM: wave size
    // the column-variance grid; row-variance plans size their forward partials with it too
    choose_splits(p.n_rb_fwd, sms * kColvarFwdRes, p.bg_pad, p.jt, 4, p.n_js_fwd, p.js_len_fwd);
    p.tiles_fwd = p.bg_pad / p.jt;
    p.seg_fwd = plan_segments(p.n_rb_fwd, p.tiles_fwd, sms * fwd_res, 21);    // column tiles per CTA: 16 / 21 / 32 time the same (profiles/r2_notes.md)
    p.slots_fwd = (p.tiles_fwd - 1) / p.seg_fwd.base + 2;
    if (p.slots_fwd > kMaxSplits) p.slots_fwd = kMaxSplits;
    // ---- backward sweep: the partial-sum slots it writes per row block fit the kMaxSplits of the backward scratch
    if (p.var_col) {
        p.bwd_rows = kBwdWarps * colvar_bwd_rows_per_warp(p.dpt);
        p.n_rb_bwd = (p.bl_pad + p.bwd_rows - 1) / p.bwd_rows;
        choose_splits(p.n_rb_bwd, sms * colvar_bwd_res(p.dpt), p.bg_pad, p.jt, 4, p.n_js_bwd, p.js_len_bwd);
    } else {
        p.bwd_cfg = (p.small ? 3 : 0) + (dp >= 128 ? 0 : dp == 64 ? 1 : 2);
        const BwdDsConfig& c = kBwdDsConfigs[p.bwd_cfg];
        p.bwd_rows = c.nw / c.ch * 2 * c.rp;
        p.n_rb_bwd = (p.bl_pad + p.bwd_rows - 1) / p.bwd_rows;
        p.slice_bwd = 32 * c.ch;
        p.n_slices_bwd = dp / p.slice_bwd;
        p.tiles_bwd = p.bg_pad / c.jt;
        p.seg_bwd = plan_segments((int64_t)p.n_rb_bwd * p.n_slices_bwd, p.tiles_bwd, sms * c.minb, 2048 / c.jt);   // 128 tiles of 16 columns per CTA (profiles/r2_notes.md)
    }

    // ---- workspace
    size_t off = 0;
    const size_t row_arr = (size_t)p.bl_pad * dp * sizeof(float);
    const size_t col_arr = (size_t)p.bg_pad * dp * sizeof(float);
    p.off_mu = off;    off = align256(off + (p.var_col ? 3 : 1) * col_arr);          // column operand(s), padded
    p.off_zs = off;    off = align256(off + row_arr);
    p.off_ns = off;    off = align256(off + row_arr);
    p.off_qmax = off;  off = align256(off + row_arr);
    p.off_shift = off; off = align256(off + row_arr);
    p.off_vr = off;    off = align256(off + row_arr);
    p.off_S = off;     off = align256(off + row_arr);
    p.off_J2 = off;    off = align256(off + (size_t)p.bl_pad * sizeof(float));
    p.n_fin_ctas = (b_loc + kFinWarps - 1) / kFinWarps;
    p.off_red = off;   off = align256(off + ((size_t)kFinRedSlots * p.n_fin_ctas + 4) * sizeof(float));   // the means per CTA, then the ticket
    p.ld_s2 = p.bg_pad;
    p.off_s2 = off;    off = align256(off + (p.save ? (size_t)p.bl_pad * p.ld_s2 * sizeof(float) : 0));
    const int n_part = p.n_js_fwd > p.slots_fwd ? p.n_js_fwd : p.slots_fwd;
    p.n_part_fwd = n_part;
    const size_t fwd_scratch = (size_t)n_part * row_arr + (size_t)n_part * p.bl_pad * 2 * sizeof(float);
    p.off_scratch = off; off = align256(off + fwd_scratch);
    p.total_bytes = off;

    size_t b = 0;
    p.boff_gps = b; b = align256(b + row_arr);
    p.boff_gj = b;  b = align256(b + (size_t)p.bl_pad * sizeof(float));
    p.boff_gk = b;  b = align256(b + (size_t)p.bl_pad * sizeof(float));
    p.boff_A = b;   b = align256(b + (size_t)kMaxSplits * row_arr);          // row-local partial sums per column split
    p.boff_CR = b;  b = align256(b + (size_t)kMaxSplits * row_arr);
    p.boff_G = b;   b = align256(b + 2 * col_arr);                           // column accumulators (mu [, logvar])
    p.boff_gpz = b; b = align256(b + (p.var_col ? (size_t)p.bl_pad * sizeof(float) : 0));   // decomposition: coefficient of log p(z_i)
    p.bwd_bytes = b;
    return true;
}

}  // namespace tcelbo
