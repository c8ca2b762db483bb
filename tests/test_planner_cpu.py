"""Host-side work planner (csrc/tc_layout.h): balanced segments must tile the (row block x column tile) space exactly,
differ by at most one tile, stay within the partial-slot budget, and number the slots of every block 0..n-1.  Whole plans:
the forward and backward grids of both sweeps write no more partial-sum slots than the workspace and the scratch hold."""
import os
import subprocess
import textwrap

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

SRC = textwrap.dedent(r"""
    #include "tc_layout.h"
    #include <cstdio>
    #include <vector>
    using namespace tcelbo;
    static int check_tiling(const Segments& s, int64_t n_blocks, int T) {
        const int64_t total = n_blocks * T;
        if (s.n_ctas < 1 || s.base < 1) return 1;
        if (seg_begin(s, s.n_ctas - 1) + seg_len(s, s.n_ctas - 1) != total) return 2;      // covers everything, no overlap
        for (int c = 0; c + 1 < s.n_ctas; ++c)
            if (seg_begin(s, c) + seg_len(s, c) != seg_begin(s, c + 1)) return 3;
        for (int c = 0; c < s.n_ctas; c += (s.n_ctas > 4096 ? 97 : 1)) {                   // inverse map
            if (seg_of(s, seg_begin(s, c)) != c) return 4;
            if (seg_of(s, seg_begin(s, c) + seg_len(s, c) - 1) != c) return 5;
        }
        for (int64_t q = 0; q < n_blocks; q += (n_blocks > 4096 ? 53 : 1)) {
            const int n = seg_slots(s, q, T);
            if (n < 1 || n > kMaxSplits) return 6;
        }
        return 0;
    }
    static int check(int64_t n_blocks, int T, int slots, int target) {
        const Segments s = plan_segments(n_blocks, T, slots, target);
        if (const int rc = check_tiling(s, n_blocks, T)) return rc;
        if (s.n_ctas > slots && s.n_ctas % slots != 0) return 7;                           // whole waves once past one wave
        return 0;
    }
    int main() {
        const int Ts[] = {1, 2, 4, 8, 16, 37, 64, 256, 512, 2048, 16384};
        const int64_t Bs[] = {1, 2, 3, 7, 32, 43, 86, 171, 342, 1366, 5462};
        const int slots[] = {1, 148, 296, 444};
        const int targets[] = {1, 21, 64, 300};
        for (int T : Ts) for (int64_t b : Bs) for (int sl : slots) for (int tg : targets) {
            const int rc = check(b, T, sl, tg);
            if (rc) { std::printf("FAIL rc=%d blocks=%lld T=%d slots=%d target=%d\n", rc, (long long)b, T, sl, tg); return 1; }
        }
        // whole plans for shapes the tests and the bench use
        const int shapes[][3] = {{8192, 8192, 128}, {1024, 8192, 128}, {2, 2, 4}, {37, 37, 20}, {24, 24, 512}, {4096, 32768, 512}, {1, 8, 3},
                                   {4096, 4096, 64}, {4000, 4000, 20}, {1000, 1000, 128}, {512, 4096, 256}, {64, 64, 128}, {3, 3, 128},
                                   {64, 64, 64}};
        int cfgs_seen = 0;
        for (auto& sh : shapes) {
            // row variance: balanced segments; the backward ones index Apart / CRpart, which hold kMaxSplits slots per row
            Plan p;
            if (!make_plan(p, sh[0], sh[1], sh[2], 4u, 148)) { std::printf("FAIL make_plan\n"); return 1; }
            if (p.slots_fwd > p.n_part_fwd || p.slots_fwd > kMaxSplits) { std::printf("FAIL slots\n"); return 1; }
            for (int q = 0; q < p.n_rb_fwd; ++q)
                if (seg_slots(p.seg_fwd, q, p.tiles_fwd) > p.slots_fwd) { std::printf("FAIL fwd slots %d %d\n", sh[0], sh[1]); return 1; }
            if (p.n_rb_bwd * p.bwd_rows < p.bl_pad || p.n_slices_bwd * p.slice_bwd != p.dp) { std::printf("FAIL bwd blocks %d %d\n", sh[0], sh[1]); return 1; }
            if (const int rc = check_tiling(p.seg_bwd, (int64_t)p.n_rb_bwd * p.n_slices_bwd, p.tiles_bwd)) {
                std::printf("FAIL bwd segments rc=%d %d %d %d\n", rc, sh[0], sh[1], sh[2]); return 1;
            }
            cfgs_seen |= 1 << p.bwd_cfg;
            // column variance: uniform splits, one partial-sum slot per split
            if (!make_plan(p, sh[0], sh[1], sh[2], 6u, 148)) { std::printf("FAIL make_plan\n"); return 1; }
            if (p.n_js_fwd > p.n_part_fwd || p.n_js_bwd > kMaxSplits) { std::printf("FAIL colvar splits %d %d %d\n", sh[0], sh[1], sh[2]); return 1; }
            if ((int64_t)p.n_js_fwd * p.js_len_fwd < p.bg_pad || (int64_t)p.n_js_bwd * p.js_len_bwd < p.bg_pad || p.n_rb_bwd * p.bwd_rows < p.bl_pad) {
                std::printf("FAIL colvar coverage %d %d %d\n", sh[0], sh[1], sh[2]); return 1;
            }
        }
        if (cfgs_seen != (1 << 6) - 1) { std::printf("FAIL backward configurations covered: %x\n", cfgs_seen); return 1; }
        std::printf("OK\n");
        return 0;
    }
""")


def test_balanced_segments(tmp_path):
    src = tmp_path / "planner_check.cpp"
    src.write_text(SRC)
    exe = tmp_path / "planner_check"
    inc = os.path.join(ROOT, "intro_tc_vae_b200", "csrc")
    subprocess.run(["g++", "-std=c++17", "-O1", "-I", inc, str(src), "-o", str(exe)], check=True)
    out = subprocess.run([str(exe)], capture_output=True, text=True)
    assert out.returncode == 0 and out.stdout.strip() == "OK", out.stdout + out.stderr
