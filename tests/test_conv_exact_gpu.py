"""Bit-exact conformance of every convolution kernel path (tcgen05 one-tile / persistent, every epilogue, split-K wgrad,
CUDA-core igemm_simt, the explicit-im2col stem) and of the weight (un)packing kernels.

The inputs are small integers (x, w, dy in [-4, 4]; [-2, 2] where the reduction is longer than 2^20).  Every bf16 x bf16
product is then exact in fp32 and every partial sum is an integer below 2^24 (checked per case by `magnitude_bound`), so
whatever the accumulation order, split-K layout or tile shape, a kernel's fp32 accumulator holds the exact sum, and so
does a float64 CPU F.conv2d on the same integers.  The expected outputs below are therefore equalities, not tolerances:

  fp32 fprop (+ integer bias)          float32(exact)
  bf16 fprop / dgrad, beta = 0         RNE_bf16(exact)          outputs reach ~+-2500: bf16 rounding and ties are exercised
  dgrad beta = 1, tcgen05 epilogues    RNE(old + RNE(acc))      the tile is staged as bf16, then added to the old value
  dgrad beta = 1, igemm_simt           RNE(old + acc)           fp32 add, one rounding
  wgrad (fresh or into a filled buffer) old + exact, in fp32, after unpack_wgrad
  BN statistics                        the exact sums of the STORED outputs (weights with <= 8 nonzeros of +-1 per output
                                       channel, so |y| <= 32 and every fp32 partial of a CTA is exact)

Each case of CASES names the kernel variant it is meant to reach; the GPU test reads the launched kernels back from
torch.profiler and fails when a case no longer reaches its variant (a retuned heuristic moves shapes between kernels), and
test_case_list_covers_every_variant checks on the CPU that the list reaches every production variant.  The run writes
`case -> variants` to conv_coverage.txt in the test session's output directory (the gpu_out_dir fixture).
test_replay_flagship_geometries replays, with the same integer data, every distinct conv geometry one training step of
bench.py's C3 and C2 configurations issues (pitches and alignments included, so the same epilogues are chosen)."""
import os
import re

import numpy as np
import pytest
import torch
import torch.nn.functional as F

if torch.cuda.is_available():
    from seg_b200 import lib, ops
    from seg_b200.lib import IMPL_AUTO
else:  # keep collection working on a machine without a GPU
    IMPL_AUTO = 0

DEV = "cuda"
OPS = ("fprop", "dgrad", "wgrad")
EPIS = ("manual", "manual_beta", "tma")
LIMIT = 1 << 24  # integers below this are exact in fp32


# ------------------------------------------------------------------------------------------------ case list
def case(name, op, N, H, W, C, K, R, stride=1, pad=None, dil=1, *, want, ldx=None, offx=0, ldy=None, offy=0, beta=0.0,
         f32=False, bias=False, stats=False, old=False, multi=False):
    """One conv call.  x side = the activation (fprop input, dgrad output, wgrad input), y side = the other tensor.
    ld*/off*: channel pitch and element offset of a slice of a wider buffer.  want: variants the case must reach.
    multi: a persistent launch must give every CTA >= 2 tiles and some CTA an odd count."""
    pad = (R // 2) * dil if pad is None else pad
    return dict(name=name, op=op, N=N, H=H, W=W, C=C, K=K, R=R, stride=stride, pad=pad, dil=dil, want=set(want),
                ldx=ldx or C, offx=offx, ldy=ldy or K, offy=offy, beta=beta, f32=f32, bias=bias, stats=stats, old=old,
                multi=multi)


CASES = [
    # ---- fprop ----
    case("fp_1x1_k64", "fprop", 2, 33, 33, 64, 64, 1, want={"fprop/tc1/bn64", "map2d", "m_tail"}),  # K <= 64: one-tile BN 64
    case("fp_3x3_256_longk", "fprop", 2, 33, 33, 256, 256, 3, want={"fprop/tc1/bn128", "map_im2col"}),  # long k-loop, few tiles
    case("fp_3x3_c304_k320_longk", "fprop", 2, 33, 33, 304, 320, 3, want={"fprop/tc1/bn128", "c_tail", "n_tail"}),
    case("fp_1x1_tma128", "fprop", 16, 49, 49, 64, 128, 1, want={"fprop/tc2/tma/128"}, multi=True),
    case("fp_1x1_tma256", "fprop", 16, 49, 49, 64, 256, 1, want={"fprop/tc2/tma/256"}, multi=True),
    case("fp_3x3_k320_tma128_ntail", "fprop", 4, 33, 33, 64, 320, 3, want={"fprop/tc2/tma/128", "n_tail"}),
    case("fp_3x3_manual_unaligned", "fprop", 16, 49, 49, 64, 128, 3, ldy=136, offy=4,  # 8-byte aligned output slice
         want={"fprop/tc2/manual/128", "slice_out"}, multi=True),
    case("fp_1x1_manual_ldy_odd", "fprop", 4, 33, 33, 128, 96, 1, ldy=130, offy=2, want={"fprop/tc2/manual/128", "n_tail"}),
    case("fp_f32_bias_k19_slice", "fprop", 2, 17, 17, 256, 19, 1, ldx=320, offx=48, f32=True, bias=True,
         want={"fprop/tc1/bn64", "f32_bias", "slice_in", "n_tail"}),
    case("fp_f32_bias_3x3_k320", "fprop", 2, 33, 33, 64, 320, 3, f32=True, bias=True, want={"fprop/tc1/bn64", "f32_bias"}),
    case("fp_3x3_s2", "fprop", 4, 65, 65, 64, 128, 3, 2, want={"fprop/tc2/tma/128", "stride2"}),
    case("fp_1x1_s2_tma256", "fprop", 2, 33, 33, 256, 512, 1, 2, want={"fprop/tc2/tma/256", "stride2"}),
    case("fp_3x3_d2", "fprop", 2, 33, 33, 128, 128, 3, dil=2, want={"fprop/tc2/tma/128", "dil2"}),
    case("fp_3x3_d6", "fprop", 2, 33, 33, 128, 256, 3, dil=6, want={"dil6"}),
    case("fp_3x3_d12_c2048", "fprop", 2, 33, 33, 2048, 256, 3, dil=12, want={"fprop/tc1/bn128", "dil12"}),
    case("fp_3x3_d18_slices", "fprop", 2, 33, 33, 128, 128, 3, dil=18, ldx=384, offx=256, ldy=640, offy=256,
         want={"dil18", "slice_in", "slice_out"}),
    case("fp_3x3_d36", "fprop", 2, 33, 33, 64, 128, 3, dil=36, want={"dil36"}),
    case("fp_3x3_c48", "fprop", 2, 33, 33, 48, 128, 3, want={"c_tail"}),
    case("fp_simt_c20", "fprop", 2, 17, 19, 20, 64, 3, want={"fprop/simt"}),
    # BN statistics (sparse +-1 weights: |y| <= 32)
    case("fp_stats_tc1", "fprop", 4, 65, 65, 64, 64, 1, stats=True, want={"fprop/tc1/bn64", "stats"}),
    case("fp_stats_tma256", "fprop", 16, 49, 49, 64, 256, 1, stats=True, want={"fprop/tc2/tma/256", "stats"}, multi=True),
    case("fp_stats_tma128_3col", "fprop", 4, 33, 33, 128, 320, 3, stats=True, want={"fprop/tc2/tma/128", "stats"}),
    case("fp_stats_manual", "fprop", 16, 49, 49, 64, 128, 1, ldy=136, offy=4, stats=True,
         want={"fprop/tc2/manual/128", "stats"}, multi=True),
    case("fp_stats_f32", "fprop", 2, 33, 33, 64, 96, 3, f32=True, stats=True, want={"fprop/tc1/bn64", "stats"}),
    case("fp_stats_longk", "fprop", 2, 33, 33, 256, 256, 3, stats=True, want={"fprop/tc1/bn128", "stats"}),
    case("fp_stats_simt", "fprop", 2, 17, 19, 20, 64, 3, stats=True, want={"fprop/simt", "stats"}),
    # ---- dgrad ----
    case("dg_1x1_s2_zero_classes_b0", "dgrad", 2, 33, 33, 256, 512, 1, 2,  # 3 of 4 parity classes have no tap: zeros
         want={"dgrad/tc2/manual/128", "dgrad/tc1/bn128", "stride2"}),
    case("dg_1x1_s2_zero_classes_b1", "dgrad", 2, 33, 33, 256, 512, 1, 2, beta=1.0,  # ... skipped at beta = 1
         want={"dgrad/tc2/manual_beta/128", "stride2"}),
    case("dg_3x3_s2_manual_b0", "dgrad", 16, 97, 97, 128, 128, 3, 2, want={"dgrad/tc2/manual/128"}, multi=True),
    case("dg_3x3_s2_manual_b1", "dgrad", 16, 97, 97, 128, 128, 3, 2, beta=1.0, want={"dgrad/tc2/manual_beta/128"}, multi=True),
    case("dg_onetile_3x3_s2_c64_b0", "dgrad", 2, 34, 30, 64, 128, 3, 2, want={"dgrad/tc1/bn64", "stride2"}),
    case("dg_onetile_1x1_s2_c64_b0", "dgrad", 2, 33, 33, 64, 256, 1, 2, want={"dgrad/tc1/bn64"}),
    case("dg_onetile_1x1_s2_c64_b1", "dgrad", 2, 33, 33, 64, 256, 1, 2, beta=1.0, want={"dgrad/tc1/bn64"}),
    case("dg_tma128_b0", "dgrad", 16, 49, 49, 128, 256, 1, want={"dgrad/tc2/tma/128"}, multi=True),
    case("dg_tma128_b1", "dgrad", 16, 49, 49, 128, 256, 1, beta=1.0, want={"dgrad/tc2/tma/128@b1"}, multi=True),
    case("dg_tma256_b0", "dgrad", 16, 49, 49, 256, 64, 3, want={"dgrad/tc2/tma/256"}, multi=True),
    case("dg_tma256_b1", "dgrad", 16, 49, 49, 256, 64, 3, beta=1.0, want={"dgrad/tc2/tma/256@b1"}, multi=True),
    case("dg_3x3_c304_longk_b1", "dgrad", 2, 33, 33, 304, 256, 3, beta=1.0, want={"dgrad/tc1/bn128", "n_tail"}),
    case("dg_slices_b1", "dgrad", 2, 33, 33, 256, 256, 1, ldx=512, offx=128, ldy=320, offy=64, beta=1.0,
         want={"slice_in", "slice_out"}),
    case("dg_3x3_d6", "dgrad", 2, 33, 33, 256, 128, 3, dil=6, want={"dil6"}),
    case("dg_3x3_d12_b1", "dgrad", 2, 33, 33, 128, 128, 3, dil=12, beta=1.0, want={"dil12"}),
    case("dg_simt_c20_b0", "dgrad", 2, 17, 19, 20, 64, 3, want={"dgrad/simt"}),
    case("dg_simt_c20_b1", "dgrad", 2, 17, 19, 20, 64, 3, beta=1.0, want={"dgrad/simt"}),
    # ---- wgrad (split-K over pixel blocks, fp32 reductions into the packed gradient) ----
    case("wg_bn64_1x1", "wgrad", 2, 33, 33, 64, 256, 1, want={"wgrad/tc1/bn64", "map2d"}),
    case("wg_bn128_3x3_acc", "wgrad", 2, 33, 33, 128, 128, 3, old=True, want={"wgrad/tc1/bn128", "map_im2col"}),
    case("wg_bn256_3x3", "wgrad", 2, 33, 33, 256, 64, 3, dil=2, want={"wgrad/tc1/bn256"}),
    case("wg_bn64_3x3_s2", "wgrad", 2, 65, 65, 64, 128, 3, 2, want={"wgrad/tc1/bn64", "stride2"}),
    case("wg_c304_k320_acc", "wgrad", 2, 33, 33, 304, 320, 3, old=True, want={"wgrad/tc1/bn128", "m_tail", "c_tail"}),
    case("wg_c3_npq", "wgrad", 16, 129, 129, 64, 64, 1, want={"wgrad/tc1/bn64"}),  # C3's largest N*P*Q = 266 256
    case("wg_slices", "wgrad", 2, 33, 33, 256, 48, 1, ldx=320, offx=48, ldy=64, offy=8, old=True, want={"slice_in"}),
    case("wg_simt_c20", "wgrad", 2, 17, 19, 20, 64, 3, want={"wgrad/simt"}),
    # ---- the stem: im2col of the NCHW fp32 image into Kpad = 152 columns, then a 1x1 GEMM ----
    case("stem_im2col", "stem", 2, 65, 65, 3, 64, 7, 2, 3, want={"stem_im2col", "fprop/tc1/bn64"}),
]

# every production variant (kernel instantiation x epilogue x beta, plus the geometry edges) the case list must reach
REQUIRED = {
    "fprop/tc1/bn64", "fprop/tc1/bn128", "fprop/tc2/tma/128", "fprop/tc2/tma/256", "fprop/tc2/manual/128", "f32_bias",
    "map2d", "map_im2col", "stem_im2col", "stride2", "stats",
    "dgrad/tc1/bn64", "dgrad/tc1/bn128", "dgrad/tc2/tma/128", "dgrad/tc2/tma/256", "dgrad/tc2/tma/128@b1",
    "dgrad/tc2/tma/256@b1", "dgrad/tc2/manual/128", "dgrad/tc2/manual_beta/128",
    "wgrad/tc1/bn64", "wgrad/tc1/bn128", "wgrad/tc1/bn256",
    "fprop/simt", "dgrad/simt", "wgrad/simt",
    "m_tail", "n_tail", "c_tail", "slice_in", "slice_out", "dil2", "dil6", "dil12", "dil18", "dil36",
}


def geometry_tags(c):
    """Variants a case reaches by its geometry alone (the kernel variants come from the profiler)."""
    N, H, W, C, K, R = c["N"], c["H"], c["W"], c["C"], c["K"], c["R"]
    P = (H + 2 * c["pad"] - c["dil"] * (R - 1) - 1) // c["stride"] + 1
    Q = (W + 2 * c["pad"] - c["dil"] * (R - 1) - 1) // c["stride"] + 1
    tags = set()
    pointwise = R == 1 and c["stride"] == 1 and c["pad"] == 0
    if c["op"] != "stem":
        tags.add("map2d" if pointwise else "map_im2col")
    if c["stride"] == 2:
        tags.add("stride2")
    if c["dil"] > 1:
        tags.add(f"dil{c['dil']}")
    if c["f32"] and c["bias"]:
        tags.add("f32_bias")
    if c["stats"]:
        tags.add("stats")
    rows = {"fprop": N * P * Q, "dgrad": N * H * W, "wgrad": K, "stem": N * P * Q}[c["op"]]
    cols = {"fprop": K, "dgrad": C, "wgrad": C, "stem": K}[c["op"]]
    red = {"fprop": C, "dgrad": K, "wgrad": C, "stem": C}[c["op"]]
    if rows % 128:
        tags.add("m_tail")
    if cols % 128:
        tags.add("n_tail")
    if red % 64:
        tags.add("c_tail")
    if c["ldx"] > C or c["offx"]:
        tags.add("slice_out" if c["op"] == "dgrad" else "slice_in")
    if c["ldy"] > K or c["offy"]:
        tags.add("slice_in" if c["op"] == "dgrad" else "slice_out")
    return tags, P, Q


def magnitude_bound(c, amp=None):
    """amp^2 * (longest reduction: fprop C*R*S, dgrad K*R*S, wgrad N*P*Q) + max |old|: every partial sum is below this."""
    _, P, Q = geometry_tags(c)
    old = 2048 if c["old"] or c["beta"] else 0
    return (amp or amplitude(c)) ** 2 * max(c["C"] * c["R"] * c["R"], c["K"] * c["R"] * c["R"], c["N"] * P * Q) + old


def amplitude(c):
    """Operands are integers in [-amp, amp]: 4, or 2 where 16x the reduction length would reach 2^24 (the stem's wgrad at
    513^2 sums N*P*Q = 1 056 656 products)."""
    return 4 if magnitude_bound(c, 4) < LIMIT else 2


def persistent_tile_counts(M, ncols, bnt, sms):
    """Tiles of each CTA of conv_gemm_tc2's static round-robin schedule (grid as launch_v2_impl sizes it)."""
    n_tiles = -(-ncols // bnt)
    num = -(-M // 128) * n_tiles
    grid = (sms // n_tiles) * n_tiles if n_tiles <= sms else sms
    grid = min(grid, num)
    return [len(range(b, num, grid)) for b in range(grid)]


def _multi_ok(c, sms):
    _, P, Q = geometry_tags(c)
    s = c["stride"]
    bnts = {int(v.split("/")[-1].split("@")[0]) for v in c["want"] if "/tc2/" in v}
    if c["op"] == "fprop":
        shapes = [(c["N"] * P * Q, c["K"])]
    else:  # dgrad: one launch per parity class of the input pixels
        shapes = [(c["N"] * -(-(c["H"] - py) // s) * -(-(c["W"] - px) // s), c["C"]) for py in range(s) for px in range(s)]
    for M, ncols in shapes:
        for bnt in bnts:
            counts = persistent_tile_counts(M, ncols, bnt, sms)
            if min(counts) >= 2 and any(n % 2 for n in counts):
                return True
    return False


def test_case_list_covers_every_variant():
    """CPU: the hand-picked list reaches every production variant, obeys the exactness bound, and its persistent
    multi-tile cases really give each CTA >= 2 tiles with an odd count somewhere (on a 148-SM B200)."""
    covered = set()
    for c in CASES:
        tags, _, _ = geometry_tags(c)
        covered |= c["want"] | tags
        assert magnitude_bound(c) < LIMIT, c["name"]
        if c["multi"]:
            assert _multi_ok(c, 148), c["name"]
    missing = REQUIRED - covered
    assert not missing, f"no case reaches {sorted(missing)}"
    assert len({c["name"] for c in CASES}) == len(CASES)


# ------------------------------------------------------------------------------------------------ exact references
def ints(shape, g, lo=-4, hi=4):
    return torch.randint(lo, hi + 1, shape, generator=g).double()


def sparse_pm1(K, C, R, g, nnz=8):
    """[K, C, R, R] with at most `nnz` entries of +-1 per output channel: |y| <= 4 * nnz for x in [-4, 4]."""
    w = torch.zeros(K, C * R * R, dtype=torch.float64)
    for k in range(K):
        pos = torch.randperm(C * R * R, generator=g)[:nnz]
        w[k, pos] = (torch.randint(0, 2, (pos.numel(),), generator=g) * 2 - 1).double()
    return w.reshape(K, C, R, R)


def bf16(t):
    """Round-to-nearest-even to bf16 (exact here: every value is an integer below 2^24, so the float32 step is exact)."""
    return t.float().to(torch.bfloat16)


def strided(flat, shape, ld, off):
    n, h, w, c = shape
    return flat.as_strided(shape, (h * w * ld, w * ld, ld, 1), off)


def placed(vals_nhwc, ld, off, fill, dtype):
    """A flat buffer holding vals_nhwc as rows of pitch ld starting at element `off`; everything else = fill."""
    n, h, w, c = vals_nhwc.shape
    flat = torch.full((n * h * w * ld + off + 8,), fill, dtype=dtype)
    strided(flat, vals_nhwc.shape, ld, off).copy_(vals_nhwc.to(dtype))
    return flat


KERNEL_RES = [
    (re.compile(r"conv_gemm_tc<\s*(?:\(int\))?(\d+)\s*,\s*(?:\(int\))?\d+\s*,\s*(?:\(int\))?(\d+)\s*>"),
     lambda m: f"{OPS[int(m[2])]}/tc1/bn{m[1]}"),
    (re.compile(r"conv_gemm_tc2<\s*(?:\(int\))?(\d+)\s*,\s*(?:\(int\))?(\d+)\s*,\s*(?:\(int\))?(\d+)\s*>"),
     lambda m: f"{OPS[int(m[1])]}/tc2/{EPIS[int(m[2])]}/{m[3]}"),
    (re.compile(r"igemm_simt<\s*(?:\(int\))?(\d+)\s*>"), lambda m: f"{OPS[int(m[1])]}/simt"),
    (re.compile(r"im2col_kernel"), lambda m: "stem_im2col"),
]


def variants_of(names, beta):
    out = set()
    for n in names:
        for rx, fn in KERNEL_RES:
            m = rx.search(n)
            if m:
                v = fn(m)
                out.add(v + "@b1" if (beta and "/tma/" in v) else v)
    return out


def run_profiled(fn, beta):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return variants_of({e.name for e in prof.events()}, beta)


def run_case(c, seed):
    """Run one case on the GPU with integer data; assert the bit-exact expectation.  Returns the variants launched."""
    g = torch.Generator().manual_seed(seed)
    a = amplitude(c)
    op, N, H, W, C, K, R = c["op"], c["N"], c["H"], c["W"], c["C"], c["K"], c["R"]
    st, pad, dil, beta = c["stride"], c["pad"], c["dil"], c["beta"]
    assert magnitude_bound(c) < LIMIT, f"{c['name']}: partial sums may exceed 2^24; the expectation would not be exact"
    _, P, Q = geometry_tags(c)
    if c["stats"]:  # y^2 <= 1024 summed over the rows of one CTA (persistent kernel, 128-wide tiles: the fewest CTAs a column)
        rows = -(-(-(-(N * P * Q) // 128)) // max(1, 148 // -(-K // 128))) * 128
        assert 1024 * rows < LIMIT, f"{c['name']}: a CTA's fp32 sum of squares may not be exact"
    if op == "stem":
        x = ints((N, C, H, W), g, -a, a)
        w = ints((K, C, R, R), g, -a, a)
        kpad = 152
        wp = ops.pack_weight(w.permute(0, 2, 3, 1).reshape(K, C * R * R, 1, 1).contiguous().float().to(DEV), cpad=kpad)
        xd = x.float().to(DEV)
        box = {}
        v = run_profiled(lambda: box.update(y=ops.conv2d_fwd(ops.im2col(xd, R, R, st, pad, dil, kpad, nchw_f32=True), wp, K, 1, 1)), 0)
        exp = bf16(F.conv2d(x, w, None, st, pad, dil).permute(0, 2, 3, 1))
        assert torch.equal(box["y"].cpu(), exp), f"{c['name']}: stem output differs from RNE(exact)"
        return v
    if op == "fprop":
        x = ints((N, C, H, W), g, -a, a)
        w = sparse_pm1(K, C, R, g) if c["stats"] else ints((K, C, R, R), g, -a, a)
        b = ints((K,), g, -64, 64) if c["bias"] else None
        ref = F.conv2d(x, w, b, st, pad, dil).permute(0, 2, 3, 1)
        odt = torch.float32 if c["f32"] else torch.bfloat16
        xflat = placed(x.permute(0, 2, 3, 1), c["ldx"], c["offx"], 0.0, torch.bfloat16).to(DEV)
        yflat0 = torch.full((N * P * Q * c["ldy"] + c["offy"] + 8,), 7.0, dtype=odt)  # sentinel outside the slice
        yflat = yflat0.to(DEV)
        wp = ops.pack_weight(w.float().to(DEV))
        stats = ops.new_stats(K, DEV) if c["stats"] else None
        bd = b.float().to(DEV) if b is not None else None
        xv = strided(xflat, (N, H, W, C), c["ldx"], c["offx"])
        yv = strided(yflat, (N, P, Q, K), c["ldy"], c["offy"])
        call = lambda: ops.conv2d_fwd(xv, wp, K, R, R, st, pad, dil, out=yv, bias=bd, stats=stats, impl=IMPL_AUTO)
        v = run_profiled(call, 0)
        exp_vals = ref.float() if c["f32"] else bf16(ref)
        exp = yflat0.clone()
        strided(exp, (N, P, Q, K), c["ldy"], c["offy"]).copy_(exp_vals)
        got = yflat.cpu()
        if not torch.equal(got, exp):
            gv, ev = strided(got, (N, P, Q, K), c["ldy"], c["offy"]), exp_vals
            bad = (gv.double() != ev.double()).nonzero()
            outside = not torch.equal(got.masked_fill(_slice_mask(got.shape[0], (N, P, Q, K), c["ldy"], c["offy"]), 0),
                                      exp.masked_fill(_slice_mask(got.shape[0], (N, P, Q, K), c["ldy"], c["offy"]), 0))
            pytest.fail(f"{c['name']}: {bad.shape[0]} outputs differ from the exact value (first {bad[:4].tolist()}: "
                        f"got {[gv[tuple(i)].item() for i in bad[:4]]} want {[ev[tuple(i)].item() for i in bad[:4]]}); "
                        f"writes outside the output slice: {outside}")
        if stats is not None:
            yd = exp_vals.double().reshape(-1, K)
            want = torch.cat([yd.sum(0), (yd * yd).sum(0)])
            assert torch.equal(stats.cpu(), want), f"{c['name']}: BN statistics differ from the exact sums of the stored output"
        return v
    if op == "dgrad":
        w = ints((K, C, R, R), g, -a, a)
        dy = ints((N, K, P, Q), g, -a, a)
        acc = torch.nn.grad.conv2d_input((N, C, H, W), w, dy, st, pad, dil).permute(0, 2, 3, 1)
        dyflat = placed(dy.permute(0, 2, 3, 1), c["ldy"], c["offy"], 0.0, torch.bfloat16).to(DEV)
        old = bf16(ints((N, H, W, C), g, -2048, 2048)) if beta else torch.full((N, H, W, C), 7.0).to(torch.bfloat16)
        xflat0 = placed(old, c["ldx"], c["offx"], 5.0, torch.bfloat16)
        xflat = xflat0.to(DEV)
        wp = ops.pack_weight(w.float().to(DEV))
        dyv = strided(dyflat, (N, P, Q, K), c["ldy"], c["offy"])
        xv = strided(xflat, (N, H, W, C), c["ldx"], c["offx"])
        call = lambda: ops.conv2d_dgrad(dyv, wp, (N, H, W, C), R, R, st, pad, dil, out=xv, beta=beta, impl=IMPL_AUTO)
        v = run_profiled(call, beta)
        simt_path = any(s.endswith("/simt") for s in v)
        if not beta:
            exp_vals = bf16(acc)
        elif simt_path:  # igemm_simt: fp32 add of the old value, one rounding
            exp_vals = bf16(old.double() + acc)
        else:  # tcgen05 epilogues: the tile is rounded to bf16 first, then added
            exp_vals = bf16(old.double() + bf16(acc).double())
        exp = xflat0.clone()
        strided(exp, (N, H, W, C), c["ldx"], c["offx"]).copy_(exp_vals)
        got = xflat.cpu()
        if not torch.equal(got, exp):
            gv = strided(got, (N, H, W, C), c["ldx"], c["offx"])
            bad = (gv.double() != exp_vals.double()).nonzero()
            alt = bf16(old.double() + acc) if beta and not simt_path else None
            pytest.fail(f"{c['name']}: {bad.shape[0]} of {exp_vals.numel()} gradients differ (first {bad[:4].tolist()}: got "
                        f"{[gv[tuple(i)].item() for i in bad[:4]]} want {[exp_vals[tuple(i)].item() for i in bad[:4]]})"
                        + (f"; equal to RNE(old + acc) instead: {torch.equal(gv, alt)}" if alt is not None else ""))
        return v
    # wgrad
    x = ints((N, C, H, W), g, -a, a)
    dy = ints((N, K, P, Q), g, -a, a)
    exact = torch.nn.grad.conv2d_weight(x, (K, C, R, R), dy, st, pad, dil)
    xflat = placed(x.permute(0, 2, 3, 1), c["ldx"], c["offx"], 0.0, torch.bfloat16).to(DEV)
    dyflat = placed(dy.permute(0, 2, 3, 1), c["ldy"], c["offy"], 0.0, torch.bfloat16).to(DEV)
    old = ints((K, C, R, R), g, -1000, 1000) if c["old"] else torch.zeros(K, C, R, R, dtype=torch.float64)
    dwp = old.permute(2, 3, 0, 1).reshape(R * R, K, C).contiguous().float().to(DEV)  # packed [tap][K][C]
    xv = strided(xflat, (N, H, W, C), c["ldx"], c["offx"])
    dyv = strided(dyflat, (N, P, Q, K), c["ldy"], c["offy"])
    call = lambda: ops.conv2d_wgrad(dyv, xv, R, R, st, pad, dil, out=dwp, impl=IMPL_AUTO)
    v = run_profiled(call, 0)
    got = ops.unpack_wgrad(dwp, (K, C, R, R)).cpu()
    want = (old + exact).float()
    if not torch.equal(got, want):
        bad = (got != want).nonzero()
        pytest.fail(f"{c['name']}: {bad.shape[0]} weight-gradient entries differ (first {bad[:4].tolist()}: got "
                    f"{[got[tuple(i)].item() for i in bad[:4]]} want {[want[tuple(i)].item() for i in bad[:4]]})")
    return v


def _slice_mask(n, shape, ld, off):
    m = torch.zeros(n, dtype=torch.bool)
    strided(m, shape, ld, off).fill_(True)
    return m


def _log(gpu_out_dir, line):
    with open(os.path.join(gpu_out_dir, "conv_coverage.txt"), "a") as f:
        f.write(line + "\n")


@pytest.mark.gpu
@pytest.mark.parametrize("c", CASES, ids=[c["name"] for c in CASES])
def test_conv_exact(c, gpu_out_dir):
    hit = run_case(c, seed=sum(map(ord, c["name"])))
    tags, _, _ = geometry_tags(c)
    _log(gpu_out_dir, f"{c['name']}: {' '.join(sorted(hit | tags))}")
    missing = c["want"] - hit - tags
    assert not missing, f"{c['name']} launched {sorted(hit)}, not {sorted(missing)}: the dispatch moved this shape"
    if c["multi"]:
        assert _multi_ok(c, torch.cuda.get_device_properties(0).multi_processor_count), c["name"]


# ------------------------------------------------------------------------------------------------ flagship replay
C_CONFIGS = {  # bench.py CONFIGS: architecture, constructor keywords, classes, crop, batch
    "C3": ("DeepLab", dict(backbone="resnet101", output_stride=16), 19, 513, 16),
    "C2": ("PSPNet", dict(backbone="resnet50"), 21, 473, 16),
}


def _align(t):
    return (t.data_ptr() // t.element_size()) % 8


def record_step_geometries(cfg, monkeypatch):
    """Distinct conv geometries (with pitches, alignments, dtype, beta, stats / bias / out= flags) of one train step."""
    import seg_b200
    from seg_b200.train import FusedTrainStep
    arch, kw, nc, size, batch = C_CONFIGS[cfg]
    torch.manual_seed(0)
    model = getattr(seg_b200, arch)(nc, pretrained=False, **kw).to(DEV).train()
    stepper = FusedTrainStep(model, ignore_index=255, lr=0.01, backbone_lr_scale=0.1, momentum=0.9, weight_decay=1e-4)
    seen = {}
    real = (ops.conv2d_fwd, ops.conv2d_dgrad, ops.conv2d_wgrad)

    def fwd(x, w_packed, K, R, S, stride=1, pad=0, dil=1, out=None, out_dtype=torch.bfloat16, bias=None, beta=0.0, stats=None, **kw):
        y = real[0](x, w_packed, K, R, S, stride, pad, dil, out=out, out_dtype=out_dtype, bias=bias, beta=beta, stats=stats, **kw)
        N, H, W, C = x.shape
        key = ("fprop", N, H, W, C, K, R, stride, pad, dil, ops.ld(x), _align(x), ops.ld(y), _align(y),
               y.dtype == torch.float32, bias is not None, float(beta), stats is not None, False)
        seen[key] = seen.get(key, 0) + 1
        return y

    def dgrad(dy, w_packed, x_shape, R, S, stride=1, pad=0, dil=1, out=None, beta=0.0, **kw):
        dx = real[1](dy, w_packed, x_shape, R, S, stride, pad, dil, out=out, beta=beta, **kw)
        N, H, W, C = x_shape
        key = ("dgrad", N, H, W, C, dy.shape[-1], R, stride, pad, dil, ops.ld(dx), _align(dx), ops.ld(dy), _align(dy),
               False, False, float(beta if out is not None else 0.0), False, False)
        seen[key] = seen.get(key, 0) + 1
        return dx

    def wgrad(dy, x, R, S, stride=1, pad=0, dil=1, out=None, **kw):
        dw = real[2](dy, x, R, S, stride, pad, dil, out=out, **kw)
        N, H, W, C = x.shape
        key = ("wgrad", N, H, W, C, dy.shape[-1], R, stride, pad, dil, ops.ld(x), _align(x), ops.ld(dy), _align(dy),
               False, False, 0.0, False, out is not None)
        seen[key] = seen.get(key, 0) + 1
        return dw

    monkeypatch.setattr(ops, "conv2d_fwd", fwd)
    monkeypatch.setattr(ops, "conv2d_dgrad", dgrad)
    monkeypatch.setattr(ops, "conv2d_wgrad", wgrad)
    g = torch.Generator().manual_seed(1234)
    x = torch.randn(batch, 3, size, size, generator=g).to(DEV)
    y = torch.randint(0, nc, (batch, size, size), generator=g).to(DEV)
    stepper.step(x, y)
    torch.cuda.synchronize()
    monkeypatch.undo()
    del stepper, model
    torch.cuda.empty_cache()
    return seen


def case_from_key(key, i):
    op, N, H, W, C, K, R, stride, pad, dil, ldx, ax, ldy, ay, f32, bias, beta, stats, has_out = key
    assert R in (1, 3), key
    return case(f"replay{i}", op, N, H, W, C, K, R, stride, pad, dil, want=set(), ldx=ldx, offx=ax, ldy=ldy, offy=ay,
                beta=beta, f32=f32, bias=bias, stats=stats, old=has_out)


@pytest.mark.gpu
@pytest.mark.parametrize("cfg", ["C3", "C2"])
def test_replay_flagship_geometries(cfg, monkeypatch, gpu_out_dir):
    """Every distinct conv call of one training step of the configuration, replayed with integer data and checked bit for
    bit: the layer shapes, pitches and slice alignments of the real model, so the real epilogue choices."""
    seen = record_step_geometries(cfg, monkeypatch)
    assert len(seen) > 20, f"{cfg}: only {len(seen)} distinct conv geometries recorded"
    hit = {}
    for i, key in enumerate(sorted(seen, key=str)):
        c = case_from_key(key, i)
        v = run_case(c, seed=1000 + i)
        for name in v:
            hit[name] = hit.get(name, 0) + 1
        _log(gpu_out_dir, f"{cfg} replay {key[0]} N{key[1]} {key[2]}x{key[3]} C{key[4]} K{key[5]} R{key[6]} s{key[7]} "
                          f"p{key[8]} d{key[9]} ldx{key[10]}+{key[11]} ldy{key[12]}+{key[13]} f32={key[14]} bias={key[15]} "
                          f"beta={key[16]} stats={key[17]} out={key[18]} x{seen[key]}: {' '.join(sorted(v))}")
    summary = f"{cfg} replay: {len(seen)} distinct geometries; variants reached: " + ", ".join(f"{k} ({n})" for k, n in sorted(hit.items()))
    print(summary)
    _log(gpu_out_dir, summary)


# ------------------------------------------------------------------------------------------------ weight packing
def _torch_pack(w, cpad, explicit):
    K, C, R, S = w.shape
    if explicit:
        m = torch.zeros(1, K, cpad)
        m[0, :, : R * S * C] = w.permute(0, 2, 3, 1).reshape(K, R * S * C)
    else:
        m = torch.zeros(R * S, K, cpad)
        m[:, :, :C] = w.permute(2, 3, 0, 1).reshape(R * S, K, C)
    return m.to(torch.bfloat16)


def _torch_unpack(p, shape, explicit):
    K, C, R, S = shape
    if explicit:
        return p[0, :, : R * S * C].reshape(K, R, S, C).permute(0, 3, 1, 2).contiguous()
    return p[:, :, :C].reshape(R, S, K, C).permute(2, 3, 0, 1).contiguous()


PACK_SHAPES = [(64, 3, 7, 7, 152, 1)] + [  # the stem, explicit [K][(r,s,c) padded to Cpad]
    (K, C, R, R, C, 0) for K, C, R in
    [(64, 64, 1), (64, 64, 3), (256, 64, 1), (128, 256, 1), (128, 128, 3), (512, 2048, 1), (256, 2048, 3), (19, 256, 1),
     (48, 256, 1), (256, 304, 3), (21, 512, 1), (64, 20, 3), (12, 12, 1)]
] + [(40, 24, 3, 3, 32, 0)]  # Cpad > C on a 3x3


@pytest.mark.gpu
def test_weight_packing_bit_exact():
    """pack_weight / unpack_wgrad (beta 0 and 1) and the batched table forms over a heterogeneous table of >= 100 entries,
    against each other and against torch permute / pad / .to(bfloat16) (round to nearest even)."""
    g = torch.Generator().manual_seed(21)
    shapes = [PACK_SHAPES[i % len(PACK_SHAPES)] for i in range(112)]
    ws = [torch.randn(K, C, R, S, generator=g) * 3 for K, C, R, S, _, _ in shapes]
    dt = np.dtype([("oihw", "<u8"), ("packed", "<u8"), ("K", "<i4"), ("C", "<i4"), ("R", "<i4"), ("S", "<i4"),
                   ("Cpad", "<i4"), ("explicit", "<i4"), ("start", "<i8")])  # seg_b200.train.WeightTables' record
    assert dt.itemsize == lib.load().seg_pack_entry_bytes()
    wd = [w.to(DEV) for w in ws]
    packed = [torch.full((1, K, cp) if ex else (R * S, K, cp), 3.0, dtype=torch.bfloat16, device=DEV)
              for K, C, R, S, cp, ex in shapes]
    tab, start = np.zeros(len(shapes), dtype=dt), 0
    for i, ((K, C, R, S, cp, ex), w, p) in enumerate(zip(shapes, wd, packed)):
        tab[i] = (w.data_ptr(), p.data_ptr(), K, C, R, S, cp, ex, start)
        start += p.numel()
    lib.call("seg_pack_weights_batched", torch.from_numpy(tab.view(np.uint8).copy()).to(DEV).data_ptr(), len(shapes), start)
    for (K, C, R, S, cp, ex), w, p in zip(shapes, ws, packed):
        want = _torch_pack(w, cp, ex)
        assert torch.equal(p.cpu(), want), f"batched pack {K}x{C}x{R}x{S} Cpad={cp} explicit={ex}"
        if ex:
            single = ops.pack_weight(w.permute(0, 2, 3, 1).reshape(K, R * S * C, 1, 1).contiguous().to(DEV), cpad=cp)
        else:
            single = ops.pack_weight(w.to(DEV), cpad=cp)
        assert torch.equal(single.cpu(), want), f"pack_weight {K}x{C}x{R}x{S} Cpad={cp}"
    # unpack: fp32 packed gradients -> OIHW, overwrite (beta 0) and accumulate (beta 1)
    dps = [torch.randn(p.shape, generator=g) for p in packed]
    olds = [torch.randn(K, C, R, S, generator=g) for K, C, R, S, _, _ in shapes]
    for beta in (0.0, 1.0):
        outs = [o.to(DEV) for o in olds]
        dpd = [d.to(DEV) for d in dps]
        tab, start = np.zeros(len(shapes), dtype=dt), 0
        for i, ((K, C, R, S, cp, ex), o, d) in enumerate(zip(shapes, outs, dpd)):
            tab[i] = (o.data_ptr(), d.data_ptr(), K, C, R, S, cp, ex, start)
            start += o.numel()
        lib.call("seg_unpack_wgrads_batched", torch.from_numpy(tab.view(np.uint8).copy()).to(DEV).data_ptr(), len(shapes), start, beta)
        for (K, C, R, S, cp, ex), o, d, old in zip(shapes, outs, dps, olds):
            want = _torch_unpack(d, (K, C, R, S), ex) + (old if beta else 0.0)
            assert torch.equal(o.cpu(), want), f"batched unpack beta={beta} {K}x{C}x{R}x{S} explicit={ex}"
            if not ex:
                single = ops.unpack_wgrad(d.to(DEV), (K, C, R, S), beta=beta, out=old.to(DEV))
                assert torch.equal(single.cpu(), want), f"unpack_wgrad beta={beta} {K}x{C}x{R}x{S}"
