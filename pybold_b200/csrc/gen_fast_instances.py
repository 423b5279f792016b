"""Writes one translation unit per register-tiled solver variant plus the dispatch table.

    python gen_fast_instances.py OUTDIR        (the Makefile runs it with OUTDIR = build/gen)

Each unit defines one Variant (pb_fast_registry.h) from its family's factory; pb_fast_table.inc
lists them per dtype for pb_fast_registry.cu.  Nothing it writes is committed: the lists below are
the record of the variants and of why each exists.  Files whose content is unchanged are left alone,
so that editing one row recompiles that unit and the table only.  Prints the units' paths.

Warp rows: (real, R, KMAX, CIRC, ...).  R = samples per lane (32 R >= T), KMAX = unrolled tap count
(>= K), CIRC = wrap-around variant (T % R == 0 and idle lanes >= halo, see pb_fast.cuh).
"""
import os
import sys

VARIANTS = [
    # (real, R, KMAX, CIRC, warps per CTA, min CTAs per SM) -- launch bounds picked by the sweep
    # in tools/exp_bd.cu on a B200 (profiles/r01_launch_bounds_sweep.txt)
    ("float", 10, 20, True, 4, 5),    # cfg2 / cfg3: T = 300, K = 20
    ("float", 40, 28, True, 8, 1),    # cfg4: T = 1200, K = 28
    ("float", 20, 20, True, 1, 12),   # cfg5: T = 600, K = 20
    ("float", 8, 28, False, 4, 4),    # ICASSP native: T = 240, K = 27
    ("float", 10, 20, False, 4, 5),
    ("float", 10, 32, False, 4, 3),
    ("float", 20, 20, False, 4, 3),
    ("float", 20, 32, False, 4, 2),
    ("float", 40, 32, False, 8, 1),
    # double: parity builds of the same template
    ("double", 10, 20, True, 4, 1),
    ("double", 8, 28, False, 4, 1),
    ("double", 10, 20, False, 4, 1),
    ("double", 10, 32, False, 4, 1),
    ("double", 20, 32, False, 4, 1),
]


# Group variants (pb_fastg.cuh): (real, R, KMAX, G lanes per voxel, TAIL, warps per CTA, min CTAs/SM).
# Used by bd when early stopping is off; 32/G voxels per warp.  Picked by tools/exp_bdg.cu.
# Round 2, end: the two-voxels-per-warp variants run as ONE-warp CTAs, twelve per SM (same 12 warps and 168
# registers as four-warp CTAs x 3, no CTA-wide barrier, one task queue reader per CTA): measured +1.6 % at
# T = 300, +3.5 % at 240 / K = 27, +7.7 % at 200, +7.4 % at 320 (tools/exp_bdg.cu sets 9, 10); the four-voxel
# variants (G = 8) gain 2 ... 6 % at R = 10, 13, 20 and nothing at R = 16, 24 (kept on four-warp CTAs).
GVARIANTS = [
    ("float", 19, 20, 16, 8, 1, 12),   # T in [296, 304], K <= 20   (cfg3: T = 300)
    ("float", 15, 28, 16, 8, 1, 12),   # T in [232, 240], K <= 28   (ICASSP native: T = 240, K = 27)
    ("double", 19, 20, 16, 8, 1, 8),   # parity build of the group kernel
] + [
    # general coverage of 192 < T <= 320 (two voxels per warp), any tail (TAIL = R)
    ("float", R, K, 16, R, 1, 12) for K in (20, 28) for R in range(13, 21)
] + [
    # 320 < T <= 352 with K <= 20 (measured +8 % over the one-warp CTA variant; with 28 taps the
    # register pressure makes it a tie, not built)
    ("float", R, 20, 16, R, 1, 12) for R in (21, 22)
] + [
    # short series, 40 < T <= 192: four voxels per warp (G = 8), every slot maskable.  Launch bounds: the
    # 28-tap variants spill at 168 registers (measured +8 % at R = 16, +23 % at R = 24 with 255, round 2)
    # (one-warp CTAs where they measured faster: T = 64 +5.9 %, 100 +2.8 %, 150 +2.4 %; R = 16 the same, R = 24 -0.9 %)
    ("float", R, 20, 8, R, 1 if R in (10, 13, 20) else 4, 12 if R in (10, 13, 20) else 3) for R in (10, 13, 16, 20, 24)
] + [
    # ... but with 28 taps the four double-precision scratch areas of a warp (8.5 KB per voxel) leave room for
    # one CTA per SM only: two voxels per warp with few samples per lane are faster (measured, round 2:
    # T = 96 +14 %, T = 128 +9 %, T = 190 +44 %; profiles/r02_exp_short_series.txt)
    ("float", R, 28, 16, R, 1, 12) for R in (4, 6, 8, 10, 12)
]


# CTA variants (pb_fastc.cuh): (real, R, KMAX, NW warps per voxel, min CTAs/SM): one CTA per voxel,
# halo exchange through shared memory.  Long series (T ~ 600 with one warp, T ~ 1200 with two).
CVARIANTS = [
    # R = 12 and R = 20 only: the per-lane stride of the halo buffers (R floats) must not be a
    # multiple of 8 banks, R = 16 (64-byte stride) stores with 4-way bank conflicts (measured 29 vs
    # 42 Tflop/s per occupied slot).  A variant serves T in (16 NW R - R, 32 NW R]; the dispatcher
    # takes the one with the fewest slots.  Three warps of R = 12 were measured slower per slot
    # (34 M vs 41 M slots/s) than two warps of R = 20 for every T in (768, 1152] and are not built.
    ("float", 20, 28, 2, 6),     # cfg4: T = 1200, K = 28  (T in (620, 1280])
    ("float", 20, 20, 1, 12),    # cfg5: T = 600, K = 20   (T in (300, 640])
    ("float", 20, 28, 1, 10),    # T ~ 600 with short TR
    ("float", 12, 20, 1, 12),    # T in (320, 384]: between the group kernels and R = 20
    ("float", 12, 28, 1, 10),
    ("float", 12, 20, 2, 8),     # T in (640, 768]
    ("float", 12, 28, 2, 8),
    ("float", 20, 20, 4, 3),     # long runs: T in (1260, 2560]
    ("float", 20, 28, 4, 3),
    ("double", 20, 28, 2, 1),    # parity builds
    ("double", 20, 20, 1, 1),
    # round 2: eight warps per voxel for 2540 < T <= 5120 (PB_MAX_T = 4096)
    ("float", 20, 20, 8, 2),
    ("float", 20, 28, 8, 2),
    # round 2: K <= 20 at 640 < T <= 1280 ran the 28-tap tile; three warps per voxel for 1260 < T <= 1920
    # (T = 1500 filled 59 % of the four-warp variant's slots)
    ("float", 20, 20, 2, 6),
    ("float", 20, 20, 3, 4),
    ("float", 20, 28, 3, 4),
] + [
    # round 2: R = 16 with the skewed shared-memory layout (pb_fastc.cuh: SKEW): fills the gaps between the
    # R = 12 and R = 20 variants -- T in (384, 512], (768, 1024], (1152, 1536], (1536, 2048], (3072, 4096]
    ("float", 16, K, NW, M) for K in (20, 28) for (NW, M) in ((1, 12), (2, 6), (3, 4), (4, 3), (8, 2))
] + [
    # six warps per voxel: two CTAs of 168-register threads per SM (eight warps leave room for one, or spill
    # at 128 registers): 2560 < T <= 4096
    # (R = 24 was measured slower than eight warps of R = 16 at T = 4096 and is not built)
    ("float", R, K, 6, 2) for K in (20, 28, 40) for R in (16, 20)
] + [
    # round 2: short-TR acquisitions, 28 < K <= 40 (TR >= 0.5 s) and K <= 64 (TR >= 0.32 s), every T <= 4096.
    # More taps, more registers (taps, halo and tile live in registers): launch bounds leave ~170 (K = 40)
    # and ~250 (K = 64) registers per thread
    ("float", R, 40, NW, M)
    for (R, NW, M) in ((4, 1, 12), (8, 1, 12), (12, 1, 12), (20, 1, 12), (20, 2, 6), (20, 4, 3), (20, 8, 1),
                       # the gaps between them (as for K <= 28): T in (384, 512], (640, 768], (768, 1024],
                       # (1280, 1536], (1536, 1920], (1920, 2048]
                       (16, 1, 12), (12, 2, 6), (16, 2, 6), (16, 3, 4), (20, 3, 4), (16, 4, 3))
] + [
    ("float", R, 64, NW, M)
    for (R, NW, M) in ((4, 1, 8), (8, 1, 8), (12, 1, 8), (20, 1, 8), (20, 2, 4), (20, 4, 2), (20, 8, 1),
                       (16, 1, 8), (12, 2, 4), (16, 2, 4), (20, 3, 2),
                       # the 64-tap scratch (double Gram matrix) leaves room for four CTAs per SM: with one
                       # warp per voxel that is four warps per SM, with two it is the eight the registers allow
                       (4, 2, 4), (8, 2, 4))
]


DTYPE = {"float": "f32", "double": "f64"}


def rows():
    """(real, tag, family header, factory call) per variant, in the order the dispatcher searches them:
    CTA rows, then group rows, then warp rows (ties go to the first row)."""
    for real, R, K, NW, M in CVARIANTS:
        yield (real, "%s_r%d_k%d_w%d" % (DTYPE[real], R, K, NW), "pb_fastc.cuh",
               "cta_variant<%s, %d, %d, %d, %d>" % (real, R, K, NW, M))
    for real, R, K, G, tail, W, M in GVARIANTS:
        yield (real, "%s_r%d_k%d_g%d_t%d" % (DTYPE[real], R, K, G, tail), "pb_fastg.cuh",
               "group_variant<%s, %d, %d, %d, %d, %d, %d>" % (real, R, K, G, tail, W, M))
    for real, R, K, circ, W, M in VARIANTS:
        yield (real, "%s_r%d_k%d_%s" % (DTYPE[real], R, K, "circ" if circ else "lin"), "pb_fast.cuh",
               "warp_variant<%s, %d, %d, %s, %d, %d>" % (real, R, K, "true" if circ else "false", W, M))


def write(path, text):
    """Writes text unless the file already holds it, so that make recompiles only what changed."""
    if os.path.exists(path):
        with open(path) as f:
            if f.read() == text:
                return
    with open(path, "w") as f:
        f.write(text)


HEAD = "// GENERATED by gen_fast_instances.py -- do not edit.\n"


def main(out):
    os.makedirs(out, exist_ok=True)
    decls, table, srcs = [], {real: [] for real in DTYPE}, []
    for real, tag, header, factory in rows():
        src = os.path.join(out, "pb_fast_inst_%s.cu" % tag)
        write(src, HEAD + '#include "%s"\n\nnamespace pb {\nextern const Variant<%s> variant_%s = %s();\n}\n'
              % (header, real, tag, factory))
        srcs.append(src)
        decls.append("extern const Variant<%s> variant_%s;\n" % (real, tag))
        table[real].append("    &variant_%s,\n" % tag)
    arrays = ["static const Variant<%s> *const variants_%s[] = {\n%s};\n" % (real, DTYPE[real], "".join(table[real]))
              for real in DTYPE]
    write(os.path.join(out, "pb_fast_table.inc"), HEAD + "".join(decls) + "".join(arrays))
    print(" ".join(srcs))


if __name__ == "__main__":
    main(sys.argv[1])
