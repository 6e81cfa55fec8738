"""Generates the committed golden fixtures from UPSTREAM ITSELF (oracle/_ref, i.e. the
unmodified reference headers compiled with the pinned flags -O2 -mavx2 -ffp-contract=off).

Run in the build container (where /root/reference exists):
    python tests/golden/make_golden.py
Each avir_*.npz holds: case tuple, seeded input image, upstream's output image.
Each lancir_*.npz holds: geometry, input, upstream CLancIR output.
Fixtures are small (<= ~100 KB each) so they can live in git.

upstream.json holds, for every other comparison of the suite and smoke() with upstream, the digest of
upstream's output (cases.digest), keyed by the call and the digest of its input (cases.upstream).  It
is recorded by running them with oracle/_ref built, on a machine with a B200 for the GPU tests:
    rm tests/golden/upstream.json; export AVIRB200_RECORD_UPSTREAM=$PWD/tests/golden/upstream.json
    python -m pytest tests; python -c "import __graft_entry__ as g; g.smoke()"
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

import cases as cs  # noqa: E402
import oracle_ref as o  # noqa: E402

u8, u16, f32, f64 = np.uint8, np.uint16, np.float32, np.float64

GOLDEN_CASES = [
    (1, 60, 34, 120, 68, 4, u8, u8, 8, {"buildmode": 1}),          # cfg2 chain
    (1, 60, 34, 120, 68, 4, u8, u8, 8, {}),                        # filtered-upsample chain
    (2, 96, 54, 48, 27, 4, f32, f32, 16, {"buildmode": 1}),        # cfg3, float8_dil mirror
    (1, 96, 54, 48, 27, 4, f32, f32, 16, {"buildmode": 0}),        # cfg3, float4 mirror
    (1, 128, 128, 32, 32, 4, u16, u16, 16, {}),                    # cfg4 chain
    (2, 96, 54, 24, 14, 4, u8, u8, 8, {"gamma": True, "alpha": 3, "buildmode": 1}),  # cfg5
    (0, 64, 48, 100, 75, 3, u8, u8, 8, {}),                        # cfg1 geometry via AVIR
    (1, 75, 50, 50, 33, 4, u8, u16, 16, {}),
    (0, 50, 30, 65, 49, 4, u8, u8, 6, {}),
    (2, 50, 30, 33, 21, 2, u16, u16, 16, {"gamma": True}),
    (1, 40, 30, 20, 15, 4, u8, u8, 8, {"ox": 0.37, "oy": -0.21}),
    (0, 90, 60, 11, 7, 1, f32, f32, 16, {}),
    # error-diffusion classes (fpclass codes 3..5), double image buffers
    (3, 60, 40, 45, 50, 4, u8, u8, 8, {}),
    (5, 60, 40, 45, 50, 4, u8, u8, 6, {"gamma": True, "alpha": 3}),   # planar class: cross-plane quirk
    (4, 60, 40, 30, 70, 3, u16, u16, 12, {}),
    (1, 60, 40, 30, 20, 4, f64, f64, 16, {}),
    (0, 60, 40, 45, 50, 3, f64, u16, 16, {"gamma": True}),
]

LANCIR_CASES = [
    (96, 54, 48, 27, u8, u8, {}),
    (64, 48, 103, 77, u8, u8, {}),
    (64, 64, 16, 16, u16, u16, {}),
    (50, 30, 33, 17, f32, f32, {}),
    (60, 40, 40, 27, u8, u16, {}),
]

# (sw, sh, nw, nh, channels, Tin, Tout, la): upstream's 1-3 channel summation trees
LANCIR_C_CASES = [
    (64, 48, 103, 77, 3, u8, u8, 3.0),      # BASELINE cfg1 ratio (k = 0.625), RGB
    (64, 48, 103, 77, 1, u8, u8, 3.0),
    (64, 48, 103, 77, 2, u16, u16, 3.0),
    (77, 51, 47, 29, 3, f32, f32, 3.0),     # kernel length 10: kl % 4 == 2 tail
    (77, 51, 47, 29, 1, f32, f32, 3.0),
    (77, 51, 47, 29, 2, f32, u8, 3.0),
]


def main():
    assert o.have_ref(), "build oracle/_ref first (make -C oracle ref)"
    for i, case in enumerate(GOLDEN_CASES):
        src = cs.make_input(case, seed=100 + i)
        out = cs.ref_output(case, src)
        c = list(case)
        c[6] = np.dtype(c[6]).name
        c[7] = np.dtype(c[7]).name
        np.savez_compressed(os.path.join(HERE, "avir_%02d.npz" % i),
                            case=np.array(c, dtype=object), src=src, out=out)
    for i, (sw, sh, nw, nh, ti, to, kw) in enumerate(LANCIR_CASES):
        src = o.lcg_image(sh, sw, 4, ti, seed=200 + i)
        r, out = o.lancir_ref(src, nw, nh, to, **kw)
        assert r == nh
        np.savez_compressed(os.path.join(HERE, "lancir_%02d.npz" % i), src=src, out=out,
                            geom=np.array([sw, sh, nw, nh]))
    for i, (sw, sh, nw, nh, ch, ti, to, la) in enumerate(LANCIR_C_CASES):
        src = o.lcg_image(sh, sw, ch, ti, seed=300 + i)
        r, out = o.lancir_ref(src, nw, nh, to, la=la)
        assert r == nh
        np.savez_compressed(os.path.join(HERE, "lancir_%02d.npz" % (len(LANCIR_CASES) + i)),
                            src=src, out=out, geom=np.array([sw, sh, nw, nh]))
    print("wrote", len(GOLDEN_CASES), "AVIR and", len(LANCIR_CASES), "LANCIR fixtures;",
          o.ref().avir_ref_version().decode())


if __name__ == "__main__":
    main()
