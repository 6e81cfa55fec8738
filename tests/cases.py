"""Shared parity cases and helpers.

A case is (fpclass, src_w, src_h, new_w, new_h, channels, in_dtype, out_dtype, res_bits, kwargs)
with kwargs drawn from: gamma, alpha, buildmode, ox, oy, k, params.
"""
import ctypes as C
import os

import numpy as np

import avir_b200 as ab
import oracle_ref as o

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")

u8, u16, f32, f64 = np.uint8, np.uint16, np.float32, np.float64

# Scaled-down versions of the BASELINE.json configs first, then coverage of every chain
# shape, type combination, channel count and option (SURVEY.md section 8f rank 4).
SMALL_CASES = [
    # cfg2: 2X upsize u8 RGBA (k = 0.5); auto mode on small images picks filtered upsample
    (1, 240, 135, 480, 270, 4, u8, u8, 8, {}),
    (1, 240, 135, 480, 270, 4, u8, u8, 8, {"buildmode": 1}),   # the chain big images select
    # cfg3: 8K->4K float RGBA (k = 2), both mirrors named by the north star
    (2, 192, 108, 96, 54, 4, f32, f32, 16, {}),
    (2, 192, 108, 96, 54, 4, f32, f32, 16, {"buildmode": 1}),
    (1, 192, 108, 96, 54, 4, f32, f32, 16, {}),
    (1, 192, 108, 96, 54, 4, f32, f32, 16, {"buildmode": 1}),
    # cfg4: 4X downsize u16 RGBA (k = 4), decimating FIR
    (1, 256, 256, 64, 64, 4, u16, u16, 16, {}),
    (1, 256, 256, 64, 64, 4, u16, u16, 16, {"buildmode": 1}),
    # cfg5: planar/DIL mirror, 4X downsize u8 + sRGB gamma, alpha exempt
    (2, 384, 216, 96, 54, 4, u8, u8, 8, {"gamma": True, "alpha": 3}),
    (2, 384, 216, 96, 54, 4, u8, u8, 8, {"gamma": True, "alpha": 3, "buildmode": 1}),
    # cfg1 geometry through AVIR (k = 0.625), default class, RGB
    (0, 64, 48, 100, 75, 3, u8, u8, 8, {}),
    (1, 64, 48, 100, 75, 4, u8, u8, 8, {}),
    (2, 64, 48, 100, 75, 4, u8, u8, 8, {}),
    (2, 64, 48, 100, 75, 4, u8, u8, 8, {"buildmode": 1}),
    # 1 < k < 2, non-integer ratios, kx != ky
    (1, 100, 60, 67, 41, 2, u16, u16, 16, {}),
    (2, 150, 90, 100, 55, 4, f32, f32, 16, {"buildmode": 1}),
    (0, 150, 90, 100, 55, 3, u8, u8, 8, {"buildmode": 1}),
    (1, 100, 60, 150, 77, 4, u8, u8, 8, {}),
    (2, 100, 60, 150, 77, 4, u8, u8, 8, {}),
    # large ratios
    (2, 200, 120, 25, 15, 4, u16, u16, 16, {}),
    (0, 400, 240, 25, 15, 1, u8, u8, 8, {}),
    (1, 333, 211, 40, 27, 4, f32, f32, 16, {"buildmode": 0}),
    # mixed types / OutMul != 1 / gamma variants / float-out quirk of the default class
    (1, 300, 200, 200, 133, 4, u8, u16, 16, {}),
    (1, 120, 80, 60, 40, 4, u16, u8, 16, {}),
    (1, 120, 80, 60, 40, 4, f32, u8, 8, {}),
    (1, 120, 80, 60, 40, 4, u8, f32, 8, {}),
    (1, 192, 108, 48, 27, 4, u8, u8, 8, {"gamma": True, "alpha": 0}),
    (0, 192, 108, 48, 27, 3, u16, f32, 16, {"gamma": True}),
    (1, 192, 108, 48, 27, 3, f32, u16, 16, {"gamma": True}),
    (2, 192, 108, 48, 27, 2, u16, u16, 16, {"gamma": True}),
    # bit-depth truncation, identity size, offsets, explicit k, negative k, other presets
    (0, 100, 60, 130, 97, 4, u8, u8, 6, {}),
    (1, 57, 33, 57, 33, 4, u8, u8, 8, {}),
    (1, 90, 70, 45, 35, 4, u8, u8, 8, {"ox": 0.37, "oy": -0.21}),
    (1, 90, 70, 45, 35, 4, u8, u8, 8, {"k": 2.0}),
    (2, 90, 70, 60, 45, 4, f32, f32, 16, {"k": -1.5}),
    (1, 96, 64, 48, 32, 4, u8, u8, 8, {"params": 1}),
    (2, 96, 64, 48, 32, 4, u8, u8, 8, {"params": 5}),
    # double image buffers: (float) cast in, (double) cast out (avir.h:2803-2806, 3168-3171);
    # double output of the default class takes the ordinary output stage, gamma included
    (1, 192, 108, 96, 54, 4, f64, f64, 16, {}),
    (2, 192, 108, 96, 54, 4, f64, f32, 16, {"buildmode": 1}),
    (0, 120, 80, 60, 40, 3, u8, f64, 8, {"gamma": True}),
    (0, 120, 80, 60, 40, 3, f32, f64, 16, {"gamma": True}),
    (1, 100, 60, 150, 77, 4, f64, u16, 16, {"gamma": True, "alpha": 3}),
    (2, 150, 90, 100, 55, 2, f64, u8, 8, {}),
    # error-diffusion ditherer (upstream CImageResizerDithererErrdINL / ErrdDIL composed into the
    # three classes: fpclass codes 3..5), integer output only; row-recursive
    (3, 120, 80, 60, 40, 4, u8, u8, 8, {}),
    (4, 120, 80, 60, 40, 4, u8, u8, 8, {}),
    (5, 120, 80, 60, 40, 4, u8, u8, 8, {}),
    (3, 100, 60, 150, 77, 3, u8, u8, 6, {}),                 # bit-depth truncation: TrMul != 1
    (4, 100, 60, 150, 97, 1, u16, u16, 12, {}),              # 3 row groups, one channel
    (5, 192, 108, 48, 27, 4, u8, u8, 5, {"gamma": True, "alpha": 3}),
    (3, 64, 48, 33, 70, 2, f32, u16, 16, {"gamma": True}),
    (4, 40, 30, 1, 65, 4, u8, u8, 8, {}),                    # one-pixel rows
    (5, 40, 30, 77, 1, 4, u8, u8, 8, {}),                    # one row
    (3, 120, 80, 60, 40, 4, u8, f32, 8, {}),                 # float output: the ditherer is skipped
    # tiny / ragged
    (1, 1, 1, 5, 7, 4, u8, u8, 8, {}),
    (1, 7, 5, 1, 1, 4, u8, u8, 8, {}),
    (2, 3, 200, 9, 50, 4, u8, u8, 8, {}),
    (0, 2, 2, 3, 3, 1, f32, f32, 16, {}),
]


def make_input(case, seed=7, structured=None):
    fp, sw, sh, nw, nh, ch, ti, to, rb, kw = case
    if structured is None:
        return o.lcg_image(sh, sw, ch, ti, seed=seed)
    mx = {u8: 255, u16: 65535, f32: 1.0, f64: 1.0}[ti]
    img = np.zeros((sh, sw, ch), dtype=ti)
    if structured == "ramp":
        xs = (np.arange(sw) / max(sw - 1, 1))[None, :, None]
        ys = (np.arange(sh) / max(sh - 1, 1))[:, None, None]
        img[:] = ((xs * 0.6 + ys * 0.4) * mx).astype(ti)
    elif structured == "impulse":
        for (y, x) in ((0, 0), (0, sw - 1), (sh - 1, 0), (sh - 1, sw - 1), (sh // 2, sw // 2)):
            img[y, x] = mx
    elif structured == "checker":
        yy, xx = np.mgrid[0:sh, 0:sw]
        img[((yy + xx) & 1) == 1] = mx
    return img


def ref_kwargs(kw):
    return dict(k=kw.get("k", 0.0), ox=kw.get("ox", 0.0), oy=kw.get("oy", 0.0),
                gamma=kw.get("gamma", False), alpha=kw.get("alpha", -1),
                buildmode=kw.get("buildmode", -1), params=kw.get("params", 0))


def ref_output(case, src):
    fp, sw, sh, nw, nh, ch, ti, to, rb, kw = case
    return o.ref_resize(src, nw, nh, to, fpclass=fp, resbits=rb, **ref_kwargs(kw))


def resizer_and_vars(case):
    fp, sw, sh, nw, nh, ch, ti, to, rb, kw = case
    rs = ab.CImageResizer(rb, 0, kw.get("params", 0), fp)
    v = ab.CImageResizerVars(ox=kw.get("ox", 0.0), oy=kw.get("oy", 0.0),
                             UseSRGBGamma=kw.get("gamma", False), AlphaIndex=kw.get("alpha", -1),
                             BuildMode=kw.get("buildmode", -1))
    return rs, v


_port = None


def port():
    global _port
    if _port is None:
        lib = C.CDLL(os.path.join(ROOT, "oracle", "libavir_port.so"))
        for f in (lib.avir_port_resize, lib.lancir_port_resize):
            f.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t]
            f.restype = C.c_int
        lib.avir_port_srgb_lut.argtypes = [C.c_void_p]
        _port = lib
    return _port


def port_output(case, src):
    """The C port executing the descriptor the product front-end builds."""
    fp, sw, sh, nw, nh, ch, ti, to, rb, kw = case
    rs, v = resizer_and_vars(case)
    h, dp, modes = rs.descriptor(src.shape, src.dtype, nw, nh, to, kw.get("k", 0.0), v)
    try:
        dst = np.zeros((nh, nw, ch), to)
        assert port().avir_port_resize(dp, src.ctypes.data, sw * ch, dst.ctypes.data, nw * ch) == 0
    finally:
        rs.free_descriptor(h)
    return dst, modes


def gpu_output(case, src):
    """The product: avir::CImageResizer<>::resizeImage through libavirb200.so."""
    fp, sw, sh, nw, nh, ch, ti, to, rb, kw = case
    rs, v = resizer_and_vars(case)
    return rs.resizeImage(src, nw, nh, kw.get("k", 0.0), v, out_dtype=to)


def count_mismatch(a, b):
    assert a.shape == b.shape and a.dtype == b.dtype
    if a.dtype == np.float32:
        return int((a.view(np.uint32) != b.view(np.uint32)).sum())
    return int((a != b).sum())


# ---- upstream's outputs, stored as digests -------------------------------------------------------
# Every comparison with upstream goes through upstream(): it returns the digest of the output upstream
# (oracle/_ref) produced for a key naming the call and its input, read from tests/golden/upstream.json,
# so the suite needs neither the reference sources nor oracle/_ref.  With AVIRB200_RECORD_UPSTREAM=<file>
# set (and oracle/_ref built) it runs upstream instead and merges every key it computed into <file>;
# tests/golden/make_golden.py describes the regeneration.

UPSTREAM_JSON = os.path.join(GOLDEN, "upstream.json")
_upstream = None
_recorded = {}


def digest(a):
    """Digest of an array's shape, type and bits (+0.0 for -0.0 in double arrays: count_mismatch
    compares those by value)."""
    import hashlib
    a = np.ascontiguousarray(a)
    if a.dtype == np.float64:
        a = a + 0.0
    h = hashlib.sha256(("%s%s" % (a.dtype.str, a.shape)).encode())
    h.update(a.view(np.uint8).reshape(-1))
    return h.hexdigest()[:32]


def avir_key(case, src):
    return case_id(case) + "/" + digest(src)[:16]


def lancir_key(src, nw, nh, to, kw):
    sh, sw, ch = src.shape
    s = "lancir-%dx%d-%dx%d-c%d-%s-%s" % (sw, sh, nw, nh, ch, src.dtype.name, np.dtype(to).name)
    for k_, v_ in sorted(kw.items()):
        s += "-%s%s" % (k_, v_)
    return s + "/" + digest(src)[:16]


def _flush_recorded():
    import json
    path = os.environ["AVIRB200_RECORD_UPSTREAM"]
    have = json.load(open(path)) if os.path.exists(path) else {}
    have.update(_recorded)
    with open(path, "w") as f:
        json.dump(have, f, indent=0, sort_keys=True)
        f.write("\n")


def upstream(key, compute):
    """The stored value for `key`; `compute()` runs upstream for it (record mode only) and returns
    an array (stored as its digest) or a JSON value."""
    global _upstream
    if os.environ.get("AVIRB200_RECORD_UPSTREAM"):
        assert o.have_ref(), "recording upstream's outputs needs oracle/_ref"
        if not _recorded:
            import atexit
            atexit.register(_flush_recorded)
        v = compute()
        _recorded[key] = digest(v) if isinstance(v, np.ndarray) else v
        return _recorded[key]
    if _upstream is None:
        import json
        _upstream = json.load(open(UPSTREAM_JSON))
    assert key in _upstream, "no stored upstream output for %s (tests/golden/make_golden.py)" % key
    return _upstream[key]


def matches_upstream(case, src, got):
    """True when `got` has the bits upstream produced for this AVIR case and input."""
    return digest(got) == upstream(avir_key(case, src), lambda: ref_output(case, src))


def case_id(case):
    fp, sw, sh, nw, nh, ch, ti, to, rb, kw = case
    s = "%s-%dx%d-%dx%d-c%d-%s-%s-b%d" % (("def", "f4", "dil", "defE", "f4E", "dilE")[fp], sw, sh, nw, nh, ch,
                                          np.dtype(ti).name, np.dtype(to).name, rb)
    for k_, v_ in sorted(kw.items()):
        s += "-%s%s" % (k_, v_)
    return s
