"""CPU tests of the oracles and the host logic (no GPU needed).

Pinning chain (SURVEY.md section 8c -- upstream has no tests, golden vectors or KATs of its own):
  upstream's plans and outputs (digests in tests/golden/upstream.json,
  recorded from upstream compiled in-tree)  --pin--->  host planner (product) and C port (oracle)
  committed fixtures (tests/golden)         --pin--->  C port
  SURVEY.md App. A hex-float coefficients   --pin--->  host planner
"""
import os

import numpy as np
import pytest

import cases as cs
import oracle_ref as o
import plan_util as pu

def hexf(strs):
    return np.array([float.fromhex(s) for s in strs.split()], dtype=np.float32)


def mirrored(half):
    return np.concatenate([half, half[-2::-1]])


# ---- planner vs SURVEY.md Appendix A golden coefficients ----------------------------------

def test_planner_appendix_a_k2_16bit_mode0():
    p = pu.host_plan(1, 7680, 64, 3840, 32, 4, np.float32, np.float32, resbits=16, buildmode=0)
    st = p["H"]["steps"]
    assert [s["kind"] for s in st] == [0, 2, 0]
    lpf = mirrored(hexf("-0x1.8bf0b8p-7 0x1.e493e4p-5 0x1.0db6f6p-2 0x1.842c26p-2"))
    assert np.array_equal(st[0]["taps"], lpf) and st[0]["lat"] == 3 and st[0]["edge"] == 3
    c0 = hexf("0x1.861df2p-11 -0x1.eeb3d2p-8 0x1.69c3c2p-7 0x1.63e384p-8 -0x1.546e5p-5 "
              "0x1.271796p-4 -0x1.bfdfcap-5 -0x1.12338cp-4 0x1.29b56ap-1")
    c1 = hexf("-0x1.ef6ep-18 0x1.efcap-15 -0x1.e036p-13 0x1.9a97ap-12 -0x1.049fp-12 -0x1.b186p-12 "
              "0x1.81e6cp-10 -0x1.259f4p-9 -0x1.ae46p-9 0x1.aadap-9 0x1.2981p-9 -0x1.81834p-10 "
              "0x1.a662p-12 0x1.0d83p-12 -0x1.9ddaep-12 0x1.df5cp-13 -0x1.e71p-15 0x1.d82fp-18")
    rs = st[1]
    assert rs["ntaps"] == 18 and rs["order"] == 1 and rs["nphases"] == 1
    assert np.array_equal(rs["taps"][:18], np.concatenate([c0, c0[::-1]]))
    assert np.array_equal(rs["taps"][18:], c1)
    assert np.array_equal(rs["src_pos"][:3], [3, 5, 7]) and np.all(rs["frac"] == 0)
    corr = mirrored(hexf("-0x1.5c0474p-11 0x1.2a05e8p-5 -0x1.ceeabap-3 0x1.617152p+0"))
    assert np.array_equal(st[2]["taps"], corr)


def test_planner_appendix_a_k2_16bit_mode1_and_k05():
    p = pu.host_plan(2, 7680, 64, 3840, 32, 4, np.float32, np.float32, resbits=16, buildmode=1)
    st = p["H"]["steps"]
    assert [s["kind"] for s in st] == [2, 0]
    c0 = hexf("-0x1.2daf84p-17 0x1.1b9668p-13 -0x1.92940cp-12 -0x1.25451ep-10 0x1.1763cp-10 "
              "0x1.671cc8p-12 -0x1.8c82a8p-10 0x1.859872p-9 -0x1.217804p-7 0x1.66144p-8 "
              "0x1.3a0c5cp-3 0x1.64e63ap-2")
    assert st[0]["ntaps"] == 24 and np.array_equal(st[0]["taps"][:24], np.concatenate([c0, c0[::-1]]))
    assert np.array_equal(st[0]["src_pos"][:3], [0, 2, 4])
    corr = hexf("-0x1.5c0478p-11 0x1.2a05eap-5 -0x1.ceeabcp-3 0x1.617152p+0")
    assert st[1]["ntaps"] == 8 and np.array_equal(st[1]["taps"][:4], corr) and st[1]["taps"][7] == 0
    # k = 0.5, 8-bit, mode 1: pre-correction, filterless 2X folded into a skip-odd resize
    q = pu.host_plan(1, 1920, 64, 3840, 128, 4, np.uint8, np.uint8, buildmode=1)["H"]["steps"]
    assert [s["kind"] for s in q] == [0, 2]
    assert q[1]["upsampled"] == 1 and q[1]["skip_odd"] == 1 and q[1]["ntaps"] == 24
    assert np.array_equal(q[1]["taps"][:12], (c0 * np.float32(2)).astype(np.float32))
    assert np.array_equal(q[1]["src_pos"][:2], [5, 6])


def test_planner_appendix_a_k4_and_auto_modes():
    p = pu.host_plan(1, 16384, 64, 4096, 16, 4, np.uint16, np.uint16, resbits=16)
    assert p["H"]["mode"] == 0
    st = p["H"]["steps"]
    lpf = mirrored(hexf("-0x1.7c80a2p-10 -0x1.8b5164p-8 0x1.867202p-11 0x1.e3d0e6p-6 0x1.3e2c2p-4 "
                        "0x1.0d4a6ep-3 0x1.632a86p-3 0x1.838ff2p-3"))
    assert st[0]["R"] == 2 and np.array_equal(st[0]["taps"], lpf)
    assert np.all(st[1]["frac"] == 0.5) and np.array_equal(st[1]["src_pos"][:3], [3, 5, 7])
    # auto-selected build modes at the BASELINE configs (SURVEY.md section 3.2)
    assert pu.host_plan(1, 7680, 4320, 3840, 2160, 4, np.float32, np.float32, resbits=16)["H"]["mode"] == 0
    assert pu.host_plan(2, 7680, 4320, 3840, 2160, 4, np.float32, np.float32, resbits=16)["H"]["mode"] == 1
    assert pu.host_plan(1, 1920, 1080, 3840, 2160, 4, np.uint8, np.uint8)["V"]["mode"] == 1
    assert pu.host_plan(2, 7680, 4320, 1920, 1080, 4, np.uint8, np.uint8, gamma=True)["H"]["mode"] == 1


# ---- planner / port vs upstream compiled in-tree -------------------------------------------

def _upstream_plan(case, src):
    """expected_axis() of both axes of the plan upstream built, arrays as digests."""
    fp, sw, sh, nw, nh, ch, ti, to, rb, kw = case

    def run():
        rp, _ = o.ref_plan(src, nw, nh, to, fpclass=fp, resbits=rb, **cs.ref_kwargs(kw))
        return {ax: [{a: (cs.digest(v) if isinstance(v, np.ndarray) else v) for a, v in e.items()}
                     for e in pu.expected_axis(rp[ax])] for ax in ("H", "V")}
    return cs.upstream("plan:" + cs.avir_key(case, src), run)


@pytest.mark.parametrize("case", cs.SMALL_CASES, ids=cs.case_id)
def test_planner_matches_upstream(case):
    fp, sw, sh, nw, nh, ch, ti, to, rb, kw = case
    fp %= 3  # the error-diffusion variants (3..5) plan exactly like their base classes
    case = (fp,) + case[1:]
    src = cs.make_input(case)
    rk = cs.ref_kwargs(kw)
    rp = _upstream_plan(case, src)
    mp = pu.host_plan(fp, sw, sh, nw, nh, ch, ti, to, k=rk["k"], resbits=rb, ox=rk["ox"], oy=rk["oy"],
                      gamma=rk["gamma"], buildmode=rk["buildmode"], params=rk["params"])
    assert pu.compare_axis(mp["H"], rp["H"]) == []
    assert pu.compare_axis(mp["V"], rp["V"]) == []


@pytest.mark.parametrize("case", cs.SMALL_CASES, ids=cs.case_id)
def test_port_matches_upstream(case):
    src = cs.make_input(case)
    mine, _ = cs.port_output(case, src)
    assert cs.matches_upstream(case, src, mine)


@pytest.mark.parametrize("structured", ["ramp", "impulse", "checker"])
@pytest.mark.parametrize("case", cs.SMALL_CASES[:10], ids=cs.case_id)
def test_port_structured_inputs(case, structured):
    src = cs.make_input(case, structured=structured)
    mine, _ = cs.port_output(case, src)
    assert cs.matches_upstream(case, src, mine)


def test_port_matches_golden_fixtures():
    files = sorted(f for f in os.listdir(cs.GOLDEN) if f.startswith("avir_") and f.endswith(".npz"))
    assert len(files) >= 8
    for f in files:
        z = np.load(os.path.join(cs.GOLDEN, f), allow_pickle=True)
        case = tuple(z["case"].tolist())
        case = case[:6] + (np.dtype(case[6]).type, np.dtype(case[7]).type) + case[8:]
        mine, _ = cs.port_output(case, z["src"])
        assert cs.count_mismatch(z["out"], mine) == 0, f


def test_lancir_port_matches_golden_fixtures():
    """Pins the LANCIR restatement (all four channel-count trees) where oracle/_ref is absent."""
    import avir_b200 as ab
    h = ab.host_lib()
    T = {np.dtype(np.uint8): 0, np.dtype(np.uint16): 1, np.dtype(np.float32): 2}
    files = sorted(f for f in os.listdir(cs.GOLDEN) if f.startswith("lancir_"))
    assert len(files) >= 11 and {np.load(os.path.join(cs.GOLDEN, f))["src"].shape[2]
                                 for f in files} == {1, 2, 3, 4}
    for f in files:
        z = np.load(os.path.join(cs.GOLDEN, f))
        src, want = np.ascontiguousarray(z["src"]), z["out"]
        sw, sh, nw, nh = [int(v) for v in z["geom"]]
        ch = src.shape[2]
        hd = h.lancirb200_host_desc_create(T[src.dtype], T[want.dtype], sw, sh, nw, nh, ch, 0.0, 0.0,
                                           0.0, 0.0, 3.0)
        assert hd
        dst = np.zeros_like(want)
        assert cs.port().lancir_port_resize(h.lancirb200_host_desc_get(hd), src.ctypes.data, sw * ch,
                                            dst.ctypes.data, nw * ch) == 0
        h.lancirb200_host_desc_free(hd)
        assert cs.count_mismatch(want, dst) == 0, f


def test_srgb_u8_table_matches_upstream():
    # feed every byte value through upstream's linearisation: 1x1 float output, no resize
    lut = np.zeros(256, np.float32)
    cs.port().avir_port_srgb_lut(lut.ctypes.data)
    # an identity-size resize is not an identity filter; probe the table through a constant
    # image instead: constant in -> constant out == de-linearised(linearised(v)) is not the
    # table either, so compare on the port/upstream pair with gamma and float output (def
    # class skips output gamma: avir.h:4956-4979), constant images reproduce the table value
    # up to the filters' DC gain; exact equality is asserted for the full pipeline instead.
    for v in (0, 1, 10, 11, 57, 128, 200, 254, 255):
        src = np.full((8, 8, 3), v, np.uint8)
        case = (0, 8, 8, 8, 8, 3, np.uint8, np.float32, 8, {"gamma": True})
        mine, _ = cs.port_output(case, src)
        assert cs.matches_upstream(case, src, mine)
    assert lut[0] == 0.0 and abs(lut[255] - 0.9999975) < 1e-7 and np.all(np.diff(lut) > 0)


def _lancir_upstream(src, nw, nh, to, kw):
    def run():
        r, ref = o.lancir_ref(src, nw, nh, to, **kw)
        assert r == nh
        return ref
    return cs.upstream(cs.lancir_key(src, nw, nh, to, kw), run)


def test_lancir_port_matches_upstream():
    import ctypes as C
    import avir_b200 as ab
    h = ab.host_lib()
    for (sw, sh, nw, nh, ti, to, kw) in [
            (96, 54, 48, 27, np.uint8, np.uint8, {}),
            (64, 48, 103, 77, np.uint8, np.uint8, {}),
            (64, 64, 16, 16, np.uint16, np.uint16, {}),
            (60, 40, 40, 27, np.uint8, np.uint16, {}),
            (50, 30, 33, 17, np.float32, np.float32, {}),
            (50, 30, 33, 17, np.float32, np.uint8, {}),
            (50, 30, 70, 45, np.uint8, np.float32, {"kx": 0.7, "ky": -0.66, "ox": 0.25, "oy": 0.1}),
            (50, 30, 25, 15, np.uint8, np.uint8, {"la": 2.0}),
            (50, 30, 25, 15, np.uint8, np.uint8, {"la": 4.5}),
            # 1-3 channels: upstream's resize1/2/3 trees, kernel lengths 6 (kl%4==2), 8, 12, 10
            (64, 48, 103, 77, np.uint8, np.uint8, {"C": 3}),
            (64, 48, 103, 77, np.uint8, np.uint8, {"C": 2}),
            (64, 48, 103, 77, np.uint8, np.uint8, {"C": 1}),
            (64, 48, 103, 77, np.float32, np.float32, {"C": 3, "la": 4.0}),
            (96, 54, 48, 27, np.uint16, np.uint16, {"C": 3}),
            (96, 54, 48, 27, np.float32, np.float32, {"C": 2}),
            (96, 54, 48, 27, np.uint8, np.float32, {"C": 1}),
            (77, 51, 50, 31, np.float32, np.float32, {"C": 3, "la": 2.0}),
            (77, 51, 50, 31, np.float32, np.float32, {"C": 1, "la": 2.0}),
            (77, 51, 47, 30, np.uint8, np.uint8, {"C": 2, "la": 3.0}),
            (77, 51, 47, 29, np.float32, np.float32, {"C": 3, "la": 3.0}),
            (77, 51, 47, 29, np.float32, np.float32, {"C": 1, "la": 3.0, "kx": 1.3, "ky": 2.2}),
            (77, 51, 47, 29, np.float32, np.float32, {"C": 2, "la": 3.0, "kx": 1.3, "ky": 2.2}),
            (77, 51, 47, 29, np.float32, np.float32, {"C": 3, "la": 3.0, "kx": 1.3, "ky": 2.2}),
            (33, 21, 7, 5, np.uint8, np.uint8, {"C": 3}),
    ]:
        kw = dict(kw)
        ch = kw.pop("C", 4)
        src = o.lcg_image(sh, sw, ch, ti, seed=3)
        T = {np.uint8: 0, np.uint16: 1, np.float32: 2}
        hd = h.lancirb200_host_desc_create(T[ti], T[to], sw, sh, nw, nh, ch, kw.get("kx", 0.0),
                                           kw.get("ky", 0.0), kw.get("ox", 0.0), kw.get("oy", 0.0),
                                           kw.get("la", 3.0))
        assert hd
        dst = np.zeros((nh, nw, ch), to)
        assert cs.port().lancir_port_resize(h.lancirb200_host_desc_get(hd), src.ctypes.data, sw * ch,
                                            dst.ctypes.data, nw * ch) == 0
        h.lancirb200_host_desc_free(hd)
        assert cs.digest(dst) == _lancir_upstream(src, nw, nh, to, kw), (sw, sh, nw, nh, ch, ti, to, kw)


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_port_fuzz_matches_upstream(seed):
    """Seeded random sweep over the whole call surface -- all six classes (the three mirrors and
    their error-diffusion variants), 1..4 channels, every Tin/Tout pair incl. double, bit depths,
    gamma / alpha, offsets, explicit and negative k, parameter presets, forced build modes,
    upsizing / downsizing / odd ratios -- host planner + C port against upstream compiled
    in-tree: 0 mismatching elements."""
    rng = np.random.default_rng(seed)
    types = [np.uint8, np.uint16, np.float32, np.float64]
    for it in range(60):
        fp, ch = int(rng.integers(0, 6)), int(rng.integers(1, 5))
        sw, sh = int(rng.integers(1, 160)), int(rng.integers(1, 160))
        mode = int(rng.integers(0, 4))
        if mode == 0:
            nw, nh = max(1, sw // int(rng.integers(1, 9))), max(1, sh // int(rng.integers(1, 9)))
        elif mode == 1:
            nw, nh = sw * int(rng.integers(1, 4)), sh * int(rng.integers(1, 4))
        else:
            nw, nh = int(rng.integers(1, 240)), int(rng.integers(1, 240))
        ti, to = types[int(rng.integers(0, 4))], types[int(rng.integers(0, 4))]
        rb = int(rng.integers(4, 9)) if to == np.uint8 else (
            int(rng.integers(8, 17)) if to == np.uint16 else int(rng.choice([8, 16])))
        kw = {}
        if rng.random() < 0.3:
            kw["gamma"] = True
        if ch == 4 and rng.random() < 0.5:
            kw["alpha"] = int(rng.choice([0, 3]))
        if rng.random() < 0.2:
            kw["ox"], kw["oy"] = float(rng.uniform(-1, 1)), float(rng.uniform(-1, 1))
        if rng.random() < 0.2:
            kw["k"] = float(rng.choice([-2.5, -1.0, 0.7, 1.5, 3.0]))
        if rng.random() < 0.2:
            kw["params"] = int(rng.integers(0, 6))
        if rng.random() < 0.3:
            kw["buildmode"] = int(rng.integers(0, 4))
        case = (fp, sw, sh, nw, nh, ch, ti, to, rb, kw)
        src = cs.make_input(case, seed=1000 * seed + it)
        mine, _ = cs.port_output(case, src)
        assert cs.matches_upstream(case, src, mine), cs.case_id(case)


def test_lancir_port_fuzz_matches_upstream():
    """Seeded random sweep of CLancIR: 1..4 channels (four summation trees), kernel lengths from
    la = 2 .. 5 and both scaling directions (kl % 4 == 0 and == 2), offsets, explicit steps,
    every u8 / u16 / float type pair."""
    import avir_b200 as ab
    h = ab.host_lib()
    rng = np.random.default_rng(7)
    types = [np.uint8, np.uint16, np.float32]
    tcode = {np.uint8: 0, np.uint16: 1, np.float32: 2}
    for it in range(80):
        ch = int(rng.integers(1, 5))
        sw, sh = int(rng.integers(2, 120)), int(rng.integers(2, 120))
        nw, nh = int(rng.integers(1, 200)), int(rng.integers(1, 200))
        ti, to = types[int(rng.integers(0, 3))], types[int(rng.integers(0, 3))]
        kw = {"la": float(rng.choice([2.0, 2.5, 3.0, 4.0, 5.0]))}
        if rng.random() < 0.3:
            kw["kx"], kw["ky"] = float(rng.choice([0.5, 0.8, 1.7, -1.3])), float(rng.choice([0.6, 1.0, 2.2, -0.9]))
        if rng.random() < 0.3:
            kw["ox"], kw["oy"] = float(rng.uniform(-1, 1)), float(rng.uniform(-1, 1))
        src = o.lcg_image(sh, sw, ch, ti, seed=500 + it)
        hd = h.lancirb200_host_desc_create(tcode[ti], tcode[to], sw, sh, nw, nh, ch, kw.get("kx", 0.0),
                                           kw.get("ky", 0.0), kw.get("ox", 0.0), kw.get("oy", 0.0), kw["la"])
        assert hd
        dst = np.zeros((nh, nw, ch), to)
        assert cs.port().lancir_port_resize(h.lancirb200_host_desc_get(hd), src.ctypes.data, sw * ch,
                                            dst.ctypes.data, nw * ch) == 0
        h.lancirb200_host_desc_free(hd)
        assert cs.digest(dst) == _lancir_upstream(src, nw, nh, to, kw), (sw, sh, nw, nh, ch, ti, to, kw)
