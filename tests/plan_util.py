"""Host planner access (product: libavirb200_host.so) and comparison with oracle plans."""
import ctypes as C
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOST_SO = os.path.join(ROOT, "avir_b200", "libavirb200_host.so")

_host = None


def host():
    global _host
    if _host is None:
        lib = C.CDLL(HOST_SO)
        lib.avirb200_host_plan_dump.restype = C.c_long
        lib.avirb200_host_plan_dump.argtypes = [C.c_int] * 9 + [C.c_double] * 3 + [C.c_int] * 6 + [
            C.c_void_p, C.c_long]
        _host = lib
    return _host


def host_plan(mirror, sw, sh, nw, nh, ch, in_dtype, out_dtype, k=0.0, resbits=8, srcbits=0,
              ox=0.0, oy=0.0, gamma=False, buildmode=-1, params=0):
    in_dtype, out_dtype = np.dtype(in_dtype), np.dtype(out_dtype)
    args = (mirror, resbits, srcbits, params, sw, sh, nw, nh, ch, k, ox, oy,
            int(in_dtype.kind == "f"), int(out_dtype.kind == "f"), in_dtype.itemsize,
            out_dtype.itemsize, int(gamma), buildmode)
    n = host().avirb200_host_plan_dump(*args, None, 0)
    buf = np.zeros(n, dtype=np.float64)
    assert host().avirb200_host_plan_dump(*args, buf.ctypes.data, n) == n
    pos = [0]

    def take(m=1):
        v = buf[pos[0]:pos[0] + m]
        pos[0] += m
        return v

    plan = dict(zip(["out_mul", "in_gamma_mult", "out_gamma_mult", "el_count"], take(4)))
    for ax in ("H", "V"):
        mode, unsup, ns = [int(v) for v in take(3)]
        steps = []
        for _ in range(ns):
            s = dict(zip(["kind", "R", "lat", "edge", "in_len", "out_len", "ntaps", "order",
                          "upsampled", "skip_odd", "nphases", "out_prefix", "out_suffix",
                          "in_prefix", "in_suffix"], [int(v) for v in take(15)]))
            nt = int(take()[0])
            s["taps"] = take(nt).astype(np.float32)
            npos = int(take()[0])
            p = take(npos * 3).reshape(npos, 3)
            s["src_pos"] = p[:, 0].astype(np.int32)
            s["phase"] = p[:, 1].astype(np.int32)
            s["frac"] = p[:, 2].astype(np.float32)
            steps.append(s)
        plan[ax] = dict(mode=mode, unsupported=bool(unsup), steps=steps)
    assert pos[0] == n
    return plan


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def expected_axis(refsteps):
    """What the host plan of one axis must hold, from the step list recorded from the upstream run:
    one dict per host step, scalars as ints and arrays as float32 bits / int32."""
    out = []
    # fold upstream's filterless upsample step into the following resize step
    pend = None
    for r in refsteps:
        if r["kind"] == 1 and r["FltOrigLen"] > 0:
            pend = r  # filterless 2X upsample: folded into the next (resize) step
            continue
        if r["kind"] == 1:
            e = dict(kind=1, R=r["R"], lat=r["lat"], in_len=r["InLen"], out_len=r["OutLen"],
                     out_prefix=r["OutPrefix"], out_suffix=r["OutSuffix"], in_prefix=r["InPrefix"],
                     in_suffix=r["InSuffix"], taps=_bits(r["Flt"]))
        elif r["kind"] == 0:
            e = dict(kind=0, R=r["R"], lat=r["lat"], edge=r["edge"], in_len=r["InLen"], out_len=r["OutLen"],
                     taps=_bits(r["Flt"]))
        else:
            e = dict(kind=2, in_len=pend["InLen"] if pend is not None else r["InLen"],
                     upsampled=int(pend is not None), skip_odd=int(r["kind"] == 3), out_len=r["OutLen"],
                     ntaps=r["FL"], order=r["order"], src_pos=np.asarray(r["SrcPosInt"], np.int32),
                     frac=_bits(r["x"]),
                     bank_taps=np.stack([_bits(r["bank"][int(r["fti"][j])]) for j in range(r["OutLen"])]))
        pend = None
        out.append(e)
    return out


def _same(a, b):
    """b: an array, or the digest of one (as stored in tests/golden/upstream.json)."""
    import cases as cs
    return cs.digest(a) == b if isinstance(b, str) else np.array_equal(a, b)


def compare_axis(mine, expected):
    """Returns a list of mismatch descriptions between the host plan of one axis and
    expected_axis() of upstream's steps (or its stored form, arrays as digests)."""
    bad = []
    if len(expected) != len(mine["steps"]):
        return ["step count %d vs ref %d" % (len(mine["steps"]), len(expected))]
    for i, (m, e) in enumerate(zip(mine["steps"], expected)):
        tag = "step %d: " % i
        if m["kind"] != e["kind"]:
            bad.append(tag + "kind")
            continue
        for a, b in e.items():
            if a in ("taps", "frac", "src_pos", "bank_taps"):
                continue
            if m[a] != b:
                bad.append(tag + "%s %d vs %d" % (a, m[a], b))
        if e["kind"] != 2:
            if not _same(_bits(m["taps"]), e["taps"]):
                bad.append(tag + ("upsample" if e["kind"] == 1 else "FIR") + " taps differ")
            continue
        if not _same(np.asarray(m["src_pos"], np.int32), e["src_pos"]):
            bad.append(tag + "src_pos differ")
        if not _same(_bits(m["frac"]), e["frac"]):
            bad.append(tag + "frac differ")
        stride = m["ntaps"] * (m["order"] + 1)
        if m["out_len"] == e["out_len"] and len(m["taps"]) % stride == 0:
            tp = _bits(m["taps"]).reshape(-1, stride)
            if not _same(tp[np.asarray(m["phase"][:m["out_len"]])], e["bank_taps"]):
                bad.append(tag + "bank taps differ")
    return bad
