#!/usr/bin/env python
"""bench.py -- headline benchmark: Mpixels/s of the AVIR separable resize hot path, 8K->4K RGBA.

  python bench.py --gpus N --steps K --warmup W            (own arm; torchrun for N > 1)
  python bench.py --impl reference --gpus N --steps K ...  (upstream's CPU path, rank 0 only)
  python bench.py ... --dump-outputs DIR                   (also save what the last timed step computed)

Workload (BASELINE.json configs[2]): CImageResizer<fpclass_float8_avx-equiv> 7680x4320 ->
3840x2160, 4-channel float.  A "step" resizes one such frame per GPU.  For N > 1 the N frames
form one 7680 x (4320*N) image that is ROW-SHARDED over the ranks: every rank runs the row
pass on its band, exchanges the filter-length halo rows with its neighbours over NCCL
(NVLink) and runs the column pass on its band -- per-GPU work is fixed (weak scaling) and the
real exchange step of the path is inside the timed region.

Besides the headline the line carries (DESIGN.md section 5 explains every field):
  parity_vs_reference  N = 1: mismatching elements between the benchmarked frame's output and
                       upstream's own output for the same input (cpu_baseline leg)
  sharded_parity       N > 1: the NCCL-sharded output against the 1-GPU output of the same tall
                       image, band by band (outside the timed region)
  configs              the other BASELINE configs (and upstream's own published case, 8-bit RGB
                       5184x3456 -> 1920x1280), device-resident: ms, per-pass split, GB/s, frac
  lancir               CLancIR 8K -> 4K RGBA u8: device-resident ms + roofline, e2e, CPU figure
  e2e_variants         pageable (malloc) host buffers next to pinned ones, u8 wire format
  batch                N frames through avirb200_resize_device_batch
  N > 1: strong scaling (ONE 8K frame over N GPUs), cfg4 row-sharded, cfg5 replicas

One JSON line is printed by rank 0.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True  # the benchmark leaves the tree as it found it
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

SRC_W, SRC_H, DST_W, DST_H, CH = 7680, 4320, 3840, 2160, 4
METRIC = "Mpixels/sec resize (8K->4K RGBA)"
MIRRORS = {"dil": 2, "f4": 1, "def": 0}
u8, u16, f32 = np.uint8, np.uint16, np.float32

# (name, fpclass, sw, sh, nw, nh, channels, tin, tout, res_bits, kwargs)
EXTRA_CONFIGS = [
    ("cfg2 1920x1080->3840x2160 RGBA u8 (float4 mirror)", 1, 1920, 1080, 3840, 2160, 4, u8, u8, 8, {}),
    ("cfg3 7680x4320->3840x2160 RGBA f32 (float4 mirror)", 1, 7680, 4320, 3840, 2160, 4, f32, f32, 16, {}),
    ("cfg4 16384x16384->4096x4096 RGBA u16 (float4 mirror, one GPU)", 1, 16384, 16384, 4096, 4096, 4, u16, u16, 16, {}),
    ("cfg5 7680x4320->1920x1080 RGBA u8 + sRGB gamma (float8_dil mirror)", 2, 7680, 4320, 1920, 1080, 4, u8, u8, 8,
     {"gamma": True, "alpha": 3}),
    ("8K->4K RGBA u8 (float4 mirror)", 1, 7680, 4320, 3840, 2160, 4, u8, u8, 8, {}),
    ("upstream README case: 5184x3456->1920x1280 RGB u8 (default class)", 0, 5184, 3456, 1920, 1280, 3, u8, u8, 8, {}),
]


def algorithmic_bytes(sw=SRC_W, sh=SRC_H, nw=DST_W, nh=DST_H, ch=CH, tin=f32, tout=f32, n_frames=1):
    """SURVEY.md 8(d): src read + intermediate write + intermediate read + dst write."""
    src = sw * sh * ch * np.dtype(tin).itemsize
    mid = nw * sh * ch * 4
    dst = nw * nh * ch * np.dtype(tout).itemsize
    return dict(row=(src + mid) * n_frames, col=(mid + dst) * n_frames,
                total=(src + 2 * mid + dst) * n_frames)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            j = json.load(open(p))
            return float(j["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100",
                 "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for (t, r) in self.rows if t0 - 0.05 <= t <= t1 + 0.15 and len(r) >= 9] or \
               [r for (_, r) in self.rows if len(r) >= 9]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm = sorted(float(r[1]) for r in rows)
        reasons = set()
        for r in rows:
            for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6),
                              ("sw_thermal_slowdown", 7), ("sw_power_cap", 8)):
                if r[col].lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(rows[0][2]), "samples": len(rows),
                "power_w_max": max(float(r[3]) for r in rows), "reasons": sorted(reasons)}


def traffic_from_profiles():
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p))
        except Exception:
            pass
    return {}


def synthetic_image(h, w, c, dtype, seed=12345):
    """SURVEY.md 8(d) generator: xorshift32, one draw per element in memory order, element =
    (T)((draw & 0xFFFF) * scale).  The sequential recurrence runs in C (libavirb200_host.so)."""
    import avir_b200 as ab
    hl = ab.host_lib()
    out = np.empty((h, w, c), dtype=dtype)
    code = {np.dtype(u8): 0, np.dtype(u16): 1, np.dtype(f32): 2}[np.dtype(dtype)]
    hl.avirb200_host_fill_xorshift32.argtypes = [C.c_void_p, C.c_size_t, C.c_uint32, C.c_int]
    hl.avirb200_host_fill_xorshift32.restype = C.c_uint32
    hl.avirb200_host_fill_xorshift32(out.ctypes.data, out.size, seed, code)
    return out


# ------------------------------------------------------------------------------------------------

def pick_threads(o, src, fp, cores):
    """Upstream's thread pool does not scale to every host core (each call allocates and
    first-touches its ~400 MB of scratch from all threads at once); use the thread count
    that is actually fastest on this host."""
    best, best_t = cores, None
    cand = sorted({c for c in (cores, cores // 2, cores // 4, 32, 16, 8, 4) if 1 <= c <= cores}, reverse=True)
    o.ref_resize(src, DST_W, DST_H, np.float32, fpclass=fp, resbits=16, nthreads=cand[0])
    for c in cand:
        t0 = time.perf_counter()
        o.ref_resize(src, DST_W, DST_H, np.float32, fpclass=fp, resbits=16, nthreads=c)
        dt = time.perf_counter() - t0
        if best_t is None or dt < best_t:
            best, best_t = c, dt
    return best


def run_reference(args):
    """Upstream's own CPU implementation (oracle/_ref: the unmodified headers compiled with the
    pinned flags) on all host threads, one full frame per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import oracle_ref as o
    if not o.have_ref():
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/libavir_ref.so missing"}))
        return
    fp = MIRRORS[args.mirror]
    src = synthetic_image(SRC_H, SRC_W, CH, np.float32)
    cores = pick_threads(o, src, fp, os.cpu_count() or 1)
    times = []
    for i in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        o.ref_resize(src, DST_W, DST_H, np.float32, fpclass=fp, resbits=16, nthreads=cores)
        dt = time.perf_counter() - t0
        if i >= args.warmup:
            times.append(dt)
    total = sum(times)
    ms = total / len(times) * 1e3
    val = SRC_W * SRC_H * len(times) / total / 1e6
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": "Mpix/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, 1),
        "cpu_baseline": {"value": val, "unit": "Mpix/s", "cores": cores, "kind": "reference",
                         "sample": "full 7680x4320 frame per step, %d steps, std::thread pool of %d "
                                   "workloads (fastest of a sweep up to %d host threads), pinned "
                                   "flags -O2 -mavx2 -ffp-contract=off"
                                   % (len(times), cores, os.cpu_count() or 1)},
        "e2e": {"value": val, "unit": "Mpix/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    fast = reference_fast_build(src, fp, cores, max(1, min(3, len(times))))
    if fast is not None:
        line["cpu_baseline_fast_build"] = fast
    print(json.dumps(line))


def reference_fast_build(src, fp, cores, n):
    """SURVEY 8(d): the same upstream headers built -O3 -mavx2 -mfma (oracle/_ref/libavir_ref_fast.so).
    FMA contraction changes upstream's bits, so this build is never a parity oracle: a labelled
    timing beside the pinned one, nothing else.  None when the build is not there or does not load."""
    path = os.path.join(ROOT, "oracle", "_ref", "libavir_ref_fast.so")
    try:
        lib = C.CDLL(path)
        lib.avir_ref_resize.restype = C.c_int
        lib.avir_ref_resize.argtypes = [
            C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p,
            C.c_int, C.c_int, C.c_int, C.c_double, C.c_int, C.c_int, C.c_double, C.c_double,
            C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]
        dst = np.zeros((DST_H, DST_W, CH), np.float32)

        def call():
            return lib.avir_ref_resize(fp, 2, 2, src.ctypes.data, SRC_W, SRC_H, 0, dst.ctypes.data, DST_W, DST_H, CH,
                                       0.0, 16, 0, 0.0, 0.0, 0, -1, -1, cores, 0)
        if call() != 0:
            return None
        ts = []
        for _ in range(n):
            t0 = time.perf_counter()
            call()
            ts.append(time.perf_counter() - t0)
        return {"value": SRC_W * SRC_H * len(ts) / sum(ts) / 1e6, "unit": "Mpix/s", "cores": cores, "kind": "reference",
                "flags": "-O3 -mavx2 -mfma (FMA contraction: bits may differ from the pinned oracle)",
                "sample": "%d full frames" % len(ts)}
    except Exception:
        return None


def workload_config(args, n):
    return {"workload": "cfg3: CImageResizer<%s>(16) 7680x%d->3840x%d RGBA float32, k=2"
                        % ({"dil": "fpclass_float8_dil", "f4": "fpclass_float4",
                            "def": "fpclass_def<float>"}[args.mirror], SRC_H * n, DST_H * n),
            "mirror": args.mirror, "frames_per_step": n,
            "parallelism": "single GPU" if n == 1 else "row-sharded x%d, halo rows exchanged through peer "
                                                       "mailboxes over NVLink (AVIRB200_OPT_OVERLAP_HALO = %s)"
                                                       % (n, "library default" if args.halo_mode is None else args.halo_mode),
            "input": "SURVEY 8(d) xorshift32, seed 12345 (+rank)",
            "l2": "inputs larger than L2 (531 MB source + 265 MB intermediate per GPU per step)"}


class SI(C.Structure):
    _fields_ = [(n_, C.c_int32) for n_ in ("src_row0", "src_rows", "dst_row0", "dst_rows",
                                           "need_row0", "need_rows", "halo_up", "halo_down")]


def declare(lib):
    lib.avirb200_resize_sharded.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p,
                                            C.c_size_t, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]
    lib.avirb200_resize_sharded_host.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p,
                                                 C.c_size_t, C.c_void_p, C.c_size_t]
    lib.avirb200_resize_device.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t,
                                           C.c_void_p, C.c_void_p]
    lib.avirb200_resize_device_batch.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p,
                                                 C.c_size_t, C.c_void_p, C.c_void_p]
    lib.avirb200_row_pass_device.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]
    lib.avirb200_col_pass_device.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]
    lib.avirb200_plan_set_option.argtypes = [C.c_void_p, C.c_int, C.c_int]
    lib.lancirb200_resize_device.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p, C.c_size_t,
                                             C.c_void_p, C.c_void_p]


class Plan:
    """A C-ABI plan for one call shape (the descriptor comes from the C++ front-end)."""
    halo_mode = None  # --halo-mode: AVIRB200_OPT_OVERLAP_HALO of every plan (None: the library's default)

    def __init__(self, ab, fp, shape, tin, nw, nh, tout, rb, kw=None):
        kw = kw or {}
        self.lib = ab.lib()
        self.rs = ab.CImageResizer(rb, 0, 0, fp)
        v = ab.CImageResizerVars(UseSRGBGamma=kw.get("gamma", False), AlphaIndex=kw.get("alpha", -1))
        self.h, dp, self.modes = self.rs.descriptor(shape, tin, nw, nh, tout, 0.0, v)
        self.plan = C.c_void_p()
        if self.lib.avirb200_plan_create(C.c_void_p(dp), C.byref(self.plan)) != 0:
            raise SystemExit("plan_create: " + self.lib.avirb200_last_error().decode())
        self.vars = v
        if Plan.halo_mode is not None:
            self.lib.avirb200_plan_set_option.argtypes = [C.c_void_p, C.c_int, C.c_int]
            assert self.lib.avirb200_plan_set_option(self.plan, 5, Plan.halo_mode) == 0  # AVIRB200_OPT_OVERLAP_HALO

    def workspace(self):
        b = C.c_size_t()
        assert self.lib.avirb200_plan_workspace_bytes(self.plan, C.byref(b)) == 0
        return b.value

    def shard(self, rank, n):
        si = SI()
        if self.lib.avirb200_shard_query(self.plan, rank, n, C.byref(si)) != 0:
            raise SystemExit("shard_query: " + self.lib.avirb200_last_error().decode())
        b = C.c_size_t()
        assert self.lib.avirb200_shard_workspace_bytes(self.plan, rank, n, C.byref(b)) == 0
        return si, b.value

    def close(self):
        self.lib.avirb200_plan_destroy(self.plan)
        self.rs.free_descriptor(self.h)


def torch_dtype(t):
    import torch
    return {np.dtype(u8): torch.uint8, np.dtype(u16): torch.uint16, np.dtype(f32): torch.float32}[np.dtype(t)]


def device_random(shape, dtype, seed):
    """Device-side uniform full-range filler for the secondary configs (their timing does not
    depend on the values; the parity tests cover their bits)."""
    import torch
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    if np.dtype(dtype) == np.dtype(f32):
        return torch.rand(shape, generator=g, device="cuda", dtype=torch.float32)
    hi = 256 if np.dtype(dtype) == np.dtype(u8) else 65536
    return torch.randint(0, hi, shape, generator=g, device="cuda", dtype=torch.int32).to(torch_dtype(dtype))


def median_ms(fn, n, warmup=3, flush=None):
    import torch
    for _ in range(warmup):
        fn()
    ts = []
    for _ in range(n):
        if flush is not None:
            flush.fill_(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return sorted(ts)[len(ts) // 2]


def run_extra_configs(ab, peak, budget_s):
    """The other BASELINE configs, device-resident on this GPU: whole call and per-pass medians."""
    import torch
    lib = ab.lib()
    out = []
    t_begin = time.time()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    for name, fp, sw, sh, nw, nh, ch, ti, to, rb, kw in EXTRA_CONFIGS:
        if time.time() - t_begin > budget_s:
            out.append({"config": name, "skipped": "time budget"})
            continue
        try:
            pl = Plan(ab, fp, (sh, sw, ch), ti, nw, nh, to, rb, kw)
            d_src = device_random((sh, sw, ch), ti, 7)
            d_dst = torch.empty((nh, nw, ch), device="cuda", dtype=torch_dtype(to))
            d_ws = torch.empty(pl.workspace(), dtype=torch.uint8, device="cuda")
            small = d_src.numel() * d_src.element_size() < (200 << 20)
            fl = flush if small else None

            def full():
                assert lib.avirb200_resize_device(pl.plan, d_src.data_ptr(), sw * ch, d_dst.data_ptr(), nw * ch,
                                                  d_ws.data_ptr(), st) == 0

            def row():
                assert lib.avirb200_row_pass_device(pl.plan, d_src.data_ptr(), sw * ch, d_ws.data_ptr(), st) == 0

            def col():
                assert lib.avirb200_col_pass_device(pl.plan, d_ws.data_ptr(), d_dst.data_ptr(), nw * ch, st) == 0
            ms = median_ms(full, 10, 3, fl)
            rms = median_ms(row, 10, 2, fl)
            cms = median_ms(col, 10, 2, fl)
            b = algorithmic_bytes(sw, sh, nw, nh, ch, ti, to)
            out.append({"config": name, "ms_per_frame": ms, "src_Mpix_per_s": sw * sh / ms / 1e3,
                        "row_ms": rms, "col_ms": cms, "algorithmic_MB": b["total"] / 1e6,
                        "GBps": b["total"] / ms / 1e6, "frac": b["total"] / ms / 1e6 / peak,
                        "row_frac": b["row"] / rms / 1e6 / peak, "col_frac": b["col"] / cms / 1e6 / peak,
                        "kernel_paths": lib.avirb200_plan_kernel_paths(pl.plan), "build_modes": list(pl.modes),
                        "l2": "flushed between iterations" if small else "inputs larger than L2"})
            pl.close()
            del d_src, d_dst, d_ws
            torch.cuda.empty_cache()
        except Exception as e:  # a secondary number must never cost the headline
            out.append({"config": name, "error": repr(e)[:200]})
    return out


def run_lancir(ab, peak, want_cpu):
    """CLancIR 8K -> 4K RGBA u8 (upstream lancir.h): device-resident, e2e, upstream on the host."""
    import torch
    lib, hl = ab.lib(), ab.host_lib()
    sw, sh, nw, nh, ch = SRC_W, SRC_H, DST_W, DST_H, 4
    res = {"workload": "CLancIR 7680x4320->3840x2160 RGBA u8, la=3"}
    try:
        h = hl.lancirb200_host_desc_create(0, 0, sw, sh, nw, nh, ch, 0.0, 0.0, 0.0, 0.0, 3.0)
        dp = hl.lancirb200_host_desc_get(h)
        plan = C.c_void_p()
        assert lib.lancirb200_plan_create(C.c_void_p(dp), C.byref(plan)) == 0, lib.avirb200_last_error()
        wsb = C.c_size_t()
        assert lib.lancirb200_plan_workspace_bytes(plan, C.byref(wsb)) == 0
        src = synthetic_image(sh, sw, ch, u8, seed=1)
        d_src = torch.from_numpy(src).cuda()
        d_dst = torch.empty((nh, nw, ch), device="cuda", dtype=torch.uint8)
        d_ws = torch.empty(wsb.value, dtype=torch.uint8, device="cuda")
        st = torch.cuda.current_stream().cuda_stream

        def run():
            assert lib.lancirb200_resize_device(plan, d_src.data_ptr(), sw * ch, d_dst.data_ptr(), nw * ch,
                                                d_ws.data_ptr(), st) == 0
        ms = median_ms(run, 10, 3)
        # B = src + 2 * mid + dst; LANCIR's intermediate is [NewH][SrcW] fp32 (columns first)
        b = sw * sh * ch + 2 * sw * nh * ch * 4 + nw * nh * ch
        res.update({"ms_per_frame": ms, "src_Mpix_per_s": sw * sh / ms / 1e3,
                    "roofline": {"bound": "hbm", "achieved": b / ms / 1e6, "peak": peak, "unit": "GB/s",
                                 "frac": b / ms / 1e6 / peak, "algorithmic_bytes_per_frame": b}})
        lr = ab.CLancIR()
        t = []
        for i in range(5):
            t0 = time.perf_counter()
            r, got = lr.resizeImage(src, nw, nh)
            t.append(time.perf_counter() - t0)
        e2e = sorted(t[1:])[len(t[1:]) // 2]
        res["e2e"] = {"value": sw * sh / e2e / 1e6, "unit": "Mpix/s", "ms_per_frame": e2e * 1e3,
                      "h2d_bytes_per_step": sw * sh * ch, "d2h_bytes_per_step": nw * nh * ch,
                      "host_buffers": "pageable (numpy)"}
        if want_cpu:
            import oracle_ref as o
            if o.have_ref():
                tc = []
                for i in range(3):
                    t0 = time.perf_counter()
                    rr, want = o.lancir_ref(src, nw, nh, u8)
                    tc.append(time.perf_counter() - t0)
                cms = sorted(tc)[len(tc) // 2]
                res["cpu_baseline"] = {"value": sw * sh / cms / 1e6, "unit": "Mpix/s", "cores": 1, "kind": "reference",
                                       "ms_per_frame": cms * 1e3,
                                       "sample": "3 full frames, upstream lancir.h (AVX2 path, single-threaded by design)"}
                res["parity_vs_reference"] = int((want != got).sum())
        lib.lancirb200_plan_destroy(plan)
        hl.lancirb200_host_desc_free(h)
    except Exception as e:
        res["error"] = repr(e)[:200]
    return res


def run_own(args):
    import torch
    import torch.distributed as dist
    import avir_b200 as ab

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torchrun --nproc-per-node %d for --gpus %d" % (args.gpus, args.gpus))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    lib = ab.lib()
    declare(lib)
    fp = MIRRORS[args.mirror]
    N = world
    stream = torch.cuda.current_stream().cuda_stream
    peak, how = peaks()

    def barrier():
        if N > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device="cuda")
        if N > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    comm = C.c_void_p()
    if N > 1:
        idbuf = torch.zeros(128, dtype=torch.uint8)
        if rank == 0:
            raw = (C.c_char * 128)()
            assert lib.avirb200_comm_unique_id(raw) == 0, lib.avirb200_last_error().decode()
            idbuf = torch.frombuffer(bytearray(raw.raw), dtype=torch.uint8).clone()
        idg = idbuf.cuda()
        dist.broadcast(idg, 0)
        raw = (C.c_char * 128).from_buffer_copy(bytes(idg.cpu().numpy().tobytes()))
        assert lib.avirb200_comm_create(raw, rank, N, C.byref(comm)) == 0, lib.avirb200_last_error().decode()

    def sharded_run(pl, shape, tin, nw, nh, tout, ch, steps, warmup, seed, check):
        """Times avirb200_resize_sharded of one global image over the N ranks; `check`: compare
        every band with the 1-GPU avirb200_resize_device output of the same image."""
        sh_, sw_ = shape[0], shape[1]
        si, wsb = pl.shard(rank, N)
        d_src = device_random((si.src_rows, sw_, ch), tin, seed + rank)
        d_dst = torch.empty((si.dst_rows, nw, ch), device="cuda", dtype=torch_dtype(tout))
        d_ws = torch.empty(wsb, dtype=torch.uint8, device="cuda")

        def step():
            rr = lib.avirb200_resize_sharded(pl.plan, comm, rank, N, d_src.data_ptr(), sw_ * ch,
                                             d_dst.data_ptr(), nw * ch, d_ws.data_ptr(), stream)
            if rr != 0:
                raise SystemExit("resize_sharded failed: " + lib.avirb200_last_error().decode())
        total_ms = timed(step, steps, warmup)
        parity = None
        if check:
            parity = sharded_parity(pl, d_src, d_dst, si, sw_, nw, nh, ch, tin, tout)
        return total_ms / steps, si, parity, (d_src, d_dst, d_ws, step)

    def sharded_parity(pl, d_src, d_dst, si, sw_, nw, nh, ch, tin, tout):
        """Rank 0 gathers the source bands, runs the SAME plan unsharded on its GPU and compares
        every rank's destination band bit for bit (avir.h:5797-5806 is why the plan is global)."""
        step_rows = [torch.zeros(2, dtype=torch.int64, device="cuda") for _ in range(N)]
        dist.all_gather(step_rows, torch.tensor([si.src_rows, si.dst_rows], dtype=torch.int64, device="cuda"))
        rows = [(int(t[0]), int(t[1])) for t in step_rows]
        srcs = [torch.empty((r[0], sw_, ch), device="cuda", dtype=d_src.dtype) for r in rows] if rank == 0 else None
        dsts = [torch.empty((r[1], nw, ch), device="cuda", dtype=d_dst.dtype) for r in rows] if rank == 0 else None
        # (gather needs equal shapes; bands may differ by a row: point-to-point instead)
        if rank == 0:
            srcs[0].copy_(d_src)
            dsts[0].copy_(d_dst)
            for r in range(1, N):
                dist.recv(srcs[r].view(torch.uint8) if d_src.dtype == torch.uint16 else srcs[r], src=r)
                dist.recv(dsts[r].view(torch.uint8) if d_dst.dtype == torch.uint16 else dsts[r], src=r)
        else:
            dist.send(d_src.view(torch.uint8) if d_src.dtype == torch.uint16 else d_src, dst=0)
            dist.send(d_dst.view(torch.uint8) if d_dst.dtype == torch.uint16 else d_dst, dst=0)
        result = None
        if rank == 0:
            whole_src = torch.cat(srcs, 0)
            whole_dst = torch.empty((nh, nw, ch), device="cuda", dtype=d_dst.dtype)
            ws = torch.empty(pl.workspace(), dtype=torch.uint8, device="cuda")
            rr = lib.avirb200_resize_device(pl.plan, whole_src.data_ptr(), sw_ * ch, whole_dst.data_ptr(),
                                            nw * ch, ws.data_ptr(), stream)
            assert rr == 0, lib.avirb200_last_error()
            torch.cuda.synchronize()
            got = torch.cat(dsts, 0)
            a = whole_dst.view(torch.uint8) if whole_dst.dtype != torch.float32 else whole_dst.view(torch.int32)
            b = got.view(torch.uint8) if got.dtype != torch.float32 else got.view(torch.int32)
            per_band, y = [], 0
            for r in rows:
                per_band.append(int((a[y:y + r[1]] != b[y:y + r[1]]).sum().item()))
                y += r[1]
            result = {"mismatches": int(sum(per_band)), "per_band": per_band, "bands": N,
                      "against": "avirb200_resize_device of the same %dx%d image on one GPU" % (sw_, whole_src.shape[0])}
            del whole_src, whole_dst, ws, got
        barrier()
        return result

    # ---- headline: N stacked frames, plan for the global image
    pl = Plan(ab, fp, (SRC_H * N, SRC_W, CH), np.float32, DST_W, DST_H * N, np.float32, 16)
    si, wsb = pl.shard(rank, N)
    # source: SURVEY 8(d) generator (host), pinned, copied to the device once
    h_src = torch.from_numpy(synthetic_image(si.src_rows, SRC_W, CH, np.float32, seed=12345 + rank)).pin_memory()
    d_src = h_src.cuda()
    d_dst = torch.empty((si.dst_rows, DST_W, CH), device="cuda", dtype=torch.float32)
    d_ws = torch.empty(max(wsb, pl.workspace() if N == 1 else 0), dtype=torch.uint8, device="cuda")

    def step():
        if N == 1:
            rr = lib.avirb200_resize_device(pl.plan, d_src.data_ptr(), SRC_W * CH, d_dst.data_ptr(),
                                            DST_W * CH, d_ws.data_ptr(), stream)
        else:
            rr = lib.avirb200_resize_sharded(pl.plan, comm, rank, N, d_src.data_ptr(), SRC_W * CH,
                                             d_dst.data_ptr(), DST_W * CH, d_ws.data_ptr(), stream)
        if rr != 0:
            raise SystemExit("resize failed: " + lib.avirb200_last_error().decode())

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    t0 = time.time()
    total_ms = timed(step, args.steps, args.warmup)
    t1 = time.time()
    clocks = sampler.stop(t0, t1) if rank == 0 else None
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, d_dst, "output" if N == 1 else "output_rank%d" % rank, N)
    launches_per_step = lib.avirb200_plan_last_launches(pl.plan)
    ms_per_step = total_ms / args.steps
    value = SRC_W * SRC_H * N / (ms_per_step * 1e-3) / 1e6
    ab_ = algorithmic_bytes()

    # ---- per-kernel timing for the roofline
    roof = None
    shard_par = None
    if N == 1:
        row_ms = timed(lambda: lib.avirb200_row_pass_device(pl.plan, d_src.data_ptr(), SRC_W * CH,
                                                           d_ws.data_ptr(), stream), args.steps, 2) / args.steps
        col_ms = timed(lambda: lib.avirb200_col_pass_device(pl.plan, d_ws.data_ptr(), d_dst.data_ptr(),
                                                           DST_W * CH, stream), args.steps, 2) / args.steps
        dom = "row" if row_ms >= col_ms else "col"
        dom_ms = max(row_ms, col_ms)
        ach = ab_[dom] / (dom_ms * 1e-3) / 1e9
        tr = traffic_from_profiles()
        roof = {"bound": "hbm", "kernel": dom + "_pass", "achieved": ach, "peak": peak, "unit": "GB/s",
                "frac": ach / peak, "traffic": tr.get(dom + "_pass"), "peak_source": how,
                "algorithmic_bytes_per_launch": ab_[dom],
                "kernels": {"row_pass": {"ms": row_ms, "GBps": ab_["row"] / row_ms / 1e6,
                                         "frac": ab_["row"] / row_ms / 1e6 / peak},
                            "col_pass": {"ms": col_ms, "GBps": ab_["col"] / col_ms / 1e6,
                                         "frac": ab_["col"] / col_ms / 1e6 / peak}},
                "whole_step": {"GBps": ab_["total"] / ms_per_step / 1e6,
                               "frac": ab_["total"] / ms_per_step / 1e6 / peak}}
    else:
        # every rank runs the same two kernels on its band; the whole job against N x the peak
        agg = ab_["total"] * N / ms_per_step / 1e6
        roof = {"bound": "hbm", "kernel": "row_pass + halo exchange + col_pass (whole step, all ranks)",
                "achieved": agg, "peak": peak * N, "unit": "GB/s", "frac": agg / (peak * N), "traffic": None,
                "peak_source": how + " x %d GPUs" % N, "algorithmic_bytes_per_launch": ab_["total"] * N}
        step()
        torch.cuda.synchronize()
        shard_par = sharded_parity(pl, d_src, d_dst, si, SRC_W, DST_W, DST_H * N, CH, np.float32, np.float32)

    # ---- end to end through the public API, host buffers, copies inside the timed region
    h_dst = torch.empty((si.dst_rows, DST_W, CH), dtype=torch.float32).pin_memory()
    e2e_variants = {}
    if N == 1:
        rs = ab.CImageResizer(16, 0, 0, fp)
        src_np, dst_np = h_src.numpy(), h_dst.numpy()

        def e2e_step():
            rs.resizeImage(src_np, DST_W, DST_H, 0.0, NewBuf=dst_np)  # H2D + passes + D2H + sync
    else:
        src_np, dst_np = h_src.numpy(), h_dst.numpy()

        def e2e_step():
            rr = lib.avirb200_resize_sharded_host(pl.plan, comm, rank, N, src_np.ctypes.data, SRC_W * CH,
                                                  dst_np.ctypes.data, DST_W * CH)
            if rr != 0:
                raise SystemExit("resize_sharded_host failed: " + lib.avirb200_last_error().decode())

    def wall(fn, steps):
        for _ in range(2):
            fn()
        barrier()
        tw0 = time.perf_counter()
        for _ in range(steps):
            fn()
        barrier()
        s = torch.tensor([time.perf_counter() - tw0], device="cuda")
        if N > 1:
            dist.all_reduce(s, op=dist.ReduceOp.MAX)
        return float(s.item()) / steps
    e2e_steps = max(3, min(args.steps, 10))
    e2e_s = wall(e2e_step, e2e_steps)
    e2e_val = SRC_W * SRC_H * N / e2e_s / 1e6
    e2e_out_first = dst_np[:2].copy() if N == 1 else None

    parity_ref = None
    cpu = None
    extras, lancir, batch = None, None, None
    if N == 1 and not args.no_extras:
        # pageable (malloc) host buffers: what a drop-in caller hands over
        pg_src = np.empty_like(src_np)
        pg_src[...] = src_np
        pg_dst = np.empty_like(dst_np)
        s_pg = wall(lambda: rs.resizeImage(pg_src, DST_W, DST_H, 0.0, NewBuf=pg_dst), 3)
        e2e_variants["pageable_f32"] = {"value": SRC_W * SRC_H / s_pg / 1e6, "unit": "Mpix/s", "ms_per_frame": s_pg * 1e3,
                                        "h2d_bytes_per_step": src_np.nbytes, "d2h_bytes_per_step": dst_np.nbytes,
                                        "matches_pinned": bool(np.array_equal(pg_dst[:2], e2e_out_first))}
        del pg_src, pg_dst
        # u8 wire format (8K -> 4K RGBA u8, float4 mirror): 133 MB in, 33 MB out
        rs8 = ab.CImageResizer(8, 0, 0, 1)
        s8 = torch.from_numpy(synthetic_image(SRC_H, SRC_W, CH, u8)).pin_memory().numpy()
        d8 = torch.empty((DST_H, DST_W, CH), dtype=torch.uint8).pin_memory().numpy()
        s_u8 = wall(lambda: rs8.resizeImage(s8, DST_W, DST_H, 0.0, NewBuf=d8), 5)
        e2e_variants["pinned_u8"] = {"value": SRC_W * SRC_H / s_u8 / 1e6, "unit": "Mpix/s", "ms_per_frame": s_u8 * 1e3,
                                     "h2d_bytes_per_step": s8.nbytes, "d2h_bytes_per_step": d8.nbytes}
        p8 = np.empty_like(s8)
        p8[...] = s8
        q8 = np.empty_like(d8)
        s_u8p = wall(lambda: rs8.resizeImage(p8, DST_W, DST_H, 0.0, NewBuf=q8), 5)
        e2e_variants["pageable_u8"] = {"value": SRC_W * SRC_H / s_u8p / 1e6, "unit": "Mpix/s", "ms_per_frame": s_u8p * 1e3,
                                       "h2d_bytes_per_step": s8.nbytes, "d2h_bytes_per_step": d8.nbytes}
        del s8, d8, p8, q8, rs8

    # ---- CPU baseline: upstream itself on the host cores (rank 0, N = 1 only) + output parity
    if rank == 0 and N == 1 and not args.no_cpu_baseline:
        import oracle_ref as o
        if o.have_ref():
            src = h_src.numpy()
            cores = pick_threads(o, src, fp, os.cpu_count() or 1)
            ts = []
            tb = time.perf_counter()
            want = None
            while len(ts) < 3 or (time.perf_counter() - tb < 12 and len(ts) < 10):
                t_ = time.perf_counter()
                want = o.ref_resize(src, DST_W, DST_H, np.float32, fpclass=fp, resbits=16, nthreads=cores)
                ts.append(time.perf_counter() - t_)
            med = sorted(ts)[len(ts) // 2]
            cpu = {"value": SRC_W * SRC_H / med / 1e6, "unit": "Mpix/s", "cores": cores,
                   "kind": "reference", "ms_per_frame": med * 1e3,
                   "sample": "%d full 7680x4320 frames, upstream headers (-O2 -mavx2 "
                             "-ffp-contract=off) on a std::thread pool of %d workloads (fastest of a "
                             "sweep up to %d host threads)" % (len(ts), cores, os.cpu_count() or 1)}
            # the benchmarked frame (device-resident path AND the host call) against upstream's frame
            step()
            torch.cuda.synchronize()
            got = d_dst.cpu().numpy()
            parity_ref = {"device_path_mismatches": int((got.view(np.uint32) != want.view(np.uint32)).sum()),
                          "host_call_mismatches": int((dst_np.view(np.uint32) != want.view(np.uint32)).sum()),
                          "elements": int(want.size), "tolerance": "bit-exact (0 ULP)"}
            del got, want

    if N == 1 and not args.no_extras:
        # ---- batch entry: 8 frames, one plan, one launch pair per frame on one stream
        nb = 8
        srcs = [d_src] + [device_random((SRC_H, SRC_W, CH), f32, 100 + i) for i in range(3)]
        dsts = [torch.empty((DST_H, DST_W, CH), device="cuda", dtype=torch.float32) for _ in range(nb)]
        sp = (C.c_void_p * nb)(*[srcs[i % len(srcs)].data_ptr() for i in range(nb)])
        dp_ = (C.c_void_p * nb)(*[t.data_ptr() for t in dsts])

        def bstep():
            assert lib.avirb200_resize_device_batch(pl.plan, nb, sp, SRC_W * CH, dp_, DST_W * CH,
                                                    d_ws.data_ptr(), stream) == 0
        bms = median_ms(bstep, 5, 2)
        batch = {"frames": nb, "ms_per_batch": bms, "value": SRC_W * SRC_H * nb / bms / 1e3, "unit": "Mpix/s",
                 "same_bits_as_single_call": bool(torch.equal(dsts[0], d_dst))}
        del srcs, dsts
        torch.cuda.empty_cache()
        extras = run_extra_configs(ab, peak, budget_s=60)
        lancir = run_lancir(ab, peak, rank == 0 and not args.no_cpu_baseline)

    multi = None
    if N > 1 and not args.no_extras:
        multi = {}
        # strong scaling: ONE 8K frame over the N GPUs
        try:
            p1 = Plan(ab, fp, (SRC_H, SRC_W, CH), f32, DST_W, DST_H, f32, 16)
            ms, si1, par, keep = sharded_run(p1, (SRC_H, SRC_W), f32, DST_W, DST_H, f32, CH, args.steps, 3, 500, True)
            b1 = algorithmic_bytes()["total"]
            multi["strong_8k_frame"] = {"workload": "one 7680x4320->3840x2160 RGBA f32 frame row-sharded over %d GPUs" % N,
                                        "scaling": "strong", "ms_per_frame": ms, "value": SRC_W * SRC_H / ms / 1e3,
                                        "unit": "Mpix/s", "halo_rows": [si1.halo_up, si1.halo_down],
                                        "roofline": {"bound": "hbm", "achieved": b1 / ms / 1e6, "peak": peak * N,
                                                     "unit": "GB/s", "frac": b1 / ms / 1e6 / (peak * N)},
                                        "sharded_parity": par}
            del keep
            p1.close()
            torch.cuda.empty_cache()
        except BaseException as e:
            multi["strong_8k_frame"] = {"error": repr(e)[:200]}
        # cfg4: 16384^2 -> 4096^2 u16 row-sharded (BASELINE configs[3])
        try:
            p4 = Plan(ab, 1, (16384, 16384, 4), u16, 4096, 4096, u16, 16)
            ms, si4, par, keep = sharded_run(p4, (16384, 16384), u16, 4096, 4096, u16, 4, max(5, args.steps // 2), 3, 700, True)
            b4 = algorithmic_bytes(16384, 16384, 4096, 4096, 4, u16, u16)["total"]
            multi["cfg4_row_sharded"] = {"workload": "cfg4 16384x16384->4096x4096 RGBA u16 row-sharded over %d GPUs" % N,
                                         "scaling": "strong", "ms_per_frame": ms, "value": 16384 * 16384 / ms / 1e3,
                                         "unit": "Mpix/s", "halo_rows": [si4.halo_up, si4.halo_down],
                                         "roofline": {"bound": "hbm", "achieved": b4 / ms / 1e6, "peak": peak * N,
                                                      "unit": "GB/s", "frac": b4 / ms / 1e6 / (peak * N)},
                                         "sharded_parity": par}
            del keep
            p4.close()
            torch.cuda.empty_cache()
        except BaseException as e:
            multi["cfg4_row_sharded"] = {"error": repr(e)[:200]}
        # cfg5: 8K -> 1080p u8 + sRGB, one frame per GPU (replicas, no exchange) -- BASELINE configs[4]
        try:
            p5 = Plan(ab, 2, (SRC_H, SRC_W, 4), u8, 1920, 1080, u8, 8, {"gamma": True, "alpha": 3})
            s5 = device_random((SRC_H, SRC_W, 4), u8, 900 + rank)
            o5 = torch.empty((1080, 1920, 4), device="cuda", dtype=torch.uint8)
            w5 = torch.empty(p5.workspace(), dtype=torch.uint8, device="cuda")

            def step5():
                assert lib.avirb200_resize_device(p5.plan, s5.data_ptr(), SRC_W * 4, o5.data_ptr(), 1920 * 4,
                                                  w5.data_ptr(), stream) == 0
            ms5 = timed(step5, args.steps, 3) / args.steps
            b5 = algorithmic_bytes(SRC_W, SRC_H, 1920, 1080, 4, u8, u8)["total"]
            multi["cfg5_replicas"] = {"workload": "cfg5 7680x4320->1920x1080 RGBA u8 + sRGB, one frame per GPU, %d GPUs" % N,
                                      "scaling": "weak", "ms_per_step": ms5, "value": SRC_W * SRC_H * N / ms5 / 1e3,
                                      "unit": "Mpix/s",
                                      "roofline": {"bound": "hbm", "achieved": b5 * N / ms5 / 1e6, "peak": peak * N,
                                                   "unit": "GB/s", "frac": b5 / ms5 / 1e6 / peak}}
            del s5, o5, w5
            p5.close()
        except BaseException as e:
            multi["cfg5_replicas"] = {"error": repr(e)[:200]}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "Mpix/s", "n_gpus": N, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": dict(workload_config(args, N), build_modes=list(pl.modes),
                           halo_rows=[si.halo_up, si.halo_down]),
            "roofline": roof, "cpu_baseline": cpu,
            "e2e": {"value": e2e_val, "unit": "Mpix/s",
                    "h2d_bytes_per_step": int(si.src_rows) * SRC_W * CH * 4 * N,
                    "d2h_bytes_per_step": int(si.dst_rows) * DST_W * CH * 4 * N,
                    "steps": e2e_steps, "host_buffers": "pinned",
                    "api": "avir::CImageResizer<>::resizeImage" if N == 1 else "avirb200_resize_sharded_host"},
            "gpu_launches": int(launches_per_step) * args.steps, "clocks": clocks,
        }
        if parity_ref is not None:
            line["parity_vs_reference"] = parity_ref
        if shard_par is not None:
            line["sharded_parity"] = shard_par
        if e2e_variants:
            line["e2e_variants"] = e2e_variants
        if batch is not None:
            line["batch"] = batch
        if extras is not None:
            line["configs"] = extras
        if lancir is not None:
            line["lancir"] = lancir
        if multi is not None:
            line["multi_gpu_configs"] = multi
        print(json.dumps(line))
    if N > 1:
        lib.avirb200_comm_destroy(comm)
        dist.destroy_process_group()
    pl.close()


DUMP_ROWS = 512  # rows of the 3840-wide RGBA float destination: 31.5 MB over all ranks


def dump_outputs(d, d_dst, name, n_ranks):
    """Saves what the last timed step left in d_dst (the caller's destination image): a fixed,
    seeded sample of whole rows, DIR/<name>.npy (float32, rows x DST_W x CH), and the row numbers
    within the band, DIR/<name>_rows.npy (float64)."""
    rows = np.sort(np.random.default_rng(0).choice(d_dst.shape[0], min(d_dst.shape[0], DUMP_ROWS // n_ranks),
                                                   replace=False))
    import torch
    os.makedirs(d, exist_ok=True)
    np.save(os.path.join(d, name + ".npy"), d_dst.index_select(0, torch.as_tensor(rows, device=d_dst.device)).cpu().numpy())
    np.save(os.path.join(d, name + "_rows.npy"), rows.astype(np.float64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="own", choices=["own", "reference"])
    ap.add_argument("--mirror", default="dil", choices=sorted(MIRRORS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--halo-mode", type=int, default=None, choices=[0, 1, 2, 3],
                    help="sharded runs: AVIRB200_OPT_OVERLAP_HALO (default: the library's)")
    ap.add_argument("--no-extras", action="store_true", help="headline only (no secondary configs / LANCIR / variants)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/*.npy (a seeded sample of its rows)")
    args = ap.parse_args()
    Plan.halo_mode = args.halo_mode
    args.warmup = max(args.warmup, 3) if args.impl == "own" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_own(args)


if __name__ == "__main__":
    main()
