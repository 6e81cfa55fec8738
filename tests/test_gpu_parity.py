"""GPU parity tests proper (run with -m gpu on a B200): the product path -- C++ front-end ->
C ABI -> sm_100a kernels -- against upstream's outputs (digests in tests/golden/upstream.json,
recorded from upstream compiled in-tree) and the committed golden fixtures.  Bit-exact
everywhere: integer output AND float output (0 ULP; the north-star tolerance for float is 1 ULP,
the tests demand 0).
"""
import ctypes as C
import os

import numpy as np
import pytest

import avir_b200 as ab
import cases as cs
import oracle_ref as o

pytestmark = pytest.mark.gpu

def _oracle_threads():
    """Threads for the multi-threaded upstream oracle: the cores this process may actually use
    (a container often sees every host core in os.cpu_count() but is scheduled on a few;
    upstream's workers spin while they wait), capped."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 8
    return max(1, min(n, 16))


@pytest.fixture(params=[0, 2, 1], ids=["product", "tile", "generic"])
def kernel_path(request):
    """Every parity case runs in the product's kernel order (warp-streaming kernel where the
    chain is regular, else the tile kernel, else the generic kernel), with the streaming
    kernel switched off (tile kernel where it applies), and through the fully generic kernel."""
    ab.set_option(ab.OPT_KERNEL_FAMILY, request.param)
    yield request.param
    ab.set_option(ab.OPT_KERNEL_FAMILY, -1)


def test_native_library_is_what_runs():
    assert ab.device_count() >= 1
    lib = ab.lib()
    assert lib.avirb200_plan_last_launches  # symbol present; launches counted per call


@pytest.mark.parametrize("case", cs.SMALL_CASES, ids=cs.case_id)
def test_small_cases_bit_exact(case, kernel_path):
    src = cs.make_input(case)
    got = cs.gpu_output(case, src)
    assert cs.matches_upstream(case, src, got)


@pytest.mark.parametrize("structured", ["ramp", "impulse", "checker"])
@pytest.mark.parametrize("case", cs.SMALL_CASES[:10], ids=cs.case_id)
def test_structured_inputs_bit_exact(case, structured, kernel_path):
    src = cs.make_input(case, structured=structured)
    got = cs.gpu_output(case, src)
    assert cs.matches_upstream(case, src, got)


def test_golden_fixtures():
    files = sorted(f for f in os.listdir(cs.GOLDEN) if f.startswith("avir_") and f.endswith(".npz"))
    for f in files:
        z = np.load(os.path.join(cs.GOLDEN, f), allow_pickle=True)
        case = tuple(z["case"].tolist())
        case = case[:6] + (np.dtype(case[6]).type, np.dtype(case[7]).type) + case[8:]
        got = cs.gpu_output(case, z["src"])
        assert cs.count_mismatch(z["out"], got) == 0, f


def test_zero_size_conventions():
    # avir.h:4686-4697: empty source -> destination zero-filled; empty destination -> no-op
    rs = ab.CImageResizer(8, 0, 0, ab.FP_FLOAT4)
    dst = np.full((4, 4, 4), 7, np.uint8)
    out = rs.resizeImage(np.zeros((0, 0, 4), np.uint8).reshape(0, 0, 4), 4, 4, NewBuf=dst)
    # upstream clears NewWidth*NewHeight ELEMENTS (not pixels): avir.h:4688-4689
    assert np.all(out.ravel()[:16] == 0) and np.all(out.ravel()[16:] == 7)


# ---- medium sizes: many tiles per pass, multi-threaded upstream as the oracle --------------

MEDIUM = [
    (2, 1920, 1080, 960, 540, 4, np.float32, np.float32, 16, {}),                 # cfg3 / 4
    (1, 1920, 1080, 960, 540, 4, np.float32, np.float32, 16, {}),
    (1, 960, 540, 1920, 1080, 4, np.uint8, np.uint8, 8, {}),                      # cfg2 / 2
    (1, 2048, 2048, 512, 512, 4, np.uint16, np.uint16, 16, {}),                   # cfg4 / 8
    (2, 1920, 1080, 480, 270, 4, np.uint8, np.uint8, 8, {"gamma": True, "alpha": 3}),  # cfg5 / 4
    (0, 1280, 720, 2000, 1125, 3, np.uint8, np.uint8, 8, {}),                     # cfg1 ratio
    (1, 1500, 1000, 1111, 741, 4, np.uint8, np.uint8, 8, {}),                     # many phases
    (2, 1500, 1000, 1111, 741, 4, np.float32, np.float32, 16, {}),
]


def _upstream_mt(case, src):
    """Upstream's output digest; recording runs upstream multi-threaded (same bits)."""
    fp, sw, sh, nw, nh, ch, ti, to, rb, kw = case
    return cs.upstream(cs.avir_key(case, src), lambda: o.ref_resize(
        src, nw, nh, to, fpclass=fp, resbits=rb, nthreads=_oracle_threads(), **cs.ref_kwargs(kw)))


@pytest.mark.parametrize("case", MEDIUM, ids=cs.case_id)
def test_medium_cases_bit_exact(case):
    src = cs.make_input(case, seed=11)
    got = cs.gpu_output(case, src)
    assert cs.digest(got) == _upstream_mt(case, src)


def test_generic_and_fast_kernels_agree_on_medium():
    case = MEDIUM[0]
    src = cs.make_input(case, seed=5)
    a = cs.gpu_output(case, src)
    ab.set_option(ab.OPT_KERNEL_FAMILY, 1)
    try:
        b = cs.gpu_output(case, src)
    finally:
        ab.set_option(ab.OPT_KERNEL_FAMILY, -1)
    assert cs.count_mismatch(a, b) == 0


# ---- streaming chains that are instantiated but not selected by default -----------------------

@pytest.mark.parametrize("case", [
    # (cfg5 chain: only in builds made with AVIRB200_BUILD_ALL_CHAINS=1; else these run the tile kernel)
    (2, 388, 220, 97, 55, 4, np.uint8, np.uint8, 8, {"gamma": True, "alpha": 3, "buildmode": 1}),
    (2, 768, 432, 192, 108, 4, np.float32, np.float32, 16, {"buildmode": 1}),
    (1, 242, 137, 484, 274, 4, np.uint8, np.uint8, 8, {"buildmode": 1}),                           # cfg2 chain
    (1, 480, 270, 960, 540, 4, np.float32, np.uint16, 16, {"buildmode": 1}),
], ids=cs.case_id)
def test_deselected_streaming_chains_bit_exact(case):
    """The upsizing and the 56-tap chain run on the tile kernel by default (it measured faster);
    the ALL_STREAM_CHAINS plan option selects their streaming instantiations, which must give
    the same bits."""
    src = cs.make_input(case, seed=31)
    ab.set_option(ab.OPT_ALL_STREAM_CHAINS, 1)
    try:
        got = cs.gpu_output(case, src)
    finally:
        ab.set_option(ab.OPT_ALL_STREAM_CHAINS, -1)
    assert cs.matches_upstream(case, src, got)


# ---- pipelined host call: row bands over copy-in / compute / copy-out streams ----------------

@pytest.mark.parametrize("bands", [2, 3, 7, 16])
@pytest.mark.parametrize("case", [MEDIUM[0], MEDIUM[2], MEDIUM[3], MEDIUM[4], MEDIUM[6],
                                  (0, 300, 200, 431, 287, 3, np.uint8, np.uint8, 8, {})], ids=cs.case_id)
def test_banded_host_call_matches_single_band(case, bands):
    """avirb200_resize_host cuts large images into row bands so that PCIe transfers overlap the
    kernels; the band count must not change a bit (the HOST_BANDS plan option forces it)."""
    src = cs.make_input(case, seed=23)
    ab.set_option(ab.OPT_HOST_BANDS, 1)
    try:
        one = cs.gpu_output(case, src)
        ab.set_option(ab.OPT_HOST_BANDS, bands)
        many = cs.gpu_output(case, src)
    finally:
        ab.set_option(ab.OPT_HOST_BANDS, -1)
    assert cs.count_mismatch(one, many) == 0
    assert cs.matches_upstream(case, src, many)


def test_banded_host_call_in_place():
    """NewBuf may alias SrcBuf (avir.h:4650-4652): the banded path must not be taken then."""
    case = (1, 512, 512, 256, 256, 4, np.uint8, np.uint8, 8, {})
    src = cs.make_input(case, seed=29)
    want = cs.gpu_output(case, src)
    ab.set_option(ab.OPT_HOST_BANDS, 4)  # the overlap check must win over the forced banding
    try:
        buf = src.copy()
        rs = ab.CImageResizer(8, 0, 0, ab.FP_FLOAT4)
        dst = buf.reshape(-1)[:256 * 256 * 4].reshape(256, 256, 4)
        out = rs.resizeImage(buf, 256, 256, NewBuf=dst)
    finally:
        ab.set_option(ab.OPT_HOST_BANDS, -1)
    assert cs.count_mismatch(want, out) == 0


# ---- BASELINE.json full sizes ----------------------------------------------------------------

def _device_run(case, src, sharded_local=0):
    """Device-resident call through the C ABI with torch-managed buffers."""
    import torch
    fp, sw, sh, nw, nh, ch, ti, to, rb, kw = case
    rs, v = cs.resizer_and_vars(case)
    tmap = {np.uint8: torch.uint8, np.uint16: torch.uint16, np.float32: torch.float32}
    d_src = torch.from_numpy(src).cuda()
    d_dst = torch.empty((nh, nw, ch), dtype=tmap[to], device="cuda")
    ws = rs.workspaceBytes(src.shape, ti, nw, nh, to, kw.get("k", 0.0), v)
    d_ws = torch.empty(ws, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    rs.resizeImageDevice(d_src.data_ptr(), src.shape, ti, d_dst.data_ptr(), nw, nh, to,
                         d_ws.data_ptr(), kw.get("k", 0.0), v, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return d_dst.cpu().numpy()


FULL = [
    ("cfg2", (1, 1920, 1080, 3840, 2160, 4, np.uint8, np.uint8, 8, {})),
    ("cfg3-dil", (2, 7680, 4320, 3840, 2160, 4, np.float32, np.float32, 16, {})),
    ("cfg3-f4", (1, 7680, 4320, 3840, 2160, 4, np.float32, np.float32, 16, {})),
    ("cfg5", (2, 7680, 4320, 1920, 1080, 4, np.uint8, np.uint8, 8, {"gamma": True, "alpha": 3})),
]


@pytest.mark.parametrize("name,case", FULL, ids=[f[0] for f in FULL])
def test_full_size_baseline_configs_bit_exact(name, case):
    """BASELINE.json configs at full size, device-resident path, vs multi-threaded upstream."""
    fp, sw, sh, nw, nh, ch, ti, to, rb, kw = case
    src = o.lcg_image(sh, sw, ch, ti, seed=12345)
    got = _device_run(case, src)
    assert cs.digest(got) == _upstream_mt(case, src)


def test_full_size_cfg4_bit_exact():
    """BASELINE configs[3] at full size, 16384^2 -> 4096^2 RGBA u16, against multi-threaded
    upstream (a few seconds per thread-second of a 1.07 GB intermediate)."""
    case = (1, 16384, 16384, 4096, 4096, 4, np.uint16, np.uint16, 16, {})
    fp, sw, sh, nw, nh, ch, ti, to, rb, kw = case
    src = o.lcg_image(sh, sw, ch, ti, seed=4)
    got = _device_run(case, src)
    assert cs.digest(got) == _upstream_mt(case, src)


@pytest.mark.parametrize("variant", [0, 1, 2])
@pytest.mark.parametrize("case", [
    (2, 1920, 1080, 960, 540, 4, np.float32, np.float32, 16, {}),          # cfg3 chain
    (2, 1000, 531, 500, 266, 4, np.float32, np.uint8, 8, {}),              # ragged strips, integer output
    (1, 1920, 1080, 960, 540, 4, np.float32, np.float32, 16, {}),          # float4 mirror: 3-step chain
    (1, 2048, 1024, 512, 256, 4, np.uint16, np.uint16, 16, {}),            # cfg4 chain, integer source
    (1, 1920, 1080, 960, 540, 4, np.uint8, np.uint8, 8, {}),               # k = 2 mode 1, u8
], ids=cs.case_id)
def test_stream_scheduling_variants_bit_exact(case, variant):
    """Scheduling variants of the streaming kernel (0 ring windows, 1 register windows, 2 register
    windows + TMA-staged column pass): same bits as upstream."""
    src = cs.make_input(case, seed=51)
    ab.set_option(ab.OPT_STREAM_VARIANT_H, variant)
    ab.set_option(ab.OPT_STREAM_VARIANT_V, variant)
    try:
        got = cs.gpu_output(case, src)
    finally:
        ab.set_option(ab.OPT_STREAM_VARIANT_H, -1)
        ab.set_option(ab.OPT_STREAM_VARIANT_V, -1)
    assert cs.matches_upstream(case, src, got)


def test_batch_entry_matches_single_calls():
    """avirb200_resize_device_batch: n frames through one plan = n single calls."""
    import torch
    case = (2, 640, 360, 320, 180, 4, np.float32, np.float32, 16, {})
    fp, sw, sh, nw, nh, ch, ti, to, rb, kw = case
    rs, v = cs.resizer_and_vars(case)
    h, dp, _ = rs.descriptor((sh, sw, ch), ti, nw, nh, to, 0.0, v)
    lib = ab.lib()
    plan = C.c_void_p()
    assert lib.avirb200_plan_create(C.c_void_p(dp), C.byref(plan)) == 0
    wsb = C.c_size_t()
    assert lib.avirb200_plan_workspace_bytes(plan, C.byref(wsb)) == 0
    n = 5
    srcs = [torch.from_numpy(cs.make_input(case, seed=60 + i)).cuda() for i in range(n)]
    dsts = [torch.zeros((nh, nw, ch), device="cuda") for _ in range(n)]
    d_ws = torch.empty(wsb.value, dtype=torch.uint8, device="cuda")
    sp = (C.c_void_p * n)(*[t.data_ptr() for t in srcs])
    dpp = (C.c_void_p * n)(*[t.data_ptr() for t in dsts])
    lib.avirb200_resize_device_batch.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t, C.c_void_p,
                                                 C.c_size_t, C.c_void_p, C.c_void_p]
    assert lib.avirb200_resize_device_batch(plan, n, sp, sw * ch, dpp, nw * ch, d_ws.data_ptr(), None) == 0
    torch.cuda.synchronize()
    lib.avirb200_plan_destroy(plan)
    rs.free_descriptor(h)
    for i in range(n):
        assert cs.matches_upstream(case, srcs[i].cpu().numpy(), dsts[i].cpu().numpy()), i


def test_full_size_properties_cfg4():
    """16384^2 -> 4096^2 u16 (cfg4) is too slow for the CPU oracle in a test; check
    size-independent properties instead: a constant image stays constant (unity DC gain of
    the whole chain incl. edges), and the sharded schedule reproduces the unsharded bits."""
    import torch
    case = (1, 16384, 4096, 4096, 1024, 4, np.uint16, np.uint16, 16, {})  # quarter height
    fp, sw, sh, nw, nh, ch, ti, to, rb, kw = case
    const = np.full((sh, sw, ch), 40000, np.uint16)
    out = _device_run(case, const)
    assert out.min() == 40000 and out.max() == 40000
    src = o.lcg_image(sh, sw, ch, ti, seed=99)
    whole = _device_run(case, src)
    # sharded-local: 8 bands on one device, halo rows moved by device copies
    rs, v = cs.resizer_and_vars(case)
    h, dp, _ = rs.descriptor(src.shape, ti, nw, nh, to, 0.0, v)
    lib = ab.lib()
    plan = C.c_void_p()
    assert lib.avirb200_plan_create(C.c_void_p(dp), C.byref(plan)) == 0
    total = 0
    for r in range(8):
        b = C.c_size_t()
        assert lib.avirb200_shard_workspace_bytes(plan, r, 8, C.byref(b)) == 0
        total += b.value
    d_src = torch.from_numpy(src).cuda()
    d_dst = torch.empty((nh, nw, ch), dtype=torch.uint16, device="cuda")
    d_ws = torch.empty(total, dtype=torch.uint8, device="cuda")
    lib.avirb200_resize_sharded_local.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t,
                                                  C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]
    assert lib.avirb200_resize_sharded_local(plan, 8, d_src.data_ptr(), sw * ch, d_dst.data_ptr(),
                                             nw * ch, d_ws.data_ptr(), None) == 0
    torch.cuda.synchronize()
    lib.avirb200_plan_destroy(plan)
    rs.free_descriptor(h)
    assert cs.count_mismatch(whole, d_dst.cpu().numpy()) == 0


@pytest.mark.parametrize("nranks", [2, 5, 8])
def test_sharded_local_matches_unsharded(nranks):
    import torch
    case = (2, 640, 720, 320, 360, 4, np.float32, np.float32, 16, {})
    fp, sw, sh, nw, nh, ch, ti, to, rb, kw = case
    src = cs.make_input(case, seed=21)
    rs, v = cs.resizer_and_vars(case)
    h, dp, _ = rs.descriptor(src.shape, ti, nw, nh, to, 0.0, v)
    lib = ab.lib()
    plan = C.c_void_p()
    assert lib.avirb200_plan_create(C.c_void_p(dp), C.byref(plan)) == 0
    total = 0
    for r in range(nranks):
        b = C.c_size_t()
        assert lib.avirb200_shard_workspace_bytes(plan, r, nranks, C.byref(b)) == 0
        total += b.value
    d_src = torch.from_numpy(src).cuda()
    d_dst = torch.zeros((nh, nw, ch), dtype=torch.float32, device="cuda")
    d_ws = torch.empty(total, dtype=torch.uint8, device="cuda")
    lib.avirb200_resize_sharded_local.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t,
                                                  C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]
    assert lib.avirb200_resize_sharded_local(plan, nranks, d_src.data_ptr(), sw * ch,
                                             d_dst.data_ptr(), nw * ch, d_ws.data_ptr(), None) == 0
    torch.cuda.synchronize()
    lib.avirb200_plan_destroy(plan)
    rs.free_descriptor(h)
    assert cs.matches_upstream(case, src, d_dst.cpu().numpy())


# The fused halo exchange (AVIRB200_OPT_OVERLAP_HALO = 3: the row kernel stores the neighbours' rows into
# their mailboxes and raises flags, the column kernel reads them in place) on ONE device: the bands of the
# sharded schedule run one after another with every mailbox in local memory -- the same kernels, parameters
# and protocol as between ranks (tests/test_gpu_nccl.py is the multi-process form).
FUSED_LOCAL = [
    (2, 640, 720, 320, 360, 4, np.float32, np.float32, 16, {}),                              # headline chain
    (1, 640, 720, 320, 360, 4, np.float32, np.float32, 16, {}),                              # three-step chain
    (1, 1024, 1536, 256, 384, 4, np.uint16, np.uint16, 16, {}),                              # cfg4 chain
    (2, 1024, 1536, 256, 384, 4, np.uint8, np.uint8, 8, {"gamma": True, "alpha": 3}),        # cfg5 chain, sRGB table
    (1, 640, 720, 320, 360, 4, np.uint8, np.uint8, 8, {}),                                   # integer source and output
    (0, 512, 600, 256, 300, 3, np.uint8, np.uint8, 8, {}),                                   # 3 channels on the 4-channel kernels
]


@pytest.mark.parametrize("overlap", [3, 1])
@pytest.mark.parametrize("nranks", [2, 3, 5])
@pytest.mark.parametrize("case", FUSED_LOCAL, ids=cs.case_id)
def test_sharded_local_fused_exchange_matches_unsharded(case, nranks, overlap):
    import torch
    fp, sw, sh, nw, nh, ch, ti, to, rb, kw = case
    src = cs.make_input(case, seed=33)
    whole = _device_run(case, src)
    rs, v = cs.resizer_and_vars(case)
    h, dp, _ = rs.descriptor(src.shape, ti, nw, nh, to, 0.0, v)
    lib = ab.lib()
    plan = C.c_void_p()
    assert lib.avirb200_plan_create(C.c_void_p(dp), C.byref(plan)) == 0
    try:
        lib.avirb200_plan_set_option.argtypes = [C.c_void_p, C.c_int, C.c_int]
        assert lib.avirb200_plan_set_option(plan, ab.OPT_OVERLAP_HALO, overlap) == 0
        total = 0
        for r in range(nranks):
            b = C.c_size_t()
            assert lib.avirb200_shard_workspace_bytes(plan, r, nranks, C.byref(b)) == 0, lib.avirb200_last_error()
            total += b.value
        d_src = torch.from_numpy(src).cuda()
        tmap = {np.uint8: torch.uint8, np.uint16: torch.uint16, np.float32: torch.float32}
        d_dst = torch.zeros(nh * nw * ch * np.dtype(to).itemsize, dtype=torch.uint8, device="cuda").view(tmap[to]).reshape(nh, nw, ch)
        d_ws = torch.empty(total, dtype=torch.uint8, device="cuda")
        lib.avirb200_resize_sharded_local.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_size_t,
                                                      C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p]
        for _ in range(2):  # (a second call: counters and flags start from what the first left)
            assert lib.avirb200_resize_sharded_local(plan, nranks, d_src.data_ptr(), sw * ch, d_dst.data_ptr(),
                                                     nw * ch, d_ws.data_ptr(), None) == 0, lib.avirb200_last_error()
            torch.cuda.synchronize()
        got = d_dst.cpu().numpy()
    finally:
        lib.avirb200_plan_destroy(plan)
        rs.free_descriptor(h)
    assert cs.count_mismatch(whole, got) == 0


def test_lin2srgb_batch_is_exhaustively_bit_identical():
    """The streaming column pass applies the output gamma to a lane's whole batch with the library
    square root's fast path written out (so that the samples' chains interleave).  The library's
    self-test compares it with the one-sample path on every float bit pattern it accepts."""
    lib = ab.lib()
    lib.avirb200_selftest_lin2srgb.argtypes = [C.POINTER(C.c_ulonglong), C.POINTER(C.c_ulonglong)]
    checked, bad = C.c_ulonglong(), C.c_ulonglong()
    assert lib.avirb200_selftest_lin2srgb(C.byref(checked), C.byref(bad)) == 0, lib.avirb200_last_error()
    # everything below 3.0e38 (positive patterns up to it, all negative non-NaN patterns incl. -inf)
    assert checked.value > (1 << 32) - (1 << 25), checked.value
    assert bad.value == 0, "%d of %d float patterns differ" % (bad.value, checked.value)


# ---- LANCIR ---------------------------------------------------------------------------------

LANCIR = [
    (96, 54, 48, 27, np.uint8, np.uint8, {}),
    (64, 48, 103, 77, np.uint8, np.uint8, {}),
    (64, 64, 16, 16, np.uint16, np.uint16, {}),
    (60, 40, 40, 27, np.uint8, np.uint16, {}),
    (50, 30, 33, 17, np.float32, np.float32, {}),
    (50, 30, 33, 17, np.float32, np.uint8, {}),
    (50, 30, 70, 45, np.uint8, np.float32, {"kx": 0.7, "ky": -0.66, "ox": 0.25, "oy": 0.1}),
    (640, 480, 1024, 768, np.uint8, np.uint8, {}),       # BASELINE cfg1 geometry (RGBA)
    (1920, 1080, 960, 540, np.uint8, np.uint8, {}),
    # 1-3 channel images: upstream's resize1/resize2/resize3 summation trees
    (640, 480, 1024, 768, np.uint8, np.uint8, {"C": 3}),     # BASELINE cfg1 as quoted (RGB)
    (640, 480, 1024, 768, np.uint8, np.uint8, {"C": 1}),
    (640, 480, 1024, 768, np.uint16, np.uint16, {"C": 2}),
    (64, 48, 103, 77, np.float32, np.float32, {"C": 3, "la": 4.0}),
    (96, 54, 48, 27, np.uint16, np.uint16, {"C": 3}),
    (96, 54, 48, 27, np.float32, np.float32, {"C": 2}),
    (96, 54, 48, 27, np.uint8, np.float32, {"C": 1}),
    (77, 51, 50, 31, np.float32, np.float32, {"C": 3, "la": 2.0}),
    (77, 51, 47, 29, np.float32, np.float32, {"C": 1, "la": 3.0, "kx": 1.3, "ky": 2.2}),
    (77, 51, 47, 29, np.float32, np.float32, {"C": 2, "la": 3.0, "kx": 1.3, "ky": 2.2}),
    (77, 51, 47, 29, np.float32, np.float32, {"C": 3, "la": 3.0, "kx": 1.3, "ky": 2.2}),
    (1920, 1080, 1280, 720, np.uint8, np.uint8, {"C": 3}),
    (33, 21, 7, 5, np.uint8, np.uint8, {"C": 3}),
]


def _lancir_upstream(src, nw, nh, to, kw):
    def run():
        r, ref = o.lancir_ref(src, nw, nh, to, **kw)
        assert r == nh
        return ref
    return cs.upstream(cs.lancir_key(src, nw, nh, to, kw), run)


@pytest.mark.parametrize("sw,sh,nw,nh,ti,to,kw", LANCIR)
def test_lancir_bit_exact(sw, sh, nw, nh, ti, to, kw):
    kw = dict(kw)
    src = o.lcg_image(sh, sw, kw.pop("C", 4), ti, seed=3)
    r, got = ab.CLancIR().resizeImage(src, nw, nh, ab.CLancIRParams(**kw), out_dtype=to)
    assert r == nh
    assert cs.digest(got) == _lancir_upstream(src, nw, nh, to, kw)


def test_lancir_golden_fixtures():
    files = sorted(f for f in os.listdir(cs.GOLDEN) if f.startswith("lancir_"))
    assert files
    for f in files:
        z = np.load(os.path.join(cs.GOLDEN, f))
        sw, sh, nw, nh = [int(v) for v in z["geom"]]
        r, got = ab.CLancIR().resizeImage(z["src"], nw, nh, out_dtype=z["out"].dtype)
        assert r == nh and cs.count_mismatch(z["out"], got) == 0, f


# ---- float sources that need the input linearisation, 4 channels ---------------------------------
# (found by the sweep below: the tile kernel's row pass streams float sources as they are and used
# to skip the sRGB linearisation; such calls now take the generic row pass)

@pytest.mark.parametrize("case", [
    (3, 84, 95, 168, 190, 4, np.float32, np.uint8, 4, {"gamma": True, "alpha": 3}),
    (2, 109, 62, 205, 190, 4, np.float64, np.float64, 8, {"gamma": True, "k": 3.0}),
    (1, 192, 108, 96, 54, 4, np.float32, np.float32, 16, {"gamma": True, "alpha": 0}),
    (2, 192, 108, 96, 54, 4, np.float32, np.uint16, 16, {"gamma": True, "buildmode": 1}),
], ids=cs.case_id)
def test_float_source_with_input_gamma_4ch(case, kernel_path):
    src = cs.make_input(case, seed=41)
    got = cs.gpu_output(case, src)
    assert cs.matches_upstream(case, src, got)


# ---- seeded random sweep over the whole call surface (same generator as the oracle's own) ------

@pytest.mark.parametrize("seed", [13, 11, 12])
def test_fuzz_product_matches_oracle(seed):
    """All six classes, 1..4 channels, every Tin/Tout pair incl. double, bit depths, gamma / alpha,
    offsets, explicit and negative k, presets, forced build modes, odd ratios: product path
    (kernel family chosen by the engine) against the oracle, 0 mismatching elements."""
    rng = np.random.default_rng(seed)
    types = [np.uint8, np.uint16, np.float32, np.float64]
    for it in range(40):
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
        got = cs.gpu_output(case, src)
        assert cs.matches_upstream(case, src, got), cs.case_id(case)


def test_lancir_fuzz_product_matches_oracle():
    """Seeded random sweep of CLancIR on the GPU: 1..4 channels, la = 2 .. 5, both scaling
    directions, offsets, explicit steps, every u8 / u16 / float type pair, against upstream."""
    rng = np.random.default_rng(17)
    types = [np.uint8, np.uint16, np.float32]
    for it in range(60):
        ch = int(rng.integers(1, 5))
        sw, sh = int(rng.integers(2, 120)), int(rng.integers(2, 120))
        nw, nh = int(rng.integers(1, 200)), int(rng.integers(1, 200))
        ti, to = types[int(rng.integers(0, 3))], types[int(rng.integers(0, 3))]
        kw = {"la": float(rng.choice([2.0, 2.5, 3.0, 4.0, 5.0]))}
        if rng.random() < 0.3:
            kw["kx"], kw["ky"] = float(rng.choice([0.5, 0.8, 1.7, -1.3])), float(rng.choice([0.6, 1.0, 2.2, -0.9]))
        if rng.random() < 0.3:
            kw["ox"], kw["oy"] = float(rng.uniform(-1, 1)), float(rng.uniform(-1, 1))
        src = o.lcg_image(sh, sw, ch, ti, seed=900 + it)
        r, got = ab.CLancIR().resizeImage(src, nw, nh, ab.CLancIRParams(**kw), out_dtype=to)
        assert r == nh
        assert cs.digest(got) == _lancir_upstream(src, nw, nh, to, kw), (sw, sh, nw, nh, ch, ti, to, kw)
