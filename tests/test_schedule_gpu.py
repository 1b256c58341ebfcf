"""The persistent kernels on long static tile schedules, under SM limits, against the fp64 references of tests/ref64.py.

Every persistent kernel walks tile ``blockIdx.x + i * gridDim.x`` (per cluster for the CTA-pair kernels) and carries
ring slots, barrier phases, TMEM accumulator stages and (in the ResBlock pair) input buffers and a weight ring from one
tile to the next.  ``as_set_sm_limit(n)`` sizes every grid for ``max(2, min(n, SMs) & ~1)`` SMs, so at a small limit
each CTA walks many tiles of a small problem.  Each case runs at no limit, 2, 7 (-> 6), 40 and 148 - 40 (the engine's
split) and checks:

  (a) the unlimited run against the reference, element by element;
  (b) every limited run bitwise against the unlimited one: kernel choice does not depend on the SM count and every tile
      is computed whole, in a fixed K order, by one CTA or CTA pair;
  (c) rows beyond ``lens`` are exact zeros (part of (a): the bound is 0 there).

The profiler names the template instantiation that ran and its grid.  The ``lens`` vector is the same in every case, so
dead and live tiles alternate within one CTA's schedule.  ``conv_halo_kernel`` is absent: it needs CinP == Cin <= 32,
i.e. Cin = 32 (16 goes to conv_cout1 or conv_small), and every such shape is taken first by ``conv_halo_sw_kernel``
(halo_sw_eligible accepts Cin = 32 for the same tile widths); the product census below confirms it never runs.
"""
import contextlib
import json
import re
import zlib

import pytest
import torch

from artspeech_b200 import _lib, ops
from tests import ref64

pytestmark = pytest.mark.gpu
DEV = "cuda"
N_SM = 148
LIMITS = (0, 2, 7, 40, N_SM - 40)
# CTAs a kernel may keep resident per SM (grid <= PER_SM * n')
PER_SM = {"conv_igemm_kernel": 2, "conv_halo_sw_kernel": 2, "conv_halo_kernel": 2, "conv_igemm_2cta_kernel": 1,
          "resblock_pair_kernel": 1, "resblock_pair2_kernel": 1, "adain_ring_kernel": 1}
PERSISTENT = tuple(PER_SM)


def _limited(n):
    return N_SM if n == 0 else max(2, min(n, N_SM) & ~1)


def _lens(T, extra_full=False):
    """T, 1, 127, 128, 129, T - 1, ceil(T / 3), 0 (clamped to T); one more full item gives odd M-tile counts."""
    v = [T, 1, 127, 128, 129, T - 1, -(-T // 3), 0] + ([T] if extra_full else [])
    return torch.tensor([min(x, T) for x in v], dtype=torch.int32)


@pytest.fixture
def sm_limit():
    """``with sm_limit(n):`` runs a block with persistent grids sized for n SMs; the process-wide setting is restored
    afterwards, also when the test fails."""
    lib = _lib.load()
    prev = lib.as_set_sm_limit(0)
    lib.as_set_sm_limit(prev)

    @contextlib.contextmanager
    def limit(n):
        old = lib.as_set_sm_limit(n)
        try:
            yield
        finally:
            lib.as_set_sm_limit(old)
    try:
        yield limit
    finally:
        lib.as_set_sm_limit(prev)


def kernel_name(name):
    """'void asb::conv_igemm_kernel<128, 64, false>(CUtensorMap, ...)' -> 'conv_igemm_kernel<128, 64, false>'."""
    m = re.search(r"(\w+_kernel)(?=[<(])", name)
    if m is None:
        return name
    out, i = m.group(1), m.end()
    if i < len(name) and name[i] == "<":
        depth, j = 0, i
        while j < len(name):
            depth += {"<": 1, ">": -1}.get(name[j], 0)
            j += 1
            if depth == 0:
                break
        out += re.sub(r"\s+", " ", name[i:j].replace("asb::", ""))
    return out


def launches(fn, tmp_path, tag):
    """Run ``fn`` under torch.profiler (CUDA activity), export the chrome trace to tmp_path and return its result and
    the (kernel name, grid) of every kernel it launched."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        res = fn()
        torch.cuda.synchronize()
    path = tmp_path / f"{tag}.json"
    prof.export_chrome_trace(str(path))
    with open(path) as f:
        ev = json.load(f)["traceEvents"]
    ks = [(kernel_name(e["name"]), tuple(e["args"].get("grid", (0, 0, 0)))) for e in ev if e.get("cat") == "kernel"]
    return res, ks


def sweep(fn, sm_limit, tmp_path, tag, kernel, work, per_cluster=False, min_per_cta=4):
    """Run ``fn`` (returns a tuple of output tensors) at every limit.  Asserts the one persistent launch is ``kernel``
    with grid <= PER_SM * n', at least ``min_per_cta`` work units (tiles, super-tiles, units) per CTA or per cluster at
    limit 2, and every limited output bitwise equal to the unlimited one.  Returns the unlimited outputs and a
    description of the schedule at limit 2."""
    base = kernel.split("<")[0]
    first, desc = None, ""
    for n in LIMITS:
        with sm_limit(n):
            outs, ks = launches(lambda: tuple(t.clone() for t in fn()), tmp_path, f"{tag}_{n}")
        pers = [k for k in ks if k[0].split("<")[0] in PERSISTENT]
        assert [k[0] for k in pers] == [kernel], f"{tag} limit {n}: launched {ks}, expected {kernel}"
        grid = pers[0][1][0]
        assert grid <= PER_SM[base] * _limited(n), f"{tag} limit {n}: grid {grid} over {PER_SM[base]} x {_limited(n)}"
        if n == 2:
            units = grid // 2 if per_cluster else grid
            per = work / units
            desc = f"{kernel} grid {grid}: {per:.1f} work units per {'cluster' if per_cluster else 'CTA'}"
            assert per >= min_per_cta, f"{tag}: only {desc} at limit 2"
        if first is None:
            first = outs
            continue
        for i, (a, b) in enumerate(zip(first, outs)):
            if not torch.equal(a.view(torch.uint8) if a.is_floating_point() else a,
                               b.view(torch.uint8) if b.is_floating_point() else b):
                d = (a.float() - b.float()).abs()
                idx = tuple(int(j) for j in torch.unravel_index(d.argmax().cpu(), d.shape))
                raise AssertionError(f"{tag}: output {i} at limit {n} differs from the unlimited run; first worst "
                                     f"index {idx}: {float(a[idx])} vs {float(b[idx])}")
    print(f"[schedule] {tag}: {desc}")
    return first, desc


DTS = [torch.float16, torch.bfloat16]


# ------------------------------------------------------------------------------------------------------------------
# as_conv_igemm: 1-CTA kernel (BN x BK), 2-D, halo-sw, CTA pairs; every epilogue
# ------------------------------------------------------------------------------------------------------------------
def _bf(dt):
    return "true" if dt == torch.bfloat16 else "false"


# name: (Cin, Cout, k, dil, T, F, epilogue, odd M-tile count, expected instantiation for a dtype)
CONV_CASES = {
    # Cin 48 (not a halo width), Cout 64: BN 64, BK 32; fp32 raw + 16-bit act, res1 16-bit + res2 fp32: direct fast
    "igemm_bn64_bk32_fast": (48, 64, 5, 2, 600, 1, "fast", False, lambda d: f"conv_igemm_kernel<64, 32, {_bf(d)}>"),
    # Cout 384 = 3 x 128 (CoutP > bn), BK 64, all-16-bit outputs and residual: the 16-bit TMA epilogue
    "igemm_bn128_bk64_tma16": (96, 384, 3, 1, 500, 1, "tma16", False, lambda d: f"conv_igemm_kernel<128, 64, {_bf(d)}>"),
    # Cin 32 -> BK 32 (no CTA pair), Cout 512 with > 74 tiles keeps BN 256; fp32 residual / raw: the fp32 TMA epilogue
    "igemm_bn256_bk32_tma32": (32, 512, 3, 1, 700, 1, "tma32", False, lambda d: f"conv_igemm_kernel<256, 32, {_bf(d)}>"),
    # mixed-dtype residual (the other 16-bit format), Cout 120 (partial 16-channel chunk), strided raw output: slow path
    "igemm_bn128_bk64_slow": (80, 120, 3, 1, 400, 1, "slow", False, lambda d: f"conv_igemm_kernel<128, 64, {_bf(d)}>"),
    # 2-D 3 x 3 over F = 80: tF = 16, tT = 8
    "igemm_2d_3x3": (64, 64, 3, 1, 40, 80, "fast2d", False, lambda d: f"conv_igemm_kernel<64, 64, {_bf(d)}>"),
    "halo_sw_bkc32_tma16": (32, 32, 7, 1, 1000, 1, "tma16", False, lambda d: f"conv_halo_sw_kernel<32, 32, {_bf(d)}>"),
    "halo_sw_bkc64_fast": (64, 64, 11, 5, 700, 1, "fast", False, lambda d: f"conv_halo_sw_kernel<64, 64, {_bf(d)}>"),
    # Cin 128 / Cout 128 and Cin 64 / Cout 16 (the product's widest and narrowest halo tiles); Cout 8, Cin 192: BN 16
    "halo_sw_bn128_bkc64_fast": (128, 128, 3, 1, 1000, 1, "fast", False,
                                 lambda d: f"conv_halo_sw_kernel<128, 64, {_bf(d)}>"),
    "halo_sw_bn16_bkc64_fast": (64, 16, 5, 1, 900, 1, "fast", False, lambda d: f"conv_halo_sw_kernel<16, 64, {_bf(d)}>"),
    "igemm_bn16_bk64_fast": (192, 8, 3, 1, 600, 1, "fast", False, lambda d: f"conv_igemm_kernel<16, 64, {_bf(d)}>"),
    # 256-wide tiles, BK 64, odd M-tile count (the padding tile lands at the end of a long schedule)
    "igemm_2cta_tma32": (256, 512, 3, 1, 600, 1, "tma32", True, lambda d: f"conv_igemm_2cta_kernel<64, {_bf(d)}>"),
}


def _conv_work(Cin, Cout, T, F, B, kernel):
    bn = ops.conv_tile_n(Cout)
    coutp = (Cout + bn - 1) // bn * bn
    tF = 1
    while tF < 128 and F % (tF * 2) == 0:
        tF *= 2
    m = B * -(-T // (128 // tF)) * -(-F // tF)
    if "2cta" in kernel:
        return -(-m // 2) * (coutp // 256), True, 8
    if "halo" in kernel:
        return m, False, 4
    return m * (coutp // bn), False, 4


@pytest.mark.parametrize("dt", DTS)
@pytest.mark.parametrize("case", list(CONV_CASES))
def test_conv_schedule(case, dt, sm_limit, tmp_path):
    Cin, Cout, k, dil, T, F, epi, odd, kern = CONV_CASES[case]
    kernel = kern(dt)
    lens = _lens(T, extra_full=odd)
    B = len(lens)
    g = torch.Generator().manual_seed(zlib.crc32(case.encode()))
    xs = (B, T, Cin) if F == 1 else (B, T, F, Cin)
    os_ = (B, T, Cout) if F == 1 else (B, T, F, Cout)
    x = (torch.randn(*xs, generator=g) * 0.5).to(dt)
    w = (torch.randn(k * (k if F > 1 else 1), Cout, Cin, generator=g) / (Cin * k) ** 0.5).to(dt)
    taps = ops.taps_1d(k, dil) if F == 1 else ops.taps_2d(k, k, k // 2, k // 2)
    bias = torch.randn(Cout, generator=g)
    other = torch.bfloat16 if dt == torch.float16 else torch.float16
    res1 = res2 = None
    outs = []                                      # (name, dtype, act, slope, channel offset, buffer width)
    if epi in ("fast", "fast2d"):
        res1 = torch.randn(*os_, generator=g).to(dt) if epi == "fast" else None
        res2 = torch.randn(*os_, generator=g) if epi == "fast" else None
        outs = [("raw", torch.float32, ops.ACT_NONE, 0.0, 0, Cout), ("act", dt, ops.ACT_LRELU, 0.2, 0, Cout)]
    elif epi == "tma16":
        res1 = torch.randn(*os_, generator=g).to(dt)
        outs = [("raw", dt, ops.ACT_NONE, 0.0, 0, Cout), ("act", dt, ops.ACT_LRELU, 0.1, 8, Cout + 24)]
    elif epi == "tma32":
        res1 = torch.randn(*os_, generator=g)
        outs = [("raw", torch.float32, ops.ACT_NONE, 0.0, 8, Cout + 16), ("act", dt, ops.ACT_LRELU, 0.2, 16, Cout + 32)]
    elif epi == "slow":
        res1 = torch.randn(*os_, generator=g).to(other)
        outs = [("raw", torch.float32, ops.ACT_NONE, 0.0, 4, Cout + 12), ("act", dt, ops.ACT_TANH, 0.0, 0, Cout)]
    scale = 0.7
    pw = ops.pack_conv(w.float(), bias, taps, dt, DEV)
    xg, lg = x.to(DEV), lens.to(DEV)
    r1g = None if res1 is None else res1.to(DEV)
    r2g = None if res2 is None else res2.to(DEV)
    act, slope = [(o[2], o[3]) for o in outs if o[0] == "act"][0]

    def run():
        bufs = {}
        for name, odt, _, _, off, width in outs:
            bufs[name] = torch.full(os_[:-1] + (width,), 7.0, dtype=odt, device=DEV)
        view = {o[0]: bufs[o[0]][..., o[4]:o[4] + Cout] for o in outs}
        ops.conv(xg, pw, res1=r1g, res2=r2g, scale=scale, raw=view["raw"], act_out=view["act"], act=act,
                 slope=slope, lens=lg)
        return tuple(bufs[o[0]] for o in outs)

    work, per_cluster, min_per = _conv_work(Cin, Cout, T, F, B, kernel)
    res, _ = sweep(run, sm_limit, tmp_path, f"{case}_{dt}", kernel, work, per_cluster, min_per)
    vb = ref64.conv_v(x, w, taps, bias=bias, res1=res1, res2=res2, scale=scale, lens=lens)
    for (name, odt, a, s, off, width), buf in zip(outs, res):
        got = buf[..., off:off + Cout]
        ref, bound = ref64.conv_out(vb, a, s, odt)
        ref64.check(got, ref, bound, f"{case} {dt} {name}", 128 // (16 if F > 1 else 1), ops.conv_tile_n(Cout))
        # neighbouring channels of a channel-slice output stay untouched
        assert bool((buf[..., :off] == 7).all()) and bool((buf[..., off + Cout:] == 7).all()), f"{case} {name}"


# ------------------------------------------------------------------------------------------------------------------
# as_hifigan_resblock_pair: 1-CTA and CTA-pair kernels, C x k, every variant
# ------------------------------------------------------------------------------------------------------------------
PAIR_CASES = [(C, k) for C in (32, 64, 128) for k in (3, 7, 11)]
VARIANTS = ("mid", "branch_end", "stage_end")
# the shared-memory plan as_hifigan_resblock_pair picks (ASB_PAIR_VERBOSE=1): (2cta, NX, NT, SW, pipelined)
EXPECTED_PLANS = {(32, 3): (0, 6, 2, 0, 1), (32, 7): (0, 6, 2, 0, 1), (32, 11): (0, 6, 2, 0, 1),
                  (64, 3): (0, 2, 2, 0, 1), (64, 7): (1, 2, 2, 0, 1), (64, 11): (1, 2, 2, 4, 1),
                  (128, 3): (0, 2, 0, 3, 0), (128, 7): (1, 1, 1, 7, 0), (128, 11): (1, 1, 1, 7, 0)}


@pytest.mark.parametrize("dt", DTS)
@pytest.mark.parametrize("C,k", PAIR_CASES)
def test_resblock_pair_schedule(C, k, dt, sm_limit, tmp_path, monkeypatch, capfd):
    variant = VARIANTS[PAIR_CASES.index((C, k)) % 3]
    dil = {3: 5, 7: 3, 11: 1}[k]
    L = 600                                          # 3 tiles per item: odd tile counts with 9 items
    lens = _lens(L, extra_full=True)
    B = len(lens)
    g = torch.Generator().manual_seed(C * 100 + k)
    x_raw = torch.randn(B, L, C, generator=g) * (torch.arange(L)[None, :] < lens[:, None])[:, :, None]
    slope = 0.1
    xa = torch.where(x_raw > 0, x_raw, slope * x_raw).to(dt)
    w1 = (torch.randn(k, C, C, generator=g) / (C * k) ** 0.5).to(dt)
    w2 = (torch.randn(k, C, C, generator=g) / (C * k) ** 0.5).to(dt)
    b1, b2 = torch.randn(C, generator=g) * 0.1, torch.randn(C, generator=g) * 0.1
    kw = dict(slope=slope)
    if variant == "mid":
        kw.update(out_act=ops.ACT_LRELU, out_slope=slope)
    elif variant == "stage_end":
        kw.update(res2=torch.randn(B, L, C, generator=g).to(dt), res3=torch.randn(B, L, C, generator=g).to(dt),
                  scale=1.0 / 3, out_act=ops.ACT_LRELU, out_slope=0.01)
    c1 = ops.pack_conv(w1.float(), b1, ops.taps_1d(k, dil), dt, DEV)
    c2 = ops.pack_conv(w2.float(), b2, ops.taps_1d(k, 1), dt, DEV)
    kwg = {n: (v.to(DEV) if torch.is_tensor(v) else v) for n, v in kw.items()}
    xg, lg = xa.to(DEV), lens.to(DEV)
    pair = C >= 64 and k >= 7                        # the product rule
    tiles = B * -(-L // (256 - (k - 1)))
    assert tiles % 2 == 1
    kernel = f"resblock_pair{'2' if pair else ''}_kernel<{C}, {_bf(dt)}>"
    monkeypatch.setenv("ASB_PAIR_VERBOSE", "1")
    capfd.readouterr()
    res, desc = sweep(lambda: (ops.resblock_pair(xg, c1, c2, k, dil, lens=lg, **kwg),), sm_limit, tmp_path,
                      f"pair_{C}_{k}_{dt}", kernel, -(-tiles // 2) if pair else tiles, pair, 6 if pair else 4)
    plans = set(re.findall(r"2cta=(\d) NX=(\d+) NT=(\d) ND=(\d) NSTG=(\d) SW=(\d+) stream=\d\d pipelined=(\d)",
                           capfd.readouterr().err))
    assert len(plans) == 1, f"plan depends on the SM limit or is missing: {plans}"
    two, nx, nt, nd, _, sw, pipe = (int(v) for v in plans.pop())
    assert two == int(pair) and nd == (2 if C <= 64 else 1)
    assert pipe == int(nd == 2 and nx >= 2) and (nt >= 1 if pair else True)
    assert (two, nx, nt, sw, pipe) == EXPECTED_PLANS[(C, k)], (two, nx, nt, sw, pipe)
    print(f"[schedule] pair C={C} k={k} {dt} {variant}: 2cta={two} NX={nx} NT={nt} SW={sw} pipelined={pipe}; {desc}")
    ref, bound = ref64.resblock_pair(xa, w1, b1, w2, b2, k, dil, lens=lens, **kw)
    ref64.check(res[0], ref, bound, f"pair C={C} k={k} {dt} {variant}", 256 - (k - 1), C)


def test_resblock_pair_plans_cover_deep_rings():
    """The table above reaches input rings of 3+ buffers with the pipelined issue order (at 13.5 tiles per CTA at
    limit 2: 27 tiles, asserted >= 6 by each case)."""
    assert any(p[1] >= 3 and p[4] == 1 for p in EXPECTED_PLANS.values()), EXPECTED_PLANS


# ------------------------------------------------------------------------------------------------------------------
# adain_ring_kernel: fp32 input up to ~1650 frames, W = 32 / 16, pool or not, MX or not
# ------------------------------------------------------------------------------------------------------------------
def _adain_inputs(B, T, C, dt, seed, up, lens=None):
    g = torch.Generator().manual_seed(seed)
    # bias-dominated channels: |mean| / std = 40
    x = (torch.randn(B, T, C, generator=g) * 0.5 + 20.0 * torch.sign(torch.randn(C, generator=g))).to(dt)
    gb = torch.randn(B, 2 * C, generator=g) * 0.3
    up_w = torch.randn(C, 3, generator=g) if up else None
    up_b = torch.randn(C, generator=g) if up else None
    return x, gb, up_w, up_b


RING_CASES = {"w32": (800, False, 0.2, 32), "w32_pool": (800, True, 0.2, 32), "w16": (1200, False, 0.2, 16),
              "w16_pool_slope1.5": (1200, True, 1.5, 16), "w32_slope-0.3": (600, False, -0.3, 32)}


@pytest.mark.parametrize("out_dt", DTS)
@pytest.mark.parametrize("case", list(RING_CASES))
def test_adain_ring_schedule(case, out_dt, sm_limit, tmp_path):
    T, up, slope, W = RING_CASES[case]
    C = 512
    lens = _lens(T)
    B = len(lens)
    x, gb, up_w, up_b = _adain_inputs(B, T, C, torch.float32, 11, up)
    xg, gbg, lg = x.to(DEV), gb.to(DEV), lens.to(DEV)
    wg = None if up_w is None else up_w.to(DEV).contiguous()
    bg = None if up_b is None else up_b.to(DEV)
    mx = "true" if 0 <= slope <= 1 else "false"
    kernel = f"adain_ring_kernel<{'true' if up else 'false'}, {mx}, {W}>"
    res, _ = sweep(lambda: (ops.adain_norm(xg, gbg, slope, lg, out_dt, wg, bg),), sm_limit, tmp_path,
                   f"ring_{case}_{out_dt}", kernel, B * C // W)
    ref, bound = ref64.adain_norm(x, gb, slope, lens, out_dt, up_w, up_b)
    ref64.check(res[0], ref, bound, f"ring {case} {out_dt}", 2 * T if up else T, W)


# ------------------------------------------------------------------------------------------------------------------
# as_adain_norm_apply dispatch: cluster kernel, two-pass fallback; as_adain_apply scalar path; as_instnorm_stats
# ------------------------------------------------------------------------------------------------------------------
def _kernels_of(fn, tmp_path, tag):
    res, ks = launches(fn, tmp_path, tag)
    return res, [k[0] for k in ks]


@pytest.mark.parametrize("up", [False, True])
@pytest.mark.parametrize("x_dt", [torch.float16, torch.bfloat16, torch.float32])
@pytest.mark.parametrize("T", [1761, 3000, 6144])
def test_adain_cluster_kernel(T, x_dt, up, tmp_path):
    C = 96
    TR = (-(-T // 4) + 31) // 32 * 32
    lens = torch.tensor([T, TR - 5, 1, 0, TR + 1], dtype=torch.int32)   # trailing cluster CTAs with no valid rows
    x, gb, up_w, up_b = _adain_inputs(len(lens), T, C, x_dt, T + 7, up)
    out_dt = torch.float16 if x_dt == torch.float32 else x_dt
    wg = None if up_w is None else up_w.to(DEV).contiguous()
    bg = None if up_b is None else up_b.to(DEV)
    out, ks = _kernels_of(lambda: ops.adain_norm(x.to(DEV), gb.to(DEV), 0.2, lens.to(DEV), out_dt, wg, bg), tmp_path,
                          "cluster")
    xdt = {torch.float16: 0, torch.bfloat16: 1, torch.float32: 2}[x_dt]
    assert ks == [f"adain_fused_kernel<{'true' if up else 'false'}, {xdt}>"], ks
    ref64.check(out, *ref64.adain_norm(x, gb, 0.2, lens, out_dt, up_w, up_b), f"cluster T={T} {x_dt} up={up}", TR, 32)


@pytest.mark.parametrize("x_dt", [torch.float32, torch.float16])
@pytest.mark.parametrize("T", [6145, 9600])
def test_adain_two_pass_fallback(T, x_dt, tmp_path):
    C, up = 64, T == 9600
    lens = torch.tensor([T, T // 3, 1, 0], dtype=torch.int32)
    x, gb, up_w, up_b = _adain_inputs(len(lens), T, C, x_dt, T, up)
    wg = None if up_w is None else up_w.to(DEV).contiguous()
    bg = None if up_b is None else up_b.to(DEV)
    out, ks = _kernels_of(lambda: ops.adain_norm(x.to(DEV), gb.to(DEV), 0.2, lens.to(DEV), torch.float32, wg, bg),
                          tmp_path, "two_pass")
    assert ks == ["instnorm_stats_kernel", f"adain_apply_vec_kernel<{'true' if up else 'false'}>"], ks
    ref64.check(out, *ref64.adain_norm(x, gb, 0.2, lens, torch.float32, up_w, up_b), f"two-pass T={T} {x_dt}")


@pytest.mark.parametrize("up", [False, True])
def test_adain_apply_scalar_kernel(up, tmp_path):
    """C % 4 != 0 and a channel slice at an odd offset take the scalar kernel; it agrees with the reference and with
    the vector kernel on the same statistics."""
    T = 333
    lens = torch.tensor([T, 100, 1, 0], dtype=torch.int32)
    B = len(lens)
    for C, off in ((250, 0), (256, 2)):
        g = torch.Generator().manual_seed(C + off)
        wide = (torch.randn(B, T, C + 8, generator=g) * 2 + 1).half()
        x = wide[..., off:off + C]
        st = torch.rand(B, C, 2, generator=g) + torch.tensor([0.5, 0.2])
        gb = torch.randn(B, 2 * C, generator=g) * 0.3
        up_w = torch.randn(C, 3, generator=g) if up else None
        up_b = torch.randn(C, generator=g) if up else None
        wg = None if up_w is None else up_w.to(DEV).contiguous()
        bg = None if up_b is None else up_b.to(DEV)
        xg = wide.to(DEV)[..., off:off + C]
        args = (st.to(DEV), gb.to(DEV), 0.2, lens.to(DEV), torch.float32, wg, bg)
        out, ks = _kernels_of(lambda: ops.adain_apply(xg, *args), tmp_path, "scalar")
        assert ks == ["adain_apply_kernel"], ks
        ref, bound = ref64.adain_apply(x, st, gb, 0.2, lens, torch.float32, up_w, up_b)
        ref64.check(out, ref, bound, f"scalar C={C} offset {off}")
        if C % 4 == 0:
            xd = xg.contiguous()
            vec, ks = _kernels_of(lambda: ops.adain_apply(xd, *args), tmp_path, "vector")
            assert ks == [f"adain_apply_vec_kernel<{'true' if up else 'false'}>"], ks
            ref64.check(vec, ref, bound, f"vector C={C}")
            assert bool(((vec - out).abs().cpu().double() <= 2 * bound).all())


@pytest.mark.parametrize("x_dt", [torch.float32, torch.bfloat16])
def test_instnorm_stats_kernel(x_dt, tmp_path):
    T, C = 1500, 200
    lens = torch.tensor([T, 700, 1, 2, 0], dtype=torch.int32)
    x, _, _, _ = _adain_inputs(len(lens), T, C, x_dt, 5, False)
    st, ks = _kernels_of(lambda: ops.instnorm_stats(x.to(DEV), lens.to(DEV)), tmp_path, "stats")
    assert ks == ["instnorm_stats_kernel"], ks
    ref64.check(st, *ref64.instnorm_stats(x, lens), f"instnorm_stats {x_dt}")


# ------------------------------------------------------------------------------------------------------------------
# the product: census of persistent instantiations and the shipped SM split
# ------------------------------------------------------------------------------------------------------------------
# instantiations asserted by the cases above (kept as a constant so that a census failure names what is missing)
CASE_TABLE = sorted({CONV_CASES[c][8](d) for c in CONV_CASES for d in DTS} |
                    {f"resblock_pair{'2' if C >= 64 and k >= 7 else ''}_kernel<{C}, {_bf(d)}>"
                     for C, k in PAIR_CASES for d in DTS} |
                    {f"adain_ring_kernel<{'true' if c[1] else 'false'}, {'true' if 0 <= c[2] <= 1 else 'false'}, {c[3]}>"
                     for c in RING_CASES.values()})


@pytest.fixture(scope="module")
def product():
    import bench
    from tests import util
    model = util.acoustic_model(0)
    gen = util.generator(0)
    tok, tl, mel, ml, dur = bench.make_inputs(0)
    return model, gen, (tok, tl, mel, ml, dur)


def test_product_census(product, tmp_path):
    """Every persistent-kernel instantiation the product launches at the benchmark's shape (16 utterances x 150
    tokens, durations summing to 400) is one the case table asserts."""
    from artspeech_b200 import engine
    model, gen, (tok, tl, mel, ml, dur) = product
    syn = engine.Synthesizer(model, gen, device=DEV, use_cuda_graph=False)
    _, ks = launches(lambda: syn.synthesize(tok.to(DEV), tl, mel.to(DEV), ml, dur, predict_durations=True), tmp_path,
                     "census")
    census = sorted({k for k, _ in ks if k.split("<")[0] in PERSISTENT})
    print("[schedule] census:", census)
    assert census, "no persistent kernel in the product's trace"
    missing = sorted(set(census) - set(CASE_TABLE))
    assert not missing, f"persistent instantiations without a schedule case: {missing}"


def test_acoustic_sms_split_is_bitwise_invariant(product):
    """Synthesizer(acoustic_sms=40) sizes the acoustic model's grids for 40 SMs and the vocoder's for the rest while
    two batches are in flight; the outputs are bitwise those of the unsplit engine."""
    from artspeech_b200 import engine
    model, gen, (tok, tl, mel, ml, dur) = product
    outs = []
    for kw in (dict(acoustic_sms=40), {}):
        syn = engine.Synthesizer(model, gen, device=DEV, pipeline_depth=2, **kw)
        got = []
        for _ in range(2):                        # the second call replays the captured graphs
            wav, lens, m = syn.synthesize(tok.to(DEV), tl, mel.to(DEV), ml, dur, predict_durations=True)
            syn.join()
            torch.cuda.synchronize()
            got.append((wav.clone(), torch.as_tensor(lens).clone(), m.clone()))
        outs.append(got)
        assert _lib.load().as_set_sm_limit(0) == 0, "the engine left an SM limit behind"
    for (w1, l1, m1), (w2, l2, m2) in zip(*outs):
        assert torch.equal(l1.cpu(), l2.cpu())
        assert torch.equal(w1, w2) and torch.equal(m1, m2)
