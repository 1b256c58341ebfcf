"""The fp64 references of tests/ref64_seq.py on the CPU: fp32 models of the kernels fall inside their bounds, and
small injected faults -- the kind a tiling, indexing or length bug produces -- fall outside them."""
import pytest
import torch

from tests import ref64, ref64_seq, sim_backend as sim


def _fails(out, ref, bound, what):
    with pytest.raises(AssertionError):
        ref64.check(out, ref, bound, what)
    err = (out.double() - ref).abs()
    return float((err / bound.clamp(min=1e-300)).max())


# ------------------------------------------------------------------------------------------------------------------
# relpos attention
# ------------------------------------------------------------------------------------------------------------------
def _relpos_inputs(T, B=2, H=2, D=128, ek_scale=1.0, seed=0):
    g = torch.Generator().manual_seed(seed)
    qkv = torch.randn(B, T, 3 * H * D, generator=g)
    ek = torch.randn(9, D, generator=g) * D ** -0.5 * ek_scale
    ev = torch.randn(9, D, generator=g)
    return qkv, ek, ev


def _relpos32(qkv, ek, ev, window, H, lens, drop_row=None, drop_cross=False, ev_shift=False):
    """fp32 model of as_relpos_attention (sim_backend's arithmetic) with injectable faults: the rel-key term missing on
    query ``drop_row``; missing where the band crosses a 64-key tile boundary; E_v read one index too far."""
    B, T, C3 = qkv.shape
    HD = C3 // 3
    D = HD // H
    q, k, v = [t.reshape(B, T, H, D).transpose(1, 2) for t in qkv.float().split(HD, dim=-1)]
    nrel = 2 * window + 1
    ek, ev = ek.float()[:nrel], ev.float()
    out = torch.zeros(B, H, T, D)
    for b in range(B):
        L = min(int(lens[b]), T)
        if L == 0:
            continue
        s = q[b, :, :L] @ k[b, :, :L].transpose(-1, -2)
        qe = q[b, :, :L] @ ek.t()
        ii = torch.arange(L)
        for r in range(nrel):
            j = ii + r - window
            ok = (j >= 0) & (j < L)
            if drop_row is not None:
                ok &= ii != drop_row
            if drop_cross:
                ok &= (j // 64) == (ii // 64)
            s[:, ii[ok], j[ok]] += qe[:, ii[ok], r]
        p = torch.softmax(s / D ** 0.5, dim=-1)
        o = p @ v[b, :, :L]
        for r in range(nrel):
            j = ii + r - window
            ok = (j >= 0) & (j < L)
            e = ev[min(r + 1, 8)] if ev_shift else ev[r]
            o[:, ii[ok]] += p[:, ii[ok], j[ok]][..., None] * e
        out[b, :, :L] = o
    return out.transpose(1, 2).reshape(B, T, HD)


@pytest.mark.parametrize("window", [0, 1, 4])
def test_relpos_fp32_model_inside_bounds(window):
    T = 150
    qkv, ek, ev = _relpos_inputs(T)
    lens = torch.tensor([T, 65])
    nrel = 2 * window + 1
    got = sim.relpos_attention(qkv, ek[:nrel], ev[:nrel], window, 2, lens, torch.float32)
    ref64.check(got, *ref64_seq.relpos_attention(qkv, ek, ev, window, 2, lens, torch.float32, "fp32"), "relpos fp32")
    # the mma bound on the operands the tensor-core kernel sees (q, k, v, E_k rounded to fp16)
    got = sim.relpos_attention(qkv.half().float(), ek[:nrel].half().float(), ev[:nrel], window, 2, lens, torch.float32)
    ref64.check(got, *ref64_seq.relpos_attention(qkv, ek, ev, window, 2, lens, torch.float32, "mma"), "relpos mma")
    for dt in (torch.float16, torch.bfloat16):
        ref, bound = ref64_seq.relpos_attention(qkv, ek, ev, window, 2, lens, dt, "mma")
        ref64.check(got.to(dt), ref, bound, f"relpos mma {dt}")


def test_relpos_faults_fail():
    T, w = 928, 4
    lens = torch.tensor([T, 700])
    qkv, ek, ev = _relpos_inputs(T)
    ref, bound = ref64_seq.relpos_attention(qkv, ek, ev, w, 2, lens, torch.float32, "mma")
    ref64.check(_relpos32(qkv, ek, ev, w, 2, lens), ref, bound, "unfaulted")
    r_row = _fails(_relpos32(qkv, ek, ev, w, 2, lens, drop_row=517), ref, bound, "row")
    r_ev = _fails(_relpos32(qkv, ek, ev, w, 2, lens, ev_shift=True), ref, bound, "E_v shift")
    qkv8, ek8, ev8 = _relpos_inputs(T, ek_scale=8.0)          # band-dominated
    ref8, bound8 = ref64_seq.relpos_attention(qkv8, ek8, ev8, w, 2, lens, torch.float32, "mma")
    ref64.check(_relpos32(qkv8, ek8, ev8, w, 2, lens), ref8, bound8, "unfaulted, band-dominated")
    r_cross = _fails(_relpos32(qkv8, ek8, ev8, w, 2, lens, drop_cross=True), ref8, bound8, "tile crossing")
    print(f"[ref64_seq] relpos fault err/bound: row {r_row:.3g}, E_v shift {r_ev:.3g}, tile crossing {r_cross:.3g}")


# ------------------------------------------------------------------------------------------------------------------
# conformer attention
# ------------------------------------------------------------------------------------------------------------------
def _conformer_inputs(T, B=3, H=4, D=64, seed=1):
    g = torch.Generator().manual_seed(seed)
    qkv = torch.randn(B, T, 3 * H * D, generator=g)
    pos = torch.randn(T, H * D, generator=g)
    u, v = torch.randn(H, D, generator=g) * 0.3, torch.randn(H, D, generator=g) * 0.3
    HD = H * D
    return qkv[..., :HD], qkv[..., HD:2 * HD], qkv[..., 2 * HD:], pos, u, v


@pytest.mark.parametrize("T", [47, 130])
def test_conformer_fp32_model_inside_bounds(T):
    q, k, v, pos, u, vb = _conformer_inputs(T)
    lens = torch.tensor([T, min(48, T), 1])
    got = sim.conformer_attention(q, k, v, pos, u, vb, 4, lens, torch.float32)
    ref64.check(got, *ref64_seq.conformer_attention(q, k, v, pos, u, vb, 4, lens, torch.float32, "fp32"), "conf fp32")
    # the mma bound allows at least what the fp32 one does
    ref, bound = ref64_seq.conformer_attention(q, k, v, pos, u, vb, 4, lens, torch.float32, "mma")
    assert float(((ref - got.double()).abs() - bound).max()) < float(bound.max())


def test_conformer_shift_index_matches_view_shift():
    """ref64_seq.shift_index is the reference's pad / view / slice relative shift (sim_backend's form)."""
    for L in (1, 2, 5, 48, 49):
        M = torch.arange(L * L, dtype=torch.float64).reshape(1, L, L) + 1
        padded = torch.cat([M.new_zeros(1, L, 1), M], -1).reshape(1, L + 1, L)
        want = padded[:, 1:].reshape(1, L, L)
        row, col, live = ref64_seq.shift_index(L)
        Mp = torch.cat([M, M.new_zeros(1, 1, L)], 1)
        got = torch.where(live, Mp[:, row, col], torch.zeros((), dtype=torch.float64))
        # the view reads row a + 1 = L (zero padding in the product: q + v of a padded row) only as M[L] below
        assert torch.equal(got, want), L


def test_conformer_faults_fail():
    T = 240
    q, k, v, pos, u, vb = _conformer_inputs(T)
    lens = torch.tensor([T, 200, 97])
    for path in ("mma", "fp32"):
        ref, bound = ref64_seq.conformer_attention(q, k, v, pos, u, vb, 4, lens, torch.float32, path)
        # the shift taken over T instead of each item's own length: only the shorter items change
        bad, _ = ref64_seq.conformer_attention(q, k, v, pos, u, vb, 4, lens, torch.float32, path, shift_len=T)
        assert torch.equal(bad[0], ref[0])
        r = _fails(bad.float(), ref, bound, f"conformer shift over T ({path})")
        print(f"[ref64_seq] conformer {path}: shift over T err/bound {r:.3g}")


# ------------------------------------------------------------------------------------------------------------------
# LSTM
# ------------------------------------------------------------------------------------------------------------------
def test_lstm_onestep_inside_bounds():
    g = torch.Generator().manual_seed(3)
    xp = torch.randn(3, 41, 8 * 256, generator=g) * 3
    for dt in (torch.float32, torch.float16):
        ref64.check(sim.lstm_onestep(xp, 256, dt), *ref64_seq.lstm_onestep(xp, 256, dt), f"onestep {dt}")


def _lstm_inputs(B, T, H, w_scale=1.0, f_bias=0.0, seed=4):
    g = torch.Generator().manual_seed(seed)
    xp = torch.randn(B, T, 8 * H, generator=g)
    for d in range(2):
        xp[..., d * 4 * H + H:d * 4 * H + 2 * H] += f_bias
    whh = torch.randn(2, H, 4 * H, generator=g) * w_scale / H ** 0.5
    return xp, whh


def _swap_if(xp, H, unit):
    """Gate pre-activations with i and f exchanged on one unit of both directions (a gate-order bug)."""
    xs = xp.clone()
    for d in range(2):
        i, f = d * 4 * H + unit, d * 4 * H + H + unit
        xs[..., [i, f]] = xs[..., [f, i]]
    return xs


@pytest.mark.parametrize("H", [64, 128, 256])
def test_bilstm_model_inside_bounds_and_faults_fail(H, monkeypatch):
    T = 60
    lens = torch.tensor([T, 1, 37, 0, T])
    xp, whh = _lstm_inputs(len(lens), T, H)
    monkeypatch.setattr(sim, "EMULATE_FP16_RECURRENCE", True)
    ref, bound = ref64_seq.bilstm(xp, whh, H, lens, torch.float32)
    got = sim.bilstm(xp, whh, H, lens, torch.float32)
    ref64.check(got, ref, bound, f"bilstm H={H}")
    n = ref64_seq.bounded_steps(bound, lens, H)
    print(f"[ref64_seq] bilstm H={H}: bounded steps per direction {n}")
    assert min(n) >= 1
    # the reverse direction started at T - 1 instead of lens[b] - 1
    bad, _ = ref64_seq.bilstm(xp, whh, H, lens, torch.float32, reverse_at_T=True)
    r_rev = _fails(bad, ref, bound, "reverse from T - 1")
    # i and f swapped on one unit: the fp32 model with the gate pre-activations exchanged there
    xs = _swap_if(xp, H, 5)
    # the swapped gates' recurrent terms must swap as well: exchange the W_hh columns too
    ws = whh.clone()
    ws[..., [5, H + 5]] = ws[..., [H + 5, 5]]
    r_if = _fails(sim.bilstm(xs, ws, H, lens, torch.float32), ref, bound, "i / f swapped")
    print(f"[ref64_seq] bilstm H={H} fault err/bound: reverse from T - 1 {r_rev:.3g}, i/f swapped {r_if:.3g}")


@pytest.mark.parametrize("H", [64, 128, 256])
def test_bilstm_contractive_regime_bound_stays_finite(H):
    """Small W_hh (0.1 / sqrt(H)) and a forget gate biased low (-3): the derived bound stays under the cap for whole
    sequences, so the GPU test checks them per element end to end."""
    T = 300
    lens = torch.tensor([T, 150, 1])
    xp, whh = _lstm_inputs(len(lens), T, H, w_scale=0.1, f_bias=-3.0)
    ref, bound = ref64_seq.bilstm(xp, whh, H, lens, torch.float32)
    n = ref64_seq.bounded_steps(bound, lens, H)
    print(f"[ref64_seq] contractive H={H}: bounded steps {n}, max bound {float(bound[torch.isfinite(bound)].max()):.3g}")
    assert n == [T, T]
