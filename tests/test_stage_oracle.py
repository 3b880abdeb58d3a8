"""Stage-by-stage fp64 oracle of the fused joint loss (-m gpu).

`rnnt_b200_joint_loss_fwd` / `_bwd` chain seven kernels: tile table, weight conversion, joint GEMM F (activations,
lse, lp), lattice, coefficients (+ work list), joint GEMM G (gradient ring), then the dW and dh GEMMs.  After one call
every intermediate is still on the device (outputs, `hidden`, and the workspace regions of rnnt_b200_debug_ws_layout),
so each stage is checked here against an fp64 computation whose inputs are the previous stage's device output.  The
checks are per element, and each bound scales with that element's own sum of absolute terms.  A missing, duplicated or
misplaced cell, column or hidden unit therefore fails wherever that element's other terms do not swamp it; a norm over
the whole tensor would not see it.

Bounds (per element; "measured" = largest error / bound-scale over the case matrix on one NVIDIA B200, 1000 W limit):
  convert_weights     W16 = fp16(W), pad 0, bias2 = fp32(b log2 e), pad -1e30           exact
  activations h       |h - tanh(enc+pred)| <= 2^-10 |tanh| + 2^-24; pad columns 0      measured 2^-10.9 relative
  F epilogue lse, lp  |err| <= 2^-21 (A + |lse| + 4) + Vp/32 * 2^-24,  A = max_v sum_k |h W| + |b|    measured 0.06 of bound
  lattice             |err| <= 1e-5 |ref| + 1e-4 (alpha, beta), 1e-5 relative (costs)  measured 0.03 of bound
  coef                |err| <= (2^-21 + 2^-22 (|alpha| + |beta'| + |log Z| + |lp|)) |ref|  measured 0.05 of bound
  tile table, work list  exact; dropped half-tiles' gradients <= 2^-25 max|dcost|
  G ring              |err| <= 2^-10 (|softmax gamma| + one-hot terms) + 2^-23           measured 0.5 of bound
  dW, db              |err| <= 2^-17 sum |terms|                                         measured 0.04 of bound
  dh: d_enc, d_pred   |err| <= sum over cells of 2^-9 |dh| h^2 + 2^-18 sum_v |g W| / S + 2^-14 |dz|   measured 0.2 of bound
"""
import numpy as np
import pytest
import torch

from helpers import fused_raw, make_inputs, tile_rows, torch_reference, ws_views

pytestmark = pytest.mark.gpu

LOG2E = 1.4426950408889634
GRAD_SHIFT = 12                                   # kGradShift: max|dcost| * S in [2^11, 2^12)
SKIP_BELOW = 2.0 ** -25 * 2 ** (GRAD_SHIFT - 1)   # kSkipBelow, in S-scaled units
DW_C = 2.0 ** -17
REPORT = {}


def _note(stage, ratio):
    REPORT[stage] = max(REPORT.get(stage, 0.0), float(ratio))


def _check(stage, got, ref, bound):
    """Every element within its bound; records the largest err / bound."""
    got, ref, bound = got.double(), ref.double(), bound.double()
    err = (got - ref).abs()
    bad = ~(err <= bound)
    if bad.any():
        i = int(bad.flatten().nonzero()[0])
        pytest.fail(f"{stage}: {int(bad.sum())} of {bad.numel()} elements out of bound; first flat index {i}: "
                    f"got {got.flatten()[i].item()!r}, want {ref.flatten()[i].item()!r}, bound {bound.flatten()[i].item()!r}")
    _note(stage, (err / bound.clamp_min(1e-300)).max() if err.numel() else 0.0)


def _case_inputs(B, T, U, H, V, blank, T_len, U_len, seed, t_major):
    inp = make_inputs(B, T, U, H, V, seed=seed)
    bl = blank % V
    g = torch.Generator().manual_seed(seed + 1)
    tg = torch.randint(0, V - 1, (B, U), generator=g, dtype=torch.int32)
    inp["targets"] = (tg + (tg >= bl).int()).cuda()                 # non-blank classes only
    inp["T_len"] = torch.tensor(T_len, dtype=torch.int32, device="cuda")
    inp["U_len"] = torch.tensor(U_len, dtype=torch.int32, device="cuda")
    if t_major:                                                       # the (B,T,H) view of a dense (B,H,T) tensor
        inp["enc"] = inp["enc"].permute(0, 2, 1).contiguous().permute(0, 2, 1)
    return inp


def _rows_dev(rows):
    a = torch.tensor([(b, t, u, int(v)) for b, t, u, v in rows], dtype=torch.long, device="cuda").view(-1, 4)
    return a[:, 0], a[:, 1], a[:, 2], a[:, 3].bool()


def check_stages(inp, out, blank, dcost, clamp, flags):
    """Checks every stage of one fused_raw call (single-chunk ring) against fp64; returns the fp64 dW / db / d_enc /
    d_pred references and their bounds, for comparing other runs of the same inputs."""
    enc, pred, W, bias = inp["enc"], inp["pred"], inp["W"], inp["b"]
    B, T, H = enc.shape
    U1, V = pred.shape[1], W.shape[0]
    bl = blank % V
    Tl, Ul = inp["T_len"].tolist(), inp["U_len"].tolist()
    v = ws_views(out)
    Hp, Vp, S = out["Hp"], out["Vp"], v["S"]
    assert out["status"] == 0

    # ---- convert_weights: exact
    W16, bias2 = v["W16"], v["bias2"]
    assert torch.equal(W16[:V, :H], W.half()), "W16"
    assert not W16[V:].any() and not W16[:, H:].any(), "W16 padding"
    assert torch.equal(bias2[:V], bias * torch.tensor(LOG2E, dtype=torch.float32)), "bias2"
    assert bool((bias2[V:] == -1e30).all()), "bias2 padding"

    # ---- tile table: exact host prefix sums
    halves = [((Tb + 15) // 16) * ((Ub + 4) // 4) for Tb, Ub in zip(Tl, Ul)]
    assert v["tile_off"].tolist() == [0] + np.cumsum(halves).tolist(), "tile table"
    total = sum(halves)

    # ---- gradient scale S: the power of two that puts max|dcost| S in [2^11, 2^12)
    mx = float(dcost.abs().max())
    assert S == 2.0 ** round(np.log2(S)) and 2 ** 11 <= mx * S < 2 ** 12, (S, mx)
    assert v["inv_S"] == 1.0 / S

    # ---- activations (saved residual: every row of every half-tile; recompute mode: the ring's rows)
    ring_rows = tile_rows(inp["T_len"].cpu(), inp["U_len"].cpu(), out=out)
    n_ring = len(ring_rows)
    wl = v["work_list"].long()
    if out["hidden"] is not None:
        h_all = out["hidden"].view(torch.float16).view(-1, Hp)
        f_rows, f_h = tile_rows(inp["T_len"].cpu(), inp["U_len"].cpu()), h_all[:total * 64]
        ridx = (wl.repeat_interleave(64) * 64 + torch.arange(64, device="cuda").repeat(wl.numel()))
        ring_h = h_all[ridx]
    else:
        f_rows, f_h = ring_rows, v["h"][:n_ring]
        ring_h = f_h
    rb, rt, ru, rv = _rows_dev(f_rows)
    assert not f_h[:, H:].any(), "activation pad columns"
    assert bool(torch.isfinite(f_h.float()).all()), "activation rows (invalid cells included) must be finite"
    hv = f_h[rv, :H].double()
    x32 = enc[rb[rv], rt[rv]] + pred[rb[rv], ru[rv]]                 # the kernel adds in fp32
    th = torch.tanh(x32.double())
    _check("h", hv, th, 2.0 ** -10 * th.abs() + 2.0 ** -24)

    # ---- F epilogue: lse, lp from the kernel's own h and W16
    W16v = W16[:V, :H].double()
    z = hv @ W16v.T + bias.double()
    A = (hv.abs() @ W16v.abs().T).max(1).values + bias.abs().max().double()
    lse_ref = torch.logsumexp(z, 1)
    cb, ct, cu = rb[rv], rt[rv], ru[rv]
    lse_k = out["lse"][cb, ct, cu].double()
    tol = 2.0 ** -21 * (A + lse_ref.abs() + 4) + Vp / 32 * 2.0 ** -24
    _check("F lse", lse_k, lse_ref, tol)
    lp_k = out["lp"][cb, ct, cu].double()
    zb = z[:, bl]
    _check("F lp blank", lp_k[:, 0], zb - lse_ref, tol + 2.0 ** -21 * zb.abs())
    Ub_c = inp["U_len"].long()[cb]
    lab = cu < Ub_c
    tgt = inp["targets"].long()[cb[lab], cu[lab]]
    zt = z[lab].gather(1, tgt[:, None])[:, 0]
    _check("F lp label", lp_k[lab, 1], zt - lse_ref[lab], tol[lab] + 2.0 ** -21 * zt.abs())
    assert not lp_k[~lab, 1].any(), "lp label at u = U_b must be 0"

    # ---- lattice on the kernel's own lp
    from oracle import rnnt_oracle as orc
    lp_np = out["lp"].double().cpu().numpy()
    valid = np.zeros((B, T, U1), bool)
    for b in range(B):
        valid[b, :Tl[b], :Ul[b] + 1] = True
    lp_np[~valid] = 0.0
    a_ref, b_ref, c_ref = orc.lattice_fast(lp_np[..., 0], lp_np[..., 1], Tl, Ul)
    vm = torch.from_numpy(valid).cuda()
    for name, ref in (("alpha", a_ref), ("beta", b_ref)):
        r = torch.from_numpy(ref).cuda()[vm]
        _check("lattice " + name, out[name][vm], r, 1e-5 * r.abs() + 1e-4)
    cr = torch.from_numpy(c_ref).cuda()
    _check("lattice costs", out["costs"], cr, 1e-5 * cr.abs())

    # ---- coefficients from the kernel's lp, alpha, beta and S
    coef = v["coef"]
    assert not coef[~vm].any(), "coef of invalid cells must be 0"
    al, be = out["alpha"].double(), out["beta"].double()
    lpB, lpE = out["lp"][..., 0].double(), out["lp"][..., 1].double()
    logZ = be[:, 0, 0][:, None, None].expand(B, T, U1)
    dcS = (dcost.double() * S)[:, None, None].expand(B, T, U1)
    Tb_g = inp["T_len"].long()[:, None, None].expand(B, T, U1)
    Ub_g = inp["U_len"].long()[:, None, None].expand(B, T, U1)
    tt = torch.arange(T, device="cuda")[None, :, None].expand(B, T, U1)
    uu = torch.arange(U1, device="cuda")[None, None, :].expand(B, T, U1)
    c = al - logZ
    be_t1 = torch.cat([be[:, 1:], torch.zeros_like(be[:, :1])], 1)
    be_u1 = torch.cat([be[:, :, 1:], torch.zeros_like(be[:, :, :1])], 2)
    zero = torch.zeros_like(c)
    gam = torch.exp(c + be) * dcS
    eB = torch.where(tt < Tb_g - 1, torch.exp(c + lpB + be_t1) * dcS,
                     torch.where(uu == Ub_g, torch.exp(c + lpB) * dcS, zero))
    eE = torch.where(uu < Ub_g, torch.exp(c + lpE + be_u1) * dcS, zero)
    mag = al.abs() + logZ.abs() + lpB.abs().maximum(lpE.abs())
    nxt_B = torch.where(tt < Tb_g - 1, be_t1, zero)
    nxt_E = torch.where(uu < Ub_g, be_u1, zero)
    for k, (name, ref, nxt) in enumerate((("gamma", gam, be), ("eB", eB, nxt_B), ("eE", eE, nxt_E))):
        rel = 2.0 ** -21 + 2.0 ** -22 * (mag + nxt.abs())
        sub = 2.0 ** -147 * dcS.abs()                       # expf results in fp32's subnormal range, then scaled by dcost S
        _check("coef " + name, coef[..., k][vm], ref[vm], (rel * ref.abs() + sub)[vm])
    assert torch.equal(coef[..., 3][vm], out["lse"][vm]), "coef lse"

    # ---- work list: in order, exactly the half-tiles with a valid cell above kSkipBelow; dropped ones are negligible
    hb_all, ht_all, hu_all, hv_all = _rows_dev(tile_rows(inp["T_len"].cpu(), inp["U_len"].cpu()))
    ht_all, hu_all = ht_all.clamp(max=T - 1), hu_all.clamp(max=U1 - 1)      # rows past the lattice: masked below
    cmax = coef[hb_all, ht_all, hu_all, :3].abs().max(1).values.masked_fill(~hv_all, 0).view(total, 64).max(1).values
    want = torch.arange(total, device="cuda") if flags & 1 else (cmax > SKIP_BELOW).nonzero()[:, 0]
    assert torch.equal(wl, want), "work list"
    ref_max = torch.stack([gam, eB, eE], -1).abs().max(-1).values[hb_all, ht_all, hu_all]
    ref_max = ref_max.masked_fill(~hv_all, 0).view(total, 64).max(1).values
    dropped = torch.ones(total, dtype=torch.bool, device="cuda")
    dropped[wl] = False
    if dropped.any():
        worst = float(ref_max[dropped].max()) / S
        assert worst <= 2.0 ** -25 * mx * (1 + 2.0 ** -20), ("dropped half-tile gradient", worst, 2.0 ** -25 * mx)
        _note("dropped / 2^-25 max|dcost|", worst / (2.0 ** -25 * mx))

    # ---- G: the gradient ring, row by row (single chunk: ring row j = work-list slot j // 64)
    assert 2 * out["ring_tiles"] >= wl.numel(), "stage checks need a single-chunk ring"
    g = v["g"][:n_ring]
    gb, gt, gu, gv = _rows_dev(ring_rows)
    assert not g[~gv].any(), "ring rows of invalid cells must be 0"
    assert not g[:, V:].any(), "ring columns V..Vp must be 0"
    hgv = ring_h[gv, :H].double()
    zg = hgv @ W16v.T + bias.double()
    cg = coef[gb[gv], gt[gv], gu[gv]].double()
    soft = torch.exp(zg - out["lse"][gb[gv], gt[gv], gu[gv]].double()[:, None]) * cg[:, 0:1]
    ref = soft.clone()
    terms = soft.abs()
    ref[:, bl] -= cg[:, 1]
    terms[:, bl] += cg[:, 1].abs()
    lab = gu[gv] < inp["U_len"].long()[gb[gv]]
    tg = torch.full_like(gu[gv], -1)
    tg[lab] = inp["targets"].long()[gb[gv][lab], gu[gv][lab]]
    ri = lab.nonzero()[:, 0]
    ref[ri, tg[ri]] -= cg[ri, 2]
    terms[ri, tg[ri]] += cg[ri, 2].abs()
    if clamp > 0:
        cbound = (clamp * dcost.abs().double() * S)[gb[gv]][:, None]
        ref = torch.maximum(torch.minimum(ref, cbound), -cbound)
    _check("G ring", g[gv, :V], ref, 2.0 ** -10 * terms + 2.0 ** -23)

    # ---- dW, db from the ring's own fp16 g and h: only the fp32 summation is left
    g64 = g[:, :V].double()
    h64 = ring_h[:, :H].double()
    dW_ref = g64.T @ h64 / S
    dW_sc = g64.abs().T @ h64.abs() / S
    db_ref = g64.sum(0) / S
    db_sc = g64.abs().sum(0) / S
    fx = (2.0 ** -27 / S * wl.numel()) if flags & 2 else 0.0          # fixed-point rounding, one per partial
    res = dict(dW=(dW_ref, DW_C * dW_sc + fx), db=(db_ref, DW_C * db_sc + fx))

    # ---- dh: (g W16 / S) * tanh'(enc + pred), summed over u (d_enc) and t (d_pred)
    dh = g64[gv] @ W16v / S
    A_dh = g64[gv].abs() @ W16v.abs() / S
    xg = (enc[gb[gv], gt[gv]] + pred[gb[gv], gu[gv]]).double()
    hx = torch.tanh(xg)
    dz = dh * (1 - hx * hx)
    sc = 2.0 ** -9 * dh.abs() * hx * hx + 2.0 ** -18 * A_dh + 2.0 ** -14 * dz.abs()
    cnt = torch.ones_like(dz[:, :1])
    ie = gb[gv] * T + gt[gv]
    ip = gb[gv] * U1 + gu[gv]
    z_e = lambda n, x: torch.zeros(n, x.shape[1], dtype=torch.float64, device="cuda")
    d_enc_ref = z_e(B * T, dz).index_add_(0, ie, dz).view(B, T, H)
    d_enc_sc = z_e(B * T, dz).index_add_(0, ie, sc).view(B, T, H)
    d_pred_ref = z_e(B * U1, dz).index_add_(0, ip, dz).view(B, U1, H)
    d_pred_sc = z_e(B * U1, dz).index_add_(0, ip, sc).view(B, U1, H)
    if flags & 2:
        d_enc_sc += z_e(B * T, cnt).index_add_(0, ie, cnt).view(B, T, 1) * 2.0 ** -27 / S
        d_pred_sc += z_e(B * U1, cnt).index_add_(0, ip, cnt).view(B, U1, 1) * 2.0 ** -27 / S
    res.update(d_enc=(d_enc_ref, d_enc_sc), d_pred=(d_pred_ref, d_pred_sc))
    check_grads(out, res, "")
    for b in range(B):
        assert not out["d_enc"][b, Tl[b]:].any() and not out["d_pred"][b, Ul[b] + 1:].any(), "padding gradients"
    return res


def check_grads(out, res, tag):
    for k, (ref, bound) in res.items():
        _check(f"{k}{tag}", out[k], ref, bound)


# (B, T, U, H, V, blank, T_len, U_len, clamp, t_major, save_hidden, dcost kind, seed).  Each case aims at tails:
#   H 8 / 72: one partial 64-column k-chunk; 320: a dh hidden block partly past H; 576, 768, 1280: a dW pair that owns a
#   single 256-column block; 2048: H > 1024.  V 2 / 5 / 257: one pass; 768, 1280: an odd number of passes (which
#   epilogue set drains a pass alternates); 4096: 16 passes.  blank 0, V//2 and V-1 put the blank column in either set.
#   U+1 = 1024 is the lattice's largest block.  B = 341 is past the shared-memory tile table (340 utterances).  Long
#   utterances with short transcripts leave half-tiles of negligible occupancy, which the backward skips.
CASES = [
    (3, 17, 4, 8, 2, 0, [17, 1, 16], [4, 0, 2], -1.0, True, True, "ones", 1),
    (2, 15, 3, 72, 5, 2, [15, 9], [3, 0], 0.01, False, False, "mixed", 2),
    (1, 17, 1023, 72, 5, -1, [17], [1023], -1.0, False, True, "ones", 3),
    (2, 16, 256, 320, 257, 0, [16, 5], [256, 131], -1.0, True, False, "mixed", 4),
    (2, 17, 4, 576, 768, 384, [17, 3], [4, 1], 0.01, False, True, "mixed", 5),
    (1, 15, 3, 1280, 1280, 0, [15], [3], -1.0, True, True, "ones", 6),
    (1, 16, 4, 2048, 4096, 2048, [16], [4], 0.01, False, False, "ones", 7),
    (341, 3, 3, 72, 1000, -1, None, None, -1.0, True, True, "mixed", 8),
    (2, 33, 8, 768, 1000, 0, [33, 1], [8, 0], -1.0, False, True, "ones", 9),
    (2, 160, 40, 128, 512, -1, [160, 97], [40, 13], -1.0, False, True, "ones", 10),     # half-tiles dropped from the
    (3, 250, 20, 64, 300, 7, [250, 180, 64], [20, 5, 12], -1.0, True, False, "ones", 11),   # work list
]


def _dcost(kind, B):
    if kind == "ones":
        return torch.ones(B, device="cuda")
    g = torch.Generator().manual_seed(B)
    d = (torch.rand(B, generator=g) * 1.5 + 0.25) * torch.where(torch.arange(B) % 2 == 0, 1.0, -1.0)
    return d.cuda()


def _build(case):
    B, T, U, H, V, blank, T_len, U_len, clamp, t_major, save, dk, seed = case
    if T_len is None:                          # ragged, with T_b = 1 and U_b = 0 in the batch
        g = torch.Generator().manual_seed(seed)
        T_len = torch.randint(1, T + 1, (B,), generator=g).tolist()
        U_len = torch.randint(0, U + 1, (B,), generator=g).tolist()
        T_len[0], U_len[0], T_len[1], U_len[2] = T, U, 1, 0
    return _case_inputs(B, T, U, H, V, blank, T_len, U_len, seed, t_major), _dcost(dk, B)


@pytest.mark.parametrize("case", CASES, ids=lambda c: "B{}T{}U{}H{}V{}bl{}".format(*c[:6]))
def test_every_stage_against_fp64(case, capsys):
    """One fused forward + backward per case, every stage checked per element against fp64 computed from the previous
    stage's device output (bounds in the module docstring).  Deterministic mode on every other case."""
    inp, dcost = _build(case)
    blank, clamp, save, seed = case[5], case[8], case[10], case[12]
    flags = 2 if seed % 2 else 0
    out = fused_raw(inp, ring_tiles=_big_ring(inp), dcost=dcost, clamp=clamp, flags=flags, save_hidden=save, blank=blank)
    check_stages(inp, out, blank, dcost, clamp, flags)
    with capsys.disabled():
        print("\n[stage-oracle] " + ", ".join(f"{k} {v:.3g}" for k, v in sorted(REPORT.items())))


def _big_ring(inp):
    import rnnt_b200  # noqa: F401
    from rnnt_b200 import _lib
    B, T, _ = inp["enc"].shape
    return int(_lib.lib().rnnt_b200_max_tiles(B, T, inp["pred"].shape[1]))


@pytest.mark.parametrize("save_hidden", [True, False])
def test_multi_chunk_and_recompute_match_single_chunk_per_element(save_hidden):
    """A ring smaller than the work list (the backward walks it in chunks) and the recomputing backward give, per
    element and within the bounds above, the gradients the fp64 reference computes from a single-chunk run's ring.  The
    last chunk's ring rows equal the single-chunk run's rows for the same half-tiles, bit for bit."""
    inp, dcost = _build((3, 40, 20, 320, 768, 0, [40, 23, 7], [20, 11, 0], -1.0, True, save_hidden, "mixed", 21))
    one = fused_raw(inp, ring_tiles=_big_ring(inp), dcost=dcost, save_hidden=save_hidden, blank=0)
    res = check_stages(inp, one, 0, dcost, -1.0, 0)
    n = one["active_halves"]
    for rt in (1, 3):
        many = fused_raw(inp, ring_tiles=rt, dcost=dcost, save_hidden=save_hidden, blank=0)
        assert 2 * rt < n and many["active_halves"] == n
        check_grads(many, res, f" ring_tiles={rt}")
        last = (n - 1) // (2 * rt) * (2 * rt)                      # first slot of the last chunk
        rows = (n - last) * 64
        assert torch.equal(ws_views(many)["g"][:rows], ws_views(one)["g"][last * 64: n * 64]), rt


@pytest.mark.parametrize("save_hidden", [True, False])
def test_results_do_not_depend_on_uninitialised_buffers(save_hidden):
    """The product path hands the kernels torch.empty buffers (workspace, hidden, every output).  Pre-filling them
    with 0xFF (NaN bit patterns) or with zeros gives bit-identical results in deterministic mode, single- and
    multi-chunk."""
    inp, dcost = _build((3, 21, 9, 72, 300, 5, [21, 1, 13], [9, 4, 0], -1.0, True, save_hidden, "mixed", 31))
    for rt in (None, 1):
        a = fused_raw(inp, ring_tiles=rt, dcost=dcost, flags=2, save_hidden=save_hidden, blank=5, fill=0xFF)
        b = fused_raw(inp, ring_tiles=rt, dcost=dcost, flags=2, save_hidden=save_hidden, blank=5, fill=0x00)
        for k in ("costs", "d_enc", "d_pred", "dW", "db"):
            assert torch.equal(a[k], b[k]), (rt, k)
        Tl, Ul = inp["T_len"].tolist(), inp["U_len"].tolist()
        for b_ in range(3):
            for k in ("lp", "lse", "alpha", "beta"):
                assert torch.equal(a[k][b_, :Tl[b_], :Ul[b_] + 1], b[k][b_, :Tl[b_], :Ul[b_] + 1]), (rt, k, b_)
        assert bool(torch.isfinite(a["d_enc"]).all() and torch.isfinite(a["dW"]).all())


@pytest.mark.parametrize("blank", [0, 150, -2])
def test_any_blank_through_the_public_api(blank):
    """joint_rnnt_loss and the dense rnnt_loss with the blank anywhere in the vocabulary, against torchaudio's CPU path
    called with the same blank: costs and every gradient."""
    import rnnt_b200
    B, T, U, H, V = 3, 19, 7, 72, 300
    inp = _case_inputs(B, T, U, H, V, blank, [19, 12, 1], [7, 0, 4], 40 + blank % V, False)
    ref = torch_reference(inp, device="cpu", blank=blank)
    leaves = {k: inp[k].clone().requires_grad_(True) for k in ("enc", "pred", "W", "b")}
    costs = rnnt_b200.joint_rnnt_loss(leaves["enc"], leaves["pred"], leaves["W"], leaves["b"], inp["targets"],
                                      inp["T_len"], inp["U_len"], blank=blank, reduction="none")
    costs.sum().backward()
    assert ((costs.detach().cpu() - ref["costs"]).abs() <= 1e-4 * ref["costs"].abs() + 3e-4).all()
    for k, kr in (("enc", "d_enc"), ("pred", "d_pred"), ("W", "dW"), ("b", "db")):
        r = ref[kr].double()
        assert float((leaves[k].grad.cpu().double() - r).norm() / r.norm()) < 2e-3, kr
    import torchaudio
    logits = ref["logits"].clone().requires_grad_(True)
    ta = torchaudio.functional.rnnt_loss(logits, inp["targets"].cpu(), inp["T_len"].cpu(), inp["U_len"].cpu(),
                                         blank=blank, reduction="none")
    ta.sum().backward()
    dl = ref["logits"].cuda().requires_grad_(True)
    mine = rnnt_b200.rnnt_loss(dl, inp["targets"], inp["T_len"], inp["U_len"], blank=blank, reduction="none")
    mine.sum().backward()
    assert torch.allclose(mine.detach().cpu(), ta.detach(), rtol=1e-5, atol=1e-5)
    assert torch.allclose(dl.grad.cpu(), logits.grad, rtol=1e-4, atol=2e-5)   # fp32 cancellation in p gamma - eB


def test_blank_out_of_range_raises_like_torchaudio():
    import rnnt_b200
    B, T, U, H, V = 2, 10, 4, 64, 40
    inp = make_inputs(B, T, U, H, V)
    logits = torch.randn(B, T, U + 1, V, device="cuda")
    for blank in (V, -V - 1):
        with pytest.raises(RuntimeError, match=r"blank must be within \[0, logits.shape\[-1\]\)"):
            rnnt_b200.joint_rnnt_loss(inp["enc"], inp["pred"], inp["W"], inp["b"], inp["targets"], inp["T_len"],
                                      inp["U_len"], blank=blank)
        with pytest.raises(RuntimeError, match=r"blank must be within \[0, logits.shape\[-1\]\)"):
            rnnt_b200.rnnt_loss(logits, inp["targets"], inp["T_len"], inp["U_len"], blank=blank)
