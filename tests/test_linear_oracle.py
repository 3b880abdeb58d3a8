"""Element-by-element fp64 oracle of the pre-projection GEMMs (`linear_gemm.cu`) across gradient scales.

`rnnt_b200_linear_fwd` / `_bwd` (the optional `audio_ln` / `text_ln` of JointNetwork) are called through the C-ABI, so
the flags and which outputs are NULL are the test's choice; the workspace is filled with 0xFF bytes and the outputs
with NaN first, so an element the kernels never write fails.  Every element of y, dx, dW and db is checked against two
fp64 references, each bound scaling with that element's own sum of absolute terms (sum|terms|):

  (a) from the operands the kernels multiply: fp16(x), fp16(W) and fp16(dy S) / S, S the power of two that puts
      max|dy| S in [2^11, 2^12) (S = 1 when max|dy| is 0 or not finite).  Only fp32 accumulation is left:
        y        |err| <= 2^-17 sum|x16 W16| + 2^-24 (sum|x16 W16| + |b|)     (+ one fp32 rounding of the bias add)
        dx, dW   |err| <= 2^-17 sum|terms|;  deterministic dW adds ksplit 2^-27 / S (one fixed-point rounding per
                 split-K partial, in S-scaled 2^-26 units)
        db       |err| <= 2^-17 sum_m |dy|;  deterministic adds gy 2^-27 / S (gy column-sum blocks)
  (b) from the fp32 inputs: |err| <= (2^-10 + 2^-16) sum|terms| + 2^-25 / S_A sum|B| + 2^-25 / S_B sum|A|  (two fp16
      roundings per product, and fp16's subnormal spacing for each operand: S_A = S for dy, 1 for x and W); the
      deterministic term of (a) is added.  This check does not depend on S, so it is what makes the test scale-free.

Measured largest err / bound over the case matrix on one NVIDIA B200 (1000 W limit):
  y (a) 0.42, (b) 0.65;  dx (a) 0.081, (b) 0.65;  dW (a) 0.090, (b) 0.85;  db 0.0076
Before dy was scaled by S, the dy scales 2^-30, 2^-20, 2^-14 and 2^16 failed (subnormal or infinite fp16 dy), and
deterministic dW / db lost inf and NaN and were not equivariant under power-of-two loss scaling.

The CPU-only checks at the end feed the same checker an emulated kernel with one defect each (a dropped 64-wide
k-chunk, a dropped 128-row tile, a split-K partial counted twice, dy rounded to fp16 without S) and require it to fail.
"""
import math

import pytest
import torch

GRAD_SHIFT = 12                 # kGradShift: max|dy| S in [2^11, 2^12)
ACC_C = 2.0 ** -17              # fp32 accumulation, per unit of sum|terms| (the stage oracle's dW / db constant)
OPS_C = 2.0 ** -10 + 2.0 ** -16  # two fp16 operand roundings per product, plus the accumulation
FX_HALF_UNIT = 2.0 ** -27       # one fixed-point rounding (2^-26 units), S-scaled
SUB = 2.0 ** -25                # half of fp16's subnormal spacing
TILE, BK = 128, 64              # output tile rows / columns, k-chunk
REPORT = {}


def grad_scale(dy):
    """The documented S of dy: 2^(12 - e) for max|dy| = m 2^e, m in [0.5, 1), exponent capped at 126; 1 for 0 / inf / NaN."""
    mx = float(dy.abs().max()) if dy.numel() else 0.0
    if not (0.0 < mx < math.inf):
        return 1.0
    return 2.0 ** min(GRAD_SHIFT - math.frexp(mx)[1], 126)


def dw_ksplit(M, K, N, sms):
    """Split-K factor of the dW launch (dW is N x K, contraction over M): clamp(sms / tiles, 1, ceil(M / 64))."""
    tiles = -(-N // TILE) * -(-K // TILE)
    return max(1, min(sms // tiles, -(-M // BK)))


def db_blocks(M):
    """Row blocks of the column-sum kernel: clamp(ceil(M / 64), 1, 64)."""
    return max(1, min(-(-M // 64), 64))


def operands(x, W, dy):
    """fp64 copies of what the kernels multiply, and S."""
    S = grad_scale(dy) if dy is not None else 1.0
    d16 = (dy * S).half().double() / S if dy is not None else None
    return x.half().double(), W.half().double(), d16, S


def _product(A16, B16, A, B, fa, fb, extra):
    """References and bounds of D = A B: ((a) ref, bound), ((b) ref, bound); fa / fb: subnormal floors of A / B."""
    ta = A16.abs() @ B16.abs()
    tb = A.abs() @ B.abs()
    floor = fa * B.abs().sum(0, keepdim=True) + fb * A.abs().sum(1, keepdim=True)
    return (A16 @ B16, ACC_C * ta + extra), (A @ B, OPS_C * tb + floor + extra)


def expectations(x, W, b, dy, want, det, ksplit, gy):
    """name -> [(label, ref, bound), ...] for the outputs in `want` (subset of y, dx, dW, db)."""
    x16, W16, d16, S = operands(x, W, dy)
    xd, Wd = x.double(), W.double()
    out = {}
    if "y" in want:
        bd = b.double()
        (ra, ba), (rb, bb) = _product(x16, W16.t(), xd, Wd.t(), SUB, SUB, 0.0)
        ta = x16.abs() @ W16.t().abs()
        out["y"] = [("a", ra + bd, ba + 2.0 ** -24 * (ta + bd.abs())), ("b", rb + bd, bb + 2.0 ** -24 * bd.abs())]
    if dy is None:
        return out
    dd = dy.double()
    if "dx" in want:
        (ra, ba), (rb, bb) = _product(d16, W16, dd, Wd, SUB / S, SUB, 0.0)
        out["dx"] = [("a", ra, ba), ("b", rb, bb)]
    if "dW" in want:
        fx = ksplit * FX_HALF_UNIT / S if det and ksplit > 1 else 0.0
        (ra, ba), (rb, bb) = _product(d16.t(), x16, dd.t(), xd, SUB / S, SUB, fx)
        out["dW"] = [("a", ra, ba), ("b", rb, bb)]
    if "db" in want:
        fx = gy * FX_HALF_UNIT / S if det else 0.0
        out["db"] = [("a", dd.sum(0), ACC_C * dd.abs().sum(0) + fx)]
    return out


def verify(got, exp, report=None):
    """Every element of every output within each of its bounds.  Returns the failures (empty: all pass); with `report`,
    records the largest err / bound per output and reference."""
    fails = []
    for name, checks in exp.items():
        g = got[name].double()
        for label, ref, bound in checks:
            err = (g - ref).abs()
            bad = ~(err <= bound)
            if bad.any():
                i = int(bad.flatten().nonzero()[0])
                fails.append(f"{name}({label}): {int(bad.sum())} of {bad.numel()} out of bound; first flat index {i}: got "
                             f"{g.flatten()[i].item()!r}, want {ref.flatten()[i].item()!r}, bound {bound.flatten()[i].item()!r}")
            elif report is not None and err.numel():
                key = f"{name}({label})"
                report[key] = max(report.get(key, 0.0), float((err / bound.clamp_min(1e-300)).max()))
    return fails


# ---------------------------------------------------------------------------------------------------------------- GPU

def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _check_rc(L, rc, what):
    assert rc == 0, f"{what}: rc {rc}: {L.rnnt_b200_last_error().decode()}"


def lib_fwd(x, W, b):
    from rnnt_b200 import _lib
    L = _lib.lib()
    (M, K), N = x.shape, W.shape[0]
    nb = L.rnnt_b200_linear_workspace_bytes(M, K, N, 0, 0)
    ws = torch.full((nb,), 0xFF, dtype=torch.uint8, device="cuda")
    y = torch.full((M, N), float("nan"), device="cuda")
    _check_rc(L, L.rnnt_b200_linear_fwd(x.data_ptr(), W.data_ptr(), b.data_ptr(), M, K, N, y.data_ptr(), ws.data_ptr(),
                                        nb, torch.cuda.current_stream().cuda_stream), "linear_fwd")
    torch.cuda.synchronize()
    return y


def lib_bwd(x, W, dy, want, det):
    """The outputs in `want` (dx, dW, db), the others passed as NULL."""
    from rnnt_b200 import _lib
    L = _lib.lib()
    (M, K), N = x.shape, W.shape[0]
    flags = _lib.FLAG_DETERMINISTIC if det else 0
    nb = L.rnnt_b200_linear_workspace_bytes(M, K, N, 1, flags)
    ws = torch.full((nb,), 0xFF, dtype=torch.uint8, device="cuda")
    shapes = {"dx": (M, K), "dW": (N, K), "db": (N,)}
    got = {k: torch.full(shapes[k], float("nan"), device="cuda") for k in want}
    ptr = lambda k: got[k].data_ptr() if k in got else None
    _check_rc(L, L.rnnt_b200_linear_bwd(x.data_ptr(), W.data_ptr(), dy.data_ptr(), M, K, N, ptr("dx"), ptr("dW"),
                                        ptr("db"), flags, ws.data_ptr(), nb, torch.cuda.current_stream().cuda_stream),
              "linear_bwd")
    torch.cuda.synchronize()
    return got


def make_case(M, K, N, dy_exp=0, x_exp=0, seed=0):
    """x ~ N(0, 1) 2^x_exp; W, b ~ U(-1, 1) / sqrt(K) (nn.Linear's init); dy ~ N(0, 1) 2^dy_exp, each entry also scaled
    by 2^u, u ~ U(-4, 0), so that a case spans five binades."""
    g = torch.Generator().manual_seed(seed * 7919 + M * 31 + K * 7 + N)
    x = torch.randn(M, K, generator=g) * 2.0 ** x_exp
    W = (torch.rand(N, K, generator=g) * 2 - 1) / K ** 0.5
    b = (torch.rand(N, generator=g) * 2 - 1) / K ** 0.5
    dy = torch.randn(M, N, generator=g) * torch.exp2(-4 * torch.rand(M, N, generator=g)) * 2.0 ** dy_exp
    return x.cuda(), W.cuda(), b.cuda(), dy.cuda()


def _run_bwd(M, K, N, dy_exp, det, want=("dx", "dW", "db"), seed=0):
    x, W, b, dy = make_case(M, K, N, dy_exp=dy_exp, seed=seed)
    got = lib_bwd(x, W, dy, want, det)
    exp = expectations(x, W, b, dy, want, det, dw_ksplit(M, K, N, _sms()), db_blocks(M))
    fails = verify(got, exp, REPORT)
    assert not fails, f"M={M} K={K} N={N} dy 2^{dy_exp} det={det}: " + "; ".join(fails)


def _print_report(capsys):
    with capsys.disabled():
        print("\n[linear-oracle] " + ", ".join(f"{k} {v:.3g}" for k, v in sorted(REPORT.items())))


# (M, K, N): M tails 1 / 127 / 128 / 129 / B(U+1) / B T at the bench shape; K, N tails 8 ... 1032; every split-K regime
# of the dW launch on 148 SMs: 1 by tile count (2048 x 2048), 1 because M < 64, 2 ... 5, and 41 (M = 2600, K = 256, N = 128)
SHAPES = [(1, 64, 64), (127, 72, 136), (128, 136, 72), (129, 264, 56), (404, 1024, 1024), (12800, 1024, 1024),
          (300, 8, 1032), (300, 1032, 8), (257, 56, 264), (40, 128, 128), (300, 2048, 2048), (1000, 640, 640),
          (2600, 256, 128)]
REF_SHAPE, TAIL_SHAPE = (3232, 1024, 1024), (129, 264, 56)
DY_EXPS = [-30, -20, -14, -8, 0, 8, 16]
_ids = lambda s: "M{}K{}N{}".format(*s)


def test_case_matrix_covers_every_split_regime():
    """The shapes above reach each ksplit regime of the dW launch on a 148-SM B200."""
    ks = {s: dw_ksplit(*s, 148) for s in SHAPES}
    assert ks[(300, 2048, 2048)] == 1 and 148 // (16 * 16) == 0          # one by tile count
    assert ks[(40, 128, 128)] == 1 and 148 // 1 > 1                      # one because M < 64
    assert ks[(404, 1024, 1024)] == 2 and ks[(1000, 640, 640)] == 5
    assert ks[(2600, 256, 128)] == 41
    assert {1, 2, 3, 5, 41} <= set(ks.values())


@pytest.mark.gpu
@pytest.mark.parametrize("shape", SHAPES + [REF_SHAPE], ids=_ids)
@pytest.mark.parametrize("x_exp", [-6, 0, 6])
def test_forward_against_fp64(shape, x_exp, capsys):
    """y = x W^T + b, K-major x K-major, at x scales 2^-6 ... 2^6."""
    M, K, N = shape
    x, W, b, _ = make_case(M, K, N, x_exp=x_exp, seed=1)
    fails = verify({"y": lib_fwd(x, W, b)}, expectations(x, W, b, None, ("y",), False, 1, 1), REPORT)
    assert not fails, f"{shape} x 2^{x_exp}: " + "; ".join(fails)
    _print_report(capsys)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", SHAPES, ids=_ids)
@pytest.mark.parametrize("det", [False, True], ids=["default", "deterministic"])
def test_backward_against_fp64(shape, det, capsys):
    """dx (K-major x MN-major), dW (MN-major x MN-major, split-K) and db at every shape, default and deterministic."""
    _run_bwd(*shape, 0, det)
    _print_report(capsys)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [REF_SHAPE, TAIL_SHAPE], ids=_ids)
@pytest.mark.parametrize("dy_exp", DY_EXPS)
@pytest.mark.parametrize("det", [False, True], ids=["default", "deterministic"])
def test_backward_across_gradient_scales(shape, dy_exp, det, capsys):
    """dy scaled by 2^-30 ... 2^16: reference (b) holds with the same constant at every scale."""
    _run_bwd(*shape, dy_exp, det)
    _print_report(capsys)


@pytest.mark.gpu
@pytest.mark.parametrize("want", [("dx",), ("dW",), ("db",), ("dx", "dW", "db")], ids="+".join)
@pytest.mark.parametrize("det", [False, True], ids=["default", "deterministic"])
def test_null_output_combinations(want, det):
    """Any of dx / dW / db may be NULL; the others are still complete and right (ksplit 5 for dW here)."""
    _run_bwd(257, 56, 264, -14, det, want=want, seed=2)


@pytest.mark.gpu
@pytest.mark.parametrize("det", [False, True], ids=["default", "deterministic"])
def test_zero_gradient_gives_exact_zeros(det):
    x, W, _, dy = make_case(404, 1024, 1024)
    got = lib_bwd(x, W, torch.zeros_like(dy), ("dx", "dW", "db"), det)
    for k, v in got.items():
        assert not v.any(), k


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(404, 256, 128), (300, 2048, 2048)], ids=_ids)
@pytest.mark.parametrize("det", [False, True], ids=["default", "deterministic"])
def test_inf_and_nan_reach_the_gradients_as_in_fp32(shape, det):
    """One inf and one NaN in dy: exactly the elements torch's fp64 product makes non-finite are non-finite (rows of dx,
    rows of dW, entries of db), with split-K (ksplit 7) and without; the others are finite.  GradScaler relies on this."""
    M, K, N = shape
    x, W, _, dy = make_case(M, K, N)
    dy[3, 5] = float("inf")
    dy[M - 2, N - 1] = float("nan")
    got = lib_bwd(x, W, dy, ("dx", "dW", "db"), det)
    dd, xd, Wd = dy.double(), x.double(), W.double()
    for k, ref in (("dx", dd @ Wd), ("dW", dd.t() @ xd), ("db", dd.sum(0))):
        assert torch.equal(torch.isfinite(got[k]), torch.isfinite(ref)), k
    assert not torch.isfinite(got["dx"][3]).any() and not torch.isfinite(got["dW"][N - 1]).any()


@pytest.mark.gpu
@pytest.mark.parametrize("dims", [(4, 120, 30, 1024, 1024, 1024, 1024), (3, 37, 11, 136, 200, 72, 300)],
                         ids=["F1024H1024V1024", "ragged"])
def test_scaled_loss_gives_scaled_gradients_bit_for_bit(dims):
    """With deterministic accumulation everywhere, the gradients of 2^k loss are exactly 2^k times those of the loss
    -- d_audio, d_text and every parameter gradient, audio_ln / text_ln included -- for k in {-24, -12, -6, 3, 8}:
    the fused backward and the pre-projection backward both absorb the binade of their incoming gradient in S."""
    import rnnt_b200
    B, T, U, Fa, Ft, H, V = dims
    torch.manual_seed(11)
    joint = rnnt_b200.JointNetwork(Fa, Ft, H, V).cuda()
    audio = torch.randn(B, T, Fa, device="cuda")
    text = torch.randn(B, U + 1, Ft, device="cuda")
    targets = torch.randint(0, V - 1, (B, U), dtype=torch.int32, device="cuda")
    T_len = torch.tensor([T] + [max(1, T - 7 * i) for i in range(1, B)], dtype=torch.int32, device="cuda")
    U_len = torch.tensor([U] + [max(0, U - 4 * i) for i in range(1, B)], dtype=torch.int32, device="cuda")

    def grads(c):
        a, t = audio.clone().requires_grad_(True), text.clone().requires_grad_(True)
        joint.zero_grad()
        (joint.loss(a, t, targets, T_len, U_len, reduction="mean") * c).backward()
        out = {n: p.grad.clone() for n, p in joint.named_parameters()}
        out["audio"], out["text"] = a.grad, t.grad
        return out

    torch.use_deterministic_algorithms(True)
    try:
        base = grads(1.0)
        assert {"audio_ln.weight", "audio_ln.bias", "text_ln.weight", "text_ln.bias"} <= set(base)
        for k in (-24, -12, -6, 3, 8):
            c = 2.0 ** k
            got = grads(c)
            for n, g in base.items():
                assert bool(torch.isfinite(g).all()), n
                want = g * c
                if not torch.equal(got[n], want):
                    d = (got[n] - want).abs().max().item()
                    pytest.fail(f"2^{k}: {n} differs from 2^{k} x the unscaled gradient (max abs diff {d:.3g}, "
                                f"{int((got[n] != want).sum())} of {g.numel()} elements)")
    finally:
        torch.use_deterministic_algorithms(False)


# ---------------------------------------------------------------------------------------------------------------- CPU

def emulate(x, W, b, dy, ksplit, defect=None):
    """The kernels' arithmetic on the CPU (fp16 operands as above, exact products, one fp32 rounding per output), split
    into the kernel's tiles, k-chunks and split-K ranges, with an optional defect."""
    M, K = x.shape
    x16, W16, d16, S = operands(x, W, dy)
    if defect == "dy_without_S":
        d16 = dy.half().double()
    y = x16 @ W16.t() + b.double()
    if defect == "dropped_row_tile":
        y[TILE:2 * TILE] = 0.0
    dyk = d16.clone()
    if defect == "dropped_k_chunk":                    # dx contracts over N in 64-wide chunks
        dyk[:, BK:2 * BK] = 0.0
    dx = dyk @ W16
    nkc = -(-M // BK)
    parts = []
    for ks in range(ksplit):                           # split-K ranges of the dW launch, in 64-row k-chunks of M
        r0, r1 = BK * (nkc * ks // ksplit), min(M, BK * (nkc * (ks + 1) // ksplit))
        parts.append(d16[r0:r1].t() @ x16[r0:r1])
    dW = sum(parts)
    if defect == "partial_counted_twice":
        dW = dW + parts[1]
    db = dy.double().sum(0)
    return {"y": y.float(), "dx": dx.float(), "dW": dW.float(), "db": db.float()}


def _cpu_case(dy_exp):
    g = torch.Generator().manual_seed(5)
    M, K, N = 300, 136, 200
    x = torch.randn(M, K, generator=g)
    W = (torch.rand(N, K, generator=g) * 2 - 1) / K ** 0.5
    b = (torch.rand(N, generator=g) * 2 - 1) / K ** 0.5
    dy = torch.randn(M, N, generator=g) * torch.exp2(-4 * torch.rand(M, N, generator=g)) * 2.0 ** dy_exp
    return x, W, b, dy


@pytest.mark.parametrize("det", [False, True])
@pytest.mark.parametrize("dy_exp", [-20, 0, 16])
def test_checker_accepts_the_emulated_kernel(det, dy_exp):
    x, W, b, dy = _cpu_case(dy_exp)
    got = emulate(x, W, b, dy, ksplit=3)
    assert not verify(got, expectations(x, W, b, dy, ("y", "dx", "dW", "db"), det, 3, db_blocks(300)))


@pytest.mark.parametrize("defect, dy_exp, hit", [("dropped_k_chunk", 0, "dx"), ("dropped_row_tile", 0, "y"),
                                                 ("partial_counted_twice", 0, "dW"), ("dy_without_S", -20, "dx")])
def test_checker_rejects_a_defective_kernel(defect, dy_exp, hit):
    """Each defect fails the check of the output it touches, against both references."""
    x, W, b, dy = _cpu_case(dy_exp)
    got = emulate(x, W, b, dy, ksplit=3, defect=defect)
    fails = verify(got, expectations(x, W, b, dy, ("y", "dx", "dW", "db"), True, 3, db_blocks(300)))
    assert any(f.startswith(f"{hit}(a)") for f in fails), fails
    assert any(f.startswith(f"{hit}(b)") for f in fails), fails
