"""Greedy decode (decode_loop.cu on decode_common.cuh) element by element against fp64, in every shared-memory plan.

The persistent kernel keeps a weight matrix's output slice in shared memory only while it fits a 92 KB budget per CTA
(`decode_smem_plan`); the rest is streamed from L2 every step, and GEMVs of K > 512 run over several K-chunks.  Each
case below reaches a stated plan (checked against a mirror of the launcher, for the device's SM count).  Per case the
batch is decoded once in one shot and once through `StreamingGreedyDecoder` fed one frame per call; the two must agree
bit for bit (tokens and margins), so what is checked on the streaming run holds for the one-shot kernel.  After every
frame the decoder's state buffer is read and `tests/decode_oracle.py` checks, against fp64:

  tables      emb_ln = LayerNorm(embedding), t1 = conv1 taps of the kernel's emb_ln
  per frame   ynew (conv1 from the kernel's t1), z (conv2 of the last five conv1 outputs), the conv1 / conv2 tap
              accumulator rings, lin (of the kernel's z), feats (LayerNorm of the kernel's lin, and end to end against
              conv_predictor on the last 7 tokens), hbuf = tanh(enc + feats), the frame's last logits row (of hbuf)
  per step    the emitted token and the margin against fp64 logits teacher-forced on the kernel's own prefix; the
              frame's advance (blank within the bound of the best, or the max_per_frame cap); no step after max_len

The bounds are derived from the kernel's summation order (tests/decode_oracle.py states them); no token is required to
equal an fp64 argmax.  Measured largest err / bound per observable on one NVIDIA B200 (1000 W power limit):
see DESIGN.md section 5.

Also here: the batched step kernel `joint_argmax` (decode.cu) against fp64 over N, V, H (up to its 2048 limit) and
strided rows, exact ties in both kernels, and CPU tests that feed the same checker an fp32 emulation of the decoder,
correct and with one planted defect each.
"""
import math

import numpy as np
import pytest
import torch

import decode_oracle as do

gpu = pytest.mark.gpu
REPORT = {}

J, C2, L = do.JOINT, do.CONV2, do.LINEAR

# name: (H, V, E, blank, lens, max_len, max_per_frame, seed, scale, blank_bias, plan on 148 SMs)
CASES = {
    # control: everything resident, joint in 2 K-chunks
    "resident": (1024, 1024, 512, 1023, [16, 13, 9], 200, 10, 1, 3.0, 5.0, J | C2 | L),
    # joint (28 rows x 4 KB per CTA) read from L2
    "joint_streamed": (1024, 4096, 512, 4095, [14, 12, 7], 200, 10, 2, 3.0, 5.0, C2 | L),
    # conv2 from L2; conv2 taps (EPI 1) and the conv1 table (EPI 2) over 2 K-chunks
    "conv2_streamed": (1024, 1024, 1024, 1023, [14, 11, 6], 200, 10, 3, 3.0, 4.0, J | L),
    # linear from L2, its K = 640 in two chunks, the second partial (K4 = 160)
    "linear_streamed": (1024, 1024, 640, 1023, [14, 12, 5], 200, 10, 4, 3.0, 4.0, J | C2),
    # predictor LayerNorm over H = 2304 > 2048 (uncached); joint in 5 K-chunks, the last partial; conv2, linear from L2
    "wide_H": (2304, 1024, 512, 1023, [13, 12, 8], 200, 10, 5, 3.0, 4.0, J),
    # embedding LayerNorm over E = 2112 > 2048 (uncached); 5-chunk conv1 table GEMV
    "wide_E": (256, 64, 2112, 63, [12, 10], 200, 10, 6, 3.0, 2.5, J | L),
    # V < grid, T_b = 0 and 1, blank at V-1 and at 0; the 10-emit cap fires and max_len is reached mid-frame
    "small_odd": (36, 29, 36, 28, [16, 0, 1, 12, 9], 24, 10, 7, 3.0, 2.0, J | C2 | L),
    "small_odd_blank0": (36, 29, 36, 0, [16, 1, 0, 14, 7], 24, 10, 8, 3.0, 2.0, J | C2 | L),
    # B = 150 > 148 CTAs: several row groups per warp, ragged lengths; exact ties (see TIES)
    "many_rows": (96, 301, 72, 300, None, 200, 10, 9, 3.0, 5.0, J | C2 | L),
}
MANY_ROWS_B, MANY_ROWS_T = 150, 16
# many_rows: joint row a copied into b (with its bias), both boosted: b = a + 256 (one thread's strided argmax scan
# sees both) and b in another CTA's slice of the joint GEMV and another warp of the argmax
TIES = [(7, 263), (20, 150)]
TIE_BOOST = 1.5


def case_lens(name):
    lens = CASES[name][4]
    if lens is not None:
        return lens
    g = torch.Generator().manual_seed(90)
    lens = torch.randint(0, MANY_ROWS_T + 1, (MANY_ROWS_B,), generator=g)
    lens[0], lens[1], lens[2] = MANY_ROWS_T, 0, 1
    return lens.tolist()


def make_model(seed, H, V, E, blank, scale, blank_bias, ties=()):
    """Seeded joint weights / ConvPredictor on the CPU generator (identical on every machine)."""
    import rnnt_b200
    torch.manual_seed(seed)
    joint = rnnt_b200.JointNetwork(-1, -1, H, V)
    pred = rnnt_b200.ConvPredictor(V, H, E, 0.3).eval()
    with torch.no_grad():
        W, b = joint.joint_ln.weight, joint.joint_ln.bias
        W.mul_(scale)
        b[blank] += blank_bias
        for a, c in ties:
            b[a] += TIE_BOOST
            W[c], b[c] = W[a], b[a]
    joint.blank_idx = blank
    return joint, pred


def case_inputs(name):
    H, V, E, blank, _, max_len, mpf, seed, scale, bb, _ = CASES[name]
    ties = TIES if name == "many_rows" else ()
    joint, pred = make_model(seed, H, V, E, blank, scale, bb, ties)
    lens = case_lens(name)
    enc = torch.randn(len(lens), max(lens), H, generator=torch.Generator().manual_seed(seed + 100))
    m = do.Model(joint.joint_ln.weight, joint.joint_ln.bias, pred, blank, max_len, mpf)
    return joint, pred, enc, lens, m


def print_report(capsys, title, report):
    with capsys.disabled():
        print(f"\n[decode-oracle] {title}: " + ", ".join(f"{k} {v:.3g}" for k, v in sorted(report.items())))


# ------------------------------------------------------------------------------------------------------------ CPU

def test_cases_reach_their_plans_on_148_sms():
    """The case list on a 148-SM B200: the residency of each case, and the chunk / LayerNorm paths it names."""
    for name, c in CASES.items():
        H, V, E = c[:3]
        assert do.smem_plan(148, H, V, E) == c[-1], name
    assert do.gemv_chunks(1024) == 2 and do.gemv_chunks(640) == 2 and 640 // 4 == 160     # joint; linear's partial chunk
    assert do.gemv_chunks(2304) == 5 and 2304 % do.CHUNK != 0 and do.gemv_chunks(2112) == 5
    assert 2304 > do.LN_CACHED and 2112 > do.LN_CACHED and 1024 <= do.LN_CACHED
    assert CASES["small_odd"][1] < 148 and MANY_ROWS_B > 148
    per_j = -(-301 // 148)
    (a1, b1), (a2, b2) = TIES
    assert b1 == a1 + 256 and a2 // per_j != b2 // per_j and a2 % 256 // 32 != b2 % 256 // 32


@pytest.mark.parametrize("B,H,V,E", [(1, 4, 2, 4), (3, 36, 29, 36), (150, 96, 301, 72), (5, 2304, 1024, 2112)])
def test_state_layout_fits_the_state_buffer(B, H, V, E):
    from rnnt_b200 import _lib
    _, end = do.state_layout(B, H, V, E)
    assert end <= _lib.lib().rnnt_b200_greedy_decode_state_bytes(B, H, V, E)


def cpu_case():
    """Wide enough for every planted defect: H = 2112 (5 joint K-chunks, uncached LayerNorm), V = 300 (argmax over all
    8 warps), a cap of 3 that fires, frames that end in a blank and an utterance that reaches max_len mid-frame."""
    joint, pred = make_model(31, 2112, 300, 36, 299, 3.0, 3.0)
    lens = [8, 5, 0, 1]
    enc = torch.randn(len(lens), 8, 2112, generator=torch.Generator().manual_seed(32))
    m = do.Model(joint.joint_ln.weight, joint.joint_ln.bias, pred, 299, 16, 3)
    return m, enc.numpy(), lens


def test_checker_accepts_the_emulated_decoder(capsys):
    m, enc, lens = cpu_case()
    trace = do.emulate(m, enc, lens)
    report = {}
    assert do.check(m, trace, report) == []
    new = [[t for fr in trace["frames"] for t in fr["new"][b]] for b in range(len(lens))]
    assert sum(map(len, new)) > 10
    per_frame = [len(fr["new"][b]) for fr in trace["frames"] for b in range(len(lens))]
    assert m.max_per_frame in per_frame                                   # the cap fires
    assert any(len(fr["margins"][b]) > len(fr["new"][b]) for fr in trace["frames"] for b in range(len(lens)))
    assert any(len(fr["margins"][b]) == len(fr["new"][b]) > 0 for fr in trace["frames"] for b in range(len(lens)))
    print_report(capsys, "emulated decoder", report)


@pytest.mark.parametrize("defect,observable", [
    ("conv2_ring_rotated", "acc2"), ("joint_last_chunk_dropped", "logits"), ("ln_first_2048", "feats"),
    ("feats_not_refreshed", "feats"), ("cap_plus_one", "cap"), ("margin_other_warps", "margin")])
def test_checker_rejects_a_defective_decoder(defect, observable):
    m, enc, lens = cpu_case()
    fails = do.check(m, do.emulate(m, enc, lens, defect=defect))
    assert any(f.startswith(observable + ":") for f in fails), fails[:5]


def test_checker_rejects_a_changed_idle_slot():
    """A slot past its frames (or past max_len) must not take a step or change its state."""
    m, enc, lens = cpu_case()
    trace = do.emulate(m, enc, lens)
    trace["frames"][-1]["regions"]["lin"][2, 0] += 1.0
    assert any(f.startswith("idle:") for f in do.check(m, trace))


# ------------------------------------------------------------------------------------------------------------ GPU

def _words(state):
    return state.view(torch.float32).cpu().numpy(), state.view(torch.int32).cpu().numpy()


def run_kernel(name):
    """One-shot and frame-by-frame streaming decode of a case on the GPU: the trace `decode_oracle.check` reads."""
    import rnnt_b200
    H, V, E, blank, _, max_len, mpf = CASES[name][:7]
    joint, pred, enc, lens, m = case_inputs(name)
    joint, pred = joint.cuda(), pred.cuda()
    B, T = enc.shape[:2]
    enc_d = enc.cuda()
    one_tok, one_mg = rnnt_b200.greedy_decode(enc_d, torch.tensor(lens), joint.joint_ln.weight, joint.joint_ln.bias,
                                              pred, blank, max_len, mpf, return_margins=True)
    dec = rnnt_b200.StreamingGreedyDecoder(joint, pred, B, max_length=max_len, max_outputs_per_step=mpf)
    assert do.state_layout(B, H, V, E)[1] <= dec.state.numel()
    dec.reset(range(B))
    frames = []
    for t in range(T):
        new, mg = dec.decode_chunk(enc_d[:, t:t + 1], [int(t < n) for n in lens], return_margins=True)
        f, i = _words(dec.state)
        frames.append(dict(new=new, margins=mg, regions=do.split_regions(f, i, B, H, V, E)))
    emb_ln, t1 = do.tables(_words(dec.state)[0], B, H, V, E)
    for b in range(B):
        assert [x for fr in frames for x in fr["new"][b]] == one_tok[b], b
        assert [x for fr in frames for x in fr["margins"][b]] == one_mg[b], b
    return m, dict(enc=enc.numpy(), lens=lens, emb_ln=emb_ln, t1=t1, frames=frames)


@gpu
@pytest.mark.parametrize("name", list(CASES))
def test_greedy_decode_against_fp64(name, capsys):
    H, V, E = CASES[name][:3]
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    assert do.smem_plan(sms, H, V, E) == CASES[name][-1], f"{name} does not reach its plan on {sms} SMs"
    m, trace = run_kernel(name)
    report = {}
    fails = do.check(m, trace, report)
    assert not fails, f"{name}: {len(fails)} failures: " + "; ".join(fails[:8])
    B = len(trace["lens"])
    tokens = [[x for fr in trace["frames"] for x in fr["new"][b]] for b in range(B)]
    assert sum(map(len, tokens)) >= B, "the case hardly emits: not a test of the predictor"
    blanks = sum(len(fr["margins"][b]) > len(fr["new"][b]) for fr in trace["frames"] for b in range(B))
    assert blanks > 0
    if name.startswith("small_odd"):
        assert any(len(fr["new"][b]) == m.max_per_frame for fr in trace["frames"] for b in range(B)), "cap never fired"
        assert any(len(fr["new"][b]) > 0 and len(fr["margins"][b]) == len(fr["new"][b])
                   for fr in trace["frames"] for b in range(B)), "max_len never reached mid-frame"
    if name == "many_rows":
        for a, c in TIES:
            assert not any(c in tk for tk in tokens), f"emitted {c}, the higher index of a tie with {a}"
            hits = [mg for fr in trace["frames"] for b in range(B)
                    for tk, mg in zip(fr["new"][b], fr["margins"][b]) if tk == a]
            assert hits and all(mg == 0.0 for mg in hits), (a, c, hits[:5])
            for fr in trace["frames"]:
                lg = fr["regions"]["logits"]
                for b in range(B):
                    if fr["margins"][b]:
                        assert lg[b, a].view(np.uint32) == lg[b, c].view(np.uint32), (a, c, b)
    for k, v in report.items():
        REPORT[(name, k)] = v
    print_report(capsys, name, report)


JA_N, JA_V, JA_H = [1, 3, 130], [2, 29, 1000, 4097], [4, 36, 2048]


@gpu
@pytest.mark.parametrize("H", JA_H)
@pytest.mark.parametrize("V", JA_V)
@pytest.mark.parametrize("N", JA_N)
def test_joint_argmax_against_fp64(N, V, H):
    """tokens / margins of the step kernel (decode.cu) from strided row views: the decision rule of the greedy checker
    (per-logit bound: ceil(H/32) FMAs per lane, 5 butterfly levels, the bias; tanhf of an fp32 add), and exact ties
    (a joint row copied to a higher index, once in the same argmax thread, once in another warp) resolved to the lower
    index with margin 0."""
    import rnnt_b200
    g = torch.Generator().manual_seed(1000 * N + 10 * V + H)
    W = (torch.rand(V, H, generator=g) * 2 - 1) * (3.0 / math.sqrt(H))
    bias = torch.rand(V, generator=g) - 0.5
    a_buf = torch.randn(N, H + 12, generator=g)
    p_buf = torch.randn(2 * N, H, generator=g)
    a, p = a_buf[:, 4:4 + H], p_buf[::2]
    h = np.tanh(a.double().numpy() + p.double().numpy())
    ties = [(3, V - 2)] if V >= 29 else []
    if V > 261:
        ties.append((5, 261))
    for x, y in ties:
        l0 = h @ W.double().numpy().T + bias.double().numpy()
        bias[x] += float(np.median(l0.max(1) - l0[:, x]))           # the pair wins about half of the rows
        W[y], bias[y] = W[x], bias[x]
    Wd, bd = W.double().numpy(), bias.double().numpy()
    l64 = h @ Wd.T + bd
    _, eh = do.tanh_add(a.double().numpy(), p.double().numpy())
    delta = (do.gamma(-(-H // 32) + 6) * (np.abs(h) @ np.abs(Wd).T + np.abs(bd)) + eh @ np.abs(Wd).T) * do.SLACK
    a_d, p_d = a_buf.cuda()[:, 4:4 + H], p_buf.cuda()[::2]
    assert a_d.stride(0) == H + 12 and p_d.stride(0) == 2 * H
    tok, mg = rnnt_b200.joint_argmax(a_d, p_d, W.cuda(), bias.cuda(), return_margin=True)
    tok, mg = tok.cpu().numpy(), mg.cpu().numpy().astype(np.float64)
    for n in range(N):
        top = int(np.argmax(l64[n]))
        s = np.sort(l64[n])
        v = int(tok[n])
        assert 0 <= v < V and l64[n, top] - l64[n, v] <= delta[n, v] + delta[n, top], (n, v, top)
        assert abs(mg[n] - (s[-1] - s[-2])) <= 2 * delta[n].max() + do.U * abs(mg[n]), (n, mg[n], s[-1] - s[-2])
    for x, y in ties:
        assert not (tok == y).any()
        assert (mg[tok == x] == 0.0).all()
        if N == 130:
            assert (tok == x).any()
