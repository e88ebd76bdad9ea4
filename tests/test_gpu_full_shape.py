"""GPU: the BENCHMARKED configuration (48 heads = one CogVideoX-5B layer-direction, 3-second / 9-second / 63-second lengths,
checkpoint group 16, the 3-buffer ring with trajectory / Q-side / K-side kernels co-resident on three streams) checked for
correctness, not only timed:
  (i)   H=48, NC=282, G=16 forward + backward vs the analytic oracle run group by group (oracle/ttt_oracle.py
        ttt_mlp_primal_backward_chunked; fp32 on the same bf16-rounded inputs), tolerance 1e-2 relative per tensor;
  (ii)  the backward run twice gives identical bits (no atomics on running sums);
  (iii) whole scan == two half scans joined through the exported final state (forward, bit-exact) and through the
        upstream state gradient (backward, ttt_b200_mlp_backward_seeded), at NC = 804 (9 s) and 5 487 (63 s): a
        size-independent property that needs no oracle;
  (iv)  the reference's 43-argument ttt_backward mirror == ttt_backward_simple;
  (v)   the per-group K-side mode == the persistent mode, batch element by batch element.
"""
import os

import pytest
import torch

from oracle import ttt_oracle as O
from ttt_video_dit_b200 import test_time_training as tt

pytestmark = pytest.mark.gpu
H48 = 48
SHAPES = ((64, 256), (1, 256), (256, 64), (1, 64))


def _bench_like_inputs(B, H, NC, seed, dev="cuda"):
    """Inputs of bench.py's shape and statistics (SURVEY 8d), generated on the device (fast at 63 s)."""
    g = torch.Generator(device=dev).manual_seed(seed)
    rn = lambda *s: torch.randn(*s, generator=g, device=dev)
    nrm = lambda t: torch.nn.functional.normalize(t, dim=-1)
    d = dict(XQ=nrm(rn(B, H, NC, 64, 64)).bfloat16(), XK=nrm(rn(B, H, NC, 64, 64)).bfloat16(), XV=rn(B, H, NC, 64, 64).bfloat16(),
             le=((0.1 / 64) * torch.sigmoid(rn(B, H, NC, 64, 1)) / 64).bfloat16(), dOut=rn(B, H, NC, 64, 64).bfloat16(),
             ln_w=(1 + 0.1 * rn(H, 64)), ln_b=0.1 * rn(H, 64),
             W1=(0.02 * rn(H, 64, 256)).unsqueeze(0).repeat(B, 1, 1, 1).contiguous(), b1=torch.zeros(B, H, 1, 256, device=dev),
             W2=(0.02 * rn(H, 256, 64)).unsqueeze(0).repeat(B, 1, 1, 1).contiguous(), b2=torch.zeros(B, H, 1, 64, device=dev))
    return d


def _forward(d, sl, state, G):
    q, k, v, le = [d[n][:, :, sl].contiguous() for n in ("XQ", "XK", "XV", "le")]
    B, H, NC = q.shape[:3]
    K = (NC + G - 1) // G
    out = torch.empty_like(q)
    ck = [torch.empty(B, H, K, a, b, device=q.device) for a, b in SHAPES]
    last = [torch.empty(B, H, a, b, device=q.device) for a, b in SHAPES]
    lw, lb = d["ln_w"].reshape(1, H, 1, 64).contiguous(), d["ln_b"].reshape(1, H, 1, 64).contiguous()
    tt.ttt_forward(q, k, v, le, lw, lb, *state, *ck, out, G, W_last=last)
    return out, ck, last, (q, k, v, le, lw, lb)


def _backward(fw, d, sl, G, dW_last=None):
    out, ck, last, (q, k, v, le, lw, lb) = fw
    return tt.ttt_backward_simple(q, k, v, le, lw, lb, *ck, d["dOut"][:, :, sl].contiguous(), G, dW_last=dW_last)


def test_h48_nc282_forward_backward_vs_chunked_oracle():
    G, NC = 16, 282
    d = _bench_like_inputs(1, H48, NC, seed=3)
    state = [d[n] for n in ("W1", "b1", "W2", "b2")]
    fw = _forward(d, slice(0, NC), state, G)
    g = _backward(fw, d, slice(0, NC), G)
    torch.cuda.synchronize()
    c = lambda t: t.float().cpu()
    torch.set_num_threads(min(32, torch.get_num_threads()))
    ref_out, _, _ = O.ttt_mlp_primal_forward(c(d["XQ"]), c(d["XK"]), c(d["XV"]), c(d["le"]), c(d["ln_w"]), c(d["ln_b"]),
                                             *[c(s) for s in state], G)
    assert O.rel_err(c(fw[0]), ref_out) < 1e-2
    ref = O.ttt_mlp_primal_backward_chunked(c(d["XQ"]), c(d["XK"]), c(d["XV"]), c(d["le"]), c(d["ln_w"]), c(d["ln_b"]),
                                            *[c(s) for s in state], c(d["dOut"]), G)
    names = ["dln_w", "dln_b", "dW1", "db1", "dW2", "db2", "dXQ", "dXV", "dXK", "dlast_eta"]
    errs = {n: O.rel_err(c(a).reshape(ref[n].shape), ref[n]) for n, a in zip(names, g)}
    bad = {n: e for n, e in errs.items() if not (e < 1e-2)}
    assert not bad, f"rel errors above 1e-2 at the benchmarked shape: {bad} (all: {errs})"


@pytest.mark.parametrize("H,NC,G", [(H48, 282, 16), (6, 37, 4)])
def test_backward_is_bitwise_reproducible(H, NC, G):
    d = _bench_like_inputs(1, H, NC, seed=4)
    state = [d[n] for n in ("W1", "b1", "W2", "b2")]
    fw = _forward(d, slice(0, NC), state, G)
    a = _backward(fw, d, slice(0, NC), G)
    b = _backward(fw, d, slice(0, NC), G)
    torch.cuda.synchronize()
    names = ["dln_w", "dln_b", "dW1", "db1", "dW2", "db2", "dXQ", "dXV", "dXK", "dlast_eta"]
    diff = [n for n, x, y in zip(names, a, b) if not torch.equal(x, y)]
    assert not diff, f"backward not reproducible bit for bit: {diff}"


@pytest.mark.parametrize("NC,cut", [(804, 400), (5487, 2752), (37, 16)])  # cuts on checkpoint-group boundaries (G = 16)
def test_whole_scan_equals_two_joined_halves(NC, cut):
    """Forward: the state exported by the first half (W_last) feeds the second half -> identical output bits.  Backward:
    the second half's gradient w.r.t. its initial state seeds the first half's backward -> the gradients of the whole scan.
    The whole-scan backward carries the state gradient across the cut in fp32 through the same scratch layout, so the two
    ways agree to fp32 round-off of the LayerNorm-parameter sums and bit for bit elsewhere."""
    G, H = 16, H48 if NC > 100 else 3
    d = _bench_like_inputs(1, H, NC, seed=5)
    state = [d[n] for n in ("W1", "b1", "W2", "b2")]
    whole = _forward(d, slice(0, NC), state, G)
    h1 = _forward(d, slice(0, cut), state, G)
    h2 = _forward(d, slice(cut, NC), h1[2], G)
    assert torch.equal(torch.cat([h1[0], h2[0]], dim=2), whole[0])
    for a, b in zip(h2[2], whole[2]):
        assert torch.equal(a, b)
    gw = _backward(whole, d, slice(0, NC), G)
    g2 = _backward(h2, d, slice(cut, NC), G)
    g1 = _backward(h1, d, slice(0, cut), G, dW_last=g2[2:6])
    torch.cuda.synchronize()
    for i, n in ((2, "dW1"), (3, "db1"), (4, "dW2"), (5, "db2")):
        assert torch.equal(g1[i], gw[i]), n
    for i, n in ((6, "dXQ"), (7, "dXV"), (8, "dXK"), (9, "dlast_eta")):
        assert torch.equal(torch.cat([g1[i], g2[i]], dim=2), gw[i]), n
    for i, n in ((0, "dln_w"), (1, "dln_b")):
        assert O.rel_err((g1[i] + g2[i]).cpu(), gw[i].cpu()) < 1e-5, n


def test_per_group_backward_equals_persistent_per_batch_element():
    """The per-group K-side mode (one K-side launch per checkpoint group, ordered by host events; taken when 2*B*H + 16
    exceeds the SM count) against the persistent mode.  H is chosen from the SM count so that B = 2 runs per group and
    B = 1 runs persistent; NC = 37, G = 4 reuses the recompute ring and ends in a partial group.  Every sequence is
    independent, so the B = 2 backward equals the two B = 1 backwards bit for bit, except d ln_w / d ln_b, whose sums
    over B and over the launches run in a different order."""
    if os.environ.get("TTT_B200_PERSISTENT", "1") == "0":
        pytest.skip("TTT_B200_PERSISTENT=0 forces the per-group mode for every batch size")
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    H, NC, G = (sms - 16) // 2, 37, 4
    assert tt.backward_is_persistent(H, sms) and not tt.backward_is_persistent(2 * H, sms)
    d = _bench_like_inputs(2, H, NC, seed=7)
    state = [d[n] for n in ("W1", "b1", "W2", "b2")]
    fw = _forward(d, slice(0, NC), state, G)
    both = _backward(fw, d, slice(0, NC), G)
    out, ck, last, inputs = fw
    one = []
    for b in range(2):
        pick = lambda t: t[b:b + 1].contiguous()
        fw_b = (pick(out), [pick(c) for c in ck], [pick(w) for w in last], [pick(t) for t in inputs[:4]] + list(inputs[4:]))
        one.append(_backward(fw_b, {"dOut": pick(d["dOut"])}, slice(0, NC), G))
    torch.cuda.synchronize()
    for i, n in enumerate(("dW1", "db1", "dW2", "db2", "dXQ", "dXV", "dXK", "dlast_eta"), start=2):
        assert torch.equal(torch.cat([one[0][i], one[1][i]]), both[i]), n
    for i, n in ((0, "dln_w"), (1, "dln_b")):
        assert O.rel_err((one[0][i] + one[1][i]).cpu(), both[i].cpu()) < 1e-5, n


def test_reference_43_argument_backward_matches_simple():
    """test_time_training.ttt_backward with the reference's buffer contract (mlp_tk.py:192-260): 16 re-materialisation
    buffers (ignored), zeroed gradient outputs written in place."""
    B, H, NC, G = 2, 3, 10, 4
    d = _bench_like_inputs(B, H, NC, seed=6)
    state = [d[n] for n in ("W1", "b1", "W2", "b2")]
    out, ck, last, (q, k, v, le, lw, lb) = _forward(d, slice(0, NC), state, G)
    ref = tt.ttt_backward_simple(q, k, v, le, lw, lb, *ck, d["dOut"], G)
    dev, f32, bf = q.device, torch.float32, torch.bfloat16
    z = lambda *s, dt=f32: torch.zeros(*s, device=dev, dtype=dt)
    remat = [z(B, H, 64, 256), z(B, H, 1, 256), z(B, H, 256, 64), z(B, H, 1, 64)] + [z(1) for _ in range(12)]
    ups = [z(B, H, 64, 256), z(B, H, 1, 256), z(B, H, 256, 64), z(B, H, 1, 64)]
    g_lw, g_lb = z(B, H, 1, 64), z(B, H, 1, 64)
    gW = [z(B, H, 64, 256), z(B, H, 1, 256), z(B, H, 256, 64), z(B, H, 1, 64)]
    g_eta = z(B, H, NC, 64, 1, dt=bf)
    gq, gk, gv = z(B, H, NC, 64, 64, dt=bf), z(B, H, NC, 64, 64, dt=bf), z(B, H, NC, 64, 64, dt=bf)
    tt.ttt_backward(q, k, v, le, lw, lb, *ck, out, *remat, *ups, d["dOut"], g_lw, g_lb, *gW, g_eta, gq, gk, gv, G)
    torch.cuda.synchronize()
    assert torch.equal(g_lw.sum(0).reshape(H, 64), ref[0]) and torch.equal(g_lb.sum(0).reshape(H, 64), ref[1])
    for a, b in zip(gW, ref[2:6]):
        assert torch.equal(a, b)
    assert torch.equal(gq, ref[6]) and torch.equal(gv, ref[7]) and torch.equal(gk, ref[8]) and torch.equal(g_eta, ref[9])
