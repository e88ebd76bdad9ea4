"""GPU parity: TTT-MLP backward (trajectory + reverse kernels through the C-ABI) vs autograd through the eager oracle
(= torch autograd through ttt/models/ssm/ops/ttt_mlp.py, pinned by tests/golden).  Tolerance 1e-2 relative per tensor
(north_star); d eta is compared after summing the eager gradient over rows (SURVEY 8c)."""
import os

import pytest
import torch

from oracle import ttt_oracle as O
from ttt_video_dit_b200 import mlp_tk

pytestmark = pytest.mark.gpu
NAMES = ["d_ln_w", "d_ln_b", "dW1", "db1", "dW2", "db2", "dXQ", "dXV", "dXK", "d_eta"]


def run_fwd_bwd(d, G):
    dev = "cuda"
    bf = lambda t: t.to(torch.bfloat16).to(dev)
    leaf = lambda t: t.clone().to(dev).requires_grad_(True)
    prm = [leaf(d[k]) for k in ("ln_w", "ln_b", "W1", "b1", "W2", "b2")]
    q, v, k = [bf(d[n]).requires_grad_(True) for n in ("XQ", "XV", "XK")]
    e = bf(d["eta"])[:, :, :, -1, :].clone().requires_grad_(True)
    out = mlp_tk.ttt_mlp_op(*prm, q, v, k, e, G)
    out.backward(bf(d["dOut"]))
    torch.cuda.synchronize()
    return out, [t.grad for t in prm] + [q.grad, v.grad, k.grad, e.grad]


def oracle_grads(d):
    r = lambda t: t.to(torch.bfloat16).float()
    grads, out = O.ttt_mlp_eager_grads(r(d["XQ"]), r(d["XK"]), r(d["XV"]), r(d["eta"]), d["ln_w"], d["ln_b"],
                                       d["W1"], d["b1"], d["W2"], d["b2"], r(d["dOut"]))
    grads[9] = grads[9].sum(dim=-2)  # eager spreads d eta over the CS rows; the op reports it per token
    return out, grads


def errors(d, G):
    out, g = run_fwd_bwd(d, G)
    ref_out, rg = oracle_grads(d)
    errs = {"out": O.rel_err(out.float().cpu(), ref_out)}
    for n, a, b in zip(NAMES, g, rg):
        errs[n] = O.rel_err(a.float().cpu().reshape(b.shape), b)
    return errs


@pytest.mark.parametrize("B,H,NC,G", [(1, 1, 1, 1), (1, 2, 3, 2), (2, 2, 7, 3), (1, 3, 20, 16)])
def test_backward_matches_autograd_of_eager(B, H, NC, G):
    d = O.make_inputs(B, H, NC, seed=40 + NC)
    errs = errors(d, G)
    bad = {k: v for k, v in errs.items() if not (v < 1e-2)}
    assert not bad, f"rel errors above 1e-2: {bad} (all: {errs})"


def test_backward_many_launch_units():
    # 10 checkpoint groups of 4 -> 10 recompute units (one group each) through the 3-slot ring: every slot is reused
    d = O.make_inputs(1, 2, 40, seed=45)
    errs = errors(d, 4)
    bad = {k: v for k, v in errs.items() if not (v < 1e-2)}
    assert not bad, f"rel errors above 1e-2: {bad} (all: {errs})"


def test_backward_golden_reference_fixture():
    fx = torch.load(os.path.join(os.path.dirname(__file__), "golden", "ttt_mlp_ref.pt"), weights_only=False)[1]
    c = fx["cfg"]
    d = O.make_inputs(c["B"], c["H"], c["NC"], seed=c["seed"])
    _, g = run_fwd_bwd(d, 2)
    for n, a, b in zip(NAMES, g, fx["grads"]):
        assert O.rel_err(a.float().cpu().reshape(b.shape), b) < 2e-2, n
