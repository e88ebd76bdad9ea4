"""Generate tests/golden/*.pt by RUNNING THE UNMODIFIED REFERENCE (a checkout of the original ttt-video-dit project).

    TORCHDYNAMO_DISABLE=1 TTT_VIDEO_DIT_ROOT=<checkout> python oracle/make_golden.py \
        [integration_patch|sampling|transformer_layer|process_input|layer]

Each fixture holds the reference's outputs (fp64, CPU, true eager) for seeded inputs that
``oracle.ttt_oracle.make_inputs`` regenerates bit-identically from the stored seed; an input
checksum guards against RNG drift.  The script also asserts that the oracle restatement agrees
with the reference before anything is written, so a committed fixture == "oracle pinned".

Reference entry points exercised (file:line in the checkout):
  ttt/models/ssm/ops/ttt_mlp.py:70      ttt_mlp      (+ torch autograd => gradient oracle)
  ttt/models/ssm/ops/ttt_linear.py:57   ttt_linear
  ttt/models/cogvideo/dit.py:224-266    SeqModelingBlock._ssm_forward (gate / flip / reverse)
  ttt/models/cogvideo/dit.py:163-211    SeqModelingBlock._attn_forward (local attention)
  ttt/models/cogvideo/utils.py:460-492  DiscreteDenoiser.forward (per-element guidance loop)
  integration/ttt_video_dit_b200.patch  applied to the checkout (hashes of the lines it replaces, CPU path unchanged)
"""
import os
import sys

os.environ.setdefault("TORCHDYNAMO_DISABLE", "1")
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
REF = os.environ.get("TTT_VIDEO_DIT_ROOT")
if REF:
    sys.path.insert(0, REF)

import torch

from oracle import ttt_oracle as O

GOLD = os.path.join(ROOT, "tests", "golden")
os.makedirs(GOLD, exist_ok=True)
torch.set_grad_enabled(True)


def checksum(d):
    return {k: float(v.double().abs().sum()) for k, v in d.items()}


def gen_mlp():
    from ttt.models.ssm.ops import ttt_mlp
    cfgs = [dict(B=1, H=2, NC=3, seed=0), dict(B=2, H=3, NC=5, seed=1)]
    fx = []
    for c in cfgs:
        d = O.make_inputs(c["B"], c["H"], c["NC"], CS=64, Fd=64, seed=c["seed"], dtype=torch.float64)
        ins = [d[k].clone().requires_grad_(True) for k in ("ln_w", "ln_b", "W1", "b1", "W2", "b2", "XQ", "XV", "XK", "eta")]
        lw, lb, w1, b1, w2, b2, q, v, k, e = ins
        out = ttt_mlp(k, q, v, e, lw, lb, w1, b1, w2, b2, 2)       # reference, checkpoint group 2
        out_op = out.permute(0, 3, 1, 2, 4)                         # ttt_layer.py:456 inverse -> [B,H,NC,CS,F]
        out_op.backward(d["dOut"])
        grads = [t.grad.clone() for t in ins]
        # pin the oracle
        (og, oo) = O.ttt_mlp_eager_grads(d["XQ"], d["XK"], d["XV"], d["eta"], d["ln_w"], d["ln_b"], d["W1"], d["b1"], d["W2"], d["b2"], d["dOut"])
        assert O.rel_err(oo, out_op.detach()) < 1e-12, "oracle eager fwd != reference"
        for a, b in zip(og, grads):
            assert O.rel_err(a, b) < 1e-10, "oracle eager grads != reference autograd"
        # primal form + analytic backward agree with the reference (row-uniform eta)
        le = d["eta"][:, :, :, -1, :, None]
        po, _, _ = O.ttt_mlp_primal_forward(d["XQ"], d["XK"], d["XV"], le, d["ln_w"], d["ln_b"], d["W1"], d["b1"], d["W2"], d["b2"], 2)
        assert O.rel_err(po, out_op.detach()) < 1e-11, "primal fwd != reference"
        pb = O.ttt_mlp_primal_backward(d["XQ"], d["XK"], d["XV"], le, d["ln_w"], d["ln_b"], d["W1"], d["b1"], d["W2"], d["b2"], d["dOut"])
        names = ["dln_w", "dln_b", "dW1", "db1", "dW2", "db2", "dXQ", "dXV", "dXK"]
        for n, b in zip(names, grads[:9]):
            assert O.rel_err(pb[n], b) < 1e-9, f"analytic bwd {n} != reference autograd: {O.rel_err(pb[n], b)}"
        # eta: eager spreads d/d eta over all rows; TK puts it in the last row -- equal after summing rows (SURVEY 8c)
        assert O.rel_err(pb["dlast_eta"].squeeze(-1), grads[9].sum(dim=-2)) < 1e-9
        fx.append(dict(cfg=c, in_checksum=checksum(d), out=out_op.detach().float(),
                       grads=[g.float() for g in grads[:9]] + [grads[9].sum(dim=-2).float()]))  # d eta stored row-summed
        print("mlp", c, "ok")
    torch.save(fx, os.path.join(GOLD, "ttt_mlp_ref.pt"))


def gen_linear():
    from ttt.models.ssm.ops import ttt_linear
    cfgs = [dict(B=1, H=2, NC=6, seed=2), dict(B=2, H=2, NC=9, seed=3)]
    fx = []
    for c in cfgs:
        d = O.make_inputs(c["B"], c["H"], c["NC"], CS=16, Fd=64, seed=c["seed"], dtype=torch.float64, base_lr=1.0, linear=True)
        ins = [d[k].clone().requires_grad_(True) for k in ("ln_w", "ln_b", "W1", "b1", "XQ", "XV", "XK", "eta")]
        lw, lb, w1, b1, q, v, k, e = ins
        out = ttt_linear(k, q, v, e, lw, lb, w1, b1, 4)
        out_op = out.permute(0, 3, 1, 2, 4)
        out_op.backward(d["dOut"])
        grads = [t.grad.clone() for t in ins]
        og, oo = O.ttt_linear_eager_grads(d["XQ"], d["XK"], d["XV"], d["eta"], d["ln_w"], d["ln_b"], d["W1"], d["b1"], d["dOut"])
        assert O.rel_err(oo, out_op.detach()) < 1e-12
        for a, b in zip(og, grads):
            assert O.rel_err(a, b) < 1e-10
        le = d["eta"][:, :, :, -1, :, None]
        po, _ = O.ttt_linear_primal_forward(d["XQ"], d["XK"], d["XV"], le, d["ln_w"], d["ln_b"], d["W1"], d["b1"])
        assert O.rel_err(po, out_op.detach()) < 1e-11
        fx.append(dict(cfg=c, in_checksum=checksum(d), out=out_op.detach().float(),
                       grads=[g.float() for g in grads[:7]] + [grads[7].sum(dim=-2).float()]))
        print("linear", c, "ok")
    torch.save(fx, os.path.join(GOLD, "ttt_linear_ref.pt"))


def gen_block():
    """Gate/flip and local attention through the reference's SeqModelingBlock (small dims, fp64)."""
    from ttt.models.cogvideo.dit import SeqModelingBlock
    from ttt.models.cogvideo.utils import SequenceMetadata
    from ttt.models.configs import ModelConfig

    torch.manual_seed(0)
    E, NH, Hh, Ww, frames, TL, chunks = 128, 2, 4, 4, 25, 8, 2
    cfg = ModelConfig(model_dim=E, num_heads=NH, num_layers=1, ssm_layer="ttt_linear", mini_batch_size=16,
                      ttt_base_lr=1.0, latent_height=Hh, latent_width=Ww, compressed_num_frames=frames, adapter_method="sft")
    blk = SeqModelingBlock(cfg).double()
    with torch.no_grad():
        for n, p in blk.named_parameters():
            if "ssm." in n:
                continue
            p.copy_(torch.randn_like(p) * (0.3 if p.dim() == 1 else 0.08))
        blk.q_norm.weight.add_(1.0); blk.k_norm.weight.add_(1.0)
    tpf = Hh * Ww
    md = SequenceMetadata(text_length=TL, seq_text_length=TL * chunks, num_frames=frames, num_chunks=chunks,
                          tokens_per_frame=tpf, latent_height=Hh, latent_width=Ww, t_emb=torch.zeros(1, 8))
    md.init_multiscene_offsets()
    B = 2
    vid = torch.randn(B, frames * tpf, E, dtype=torch.float64)
    txt = torch.randn(B, TL * chunks, E, dtype=torch.float64)

    # --- local attention (dit.py:163-211)
    with torch.no_grad():
        attn_ref = blk._attn_forward(vid, txt, md)
    P = {k: v.detach().clone() for k, v in blk.state_dict().items() if not k.startswith("ssm.") and "gating" not in k}
    sin, cos = O.rope3d_tables(Hh, Ww, frames, E // NH)
    mine = O.local_attention_block(vid, txt, {k: v for k, v in P.items()}, NH, TL, tpf, chunks, cfg.attn_length,
                                   cfg.prefix_temporal_length, sin.double(), cos.double(), cfg.layer_norm_eps)
    assert O.rel_err(mine, attn_ref) < 1e-10, O.rel_err(mine, attn_ref)
    print("attention ok")

    # --- gate / flip (dit.py:213-266) with an order-sensitive stub in place of the TTT layer
    class Stub(torch.nn.Module):
        def forward(self, x, seq_metadata):
            return torch.cumsum(x, dim=1) * 0.01 + torch.roll(x, 1, dims=-1) * 0.5
    blk.ssm = Stub()
    emb = torch.cat((txt, vid), dim=1)
    with torch.no_grad():
        ssm_ref = blk._ssm_forward(emb.clone(), md)
    al = {k: v.detach().clone() for k, v in blk.state_dict().items() if "gating" in k}
    stub = Stub()
    mine = O.ssm_bidirectional(emb.clone(), lambda x: stub(x, None), TL * chunks, chunks, True,
                               al["forward_ssm_gating_text.gating_alpha"], al["forward_ssm_gating_video.gating_alpha"],
                               al["backward_ssm_gating_text.gating_alpha"], al["backward_ssm_gating_video.gating_alpha"])
    assert O.rel_err(mine, ssm_ref) < 1e-12, O.rel_err(mine, ssm_ref)
    print("gate/flip ok")
    torch.save(dict(cfg=dict(E=E, NH=NH, Hh=Hh, Ww=Ww, frames=frames, TL=TL, chunks=chunks, B=B,
                             attn_length=cfg.attn_length, prefix=cfg.prefix_temporal_length, ln_eps=cfg.layer_norm_eps),
                    vid=vid.float(), txt=txt.float(), P={k: v.float() for k, v in P.items()},
                    alphas={k: v.float() for k, v in al.items()},
                    attn_ref=attn_ref.float(), ssm_ref=ssm_ref.float()),
               os.path.join(GOLD, "seq_block_ref.pt"))


def gen_process_input():
    """TTTBase.process_input (ttt_layer.py:252-306) through the reference's own module, single- and multi-scene."""
    from ttt.models.cogvideo.utils import SequenceMetadata
    from ttt.models.configs import ModelConfig
    from ttt.models.ssm.ttt_layer import TTTLinear
    from ttt.models.ssm.utils import precompute_freqs_cis_3d

    torch.manual_seed(0)
    out = []
    for (frames, TL, chunks) in ((13, 16, 1), (25, 8, 2)):
        E, NH, Hh, Ww, CS = 128, 2, 4, 4, 16
        cfg = ModelConfig(model_dim=E, num_heads=NH, num_layers=1, ssm_layer="ttt_linear", mini_batch_size=CS,
                          ttt_base_lr=1.0, latent_height=Hh, latent_width=Ww, compressed_num_frames=frames, adapter_method="sft")
        m = TTTLinear(cfg, use_kernel=False).double()
        with torch.no_grad():
            for n, p_ in m.named_parameters():
                p_.copy_(torch.randn_like(p_) * (0.3 if p_.dim() <= 2 and "ttt_norm" in n else 0.08))
            m.ttt_norm_weight.add_(1.0)
        tpf = Hh * Ww
        md = SequenceMetadata(text_length=TL, seq_text_length=TL * chunks, num_frames=frames, num_chunks=chunks,
                              tokens_per_frame=tpf, latent_height=Hh, latent_width=Ww, t_emb=torch.zeros(1, 8))
        if chunks > 1:
            md.init_multiscene_offsets()
        B, L = 1, TL * chunks + frames * tpf
        assert L % CS == 0
        X = torch.randn(B, L, E, dtype=torch.float64)
        fc = precompute_freqs_cis_3d(E // NH, Hh, Ww, frames)
        with torch.no_grad():
            ref = m.process_input(X, fc, md)
            q0, k0, v0 = (lin(X).reshape(B, L, NH, E // NH) for lin in (m.wq, m.wk, m.wv))
            logit = torch.einsum("blc,hdc->blh", X, m.learnable_ttt_lr_weight) + m.learnable_ttt_lr_bias.reshape(1, 1, -1)
        cos, sin = O.ttt_rope_tables(Hh, Ww, frames, E // NH)
        assert torch.allclose(torch.complex(cos, sin), fc, atol=1e-6)
        idx = O.interleave_index(L, TL, chunks, md.init_offset) if chunks > 1 else None
        mine = O.ttt_process_input(q0, k0, v0, logit, cos.double(), sin.double(), m.ttt_norm_weight.detach(),
                                   m.ttt_norm_bias.detach(), TL * chunks, cfg.ttt_base_lr, CS, idx)
        for a, n in zip(mine, ("XQ", "XK", "XV", "eta")):
            assert O.rel_err(a, ref[n]) < 1e-6, (n, O.rel_err(a, ref[n]))
        # output side (ttt_layer.py:324-331): post_norm, then undo_interleave (moved before the per-token wo Linear)
        Oop = torch.randn(B, NH, L // CS, CS, E // NH, dtype=torch.float64)
        with torch.no_grad():
            pn = m.post_norm(Oop.permute(0, 2, 3, 1, 4).reshape(B, L, E))
            ep_ref = m.undo_interleave(pn, md) if chunks > 1 else pn
            wo_then_undo = m.undo_interleave(m.wo(pn), md) if chunks > 1 else m.wo(pn)
            assert O.rel_err(m.wo(ep_ref), wo_then_undo) < 1e-12  # the permutation commutes with wo
        uidx = O.undo_interleave_index(L, TL, chunks, md.init_offset, md.base_offset) if chunks > 1 else None
        mine_ep = O.ttt_output_epilogue(Oop, m.post_norm.weight.detach(), m.post_norm.bias.detach(), 1e-6, uidx)
        assert O.rel_err(mine_ep, ep_ref) < 1e-10, O.rel_err(mine_ep, ep_ref)
        out.append(dict(cfg=dict(E=E, NH=NH, Hh=Hh, Ww=Ww, frames=frames, TL=TL, chunks=chunks, CS=CS, B=B, L=L,
                                 base_lr=cfg.ttt_base_lr, init_offset=md.init_offset, base_offset=md.base_offset),
                        ep_in=Oop.float(), ep_ref=ep_ref.float(), pn_w=m.post_norm.weight.detach().float(),
                        pn_b=m.post_norm.bias.detach().float(),
                        q0=q0.float(), k0=k0.float(), v0=v0.float(), logit=logit.float(),
                        ln_w=m.ttt_norm_weight.detach().float(), ln_b=m.ttt_norm_bias.detach().float(),
                        ref={n: ref[n].float() for n in ("XQ", "XK", "XV")}, ref_last_eta=ref["eta"][:, :, :, -1, :].float()))
    print("process_input ok")
    torch.save(out, os.path.join(GOLD, "process_input_ref.pt"))


def gen_layer():
    """Whole TTT layer forward through the reference modules in eager mode (TTTMLP / TTTLinear, use_kernel=False),
    single scene (uniform eta rows: the eager dual form equals the kernels' last-row form, SURVEY trap #1)."""
    from ttt.models.cogvideo.utils import SequenceMetadata
    from ttt.models.configs import ModelConfig
    from ttt.models.ssm.ttt_layer import TTTLinear, TTTMLP
    from ttt.models.ssm.utils import precompute_freqs_cis_3d

    torch.manual_seed(0)
    out = []
    for kind, cls, CS, lr in (("ttt_mlp", TTTMLP, 64, 0.1), ("ttt_linear", TTTLinear, 16, 1.0)):
        E, NH, Hh, Ww, frames, TL = 128, 2, 4, 4, 13, 48
        cfg = ModelConfig(model_dim=E, num_heads=NH, num_layers=1, ssm_layer=kind, mini_batch_size=CS, ttt_base_lr=lr,
                          latent_height=Hh, latent_width=Ww, compressed_num_frames=frames, adapter_method="sft",
                          scan_checkpoint_group_size=2)
        m = cls(cfg, use_kernel=False).double()
        with torch.no_grad():
            for n, p_ in m.named_parameters():
                if n in ("W1", "W2"):
                    p_.copy_(torch.randn_like(p_) * 0.02)
                elif n in ("b1", "b2"):
                    p_.zero_()
                else:
                    p_.copy_(torch.randn_like(p_) * 0.08)
            m.ttt_norm_weight.add_(1.0); m.post_norm.weight.add_(1.0)
        tpf = Hh * Ww
        md = SequenceMetadata(text_length=TL, seq_text_length=TL, num_frames=frames, num_chunks=1, tokens_per_frame=tpf,
                              latent_height=Hh, latent_width=Ww, t_emb=torch.zeros(1, 8))
        B, L = 2, TL + frames * tpf
        assert L % CS == 0
        X = torch.randn(B, L, E, dtype=torch.float64, requires_grad=True)
        fc = precompute_freqs_cis_3d(E // NH, Hh, Ww, frames)
        ref = m(X, fc, md)
        gout = torch.randn(B, L, E, dtype=torch.float64)
        ref.backward(gout)  # autograd through the reference's eager layer
        grads = {n: p_.grad.detach().float() for n, p_ in m.named_parameters()}
        grads["X"] = X.grad.detach().float()
        out.append(dict(kind=kind, cfg=dict(E=E, NH=NH, Hh=Hh, Ww=Ww, frames=frames, TL=TL, CS=CS, B=B, L=L, base_lr=lr, group=2),
                        X=X.detach().float(), P={k: v.detach().float() for k, v in m.state_dict().items()},
                        ref=ref.detach().float(), gout=gout.float(), grads=grads))
    print("layer ok")
    torch.save(out, os.path.join(GOLD, "ttt_layer_ref.pt"))


def gen_transformer_layer():
    """The reference's whole ``TransformerLayer`` (adaLN shell + SeqModelingBlock: local attention, bidirectional gated
    TTT-MLP, eager scan + autograd; dit.py:281-382), single scene and THREE scenes, fp64 on CPU.

    Multi-scene eta semantics (SURVEY trap #1): ``interleave`` permutes the eta rows, the eager dual form reads the full
    [CS, CS] eta (ops/ttt_mlp.py:40-46) while the native kernel path reads only the last row (mlp_tk.py:105).  Both are
    recorded: ``ref`` / ``grads`` with the rows forced to the last row (what ``use_kernel=True`` computes: the semantics the
    B200 kernels implement) and ``ref_full_eta`` as the module runs it eagerly, so the test can state the distance."""
    import ttt.models.ssm.ttt_layer as ref_layer
    from ttt.models.cogvideo.dit import TransformerLayer
    from ttt.models.cogvideo.utils import SequenceMetadata
    from ttt.models.configs import ModelConfig

    eager_mlp = ref_layer.ttt_mlp

    def last_row_eta(XK, XQ, XV, eta, *rest):
        return eager_mlp(XK, XQ, XV, eta[:, :, :, -1:, :].expand_as(eta).contiguous(), *rest)

    out = []
    for frames, TL, chunks in ((13, 48, 1), (37, 16, 3)):
        torch.manual_seed(100 + chunks)
        E, NH, Hh, Ww, TE = 128, 2, 4, 4, 32
        cfg = ModelConfig(model_dim=E, num_heads=NH, num_layers=1, ssm_layer="ttt_mlp", mini_batch_size=64, ttt_base_lr=0.1,
                          latent_height=Hh, latent_width=Ww, compressed_num_frames=frames, adapter_method="sft",
                          scan_checkpoint_group_size=2, time_embed_dim=TE)
        layer = TransformerLayer(cfg).double()
        layer.seq_modeling_block.ssm.ttt.use_kernel = False
        layer.seq_modeling_block.ssm.init_freqs()
        with torch.no_grad():
            for n, p_ in layer.named_parameters():
                if n.endswith((".W1", ".W2")):
                    p_.copy_(torch.randn_like(p_) * 0.02)
                elif n.endswith((".b1", ".b2")):
                    p_.zero_()
                elif "gating_alpha" in n:
                    p_.copy_(0.1 + 0.05 * torch.randn_like(p_))
                else:
                    p_.copy_(torch.randn_like(p_) * (0.2 if p_.dim() == 1 else 0.06))
            for m in (layer.pre_seq_layernorm, layer.pre_mlp_layernorm, layer.seq_modeling_block.q_norm, layer.seq_modeling_block.k_norm,
                      layer.seq_modeling_block.ssm.ttt.post_norm):
                m.weight.add_(1.0)
            layer.seq_modeling_block.ssm.ttt.ttt_norm_weight.add_(1.0)
        tpf = Hh * Ww
        B, Lv, Lt = 2, frames * tpf, TL * chunks
        assert (Lv + Lt) % 64 == 0
        t_emb = torch.randn(B, TE, dtype=torch.float64)
        md = SequenceMetadata(text_length=TL, seq_text_length=Lt, num_frames=frames, num_chunks=chunks, tokens_per_frame=tpf,
                              latent_height=Hh, latent_width=Ww, t_emb=t_emb)
        md.init_multiscene_offsets()
        vid = torch.randn(B, Lv, E, dtype=torch.float64, requires_grad=True)
        txt = torch.randn(B, Lt, E, dtype=torch.float64, requires_grad=True)
        with torch.no_grad():
            v_full, t_full = layer(vid, txt, md)
        blk_out = {}
        hook = layer.seq_modeling_block.register_forward_hook(lambda m, i, o: blk_out.update(vid=o[0].detach(), txt=o[1].detach(), x_vid=i[0].detach(), x_txt=i[1].detach()))
        ref_layer.ttt_mlp = last_row_eta
        try:
            v_ref, t_ref = layer(vid, txt, md)
            gv = torch.randn_like(v_ref); gt = torch.randn_like(t_ref)
            (v_ref * gv).sum().add((t_ref * gt).sum()).backward()
        finally:
            ref_layer.ttt_mlp = eager_mlp
            hook.remove()
        keep = ("pre_seq_adaLN_modulation.1.weight", "pre_seq_layernorm.weight", "seq_modeling_block.q.weight", "seq_modeling_block.o.bias",
                "seq_modeling_block.k_norm.weight", "seq_modeling_block.ssm.ttt.W1", "seq_modeling_block.ssm.ttt.b2",
                "seq_modeling_block.ssm.ttt.wq.weight", "seq_modeling_block.ssm.ttt.ttt_norm_weight",
                "seq_modeling_block.ssm.ttt.learnable_ttt_lr_weight", "seq_modeling_block.ssm.ttt.post_norm.weight",
                "seq_modeling_block.forward_ssm_gating_video.gating_alpha", "seq_modeling_block.backward_ssm_gating_text.gating_alpha",
                "mlp.layer1.weight", "mlp.layer2.bias", "pre_mlp_adaLN_modulation.1.bias")
        named = dict(layer.named_parameters())
        f = lambda t: t.detach().float()
        out.append(dict(cfg=dict(E=E, NH=NH, Hh=Hh, Ww=Ww, frames=frames, TL=TL, chunks=chunks, B=B, TE=TE, CS=64, base_lr=0.1, group=2,
                                 attn_length=cfg.attn_length, prefix=cfg.prefix_temporal_length, ln_eps=cfg.layer_norm_eps),
                        vid=f(vid), txt=f(txt), t_emb=f(t_emb), P={k: f(v) for k, v in layer.state_dict().items()},
                        ref_vid=f(v_ref), ref_txt=f(t_ref), ref_full_eta_vid=f(v_full), ref_full_eta_txt=f(t_full),
                        block_in_vid=f(blk_out["x_vid"]), block_in_txt=f(blk_out["x_txt"]), block_vid=f(blk_out["vid"]), block_txt=f(blk_out["txt"]),
                        gout_vid=f(gv), gout_txt=f(gt), grads=dict({k: f(named[k].grad) for k in keep}, vid=f(vid.grad), txt=f(txt.grad)),
                        eta_semantics_distance=O.rel_err(torch.cat((t_full, v_full), 1), torch.cat((t_ref, v_ref), 1))))
        print(f"transformer layer ({chunks} scene(s)) ok; full-eta vs last-row-eta output distance = {out[-1]['eta_semantics_distance']:.3e}")
    torch.save(out, os.path.join(GOLD, "transformer_layer_ref.pt"))


def sampling_network(calls):
    """Stand-in for the DiT in the denoiser fixture: per-element results do not depend on the batching; records the batch size
    of every call.  tests/test_sampling_host.py restates it."""
    def network(x, crossattn, c_noise):
        calls.append(x.shape[0])
        return torch.tanh(x) * (1 + 0.01 * c_noise.float().reshape(-1, 1, 1, 1, 1)) + crossattn.mean(dim=(1, 2)).reshape(-1, 1, 1, 1, 1)
    return network


def gen_sampling():
    """The reference's DiscreteDenoiser.forward (utils.py:460-492) on a classifier-free-guidance pair, fp32 on CPU: its output,
    the batch size of each network call it makes, and its discretisation table."""
    from ttt.models.cogvideo import utils as RU
    torch.manual_seed(0)
    calls = []
    ref = RU.DiscreteDenoiser.__new__(RU.DiscreteDenoiser)
    torch.nn.Module.__init__(ref)
    ref.scaling = RU.VideoScaling()
    ref.sigmas = RU.ZeroSNRDDPMDiscretization()(1000, do_append_zero=False, device="cpu", flip=True)
    ref.quantize_c_noise, ref.network, ref.dtype = True, sampling_network(calls), torch.float32
    x = torch.randn(2, 3, 4, 5, 6)
    crossattn = torch.randn(2, 7, 8)
    step = 400
    with torch.no_grad():
        out = ref(x, ref.sigmas[[step, step]].clone(), {"crossattn": crossattn}, idx=ref.sigmas[[step, step]])
    print("sampling ok, network calls", calls)
    torch.save(dict(sigmas=ref.sigmas.clone(), x=x, crossattn=crossattn, step=step, calls=calls, out=out),
               os.path.join(GOLD, "sampling_ref.pt"))


PATCH_SCRIPT = r'''
import sys, torch
torch.manual_seed(0)
from ttt.models.cogvideo.dit import SeqModelingBlock
from ttt.models.cogvideo.utils import SequenceMetadata
from ttt.models.configs import ModelConfig
import ttt.models.ssm.ttt_layer as TL
print("TKMLP", TL.TkMLP.__module__, "LINEAR", TL.TritonLinear.__module__)
E, NH, Hh, Ww, frames, T, chunks = 128, 2, 4, 4, 25, 8, 2
cfg = ModelConfig(model_dim=E, num_heads=NH, num_layers=1, ssm_layer="ttt_linear", mini_batch_size=16, ttt_base_lr=1.0,
                  latent_height=Hh, latent_width=Ww, compressed_num_frames=frames, adapter_method="sft")
blk = SeqModelingBlock(cfg).double()
class Stub(torch.nn.Module):
    def forward(self, x, seq_metadata):
        return torch.cumsum(x, dim=1) * 0.01 + torch.roll(x, 1, dims=-1) * 0.5
blk.ssm = Stub()
md = SequenceMetadata(text_length=T, seq_text_length=T * chunks, num_frames=frames, num_chunks=chunks, tokens_per_frame=Hh * Ww,
                      latent_height=Hh, latent_width=Ww, t_emb=torch.zeros(1, 8))
md.init_multiscene_offsets()
vid = torch.randn(2, frames * Hh * Ww, E, dtype=torch.float64)
txt = torch.randn(2, T * chunks, E, dtype=torch.float64)
with torch.no_grad():
    a = blk._attn_forward(vid, txt, md)
    s = blk._ssm_forward(torch.cat((txt, vid), dim=1), md)
print("SUM %.12e %.12e" % (a.double().sum().item(), s.double().sum().item()))
'''


def gen_integration_patch():
    """integration/ttt_video_dit_b200.patch against the checkout: `patch -p1` applies it without offset or fuzz, the patched
    tree binds TkMLP / TritonLinear to this package, and a SeqModelingBlock (attention + gate/flip, fp64 on CPU) gives
    bit-identical results patched and stock.  Records the patch's sha256, for every hunk the sha256 of the lines it replaces
    in the checkout, and the two runs' results (tests/test_integration_patch.py)."""
    import json
    import shutil
    import subprocess
    import tempfile
    from oracle import patch_hunks
    patch_path = os.path.join(ROOT, "integration", "ttt_video_dit_b200.patch")
    text = open(patch_path).read()

    def run(pythonpath):
        env = dict(os.environ, TORCHDYNAMO_DISABLE="1", PYTHONPATH=os.pathsep.join(pythonpath))
        r = subprocess.run([sys.executable, "-c", PATCH_SCRIPT], capture_output=True, text=True, env=env, timeout=900)
        assert r.returncode == 0, r.stderr[-3000:]
        return [l for l in r.stdout.splitlines() if l.startswith(("TKMLP", "SUM"))]
    with tempfile.TemporaryDirectory() as tmp:
        shutil.copytree(os.path.join(REF, "ttt"), os.path.join(tmp, "ttt"))
        r = subprocess.run(["patch", "-p1", "--no-backup-if-mismatch", "-i", patch_path], cwd=tmp, capture_output=True, text=True)
        assert r.returncode == 0 and "offset" not in r.stdout and "fuzz" not in r.stdout, r.stdout + r.stderr
        patched = run([tmp, ROOT])
    stock = run([REF])
    assert patched[0] == "TKMLP ttt_video_dit_b200.mlp_tk LINEAR ttt_video_dit_b200.linear_triton", patched
    assert stock[0] == "TKMLP ttt.models.ssm.mlp_tk LINEAR ttt.models.ssm.linear_triton", stock
    assert patched[1] == stock[1], (patched, stock)
    files = {}
    for path, hunks in patch_hunks.parse(text).items():
        lines = open(os.path.join(REF, path)).read().splitlines()
        files[path] = [dict(old_start=h["old_start"], old_len=h["old_len"],
                            sha256=patch_hunks.digest(lines[h["old_start"] - 1:h["old_start"] - 1 + h["old_len"]])) for h in hunks]
        for h, rec in zip(hunks, files[path]):
            assert patch_hunks.digest(patch_hunks.pre_image(h)) == rec["sha256"], (path, h["old_start"])
    out = dict(patch_sha256=patch_hunks.digest(text.splitlines()), files=files, patched_binding=patched[0],
               stock_binding=stock[0], patched_sums=patched[1], stock_sums=stock[1])
    with open(os.path.join(GOLD, "integration_patch_ref.json"), "w") as f:
        json.dump(out, f, indent=1)
        f.write("\n")
    print("integration patch ok:", patched[1])


if __name__ == "__main__":
    assert REF and os.path.isdir(os.path.join(REF, "ttt")), "set TTT_VIDEO_DIT_ROOT to a checkout of the original project"
    if len(sys.argv) > 1 and sys.argv[1] == "integration_patch":
        gen_integration_patch()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "sampling":
        gen_sampling()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "transformer_layer":
        gen_transformer_layer()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "process_input":
        gen_process_input()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "layer":
        gen_layer()
        sys.exit(0)
    gen_mlp()
    gen_linear()
    gen_block()
    gen_process_input()
    gen_layer()
    gen_transformer_layer()
    gen_sampling()
    gen_integration_patch()
    for f in sorted(os.listdir(GOLD)):
        print(f, os.path.getsize(os.path.join(GOLD, f)))
