#!/usr/bin/env python
"""bench.py -- TTT hot path benchmark (contract: see task statement / DESIGN.md "Measurement").

A *step* is one pass of the TTT-MLP op (forward scan + backward scan) over one batch of synthetic token tensors for ONE
layer-direction of CogVideoX-5B (48 heads x 64, mini-batch 64, checkpoint group 16).

  N = 1 (default)   workload = the 63-second video of BASELINE.json's metric: NC = 5 487 mini-batches (L = 351 168 tokens),
                    B = 1.  Secondary key "nc804": the same at the 9-second length (the metric's other quoted point).
  N > 1 (torchrun)  the north-star multi-GPU mode: the sequence is SHARDED over the N ranks (contiguous mini-batch ranges,
                    ttt_video_dit_b200.seq_shard.ShardedTTTMLP); the only data-path collective is the NCCL send/recv of the
                    fp32 state {W1,b1,W2,b2} (forward) and of its gradient (backward) at the shard boundaries.  M = 8N
                    independent sequences are in flight so the serial chain is full (pipeline over sequences); secondary
                    keys: single-sequence latency through the chain, and plain data-parallel replicas.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--mode fwd|fwdbwd] [--nc 5487] [--batch 1] [--seqs M]
                    [--dump-outputs DIR]
    python bench.py --impl reference ...      # the reference's eager CPU path on the host cores

--dump-outputs DIR writes what the last timed step handed back to its caller as DIR/<name>.npy (float32): the op's output
`out` and, in fwd+bwd mode, the token gradients dXQ/dXK/dXV and the parameter gradients.  The inputs are seeded, so two builds
run with the same arguments can be compared array by array.  An array of more than DUMP_ELEMS elements is reduced to a fixed,
seeded sample of rows of its last dimension (the same rows for every array of the same shape).

value   = tokens/s with inputs resident in HBM (CUDA-event time, max over ranks, whole-job aggregate)
e2e     = same through the public op with HOST (pinned) inputs: H2D of q,k,v,eta(,dOut) + op + D2H of the op's output per
          step, copies placed beside the kernels on copy streams
roofline= algorithmic TTT FLOPs (7U fwd, +15U bwd per head per mini-batch, U = 2*64*64*256) / op time vs
          MEASURED_PEAKS.json bf16 peak
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark may run from a read-only tree and leaves nothing behind in it
os.environ.setdefault("TORCHDYNAMO_DISABLE", "1")

U_FLOP = 2 * 64 * 64 * 256
FWD_U, BWD_U = 7, 15
H_5B = 48
NC_63S, NC_9S, NC_3S = 5487, 804, 282
CPU_SAMPLE_NC = 64  # BASELINE.md section 3: time a prefix of >= 64 mini-batches, the scan cost is linear in NC
PARAM_NAMES = ("ln_w", "ln_b", "W1", "b1", "W2", "b2")
DUMP_ELEMS = 1 << 20  # per dumped array (4 MB in float32): at most 10 arrays stay well inside 64 MB
DUMP_SEED = 0


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10, help="timed steps (>= 1)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--mode", default="fwdbwd", choices=["auto", "fwd", "fwdbwd"])
    ap.add_argument("--nc", type=int, default=NC_63S, help="mini-batches per sequence (282 = 3 s, 804 = 9 s, 5487 = 63 s)")
    ap.add_argument("--batch", type=int, default=1)
    ap.add_argument("--heads", type=int, default=H_5B)
    ap.add_argument("--ckpt", type=int, default=16)
    ap.add_argument("--seqs", type=int, default=0, help="N>1: sequences in flight through the sharded chain (default 8N)")
    ap.add_argument("--parallel", default="auto", choices=["auto", "seqshard", "replicas"],
                    help="N>1: sequence-sharded chain (default) or independent data-parallel replicas")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the secondary keys (nc804 / latency / replicas)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's outputs as DIR/<name>.npy (un-sharded runs; rank 0)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    return args


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops", 1590.0), d.get("bf16_tflops_sustained", 1400.0), "measured (MEASURED_PEAKS.json)"
    return 1590.0, 1400.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons during the timed region."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.stop_flag = False

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        mhz = sorted(int(s[0]) for s in self.samples if s[0].isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(s[2 + i].lower().startswith("active") for s in self.samples if len(s) > 2 + i)]
        return {"sm_mhz": mhz[len(mhz) // 2] if mhz else None, "sm_max_mhz": int(self.samples[0][1]) if self.samples[0][1].isdigit() else None,
                "reasons": reasons, "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------------ CPU baseline
def usable_cores():
    return len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)


class CpuEager:
    """The reference's eager CPU path of the op on a bounded sample, as restated in oracle/ttt_oracle.py (kind "port"; the
    restatement is pinned to the reference's outputs by tests/test_oracle.py).  fp32, eta materialised [.., CS, CS] as the
    reference does (ttt_layer.py:288), autograd backward."""

    def __init__(self, heads, mode, sample_nc=CPU_SAMPLE_NC):
        import torch
        from oracle import ttt_oracle as O
        self.torch, self.mode, self.heads, self.nc = torch, mode, heads, sample_nc
        self.d = O.make_inputs(1, heads, sample_nc, seed=0)
        self.kind = "port"
        self.fn = lambda *a: O.ttt_mlp_eager(*a)[0]

    def once(self):
        torch, d = self.torch, self.d
        names = ("XK", "XQ", "XV", "eta", "ln_w", "ln_b", "W1", "b1", "W2", "b2")
        t0 = time.perf_counter()
        if self.mode == "fwd":
            with torch.no_grad():
                self.fn(*[d[n] for n in names])
        else:
            ins = [d[n].detach().clone().requires_grad_(True) for n in names]
            out = self.fn(*ins)  # [B,NC,CS,H,F]
            out.backward(d["dOut"].permute(0, 2, 3, 1, 4))
        return time.perf_counter() - t0

    def pick_threads(self):
        """Thread count at which this path is fastest on this host: the ops are small ([heads,64,256] batched matmuls), so
        'every core' is not the optimum (measured on the 128-core GPU host: 16 threads ~1.5-4 k tok/s, 128 threads 4-150
        tok/s).  Searched over 1..32 on an 8-mini-batch prefix (the per-mini-batch cost does not depend on the length)."""
        torch = self.torch
        cores = usable_cores()
        cands = sorted({c for c in (1, 2, 4, 8, 16, 32) if c <= cores})
        full, self.d = self.d, {k: (v[:, :, :8].contiguous() if v.dim() == 5 else v) for k, v in self.d.items()}
        try:
            return self._search(cands)
        finally:
            self.d = full

    def _search(self, cands):
        torch = self.torch
        best_n, best_dt = 1, None
        for n in cands:
            torch.set_num_threads(n)
            self.once()  # thread-pool start-up
            dt = min(self.once(), self.once())
            if best_dt is None or dt < best_dt:
                best_n, best_dt = n, dt
            elif dt > 2.0 * best_dt:
                break
        torch.set_num_threads(best_n)
        return best_n

    def describe(self, threads):
        return (f"first {self.nc} mini-batches ({self.nc * 64} tokens) x {self.heads} heads, fp32 eager dual form "
                f"(oracle port of ttt/models/ssm/ops/ttt_mlp.py), "
                f"{'fwd' if self.mode == 'fwd' else 'fwd + autograd bwd'}, {threads} threads = fastest of 1..{usable_cores()} usable cores, "
                f"median of the timed passes after one warm-up")


def cpu_baseline(heads, mode, reps=3):
    eager = CpuEager(heads, mode)
    threads = eager.pick_threads()
    eager.once()
    dts = sorted(eager.once() for _ in range(reps))
    dt = dts[len(dts) // 2]
    return {"value": eager.nc * 64 / dt, "unit": "tokens/s", "cores": usable_cores(), "threads": threads, "kind": eager.kind,
            "sample": eager.describe(threads), "seconds_per_pass": dt}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    mode = "fwd" if args.mode == "fwd" else "fwdbwd"
    eager = CpuEager(args.heads, mode)
    threads = eager.pick_threads()
    for _ in range(args.warmup):
        eager.once()
    dts = [eager.once() for _ in range(args.steps)]
    dt = sum(dts) / len(dts)
    tok_s = eager.nc * 64 / dt
    line = {
        "impl": "reference", "metric": f"video-tokens/sec TTT-MLP layer-direction ({'fwd+bwd' if mode == 'fwdbwd' else 'fwd'})",
        "value": tok_s, "unit": "tokens/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"CogVideoX-5B TTT-MLP op, {args.heads} heads x 64, mini-batch 64, NC={args.nc} "
                               f"(each step = the first {eager.nc} mini-batches; the scan is linear in NC)", "mode": mode},
        "cpu_baseline": {"value": tok_s, "unit": "tokens/s", "cores": usable_cores(), "threads": threads, "kind": eager.kind,
                         "sample": eager.describe(threads)},
        "e2e": {"value": tok_s, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------ GPU arms
def synth(torch, dev, B, H, NC, seed, want_dout=True):
    """Synthetic inputs of SURVEY 8d, generated on the device (63 s = 1.1 G elements per tensor: too slow on the host)."""
    g = torch.Generator(device=dev).manual_seed(seed)
    rn = lambda *s: torch.randn(*s, generator=g, device=dev)
    nrm = torch.nn.functional.normalize
    q = nrm(rn(B, H, NC, 64, 64), dim=-1).to(torch.bfloat16)
    k = nrm(rn(B, H, NC, 64, 64), dim=-1).to(torch.bfloat16)
    v = rn(B, H, NC, 64, 64).to(torch.bfloat16)
    e = ((0.1 / 64) * torch.sigmoid(rn(B, H, NC, 64)) / 64).to(torch.bfloat16)  # the one eta row the scan reads
    go = rn(B, H, NC, 64, 64).to(torch.bfloat16) if want_dout else None
    return q, k, v, e, go


def synth_params(torch, dev, B, H, seed=99):
    g = torch.Generator(device=dev).manual_seed(seed)
    rn = lambda *s: torch.randn(*s, generator=g, device=dev)
    ln_w, ln_b = 1 + 0.1 * rn(H, 64), 0.1 * rn(H, 64)
    W1 = (0.02 * rn(H, 64, 256)).unsqueeze(0).repeat(B, 1, 1, 1).contiguous()
    W2 = (0.02 * rn(H, 256, 64)).unsqueeze(0).repeat(B, 1, 1, 1).contiguous()
    return [ln_w, ln_b, W1, torch.zeros(B, H, 1, 256, device=dev), W2, torch.zeros(B, H, 1, 64, device=dev)]


def timed(torch, dist, world, fn, steps, warmup, sampler=None):
    """W warm-up steps, then K steps between barrier + synchronize, CUDA events on the launching stream; returns ms."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    if sampler is not None:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    if sampler is not None:
        sampler.stop_flag = True
    return e0.elapsed_time(e1)


def max_over_ranks(torch, dist, world, dev, *vals):
    t = torch.tensor(list(vals), device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return [float(x) for x in t]


def single_gpu_op(torch, mlp_tk, params, mode, G, outputs=None):
    def step(q, k, v, e, go):
        """One pass of the hot path through the public op (TkMLP.apply-compatible entry, last-row eta form).  `outputs`, when
        given, holds what the pass hands back to its caller until the next pass starts."""
        if outputs is not None:
            outputs.clear()
        if mode == "fwdbwd":
            for p in params:  # each pass leaves its own parameter gradients, as a training step does
                p.grad = None
            q = q.detach().requires_grad_(True); k = k.detach().requires_grad_(True); v = v.detach().requires_grad_(True)
        out = mlp_tk.ttt_mlp_op(*params, q, v, k, e, G)
        if mode == "fwdbwd":
            out.backward(go)
        if outputs is not None:
            outputs["out"] = out
            if mode == "fwdbwd":
                outputs.update(dXQ=q.grad, dXK=k.grad, dXV=v.grad, **{"d" + n: p.grad for n, p in zip(PARAM_NAMES, params)})
        return out
    return step


def dump_outputs(torch, outputs, path):
    """Each array as path/<name>.npy in float32; one of more than DUMP_ELEMS elements as the rows (of its last dimension) at
    DUMP_ELEMS // last_dim indices drawn with a fixed seed, in ascending order."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    total = 0
    for name, t in outputs.items():
        t = t.detach().reshape(-1, t.shape[-1])
        if t.numel() > DUMP_ELEMS:
            g = torch.Generator().manual_seed(DUMP_SEED)
            rows = torch.randint(t.shape[0], (DUMP_ELEMS // t.shape[1],), generator=g).sort().values
            t = t[rows.to(t.device)]
        a = t.float().cpu().numpy()
        np.save(os.path.join(path, name + ".npy"), a)
        total += a.nbytes
    assert total <= 64 << 20, total


def bench_replica(args, torch, dist, mlp_tk, world, rank, dev, mode, NC, with_e2e, steps, warmup, sampler=None, dump=None):
    """B sequences per GPU, un-sharded: the N = 1 workload, and the data-parallel-replica secondary key at N > 1.  `dump`: a
    directory that receives this rank's outputs of the last timed step."""
    B, H, G = args.batch, args.heads, args.ckpt
    params = synth_params(torch, dev, B, H)
    if mode == "fwdbwd":
        params = [p.requires_grad_(True) for p in params]
    q, k, v, e, go = synth(torch, dev, B, H, NC, 1234 + rank, mode == "fwdbwd")
    outputs = {} if dump else None
    step = single_gpu_op(torch, mlp_tk, params, mode, G, outputs)
    ms = timed(torch, dist, world, lambda: step(q, k, v, e, go), steps, warmup, sampler)
    if dump:
        dump_outputs(torch, outputs, dump)
        outputs.clear()
    res = {"ms_per_step": ms / steps, "tokens_per_step": B * NC * 64 * world,
           "launches": steps * mlp_tk.launches_per_call(mode)}
    if with_e2e:
        # end to end from pinned host memory.  Every step copies its own inputs host->device and its result device->host inside
        # the timed region; HostPipeline places H2D(i+1) and D2H(i-1) beside op(i) instead of in front of it.
        from ttt_video_dit_b200.host_stream import HostPipeline
        pin = lambda t: torch.empty(t.shape, dtype=t.dtype, pin_memory=True).copy_(t)
        host = [pin(t) if t is not None else None for t in (q, k, v, e, go)]
        host_out = torch.empty(B, H, NC, 64, 64, dtype=torch.bfloat16, pin_memory=True)
        h2d = sum(t.numel() * t.element_size() for t in host if t is not None)
        d2h = host_out.numel() * 2
        del q, k, v, go
        pipe = HostPipeline(dev)
        pipe.run((host for _ in range(2)), step, host_out)
        torch.cuda.synchronize()
        pipe.h2d_bytes = pipe.d2h_bytes = 0
        # as many steps as the device-timed region: the pipeline's fill (first H2D) and drain (last op + D2H) are inside the
        # timed region and are amortised over these steps only (63 s: 8.7 GB in + 2.2 GB out per step over PCIe)
        n_e2e = steps
        if world > 1:
            dist.barrier()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record()
        n = pipe.run((host for _ in range(n_e2e)), step, host_out)
        f1.record()
        torch.cuda.synchronize()
        assert n == n_e2e and pipe.h2d_bytes == h2d * n_e2e and pipe.d2h_bytes == d2h * n_e2e
        res.update(e2e_ms_per_step=f0.elapsed_time(f1) / n_e2e, h2d=h2d, d2h=d2h, e2e_steps=n_e2e)
    return res


_PAIRS = {}


def _pair_groups(seq_shard):
    """Two-rank NCCL communicators for the chain neighbours, created once per process (collective call)."""
    if "g" not in _PAIRS:
        _PAIRS["g"] = seq_shard.make_pair_groups()
    return _PAIRS["g"]


def bench_sharded(args, torch, dist, world, rank, dev, mode, NC, M, with_e2e, steps, warmup, sampler=None):
    """The sequence-sharded chain: this rank owns mini-batch range `rank` of each of the M sequences."""
    from ttt_video_dit_b200 import seq_shard, test_time_training as tt
    H, G = args.heads, args.ckpt
    s, e_ = seq_shard.partition_minibatches(NC, world)[rank]
    n_local = e_ - s
    ln_w, ln_b, W1, b1, W2, b2 = synth_params(torch, dev, 1, H)
    impl = seq_shard.CudaMLPRange(ln_w, ln_b, checkpoint_group_size=G)
    pairs = _pair_groups(seq_shard)
    stage = seq_shard.ShardedTTTMLP(impl, rank=rank, world=world, pair_groups=pairs)
    items, gouts = [], []
    for m in range(M):
        q, k, v, e, go = synth(torch, dev, 1, H, n_local, 5000 + 97 * m + rank, True)
        items.append((q, k, v, e)); gouts.append(go)

    def step():  # outputs / token gradients are dropped item by item: M sequences of results would not fit beside the inputs
        stage.forward(items, (W1, b1, W2, b2), collect=False)
        if mode == "fwdbwd":
            stage.backward(gouts, collect=False)
    ms = timed(torch, dist, world, step, steps, warmup, sampler)
    groups = (n_local + min(G, n_local) - 1) // min(G, n_local)
    per_item = tt.LAUNCHES_FWD + ((3 * groups + (1 if rank != world - 1 else 0)) if mode == "fwdbwd" else 0)
    res = {"ms_per_step": ms / steps, "tokens_per_step": M * NC * 64, "launches": steps * M * per_item}
    if with_e2e:
        # every step, every item: H2D of this rank's range of q,k,v,eta,dOut from pinned host memory on a copy stream (ahead of
        # the chain), D2H of the item's output range on a second copy stream.  The pinned source holds ONE item (synthetic
        # data); each of the M items is a separate copy into its own device buffers.
        s_in, s_out = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
        pin = lambda t: torch.empty(t.shape, dtype=t.dtype, pin_memory=True).copy_(t)
        host = [pin(t) for t in (*items[0], gouts[0])]
        host_out = torch.empty(host[0].shape, dtype=host[0].dtype, pin_memory=True)
        ev_in = [torch.cuda.Event() for _ in range(M)]
        ev_done = [torch.cuda.Event() for _ in range(M)]
        h2d = M * sum(t.numel() * t.element_size() for t in host)
        d2h = M * host_out.numel() * 2
        main = torch.cuda.current_stream(dev)

        class Feed:  # the stage's implementation with the copies around it
            def forward(self, q, k, v, le, st):
                m = self.m
                main.wait_event(ev_in[m])
                out, st_out, ctx = impl.forward(q, k, v, le, st)
                ev = torch.cuda.Event(); ev.record(main)
                with torch.cuda.stream(s_out):
                    s_out.wait_event(ev)
                    host_out.copy_(out, non_blocking=True)
                    out.record_stream(s_out)
                self.m += 1
                return out, st_out, ctx

            def backward(self, ctx, go, d_state):
                r = impl.backward(ctx, go, d_state)
                ev_done[self.mb].record(main)
                self.mb += 1
                return r
        feed = Feed()
        stage_e2e = seq_shard.ShardedTTTMLP(feed, rank=rank, world=world, pair_groups=pairs)

        def step_e2e(first=False):
            with torch.cuda.stream(s_in):
                for m in range(M):
                    if not first:
                        s_in.wait_event(ev_done[m])  # the previous step's backward has consumed item m's buffers
                    for dst, src in zip((*items[m], gouts[m]), host):
                        dst.copy_(src, non_blocking=True)
                    ev_in[m].record(s_in)
            feed.m = feed.mb = 0
            stage_e2e.forward(items, (W1, b1, W2, b2), collect=False)
            if mode == "fwdbwd":
                stage_e2e.backward(gouts, collect=False)
            else:
                for m in range(M):
                    ev_done[m].record(main)
            main.wait_stream(s_out)
        s_in.wait_stream(main)
        step_e2e(first=True)
        torch.cuda.synchronize()
        n_e2e = steps  # fill / drain of the copy pipeline are inside the timed region, amortised over these steps
        if world > 1:
            dist.barrier()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record()
        for _ in range(n_e2e):
            step_e2e()
        f1.record()
        torch.cuda.synchronize()
        res.update(e2e_ms_per_step=f0.elapsed_time(f1) / n_e2e, h2d=h2d * world, d2h=d2h * world, e2e_steps=n_e2e)
    return res


def synth_layer_params(torch, dev, E, H, TE=512, seed=7):
    """Random-init TransformerLayer state_dict with the reference's names and init scales (dit.py:281-320, ttt_layer.py:404-416),
    GEMM weights in bf16, norm / TTT-state parameters in fp32."""
    g = torch.Generator(device=dev).manual_seed(seed)
    rn = lambda *s: torch.randn(*s, generator=g, device=dev)
    bf = torch.bfloat16
    P = {}
    lin = lambda name, o, i: P.update({f"{name}.weight": (rn(o, i) / i ** 0.5).to(bf), f"{name}.bias": torch.zeros(o, device=dev, dtype=bf)})
    for n in ("pre_seq_adaLN_modulation.1", "pre_mlp_adaLN_modulation.1"):
        lin(n, 6 * E, TE)
    for n in ("pre_seq_layernorm", "pre_mlp_layernorm"):
        P[f"{n}.weight"], P[f"{n}.bias"] = torch.ones(E, device=dev), torch.zeros(E, device=dev)
    sb = "seq_modeling_block."
    for n in ("q", "k", "v", "o"):
        lin(sb + n, E, E)
    for n in ("q_norm", "k_norm"):
        P[sb + n + ".weight"], P[sb + n + ".bias"] = torch.ones(64, device=dev), torch.zeros(64, device=dev)
    for n in ("forward_ssm_gating_video", "forward_ssm_gating_text", "backward_ssm_gating_video", "backward_ssm_gating_text"):
        P[sb + n + ".gating_alpha"] = torch.full((E,), 0.1, device=dev)
    t = sb + "ssm.ttt."
    for n in ("wq", "wk", "wv", "wo"):
        lin(t + n, E, E)
    P[t + "learnable_ttt_lr_weight"] = (0.02 * rn(H, 1, E)).to(bf); P[t + "learnable_ttt_lr_bias"] = torch.zeros(H, 1, device=dev, dtype=bf)
    P[t + "ttt_norm_weight"], P[t + "ttt_norm_bias"] = torch.ones(H, 64, device=dev), torch.zeros(H, 64, device=dev)
    P[t + "post_norm.weight"], P[t + "post_norm.bias"] = torch.ones(E, device=dev), torch.zeros(E, device=dev)
    P[t + "W1"], P[t + "b1"] = 0.02 * rn(H, 64, 256), torch.zeros(H, 1, 256, device=dev)
    P[t + "W2"], P[t + "b2"] = 0.02 * rn(H, 256, 64), torch.zeros(H, 1, 64, device=dev)
    lin("mlp.layer1", 4 * E, E); lin("mlp.layer2", E, 4 * E)
    return P


def bench_dit_layer(torch, dev, steps=3, warmup=2):
    """Secondary key: ONE whole CogVideoX-5B TransformerLayer (adaLN shell, local attention, forward + reversed gated TTT-MLP,
    token MLP; all Linears) forward + backward at the 3-second length, B = 1 -- the "DiT+TTT" of BASELINE.json's metric at
    layer granularity (the 5B model is 42 such layers).  Measured twice: attention on this repo's kernel, and on the library
    SDPA the reference calls."""
    from ttt_video_dit_b200 import transformer_layer as TL
    E, H, TLen, frames = 3072, 48, 498, 13
    out = {}
    P = {k: v.requires_grad_(True) for k, v in synth_layer_params(torch, dev, E, H).items()}
    L = TLen + frames * 30 * 45
    g = torch.Generator(device=dev).manual_seed(3)
    emb = torch.randn(1, L, E, generator=g, device=dev).to(torch.bfloat16).requires_grad_(True)
    t_emb = torch.randn(1, 512, generator=g, device=dev).to(torch.bfloat16)
    go = torch.randn(1, L, E, generator=g, device=dev).to(torch.bfloat16)
    for impl in ("b200", "library"):
        meta = TL.LayerMeta(num_heads=H, text_length=TLen, num_chunks=1, num_frames=frames, latent_height=30, latent_width=45,
                            attention_impl=impl)

        def step():
            y = TL.transformer_layer_forward(emb, t_emb, P, meta)
            y.backward(go)
            emb.grad = None
            for v in P.values():
                v.grad = None
        for _ in range(warmup):
            step()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            step()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        out[f"attention_{impl}"] = {"ms_per_layer": ms, "tokens_per_s_per_layer": L / (ms * 1e-3), "model_tokens_per_s_42_layers": L / (42 * ms * 1e-3)}
    out["note"] = (f"one TransformerLayer fwd+bwd, CogVideoX-5B dims (E={E}, {H} heads), 3-sec video (L={L} tokens), B=1, bf16 GEMMs by cuBLAS; "
                   "attention_b200 = csrc/attn_*.cu, attention_library = F.scaled_dot_product_attention as in the reference")
    return out


def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    sharded = world > 1 and args.parallel in ("auto", "seqshard")
    if args.dump_outputs and sharded:
        sys.exit("bench.py: --dump-outputs needs an un-sharded run (one GPU, or --parallel replicas)")
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    from ttt_video_dit_b200 import _lib, mlp_tk
    _lib.lib()  # the library build() made; raises if it is missing (the benchmark compiles nothing into the tree)

    mode = "fwd" if args.mode == "fwd" else "fwdbwd"
    H, NC, G = args.heads, args.nc, args.ckpt
    M = (args.seqs or 8 * world) if sharded else None
    sampler = ClockSampler(local)
    if sharded:
        r = bench_sharded(args, torch, dist, world, rank, dev, mode, NC, M, True, args.steps, args.warmup, sampler)
    else:
        r = bench_replica(args, torch, dist, mlp_tk, world, rank, dev, mode, NC, True, args.steps, args.warmup, sampler,
                          dump=args.dump_outputs if rank == 0 else None)
    ms_step, ms_e2e = max_over_ranks(torch, dist, world, dev, r["ms_per_step"], r["e2e_ms_per_step"])

    secondary = {}
    if not args.no_secondary:
        torch.cuda.empty_cache()
        if sharded:
            lat = bench_sharded(args, torch, dist, world, rank, dev, mode, NC, 1, False, 3, 1)
            (ms_lat,) = max_over_ranks(torch, dist, world, dev, lat["ms_per_step"])
            secondary["single_sequence"] = {"ms": ms_lat, "tokens_per_s": NC * 64 / (ms_lat * 1e-3),
                                            "note": "ONE sequence through the N-rank chain (serial recurrence: no speed-up over one "
                                                    "GPU is possible; this is the latency the hand-offs add)"}
            torch.cuda.empty_cache()
            rep = bench_replica(args, torch, dist, mlp_tk, world, rank, dev, mode, NC, False, 3, 1)
            (ms_rep,) = max_over_ranks(torch, dist, world, dev, rep["ms_per_step"])
            secondary["replicas"] = {"ms_per_step": ms_rep, "tokens_per_s": rep["tokens_per_step"] / (ms_rep * 1e-3),
                                     "note": f"dp{world}: independent un-sharded replicas, B={args.batch} per GPU, no data-path collective"}
        elif NC != NC_9S and world == 1:
            r9 = bench_replica(args, torch, dist, mlp_tk, world, rank, dev, mode, NC_9S, False, 5, 2)
            secondary["nc804"] = {"ms_per_step": r9["ms_per_step"], "tokens_per_s": r9["tokens_per_step"] / (r9["ms_per_step"] * 1e-3),
                                  "note": "the 9-second video (3 interleaved segments, NC = 804), same op and mode"}
            if mode == "fwdbwd" and H == H_5B:
                torch.cuda.empty_cache()
                try:  # a secondary key must never cost the contract line
                    secondary["dit_layer"] = bench_dit_layer(torch, dev)
                except Exception as e:  # noqa: BLE001
                    secondary["dit_layer"] = {"error": f"{type(e).__name__}: {e}"[:300]}
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    tokens = r["tokens_per_step"]
    value = tokens / (ms_step * 1e-3)
    e2e_val = tokens / (ms_e2e * 1e-3)
    seqs_per_step = M if sharded else args.batch * world
    flop_per_step = seqs_per_step * H * NC * U_FLOP * (FWD_U + (BWD_U if mode == "fwdbwd" else 0))
    burst, sustained, src = peaks()
    achieved = flop_per_step / (ms_step * 1e-3) / 1e12 / world  # per GPU
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "r02_traffic.json")
    if not os.path.exists(tpath):
        tpath = os.path.join(ROOT, "profiles", "r01_traffic.json")
    if os.path.exists(tpath):  # DRAM bytes of the dominant kernel from the committed ncu capture, scaled to one launch
        tj = json.load(open(tpath)).get(mode)
        if tj:
            per_launch_units = args.batch * H * (NC if mode == "fwd" else min(G, NC))
            traffic = {"bytes_per_launch": tj["bytes_per_head_minibatch"] * per_launch_units, "kernel": tj["kernel"], "source": tj["source"]}
    secs = {NC_63S: "63-sec video, 21 segments", NC_9S: "9-sec video, 3 segments", NC_3S: "3-sec segment"}.get(NC, f"{NC} mini-batches")
    if sharded:
        par = (f"sequence-sharded x{world}: rank r owns mini-batch range r of every sequence ({NC // world}-{-(-NC // world)} "
               f"mini-batches); NCCL send/recv of the fp32 state (forward, 6.35 MB per sequence and boundary) and of its gradient "
               f"(backward) is the only data-path collective; {M} sequences in flight (pipeline over sequences, bubble "
               f"{(world - 1)}/{(M + world - 1)})")
    else:
        par = f"dp{world}: un-sharded replicas, no data-path collective" if world > 1 else "single GPU"
    line = {
        "metric": f"video-tokens/sec TTT-MLP layer-direction ({'fwd+bwd' if mode == 'fwdbwd' else 'fwd'})",
        "value": value, "unit": "tokens/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic",
        "config": {"workload": f"CogVideoX-5B TTT-MLP op ({secs}): {seqs_per_step} sequence(s) per step, {H} heads x 64, mini-batch 64, "
                               f"NC={NC} (L={NC * 64} tokens), checkpoint group {G}, one layer-direction",
                   "mode": mode, "parallelism": par,
                   "l2": "inputs (q,k,v = %.0f MB per sequence) larger than the 126 MB L2; no explicit flush" % (3 * H * NC * 8192 / 1e6)},
        "e2e": {"value": e2e_val, "unit": "tokens/s", "h2d_bytes_per_step": r["h2d"], "d2h_bytes_per_step": r["d2h"],
                "ms_per_step": ms_e2e, "steps": r["e2e_steps"],
                "pipeline": "pinned host -> H2D on a copy stream (ahead of the op) -> op -> D2H of the op's output on a second copy "
                            "stream; all copies of all steps inside the timed region; in fwd+bwd mode dXQ/dXK/dXV stay on the "
                            "device (they feed the upstream layer's backward), only the forward output is read back"
                            + ("; byte counts are whole-job (all ranks)" if world > 1 else "")},
        "gpu_launches": r["launches"],
        "clocks": sampler.summary(),
        "roofline": {"bound": "tensor", "achieved": achieved, "peak": burst, "unit": "TFLOP/s", "frac": achieved / burst,
                     "traffic": traffic, "peak_source": src + ", burst figure (op timed alone)",
                     "algorithmic_flop_per_step": flop_per_step,
                     "scope": "whole step, per GPU (all our kernels of the op: 7U fwd + 15U bwd per head per mini-batch; recompute not counted)"},
    }
    line.update(secondary)
    if not args.no_cpu_baseline and world == 1:
        line["cpu_baseline"] = cpu_baseline(H, mode)
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
