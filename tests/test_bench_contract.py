"""CPU: the reference arm of bench.py (`--impl reference`) honours the JSON-line contract and the rank rules -- rank 0 alone
runs and prints, other ranks exit 0 without work -- and the host thread-count search returns a usable count; --dump-outputs
writes a fixed sample of the last timed step's outputs."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(extra_env=None, *args):
    env = dict(os.environ, TORCHDYNAMO_DISABLE="1")
    env.update(extra_env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                           "--heads", "2", *args], capture_output=True, text=True, env=env, timeout=600, cwd=ROOT)


def test_reference_arm_prints_one_contract_line():
    r = run_bench()
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "tokens/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["steps"] == 1 and d["warmup"] == 0
    assert d["metric"].startswith("video-tokens/sec TTT-MLP layer-direction")
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["value"] == d["value"] and cb["sample"]
    assert cb["cores"] == len(os.sched_getaffinity(0)) and 1 <= cb["threads"] <= cb["cores"]
    assert d["e2e"] == {"value": d["value"], "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_other_ranks_do_no_work():
    r = run_bench({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"}, "--gpus", "2")
    assert r.returncode == 0, r.stderr[-2000:]
    assert r.stdout.strip() == ""


def test_dump_outputs_samples_large_arrays_with_a_fixed_seed(tmp_path):
    import numpy as np
    import torch
    import bench
    big = torch.arange(3 * bench.DUMP_ELEMS, dtype=torch.float32).reshape(-1, 64)  # row r holds 64 r .. 64 r + 63
    small = torch.randn(4, 256).to(torch.bfloat16)
    for d in ("a", "b"):
        bench.dump_outputs(torch, {"big": big, "small": small}, str(tmp_path / d))
    a, b = np.load(tmp_path / "a" / "big.npy"), np.load(tmp_path / "b" / "big.npy")
    assert a.dtype == np.float32 and a.shape == (bench.DUMP_ELEMS // 64, 64) and np.array_equal(a, b)
    rows = a[:, 0].astype(np.int64) // 64
    assert np.all(np.diff(rows) >= 0) and rows[-1] < big.shape[0] and np.array_equal(a, big.numpy()[rows])
    s = np.load(tmp_path / "a" / "small.npy")
    assert s.dtype == np.float32 and np.array_equal(s, small.float().numpy())


@pytest.mark.gpu
def test_dump_outputs_are_one_step_of_the_op(tmp_path):
    """bench.py --dump-outputs writes exactly what one call of the op (+ backward) returns on the benchmark's seeded inputs:
    the last timed step, not gradients accumulated over the warm-up and timed steps."""
    import numpy as np
    import torch
    import bench
    from oracle import ttt_oracle as O
    from ttt_video_dit_b200 import mlp_tk
    H, NC, G = 4, 80, 16  # 1.3 M elements per token tensor: those are sampled
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--heads", str(H), "--nc", str(NC), "--ckpt", str(G),
                        "--steps", "3", "--warmup", "1", "--no-cpu-baseline", "--no-secondary", "--dump-outputs", str(tmp_path / "bench")],
                       capture_output=True, text=True, env=dict(os.environ, TORCHDYNAMO_DISABLE="1"), timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 3
    dev = torch.device("cuda")
    params = [p.requires_grad_(True) for p in bench.synth_params(torch, dev, 1, H)]
    q, k, v, e, go = bench.synth(torch, dev, 1, H, NC, 1234, True)
    q, k, v = (t.detach().requires_grad_(True) for t in (q, k, v))
    out = mlp_tk.ttt_mlp_op(*params, q, v, k, e, G)
    out.backward(go)
    direct = dict(out=out, dXQ=q.grad, dXK=k.grad, dXV=v.grad, **{"d" + n: p.grad for n, p in zip(bench.PARAM_NAMES, params)})
    bench.dump_outputs(torch, direct, str(tmp_path / "direct"))
    assert sorted(os.listdir(tmp_path / "bench")) == sorted(n + ".npy" for n in direct)
    assert sum(os.path.getsize(tmp_path / "bench" / f) for f in os.listdir(tmp_path / "bench")) <= 64 << 20
    for n in direct:
        a, b = np.load(tmp_path / "bench" / (n + ".npy")), np.load(tmp_path / "direct" / (n + ".npy"))
        assert a.dtype == np.float32 and a.shape == b.shape, n
        assert O.rel_err(torch.from_numpy(a), torch.from_numpy(b)) < 1e-3, n
