"""CPU: ``sampling.BatchedDenoiser`` reproduces the reference's ``DiscreteDenoiser.forward``
(ttt/models/cogvideo/utils.py:460-492) on the classifier-free-guidance pair with ONE network call instead of one per batch
element.  The reference side is tests/golden/sampling_ref.pt, written by oracle/make_golden.py from the unmodified reference."""
import os

import pytest
import torch

GOLD = os.path.join(os.path.dirname(__file__), "golden", "sampling_ref.pt")


def test_batched_denoiser_matches_reference_loop():
    from ttt_video_dit_b200.sampling import BatchedDenoiser
    fx = torch.load(GOLD)
    calls = []

    def network(x, crossattn, c_noise):  # per-element results must not depend on the batching (= make_golden.sampling_network)
        calls.append(x.shape[0])
        return torch.tanh(x) * (1 + 0.01 * c_noise.float().reshape(-1, 1, 1, 1, 1)) + crossattn.mean(dim=(1, 2)).reshape(-1, 1, 1, 1, 1)
    mine = BatchedDenoiser(network, fx["sigmas"], dtype=torch.float32)
    s = fx["step"]
    b = mine(fx["x"], fx["sigmas"][[s, s]].clone(), {"crossattn": fx["crossattn"]}, idx=fx["sigmas"][[s, s]])
    assert fx["calls"] == [1, 1] and calls == [2]
    assert torch.allclose(fx["out"], b, rtol=0, atol=1e-6)


def test_sampling_ops_need_the_cuda_library_and_device():
    from ttt_video_dit_b200 import sampling
    from ttt_video_dit_b200.transformer_layer import LayerMeta
    meta = LayerMeta(num_heads=2, text_length=16, num_chunks=1, num_frames=13, latent_height=4, latent_width=4)
    with pytest.raises(RuntimeError):
        sampling.dit_stack_forward(torch.zeros(1, 64, 128, dtype=torch.bfloat16), torch.zeros(1, 8), [{}], meta)
