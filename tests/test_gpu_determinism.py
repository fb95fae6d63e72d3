"""GPU: training steps are reproducible bit for bit.  Every cross-block reduction of the library — the weight gradients of the
tensor-core and generic convolution kernels, split-K linears, the bias / noise-weight / style / ToRGB gradients — sums
per-block partials in a fixed order instead of with float atomics, so two runs from identical state give identical losses,
gradients and parameters."""
import pytest
import torch

import swapping_autoencoder_pytorch_b200 as S

pytestmark = pytest.mark.gpu


def _train(opt, real, steps):
    torch.manual_seed(0)
    model = S.create_model(opt)
    trainer = S.create_optimizer(opt, model)
    torch.manual_seed(1)
    losses = [{k: float(v) for k, v in trainer.train_one_step({"real_A": real}, 0).items()} for _ in range(steps)]
    torch.cuda.synchronize()
    inner = model.singlegpu_model
    params = {n: p.detach().clone() for n, p in inner.named_parameters()}
    grads = {n: p.grad.detach().clone() for n, p in inner.named_parameters() if p.grad is not None}
    return losses, params, grads


def test_training_steps_are_bitwise_reproducible():
    # the benchmark's networks (default options, 256x256) at batch 4, lazy R1 on every D step: D+R1, G, D+R1, G
    opt = S.default_options(num_gpus=1, batch_size=4, crop_size=256, R1_once_every=1)
    real = torch.randn(4, 3, 256, 256, generator=torch.Generator().manual_seed(2)).clamp(-1, 1).cuda()
    losses_a, params_a, grads_a = _train(opt, real, 4)
    losses_b, params_b, grads_b = _train(opt, real, 4)
    assert losses_a == losses_b
    assert params_a.keys() == params_b.keys()
    for n in params_a:
        assert torch.equal(params_a[n], params_b[n]), n
    assert len(grads_a) > 0 and grads_a.keys() == grads_b.keys()
    for n in grads_a:
        assert torch.equal(grads_a[n], grads_b[n]), n
