"""BASELINE.json configs[0]: usps_mnist.py USPS->MNIST, group_size=4, 1 epoch -- plumbing.

CPU side: the LeNet restatement used on the GPU is checked against the script's own LeNet, through the
outputs that LeNet gave on the same weights and input (tests/golden/lenet.npz, written by
tests/golden/make_golden_models.py from the unmodified reference).  GPU side: one epoch of the restated
LeNet on the CUDA layers.
"""
import os

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LENET_SEED = 0


def init_lenet(model, seed):
    """Deterministic weights for the LeNet parity check, drawn from one seeded generator in parameter order:
    gamma ~ 1 + 0.1 N(0, 1), beta ~ 0.1 N(0, 1), weights and biases ~ U(-1/sqrt(fan_in), 1/sqrt(fan_in))."""
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for name, p in model.named_parameters():
            if name.startswith(("gamma", "beta")):
                p.copy_(float(name.startswith("gamma")) + 0.1 * torch.randn(p.shape, generator=g))
            else:
                bound = (p[0].numel() if p.dim() > 1 else p.numel()) ** -0.5
                p.uniform_(-bound, bound, generator=g)


def lenet_input(seed):
    return torch.randn(16, 1, 28, 28, generator=torch.Generator().manual_seed(seed))


def test_lenet_restatement_matches_reference_lenet(golden_dir):
    import oracle.torch_port as port
    from harness.lenet_dwt import LeNetDWT
    z = np.load(os.path.join(golden_dir, "lenet.npz"))
    mine = LeNetDWT(port, group_size=4)
    init_lenet(mine, LENET_SEED)
    assert sorted(mine.state_dict()) == sorted(z["keys"])    # the reference LeNet loaded these weights with strict=True
    x = lenet_input(LENET_SEED)
    mine.train()
    assert torch.allclose(mine(x), torch.from_numpy(z["y_train"]), atol=1e-5)
    mine.eval()
    with torch.no_grad():
        assert torch.allclose(mine(x), torch.from_numpy(z["y_eval"]), atol=1e-5)


@pytest.mark.gpu
def test_config1_lenet_epoch_on_cuda_layers():
    import dwt_b200
    import oracle.torch_port as port
    from dwt_b200 import _native
    from harness.lenet_dwt import LeNetDWT, train_epoch
    from harness.synth_digits import digit_batches
    dev = torch.device("cuda", 0)
    torch.manual_seed(1)
    model = LeNetDWT(dwt_b200, group_size=4).to(dev)
    twin = LeNetDWT(port, group_size=4).to(dev)           # same topology on stock ATen ops, same weights
    twin.load_state_dict(model.state_dict())
    batches = digit_batches(seed=3, steps=16)
    log = train_epoch(model, torch.optim.SGD(model.parameters(), lr=1e-2, momentum=0.5), batches, dev)
    log_twin = train_epoch(twin, torch.optim.SGD(twin.parameters(), lr=1e-2, momentum=0.5), batches, dev)   # (Adam's sign-like steps amplify 1e-7 differences)
    assert _native.status(dev) == 0
    assert all(abs(a[0] - b[0]) < 2e-2 * max(1.0, abs(b[0])) for a, b in zip(log, log_twin)), (log[-3:], log_twin[-3:])
    assert log[-1][0] < log[0][0]                          # the plumbing run learns
    model.eval(); twin.eval()
    x = batches[0][2].to(dev)
    with torch.no_grad():
        assert (model(x) - twin(x)).abs().max() < 5e-2 * twin(x).abs().max()
