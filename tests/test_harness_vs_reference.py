"""The measurement harness (harness/resnet50_dwt.py) against the UNMODIFIED reference model
(resnet50_dwt_mec_officehome.py ResNet) on CPU, both built on stock ATen layers:
same synthetic checkpoint, same batch -> same logits, loss, gradients, buffers, eval logits.
Guards the topology restatement (incl. the Bottleneck tail that the fused site folds in).

The reference side is stored: tests/golden/make_golden_models.py ran the reference on the same inputs and
wrote what it gave to tests/golden/ (resnet_harness.npz, resnet_stem.npz, module_surface.json).  Tensors
too large to store whole are compared on a fixed sample of their elements and on their full norm."""
import json
import os

import numpy as np
import torch
import torch.nn.functional as F

PROBE_SEED = 5
BN_KWARGS = [dict(affine=True), dict(affine=False), dict(affine=True, track_running_stats=False),
             dict(momentum=None, eps=1e-3)]


def whitening_configs():
    return [dict(num_features=8, group_size=4), dict(num_features=8, group_size=16), dict(num_features=48, group_size=32),
            dict(num_features=8, group_size=4, running_m=torch.zeros(1, 8, 1, 1), running_var=torch.ones(2, 4, 4)),
            dict(num_features=8, group_size=4, running_m=torch.zeros(1, 8, 1, 1), running_var=torch.ones(2, 4, 4),
                 track_running_stats=False, momentum=0.3, eps=1e-2, alpha=2)]


def check_errors(m, channels, bn=False):
    """The ValueError text (or None) of the module's input checks on a fixed set of malformed inputs."""
    def err(fn, *a):
        try:
            fn(*a)
        except ValueError as e:
            return str(e)
        return None
    if bn:
        return [err(m._check_input_dim, torch.zeros(*([2, 6] + [3] * (nd - 2)))) for nd in range(2, 7)]
    return [err(lambda b: (m._check_input_dim(b), m._check_group_size()), bad)
            for bad in [torch.zeros(2, 8, 3), torch.zeros(2, channels, 3, 3)]]


def _golden(golden_dir, name):
    return np.load(os.path.join(golden_dir, name))


def _stored(z, prefix):
    """-> [(flat indices, reference values)] per tensor, in the order the generator stored them."""
    ends = np.cumsum(z[prefix + "_counts"])
    return [(z[prefix + "_index"][e - c:e], z[prefix + "_values"][e - c:e].astype(np.float64))
            for c, e in zip(z[prefix + "_counts"], ends)]


def test_harness_equals_reference_model(golden_dir):
    import oracle.torch_port as port
    from harness.resnet50_dwt import build_resnet50_dwt
    from harness.synth import synth_batch, synth_state_dict
    z = _golden(golden_dir, "resnet_harness.npz")
    torch.set_num_threads(8)
    sd = synth_state_dict(1)
    x, y = synth_batch(2, 2, size=64)
    mine = build_resnet50_dwt({k: v.clone() for k, v in sd.items()}, port)
    assert set(z["keys"]) == set(mine.state_dict())

    mine.train()
    out = mine(x)
    s, t, a = out.split(out.shape[0] // 3)
    loss = F.nll_loss(F.log_softmax(s, 1), y) + 0.1 * port.MinEntropyConsensusLoss(65, "cpu")(t, a)
    loss.backward()
    assert torch.allclose(torch.from_numpy(z["logits"]), out.detach(), atol=1e-5) and abs(float(z["loss"]) - loss.item()) < 1e-5
    params = dict(mine.named_parameters())
    assert set(z["grad_names"]) == set(params)
    for name, norm, (idx, want) in zip(z["grad_names"], z["grad_norms"], _stored(z, "grad")):
        g = params[name].grad.reshape(-1).double().numpy()
        # ||g_ref - g|| <= 1e-4 ||g_ref|| holds on any subset of the elements too, and bounds the difference of the norms
        assert np.linalg.norm(g[idx] - want) <= 1e-4 * norm + 1e-9, name
        assert abs(np.linalg.norm(g) - norm) <= 1e-4 * norm + 1e-9, name
    sd_mine = mine.state_dict()
    for name, norm, (idx, want) in zip(z["keys"], z["buf_norms"], _stored(z, "buf")):
        b = sd_mine[name].reshape(-1).double().numpy()
        assert np.allclose(b[idx], want, atol=1e-5, rtol=1e-5), name
        assert abs(np.linalg.norm(b) - norm) <= 1e-5 * (1 + norm) * b.size ** 0.5, name      # implied by allclose
    mine.eval()
    with torch.no_grad():
        assert torch.allclose(torch.from_numpy(z["logits_eval"]), mine(x), atol=1e-4)


def test_module_surface_is_the_references_own(golden_dir):
    """Against the UNMODIFIED reference modules: attributes, buffer identity, state-dict keys and initial values (same
    RNG stream), repr, checkpoint-version shim and every error text, string for string."""
    import warnings
    warnings.filterwarnings("ignore")
    from dwt_b200 import batch_norm as B, whitening as W
    with open(os.path.join(golden_dir, "module_surface.json")) as f:
        ref = json.load(f)

    def same_state(m, want):
        sd = m.state_dict()
        assert list(sd) == list(want)
        for k, v in sd.items():
            r = torch.tensor(want[k]["values"], dtype=v.dtype).reshape(want[k]["shape"])
            assert torch.equal(v.cpu(), r), k

    configs = whitening_configs()
    assert len(configs) == len(ref["whitening"])
    for args, r in zip(configs, ref["whitening"]):
        a = W.WTransform2d(**args)
        for k, v in r["attrs"].items():
            assert getattr(a, k) == v, (k, args)
        assert a.running_m is args.get("running_m") and a.running_var is args.get("running_var")
        same_state(a, r["state"])
        assert check_errors(a, args["num_features"]) == r["errors"]
    for cls in ("BatchNorm1d", "BatchNorm2d", "BatchNorm3d"):
        assert len(BN_KWARGS) == len(ref["batch_norm"][cls])
        for kw, r in zip(BN_KWARGS, ref["batch_norm"][cls]):
            torch.manual_seed(0)
            a = getattr(B, cls)(6, torch.zeros(6), torch.ones(6), **kw)
            assert repr(a) == r["repr"] and a._version == r["version"]
            same_state(a, r["state"])
            assert [n for n, _ in a.named_parameters()] == r["parameters"]
            assert [n for n, _ in a.named_buffers()] == r["buffers"]
            assert check_errors(a, 6, bn=True) == r["errors"], cls
            if kw.get("track_running_stats", True):
                v1 = {k: v for k, v in a.state_dict().items() if "num_batches" not in k}
                a.load_state_dict(v1)                             # pre-version-2 checkpoint: no counter


def test_space_to_depth_stem_equals_the_reference_stem(golden_dir):
    """The harness option stem_s2d (7x7/2 convolution evaluated as the 4x4/1 convolution of the 2x2 space-to-depth image)
    against the UNMODIFIED reference model's conv1: same output and the same gradient of the [64, 3, 7, 7] weight (fp32
    summation order is the only difference), in both memory formats; and the whole model's logits on top of it.  (The
    GPU golden test at 224x224 runs the same option on the CUDA layers.)"""
    import oracle.torch_port as port
    from harness.resnet50_dwt import build_resnet50_dwt
    from harness.synth import synth_batch, synth_state_dict
    z = _golden(golden_dir, "resnet_stem.npz")
    torch.set_num_threads(8)
    sd = synth_state_dict(1)
    x, _ = synth_batch(3, 2, size=64)
    probe = torch.randn(6, 64, 32, 32, generator=torch.Generator().manual_seed(PROBE_SEED))
    idx = torch.from_numpy(z["stem_idx"])
    r_stem, gr, r_logits = torch.from_numpy(z["stem"]), torch.from_numpy(z["weight_grad"]), torch.from_numpy(z["logits"])
    for cl in (False, True):
        mine = build_resnet50_dwt({k: v.clone() for k, v in sd.items()}, port, channels_last=cl, stem_s2d=True).train()
        xi = x.contiguous(memory_format=torch.channels_last) if cl else x
        assert mine.conv1.weight.shape == gr.shape == (64, 3, 7, 7)
        m_stem = mine._stem(xi)
        assert tuple(m_stem.shape) == tuple(z["stem_shape"])
        m_flat = m_stem.detach().reshape(-1)[idx]
        assert torch.allclose(r_stem, m_flat, atol=1e-5), (r_stem - m_flat).abs().max()
        assert abs(m_stem.detach().abs().max().item() - float(z["stem_absmax"])) <= 1e-5
        (gm,) = torch.autograd.grad((m_stem * probe).sum(), mine.conv1.weight)
        assert (gr - gm).norm() <= 1e-5 * gr.norm(), ((gr - gm).norm() / gr.norm()).item()
        # 2 x 2 pixels per image reach layer4 at this size: the batch statistics amplify the rounding differences
        assert (r_logits - mine(xi)).abs().max() <= 1e-3 * r_logits.abs().max()
