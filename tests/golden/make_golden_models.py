"""Golden fixtures for the model-level CPU tests, produced by the UNMODIFIED reference models.

    python tests/golden/make_golden_models.py REFERENCE_DIR      # a checkout of the original project

REFERENCE_DIR is the original dwt-domain-adaptation checkout (usps_mnist.py, resnet50_dwt_mec_officehome.py,
utils/).  Writes, next to this file:
  lenet.npz           the reference LeNet (its own utils/whitening.py) on weights drawn by tests/test_config1_plumbing.py
  resnet_harness.npz  one train step + eval of the reference ResNet on the synthetic checkpoint (test_harness_vs_reference)
  resnet_stem.npz     the reference conv1 output, its weight gradient and the model's logits (space-to-depth stem test)
  module_surface.json attributes, state dicts, reprs and error texts of the reference layer modules
Tensors larger than FULL elements are stored as a fixed sample (flat indices kept beside the values) so every
file stays small; the tests compare on the stored elements and on the stored full norms.
"""
from __future__ import annotations

import json
import os
import sys
import types
import warnings

import numpy as np
import torch
import torch.nn.functional as F

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
TESTS = os.path.dirname(HERE)
FULL, SAMPLE = 32, 32


def sampled(out, prefix, tensors):
    """Each tensor whole when small, else SAMPLE elements at seeded flat indices; stored as one array each of values,
    flat indices and per-tensor counts (<prefix>_values / _index / _counts), in the order given."""
    idx, val = [], []
    for i, t in enumerate(tensors):
        flat = t.detach().reshape(-1).float().numpy()
        k = np.arange(flat.size) if flat.size <= FULL else np.sort(np.random.default_rng(i).choice(flat.size, SAMPLE, replace=False))
        idx.append(k)
        val.append(flat[k])
    out[prefix + "_values"] = np.concatenate(val)
    out[prefix + "_index"] = np.concatenate(idx).astype(np.int32)
    out[prefix + "_counts"] = np.array([len(k) for k in idx], dtype=np.int32)


def load_reference(ref):
    sys.path[:0] = [os.path.join(ref, "utils"), ref]
    sys.modules.setdefault("matplotlib", types.ModuleType("matplotlib"))          # usps_mnist.py only plots
    sys.modules.setdefault("matplotlib.pyplot", types.ModuleType("matplotlib.pyplot"))
    cwd = os.getcwd()
    os.chdir(ref)                                                                  # the scripts append 'utils' relatively
    try:
        import consensus_loss
        import resnet50_dwt_mec_officehome as resnet_script
        import usps_mnist
    finally:
        os.chdir(cwd)
    assert resnet_script.__file__.startswith(os.path.abspath(ref)), resnet_script.__file__
    return usps_mnist, resnet_script, consensus_loss


def lenet_case(usps_mnist):
    import oracle.torch_port as port
    from harness.lenet_dwt import LeNetDWT
    from test_config1_plumbing import LENET_SEED, init_lenet, lenet_input
    mine = LeNetDWT(port, group_size=4)
    init_lenet(mine, LENET_SEED)
    ref = usps_mnist.LeNet(group_size=4)
    ref.load_state_dict(mine.state_dict(), strict=True)
    x = lenet_input(LENET_SEED)
    ref.train()
    y_train = ref(x)
    ref.eval()
    with torch.no_grad():
        y_eval = ref(x)
    np.savez_compressed(os.path.join(HERE, "lenet.npz"), torch=torch.__version__, keys=np.array(list(ref.state_dict())),
                        y_train=y_train.detach().numpy(), y_eval=y_eval.numpy())


def resnet_harness_case(script, ref_mec):
    from harness.synth import synth_batch, synth_state_dict
    sd = synth_state_dict(1)
    x, y = synth_batch(2, 2, size=64)
    clone = lambda: {k: v.clone() for k, v in sd.items()}                        # noqa: E731
    ref = script.ResNet(script.Bottleneck, [3, 4, 6, 3], clone())
    ref.load_state_dict(clone(), strict=False)
    ref.train()
    out = ref(x)
    s, t, a = out.split(out.shape[0] // 3)
    loss = F.nll_loss(F.log_softmax(s, 1), y) + 0.1 * ref_mec.MinEntropyConsensusLoss(65, "cpu")(t, a)
    loss.backward()
    res = dict(torch=torch.__version__, keys=np.array(list(ref.state_dict())), logits=out.detach().numpy(),
               loss=np.float64(loss.item()))
    names = [n for n, _ in ref.named_parameters()]
    res["grad_names"] = np.array(names)
    res["grad_norms"] = np.array([p.grad.double().norm().item() for _, p in ref.named_parameters()])
    sampled(res, "grad", [p.grad for _, p in ref.named_parameters()])
    res["buf_norms"] = np.array([b.double().norm().item() for b in ref.state_dict().values()])
    sampled(res, "buf", list(ref.state_dict().values()))
    ref.eval()
    with torch.no_grad():
        res["logits_eval"] = ref(x).numpy()
    np.savez_compressed(os.path.join(HERE, "resnet_harness.npz"), **res)


def resnet_stem_case(script):
    from harness.synth import synth_batch, synth_state_dict
    from test_harness_vs_reference import PROBE_SEED
    sd = synth_state_dict(1)
    x, _ = synth_batch(3, 2, size=64)
    clone = lambda: {k: v.clone() for k, v in sd.items()}                        # noqa: E731
    ref = script.ResNet(script.Bottleneck, [3, 4, 6, 3], clone())
    ref.load_state_dict(clone(), strict=False)
    ref.train()
    probe = torch.randn(6, 64, 32, 32, generator=torch.Generator().manual_seed(PROBE_SEED))
    r_stem = ref.conv1(x)
    (gr,) = torch.autograd.grad((r_stem * probe).sum(), ref.conv1.weight)
    res = dict(torch=torch.__version__, stem_shape=np.array(r_stem.shape), stem_absmax=np.float64(r_stem.abs().max()),
               weight_grad=gr.numpy(), logits=ref(x).detach().numpy())
    flat = r_stem.detach().reshape(-1).numpy()
    idx = np.sort(np.random.default_rng(0).choice(flat.size, 4096, replace=False))
    res["stem_idx"], res["stem"] = idx.astype(np.int32), flat[idx]
    np.savez_compressed(os.path.join(HERE, "resnet_stem.npz"), **res)


def module_surface_case(ref):
    """The reference layer modules' observable surface for the constructor arguments test_harness_vs_reference lists."""
    import importlib.util
    from test_harness_vs_reference import BN_KWARGS, check_errors, whitening_configs

    def load(name):
        spec = importlib.util.spec_from_file_location("ref_" + name, os.path.join(ref, "utils", name + ".py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        return mod

    def state(m):
        return {k: {"shape": list(v.shape), "values": v.detach().cpu().reshape(-1).tolist()} for k, v in m.state_dict().items()}

    RW, RB = load("whitening"), load("batch_norm")
    out = {"torch": torch.__version__, "whitening": [], "batch_norm": {}}
    for args in whitening_configs():
        r = RW.WTransform2d(**args)
        out["whitening"].append({
            "attrs": {k: getattr(r, k) for k in ["num_features", "momentum", "track_running_stats", "eps", "alpha",
                                                 "group_size", "num_groups"]},
            "state": state(r), "errors": check_errors(r, args["num_features"])})
    for cls in ("BatchNorm1d", "BatchNorm2d", "BatchNorm3d"):
        rows = []
        for kw in BN_KWARGS:
            torch.manual_seed(0)
            r = getattr(RB, cls)(6, torch.zeros(6), torch.ones(6), **kw)
            rows.append({"repr": repr(r), "version": r._version, "state": state(r),
                         "parameters": [n for n, _ in r.named_parameters()], "buffers": [n for n, _ in r.named_buffers()],
                         "errors": check_errors(r, 6, bn=True)})
        out["batch_norm"][cls] = rows
    with open(os.path.join(HERE, "module_surface.json"), "w") as f:
        json.dump(out, f, indent=0)
        f.write("\n")


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    ref_dir = os.path.abspath(sys.argv[1])
    warnings.filterwarnings("ignore")
    sys.path[:0] = [TESTS, os.path.join(ROOT, "dwt-domain-adaptation_b200"), ROOT]
    torch.set_num_threads(8)
    usps_mnist, resnet_script, ref_mec = load_reference(ref_dir)
    lenet_case(usps_mnist)
    resnet_harness_case(resnet_script, ref_mec)
    resnet_stem_case(resnet_script)
    module_surface_case(ref_dir)
    print("wrote lenet.npz resnet_harness.npz resnet_stem.npz module_surface.json")
