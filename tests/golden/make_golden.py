"""Generate the committed golden fixtures by running the UNMODIFIED reference UNet3D on CPU.

Needs the reference source tree (located by oracle/ref_loader.py):   python tests/golden/make_golden.py
Writes tests/golden/*.npz .  Inputs/weights are NOT stored: they are regenerated from seeds by
``oracle.make_state_dict`` / ``golden_inputs`` so the fixtures stay small.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import UNetConfig, make_state_dict, unet3d_state_dict_spec, dice_loss  # noqa: E402
from oracle.ref_loader import reference_unet3d  # noqa: E402

sys.path.insert(0, HERE)
from recipe import CASES, REFERENCE_CASES, SUB2, golden_inputs, dropout_mask, reference_eval_input  # noqa: E402


def run_case(name, kw, shape, dtype):
    cfg = UNetConfig(**kw)
    model = reference_unet3d(**kw).to(dtype)
    sd = make_state_dict(cfg, seed=0, dtype=dtype)
    ref_keys = [(k, tuple(v.shape)) for k, v in model.state_dict().items()]
    assert ref_keys == unet3d_state_dict_spec(cfg), "state-dict spec mismatch for %s" % name
    model.load_state_dict(sd, strict=True)
    x, t, g3 = golden_inputs(shape, cfg.n_outputs)
    x = x.to(dtype)
    mask = dropout_mask(shape[0], cfg.enc_widths()[0], cfg.dropout, g3)

    # train-mode forward with a shared dropout mask: monkeypatch Dropout3d to apply our mask
    drop = model.encoder.layers[0].dropout

    def fake_dropout(inp):
        return inp * mask.to(inp.dtype).view(inp.shape[0], inp.shape[1], 1, 1, 1)
    drop.forward = fake_dropout
    model.train()
    logits = model(x)
    loss = dice_loss(logits, t)
    loss.backward()
    grads = {k: p.grad.detach().double().numpy() for k, p in model.named_parameters()}
    del drop.forward            # back to the real Dropout3d (identity in eval mode)
    model.eval()
    with torch.no_grad():
        logits_eval = model(x)
    return cfg, logits.detach(), loss.detach(), grads, logits_eval


def main():
    for name, (kw, shape) in CASES.items():
        cfg, logits, loss, grads, logits_eval = run_case(name, kw, shape, torch.float64)
        _, logits32, loss32, _, _ = run_case(name, kw, shape, torch.float32)
        rel32 = float((logits32.double() - logits).norm() / logits.norm())
        sub = (slice(None), slice(None), slice(None, None, 4), slice(None, None, 4), slice(None, None, 4))
        out = {
            "logits_sub4": logits[sub].numpy().astype(np.float32),
            "logits_eval_sub4": logits_eval[sub].numpy().astype(np.float32),
            "logits_norm": np.float64(logits.norm()),
            "logits_sum": np.float64(logits.sum()),
            "logits_eval_norm": np.float64(logits_eval.norm()),
            "dice": np.float64(loss),
            "dice_fp32_ref": np.float64(loss32),
            "fp32_vs_fp64_logits_rel": np.float64(rel32),
        }
        keys = sorted(grads)
        out["grad_keys"] = np.array(keys)
        out["grad_norms"] = np.array([np.linalg.norm(grads[k]) for k in keys])
        # a few full small gradients for direction checks
        for k in keys:
            if grads[k].size <= 4096:
                out["grad::" + k] = grads[k].astype(np.float32)
        path = os.path.join(HERE, name + ".npz")
        np.savez_compressed(path, **out)
        print(name, "dice", float(loss), "fp32 rel", rel32, "->", os.path.getsize(path), "bytes")
    reference_unet3d_fixture()


def reference_unet3d_fixture():
    out = {}
    for name, (kw, shape) in REFERENCE_CASES.items():
        model = reference_unet3d(**kw).double()
        sd = model.state_dict()
        out["keys::" + name] = np.array(list(sd))
        out["shapes::" + name] = np.array(["x".join(str(d) for d in v.shape) for v in sd.values()])
        model.load_state_dict(make_state_dict(UNetConfig(**kw), seed=3, dtype=torch.float64), strict=True)
        model.eval()
        with torch.no_grad():
            y = model(reference_eval_input(shape))
        out["eval_sub2::" + name] = y[SUB2].numpy()
        out["eval_norm::" + name] = np.float64(y.norm())
    path = os.path.join(HERE, "reference_unet3d.npz")
    np.savez_compressed(path, **out)
    print("reference_unet3d ->", os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
