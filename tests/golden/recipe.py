"""Seed recipe shared by the golden generator and the tests (inputs are regenerated, never stored)."""
import torch

CASES = {
    "c1_bw8_32": (dict(n_features=4, n_outputs=3, base_width=8), (1, 4, 32, 32, 32)),
    "c1_bw8_64": (dict(n_features=4, n_outputs=3, base_width=8), (1, 4, 64, 64, 64)),
    "bw16_n2_32": (dict(n_features=4, n_outputs=3, base_width=16), (2, 4, 32, 32, 32)),
    "bw8_convT_32": (dict(n_features=4, n_outputs=3, base_width=8, use_transposed_convolutions=True), (1, 4, 32, 32, 32)),
    "c5like_1ch_5lev_32": (dict(n_features=1, n_outputs=1, base_width=8, encoder_blocks=[1, 2, 2, 4, 4]), (1, 1, 32, 32, 32)),
    "bw8_nonpow2_24x32x40": (dict(n_features=4, n_outputs=3, base_width=8), (1, 4, 24, 32, 40)),
}


# reference_unet3d.npz: the reference UNet3D's state-dict spec and eval-mode forward (weights make_state_dict(seed=3), fp64
# input from seed 5) per case; the forward is stored at every second voxel along each spatial axis, plus its full norm
REFERENCE_CASES = {
    "bw8_16": (dict(n_features=4, n_outputs=3, base_width=8), (1, 4, 16, 16, 16)),
    "bw8_3lev_n2_16x24x16": (dict(n_features=2, n_outputs=2, base_width=8, encoder_blocks=[1, 1, 2]), (2, 2, 16, 24, 16)),
    "bw8_convT_16": (dict(n_features=4, n_outputs=3, base_width=8, use_transposed_convolutions=True), (1, 4, 16, 16, 16)),
}
SUB2 = (slice(None), slice(None), slice(None, None, 2), slice(None, None, 2), slice(None, None, 2))


def reference_eval_input(shape):
    return torch.randn(shape, dtype=torch.float64, generator=torch.Generator().manual_seed(5))


def stored_spec(gold, name):
    """The reference's ordered (key, shape) state-dict spec of case ``name`` from reference_unet3d.npz."""
    return [(str(k), tuple(int(d) for d in str(s).split("x") if d)) for k, s in zip(gold["keys::" + name], gold["shapes::" + name])]


def golden_inputs(shape, n_outputs, seed=1):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(shape, generator=g, dtype=torch.float32)
    g2 = torch.Generator().manual_seed(seed + 1)
    t = (torch.rand((shape[0], n_outputs) + tuple(shape[2:]), generator=g2) > 0.7).to(torch.uint8)
    g3 = torch.Generator().manual_seed(seed + 2)
    return x, t, g3


def dropout_mask(n, c, p, gen):
    keep = (torch.rand((n, c), generator=gen) >= p).to(torch.float32)
    return keep / (1.0 - p)
