"""Host-side mirror of the reference interface (CPU only): factories, state-dict handling, error behaviour, the
step loop and the inference contract.  The CUDA path itself is exercised by the -m gpu tests."""
import os
import sys

import numpy as np
import pytest
import torch
from torch import nn

from oracle import UNetConfig, make_state_dict, sliding_window_inference

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
from recipe import REFERENCE_CASES, stored_spec  # noqa: E402


def test_fetch_model_by_name(pkg):
    m = pkg.fetch_model_by_name("UNet3D", n_features=4, n_outputs=3, base_width=8)
    assert isinstance(m, pkg.UNet3D) and m.n_outputs == 3
    with pytest.raises(ValueError, match="model name NoSuch not supported"):        # build.py:12-13
        pkg.fetch_model_by_name("NoSuch")


def test_ctor_rejects_unimplemented_options(pkg):
    for kw in (dict(downsampling_stride=3), dict(interpolation_mode="nearest"), dict(kernel_size=5), dict(layer_widths=[8, 16])):
        with pytest.raises(NotImplementedError):
            pkg.UNet3D(**kw)
    with pytest.raises(ValueError):
        pkg.UNet3D(activation="tanh")


def test_no_cpu_fallback(pkg):
    m = pkg.UNet3D(n_features=4, n_outputs=3, base_width=8)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m(torch.zeros(1, 4, 16, 16, 16))
    crit = pkg.DiceLoss(sigmoid=True)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        crit(torch.zeros(1, 3, 4, 4, 4), torch.zeros(1, 3, 4, 4, 4, dtype=torch.uint8))
    with pytest.raises(NotImplementedError):
        pkg.DiceLoss(softmax=True)


def test_state_dict_roundtrip_and_build_or_load(pkg, tmp_path):
    kw = dict(n_features=4, n_outputs=3, base_width=8)
    sd = make_state_dict(UNetConfig(**kw), seed=7)
    path = os.path.join(tmp_path, "model.pth")
    torch.save(sd, path)
    m = pkg.build_or_load_model("UNet3D", path, n_gpus=0, strict=True, **kw)
    for k, v in m.state_dict().items():
        assert torch.equal(v, sd[k]), k
    # non-strict load tiles/narrows mismatching tensors (build.py:47-64)
    sd_small = make_state_dict(UNetConfig(n_features=2, n_outputs=3, base_width=8), seed=7)
    torch.save(sd_small, path)
    m2 = pkg.build_or_load_model("UNet3D", path, n_gpus=0, strict=False, **kw)
    w = m2.state_dict()["encoder.layers.0.blocks.0.conv1.conv.weight"]
    assert w.shape == (8, 4, 3, 3, 3)
    assert torch.equal(w[:, :2], sd_small["encoder.layers.0.blocks.0.conv1.conv.weight"])
    assert torch.equal(w[:, 2:], sd_small["encoder.layers.0.blocks.0.conv1.conv.weight"])


def test_checkpoint_interchange_with_reference(pkg, golden_dir):
    """Checkpoints move both ways between the reference UNet3D and this module: the two state dicts have the same keys, in
    the same order, with the same shapes (the reference's, stored in tests/golden/reference_unet3d.npz)."""
    kw, _ = REFERENCE_CASES["bw8_16"]
    spec = stored_spec(np.load(os.path.join(golden_dir, "reference_unet3d.npz")), "bw8_16")
    g = torch.Generator().manual_seed(0)
    ref_sd = {k: torch.randn(shape, generator=g) for k, shape in spec}
    mine = pkg.UNet3D(**kw)
    mine.load_state_dict(ref_sd, strict=True)                     # reference checkpoint -> B200 module
    assert [(k, tuple(v.shape)) for k, v in mine.state_dict().items()] == spec      # and back
    for k, v in mine.state_dict().items():
        assert torch.equal(v, ref_sd[k]), k


def test_default_init_matches_torch_bounds(pkg):
    torch.manual_seed(0)
    m = pkg.UNet3D(n_features=4, n_outputs=3, base_width=8)
    sd = m.state_dict()
    w = sd["encoder.layers.1.blocks.0.conv1.conv.weight"]          # [16, 8, 3,3,3]: bound 1/sqrt(8*27)
    assert float(w.abs().max()) <= (8 * 27) ** -0.5 + 1e-7 and float(w.abs().max()) > 0.9 * (8 * 27) ** -0.5
    assert torch.all(sd["encoder.layers.0.blocks.0.conv1.norm1.weight"] == 1)
    assert torch.all(sd["encoder.layers.0.blocks.0.conv1.norm1.bias"] == 0)


class _Meta(torch.Tensor):
    pass


def test_volumetric_predictions_contract(pkg):
    """Re-creation of /root/reference/test/test_predict_volumetric.py's calling contract with a 1x1x1 dummy model."""
    model = nn.Conv3d(1, 1, kernel_size=1)
    x = torch.randn(2, 1, 10, 10, 10)
    with pytest.raises(TypeError):
        pkg.predict.volumetric_predictions(model, [{"image": x}], "unused")
    xm = x.as_subclass(_Meta)
    xm.meta = {}
    with pytest.raises(KeyError):
        pkg.predict.volumetric_predictions(model, [{"image": xm}], "unused")
    xm.meta = {"filename_or_obj": ["a.nii.gz", "b.nii.gz"]}
    written = []
    res = pkg.predict.volumetric_predictions(model, [{"image": xm}], "out", activation="sigmoid",
                                             writer=lambda fn, t, d: written.append((fn, d)))
    assert [r[0] for r in res] == ["a.nii.gz", "b.nii.gz"] and written == [("a.nii.gz", "out"), ("b.nii.gz", "out")]
    assert res[0][1].shape == (1, 10, 10, 10)
    assert float((res[0][1] - torch.sigmoid(model(x))[0]).abs().max()) < 1e-6


def test_sliding_window_scan_logic_matches_oracle(pkg):
    """Host side of the inferer (scan starts, importance map, config hook); the tiling kernels themselves are compared
    with the oracle inferer in tests/test_gpu_prepost.py.  A CPU tensor must raise: there is no CPU fallback."""
    from oracle.unet3d_oracle import _scan_starts, gaussian_importance
    for size, roi, ov in [(20, 16, 0.25), (24, 16, 0.25), (28, 16, 0.5), (256, 128, 0.25), (16, 16, 0.25), (10, 16, 0.25), (37, 8, 0.1)]:
        assert pkg.predict._scan_starts(size, roi, ov) == _scan_starts(size, roi, ov)
    assert pkg.predict._scan_starts(256, 128, 0.25) == [0, 96, 128]                      # config 5: 3 per axis -> 27 tiles
    g = pkg.predict._gaussian_importance((8, 12, 16), "cpu")
    assert float((g - gaussian_importance((8, 12, 16))).abs().max()) == 0.0
    inf = pkg.predict.SlidingWindowInferer(roi_size=(16, 16, 16), sw_batch_size=4, overlap=0.25)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        inf(torch.zeros(1, 2, 20, 24, 28), nn.Conv3d(2, 3, 1))
    with pytest.raises(ValueError):
        pkg.predict.SlidingWindowInferer(roi_size=16, sw_batch_size=64)
    built = pkg.predict.build_inferer_from_config({"name": "SlidingWindowInferer", "roi_size": [16, 16, 16]})
    assert isinstance(built, pkg.predict.SlidingWindowInferer)


def test_epoch_training_plumbing_cpu(pkg):
    """training_utils.py:20-85 call contract with n_gpus=None (the only CPU entry that works in the reference)."""
    torch.manual_seed(0)
    model = nn.Sequential(nn.Conv3d(2, 3, 1))
    from oracle import dice_loss

    class Crit(nn.Module):
        def forward(self, o, t):
            return dice_loss(o, t)
    loader = [{"image": torch.randn(2, 2, 4, 4, 4), "label": (torch.rand(2, 3, 4, 4, 4) > 0.5).to(torch.uint8)} for _ in range(3)]
    opt = torch.optim.Adam(model.parameters(), lr=1e-2)
    before = [p.detach().clone() for p in model.parameters()]
    synced = []
    avg = pkg.train.epoch_training(loader, model, Crit(), opt, epoch=0, n_gpus=None, print_frequency=0,
                                   grad_sync=lambda: synced.append(1))
    assert 0 < avg < 1 and len(synced) == 3
    assert any(not torch.equal(a, b) for a, b in zip(before, model.parameters()))
    v = pkg.train.epoch_validation(loader, model, Crit(), n_gpus=None)
    assert 0 < v < 1


# ------------------------------------------------------------------------------------------------ kernel index arithmetic
# Executable restatement of the stacked-MMA bookkeeping of csrc/conv_halo.cu and csrc/wgrad_halo.cu: every (output plane,
# kd tap) pair must be produced exactly once, into the accumulator columns the epilogue later reads.
@pytest.mark.parametrize("TD", [1, 2, 4])
def test_conv_halo_kd_stacking_covers_every_plane_tap_pair_once(TD):
    seen = {}
    for hq in range(TD + 2):                                   # halo plane = input depth d0 - 1 + hq
        kdmin = max(0, hq - (TD - 1))
        kdmax = min(2, hq)
        nkd = kdmax - kdmin + 1
        assert 1 <= nkd <= 3
        d_slot0 = TD - 1 - hq + kdmin                          # accumulators sit in DESCENDING plane order (units of BN)
        assert 0 <= d_slot0 and d_slot0 + nkd <= TD            # the N-stacked MMA stays inside the tile's accumulators
        for j in range(nkd):
            kd = kdmin + j                                     # weight row block kdmin + j  <->  column block d_slot0 + j
            plane = TD - 1 - (d_slot0 + j)
            assert plane == hq - kd                            # tap kd of output plane p reads halo plane p + kd
            assert (plane, kd) not in seen
            seen[(plane, kd)] = hq
    assert sorted(seen) == [(p, kd) for p in range(TD) for kd in range(3)]


@pytest.mark.parametrize("TD", [2, 4])
def test_wgrad_halo_kd_stacking_pairs_each_halo_plane_with_the_right_dy_planes(TD):
    seen = set()
    for hq in range(TD + 2):
        kdmin = max(0, hq - (TD - 1))
        kdmax = min(2, hq)
        nkd = kdmax - kdmin + 1
        blk0 = 2 - kdmax                                       # column block b holds kd = 2 - b
        dy0 = hq - kdmax                                       # first dY plane of the N atoms (ascending addresses)
        assert 0 <= dy0 and dy0 + nkd <= TD and 0 <= blk0 and blk0 + nkd <= 3
        for j in range(nkd):
            kd = 2 - (blk0 + j)
            assert dy0 + j == hq - kd                          # dY plane d pairs with input plane d + kd
            seen.add((dy0 + j, kd))
    assert seen == {(p, kd) for p in range(TD) for kd in range(3)}


@pytest.mark.parametrize("stacked", [True, False])
def test_conv_halo_incremental_tap_offsets(stacked):
    """the rolled stage loop advances the A-descriptor offset incrementally (kw fastest, then kh, then kd)"""
    rb = 4                                                     # halo row bytes >> 4 for KC = 32
    a_off, kw, kh = 0, 0, 0
    for st in range(9 if stacked else 27):
        kd_, kh_, kw_ = (0, st // 3, st % 3) if stacked else (st // 9, (st // 3) % 3, st % 3)
        assert a_off == ((kd_ * 18 + kh_) * 10 + kw_) * rb
        a_off += rb
        kw += 1
        if kw == 3:
            kw = 0
            a_off += 7 * rb
            kh += 1
            if kh == 3:
                kh = 0
                a_off += 15 * 10 * rb


def test_conv_halo_kw_grouped_stage_offsets():
    """BN <= 32: a weight stage holds the kw = 0,1,2 boxes of one kh (HaloCfg::KWS = 3).  Stage st = kh advances the A offset by
    one halo row (10 voxels); box q of the stage is kw = q (+1 voxel) and sits q boxes into the stage; the TMA box index of
    the 4-D (Cin, Cout, khkw, kd) weight view is st * 3 + q."""
    rb = 4
    b_box = 3 * 2048                                           # three kd tiles of a 32 x 32 tap
    a_off = 0
    taps = set()
    for st in range(3):
        for q in range(3):
            khkw = st * 3 + q
            assert khkw == st * 3 + q and khkw // 3 == st and khkw % 3 == q
            a_q = a_off + q * rb
            for kd in range(3):
                assert a_q + kd * 180 * rb == ((kd * 18 + st) * 10 + q) * rb
                taps.add((kd, st, q, q * b_box + kd * 2048))    # B operand offset inside the stage
        a_off += 10 * rb
    assert len(taps) == 27 and len({t[3] for t in taps}) == 9   # 9 distinct tile offsets per stage x 3 stages


def test_stride2_dgrad_parity_class_tap_lists():
    """cls_mode 1 (igemm_conv.cu): dx[i] = sum_o sum_k dy[o] w[k] [2o + k - 1 == i].  With the flipped pack Wd[k'] = w[2 - k'],
    class parity p lists (k', delta) with source index j + delta for output 2j + p; the 8 classes hold 27 tap products."""
    import itertools
    for p in (0, 1):
        lst = [(k, 1 if k == 2 else 0) for k in range(3) if (k != 1 if p else k == 1)]
        for j in range(1, 5):
            i = 2 * j + p
            direct = sorted((o, k) for o in range(0, 8) for k in range(3) if 2 * o + k - 1 == i)
            via = sorted((j + delta, 2 - kp) for kp, delta in lst)      # (dy index, un-flipped w index)
            assert direct == via
    total = sum(len([k for k in range(3) if (k != 1 if pd else k == 1)]) * len([k for k in range(3) if (k != 1 if ph else k == 1)]) *
                len([k for k in range(3) if (k != 1 if pw else k == 1)]) for pd, ph, pw in itertools.product((0, 1), repeat=3))
    assert total == 27


def test_transposed_conv_k2s2_roles():
    """ConvTranspose3d(kernel = stride = 2): U[2j + p] = sum_ci X[j] W[ci][co][p] -> class p uses tap p (cls_mode 2); its data
    gradient is the unpadded kernel-2 stride-2 convolution of dU and its weight gradient the same convolution's filter
    gradient with roles swapped (checked numerically against torch in 1-D per axis)."""
    import torch.nn.functional as F
    torch.manual_seed(0)
    x = torch.randn(1, 3, 5, dtype=torch.float64, requires_grad=True)
    w = torch.randn(3, 4, 2, dtype=torch.float64, requires_grad=True)
    u = F.conv_transpose1d(x, w, stride=2)
    for p in (0, 1):
        assert torch.allclose(u[0, :, p::2], torch.einsum("cj,co->oj", x[0], w[:, :, p]))
    du = torch.randn_like(u)
    u.backward(du)
    dx = F.conv1d(du, w.permute(0, 1, 2).reshape(3, 4, 2), stride=2)          # V[p][ci][co] = w[ci][co][p], no padding
    assert torch.allclose(dx, x.grad)
    dw = torch.stack([torch.einsum("cj,oj->co", x[0].detach(), du[0, :, t::2]) for t in (0, 1)], dim=-1)
    assert torch.allclose(dw, w.grad)


def test_tile_decode_fast_division_restatement():
    """conv_halo_kernel.cuh make_fastdiv / fast_divmod: q = umulhi(x, mul) >> shr with p = 31 + ceil(log2 d), mul = ceil(2^p / d),
    shr = p - 32 must equal x // d for every tile index (x < 2^31) and every tile-count divisor."""
    import random

    def mk(d):
        if d <= 1:
            return 0, 0
        lg = d.bit_length() - 1 + (1 if d & (d - 1) else 0)
        p = 31 + lg
        return ((1 << p) + d - 1) // d, p - 32
    rnd = random.Random(0)
    for d in list(range(1, 300)) + [511, 512, 513, 1000, 4096, 65535]:
        mul, shr = mk(d)
        assert mul < 2 ** 32
        for x in list(range(0, 600)) + [rnd.randrange(0, 2 ** 31) for _ in range(300)] + [2 ** 31 - 1]:
            q = (((x * mul) >> 32) >> shr) if d > 1 else x
            assert q == x // d and x - q * d == x % d


@pytest.mark.parametrize("n", [2, 4, 6, 10])
def test_register_blocked_trilinear_adjoint_weights(n):
    """elementwise.cu:k_upsample2x_bwd_blk: per axis, block m (outputs 2m, 2m+1) meets dy indices 4m-1+i, i = 0..5, with the
    weights blk_w0 / blk_w1.  Restated here and held to the transpose of the oracle's 1-D upsampling matrix."""
    import numpy as np

    def blk_w0(i, first):
        return {0: 0.0 if first else 0.25, 1: 1.0 if first else 0.75, 2: 0.75, 3: 0.25}.get(i, 0.0)

    def blk_w1(i, last):
        return {2: 0.25, 3: 0.75, 4: 1.0 if last else 0.75, 5: 0.0 if last else 0.25}.get(i, 0.0)

    # 1-D upsampling matrix U (2n x n) from the oracle: column k = upsampled unit vector e_k along the last axis
    U = np.zeros((2 * n, n))
    for k in range(n):
        e = np.zeros((1, 1, 1, 1, n))
        e[..., k] = 1.0
        U[:, k] = _up_last_axis(e)
    A = np.zeros((n, 2 * n))      # the kernel's adjoint
    for m in range(n // 2):
        first, last = m == 0, m == n // 2 - 1
        for i in range(6):
            g = 4 * m - 1 + i
            w0, w1 = blk_w0(i, first), blk_w1(i, last)
            if w0 == 0.0 and w1 == 0.0:
                continue
            assert 0 <= g < 2 * n, (m, i)
            A[2 * m, g] += w0
            A[2 * m + 1, g] += w1
    assert np.allclose(A, U.T, atol=1e-12)


def _up_last_axis(e):
    """the oracle's trilinear x2 restricted to the last axis: upsample a (1,1,1,1,n) array and undo the two unit axes"""
    from oracle import trilinear_upsample2x
    y = trilinear_upsample2x(e)            # (1, 1, 2, 2, 2n): the unit axes are replicated, the last axis is interpolated
    return y[0, 0, 0, 0, :]
