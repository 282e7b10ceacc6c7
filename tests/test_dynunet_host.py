"""Host logic of the DynUNet mirror (no GPU): MONAI kwarg surface, state-dict spec == the restated oracle spec == the
library plan's spec, loud rejection of what is not implemented, the reference's JSON config builds."""
import pytest
import torch

from oracle.dynunet_oracle import dynunet_state_dict_spec, make_dynunet_state_dict, dynunet_forward

KW = dict(spatial_dims=3, in_channels=4, out_channels=3, kernel_size=[[3, 3, 3]] * 4, strides=[[1, 1, 1]] + [[2, 2, 2]] * 3,
          upsample_kernel_size=[[2, 2, 2]] * 3, filters=[8, 16, 24, 32])


def test_state_dict_and_plan_spec(pkg):
    m = pkg.DynUNet(**KW)
    spec = dynunet_state_dict_spec(4, 3, [8, 16, 24, 32])
    assert [(k, tuple(v.shape)) for k, v in m.state_dict().items()] == spec
    plan = pkg.models._Plan(m._net_desc(1, 32, 32, 32), torch.device("cpu"))
    assert plan.param_spec() == spec
    d = m._net_desc(1, 32, 32, 32)
    d.inference_only = 1
    assert pkg.models._Plan(d, torch.device("cpu")).ws_bytes < 0.5 * plan.ws_bytes
    m.load_state_dict(make_dynunet_state_dict(4, 3, [8, 16, 24, 32]), strict=True)
    assert isinstance(pkg.fetch_model_by_name("DynUNet", **KW), pkg.DynUNet)          # build.py:9-13 lookup


def test_default_filters_and_ints(pkg):
    m = pkg.DynUNet(3, 1, 2, kernel_size=[3, 3, 3, 3, 3], strides=[1, 2, 2, 2, 2], upsample_kernel_size=[2, 2, 2, 2])
    assert m.filters == [32, 64, 128, 256, 320]
    assert m.act_slope == pytest.approx(0.01)


@pytest.mark.parametrize("bad", [dict(deep_supervision=True), dict(res_block=True), dict(trans_bias=True), dict(dropout=0.1),
                                 dict(norm_name="batch"), dict(spatial_dims=2), dict(kernel_size=[[3, 3, 3], [3, 3, 3], [5, 5, 5], [3, 3, 3]]),
                                 dict(strides=[[1, 1, 1], [2, 2, 2], [2, 2, 1], [2, 2, 2]]), dict(upsample_kernel_size=[[2, 2, 2], [2, 2, 2], [4, 4, 4]])])
def test_unimplemented_options_raise(pkg, bad):
    with pytest.raises(NotImplementedError):
        pkg.DynUNet(**{**KW, **bad})


def test_reference_example_config_builds(pkg):
    # the "model" block of the reference's examples/brats2020/brats2020_config.json
    cfg = dict(name="DynUNet", in_channels=4, out_channels=3, spatial_dims=3, deep_supervision=False,
               strides=[[1, 1, 1]] + [[2, 2, 2]] * 5, filters=[64, 96, 128, 192, 256, 384], kernel_size=[[3, 3, 3]] * 6,
               upsample_kernel_size=[[2, 2, 2]] * 5)
    name = cfg.pop("name")
    m = pkg.fetch_model_by_name(name, **cfg)
    assert m.filters == [64, 96, 128, 192, 256, 384]
    plan = pkg.models._Plan(m._net_desc(2, 128, 128, 128), torch.device("cpu"))
    assert plan.n_params == len(list(m.parameters())) and plan.ws_bytes < 40 * 2 ** 30


def test_oracle_restatement_shapes():
    sd = make_dynunet_state_dict(2, 2, [8, 16, 16])
    y = dynunet_forward(sd, torch.randn(2, 2, 16, 24, 16), 3)
    assert y.shape == (2, 2, 16, 24, 16) and torch.isfinite(y).all()
