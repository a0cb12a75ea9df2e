"""GPU: NBC2 inference (BASELINE configs[3]) against oracle/nbc2_oracle.py (pinned to the unmodified reference by
tests/golden/nbc2_small_f17_t12.npz).  Tolerance: 1e-3 rel-L2 of the network output (fp16 tensor-core operands)."""
import pytest
import torch

from nbss_b200 import ops
from nbss_b200.nbc2 import NBC2
from oracle import nbc2_oracle as N2
from oracle import spatialnet_oracle as O


def _net(cfg, P):
    net = NBC2(dim_input=cfg["dim_input"], dim_output=cfg["dim_output"], n_layers=cfg["n_layers"], dim_hidden=96, dim_ffn=192,
               num_freqs=cfg["num_freqs"]).cuda()
    net.load_state_dict({k: v.clone() for k, v in P.items()}, strict=True)
    return net


@pytest.mark.gpu
@pytest.mark.parametrize("T", [250, 251, 64, 37])
def test_mhsa_two_heads(T):
    """The attention kernel instantiated for 2 heads x 48 (NBC2) against the oracle's MHSA, incl. the GroupBatchNorm partials."""
    cfg = dict(N2.NBC2_SMALL, n_layers=1, num_freqs=5)
    P = N2.synth_params(cfg, 7)
    Pd = {k: v.cuda() for k, v in P.items()}
    pre = "sa_layers.0."
    x = torch.randn(2, 5, T, 96, generator=torch.Generator().manual_seed(T))
    with torch.no_grad():
        xr = x.reshape(10, T, 96)
        ref = N2.mhsa(N2.layer_norm(xr, P[pre + "norm1.weight"], P[pre + "norm1.bias"]), P, pre + "self_attn.", 2).reshape(2, 5, T, 96)
    img = ops.nbc2_pack_block(Pd, pre)
    xd = x.cuda()
    y = torch.empty_like(xd)
    part = torch.zeros(10 * T, 2, device="cuda")
    err = ops.device_err_flag(xd.device)
    st = ops._K("nbss_mhsa_fwd_nh")(ops.ptr(xd), ops.ptr(y), 10, T, ops.ptr(Pd[pre + "norm1.weight"]), ops.ptr(Pd[pre + "norm1.bias"]),
                                    ops.ptr(Pd[pre + "self_attn.in_proj_bias"]), ops.ptr(Pd[pre + "self_attn.out_proj.bias"]), ops.ptr(img),
                                    ops.ptr(None), ops.ptr(None), ops.ptr(None), ops.ptr(None), ops.ptr(part), 2, ops.FMT_F16, ops.ptr(err),
                                    ops.stream_ptr())
    ops.check(st, "nbss_mhsa_fwd_nh")
    torch.cuda.synchronize()
    ops.check_err_flag(err, "mhsa_fwd_nh")
    e = O.rel_l2(y.cpu() - x, ref)
    assert e < 1e-3, f"branch rel-L2 {e:.3e}"
    yr = (x + ref).reshape(10 * T, 96)
    assert O.rel_l2(part.cpu()[:, 0], yr.sum(-1)) < 1e-3 and O.rel_l2(part.cpu()[:, 1], (yr * yr).sum(-1)) < 1e-3


@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(2, 17, 12), (1, 257, 250), (3, 33, 100)])
def test_nbc2_forward(shape):
    B, F, T = shape
    cfg = dict(N2.NBC2_SMALL, n_layers=3 if F == 257 else 8, num_freqs=F)
    P = N2.synth_params(cfg, 11)
    net = _net(cfg, P)
    x = torch.randn(B, F, T, 16, generator=torch.Generator().manual_seed(F + T))
    y = net(x.cuda())
    torch.cuda.synchronize()
    net.check_device_errors()
    with torch.no_grad():
        ref = N2.nbc2_forward({k: v.double() for k, v in P.items()}, x.double(), cfg)
    e = O.rel_l2(y.cpu(), ref)
    print(f"NBC2 {shape}: forward rel-L2 {e:.2e}")
    assert e < 1e-3, e


@pytest.mark.gpu
def test_nbc2_state_dict_and_no_cpu_path():
    cfg = dict(N2.NBC2_SMALL, n_layers=2, num_freqs=9)
    net = NBC2(dim_input=16, dim_output=4, n_layers=2, dim_hidden=96, dim_ffn=192, num_freqs=9)
    shapes = N2.param_shapes(cfg)
    sd = net.state_dict()
    assert set(sd.keys()) == set(shapes.keys())
    for k, shp in shapes.items():
        assert tuple(sd[k].shape) == tuple(shp), k
    with pytest.raises(Exception):
        net(torch.zeros(1, 9, 8, 16))


@pytest.mark.gpu
def test_nbc2_forward_against_the_unmodified_reference_module():
    """Parity with the reference ITSELF: the unmodified `models.arch.NBC2.NBC2` ran on the host in fp32 on the case of
    test_nbc2_forward[(3, 33, 100)] (every 7th output value stored by tests/golden/make_golden_parity.py)."""
    import os

    import numpy as np

    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "nbc2_f33_t100.npz"))
    B, F, T = 3, 33, 100
    cfg = dict(N2.NBC2_SMALL, n_layers=8, num_freqs=F)
    P = N2.synth_params(cfg, 11)
    net = _net(cfg, P)
    x = torch.randn(B, F, T, 16, generator=torch.Generator().manual_seed(F + T))
    assert abs(x.double().sum().item() - float(z["x_sum"])) < 1e-6, "torch's seeded generator no longer gives the stored input"
    y = net(x.cuda())
    torch.cuda.synchronize()
    net.check_device_errors()
    e = O.rel_l2(y.cpu().reshape(-1)[::7], torch.from_numpy(z["y_every7"]))
    assert e < 1e-3, f"rel-L2 vs the unmodified reference {e:.3e}"
