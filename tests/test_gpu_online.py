"""GPU: the causal / streaming SpatialNet (BASELINE configs[4]) against oracle/online_oracle.py, which is pinned to the unmodified
reference by tests/golden/online_f9_t270.npz."""
import os

import numpy as np
import pytest
import torch

from nbss_b200.online import OnlineSpatialNet
from oracle import online_oracle as OO
from oracle import spatialnet_oracle as O

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def _net(cfg, P):
    net = OnlineSpatialNet(dim_input=cfg["dim_input"], dim_output=cfg["dim_output"], num_layers=cfg["num_layers"], dim_squeeze=8,
                           num_freqs=cfg["num_freqs"], dim_hidden=96, dim_ffn=192, num_heads=4, attention="mhsa(251)").cuda()
    net.load_state_dict({k: v.clone() for k, v in P.items()}, strict=True)
    return net


def _x(z):
    """The seeded input of tests/golden/online_f9_t270.npz (make_golden_online.py), checked against its stored sum."""
    x = torch.randn(2, 9, 270, 12, generator=torch.Generator().manual_seed(270))
    assert abs(x.double().sum().item() - float(z["x_sum"])) < 1e-6, "torch's seeded generator no longer gives the stored input"
    return x


@pytest.mark.gpu
def test_online_matches_reference_golden():
    """The unmodified reference's own output (T = 270 > 251: causal attention over all past frames, the function torch executes)."""
    z = np.load(os.path.join(G, "online_f9_t270.npz"))
    cfg = dict(O.SMALL_CFG, num_layers=2, num_freqs=9)
    P = O.synth_params(cfg, 107)
    net = _net(cfg, P)
    y = net(_x(z).cuda())
    torch.cuda.synchronize()
    net.check_device_errors()
    e = O.rel_l2(y.cpu(), torch.from_numpy(z["y"]))
    print(f"online vs reference golden: rel-L2 {e:.2e}")
    assert e < 1e-3


@pytest.mark.gpu
def test_online_window_ring_wraps():
    """window=True: the key/value ring of 251 frames wraps at T = 270; against the oracle with the mask the reference builds."""
    z = np.load(os.path.join(G, "online_f9_t270.npz"))
    cfg = dict(O.SMALL_CFG, num_layers=2, num_freqs=9)
    P = O.synth_params(cfg, 107)
    net = _net(cfg, P)
    x = _x(z)
    y = net(x.cuda(), window=True)
    with torch.no_grad():
        ref = OO.online_forward({k: v.double() for k, v in P.items()}, x.double(), cfg, scope=251)
    assert O.rel_l2(y.cpu(), ref) < 1e-3
    assert O.rel_l2(y.cpu()[:, :, 251:], ref[:, :, 251:]) < 1e-3


@pytest.mark.gpu
def test_online_streaming_state_and_f129():
    """step() with an explicit state at the bench shape (F = 129, 8 layers): frame-by-frame outputs equal the oracle's offline
    causal forward; two independent streams do not interfere; the state has constant size."""
    cfg = dict(O.SMALL_CFG, num_layers=8, num_freqs=129)
    P = O.synth_params(cfg, 91)
    net = _net(cfg, P)
    g = torch.Generator().manual_seed(3)
    x = torch.randn(2, 129, 20, 12, generator=g)
    with torch.no_grad():
        ref = OO.online_forward({k: v.double() for k, v in P.items()}, x.double(), cfg)
    sa, sb = net.init_state(1), net.init_state(1)
    ya, yb = [], []
    for t in range(20):  # interleave the two utterances as two separate streams
        ya.append(net.step(x[0:1, :, t].cuda(), sa).clone())
        yb.append(net.step(x[1:2, :, t].cuda(), sb).clone())
    torch.cuda.synchronize()
    net.check_device_errors()
    y = torch.stack([torch.cat(ya, 0), torch.cat(yb, 0)], 0).permute(0, 2, 1, 3)  # [2, F, T, Cout]
    e = O.rel_l2(y.cpu(), ref)
    print(f"streaming F=129, 8 layers: rel-L2 {e:.2e}")
    assert e < 1e-3
    assert int(sa.pos.item()) == 20 and sa.kcache[0].shape == (129, 251, 96)


@pytest.mark.gpu
@pytest.mark.parametrize("scope", [251, 600, 2048])
def test_online_many_streams_row_blocked_kernels(scope):
    """More than 600 rows: the kernels that give one CTA 4 rows (2 / 1 for longer rings), with a ragged last CTA (645 % 4 = 1);
    the step replayed from a CUDA graph (capture_step) gives the same numbers as the plain launches."""
    cfg = dict(O.SMALL_CFG, num_layers=2, num_freqs=129)
    P = O.synth_params(cfg, 17)
    net = _net(cfg, P)
    g = torch.Generator().manual_seed(5)
    x = torch.randn(5, 129, 10, 12, generator=g)
    with torch.no_grad():
        ref = OO.online_forward({k: v.double() for k, v in P.items()}, x.double(), cfg)
    st, stg = net.init_state(5, scope=scope), net.capture_step(net.init_state(5, scope=scope))
    assert stg.graph is not None and int(stg.pos.item()) == 0  # capturing advanced nothing
    ys, yg = [], []
    for t in range(10):
        ys.append(net.step(x[:, :, t].cuda(), st).clone())
        yg.append(net.step(x[:, :, t].cuda(), stg).clone())
    torch.cuda.synchronize()
    net.check_device_errors()
    y, y2 = torch.stack(ys, 2), torch.stack(yg, 2)
    assert O.rel_l2(y.cpu(), ref) < 1e-3
    assert torch.equal(y, y2)


def test_online_state_dict_matches_reference_names():
    cfg = dict(O.SMALL_CFG, num_layers=2, num_freqs=9)
    net = OnlineSpatialNet(dim_input=12, dim_output=4, num_layers=2, dim_squeeze=8, num_freqs=9, dim_hidden=96, dim_ffn=192, num_heads=4)
    z = np.load(os.path.join(G, "online_f9_t270.npz"))
    ref_keys = {k[6:]: tuple(z[k]) for k in z.files if k.startswith("shape.")}
    sd = net.state_dict()
    assert set(sd.keys()) == set(ref_keys.keys())
    for k, shp in ref_keys.items():
        assert tuple(sd[k].shape) == tuple(shp), k
