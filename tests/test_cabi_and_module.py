"""CPU: the C-ABI library loads and exports every symbol include/nbss_b200.h declares; the drop-in module exposes the
reference's parameter names / shapes; the product path refuses to run without CUDA (no fallback)."""
import os
import re

import pytest
import torch

from nbss_b200 import _lib
from nbss_b200.spatialnet import SpatialNet
from oracle import spatialnet_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "nbss_b200.h")).read()
    names = set(re.findall(r"\b(nbss_[a-z0-9_]+)\s*\(", hdr))
    assert len(names) >= 20
    L = _lib.lib()
    missing = [n for n in sorted(names) if not hasattr(L, n)]
    assert not missing, missing


def test_cabi_error_behaviour_without_a_gpu():
    """Every entry point validates its arguments BEFORE touching CUDA and answers with the status codes of include/nbss_b200.h
    (-1 shape, -2 null pointer, -3 unsupported); nothing throws, nothing is launched — so this runs without a GPU.  The dummy
    non-null addresses are never dereferenced on the host."""
    import ctypes as C

    L = _lib.lib()
    nul, d = C.c_void_p(0), C.c_void_p(0x1000)
    assert L.nbss_version() == 200
    L.nbss_workspace_bytes.restype = C.c_longlong
    assert L.nbss_workspace_bytes(32, 129, 250, 0) == 0
    per_layer = L.nbss_workspace_bytes(32, 129, 250, 1)
    assert 4.0e9 < per_layer < 9.0e9  # DESIGN.md §2: ~4.4 GB saved per layer at batch 32 + transient gradient operands
    assert L.nbss_workspace_bytes(0, 129, 250, 1) == -1
    L.nbss_layer_image_bytes.restype = C.c_uint
    assert L.nbss_layer_image_bytes() == 626688            # csrc/layout.cuh IMG_LAYER_BYTES
    L.nbss_fconv_image_bytes.restype = C.c_uint
    assert L.nbss_fconv_image_bytes() == 2 * 46080          # forward + transposed F-conv images
    # null pointers
    assert L.nbss_mhsa_fwd(nul, d, 4, 250, d, d, d, d, d, nul, nul, nul, nul, 0, nul, nul) == -2
    assert L.nbss_fconv_tc_fwd(d, nul, 1, 129, 250, d, d, d, d, d, 0, nul, nul) == -2
    assert L.nbss_pack_layer_weights(d, d, d, nul, d, d, d, d, 0, 0, nul) == -2
    assert L.nbss_sisdr_pit_fwd(nul, d, 1, 2, C.c_longlong(100), 0, d, d, nul, nul, nul, nul) == -2
    # shapes: the training kernels hold one (b,f) slab of at most 256 frames per CTA
    assert L.nbss_mhsa_fwd(d, d, 4, 257, d, d, d, d, d, nul, nul, nul, nul, 0, nul, nul) == -1
    assert L.nbss_mhsa_fwd(d, d, 0, 250, d, d, d, d, d, nul, nul, nul, nul, 0, nul, nul) == -1
    assert L.nbss_ffn_fwd(d, d, 4, 0, d, d, d, d, d, d, d, d, d, d, nul, nul, nul, nul, nul, nul, 0, nul, nul) == -1
    assert L.nbss_fconv_tc_fwd(d, d, 0, 129, 250, d, d, d, d, d, 0, nul, nul) == -1
    assert L.nbss_sisdr_pit_fwd(d, d, 0, 2, C.c_longlong(100), 0, d, d, nul, nul, nul, nul) == -1
    # unsupported configurations
    assert L.nbss_mhsa_fwd_nh(d, d, 4, 250, d, d, d, d, d, nul, nul, nul, nul, nul, 3, 0, nul, nul) == -3   # heads: 4 or 2
    assert L.nbss_ffn_fwd(d, d, 4, 250, d, d, d, d, d, d, d, d, d, d, nul, nul, nul, nul, nul, nul, 2, nul, nul) == -3  # fmt
    assert L.nbss_sisdr_pit_fwd(d, d, 1, 3, C.c_longlong(100), 0, d, d, nul, nul, nul, nul) == -3           # 2 speakers
    # the Python wrapper turns a status into NbssError with the entry point's name
    with pytest.raises(_lib.NbssError, match="nbss_mhsa_fwd.*shape"):
        _lib.check(-1, "nbss_mhsa_fwd")


def test_state_dict_contract_matches_reference_names_and_shapes():
    net = SpatialNet(dim_input=12, dim_output=4, dim_squeeze=8, num_layers=8, num_freqs=129, dim_hidden=96, dim_ffn=192, num_heads=4)
    sd = net.state_dict()
    shapes = O.param_shapes(O.SMALL_CFG)
    assert set(sd.keys()) == set(shapes.keys())
    for k, shp in shapes.items():
        assert tuple(sd[k].shape) == tuple(shp), k
    # the full-band linear is one tensor shared by all layers (SpatialNet.py:192-195)
    assert sd["layers.0.full.weight"].data_ptr() == sd["layers.7.full.weight"].data_ptr()
    assert sum(p.numel() for p in net.parameters()) == 1_191_092
    # loading oracle-style parameters round-trips
    P = O.synth_params(O.SMALL_CFG, 1)
    net.load_state_dict({k: v.clone() for k, v in P.items()}, strict=True)


def test_no_cpu_fallback():
    net = SpatialNet(dim_input=12, dim_output=4, dim_squeeze=8, num_layers=1, num_freqs=129, dim_hidden=96, dim_ffn=192, num_heads=4)
    with pytest.raises(Exception):
        with torch.no_grad():
            net(torch.zeros(1, 129, 8, 12))


def test_unsupported_configuration_is_rejected():
    with pytest.raises(NotImplementedError):
        SpatialNet(dim_input=12, dim_output=4, dim_squeeze=16, num_layers=12, num_freqs=129, dim_hidden=192, dim_ffn=384, num_heads=4)


def test_same_init_as_reference_under_same_seed():
    """The reference's SpatialNet initialised under the same seed (tests/golden/make_golden_parity.py stores its key order, and
    per tensor the float64 sum, sum of squares and a strided sample)."""
    import numpy as np

    z = np.load(os.path.join(ROOT, "tests", "golden", "init_seed2_l2.npz"))
    kw = dict(dim_input=12, dim_output=4, dim_squeeze=8, num_layers=2, num_freqs=129, dim_hidden=96, dim_ffn=192, num_heads=4)
    torch.manual_seed(2)
    msd = SpatialNet(**kw).state_dict()
    assert list(msd.keys()) == z["keys"].tolist()
    samples = torch.from_numpy(z["samples"]).split(z["sample_len"].tolist())
    for i, (k, v) in enumerate(msd.items()):
        flat = v.reshape(-1)
        assert torch.equal(flat[::max(1, flat.numel() // 64)], samples[i]), k
        for stat, got in (("sum", flat.double().sum()), ("sumsq", flat.double().square().sum())):
            want = float(z[stat][i])
            assert abs(got.item() - want) <= 1e-12 * max(1.0, abs(want)), (k, stat)


def test_flat_clip_adam_state_dict_speaks_torch_adam_format():
    """CPU (host logic only; the update kernel itself is a GPU test): FlatClipAdam.state_dict() loads into torch.optim.Adam over
    the same parameters and torch.optim.Adam's state_dict() loads back — the checkpoint / resume path of the reference's trainer
    (Lightning stores optimizer.state_dict(), models/utils/general_steps.py:243-271)."""
    from nbss_b200.optim import FlatClipAdam

    net = SpatialNet(dim_input=12, dim_output=4, dim_squeeze=8, num_layers=1, num_freqs=17, dim_hidden=96, dim_ffn=192, num_heads=4)
    params = [p for _, p in net._unique_params()]
    n = sum(p.numel() for p in params)
    opt = FlatClipAdam.__new__(FlatClipAdam)  # the constructor insists on CUDA parameters; the state logic does not
    opt.module, opt._params, opt.n = net, params, n
    opt.lr, opt.betas, opt.eps, opt.max_norm = 1e-3, (0.9, 0.999), 1e-8, 5.0
    opt.exp_avg, opt.exp_avg_sq = torch.zeros(n), torch.zeros(n)
    opt.step_count = torch.zeros(1)

    ref = torch.optim.Adam(params, lr=3e-4)
    g = torch.Generator().manual_seed(0)
    for _ in range(3):
        for p in params:
            p.grad = torch.randn(p.shape, generator=g)
        ref.step()
    opt.load_state_dict(ref.state_dict())
    assert opt.lr == 3e-4 and opt.step_count.item() == 3.0
    off = 0
    for i, p in enumerate(params):
        assert torch.equal(opt.exp_avg[off:off + p.numel()].view_as(p), ref.state[p]["exp_avg"])
        assert torch.equal(opt.exp_avg_sq[off:off + p.numel()].view_as(p), ref.state[p]["exp_avg_sq"])
        off += p.numel()
    ref2 = torch.optim.Adam(params, lr=1.0)
    ref2.load_state_dict(opt.state_dict())  # torch validates the group / state structure
    assert ref2.param_groups[0]["lr"] == 3e-4
    for p in params:
        assert torch.equal(ref2.state[p]["exp_avg"], ref.state[p]["exp_avg"]) and float(ref2.state[p]["step"]) == 3.0
    for p in params:  # and the restored torch optimizer steps exactly like the original one
        p.grad = torch.randn(p.shape, generator=g)
    before = [p.detach().clone() for p in params]
    ref.step()
    after_ref = [p.detach().clone() for p in params]
    with torch.no_grad():
        for p, b in zip(params, before):
            p.copy_(b)
    ref2.step()
    for p, a in zip(params, after_ref):
        assert torch.equal(p.detach(), a)
    with pytest.raises(ValueError):
        opt.load_state_dict({"state": {}, "param_groups": [{"params": [0, 1], "lr": 1e-3, "betas": (0.9, 0.999), "eps": 1e-8}]})
    opt.load_state_dict(torch.optim.Adam(params, lr=1e-3).state_dict())  # fresh optimizer: empty state
    assert opt.step_count.item() == 0.0 and not opt.exp_avg.any()
