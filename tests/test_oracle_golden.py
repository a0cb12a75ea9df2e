"""CPU: pins oracle/spatialnet_oracle.py against fixtures generated from the UNMODIFIED reference modules
(tests/golden/make_golden*.py)."""
import os

import numpy as np
import torch

from oracle import spatialnet_oracle as O

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
TINY = dict(dim_input=4, dim_output=4, dim_squeeze=4, num_layers=2, num_freqs=17, encoder_kernel_size=5,
            dim_hidden=32, dim_ffn=64, num_heads=4, kernel_size=(5, 3), conv_groups=(8, 8))
CFG1 = dict(dim_input=4, dim_output=4, dim_squeeze=8, num_layers=8, num_freqs=65, encoder_kernel_size=5,
            dim_hidden=96, dim_ffn=192, num_heads=4, kernel_size=(5, 3), conv_groups=(8, 8))


LARGE = dict(dim_input=12, dim_output=4, dim_squeeze=16, num_layers=2, num_freqs=129, encoder_kernel_size=5,
             dim_hidden=192, dim_ffn=384, num_heads=4, kernel_size=(5, 3), conv_groups=(8, 8))


def _leaf_params(P):
    """requires_grad leaves; the shared full.* tensor stays ONE leaf under all its keys."""
    seen, out = {}, {}
    for k, v in P.items():
        if id(v) not in seen:
            seen[id(v)] = v.clone().requires_grad_(True)
        out[k] = seen[id(v)]
    return out


def test_tiny_forward_backward_matches_reference():
    z = np.load(os.path.join(G, "tiny_fwd_bwd.npz"))
    P = _leaf_params(O.synth_params(TINY, seed=101))
    x = torch.from_numpy(z["x"]).requires_grad_(True)
    y = O.spatialnet_forward(P, x, TINY)
    assert O.rel_l2(y.detach(), torch.from_numpy(z["y"])) < 2e-6
    y.backward(torch.from_numpy(z["dy"]))
    assert O.rel_l2(x.grad, torch.from_numpy(z["dx"])) < 1e-5
    checked = 0
    for k in z.files:
        if not k.startswith("grad."):
            continue
        name = k[5:]
        assert O.rel_l2(P[name].grad, torch.from_numpy(z[k])) < 2e-5, name
        checked += 1
    assert checked >= 60


def test_large_widths_forward_and_grad_norms():
    """The 'large' layer widths of configs/SpatialNet.yaml (H=192, Hf=384, dim_squeeze=16; SURVEY 8f rank 4): the oracle is
    already pinned for the next tile shapes."""
    z = np.load(os.path.join(G, "large_widths_f129_t10.npz"))
    P = _leaf_params(O.synth_params(LARGE, seed=105))
    y = O.spatialnet_forward(P, torch.from_numpy(z["x"]), LARGE)
    assert O.rel_l2(y.detach(), torch.from_numpy(z["y"])) < 5e-6
    y.backward(torch.from_numpy(z["dy"]))
    n = 0
    for k in z.files:
        if k.startswith("gnorm."):
            got = float(P[k[6:]].grad.double().norm())
            assert abs(got - float(z[k])) <= 1e-4 * float(z[k]) + 1e-12, k
            n += 1
    assert n >= 60


def test_nbc2_oracle_matches_reference():
    """oracle/nbc2_oracle.py (BASELINE configs[3]; SURVEY 8f rank 2) against the unmodified reference NBC2."""
    from oracle import nbc2_oracle as N2

    z = np.load(os.path.join(G, "nbc2_small_f17_t12.npz"))
    cfg = dict(N2.NBC2_SMALL, n_layers=2, num_freqs=17)
    P = {k: v.clone().requires_grad_(True) for k, v in N2.synth_params(cfg, seed=106).items()}
    y = N2.nbc2_forward(P, torch.from_numpy(z["x"]), cfg)
    assert O.rel_l2(y.detach(), torch.from_numpy(z["y"])) < 5e-6
    y.backward(torch.from_numpy(z["dy"]))
    n = 0
    for k in z.files:
        if k.startswith("gnorm."):
            got = float(P[k[6:]].grad.double().norm())
            assert abs(got - float(z[k])) <= 1e-4 * float(z[k]) + 1e-12, k
            n += 1
    assert n == len(P)


def test_cfg1_small_2ch_forward_and_grad_norms():
    """BASELINE.json configs[0]: SpatialNet-small 2ch F=65 T=64 forward on CPU, batch=1."""
    z = np.load(os.path.join(G, "cfg1_small_2ch_f65_t64.npz"))
    P = _leaf_params(O.synth_params(CFG1, seed=102))
    y = O.spatialnet_forward(P, torch.from_numpy(z["x"]), CFG1)
    assert tuple(y.shape) == (1, 65, 64, 4)
    assert O.rel_l2(y.detach(), torch.from_numpy(z["y"])) < 5e-6
    y.backward(torch.from_numpy(z["dy"]))
    for k in z.files:
        if k.startswith("gnorm."):
            got = float(P[k[6:]].grad.double().norm())
            assert abs(got - float(z[k])) <= 1e-4 * float(z[k]) + 1e-12, k


def test_small_6ch_f129_forward():
    z = np.load(os.path.join(G, "small_6ch_f129_t12.npz"))
    P = O.synth_params(O.SMALL_CFG, seed=103)
    with torch.no_grad():
        y = O.spatialnet_forward(P, torch.from_numpy(z["x"]), O.SMALL_CFG)
    assert O.rel_l2(y, torch.from_numpy(z["y"])) < 5e-6


def test_param_count_matches_published():
    """1.2 M parameters for SpatialNet-small (images/model_size_and_flops.png; SURVEY.md §2.2: 1,191,092)."""
    P = O.synth_params(O.SMALL_CFG, seed=0)
    n = sum(v.numel() for v in {id(v): v for v in P.values()}.values())
    assert n == 1_191_092


def test_framing_matches_reference():
    z = np.load(os.path.join(G, "framing.npz"))
    wave = torch.from_numpy(z["wave"])
    X = O.stft(wave, 32, 16)
    Xg = torch.complex(torch.from_numpy(z["X_re"]), torch.from_numpy(z["X_im"]))
    assert O.rel_l2(torch.view_as_real(X), torch.view_as_real(Xg)) < 2e-6
    P = O.synth_params(TINY, seed=101)
    with torch.no_grad():
        yw = O.io_forward(P, wave, TINY, n_fft=32, n_hop=16)
    assert O.rel_l2(yw, torch.from_numpy(z["y_wave"])) < 1e-5
    # 8 kHz framing of configs/SpatialNet.yaml (n_fft 256, hop 128)
    w8 = torch.from_numpy(z["wave8"])
    X8 = O.stft(w8, 256, 128)
    X8g = torch.complex(torch.from_numpy(z["X8_re"]), torch.from_numpy(z["X8_im"]))
    assert O.rel_l2(torch.view_as_real(X8), torch.view_as_real(X8g)) < 2e-6
    Xn, Xr, XrMM = O.norm_frequency_online(X8g, 0)  # norm applied to the reference's own STFT output
    Xng = torch.complex(torch.from_numpy(z["Xn8_re"]), torch.from_numpy(z["Xn8_im"]))
    assert O.rel_l2(torch.view_as_real(Xn), torch.view_as_real(Xng)) < 2e-6
    assert O.rel_l2(XrMM, torch.from_numpy(z["XrMM8"])) < 1e-6
    rt = O.istft(X8, 256, 128, w8.shape[-1])
    assert O.rel_l2(rt, torch.from_numpy(z["rt8"])) < 2e-6
    assert O.rel_l2(rt, w8) < 1e-5  # STFT -> iSTFT round trip (models/io/stft.py:106-113)


def test_live_reference_layer_taps():
    """The reference's whole network, and its layer 1 alone on the oracle's encoder output (tests/golden/make_golden_parity.py)."""
    z = np.load(os.path.join(G, "layer_taps_tiny.npz"))
    P = O.synth_params(TINY, seed=7)
    x = torch.from_numpy(z["x"])
    with torch.no_grad():
        assert O.rel_l2(O.spatialnet_forward(P, x, TINY), torch.from_numpy(z["y"])) < 2e-6
        assert O.rel_l2(O.layer_forward(torch.from_numpy(z["h"]), P, 1, TINY), torch.from_numpy(z["layer1"])) < 2e-6


def test_oracle_si_sdr_pit_properties():
    """The loss restatement has no golden vector (torchmetrics is absent): pin its defining properties instead —
    scale invariance, the right permutation, and the closed form for a known SNR."""
    g = torch.Generator().manual_seed(0)
    ref = torch.randn(4, 2, 4000, generator=g, dtype=torch.float64)
    noise = torch.randn(4, 2, 4000, generator=g, dtype=torch.float64)
    noise = noise - (noise * ref).sum(-1, keepdim=True) / (ref * ref).sum(-1, keepdim=True) * ref  # orthogonal to ref
    noise = noise * (ref.norm(dim=-1, keepdim=True) / noise.norm(dim=-1, keepdim=True)) * 10 ** (-20 / 20)  # 20 dB
    est = (3.7 * (ref + noise))[:, [1, 0]]  # scaled and speaker-swapped
    loss, loss_b, perms = O.neg_si_sdr_pit(est, ref)
    assert torch.allclose(loss_b, torch.full((4,), -20.0, dtype=torch.float64), atol=1e-6)
    assert abs(loss.item() + 20.0) < 1e-6
    assert torch.equal(perms, torch.tensor([[1, 0]] * 4))
    # zero_mean=True is the plain formula on the centred signals, whatever DC offset they carry
    centred = O.si_sdr(est - est.mean(-1, keepdim=True), ref - ref.mean(-1, keepdim=True))
    assert torch.allclose(O.si_sdr(est + 0.3, ref - 0.1, zero_mean=True), centred, atol=1e-9)


def test_loss_oracle_torchmetrics_known_answers():
    """Pins the loss restatement (oracle si_sdr / snr / neg_si_sdr_pit) to the known-answer vectors torchmetrics publishes in
    the doctests of the three functions models/io/loss.py:5-9 imports (tests/golden/torchmetrics_kat.json; 4 printed decimals)."""
    import json
    import os

    kat = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "torchmetrics_kat.json")))
    k = kat["si_sdr"]
    assert abs(O.si_sdr(torch.tensor(k["preds"]), torch.tensor(k["target"])).item() - k["value"]) < 5e-5
    k = kat["snr"]
    assert abs(O.snr(torch.tensor(k["preds"]), torch.tensor(k["target"])).item() - k["value"]) < 5e-5
    k = kat["pit_si_sdr_max"]
    # torchmetrics maximises si_sdr over the permutations; the reference minimises neg_si_sdr (loss.py:109-110): same optimum
    loss, loss_b, perms = O.neg_si_sdr_pit(torch.tensor(k["preds"]), torch.tensor(k["target"]))
    assert torch.allclose(-loss_b, torch.tensor(k["best_metric"]), atol=5e-5)
    assert perms.tolist() == k["best_perm"]
    assert abs(loss.item() + k["best_metric"][0]) < 5e-5


def test_eager_opset_restatement_matches_oracle():
    """oracle/eager_gpu.py (the reference's op-set as torch.nn.functional calls: what bench.py times on the GPU as the
    eager baseline and on the host cores as the CPU arm) computes the same function as the pinned oracle: identical in
    fp64 (1e-10), and its fp32 gradients are within 5e-4 of fp64 autograd (the explicit-math oracle's own fp32 gradients are
    only good to ~3e-3 on some tensors, which is why the GPU gradient tests compare against fp64)."""
    from oracle import eager_gpu as E

    cfg = dict(O.SMALL_CFG, num_layers=2)
    g = torch.Generator().manual_seed(0)
    x = 0.1 * torch.randn(2, 6, 128 * 20, generator=g)
    tgt = 0.1 * torch.randn(2, 2, 128 * 20, generator=g)

    def run(fwd, loss, dt):
        P = O.synth_params(cfg, 3, dtype=dt)
        seen, Pl = {}, {}
        for k, v in P.items():
            if id(v) not in seen:
                seen[id(v)] = v.clone().requires_grad_(True)
            Pl[k] = seen[id(v)]
        est = fwd(Pl, x.to(dt), cfg)
        loss(est, tgt.to(dt)).backward()
        return est.detach(), {k: v.grad for k, v in Pl.items()}

    o64, g_o64 = run(O.io_forward, lambda e, t: O.neg_si_sdr_pit(e, t)[0], torch.float64)
    e64, g_e64 = run(E.io_forward, E.neg_si_sdr_pit2, torch.float64)
    e32, g_e32 = run(E.io_forward, E.neg_si_sdr_pit2, torch.float32)
    assert O.rel_l2(e64, o64) < 1e-10
    for k in g_o64:
        assert O.rel_l2(g_e64[k], g_o64[k]) < 1e-10, k
        assert O.rel_l2(g_e32[k], g_o64[k]) < 5e-4, k
    assert O.rel_l2(e32, o64) < 5e-5


def test_online_oracle_matches_reference():
    """oracle/online_oracle.py (BASELINE configs[4]; SURVEY 8f rank 3) against the unmodified reference OnlineSpatialNet
    (attention='mhsa(251)', T = 270): the executed function is causal attention over all past frames (torch drops the window mask
    for need_weights=False, see the oracle's header); the windowed restatement agrees on the first 251 frames."""
    from oracle import online_oracle as OO

    z = np.load(os.path.join(G, "online_f9_t270.npz"))
    cfg = dict(O.SMALL_CFG, num_layers=2, num_freqs=9)
    P = O.synth_params(cfg, 107)
    x = torch.randn(2, 9, 270, 12, generator=torch.Generator().manual_seed(270))
    assert abs(x.double().sum().item() - float(z["x_sum"])) < 1e-6, "torch's seeded generator no longer gives the stored input"
    y = torch.from_numpy(z["y"])
    with torch.no_grad():
        assert O.rel_l2(OO.online_forward(P, x, cfg), y) < 2e-6
        assert O.rel_l2(OO.online_forward(P, x[:, :, :251], cfg, scope=251), y[:, :, :251]) < 2e-6
        yw = OO.online_forward(P, x, cfg, scope=251)
        assert O.rel_l2(yw[:, :, :251], y[:, :, :251]) < 2e-6 and O.rel_l2(yw, y) > 1e-4  # the window matters beyond frame 251
