"""GPU: whole-network parity of the drop-in modules against the oracle (north_star tolerance: outputs within 1e-3
relative-L2 of the fp32 reference; gradients within 2e-2 with bf16 gradient operands)."""
import pytest
import torch

from nbss_b200.io import Norm, STFT, SeparationPipeline
from nbss_b200.spatialnet import SpatialNet
from oracle import spatialnet_oracle as O


def _net(cfg, P):
    net = SpatialNet(dim_input=cfg["dim_input"], dim_output=cfg["dim_output"], dim_squeeze=8, num_layers=cfg["num_layers"],
                     num_freqs=cfg["num_freqs"], dim_hidden=96, dim_ffn=192, num_heads=4).cuda()
    net.load_state_dict({k: v.clone() for k, v in P.items()}, strict=True)
    return net


def _leaf(P):
    seen, out = {}, {}
    for k, v in P.items():
        if id(v) not in seen:
            seen[id(v)] = v.clone().requires_grad_(True)
        out[k] = seen[id(v)]
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("T", [250, 251])
def test_forward_small_6ch_f129(T):
    """BASELINE configs[1] shape per utterance: 6ch, F=129, T=250 (and the 4 s / T=251 case)."""
    cfg = O.SMALL_CFG
    P = O.synth_params(cfg, 21)
    net = _net(cfg, P).eval()
    x = torch.randn(2, 129, T, 12, generator=torch.Generator().manual_seed(T))
    with torch.no_grad():
        y = net(x.cuda())
        net.check_device_errors()
        ref = O.spatialnet_forward(P, x, cfg)
    e = O.rel_l2(y.cpu(), ref)
    assert e < 1e-3, f"rel-L2 {e:.3e}"


@pytest.mark.gpu
def test_cfg1_small_2ch_f65_t64():
    """BASELINE configs[0] (2ch, F=65, T=64, batch 1) on the GPU path against the oracle."""
    cfg = dict(O.SMALL_CFG, dim_input=4, num_freqs=65)
    P = O.synth_params(cfg, 102)
    net = _net(cfg, P).eval()
    x = torch.randn(1, 65, 64, 4, generator=torch.Generator().manual_seed(12))
    with torch.no_grad():
        y = net(x.cuda())
        ref = O.spatialnet_forward(P, x, cfg)
    assert O.rel_l2(y.cpu(), ref) < 1e-3


@pytest.mark.gpu
def test_forward_backward_16khz_f257():
    """The reference's 16 kHz framing (n_fft 512, F = 257; models/io/stft.py:8-12): forward 1e-3, parameter gradients of a
    2-layer network against fp64 autograd (the full-band LinearGroup runs on the fp32 kernels for F > 256)."""
    cfg = dict(O.SMALL_CFG, num_layers=2, num_freqs=257)
    P = O.synth_params(cfg, 35)
    Pl = {}
    seen = {}
    for k, v in P.items():
        if id(v) not in seen:
            seen[id(v)] = v.double().requires_grad_(True)
        Pl[k] = seen[id(v)]
    net = _net(cfg, P)
    g = torch.Generator().manual_seed(6)
    x = torch.randn(1, 257, 60, 12, generator=g)
    dy = torch.randn(1, 257, 60, 4, generator=g)
    y = net(x.cuda())
    y.backward(dy.cuda())
    torch.cuda.synchronize()
    net.check_device_errors()
    ref = O.spatialnet_forward(Pl, x.double(), cfg)
    ref.backward(dy.double())
    assert O.rel_l2(y.detach().cpu(), ref.detach()) < 1e-3
    errs = {n: O.rel_l2(p.grad.cpu().reshape(-1), Pl[n].grad.reshape(-1)) for n, p in net.named_parameters()}
    bad = {k: f"{v:.2e}" for k, v in errs.items() if not v < 3e-2}
    assert not bad, bad


@pytest.mark.gpu
def test_forward_backward_grads():
    cfg = dict(O.SMALL_CFG, num_layers=3)
    P = O.synth_params(cfg, 33)
    Pl = _leaf(P)
    net = _net(cfg, P)
    g = torch.Generator().manual_seed(5)
    x = torch.randn(2, 129, 100, 12, generator=g)
    dy = torch.randn(2, 129, 100, 4, generator=g)
    y = net(x.cuda())
    y.backward(dy.cuda())
    torch.cuda.synchronize()
    net.check_device_errors()
    assert net.grads_alias_flat(), "parameter gradients must be views of the single flat buffer (one all-reduce)"
    ref = O.spatialnet_forward(Pl, x, cfg)
    ref.backward(dy)
    assert O.rel_l2(y.detach().cpu(), ref.detach()) < 1e-3
    errs = {}
    for name, p in net.named_parameters():
        errs[name] = O.rel_l2(p.grad.cpu().reshape(-1), Pl[name].grad.reshape(-1))
    bad = {k: f"{v:.2e}" for k, v in errs.items() if not v < 3e-2}
    assert not bad, f"gradient rel-L2 > 3e-2: {bad}"
    worst = max(errs.values())
    print(f"worst parameter-gradient rel-L2 {worst:.2e}")


@pytest.mark.gpu
def test_wave_to_wave_pipeline_and_module_api():
    """TrainModule.forward (SharedTrainer.py:104-132) two ways: the fused SeparationPipeline, and the reference's own
    call sequence written against the drop-in STFT / Norm / SpatialNet modules."""
    cfg = dict(O.SMALL_CFG, num_layers=2)
    P = O.synth_params(cfg, 44)
    net = _net(cfg, P)
    wave = 0.1 * torch.randn(2, 6, 128 * 63, generator=torch.Generator().manual_seed(9))
    with torch.no_grad():
        ref = O.io_forward(P, wave, cfg, 256, 128, 0)
    pipe = SeparationPipeline(net, 256, 128, channels=[0, 1, 2, 3, 4, 5], ref_channel=0)
    est = pipe(wave.cuda())
    assert O.rel_l2(est.detach().cpu(), ref) < 1e-3
    # gradient flows from the time-domain output to the network parameters
    est.square().mean().backward()
    assert net.decoder.weight.grad is not None and torch.isfinite(net.decoder.weight.grad).all()
    # reference call sequence with the drop-in modules
    stft, norm = STFT(256, 128).cuda(), Norm("frequency")
    with torch.no_grad():
        x = wave.cuda()
        X, stft_paras = stft.stft(x)
        B, C, F, T = X.shape
        X, (Xr, XrMM) = norm.norm(X, ref_channel=0)
        Xp = torch.view_as_real(X.permute(0, 2, 3, 1)).reshape(B, F, T, -1)
        out = net(Xp)
        out = torch.view_as_complex(out.float().reshape(B, F, T, -1, 2)).permute(0, 3, 1, 2)
        Yr = norm.inorm(out, (Xr, XrMM))
        y2 = stft.istft(Yr, stft_paras)
    assert O.rel_l2(y2.cpu(), ref) < 1e-3


@pytest.mark.gpu
@pytest.mark.parametrize("B,Ts,zero_mean", [(3, 32000, False), (1, 1000, False), (5, 31872, True)])
def test_si_sdr_pit_loss(B, Ts, zero_mean):
    """csrc/loss.cu against the oracle restatement of torchmetrics SI-SDR + permutation-wise PIT (models/io/loss.py:21-29,
    95-118): loss 1e-5, permutations equal, gradient wrt the estimate 1e-4 rel-L2."""
    from nbss_b200.loss import NegSiSdrPitLoss, neg_si_sdr_pit

    g = torch.Generator().manual_seed(B + Ts)
    ref = 0.1 * torch.randn(B, 2, Ts, generator=g) + (0.02 if zero_mean else 0.0)
    mix = torch.rand(B, 1, 1, generator=g)
    est = ref[:, [1, 0]] * (0.5 + mix) + 0.05 * torch.randn(B, 2, Ts, generator=g)  # mostly the swapped permutation
    est[0] = ref[0] * 0.8 + 0.03 * torch.randn(2, Ts, generator=g)                  # ... and one identity case
    est = est.requires_grad_(True)
    l_ref, lb_ref, p_ref = O.neg_si_sdr_pit(est.double(), ref.double(), zero_mean)
    l_ref.backward()
    est_d = est.detach().cuda().requires_grad_(True)
    loss, loss_b, perms = neg_si_sdr_pit(est_d, ref.cuda(), zero_mean)
    (2.0 * loss).backward()
    torch.cuda.synchronize()
    assert abs(loss.item() - l_ref.item()) < 1e-5 * max(1.0, abs(l_ref.item()))
    assert torch.allclose(loss_b.cpu().double(), lb_ref, rtol=1e-5, atol=1e-5)
    assert torch.equal(perms.cpu().long(), p_ref)
    assert O.rel_l2(est_d.grad.cpu().double(), 2.0 * est.grad.double()) < 1e-4
    # module form mirrors Loss.forward (loss, perms, reordered estimate)
    with torch.no_grad():
        lm_ref, _, pm_ref = O.neg_si_sdr_pit(est.double(), ref.double(), False)  # the module uses the reference's zero_mean=False
    l2, p2, yh = NegSiSdrPitLoss()(est_d.detach(), ref.cuda(), reorder=True)
    assert abs(l2.item() - lm_ref.item()) < 1e-5 * max(1.0, abs(lm_ref.item()))
    assert torch.equal(p2.cpu(), pm_ref)
    assert torch.equal(yh.cpu(), torch.gather(est.detach(), 1, pm_ref[:, :, None].expand(-1, -1, Ts)))


@pytest.mark.gpu
def test_flat_clip_adam_resume_across_optimizers():
    """Checkpoint / resume: FlatClipAdam.state_dict() is torch.optim.Adam's format (what Lightning stores), in both directions —
    after two steps the two optimizers swap states and the third step still agrees to 2e-6."""
    import copy

    from nbss_b200.optim import FlatClipAdam

    cfg = dict(O.SMALL_CFG, num_layers=1)
    net = _net(cfg, O.synth_params(cfg, 13))
    ref = copy.deepcopy(net)
    ref_params = [p for _, p in ref.named_parameters()]
    opt_ref = torch.optim.Adam(ref_params, lr=1e-3)
    opt = FlatClipAdam(net, lr=1e-3, max_norm=5.0)
    g = torch.Generator().manual_seed(5)
    for it in range(3):
        if it == 2:  # swap: each optimizer continues from the OTHER one's saved state
            sd_flat, sd_torch = opt.state_dict(), copy.deepcopy(opt_ref.state_dict())
            opt = FlatClipAdam(net, lr=7.0, max_norm=5.0)
            opt.load_state_dict(sd_torch)
            opt_ref = torch.optim.Adam(ref_params, lr=7.0)
            opt_ref.load_state_dict(sd_flat)
            assert opt.lr == 1e-3 and opt_ref.param_groups[0]["lr"] == 1e-3 and opt.step_count.item() == 2.0
        x = torch.randn(1, 129, 24, 12, generator=g).cuda()
        dy = 2e-4 * torch.randn(1, 129, 24, 4, generator=g).cuda()
        opt.zero_grad(set_to_none=True)
        net(x).backward(dy)
        for (_, p1), p2 in zip(net.named_parameters(), ref_params):
            p2.grad = p1.grad.detach().clone()
        torch.nn.utils.clip_grad_norm_(ref_params, 5.0)
        opt_ref.step()
        opt.step()
        torch.cuda.synchronize()
        for (n1, p1), p2 in zip(net.named_parameters(), ref_params):
            assert torch.allclose(p1, p2, rtol=0, atol=2e-6), (it, n1, (p1 - p2).abs().max().item())


@pytest.mark.gpu
def test_si_sdr_pit_loss_torchmetrics_known_answer():
    """csrc/loss.cu on the vector torchmetrics publishes in the doctest of permutation_invariant_training (the library
    models/io/loss.py:5-9 calls): best SI-SDR -5.1091 dB with the identity permutation (tests/golden/torchmetrics_kat.json)."""
    import json
    import os

    from nbss_b200.loss import neg_si_sdr_pit

    k = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "torchmetrics_kat.json")))["pit_si_sdr_max"]
    loss, loss_b, perms = neg_si_sdr_pit(torch.tensor(k["preds"]).cuda(), torch.tensor(k["target"]).cuda())
    torch.cuda.synchronize()
    assert abs(loss.item() + k["best_metric"][0]) < 2e-4
    assert abs(loss_b.cpu()[0].item() + k["best_metric"][0]) < 2e-4
    assert perms.cpu().tolist() == k["best_perm"]


@pytest.mark.gpu
def test_flat_clip_adam_matches_torch():
    """nbss_clip_adam (two launches over the flat gradient buffer) against clip_grad_norm_(5) + torch.optim.Adam(1e-3) fed
    with the SAME gradients (Adam's first steps are sign-like, so independently computed gradients would not do)."""
    import copy

    from nbss_b200.optim import FlatClipAdam

    cfg = dict(O.SMALL_CFG, num_layers=2)
    P = O.synth_params(cfg, 12)
    net = _net(cfg, P)
    ref = copy.deepcopy(net)
    ref_params = [p for _, p in ref.named_parameters()]
    opt_ref = torch.optim.Adam(ref_params, lr=1e-3)
    opt = FlatClipAdam(net, lr=1e-3, max_norm=5.0)
    g = torch.Generator().manual_seed(3)
    for it in range(4):
        x = torch.randn(1, 129, 40, 12, generator=g).cuda()
        dy = (30.0 if it == 0 else 2e-4) * torch.randn(1, 129, 40, 4, generator=g).cuda()  # step 0 is clipped, the others not
        opt.zero_grad(set_to_none=True)
        net(x).backward(dy)
        for (_, p1), p2 in zip(net.named_parameters(), ref_params):
            p2.grad = p1.grad.detach().clone()
        total = torch.nn.utils.clip_grad_norm_(ref_params, 5.0)
        opt_ref.step()
        opt.step()
        torch.cuda.synchronize()
        assert (it == 0) == (total.item() > 5.0), total.item()
        assert abs(opt.grad_norm().item() - total.item()) < 1e-5 * total.item()
        for (n1, p1), p2 in zip(net.named_parameters(), ref_params):
            assert torch.allclose(p1, p2, rtol=0, atol=2e-6), (it, n1, (p1 - p2).abs().max().item())
    # the optimiser invalidated the cached weight images: the next forward uses the updated weights
    y1 = net(x)
    net.engine.invalidate_images()
    assert torch.equal(y1, net(x))


@pytest.mark.gpu
def test_forward_against_the_unmodified_reference_module():
    """Parity with the reference ITSELF: the unmodified `models.arch.SpatialNet.SpatialNet` ran on the host in fp32 on the input of
    test_forward_small_6ch_f129[250] (every 29th output value stored by tests/golden/make_golden_parity.py); the CUDA path is within
    1e-3 of it, and the oracle within 2e-5 (what pins the oracle here too)."""
    import os

    import numpy as np

    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "spatialnet_f129_t250.npz"))
    cfg = O.SMALL_CFG
    P = O.synth_params(cfg, 21)
    net = _net(cfg, P).eval()
    x = torch.randn(2, 129, 250, 12, generator=torch.Generator().manual_seed(250))
    assert abs(x.double().sum().item() - float(z["x_sum"])) < 1e-6, "torch's seeded generator no longer gives the stored input"
    ref = torch.from_numpy(z["y_every29"])
    with torch.no_grad():
        y = net(x.cuda())
        net.check_device_errors()
        orc = O.spatialnet_forward(P, x, cfg)
    assert O.rel_l2(orc.reshape(-1)[::29], ref) < 2e-5
    e = O.rel_l2(y.cpu().reshape(-1)[::29], ref)
    assert e < 1e-3, f"rel-L2 vs the unmodified reference {e:.3e}"
