#!/usr/bin/env python
"""bench.py — T-F frames/sec of the SpatialNet hot path on B200 (BASELINE.json metric, configs[1]).

    python bench.py [--gpus N] [--steps K] [--warmup W]            # N>1: launched by torch.distributed.run
    python bench.py --impl reference ...                           # CPU arm: the oracle port on the host cores

One STEP = one training pass of the hot path over one batch of synthetic 6-channel mixtures:
    stft+norm+pack -> SpatialNet fwd (8 layers) -> unpack+inorm+iSTFT -> SI-SDR/PIT loss -> backward of all of it ->
    (N>1: one NCCL all-reduce of the flat 4.76 MB gradient) -> grad-clip(5) + Adam.
Workload: SpatialNet-small 6ch F=129 T=250, global batch 32 (strong scaling: 32/N utterances per GPU), fp16/bf16
tensor-core operands with fp32 accumulation and fp32 residual stream.
  value : whole-job frames/s with the waveforms already resident in HBM (CUDA events, max over ranks)
  e2e   : the same step through nbss_b200.SeparationPipeline with HOST (pinned) waveforms/targets copied in and the loss
          copied back inside the timed region
  roofline : the dominant kernel of the step, timed live with CUDA events on the launching stream
  cpu_baseline : oracle/ (torch-CPU restatement of the reference) on the host cores, bounded sample, rank 0, N=1
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the bench writes nothing into the tree it runs from (which may be read-only)

import torch  # noqa: E402

CFG = dict(B=32, C=6, F=129, T=250, n_fft=256, hop=128, S=2, L=8)
TS = CFG["hop"] * (CFG["T"] - 1)  # 31872 samples -> T = 250 frames
FLOP_PER_POINT = {  # algorithmic FLOPs per T-F point (SURVEY.md §8d)
    "ffn_fwd": 156_672, "mhsa_fwd": 169_728, "ffn_bwd": 156_672, "ffn_wgrad": 156_672, "mhsa_bwd": 265_728,
    "mhsa_wgrad": 73_728, "fconv_fwd": 11_520, "fconv_bwd": 34_560, "fconv_tc_fwd": 11_520, "fconv_tc_bwd": 34_560, "full_fwd": 5_136, "full_bwd": 10_272, "full_fwd_tc": 5_136, "full_bwd_tc": 10_272,
}
# algorithmic HBM bytes per T-F point with one fused kernel per sub-block and an fp32 stream (SURVEY.md §8d):
# forward = x in + y out; data-gradient = x, dy in + dx out; weight-gradient = x, dy in.  (What the kernels move on top
# of this — 16-bit saves and gradient operands — is design overhead and shows up as a lower fraction.)
BYTES_PER_POINT = {"ffn_fwd": 768, "mhsa_fwd": 768, "fconv_tc_fwd": 768, "full_fwd": 768, "full_fwd_tc": 768, "full_bwd_tc": 1152, "ffn_bwd": 1152, "mhsa_bwd": 1152,
                   "fconv_tc_bwd": 1152, "full_bwd": 1152, "ffn_wgrad": 768, "mhsa_wgrad": 768}


def synth_batch(b, seed, device="cpu"):
    """Synthetic 6-ch mixtures: 2 'speakers' = white noise through random 64-tap 6-ch FIRs + white noise at 10 dB."""
    g = torch.Generator().manual_seed(seed)
    src = torch.randn(b, CFG["S"], 1, TS + 63, generator=g)
    fir = torch.randn(b, CFG["S"], CFG["C"], 64, generator=g) * torch.exp(-torch.arange(64) / 8.0)
    img = torch.nn.functional.conv1d(src.reshape(1, b * CFG["S"], -1), fir.reshape(b * CFG["S"] * CFG["C"], 1, 64),
                                     groups=b * CFG["S"]).reshape(b, CFG["S"], CFG["C"], TS)
    mix = img.sum(1)
    mix = mix + torch.randn(mix.shape, generator=g) * mix.std() * 10 ** (-10 / 20)
    scale = 0.1 / mix.std()
    return (mix * scale).contiguous(), (img[:, :, 0] * scale).contiguous()  # x [b,C,Ts], targets at ref channel [b,S,Ts]


class ClockSampler:
    def __init__(self, dev):
        self.dev, self.proc, self.rows = dev, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.dev}", "--query-gpu=clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
                 "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap",
                 "--format=csv,noheader,nounits", "-lms", "200"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        rows = [r for r in self.rows if len(r) >= 7]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        clk = sorted(float(r[0]) for r in rows)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[3 + i].lower().startswith("active") for r in rows)]
        return {"sm_mhz": clk[len(clk) // 2], "sm_max_mhz": float(rows[0][1]), "power_w_max": max(float(r[2]) for r in rows),
                "samples": len(rows), "reasons": reasons}


def log(msg):
    sys.stderr.write(f"[bench {time.strftime('%H:%M:%S')}] {msg}\n")
    sys.stderr.flush()


def cpu_oracle_subprocess(threads, reps, timeout_s=420):
    """Runs cpu_oracle_step in a child process under a timeout so a slow host cannot stall the GPU bench line.
    Returns (frames/s, seconds per pass, sample description)."""
    code = (f"import sys, json; sys.path.insert(0, {ROOT!r}); import bench; "
            f"print(json.dumps(bench.cpu_oracle_step({threads}, 4, {reps})))")
    try:
        r = subprocess.run([sys.executable, "-B", "-c", code], capture_output=True, text=True, timeout=timeout_s)
        return tuple(json.loads(r.stdout.strip().splitlines()[-1]))
    except Exception as e:  # timeout / parse error
        return None, None, f"cpu baseline unavailable: {type(e).__name__}"


def cpu_oracle_step(threads, b=4, reps=2):
    """One training pass of the same path on the host cores through the reference's own op-set (oracle/eager_gpu.py: the
    torch.nn.functional calls the reference's modules make, pinned to the oracle and the golden vectors by
    tests/test_oracle_golden.py): forward + autograd backward, all host threads."""
    from oracle import eager_gpu as E
    from oracle import spatialnet_oracle as O
    torch.set_num_threads(threads)
    P = O.synth_params(O.SMALL_CFG, 2)
    leaves, Pl = {}, {}
    for k, v in P.items():
        if id(v) not in leaves:
            leaves[id(v)] = v.clone().requires_grad_(True)
        Pl[k] = leaves[id(v)]
    x, tgt = synth_batch(b, 1234)
    ts = []
    for i in range(reps + 1):
        t0 = time.perf_counter()
        est = E.io_forward(Pl, x, O.SMALL_CFG, CFG["n_fft"], CFG["hop"], 0)
        loss = E.neg_si_sdr_pit2(est, tgt)
        loss.backward()
        ts.append(time.perf_counter() - t0)
        if sum(ts) > 120:  # bounded sample: stop once ~2 minutes of CPU work have been spent
            break
    timed = ts[1:] if len(ts) > 1 else ts
    t = min(timed)
    note = f"1 warm-up + {len(ts) - 1} timed (best)" if len(ts) > 1 else "single cold pass (host too slow for a warm-up within the bound)"
    return b * CFG["T"] / t, t, f"B={b} utterance(s) x T=250 frames, wave->wave fwd+bwd, reference op-set (torch CPU kernels), {threads} threads, {note}"


def gpu_eager_baseline(dev, batch, steps=3, warmup=2):
    """The reference's op-set in PyTorch eager on this GPU (oracle/eager_gpu.py: cuDNN / cuBLAS / SDPA / cuFFT calls in the
    reference's module order), the same training step (wave -> wave, SI-SDR + PIT, backward, clip + Adam): fp32 with TF32
    allowed (models/utils/base_cli.py:24-25) and bf16 autocast (Lightning 'bf16-mixed').  Largest batch <= `batch` that fits."""
    from oracle import eager_gpu as E
    from oracle import spatialnet_oracle as O

    out = {}
    old = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    torch.backends.cuda.matmul.allow_tf32 = True
    torch.backends.cudnn.allow_tf32 = True
    try:
        for mode in ("fp32_tf32", "bf16_autocast"):
            b = batch
            while b >= 1:
                try:
                    torch.manual_seed(2)
                    P = O.synth_params(O.SMALL_CFG, 2)
                    leaves, Pl = {}, {}
                    for k, v in P.items():
                        if id(v) not in leaves:
                            leaves[id(v)] = v.to(dev).requires_grad_(True)
                        Pl[k] = leaves[id(v)]
                    params = list(leaves.values())
                    opt = torch.optim.Adam(params, lr=1e-3, fused=True)
                    x, y = (t.to(dev) for t in synth_batch(b, seed=777))

                    def one():
                        opt.zero_grad(set_to_none=True)
                        with torch.autocast("cuda", dtype=torch.bfloat16, enabled=(mode == "bf16_autocast")):
                            est = E.io_forward(Pl, x, O.SMALL_CFG, CFG["n_fft"], CFG["hop"], 0)
                        loss = E.neg_si_sdr_pit2(est.float(), y)
                        loss.backward()
                        torch.nn.utils.clip_grad_norm_(params, 5.0, foreach=True)
                        opt.step()
                        return loss

                    for _ in range(warmup):
                        one()
                    torch.cuda.synchronize()
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    for _ in range(steps):
                        loss = one()
                    e1.record()
                    torch.cuda.synchronize()
                    ms = e0.elapsed_time(e1) / steps
                    out[mode] = {"ms_per_step": round(ms, 2), "frames_per_s": round(b * CFG["T"] / (ms * 1e-3), 1), "batch": b,
                                 "ms_per_step_scaled_to_batch": round(ms * batch / b, 2), "loss": float(loss),
                                 "peak_mem_gb": round(torch.cuda.max_memory_allocated(dev) / 2**30, 1)}
                    break
                except torch.OutOfMemoryError:
                    b //= 2
                finally:
                    Pl = leaves = params = opt = x = y = None
                    import gc
                    gc.collect()
                    torch.cuda.empty_cache()
                    torch.cuda.reset_peak_memory_stats(dev)
            log(f"eager baseline {mode}: {out.get(mode)}")
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old
    out["what"] = ("reference op-set (oracle/eager_gpu.py: F.conv1d / F.multi_head_attention_forward (SDPA) / F.layer_norm / "
                   "F.group_norm / torch.stft / torch.istft in the reference's module order), same training step, PyTorch eager")
    return out


def bench_nbc2(dev, steps=5, warmup=3, batch=64, eager=True):
    """BASELINE configs[3]: NBC2 (models/arch/NBC2.py) small, 8-channel input (dim_input 16), F=257, T=250, inference, batch 64.
    Device-resident and end-to-end (pinned host input copied in, output copied back) frames/s of nbss_b200.nbc2.NBC2, next to
    the oracle's eager torch restatement of the reference on the same GPU (largest batch <= `batch` that fits)."""
    from nbss_b200.nbc2 import NBC2
    from oracle import nbc2_oracle as N2

    B, F, T, Cin = batch, 257, 250, 16
    cfg = N2.NBC2_SMALL
    torch.manual_seed(2)
    net = NBC2(dim_input=Cin, dim_output=4, n_layers=cfg["n_layers"], dim_hidden=96, dim_ffn=192, num_freqs=F).to(dev).eval()
    g = torch.Generator().manual_seed(5)
    x_host = torch.randn(B, F, T, Cin, generator=g).pin_memory()
    x = x_host.to(dev)
    y_host = torch.empty(B, F, T, 4).pin_memory()

    def timed(fn):
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / steps

    ms = timed(lambda: net(x))

    def e2e():
        xd = x_host.to(dev, non_blocking=True)
        y_host.copy_(net(xd), non_blocking=True)

    ms_e2e = timed(e2e)
    net.check_device_errors()
    out = {"workload": f"NBC2-small 8ch F=257 T=250 inference, batch={B} (BASELINE configs[3])", "ms_per_step": round(ms, 3),
           "frames_per_s": round(B * T / (ms * 1e-3), 1), "e2e": {"ms_per_step": round(ms_e2e, 3), "frames_per_s": round(B * T / (ms_e2e * 1e-3), 1),
                                                                  "h2d_bytes_per_step": x_host.numel() * 4, "d2h_bytes_per_step": y_host.numel() * 4},
           "launches_per_step": 2 + 5 * cfg["n_layers"] + cfg["n_layers"]}
    del net
    if eager:
        P = {k: v.to(dev) for k, v in N2.synth_params(cfg, 2).items()}
        b = B
        while b >= 1:
            try:
                xe = x[:b].contiguous()
                with torch.no_grad():
                    ms_e = timed(lambda: N2.nbc2_forward(P, xe, cfg))
                out["gpu_eager_baseline"] = {"ms_per_step": round(ms_e, 2), "batch": b, "frames_per_s": round(b * T / (ms_e * 1e-3), 1),
                                             "what": "oracle/nbc2_oracle.py (torch restatement of the reference's NBC2) in PyTorch eager, fp32"}
                break
            except torch.OutOfMemoryError:
                b //= 2
                torch.cuda.empty_cache()
    torch.cuda.empty_cache()
    return out


def bench_long(dev, seconds=32, steps=3, warmup=2, eager=True):
    """Validation / test-time inference on a whole utterance (SharedTrainer.py:134-189: no 4 s crop): one 32 s, 8 kHz, 6-channel
    recording = T = 2001 STFT frames, wave -> wave through nbss_b200.SeparationPipeline under torch.no_grad() — the chunked
    long-sequence kernels (mhsa_fwd.cu LONG 1/2, ffn_fwd.cu MODE 3/4).  Device-resident and end to end (pinned host wave in, host
    estimates out); next to it the reference's op-set in PyTorch eager on the same GPU (forward only)."""
    from nbss_b200.io import SeparationPipeline
    from nbss_b200.spatialnet import SpatialNet
    from oracle import eager_gpu as E
    from oracle import spatialnet_oracle as O

    Ts = CFG["hop"] * (seconds * 8000 // CFG["hop"])
    T = Ts // CFG["hop"] + 1
    torch.manual_seed(2)
    net = SpatialNet(dim_input=2 * CFG["C"], dim_output=2 * CFG["S"], dim_squeeze=8, num_layers=CFG["L"], num_freqs=CFG["F"], dim_hidden=96,
                     dim_ffn=192, num_heads=4).to(dev).eval()
    pipe = SeparationPipeline(net, CFG["n_fft"], CFG["hop"], channels=None, ref_channel=0)
    x_host = (0.1 * torch.randn(1, CFG["C"], Ts, generator=torch.Generator().manual_seed(9))).pin_memory()
    y_host = torch.empty(1, CFG["S"], Ts).pin_memory()
    x = x_host.to(dev)

    def timed(fn):
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / steps

    with torch.no_grad():
        ms = timed(lambda: pipe(x))

        def e2e():
            y_host.copy_(pipe(x_host.to(dev, non_blocking=True)), non_blocking=True)

        ms_e2e = timed(e2e)
    net.check_device_errors()
    out = {"workload": f"SpatialNet-small 6ch F=129, one {seconds} s utterance (T={T} frames), inference wave->wave", "ms_per_utt": round(ms, 2),
           "frames_per_s": round(T / (ms * 1e-3), 1), "real_time_factor": round(ms * 1e-3 / seconds, 5),
           "e2e": {"ms_per_utt": round(ms_e2e, 2), "h2d_bytes_per_step": x_host.numel() * 4, "d2h_bytes_per_step": y_host.numel() * 4}}
    if eager:
        P = {k: v.to(dev) for k, v in O.synth_params(O.SMALL_CFG, 2).items()}
        old = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
        torch.backends.cuda.matmul.allow_tf32 = True
        torch.backends.cudnn.allow_tf32 = True
        try:
            eg = {}
            for mode in ("fp32_tf32", "bf16_autocast"):
                def one():
                    with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16, enabled=(mode == "bf16_autocast")):
                        return E.io_forward(P, x, O.SMALL_CFG, CFG["n_fft"], CFG["hop"], 0)
                try:
                    eg[mode] = {"ms_per_utt": round(timed(one), 2)}
                except torch.OutOfMemoryError:
                    eg[mode] = {"unavailable": "out of memory"}
                    torch.cuda.empty_cache()
            out["gpu_eager_baseline"] = eg
        finally:
            torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old
    return out


def bench_online(dev, frames=1000, batches=(1, 8, 64)):
    """BASELINE configs[4]: online (causal) SpatialNet, 6 channels, F=129, one 16 ms frame (hop 128 at 8 kHz) per call through
    nbss_b200.online.OnlineSpatialNet.step, the whole step replayed as one CUDA graph.  Latency = host wall clock from handing a
    pinned host frame to having the output frame back on the host (H2D copy + graph + D2H copy + stream sync), p50 / p95 over
    `frames` consecutive frames of one stream (B=1); throughput = frames/s of B parallel streams (device time).  The rings are
    filled before timing, so every step attends over the full 251-frame window (steady state of a long stream)."""
    from nbss_b200.online import OnlineSpatialNet

    torch.manual_seed(2)
    net = OnlineSpatialNet(dim_input=12, dim_output=4, num_layers=8, dim_squeeze=8, num_freqs=129, dim_hidden=96, dim_ffn=192, num_heads=4,
                           attention="mhsa(251)").to(dev).eval()
    out = {"workload": "OnlineSpatialNet mhsa(251) 6ch F=129, 8 layers, one 16 ms frame per call (BASELINE configs[4])", "hop_ms": 16.0, "streams": {}}
    for B in batches:
        state = net.init_state(B)
        x_host = torch.randn(B, 129, 12).pin_memory()
        y_host = torch.empty(B, 129, 4).pin_memory()
        x_dev = x_host.to(dev)
        for _ in range(3):  # warm-up (packs the weights, fills caches)
            net.step(x_dev, state)
        for kc, vc in zip(state.kcache, state.vcache):  # steady state: a full ring (every step then reads all `scope` cached frames)
            kc.normal_(0, 0.3)
            vc.normal_(0, 0.3)
        state.pos.fill_(4 * state.scope)
        torch.cuda.synchronize()
        net.capture_step(state)  # from here on step() = copy the frame into the graph's input + one graph replay
        lat = []
        n = frames if B == 1 else max(100, frames // 5)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(n):
            t0 = time.perf_counter()
            y_dev = net.step(x_host, state)  # pinned host frame in (H2D inside)
            y_host.copy_(y_dev, non_blocking=True)
            torch.cuda.current_stream().synchronize()
            lat.append((time.perf_counter() - t0) * 1e3)
        e1.record()
        torch.cuda.synchronize()
        lat.sort()
        dev_ms = e0.elapsed_time(e1) / n
        out["streams"][str(B)] = {"latency_ms_p50": round(lat[len(lat) // 2], 4), "latency_ms_p95": round(lat[int(len(lat) * 0.95)], 4),
                                  "frames": n, "ms_per_frame_wall": round(dev_ms, 4), "frames_per_s": round(B / (dev_ms * 1e-3), 1),
                                  "real_time_factor": round(dev_ms / 16.0, 5), "state_mb": round(sum(t.numel() * 4 for t in state.kcache + state.vcache) / 2**20, 1)}
    net.check_device_errors()
    return out


def run_torch_gpu(args):
    """--impl torch-gpu: the eager baseline as a bench line of its own (rank 0 only)."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    r = gpu_eager_baseline(dev, args.batch, steps=max(1, min(args.steps, 5)), warmup=max(2, min(args.warmup, 3)))
    best = min((v for k, v in r.items() if isinstance(v, dict)), key=lambda v: v["ms_per_step_scaled_to_batch"])
    _emit(json.dumps({
        "impl": "torch-gpu", "metric": "T-F frames/sec (SpatialNet-small 6ch F=129, training step fwd+bwd incl. STFT/iSTFT)",
        "value": best["frames_per_s"], "unit": "frames/s", "n_gpus": 1, "steps": max(1, min(args.steps, 5)), "warmup": max(2, min(args.warmup, 3)),
        "ms_per_step": best["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "tf32 / bf16 autocast",
        "data": "synthetic", "config": {"workload": "SpatialNet-small 6ch F=129 T=250 fwd+bwd, batch=32 (BASELINE configs[1])", "global_batch": best["batch"]},
        "gpu_eager_baseline": r}))


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = min(os.cpu_count() or 1, 32)
    steps = max(1, min(args.steps, 3))
    fps, t, sample = cpu_oracle_step(cores, b=4, reps=steps)
    _emit(json.dumps({
        "impl": "reference", "metric": "T-F frames/sec (SpatialNet-small 6ch F=129, training step fwd+bwd incl. STFT/iSTFT)",
        "value": fps, "unit": "frames/s", "n_gpus": args.gpus, "steps": steps, "warmup": 1, "ms_per_step": t * 1e3,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "SpatialNet-small 6ch F=129 T=250 fwd+bwd, batch=32 (BASELINE configs[1])", "global_batch": 32,
                   "cpu_sample_batch": 4, "frames_per_utt": CFG["T"]},
        "cpu_baseline": {"value": fps, "unit": "frames/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "rtf": t / (4 * TS / 8000.0),
    }))


_JSON_OUT = None


def _emit(line: str) -> None:
    out = _JSON_OUT if _JSON_OUT is not None else sys.stdout
    out.write(line + "\n")
    out.flush()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="nbss_b200")
    ap.add_argument("--torch-adam", action="store_true", help="clip_grad_norm_ + torch.optim.Adam(fused, capturable) instead of FlatClipAdam")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-eager-baseline", action="store_true", help="skip the PyTorch-eager reference op-set timed on this GPU")
    ap.add_argument("--no-nbc2", action="store_true", help="skip the extra workloads (NBC2 inference = BASELINE configs[3], online streaming = configs[4]) reported under 'extra_workloads'")
    ap.add_argument("--batch", type=int, default=CFG["B"], help="global batch (utterances)")
    ap.add_argument("--profile", action="store_true", help="1 warm-up + 1 step only (for ncu); prints no bench line")
    ap.add_argument("--layers", type=int, default=CFG["L"], help="number of SpatialNet layers (profiling only; default 8)")
    ap.add_argument("--no-graphs", action="store_true", help="launch every kernel eagerly instead of replaying CUDA graphs")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed (estimates, loss, flat gradient, "
                    "updated parameters; rank 0) to DIR/<name>.npy in float32")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    # stdout carries exactly ONE line, the JSON result: everything else that a library writes to file descriptor 1 (NCCL's
    # version banner, for one) is routed to stderr, and the JSON line goes to the saved original stdout
    global _JSON_OUT
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    if args.impl == "reference":
        return run_reference(args)
    if args.impl == "torch-gpu":
        return run_torch_gpu(args)

    import torch.distributed as dist
    from nbss_b200 import ops
    from nbss_b200.io import SeparationPipeline
    from nbss_b200.spatialnet import SpatialNet

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world} (launch with torch.distributed.run)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # stdout carries exactly one JSON line: NCCL's own banner / debug lines (NCCL_DEBUG=VERSION|INFO) go to stderr
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)
    assert args.batch % world == 0
    b_local = args.batch // world

    eager = None
    if world == 1 and not args.no_eager_baseline and not args.profile:
        # the kernel set to beat (SURVEY.md §2.3, §8d): timed first, in this process, then freed
        try:
            eager = gpu_eager_baseline(dev, args.batch)
        except Exception as e:  # never let the baseline take the bench line down
            eager = {"unavailable": f"{type(e).__name__}: {e}"[:200]}
            log(f"eager baseline failed: {eager}")

    torch.manual_seed(2)  # configs/SpatialNet.yaml:1
    net = SpatialNet(dim_input=2 * CFG["C"], dim_output=2 * CFG["S"], dim_squeeze=8, num_layers=args.layers, num_freqs=CFG["F"],
                     dim_hidden=96, dim_ffn=192, num_heads=4).to(dev)
    pipe = SeparationPipeline(net, CFG["n_fft"], CFG["hop"], channels=None, ref_channel=0)
    params = [p for p in net.parameters()]
    from nbss_b200.optim import FlatClipAdam  # clip_grad_norm_(5) + Adam(1e-3) over the flat gradient buffer, two launches

    opt = FlatClipAdam(net, lr=1e-3, max_norm=5.0) if not args.torch_adam else torch.optim.Adam(params, lr=1e-3, fused=True, capturable=True)

    # rank r takes utterances r::world of the global batch (data_loaders/utils/my_distributed_sampler.py:78)
    x_all, y_all = synth_batch(args.batch, seed=777)
    x_host = x_all[rank::world].contiguous().pin_memory()
    y_host = y_all[rank::world].contiguous().pin_memory()
    x_dev, y_dev = x_host.to(dev), y_host.to(dev)
    loss_host = torch.zeros(1).pin_memory()

    from nbss_b200.loss import neg_si_sdr_pit  # CUDA SI-SDR + PIT (csrc/loss.cu; models/io/loss.py:21-29,95-118)

    def fwd_bwd(x, y):
        opt.zero_grad(set_to_none=True)
        est = pipe(x)
        loss = neg_si_sdr_pit(est, y)[0]
        loss.backward()
        return loss, est

    def reduce_grads():
        if world > 1:
            flat = net._last_flat_grad  # every p.grad is a view of this buffer (checked below): ONE all-reduce
            dist.all_reduce(flat)
            flat.mul_(1.0 / world)

    def opt_step():
        if args.torch_adam:
            torch.nn.utils.clip_grad_norm_(params, 5.0, foreach=True)
        opt.step()

    def step(x, y):  # eager step
        loss, est = fwd_bwd(x, y)
        reduce_grads()
        opt_step()
        return loss, est

    graphs = {}

    def build_graphs():
        """Capture the step as CUDA graphs: A = (H2D copies +) forward + backward (+ D2H loss), B = clip + Adam.  The
        gradient all-reduce runs between them, outside any capture.  Replays cost microseconds of CPU time, which
        matters at 4 utterances per GPU (8-GPU strong scaling), where eager launches would bound the step."""
        x_st, y_st = x_dev.clone(), y_dev.clone()
        gA = torch.cuda.CUDAGraph()
        ops.LAUNCHES = 0
        with torch.cuda.graph(gA):
            lossA, estA = fwd_bwd(x_st, y_st)
        graphs["launches"] = ops.LAUNCHES
        gH = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gH, pool=gA.pool()):
            x_st.copy_(x_host, non_blocking=True)
            y_st.copy_(y_host, non_blocking=True)
            lossH, estH = fwd_bwd(x_st, y_st)
            loss_host.copy_(lossH.detach().reshape(1), non_blocking=True)
        gB = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gB, pool=gA.pool()):
            opt_step()
        graphs.update(A=gA, H=gH, B=gB, lossA=lossA, lossH=lossH, estA=estA, estH=estH)

    def gstep(host_io):
        (graphs["H"] if host_io else graphs["A"]).replay()
        reduce_grads()
        graphs["B"].replay()
        return (graphs["lossH"], graphs["estH"]) if host_io else (graphs["lossA"], graphs["estA"])

    def timed(nsteps, host_io):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(nsteps):
            if use_graphs:
                loss, est = gstep(host_io)
            elif host_io:
                x = x_host.to(dev, non_blocking=True)
                y = y_host.to(dev, non_blocking=True)
                loss, est = step(x, y)
                loss_host.copy_(loss.detach().reshape(1), non_blocking=True)
            else:
                loss, est = step(x_dev, y_dev)
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.barrier()
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()) / nsteps, loss.detach(), est.detach()

    if args.profile:
        step(x_dev, y_dev)
        torch.cuda.synchronize()
        torch.cuda.profiler.start()
        step(x_dev, y_dev)
        torch.cuda.synchronize()
        torch.cuda.profiler.stop()
        return
    log("setup done; warm-up")
    use_graphs = False
    for i in range(max(args.warmup, 3)):
        step(x_dev, y_dev)
        torch.cuda.synchronize()
        log(f"warm-up step {i} done")
    assert net.grads_alias_flat(), "p.grad tensors are not views of the flat gradient buffer"
    if not args.no_graphs:
        try:
            build_graphs()
            use_graphs = True
            for _ in range(2):
                gstep(False)
            torch.cuda.synchronize()
            log("CUDA graphs captured (fwd+bwd, host-I/O variant, optimizer)")
        except Exception as e:  # fall back to eager launches, say so in the JSON line
            log(f"CUDA graph capture failed ({type(e).__name__}: {e}); running eagerly")
            use_graphs = False
            torch.cuda.synchronize()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ops.LAUNCHES = 0
    ms_dev, loss_t, est_t = timed(args.steps, host_io=False)
    loss_v = float(loss_t)
    log(f"device-resident: {ms_dev:.2f} ms/step")
    if args.dump_outputs and rank == 0:
        # the outputs of the last timed step, taken before any later pass moves the parameters on (about 18 MB at batch 32)
        dump = {"estimates": est_t, "loss": loss_t.reshape(1), "grad_flat": net._last_flat_grad,
                "params_flat": torch.cat([p.detach().reshape(-1) for p in params])}
        dump = {k: v.float().cpu().numpy() for k, v in dump.items()}
    launches = graphs["launches"] if use_graphs else ops.LAUNCHES // args.steps
    ms_e2e, _, _ = timed(args.steps, host_io=True)
    log(f"e2e: {ms_e2e:.2f} ms/step")
    clocks = sampler.stop() if rank == 0 else None

    # per-kernel live timing (CUDA events around every C-ABI call on the launching stream) for the roofline
    ops.TIMING = {}
    was_graphs, use_graphs = use_graphs, False  # the per-kernel event timing pass launches eagerly ...
    was_side, net.engine.use_side = net.engine.use_side, False  # ... and on one stream, so that every kernel is timed alone
    timed(max(2, min(args.steps, 5)), host_io=False)
    use_graphs, net.engine.use_side = was_graphs, was_side
    torch.cuda.synchronize()
    per_kernel = {k: (sum(a.elapsed_time(b) for a, b in v) / len(v), len(v)) for k, v in ops.TIMING.items()}
    ops.TIMING = None
    nsteps_prof = max(2, min(args.steps, 5))

    net.check_device_errors()  # sticky device flag: no kernel hit an mbarrier time-out during the whole run
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    frames = args.batch * CFG["T"]
    npts = b_local * CFG["F"] * CFG["T"]
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak_tf = peaks.get("bf16_tflops_sustained", 1400.0)
    peak_bw = peaks.get("hbm_gbs", 6650.0)
    peak_src = "measured (MEASURED_PEAKS.json, sustained)" if peaks else "fallback (B200_PROFILING.md)"
    kernels = {}
    for k, (ms, cnt) in per_kernel.items():
        per_step = ms * cnt / nsteps_prof
        ent = {"ms_per_launch": round(ms, 4), "launches_per_step": cnt // nsteps_prof, "ms_per_step": round(per_step, 3)}
        if k in FLOP_PER_POINT:
            ent["tflops"] = round(FLOP_PER_POINT[k] * npts / (ms * 1e-3) / 1e12, 2)
        kernels[k] = ent
    # DRAM bytes per call from the committed ncu capture of the r02 build (tools/profile.sh + tools/traffic_from_ncu.py;
    # profiles/r02_traffic.json names its commit and command), scaled linearly to this batch (one slab = one unit of traffic)
    traffic, traffic_src = {}, None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))
        traffic = {k: v * b_local / tj["batch_per_gpu"] for k, v in tj["dram_bytes_per_call"].items()}
        traffic_src = (f"profiles/r02_traffic.json (ncu --set full, commit {tj.get('commit')}, batch {tj['batch_per_gpu']}"
                       + ("" if tj["batch_per_gpu"] == b_local else f" scaled to {b_local}") + ")")
    except Exception:
        pass

    def roof(k):
        sec = kernels[k]["ms_per_launch"] * 1e-3
        tf = FLOP_PER_POINT[k] * npts / sec / 1e12
        gb = BYTES_PER_POINT[k] * npts / sec / 1e9
        # roofline side: arithmetic intensity of the ALGORITHMIC work against the machine balance of the measured peaks
        if FLOP_PER_POINT[k] / BYTES_PER_POINT[k] >= peak_tf * 1e12 / (peak_bw * 1e9):
            return {"kernel": k, "bound": "tensor", "achieved": round(tf, 2), "peak": peak_tf, "unit": "TFLOP/s", "frac": round(tf / peak_tf, 4),
                    "traffic": traffic.get(k), "traffic_source": traffic_src, "also_hbm_gbs": round(gb, 1), "peak_source": peak_src}
        return {"kernel": k, "bound": "hbm", "achieved": round(gb, 1), "peak": peak_bw, "unit": "GB/s", "frac": round(gb / peak_bw, 4),
                "traffic": traffic.get(k), "traffic_source": traffic_src, "also_tflops": round(tf, 2), "peak_source": peak_src}
    cands = [k for k in kernels if k in FLOP_PER_POINT and k in BYTES_PER_POINT]
    top = max(cands, key=lambda k: kernels[k]["ms_per_step"])
    rooflines = sorted((dict(roof(k), ms_per_step=kernels[k]["ms_per_step"]) for k in cands), key=lambda r: -r["ms_per_step"])
    roof = dict(roof(top), share_of_step=round(kernels[top]["ms_per_step"] / ms_dev, 3))
    out = {
        "metric": "T-F frames/sec (SpatialNet-small 6ch F=129, training step fwd+bwd incl. STFT/iSTFT)",
        "value": frames / (ms_dev * 1e-3), "unit": "frames/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms_dev, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "fp16 tensor-core operands (fwd + loss-scaled bwd), fp32 accumulate, fp32 stream", "data": "synthetic",
        "config": {"workload": "SpatialNet-small 6ch F=129 T=250 fwd+bwd, batch=32 (BASELINE configs[1])", "global_batch": args.batch,
                   "per_gpu_batch": b_local, "frames_per_utt": CFG["T"], "parallelism": f"dp{world}", "cuda_graphs": bool(use_graphs),
                   "l2": "activations per step (>10 GB) far exceed the 126 MB L2; no explicit flush"},
        "e2e": {"value": frames / (ms_e2e * 1e-3), "unit": "frames/s", "ms_per_step": ms_e2e,
                "h2d_bytes_per_step": int(x_host.numel() * 4 + y_host.numel() * 4) * world, "d2h_bytes_per_step": 4 * world},
        "gpu_launches": launches, "loss": loss_v, "rtf": ms_dev * 1e-3 / (args.batch * TS / 8000.0),
        "roofline": roof, "rooflines": rooflines, "kernels": kernels, "clocks": clocks,
    }
    if eager is not None:
        out["gpu_eager_baseline"] = eager
    if world == 1 and not args.no_nbc2:
        out["extra_workloads"] = {}
        for name, fn in (("nbc2_inference", lambda: bench_nbc2(dev, eager=not args.no_eager_baseline)), ("online_streaming", lambda: bench_online(dev)),
                         ("long_utterance_inference", lambda: bench_long(dev, eager=not args.no_eager_baseline))):
            try:
                out["extra_workloads"][name] = fn()
            except Exception as e:
                out["extra_workloads"][name] = {"unavailable": f"{type(e).__name__}: {e}"[:200]}
    if world == 1 and not args.no_cpu_baseline:
        cores = min(os.cpu_count() or 1, 32)
        log(f"cpu baseline on {cores} threads")
        fps, t, sample = cpu_oracle_subprocess(cores, reps=2)
        out["cpu_baseline"] = {"value": fps, "unit": "frames/s", "cores": cores, "kind": "port", "sample": sample}
    if args.dump_outputs:
        import numpy as np

        os.makedirs(args.dump_outputs, exist_ok=True)
        for k, v in dump.items():
            np.save(os.path.join(args.dump_outputs, k + ".npy"), v)
    _emit(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
