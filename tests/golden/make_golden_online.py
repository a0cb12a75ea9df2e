"""Generates tests/golden/online_f9_t270.npz from the UNMODIFIED reference:
    python tests/golden/make_golden_online.py <path to a checkout of the reference>
OnlineSpatialNet(attention='mhsa(251)') — causal encoder / T-convs, attention over the last 251 frames, GroupNorm over
(24 channels x F) per frame (models/arch/OnlineSpatialNet.py).  The reference imports mamba_ssm at module level and calls
isinstance(..., Mamba), so a stub module is injected (the mhsa variant never touches it).  T = 270 > 251 exercises the window.
The weights are oracle.spatialnet_oracle.synth_params(seed 107) and the input is seeded: the tests regenerate both rather than
load them (the fixture keeps the input's float64 sum), and the fixture keeps the shape of every state-dict entry of the reference."""
import os
import sys
import types

import numpy as np
import torch

m = types.ModuleType("mamba_ssm")


class Mamba(torch.nn.Module):
    def __init__(self, *a, **k):
        super().__init__()


m.Mamba = Mamba
u, g = types.ModuleType("mamba_ssm.utils"), types.ModuleType("mamba_ssm.utils.generation")
g.InferenceParams = type("InferenceParams", (), {"__init__": lambda self, *a, **k: None})
sys.modules.update({"mamba_ssm": m, "mamba_ssm.utils": u, "mamba_ssm.utils.generation": g})
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
sys.path.insert(0, os.path.abspath(sys.argv[1]))
from models.arch.OnlineSpatialNet import OnlineSpatialNet  # noqa: E402

from oracle import spatialnet_oracle as O  # noqa: E402

torch.manual_seed(7)
F, T = 9, 270
net = OnlineSpatialNet(dim_input=12, dim_output=4, num_layers=2, dim_hidden=96, dim_ffn=192, num_heads=4, kernel_size=(5, 3),
                       conv_groups=(8, 8), norms=["LN", "LN", "GN", "LN", "LN", "LN"], dim_squeeze=8, num_freqs=F, full_share=0,
                       attention="mhsa(251)", rope=False).eval()
sd = net.state_dict()
P = O.synth_params(dict(O.SMALL_CFG, num_layers=2, num_freqs=F), seed=107)
net.load_state_dict({k: v.clone() for k, v in P.items()}, strict=True)
x = torch.randn(2, F, T, 12, generator=torch.Generator().manual_seed(270))
with torch.no_grad():
    y = net(x)
out = {"x_sum": np.float64(x.double().sum().item()), "y": y.numpy()}
for k, v in sd.items():
    out["shape." + k] = np.array(v.shape, dtype=np.int64)
np.savez_compressed(os.path.join(os.path.dirname(os.path.abspath(__file__)), "online_f9_t270.npz"), **out)
print("saved", y.shape, float(y.abs().mean()))
