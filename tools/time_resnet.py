"""Device timing of the ResNet variant (riser_b200/resnet.py) on a fixed-length batch.
usage: python tools/time_resnet.py [B] [L] [basic|bottleneck] [x3|f8|w2|f16]
The precision mode applies to the tensor-core launches (ResNetModel(precision=)); default x3.  The GPU's name and
power limit are printed with the result."""
import json
import logging
import subprocess
import sys

import torch

sys.path.insert(0, ".")
from riser_b200 import synth                       # noqa: E402
from riser_b200.config import AttrDict             # noqa: E402
from riser_b200.model import PREC_F16, PREC_F16_F8, PREC_F16_W2, PREC_F16_X3   # noqa: E402
from riser_b200.resnet import ResNetModel          # noqa: E402

MODES = {"f16": PREC_F16, "w2": PREC_F16_W2, "x3": PREC_F16_X3, "f8": PREC_F16_F8}
B = int(sys.argv[1]) if len(sys.argv) > 1 else 512
L = int(sys.argv[2]) if len(sys.argv) > 2 else 12048
name = sys.argv[3] if len(sys.argv) > 3 else "basic"
mode = sys.argv[4] if len(sys.argv) > 4 else "x3"
if mode not in MODES:
    sys.exit(f"unknown precision {mode!r}: one of {', '.join(MODES)}")


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                        str(torch.cuda.current_device())], capture_output=True, text=True)
    return q.stdout.strip() if q.returncode == 0 else torch.cuda.get_device_name() + ", power limit unknown"


cfg = synth.RESNET_CONFIGS[name]
model = ResNetModel(synth.resnet_state_dict(cfg, 0), AttrDict({"model": "resnet", "resnet": cfg}), logging.getLogger("t"),
                    "mRNA", precision=MODES[mode])
x = torch.randn(B, L, device="cuda")
lens = torch.full((B,), L, dtype=torch.int32, device="cuda")
for _ in range(2):
    p = model.classify_batch(x, lens, max_len=L)
torch.cuda.synchronize()
a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
a.record()
for _ in range(3):
    p = model.classify_batch(x, lens, max_len=L)
b.record()
b.synchronize()
ms = a.elapsed_time(b) / 3
print(json.dumps({"net": "resnet-" + name, "precision": mode, "B": B, "L": L, "ms": ms, "reads_per_s": B / ms * 1e3,
                  "fused": model.n_tc_fused, "tc_convs": model.n_tc_convs, "cuda_core_convs": model.n_cuda_core_convs,
                  "gpu": gpu_info(), "p_on_first": p[:3, 1].tolist()}))
