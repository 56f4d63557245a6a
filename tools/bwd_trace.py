"""One native training step (forward + backward) at the HERMES-CR-120 shape, batch 64, run three times: the workload of
gpu_ll_train.sh (launch list) and, with PROFILE_API=1, of ll_split.py (third step only)."""
import os, sys
import torch
import torch.nn.functional as F
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from bench import ATC, synthetic_macroprops
from crowdmod_ddpm_4d_b200.models.backbones.unet import UNet
dev = torch.device("cuda", 0)
torch.manual_seed(42)
net = UNet(**ATC).to(dev).train()
n, R, Cc = 64, 28, 24
past = synthetic_macroprops(n, 3, R, Cc, 5, 1, dev); fut = synthetic_macroprops(n, 3, R, Cc, 3, 2, dev)
t = torch.randint(0, 1000, (n,), device=dev)
for i in range(3):
    if i == 2:
        print("=== measured pass", file=sys.stderr, flush=True)
        if os.environ.get("PROFILE_API"):      # ncu --profile-from-start off: the third step only (forward + backward)
            torch.cuda.synchronize(); torch.cuda.profiler.start()
    loss = F.mse_loss(net(fut, t, past), torch.randn_like(fut))
    net.zero_grad(set_to_none=True)
    loss.backward()
torch.cuda.synchronize()
if os.environ.get("PROFILE_API"): torch.cuda.profiler.stop()
