"""VQ kernel (vq2.cu) alone at streaming sizes: N = 2^20 rows, K in {512, 1024, 8192}."""
import sys
import numpy as np
import torch
sys.path.insert(0, ".")
from vqvae_b200 import ops

dev = torch.device("cuda")
rng = np.random.RandomState(0)
N = 1 << 20
z = torch.from_numpy(rng.standard_normal((N, 64)).astype(np.float32)).to(dev)
for K in (512, 1024, 8192):
    E = torch.from_numpy(rng.standard_normal((K, 64)).astype(np.float32)).to(dev)
    ops.set_vq_kernel("tc")
    for _ in range(2):
        ops.vq_forward(z, E)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(5):
        ops.vq_forward(z, E)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 5
    print(f"K={K:5d} {ms * 1e3:9.1f} us  {N * 520 / ms / 1e6:8.1f} GB/s  {2.0 * N * K * 64 / ms / 1e9:7.1f} TFLOP/s", flush=True)
ops.set_vq_kernel("auto")
