"""Diagnostic (not a test): which batches of the eager HostPipeline differ from the direct forward."""
import os, sys
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))
import vqvae_b200
from oracle import weights

prec = sys.argv[1] if len(sys.argv) > 1 else "tf32"
use_graph = (sys.argv[2] == "graph") if len(sys.argv) > 2 else False
depth = int(sys.argv[3]) if len(sys.argv) > 3 else 3
sd = weights.make_state_dict(128, 32, 2, 512, 64, seed=5)
m = vqvae_b200.VQVAE(128, 32, 2, 512, 64, 0.25)
m.load_state_dict({k: torch.from_numpy(np.array(v)) for k, v in sd.items()})
vqvae_b200.set_precision(prec)
m = m.cuda().eval()
rng = np.random.default_rng(11)
batches = [torch.from_numpy(rng.standard_normal((16, 3, 32, 32)).astype(np.float32)).pin_memory() for _ in range(9)]
want = []
with torch.no_grad():
    for x in batches:
        loss, x_hat, perp = m(x.cuda())
        want.append((float(loss), x_hat.cpu().clone(), float(perp)))
pipe = vqvae_b200.HostPipeline(m, (16, 3, 32, 32), depth=depth, use_graph=use_graph)
got = []
pipe.run(batches, lambda r: got.append((r.index, float(r.loss), r.x_hat.clone(), float(r.perplexity))))
for i, (w, g) in enumerate(zip(want, got)):
    same = w[0] == g[1] and torch.equal(w[1], g[2]) and w[2] == g[3]
    alias = [j for j, ww in enumerate(want) if ww[0] == g[1]]
    xalias = [j for j, ww in enumerate(want) if torch.equal(ww[1], g[2])]
    print(f"{prec} graph={use_graph} depth={depth} batch {i}: same={same} loss_of={alias} xhat_of={xalias} "
          f"loss {w[0]:.9f} vs {g[1]:.9f}")
