"""Generate tests/golden/*.npz from the UNMODIFIED reference (authoring container only).

TEST INFRASTRUCTURE ONLY.  Run as ``python -m oracle.make_golden`` from the repo root
in a container that has /root/reference.  The reference is imported in a subprocess
with cwd=/root/reference (its modules use absolute ``from models.x import``, which
collides with this repo's drop-in ``models`` package) and CUDA hidden (SURVEY Q5).

Weights and inputs are NOT stored: they are regenerated from (hyper-params, seed) by
oracle/weights.py, so each fixture only holds the reference's outputs.
"""
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

from .weights import make_images, make_state_dict

REF = "/root/reference"
OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")

# name -> (model hyper-params, codebook kind/scale, batch, image size)
MODEL_CASES = {
    # BASELINE cfg1/cfg2 architecture, default codebook init = near-tie stress (SURVEY Q10)
    "cifar_default": dict(h_dim=128, res_h_dim=32, n_res_layers=2, n_embeddings=512,
                          embedding_dim=64, codebook="default", codebook_scale=1.0,
                          batch=4, size=32, wseed=0, xseed=1),
    # same architecture, trained-like codebook spread over the z_e range
    "cifar_spread": dict(h_dim=128, res_h_dim=32, n_res_layers=2, n_embeddings=512,
                         embedding_dim=64, codebook="normal", codebook_scale=0.05,
                         batch=4, size=32, wseed=2, xseed=3),
    # odd sizes: K not a multiple of any tile, 3 shared residual applications, S=20
    "small_odd": dict(h_dim=32, res_h_dim=8, n_res_layers=3, n_embeddings=50,
                      embedding_dim=16, codebook="normal", codebook_scale=0.08,
                      batch=3, size=20, wseed=4, xseed=5),
    # empty residual stack (ModuleList of 0 layers -> just F.relu)
    "no_res": dict(h_dim=64, res_h_dim=16, n_res_layers=0, n_embeddings=128,
                   embedding_dim=32, codebook="normal", codebook_scale=0.07,
                   batch=2, size=16, wseed=6, xseed=7),
    # cfg3 architecture (K=1024) on a 64x64 image
    "k1024_s64": dict(h_dim=128, res_h_dim=32, n_res_layers=2, n_embeddings=1024,
                      embedding_dim=64, codebook="normal", codebook_scale=0.05,
                      batch=2, size=64, wseed=8, xseed=9),
    # BASELINE configs[2] (cfg3) at its real image size: 256x256, K=1024 (B=2 instead of 128).  Its full z_e and x_hat
    # take 3.5 MB, so the fixture keeps idx, hist, loss and perplexity of the whole forward and z_e / x_hat of one
    # window (see window()), plus the reference's VQ step and decoder run on that window of z_e.
    "cfg3_s256": dict(h_dim=128, res_h_dim=32, n_res_layers=2, n_embeddings=1024,
                      embedding_dim=64, codebook="normal", codebook_scale=0.05,
                      batch=2, size=256, wseed=18, xseed=19, window=[1, 40, 0, 16]),
}


def window(a, case):
    """The part of a full-size NCHW output of a model case that its fixture stores.  All of it, unless the case has a
    ``window`` [image, y0, x0, n]: then image ``image``, latent rows and columns [y0, y0 + n) (x0 likewise), scaled to
    the resolution of ``a`` (z_e is at 1/4 of the image size, x_hat at the full size)."""
    if "window" not in case:
        return a
    i, y0, x0, n = case["window"]
    s = a.shape[2] // (case["size"] // 4)
    return a[i:i + 1, :, s * y0:s * (y0 + n), s * x0:s * (x0 + n)]


# VectorQuantizer-only cases (BASELINE cfg4 grid at a size the CPU finishes in seconds)
VQ_CASES = {
    "vq_k512_d64": dict(K=512, D=64, B=4, H=16, W=16, seed=11, kind="normal"),
    "vq_k1024_d64": dict(K=1024, D=64, B=4, H=16, W=16, seed=12, kind="normal"),
    "vq_k8192_d64": dict(K=8192, D=64, B=2, H=16, W=16, seed=13, kind="normal"),
    "vq_k512_d256": dict(K=512, D=256, B=2, H=16, W=16, seed=14, kind="normal"),
    "vq_k8192_d256": dict(K=8192, D=256, B=1, H=16, W=16, seed=15, kind="normal"),
    "vq_default_init": dict(K=512, D=64, B=4, H=16, W=16, seed=16, kind="default"),
    # adversarial: duplicated codebook rows (lowest index must win), z equal to a code,
    # one NaN row (argmin returns the NaN column), K=37 / N=3*5*7 ragged sizes
    "vq_adversarial": dict(K=37, D=8, B=3, H=5, W=7, seed=17, kind="adversarial"),
    # 65 536 rows at the default codebook init (near-tie stress, SURVEY Q10): pins the canonical summation order
    # against MKL at a size where its blocking could differ.  z_q (16 MB) is stored as a SHA-256 of its bytes.
    "vq_default_init_64k": dict(K=512, D=64, B=16, H=64, W=64, seed=20, kind="default", hash_zq=True),
    "vq_k1024_d64_64k": dict(K=1024, D=64, B=16, H=64, W=64, seed=21, kind="normal", hash_zq=True),
}

_REF_SCRIPT = r"""
import sys, json, numpy as np, torch
sys.path.insert(0, %(ref)r)
import models.quantizer as Q
Q.device = torch.device("cpu")
from models.vqvae import VQVAE
from models.quantizer import VectorQuantizer
torch.set_num_threads(1)   # fixed thread count -> reproducible MKL blocking
job = json.load(open(sys.argv[1]))
data = np.load(job["in"])
out = {}
with torch.no_grad():
    if job["kind"] == "model":
        hp = job["hp"]
        m = VQVAE(hp["h_dim"], hp["res_h_dim"], hp["n_res_layers"], hp["n_embeddings"],
                  hp["embedding_dim"], 0.25).eval()
        sd = {k: torch.from_numpy(data[k]) for k in m.state_dict().keys()}
        m.load_state_dict(sd)
        x = torch.from_numpy(data["__x"])
        z_e = m.pre_quantization_conv(m.encoder(x.clone()))
        loss, z_q, perp, onehot, idx = m.vector_quantization(z_e)
        x_hat = m.decoder(z_q.clone())
        l2, xh2, p2 = m(x.clone())
        assert torch.equal(xh2, x_hat) and torch.equal(l2, loss) and torch.equal(p2, perp)
        out = dict(z_e=z_e.numpy(), idx=idx.numpy(), z_q=z_q.numpy(), x_hat=x_hat.numpy(),
                   loss=loss.numpy(), perplexity=perp.numpy(),
                   hist=onehot.sum(0).numpy().astype(np.int32))
    elif job["kind"] == "window":
        # the VQ step and the decoder on a window of z_e (the VQ boundary and decoder checks of a windowed case)
        hp = job["hp"]
        m = VQVAE(hp["h_dim"], hp["res_h_dim"], hp["n_res_layers"], hp["n_embeddings"],
                  hp["embedding_dim"], 0.25).eval()
        m.load_state_dict({k: torch.from_numpy(data[k]) for k in m.state_dict().keys()})
        loss, z_q, perp, _, idx = m.vector_quantization(torch.from_numpy(data["__z"]))
        out = dict(vq_idx=idx.numpy(), vq_loss=loss.numpy(), vq_perplexity=perp.numpy(),
                   dec_x_hat=m.decoder(z_q.clone()).numpy())
    else:
        vq = VectorQuantizer(int(job["K"]), int(job["D"]), 0.25)
        vq.embedding.weight.data.copy_(torch.from_numpy(data["E"]))
        z = torch.from_numpy(data["z"])
        loss, z_q, perp, onehot, idx = vq(z)
        out = dict(idx=idx.numpy(), z_q=z_q.numpy(), loss=loss.numpy(),
                   perplexity=perp.numpy(), hist=onehot.sum(0).numpy().astype(np.int32),
                   onehot_shape=np.array(onehot.shape))
np.savez(job["out"], **out)
"""


_CKPT_SCRIPT = r"""
# writes a checkpoint exactly as utils.save_model_and_results does (utils.py:106-115) from the unmodified reference model
import sys, json, numpy as np, torch
sys.path.insert(0, %(ref)r)
import models.quantizer as Q
Q.device = torch.device("cpu")
from models.vqvae import VQVAE
job = json.load(open(sys.argv[1]))
data = np.load(job["in"])
hp = job["hp"]
m = VQVAE(hp["h_dim"], hp["res_h_dim"], hp["n_res_layers"], hp["n_embeddings"], hp["embedding_dim"], 0.25)
m.load_state_dict({k: torch.from_numpy(data[k]) for k in m.state_dict().keys()})
results = {"n_updates": 3, "recon_errors": [np.float32(0.5), np.float32(0.4)], "loss_vals": [np.float32(0.9), np.float32(0.8)],
           "perplexities": [np.float32(3.0), np.float32(4.0)]}                     # main.py:59-64, 81-84
hyper = {"batch_size": 32, "n_updates": 5000, "n_hiddens": hp["h_dim"], "n_residual_hiddens": hp["res_h_dim"],
         "n_residual_layers": hp["n_res_layers"], "embedding_dim": hp["embedding_dim"], "n_embeddings": hp["n_embeddings"],
         "beta": 0.25, "learning_rate": 3e-4, "log_interval": 50, "dataset": "CIFAR10", "save": True, "filename": "golden"}   # vars(args), main.py:9-32
torch.save({"model": m.state_dict(), "results": results, "hyperparameters": hyper}, job["ckpt"])
"""


def make_checkpoint(name="small_odd"):
    """tests/golden/ckpt_<name>.pth: the reference's own checkpoint format holding the weights of golden case <name>."""
    c = MODEL_CASES[name]
    hp = {k: c[k] for k in ("h_dim", "res_h_dim", "n_res_layers", "n_embeddings", "embedding_dim")}
    sd = make_state_dict(seed=c["wseed"], codebook=c["codebook"], codebook_scale=c["codebook_scale"], **hp)
    with tempfile.TemporaryDirectory() as td:
        job = {"in": os.path.join(td, "in.npz"), "hp": hp, "ckpt": os.path.join(OUT, f"ckpt_{name}.pth")}
        np.savez(job["in"], **sd)
        with open(os.path.join(td, "job.json"), "w") as f:
            json.dump(job, f)
        subprocess.run([sys.executable, "-c", _CKPT_SCRIPT % dict(ref=REF), os.path.join(td, "job.json")], check=True, cwd=REF,
                       env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    return job["ckpt"]


def make_vq_inputs(K, D, B, H, W, seed, kind, hash_zq=False):
    """(z NCHW, codebook) for a VectorQuantizer-only case; shared with the tests."""
    rng = np.random.RandomState(seed)
    z = rng.standard_normal((B, D, H, W)).astype(np.float32)
    if kind == "default":
        E = rng.uniform(-1.0 / K, 1.0 / K, size=(K, D)).astype(np.float32)
        z *= np.float32(0.06)
    elif kind == "normal":
        E = rng.standard_normal((K, D)).astype(np.float32)
    else:  # adversarial
        E = rng.standard_normal((K, D)).astype(np.float32)
        E[5] = E[3]; E[20] = E[3]; E[36] = E[0]          # duplicates: lowest index wins
        rows = z.transpose(0, 2, 3, 1).reshape(-1, D)     # a copy
        rows[0] = E[3]; rows[1] = E[36]; rows[2] = E[17]  # exact hits
        rows[7, 2] = np.nan                               # NaN row
        rows[9] = 0.0
        z = np.ascontiguousarray(rows.reshape(B, H, W, D).transpose(0, 3, 1, 2))
    return z, E


def _run_ref(job, arrays):
    with tempfile.TemporaryDirectory() as td:
        job = dict(job, **{"in": os.path.join(td, "in.npz"), "out": os.path.join(td, "out.npz")})
        np.savez(job["in"], **arrays)
        with open(os.path.join(td, "job.json"), "w") as f:
            json.dump(job, f)
        env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
        subprocess.run([sys.executable, "-c", _REF_SCRIPT % dict(ref=REF),
                        os.path.join(td, "job.json")], check=True, cwd=REF, env=env)
        with np.load(job["out"]) as d:
            return {k: d[k] for k in d.files}


def main():
    assert os.path.isdir(REF), "needs the reference checkout (authoring container only)"
    os.makedirs(OUT, exist_ok=True)
    only = set(sys.argv[1:])          # optional: regenerate just the named cases
    if not only or "ckpt" in only:
        print("checkpoint", make_checkpoint("small_odd"))
    for name, c in MODEL_CASES.items():
        if only and name not in only:
            continue
        hp = {k: c[k] for k in ("h_dim", "res_h_dim", "n_res_layers", "n_embeddings", "embedding_dim")}
        sd = make_state_dict(seed=c["wseed"], codebook=c["codebook"],
                             codebook_scale=c["codebook_scale"], **hp)
        x = make_images(c["batch"], c["size"], c["xseed"])
        out = _run_ref(dict(kind="model", hp=hp), dict(sd, __x=x))
        if "window" in c:
            z = np.ascontiguousarray(window(out["z_e"], c))
            out = dict(_run_ref(dict(kind="window", hp=hp), dict(sd, __z=z)), z_e=z, idx=out["idx"],
                       x_hat=np.ascontiguousarray(window(out["x_hat"], c)), loss=out["loss"],
                       perplexity=out["perplexity"], hist=out["hist"])
        np.savez_compressed(os.path.join(OUT, name + ".npz"), case=json.dumps(c), **out)
        print(name, {k: v.shape for k, v in out.items()}, "codes used", int((out["hist"] > 0).sum()))
    for name, c in VQ_CASES.items():
        if only and name not in only:
            continue
        z, E = make_vq_inputs(**c)
        out = _run_ref(dict(kind="vq", K=c["K"], D=c["D"]), dict(z=z, E=E))
        out.pop("onehot_shape")
        if c.get("hash_zq"):
            import hashlib
            zq = np.ascontiguousarray(out.pop("z_q"))
            out["z_q_sha256"] = np.array(hashlib.sha256(zq.tobytes()).hexdigest())
            out["idx"] = out["idx"].astype(np.int32)
        np.savez_compressed(os.path.join(OUT, name + ".npz"), case=json.dumps(c), **out)
        print(name, "codes used", int((out["hist"] > 0).sum()))


if __name__ == "__main__":
    main()
