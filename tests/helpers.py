"""Shared helpers of the parity tests (test infrastructure; may import oracle/)."""
import json
import os

import numpy as np

from oracle.make_golden import MODEL_CASES, VQ_CASES, make_vq_inputs, window  # noqa: F401
from oracle.weights import make_images, make_state_dict

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
HP_KEYS = ("h_dim", "res_h_dim", "n_res_layers", "n_embeddings", "embedding_dim")


def load_golden(name):
    """A golden case.  Model cases also carry the reference's VQ step on the stored z_e (vq_idx, vq_loss,
    vq_perplexity) and its decoder on the resulting z_q (dec_x_hat): for a full-size fixture these are the forward's
    own idx, loss, perplexity and x_hat; a windowed fixture (cfg3_s256) stores them for its window."""
    with np.load(os.path.join(GOLDEN, name + ".npz")) as d:
        out = {k: d[k] for k in d.files}
    out["case"] = json.loads(str(out["case"]))
    if "z_e" in out:
        for k, full in (("vq_idx", "idx"), ("vq_loss", "loss"), ("vq_perplexity", "perplexity"), ("dec_x_hat", "x_hat")):
            out.setdefault(k, out[full])
    return out


def model_case_inputs(case):
    hp = {k: case[k] for k in HP_KEYS}
    sd = make_state_dict(seed=case["wseed"], codebook=case["codebook"],
                         codebook_scale=case["codebook_scale"], **hp)
    x = make_images(case["batch"], case["size"], case["xseed"])
    return hp, sd, x


def build_model(hp, sd, device="cuda"):
    """The product model (drop-in import path) loaded with a numpy state dict."""
    import torch
    from models.vqvae import VQVAE
    m = VQVAE(hp["h_dim"], hp["res_h_dim"], hp["n_res_layers"], hp["n_embeddings"],
              hp["embedding_dim"], 0.25)
    m.load_state_dict({k: torch.from_numpy(np.array(v)) for k, v in sd.items()})
    return m.to(device).eval()


def expected_zq(g, E=None):
    """The reference's z_q (NCHW) of a golden case, or None when only its hash is stored.  Cases that do not store z_q
    to stay small (cfg3_s256) hold z_e and vq_idx, from which z_q = fl(z_e + fl(E[idx] - z_e)) follows
    (quantizer.py:60,67)."""
    if "z_q" in g:
        return g["z_q"]
    if "z_e" in g and E is not None:
        z = g["z_e"]
        B, D, H, W = z.shape
        rows = np.ascontiguousarray(z.transpose(0, 2, 3, 1)).reshape(-1, D)
        e = np.asarray(E, dtype=np.float32)[g["vq_idx"].ravel()]
        zq = (rows + (e - rows).astype(np.float32)).astype(np.float32)
        return np.ascontiguousarray(zq.reshape(B, H, W, D).transpose(0, 3, 1, 2))
    return None


def assert_zq_matches(g, zq_nchw, E=None):
    """Bitwise comparison of a z_q (NCHW fp32 array) with the golden case, through the stored array, the
    reconstruction above, or the stored SHA-256 of the reference's bytes."""
    import hashlib
    zq_nchw = np.ascontiguousarray(zq_nchw, dtype=np.float32)
    want = expected_zq(g, E)
    if want is not None:
        assert np.array_equal(zq_nchw, want, equal_nan=True)
    else:
        assert hashlib.sha256(zq_nchw.tobytes()).hexdigest() == str(g["z_q_sha256"])
