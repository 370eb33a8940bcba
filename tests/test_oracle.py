"""The oracle pinned against the unmodified reference's outputs (tests/golden/*.npz,
made by oracle/make_golden.py).  CPU only."""
import numpy as np
import pytest
import torch

from oracle import cref, torch_port
from tests.helpers import (MODEL_CASES, VQ_CASES, assert_zq_matches, expected_zq, load_golden, make_vq_inputs,
                           model_case_inputs, window)


@pytest.mark.parametrize("name", sorted(VQ_CASES))
def test_c_oracle_vq_matches_reference_bit_exact(name):
    g = load_golden(name)
    z, E = make_vq_inputs(**g["case"])
    r = cref.vq_nchw(z, E)
    assert np.array_equal(r["idx"], g["idx"])                      # int64, bit-exact
    assert r["idx"].dtype == np.int64 and r["idx"].shape == g["idx"].shape
    assert_zq_matches(g, r["zq_nchw"])                             # fp32 bitwise (Q4)
    assert np.array_equal(r["hist"], g["hist"])
    np.testing.assert_allclose(r["loss"], g["loss"], rtol=1e-6, equal_nan=True)
    np.testing.assert_allclose(r["perplexity"], g["perplexity"], rtol=2e-5)


def test_adversarial_known_answers():
    g = load_golden("vq_adversarial")
    z, E = make_vq_inputs(**g["case"])
    idx = cref.vq_nchw(z, E)["idx"].ravel()
    assert idx[0] == 3      # z == E[3] == E[5] == E[20]: lowest duplicate wins
    assert idx[1] == 0      # z == E[36] == E[0]
    assert idx[2] == 17     # exact hit
    assert idx[7] == 0      # NaN row: every distance is NaN, argmin returns column 0
    assert np.array_equal(idx, g["idx"].ravel())


@pytest.mark.parametrize("name", sorted(MODEL_CASES))
def test_c_oracle_model_matches_reference(name):
    g = load_golden(name)
    hp, sd, x = model_case_inputs(g["case"])
    o = cref.vqvae_forward(x, sd, hp["n_res_layers"])
    np.testing.assert_allclose(window(o["z_e"], g["case"]), g["z_e"], atol=2e-7, rtol=0)
    # VQ boundary: same z_e in -> identical indices and bitwise z_q
    b = cref.vq_nchw(g["z_e"], sd["vector_quantization.embedding.weight"])
    assert np.array_equal(b["idx"], g["vq_idx"])
    assert_zq_matches(g, b["zq_nchw"], sd["vector_quantization.embedding.weight"])
    # end to end (oracle convs accumulate in double, the reference in fp32)
    assert np.array_equal(o["idx"], g["idx"])
    np.testing.assert_allclose(window(o["x_hat"], g["case"]), g["x_hat"], atol=2e-7, rtol=0)
    np.testing.assert_allclose(o["loss"], g["loss"], rtol=1e-5)
    np.testing.assert_allclose(o["perplexity"], g["perplexity"], rtol=2e-5)


@pytest.mark.parametrize("name", sorted(MODEL_CASES))
def test_torch_port_matches_reference(name):
    g = load_golden(name)
    hp, sd, x = model_case_inputs(g["case"])
    torch.set_num_threads(1)
    tsd = {k: torch.from_numpy(np.array(v)) for k, v in sd.items()}
    o = torch_port.vqvae_forward(torch.from_numpy(x), tsd, hp["n_res_layers"], intermediates=True)
    assert np.array_equal(o["idx"].numpy(), g["idx"])
    np.testing.assert_allclose(window(o["z_e"].numpy(), g["case"]), g["z_e"], atol=1e-6, rtol=0)
    np.testing.assert_allclose(window(o["x_hat"].numpy(), g["case"]), g["x_hat"], atol=1e-6, rtol=0)
    np.testing.assert_allclose(o["loss"].numpy(), g["loss"], rtol=1e-5)
    np.testing.assert_allclose(o["perplexity"].numpy(), g["perplexity"], rtol=1e-5)
