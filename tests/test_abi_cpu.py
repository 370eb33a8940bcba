"""CPU-only checks of the C-ABI boundary and of the drop-in nn.Module API (no compute:
there is no GPU here and the product has no CPU fallback)."""
import ctypes
import inspect
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_functions():
    src = open(os.path.join(ROOT, "include", "vqvae_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(vqb_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol_at_abi_version_3():
    from vqvae_b200.build import build
    lib = ctypes.CDLL(build())
    names = _header_functions()
    assert len(names) >= 15
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/vqvae_b200.h but not exported"
    lib.vqb_abi_version.restype = ctypes.c_int
    assert lib.vqb_abi_version() == 3
    assert lib.vqb_diag_build() == 0          # the shipped library never reads the environment
    lib.vqb_error_string.restype = ctypes.c_char_p
    assert b"workspace" in lib.vqb_error_string(-3)


def test_ctypes_signature_table_matches_header():
    from vqvae_b200 import _lib
    assert sorted(_lib.SIGNATURES) == _header_functions()


def test_argument_validation_without_a_gpu():
    """Bad arguments are rejected before any CUDA call (safe on a CPU box)."""
    from vqvae_b200 import _lib
    lib = _lib.lib()
    assert lib.vqb_conv2d_f32(None, None, None, None, None, 1, 3, 8, 8, 4, 3, 3, 1, 1, 0, 0, 0, 0, 0, None) == -1
    assert lib.vqb_vq_forward_f32(None, None, 1, 1, 4, None, None, None, None, None, 0, None) == -1
    assert lib.vqb_set_vq_kernel(7) == -1
    assert lib.vqb_vq_workspace_bytes(1024, 512, 64) > 0
    assert lib.vqb_vq_forward_deferred_f32(None, None, 1, 1, 4, None, None, None, None, None, 0, None) == -1
    assert lib.vqb_vq_reduce_sse_f32(None, 1, 1, 4, None, None) == -1
    assert lib.vqb_residual_layer_f32(None, None, None, None, None, 1, 8, 8, 32, 32, 1, 1, None) == -1
    assert lib.vqb_residual_stack_f32(None, None, None, None, None, None, 1, 8, 8, 32, 32, 2, 1, None) == -1
    import ctypes
    buf = (ctypes.c_float * 4)()
    p = ctypes.cast(buf, ctypes.c_void_p)
    assert lib.vqb_residual_stack_f32(p, p, p, p, p, p, 1, 8, 8, 32, 32, 0, 1, None) == -1      # n_layers < 1
    assert lib.vqb_residual_stack_f32(p, p, p, p, None, p, 1, 8, 8, 32, 32, 2, 1, None) == -1   # scratch needed for n > 1
    assert lib.vqb_memcpy_async(None, p, 16, 1, None) == -1
    assert lib.vqb_memcpy_async(p, p, 16, 9, None) == -1                                        # unknown kind
    assert lib.vqb_memcpy_async(p, p, 0, 1, None) == 0                                          # empty copy is a no-op


def test_reference_constructor_signatures_and_import_paths():
    from models.vqvae import VQVAE
    from models.encoder import Encoder
    from models.decoder import Decoder
    from models.quantizer import VectorQuantizer
    from models.residual import ResidualLayer, ResidualStack
    sig = lambda c: list(inspect.signature(c.__init__).parameters)[1:]   # noqa: E731
    assert sig(VQVAE) == ["h_dim", "res_h_dim", "n_res_layers", "n_embeddings", "embedding_dim", "beta",
                          "save_img_embedding_map"]                       # vqvae.py:11-12
    assert sig(Encoder) == ["in_dim", "h_dim", "n_res_layers", "res_h_dim"]   # encoder.py:24
    assert sig(Decoder) == ["in_dim", "h_dim", "n_res_layers", "res_h_dim"]   # decoder.py:22
    assert sig(VectorQuantizer) == ["n_e", "e_dim", "beta"]                   # quantizer.py:20
    assert sig(ResidualLayer) == ["in_dim", "h_dim", "res_h_dim"]             # residual.py:16
    assert sig(ResidualStack) == ["in_dim", "h_dim", "res_h_dim", "n_res_layers"]   # residual.py:41
    assert list(inspect.signature(VQVAE.forward).parameters) == ["self", "x", "verbose"]


def test_state_dict_keys_shapes_and_shared_residual_weights():
    from models.vqvae import VQVAE
    from oracle.weights import state_dict_shapes
    m = VQVAE(128, 32, 2, 512, 64, 0.25)
    sd = m.state_dict()
    want = state_dict_shapes(128, 32, 2, 512, 64)
    assert list(sd.keys()) == [k for k, _, _ in want]            # 23 keys, reference order (SURVEY 8b)
    for k, shape, _ in want:
        assert tuple(sd[k].shape) == tuple(shape), k
    assert sum(v.numel() for v in sd.values()) == 694851          # duplicated stack.1.* keys included
    assert sum(p.numel() for p in m.parameters()) == 612931       # unique parameters (Q1)
    st = m.encoder.conv_stack[5].stack
    assert st[0] is st[1]
    assert sd["encoder.conv_stack.5.stack.0.res_block.1.weight"].data_ptr() == \
        sd["encoder.conv_stack.5.stack.1.res_block.1.weight"].data_ptr()
    # load_state_dict accepts the duplicated keys; attributes callers touch exist
    m.load_state_dict({k: v.clone() for k, v in sd.items()})
    assert m.img_to_embedding_map is None and m.vector_quantization.n_e == 512
    assert VQVAE(32, 8, 1, 16, 8, 0.25, save_img_embedding_map=True).img_to_embedding_map == {i: [] for i in range(16)}
    w = m.vector_quantization.embedding.weight
    assert float(w.abs().max()) <= 1.0 / 512 + 1e-9               # quantizer.py:27 init


def test_same_seed_gives_reference_init_order():
    """Parameter creation order equals the reference's, so the same torch seed gives the same
    weights; pinned by a fingerprint taken from the unmodified reference (tests/golden)."""
    import json
    from models.vqvae import VQVAE
    fp = json.load(open(os.path.join(ROOT, "tests", "golden", "init_fingerprint.json")))
    torch.manual_seed(fp["seed"])
    m = VQVAE(*fp["args"])
    for k, v in m.state_dict().items():
        assert abs(float(v.double().sum()) - fp["sums"][k]) <= 1e-9 + 1e-12 * abs(fp["sums"][k]), k


def test_default_precision_is_the_reference_gpu_arithmetic():
    from vqvae_b200 import modules
    assert modules.DEFAULT_PRECISION == "tf32"
    import vqvae_b200
    for name in ("fp32", "tf32", "bf16"):
        with vqvae_b200.precision(name):
            assert vqvae_b200.get_precision() == name
    with pytest.raises(ValueError):
        vqvae_b200.set_precision("fp8")


def test_entry_points_and_vq_kernel_choice_validate_arguments_without_a_gpu():
    """bf16 pipeline entry points and the VQ kernel choice: bad arguments / unsupported shapes are rejected before any
    CUDA call."""
    from vqvae_b200 import _lib
    lib = _lib.lib()
    buf = (ctypes.c_float * 64)()
    p = ctypes.cast(buf, ctypes.c_void_p)
    assert lib.vqb_conv2d_bf16(None, None, None, None, 1, 64, 8, 8, 64, _lib.CONV_K3, 0, 0, None) == -1
    assert lib.vqb_conv2d_bf16(p, p, None, p, 1, 48, 8, 8, 64, _lib.CONV_K3, 0, 0, None) == -2          # Cin % 64
    assert lib.vqb_conv2d_bf16(p, p, None, p, 1, 64, 7, 8, 64, _lib.CONV_K4S2, 0, 0, None) == -2        # odd height
    assert lib.vqb_conv_bf16_packed_bytes(_lib.CONV_K3, 128, 128) == 9 * 2 * 128 * (128 + 16) + 256
    assert lib.vqb_conv_bf16_packed_bytes(_lib.CONV_K3, 128, 100) == 0                                  # not covered
    assert lib.vqb_conv_bf16_packed_bytes(_lib.CONVT_K4S2, 64, 128) > 0
    assert lib.vqb_pack_conv_weight_bf16(None, None, _lib.CONV_K3, 128, 128, None) == -1
    assert lib.vqb_residual_layer_bf16(None, None, None, None, 1, 8, 8, 128, 32, 1, None) == -1
    assert lib.vqb_residual_layer_bf16(p, p, p, p, 1, 8, 8, 256, 32, 1, None) in (-1, -2)               # C = 256 / r == out
    assert lib.vqb_conv_in_bf16(None, None, None, None, 1, 32, 32, 64, 1, None) == -1
    assert lib.vqb_vq_forward_bf16zq_f32(None, None, 1, 1, 64, None, None, None, None, None, 0, None) == -1
    # the fp32-activation entry points refuse the bf16 enum instead of silently running TF32 (round-1 verdict)
    assert lib.vqb_conv2d_f32(p, p, None, None, p, 1, 64, 8, 8, 64, 3, 3, 1, 1, 0, 1, 1, 0, _lib.BF16, None) == -2
    assert lib.vqb_residual_layer_f32(p, p, p, p, p, 1, 8, 8, 32, 32, 1, _lib.BF16, None) == -2
    assert lib.vqb_set_vq_kernel(3) == -1 and lib.vqb_set_vq_kernel(0) == 0


def test_no_cpu_fallback():
    from models.vqvae import VQVAE
    m = VQVAE(32, 8, 1, 16, 8, 0.25)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m(torch.zeros(1, 3, 8, 8))
    with pytest.raises(RuntimeError):
        m.encoder(torch.zeros(1, 3, 8, 8))


def test_product_never_imports_the_oracle():
    for d in ("vqvae_b200", "models"):
        for root, _, files in os.walk(os.path.join(ROOT, d)):
            for f in files:
                if f.endswith(".py"):
                    src = open(os.path.join(root, f)).read()
                    assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), os.path.join(root, f)


def test_reference_checkpoint_loads_on_cpu(tmp_path):
    """vqvae_b200.load_checkpoint reads the reference's {'model','results','hyperparameters'} file (utils.py:106-115; written by
    oracle/make_golden.py from the unmodified reference model): architecture from the hyper-parameters, all 23 keys loaded."""
    import numpy as np
    import vqvae_b200
    from tests.helpers import load_golden, model_case_inputs
    path = os.path.join(ROOT, "tests", "golden", "ckpt_small_odd.pth")
    m, data = vqvae_b200.load_checkpoint(path, device="cpu")
    hp, sd, _ = model_case_inputs(load_golden("small_odd")["case"])
    assert data["hyperparameters"]["n_hiddens"] == hp["h_dim"] and len(data["results"]["recon_errors"]) == 2
    got = m.state_dict()
    assert list(got.keys()) == list(sd.keys())
    for k, v in sd.items():
        assert np.array_equal(got[k].numpy(), v), k
    assert len(m.encoder.conv_stack[5].stack) == hp["n_res_layers"] and not m.training
    # save_checkpoint writes the same format back
    out = str(tmp_path / "roundtrip.pth")
    vqvae_b200.save_checkpoint(m, data["results"], data["hyperparameters"], out)
    m2, d2 = vqvae_b200.load_checkpoint(out, device="cpu")
    assert all(torch.equal(a, b) for a, b in zip(m.state_dict().values(), m2.state_dict().values()))
    assert d2["hyperparameters"] == data["hyperparameters"]


def test_convt_out_scatter_column_layout():
    """convt_out_bf16.cu orders the 64 GEMM columns of the output layer by DESTINATION pixel.  Host logic, pinned here:
    every (ky, kx, co) of the 4x4x3 ConvTranspose2d weight appears exactly once, the 16 pad columns are marked, and the
    group a column sits in is the one the epilogue reads it from: a tap (ky, kx) of input pixel (y, x) lands on output pixel
    (2y - 1 + ky, 2x - 1 + kx) (decoder.py:34, k4 s2 p1), i.e. in the 2x2 block of input pixel (y + dy, x + dx) with
    dy = -1 for ky = 0, +1 for ky = 3, else 0 (same for dx), at block row r = (2y - 1 + ky) - 2(y + dy)."""
    import ctypes
    from vqvae_b200 import _lib
    fn = _lib.lib().vqb_debug_convt_out_scatter_column
    fn.argtypes = [ctypes.c_int] + [ctypes.POINTER(ctypes.c_int)] * 3
    seen = {}
    pads = 0
    for n in range(64):
        co, ky, kx = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
        assert fn(n, ctypes.byref(co), ctypes.byref(ky), ctypes.byref(kx)) == 0
        if co.value < 0:
            pads += 1
            continue
        key = (ky.value, kx.value, co.value)
        assert key not in seen
        seen[key] = n
        dy = -1 if ky.value == 0 else (1 if ky.value == 3 else 0)
        dx = -1 if kx.value == 0 else (1 if kx.value == 3 else 0)
        r, s_ = (ky.value - 1) - 2 * dy, (kx.value - 1) - 2 * dx          # position inside the destination's 2x2 block
        assert r in (0, 1) and s_ in (0, 1)
        # the column groups the epilogue addresses: own [0,12), up [12,20), down [20,28), left [28,36), right [36,44), corners
        if (dy, dx) == (0, 0):
            assert n == (r * 2 + s_) * 3 + co.value
        elif dx == 0:
            assert n == (12 if dy == -1 else 20) + s_ * 3 + co.value and r == (1 if dy == -1 else 0)
        elif dy == 0:
            assert n == (28 if dx == -1 else 36) + r * 3 + co.value and s_ == (1 if dx == -1 else 0)
        else:
            base = {(-1, -1): 44, (-1, 1): 48, (1, -1): 52, (1, 1): 56}[(dy, dx)]
            assert n == base + co.value and (r, s_) == ((1 if dy == -1 else 0), (1 if dx == -1 else 0))
    assert len(seen) == 48 and pads == 16
    assert fn(64, ctypes.byref(ctypes.c_int()), ctypes.byref(ctypes.c_int()), ctypes.byref(ctypes.c_int())) != 0


def test_bf16_conv_plans_row_counts():
    """hconv.cu's host-built GEMM step plans (no GPU needed): one packed 128-byte weight row per (output column, tap,
    64-channel chunk).  Every useful row count follows from the layer: conv Cout x taps x chunks; the stride-2 conv on its
    space-to-depth view 4 chunks x 4 taps; the stride-2 transposed conv 2 passes x chunks x 2 row taps x (2 Cout + Cout +
    Cout) columns; the output layer 9 x 16 gather-form rows + the 64 scatter-form columns."""
    from vqvae_b200 import _lib
    L = _lib.lib()
    expect = [
        (_lib.CONV_K1, 64, 128, 2 * 64),                     # vqvae.py:16
        (_lib.CONV_K3, 128, 128, 9 * 2 * 128),               # encoder.py:35
        (_lib.CONV_K3, 32, 128, 9 * 2 * 32),                 # residual.py:20 (W1)
        (_lib.CONVT_K3, 128, 64, 9 * 128),                   # decoder.py:28
        (_lib.CONV_K4S2, 128, 64, 4 * 4 * 128),              # encoder.py:32
        (_lib.CONVT_K4S2, 64, 128, 2 * 2 * 2 * 4 * 64),      # decoder.py:31
        (_lib.CONVT_K4S2_OUT, 3, 64, 9 * 16 + 64),           # decoder.py:34
        (_lib.RES_W2, 128, 32, 128),                         # residual.py:23 (W2, Cmid padded to one 64-channel chunk)
    ]
    for kind, cout, cin, rows in expect:
        assert L.vqb_conv_bf16_packed_bytes(kind, cout, cin) == rows * (128 + 16) + 256, (kind, cout, cin)
    assert L.vqb_conv_bf16_packed_bytes(_lib.CONV_K3, 128, 100) == 0          # Cin must be a multiple of 64: not covered
