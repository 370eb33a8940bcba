"""Build recipe for the C oracle (gcc only; output stays under oracle/_build/)."""
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "csrc", "oracle.c")
_OUT_DIR = os.path.join(_HERE, "_build")
_OUT = os.path.join(_OUT_DIR, "liboracle.so")


def lib_path() -> str:
    return _OUT


def build(force: bool = False) -> str:
    """Compile oracle/csrc/oracle.c -> oracle/_build/liboracle.so (idempotent)."""
    if (not force and os.path.exists(_OUT)
            and os.path.getmtime(_OUT) >= os.path.getmtime(_SRC)):
        return _OUT
    os.makedirs(_OUT_DIR, exist_ok=True)
    # Processes that build at once (the spawned workers of tests/test_dist_cpu.py on a fresh tree) each compile to
    # their own file and rename it into place, so none of them can load a library another one is still writing.
    tmp = f"{_OUT}.{os.getpid()}.tmp"
    # -ffp-contract=off: the restatement spells out every fmaf itself.
    cmd = ["gcc", "-O2", "-std=c11", "-fPIC", "-shared", "-fopenmp",
           "-ffp-contract=off", "-fno-fast-math", "-o", tmp, _SRC, "-lm"]
    subprocess.run(cmd, check=True)
    os.replace(tmp, _OUT)
    return _OUT


# ---- the unmodified reference, for bench.py --impl reference on the GPU box ---------------------------------
# /root/reference exists only in the authoring container.  The reference is pure Python (no build step): this
# recipe copies its hot-path package (models/*.py, the files SURVEY.md section 8a names) verbatim into oracle/_ref/,
# which is git-ignored (no reference source enters the history) but NOT gpurun-ignored, so it travels to the GPU
# box next to the built .so files.  bench.py's reference arm imports it from there ("kind": "reference") and
# falls back to oracle/torch_port.py ("kind": "port") when the copy is absent.
REF_SRC = "/root/reference"
_REF_OUT = os.path.join(_HERE, "_ref")
_REF_FILES = ("models/__init__.py", "models/vqvae.py", "models/quantizer.py", "models/encoder.py",
              "models/decoder.py", "models/residual.py")


def ref_path() -> str:
    """oracle/_ref when the verbatim copy of the reference's models package is present, else ''."""
    return _REF_OUT if all(os.path.exists(os.path.join(_REF_OUT, f)) for f in _REF_FILES) else ""


def build_ref() -> str:
    """Copy the reference's models package into oracle/_ref/ (authoring container only; a no-op elsewhere)."""
    if not os.path.isdir(REF_SRC):
        return ref_path()
    import shutil
    for f in _REF_FILES:
        dst = os.path.join(_REF_OUT, f)
        os.makedirs(os.path.dirname(dst), exist_ok=True)
        shutil.copyfile(os.path.join(REF_SRC, f), dst)
    return _REF_OUT
