"""CPU-only checks of the drop-in boundary: the C-ABI library builds, loads, and exports every symbol that
include/pg_b200.h declares; the Python binding covers the same set; the product refuses to run without CUDA
(no CPU fallback) and keeps the reference's constructor signatures / state-dict keys."""

import inspect
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")


@pytest.fixture(scope="module")
def lib():
    from pytorch_generative_b200 import _build, _lib

    _build.build(verbose=False)
    return _lib.load()


def _declared_symbols():
    text = open(os.path.join(ROOT, "include", "pg_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(pg_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol(lib):
    from pytorch_generative_b200 import _lib

    declared = _declared_symbols()
    assert len(declared) >= 20
    for sym in declared:
        assert hasattr(lib, sym), f"{sym} declared in include/pg_b200.h but not exported by libpg_b200.so"
    assert sorted(_lib.EXPORTED_SYMBOLS) == declared, set(_lib.EXPORTED_SYMBOLS) ^ set(declared)
    assert lib.pg_abi_version() == 1


def test_no_cpu_fallback():
    from pytorch_generative_b200 import models, nn

    with pytest.raises(RuntimeError):
        models.ImageGPT(3, 3, 8, 1, 2, 16)(torch.zeros(1, 3, 8, 8))
    with pytest.raises(RuntimeError):
        nn.NCHWLayerNorm(8)(torch.zeros(1, 8, 2, 2))
    with pytest.raises(RuntimeError):
        nn.CausalConv2d(True, 3, 8, 3, padding=1)(torch.zeros(1, 3, 4, 4))
    with pytest.raises(RuntimeError):
        models.PixelCNN(1, 1, 1, 8, 8)(torch.zeros(1, 1, 8, 8))


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "pytorch_generative_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh")):
                src = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in src.replace("# oracle", ""), f"{f} mentions the oracle"


@pytest.mark.parametrize("name,cls", [("pixel_cnn", "PixelCNN"), ("gated_pixel_cnn", "GatedPixelCNN"),
                                      ("pixel_snail", "PixelSNAIL"), ("image_gpt", "ImageGPT")])
def test_constructor_and_state_dict_match_reference_fixture(name, cls):
    from pytorch_generative_b200 import models

    fx = torch.load(os.path.join(GOLD, f"model_{name}.pt"), weights_only=False)
    m = getattr(models, cls)(**fx["cfg"])
    sd = m.state_dict()
    assert set(sd) == set(fx["state_before"])
    for k, v in fx["state_before"].items():
        assert sd[k].shape == v.shape and sd[k].dtype == v.dtype, k
    m.load_state_dict(fx["state_before"])  # a reference checkpoint loads as is
    m.load_state_dict(fx["state_after"])   # ... including the dynamic _c/_h/_w buffers
    assert int(m._h) == fx["x"].shape[2]
    sig = inspect.signature(getattr(models, cls).__init__)
    assert list(sig.parameters)[-1] == "sample_fn" and sig.parameters["sample_fn"].default is None


def test_sample_argument_contract():
    from pytorch_generative_b200 import models

    m = models.PixelCNN(1, 1, 1, 8, 8)
    with pytest.raises(AssertionError):
        m.sample()  # neither n_samples nor conditioned_on (reference base.py:87-89)
    with pytest.raises(AttributeError):
        m.sample(n_samples=1)  # before any forward: shape buffers do not exist yet, as in the reference


# Where the reference package (pytorch_generative) defines the names the overlay rebinds: `nn` re-exports them from
# two modules, `models` from one module per model under the namespace package `models.autoregressive`.
_REF_LAYOUT = {
    "nn/attention.py": ["CausalAttention", "LinearCausalAttention", "image_positional_encoding"],
    "nn/convolution.py": ["CausalConv2d", "GatedActivation", "NCHWLayerNorm"],
    "models/autoregressive/pixel_cnn.py": ["PixelCNN"],
    "models/autoregressive/gated_pixel_cnn.py": ["GatedPixelCNN"],
    "models/autoregressive/pixel_snail.py": ["PixelSNAIL"],
    "models/autoregressive/image_gpt.py": ["ImageGPT"],
}


def _write_reference_stand_in(root):
    """A package with the reference's module layout whose names are placeholders (the overlay only rebinds them)."""
    pkg = root / "pytorch_generative"
    inits = {"": "from pytorch_generative import models, nn\n", "nn": "", "models": ""}
    for rel, names in _REF_LAYOUT.items():
        (pkg / rel).parent.mkdir(parents=True, exist_ok=True)
        (pkg / rel).write_text("".join(f"class {n}:\n    pass\n" for n in names))
        mod = "pytorch_generative." + rel[:-3].replace("/", ".")
        inits[rel.split("/")[0]] += f"from {mod} import {', '.join(names)}\n"
    for sub, text in inits.items():
        (pkg / sub / "__init__.py").write_text(text)


def test_overlay_rebinds_reference_names(tmp_path):
    """overlay.install() makes the reference package hand out the B200 classes (and uninstall() restores it)."""
    import sys

    _write_reference_stand_in(tmp_path)
    sys.path.insert(0, str(tmp_path))
    try:
        import pytorch_generative as ref

        from pytorch_generative_b200 import models, nn, overlay

        orig = ref.models.ImageGPT
        bound = overlay.install()
        try:
            assert ref.models.ImageGPT is models.ImageGPT and ref.nn.CausalAttention is nn.CausalAttention
            assert ref.models.autoregressive.pixel_snail.PixelSNAIL is models.PixelSNAIL
            assert len(bound) == 6 + 2 * 4  # 6 nn names (incl. LinearCausalAttention) + 4 models in 2 namespaces
            m = ref.models.PixelCNN(in_channels=1, out_channels=1, n_residual=1, residual_channels=4, head_channels=4)
            assert isinstance(m, models.PixelCNN)
        finally:
            overlay.uninstall()
        assert ref.models.ImageGPT is orig
        assert ref.models.autoregressive.pixel_snail.PixelSNAIL is not models.PixelSNAIL
        assert ref.nn.CausalAttention is not nn.CausalAttention
    finally:
        sys.path.remove(str(tmp_path))
        for name in [n for n in sys.modules if n == "pytorch_generative" or n.startswith("pytorch_generative.")]:
            del sys.modules[name]


def test_ctypes_structs_and_signatures_match_the_header(tmp_path):
    """The header is the contract: compile it with gcc (plain C, no CUDA), compare sizeof / offsetof of
    pg_gemm_epilogue with the ctypes mirror, and the arity of every declared function with the Python binding."""
    import ctypes
    import shutil
    import subprocess

    from pytorch_generative_b200 import _lib

    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("gcc not available")
    fields = [name for name, _ in _lib.GemmEpilogue._fields_]
    prog = ['#include <stddef.h>', '#include <stdio.h>', '#include "pg_b200.h"', "int main(void) {",
            '  printf("size %zu\\n", sizeof(pg_gemm_epilogue));']
    prog += [f'  printf("{f} %zu\\n", offsetof(pg_gemm_epilogue, {f}));' for f in fields]
    prog += ['  printf("acts %d %d %d\\n", PG_ACT_GELU, PG_ACT_GIVEN, PG_ACT_STORE_DERIV);', "  return 0;", "}"]
    src = tmp_path / "layout.c"
    src.write_text("\n".join(prog))
    exe = tmp_path / "layout"
    subprocess.run([gcc, "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)],
                   check=True)
    got = dict(line.split(" ", 1) for line in subprocess.run([str(exe)], capture_output=True, text=True,
                                                             check=True).stdout.strip().splitlines())
    assert int(got["size"]) == ctypes.sizeof(_lib.GemmEpilogue)
    for f in fields:
        assert int(got[f]) == getattr(_lib.GemmEpilogue, f).offset, f
    assert got["acts"].split() == [str(_lib.ACT_GELU), str(_lib.ACT_GIVEN), str(_lib.ACT_STORE_DERIV)]

    # arity of every prototype in the header == len(argtypes) of the binding
    text = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "pg_b200.h")).read(), flags=re.S)
    for name, args in re.findall(r"\b(pg_[a-z0-9_]+)\s*\(([^)]*)\)\s*;", text):
        n_args = 0 if args.strip() in ("", "void") else len(args.split(","))
        if name in _lib._SIGNATURES:
            assert len(_lib._SIGNATURES[name]) == n_args, (name, n_args, len(_lib._SIGNATURES[name]))
