"""CPU-side checks of the drop-in boundary: the C-ABI library builds / loads without a GPU, exports every entry point
declared in include/gecco_b200.h, and the product path refuses to run without CUDA (there is no CPU fallback)."""
import ctypes
import re
from pathlib import Path

import pytest
import torch

ROOT = Path(__file__).resolve().parent.parent
HEADER = ROOT / "include" / "gecco_b200.h"


def declared_symbols():
    text = re.sub(r"/\*.*?\*/", "", HEADER.read_text(), flags=re.S)
    names = re.findall(r"^\s*(?:const\s+)?[A-Za-z_][A-Za-z0-9_]*\s*\*?\s*(gecco_[a-z0-9_]+)\s*\(", text, flags=re.M)
    return sorted(set(names))


def test_header_declares_the_hot_path_entry_points():
    names = declared_symbols()
    for required in ("gecco_init", "gecco_last_error", "gecco_create", "gecco_destroy", "gecco_workspace_bytes", "gecco_denoise",
                     "gecco_sample", "gecco_lookup", "gecco_pool_attention", "gecco_unpool_attention", "gecco_gemm", "gecco_reparam"):
        assert required in names, (required, names)


def test_library_exports_every_declared_symbol():
    from gecco_b200 import _abi

    assert _abi.lib_path().exists(), "libgecco_b200.so is missing: run `python -m gecco_b200.build`"
    lib = ctypes.CDLL(str(_abi.lib_path()))
    missing = [n for n in declared_symbols() if not hasattr(lib, n)]
    assert not missing, f"declared in include/gecco_b200.h but not exported: {missing}"


def test_no_cpu_fallback():  # CPU tensors are refused whether or not the machine has a GPU
    import gecco_b200 as G
    from gecco_b200 import _abi
    from tests.models_b200 import build

    model = build("uncond", "gaussian", [0.0, 0.0, 0.0], [1.0, 1.0, 1.0], 165.0, 1, torch.device("cpu"))
    with pytest.raises((_abi.GeccoError, RuntimeError)):
        model(torch.randn(1, 128, 3), torch.tensor([1.0]), None)
    with pytest.raises((_abi.GeccoError, RuntimeError)):
        model.sample_stochastic((1, 128, 3), None, num_steps=2)
    assert isinstance(model, G.Diffusion)
