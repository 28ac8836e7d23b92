"""Import the live reference (/root/reference) under the alias ``refsrc`` (SURVEY.md §8c recipe).

Only usable in the build container (the GPU box has no /root/reference). Used by
make_golden.py and make_host_curve_golden.py, which write the fixtures the tests compare against.
"""
import importlib
import os
import sys
import types

REF_ROOT = "/root/reference"

_REF_MODULES = [
    "src.curves.space_filling_curves",
    "src.tokenizers.base_patch_embedding",
    "src.tokenizers._2D.zigzag_embedding", "src.tokenizers._2D.hilbert_embedding",
    "src.tokenizers._1D.zigzag_embedding1D", "src.tokenizers._1D.hilbert_embedding1D",
    "src.tokenizers._1D.peano_embedding1D", "src.tokenizers._1D.moore_embedding1D",
    "src.tokenizers._1D.morton_embedding1D", "src.tokenizers._1D.onion_embedding1D",
    "src.tokenizers._2D.random_embedding", "src.tokenizers.multiscale.multi_onion",
    "src.tokenizers.multiscale.multi_morton", "src.tokenizers.multiscale.multi_zigzag",
    "src.tokenizers.multiscale.multi_hilbert", "src.tokenizers.multiscale.multi_peano",
    "src.tokenizers.multiscale.multi_moore",
    "src.models.vit", "src.models.altvit",
    "src.training.train", "src.training.scheduler",
]


def available() -> bool:
    return os.path.isdir(os.path.join(REF_ROOT, "src"))


def load_reference():
    """Returns a dict name -> module, e.g. ref['curves'], ref['vit'], ref['multi_hilbert']."""
    if "refsrc" in sys.modules:
        return sys.modules["refsrc"]._graft_index
    if not available():
        raise RuntimeError("reference not mounted")
    for stub in ("matplotlib", "matplotlib.pyplot"):
        if stub not in sys.modules:
            sys.modules[stub] = types.ModuleType(stub)
    saved_path = list(sys.path)
    saved_mods = {k: v for k, v in sys.modules.items() if k == "src" or k.startswith("src.")}
    for k in saved_mods:
        del sys.modules[k]
    try:
        sys.path = [REF_ROOT] + [p for p in sys.path
                                 if not os.path.isdir(os.path.join(p or os.getcwd(), "src"))]
        loaded = {}
        for name in _REF_MODULES:
            loaded[name] = importlib.import_module(name)
    finally:
        sys.path = saved_path
    index = {}
    for k in [k for k in sys.modules if k == "src" or k.startswith("src.")]:
        mod = sys.modules.pop(k)
        sys.modules["ref" + k] = mod
    sys.modules.update(saved_mods)
    for name, mod in loaded.items():
        index[name.split(".")[-1]] = mod
    index["curves"] = loaded["src.curves.space_filling_curves"]
    sys.modules["refsrc"]._graft_index = index
    return index
