"""Drop-in check: every public module-level name of the reference's packages exists under the same name here
(``import lca_b200 as yunchang`` must keep working for user code).  The names were read from the reference tree
(long-context-attention / yunchang 0.6.4, commit 56118e0d) by ``tools/reference_api_surface.py`` and are stored in
``tests/golden/reference_api_surface.json``."""
import importlib
import json
import os

import pytest

with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_api_surface.json")) as _f:
    REF = json.load(_f)

# names that are implementation details of the reference's optional third-party backends (symbols of flash_attn /
# flashinfer / aiter / sageattention that it merely imports at module level) or plain helper imports
THIRD_PARTY = {
    "yunchang.globals": {"flash3_attn_func", "flash_attn_forward_hopper", "flash_attn_func_hopper_backward",
                         "flash_attn_func_aiter", "single_prefill_with_kv_cache", "cuda_arch"},
    "yunchang.kernels": {"SparseAttentionMeansim", "flash3_attn_func", "partial", "auto"},
}


@pytest.mark.parametrize("mod", ["yunchang", "yunchang.ring", "yunchang.hybrid", "yunchang.ulysses", "yunchang.comm",
                                 "yunchang.kernels", "yunchang.globals"])
def test_every_reference_name_resolves(mod):
    ours = importlib.import_module(mod.replace("yunchang", "lca_b200", 1))
    wanted = set(REF["packages"][mod]) - THIRD_PARTY.get(mod, set())
    wanted -= {"torch", "dist", "os", "Enum", "Optional", "Tuple", "Any", "Tensor", "Function", "Module"}
    missing = sorted(n for n in wanted if not hasattr(ours, n))
    assert not missing, f"{mod}: {missing}"


def test_singleton_aliases():
    import lca_b200.globals as g
    assert g.ProcessGroupSingleton() is g.PROCESS_GROUP
    assert g.Singleton() is g.Singleton()
    assert g.get_cuda_arch().count(".") == 1


@pytest.mark.parametrize("mod", sorted(REF["modules"]))
def test_every_reference_module_path_imports_with_its_public_defs(mod):
    """``from yunchang.ring.zigzag_ring_flash_attn import zigzag_ring_flash_attn_forward`` style imports of third-party
    code: same module path, same top-level function / class names."""
    ours = importlib.import_module(mod.replace("yunchang", "lca_b200", 1))
    missing = sorted(n for n in REF["modules"][mod] if not hasattr(ours, n))
    assert not missing, f"{mod}: {missing}"
