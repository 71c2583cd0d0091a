"""CPU checks of the boundary: the library loads without a GPU, exports every symbol that
include/b2nerf.h declares, reports errors through the C convention, and the host logic that
needs no device (hash geometry, z tables contract, loud failure on CPU tensors) behaves."""
import ctypes
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as ge
    ge.build()
    from b2n import _lib
    return _lib


def test_exports_every_declared_symbol(lib):
    hdr = open(os.path.join(ROOT, "include", "b2nerf.h")).read()
    declared = set(re.findall(r"\b(b2n_[a-z0-9_]+)\s*\(", hdr))
    assert len(declared) >= 20
    raw = ctypes.CDLL(lib.LIB_PATH)
    for name in declared:
        assert hasattr(raw, name), name
    assert declared == set(lib.SIGNATURES), declared ^ set(lib.SIGNATURES)
    assert not any(n.startswith("b2n_debug") for n in declared)        # debug aids live in b2nerf_debug.h only
    dbg = open(os.path.join(ROOT, "include", "b2nerf_debug.h")).read()
    declared_dbg = set(re.findall(r"\b(b2n_[a-z0-9_]+)\s*\(", dbg)) - {"b2n_last_error"}
    for name in declared_dbg:
        assert hasattr(raw, name), name
    assert declared_dbg == set(lib.DEBUG_SIGNATURES), declared_dbg ^ set(lib.DEBUG_SIGNATURES)
    assert raw.b2n_abi_version() == lib.ABI_VERSION


def test_error_convention_without_gpu(lib):
    # argument validation happens before any launch, so it can be exercised on a CPU box
    with pytest.raises(ValueError, match="b2n_composite_fwd"):
        lib.call("b2n_composite_fwd", None, None, None, None, None, None, 0, None, None, 4, 5000, None, None, None,
                 None, None)
    with pytest.raises(ValueError):
        lib.call("b2n_hash_fwd", None, 8, 1.0, None, None, 0, 2, None, 32, 0, None)
    # empty inputs are a no-op (rc 0) even with null pointers
    lib.call("b2n_pe_fwd", None, 0, 3, None, 4, None, 27, 0, None)
    assert lib.lib.b2n_march_scan_scratch(2 ** 18) >= 4 * (128 + 2)


def test_hash_variant_switch_reports_and_validates(lib):
    """b2n_debug_hash_variant / b2n_debug_hash_config are host state: the shipped configuration is readable, a switch
    restores what it found, and values the kernels cannot run (a merge threshold whose res^3 cell id overflows uint32, an
    unknown variant) are refused without changing anything"""
    shipped = lib.hash_config()
    assert shipped == (3, 128)
    with lib.hash_variant(1, 1625):
        assert lib.hash_config() == (1, 1625)
        with lib.hash_variant(2, 0):
            assert lib.hash_config() == (2, 0)
        assert lib.hash_config() == (1, 1625)
    assert lib.hash_config() == shipped
    for bad in ((3, 1626), (3, 2 ** 20), (4, 128), (-1, 128)):
        with pytest.raises(ValueError, match="b2n_debug_hash_variant"):
            with lib.hash_variant(*bad):
                pass
        assert lib.hash_config() == shipped


def test_product_has_no_cpu_path(lib):
    import b2n
    with pytest.raises(ValueError, match="no CPU path"):
        b2n.fourier_encode(torch.zeros(4, 3), torch.ones(2))
    with pytest.raises(ValueError, match="no CPU path"):
        b2n.composite(torch.zeros(8, 3), torch.zeros(8), torch.zeros(2, 4), torch.zeros(2, 3))


def test_optional_helpers_have_no_cpu_path_either(lib):
    """b2n.optim.FusedAdamW / b2n.graphs.GraphedStep: host logic only (descriptor layout, option validation); on CPU tensors
    they refuse to run instead of falling back."""
    import ctypes
    import b2n
    from b2n.optim import _OptTensor
    assert ctypes.sizeof(_OptTensor) == 80                       # b2n_opt_tensor of include/b2nerf.h: 4 ptr, i64, 8 f32, 2 i32
    p = torch.nn.Parameter(torch.zeros(10))
    opt = b2n.optim.FusedAdamW([{"params": [p], "tv_weight": 1e-3, "max_norm": 1.0}], lr=1e-2)
    assert opt.defaults["weight_decay"] == 1e-2 and opt.param_groups[0]["tv_weight"] == 1e-3
    assert opt._step_supports_amp_scaling
    opt.step()                                                   # no gradients: nothing to do, no kernel call
    p.grad = torch.ones(10)
    with pytest.raises(ValueError, match="no CPU path"):
        opt.step()
    with pytest.raises(ValueError):
        b2n.optim.FusedAdamW([p], lr=-1.0)
    with pytest.raises(ValueError, match="no CPU path"):
        b2n.graphs.GraphedStep(lambda x: x + 1, (torch.zeros(3),))


def test_hash_geometry_matches_oracle_table(lib):
    import b2n
    from oracle import nerf_oracle as O
    for args in ((16, 16, 1.5, 19), (16, 16, 1.5, 20), (12, 16, 1.5, 16), (14, 16, 1.5, 19), (6, 4, 1.7, 11)):
        g = b2n.HashGeometry(*args, 2)
        lv = O.hash_level_table(*args)
        assert g.levels == [(l.scale, l.res, l.size, l.offset, l.hashed) for l in lv]
        assert g.n_entries == O.hash_table_entries(lv)
    assert b2n.HashGeometry(16, 16, 1.5, 19, 2).n_params == 13026992       # SURVEY.md A2


def test_dropin_module_surface(lib):
    """names run.py reaches for (SURVEY.md 8b / F10) exist with the reference's shapes."""
    from src.core import NeuralField
    from src.renderer import DensityGrid, render_image, render_rays, sample_stratified, volume_render  # noqa: F401
    m = NeuralField(dict(mode="part4", scene_bound=1.5, deform_n_levels=12, deform_log2_hashmap_size=16,
                         log2_hashmap_size=20))
    assert m.deformation_grid is m.deform_grid_start
    assert m.canonical_repr.encoding.params.dim() == 1 and m.canonical_repr.encoding.params.numel() == 24575648
    assert m.canonical_repr.encoding.n_output_dims == 32 and m.canonical_repr.out_dim == 32
    assert not torch.equal(m.deform_grid_mid.encoding.params, m.deform_grid_start.encoding.params)
    assert m.deform_decoder.displacement_scale.item() == pytest.approx(0.1)
    names = [n for n, _ in m.deform_decoder.named_parameters()]
    assert "displacement_scale" in names and any("deform_net" in n for n in names)
    g = DensityGrid(resolution=8, bound=1.5, threshold=0.01)
    assert set(g.state_dict()) == {"grid", "binary_grid"} and g.binary_grid.dtype == torch.bool
    assert g.should_update(32, 16, 0) and not g.should_update(8, 16, 16) and not g.should_update(33, 16, 0)
    assert float(g.binary_grid.float().mean()) == 1.0
    with pytest.raises(ValueError):
        NeuralField(dict(mode="part3"))(torch.zeros(1, 3), torch.zeros(1, 3))
    with pytest.raises(ValueError):
        NeuralField(dict(mode="part2_nerf", L_embed=4))(torch.zeros(1, 3))
