"""Drop-in surface (SURVEY.md section 4 (v)): every name the reference's own modules reach in `diff_gaussian_rasterization`,
`simple_knn._C`, `plyfile` and `gsplat`, the keywords it builds GaussianRasterizationSettings with and calls the operator
with, and the tile grid it derives from get_block_XY() -- recorded from the reference by
tests/golden/make_dropin_golden.py into tests/golden/dropin.json -- resolve against our packages, unchanged.  Nothing is
executed on a device: the reference hard-codes "cuda" everywhere (SURVEY F3)."""
import importlib
import importlib.util
import inspect
import json
import os

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
PKG = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "grendel-gs_b200")


def _shim(name, path):
    """The opt-in stand-ins under shims/, loaded from their files so they cannot shadow a real install."""
    spec = importlib.util.spec_from_file_location(f"{name}_shim", os.path.join(PKG, "shims", *path))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_reference_modules_import_against_our_package():
    rec = json.load(open(os.path.join(G, "dropin.json")))
    import diff_gaussian_rasterization as dgr
    from gs_b200 import ops
    assert dgr.__file__.startswith(PKG), dgr.__file__
    modules = {"diff_gaussian_rasterization": dgr, "simple_knn._C": importlib.import_module("simple_knn._C"),
               "plyfile": _shim("plyfile", ("plyfile.py",)), "gsplat": _shim("gsplat", ("gsplat", "__init__.py"))}
    assert set(rec["names_used"]) == set(modules)
    for mod, names in rec["names_used"].items():
        assert names, mod
        for dotted in names:
            obj = modules[mod]
            for part in dotted.split("."):
                assert hasattr(obj, part), f"{mod}.{dotted}"
                obj = getattr(obj, part)
    # arguments/__init__.py:254-257: the block sizes come from the extension, the reference derives its tile grid from them
    g = rec["grid_1080p"]
    assert dgr._C.get_block_XY() == (g["BLOCK_X"], g["BLOCK_Y"], g["ONE_DIM_BLOCK_SIZE"])
    rs_1080p = dgr.GaussianRasterizationSettings(1080, 1920, 1.0, 1.0, None, 1.0, None, None, 3, None, False, False)
    assert ops._tiles(rs_1080p) == (g["TILE_Y"], g["TILE_X"])
    # the settings object is built with exactly these keywords at gaussian_renderer/__init__.py:930-943
    assert tuple(rec["settings_keywords"]) == dgr.GaussianRasterizationSettings._fields, rec["settings_keywords"]
    # and the operator is called with exactly these keywords (:949-956, :1271-1282)
    sig_p = inspect.signature(dgr.GaussianRasterizer.preprocess_gaussians).parameters
    for name in rec["preprocess_keywords"]:
        assert name in sig_p, name
    sig_r = inspect.signature(dgr.GaussianRasterizer.render_gaussians).parameters
    for name in rec["render_keywords"]:
        assert name in sig_r, name
