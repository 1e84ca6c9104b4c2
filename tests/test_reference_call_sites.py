"""The drop-in contract checked against DreamScene's OWN call sites (CPU).

DreamScene's scene_gaussian.py constructs GaussianRasterizationSettings and calls the rasterizer by
keyword in three renderers (score_render :586-646, scene_render :737-870, object_render :951-1021).
Its call sites were read from its AST by tests/golden/make_call_sites.py into ref_call_sites.json;
every keyword it passes is checked against the signatures this package exports under the same import
name, plus the way it unpacks the results."""
import inspect
import json
import os

SITES = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "ref_call_sites.json")))
SCENE = SITES["scene_gaussian.py"]


def test_reference_imports_exactly_what_the_alias_package_exports():
    names = sorted(SCENE["imports"])
    assert names == ["GaussianRasterizationSettings", "GaussianRasterizer"]
    import diff_gaussian_rasterization as D
    for n in names:
        assert hasattr(D, n)


def test_every_keyword_the_reference_passes_is_accepted():
    from diff_gaussian_rasterization import GaussianRasterizationSettings, GaussianRasterizer
    settings, ctor, call = SCENE["settings"], SCENE["ctor"], SCENE["call"]
    assert len(settings) == 3 and len(ctor) == 3 and len(call) == 3       # score / scene / object renderers
    fields = set(GaussianRasterizationSettings._fields)
    for n in settings:
        assert not n["n_args"], "settings are passed by keyword"
        kws = set(n["keywords"])
        assert kws <= fields, kws - fields
        required = {f for f in GaussianRasterizationSettings._fields if f not in GaussianRasterizationSettings._field_defaults}
        assert required <= kws, required - kws
    init = inspect.signature(GaussianRasterizer.__init__)
    for n in ctor:
        assert set(n["keywords"]) == {"raster_settings"} and "raster_settings" in init.parameters
    fwd = inspect.signature(GaussianRasterizer.forward)
    for n in call:
        assert not n["n_args"]
        kws = set(n["keywords"])
        assert kws == {"means3D", "means2D", "shs", "colors_precomp", "opacities", "scales", "rotations", "cov3D_precomp"}
        assert kws <= set(fwd.parameters)


def test_result_unpacking_matches_the_return_arity():
    """score_render unpacks 4 values (important_score first), scene/object_render 3."""
    arities = [n["targets"] for n in SCENE["unpack"]]
    assert sorted(len(a) for a in arities) == [3, 3, 4]
    four = [a for a in arities if len(a) == 4][0]
    assert four[0] == "important_score" and four[1:] == ["rendered_image", "radii", "depth_alpha"]
    for a in arities:
        if len(a) == 3:
            assert a == ["rendered_image", "radii", "depth_alpha"]


def test_simple_knn_call_site():
    """gs_renderer.py:9 imports distCUDA2 from simple_knn._C and calls it with one positional tensor (:590-593)."""
    knn = SITES["gs_renderer.py"]
    assert knn["imports"] and knn["imports"][0] == ["distCUDA2"]
    calls = knn["call"]
    assert calls and all(c["n_args"] == 1 and not c["keywords"] for c in calls)
    from simple_knn._C import distCUDA2
    assert list(inspect.signature(distCUDA2).parameters) == ["points"]
