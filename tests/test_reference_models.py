"""The drop-in boundary at MODEL level (SURVEY.md 8b): after `install()`, the reference's own
`model.py` builds `Transformer_Net_Cross_Attention`, `SwinTransformerV2`, `Func_Struct_Cross` and
`SwinFusion` with `main.py`'s default arguments on top of our modules, with the same state_dict
keys and shapes as the reference build, and loads a reference-built state_dict strictly.

test_model_builds_on_dropin_modules and test_star_exports_cover_the_reference need a checkout of
the reference, named by MMN_REFERENCE=<dir>, and skip without one.  Stored data cannot stand in
for it: the first builds the models with the reference's own model.py (our side of the comparison
needs that code as much as the reference's side does), and the second lists the public names of
the reference's modules, which no committed fixture records.  Each mode runs in its own
subprocess -- the two `modules.*` sets cannot share one interpreter.
test_install_serves_the_dropin_modules checks, without the reference, the part of the boundary
that is ours: the names model.py imports resolve to our modules.
"""
import importlib
import json
import os
import subprocess
import sys
import types

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import ref_harness as H  # noqa: E402

needs_reference = pytest.mark.skipif(not H.reference_available(), reason="no reference checkout (set MMN_REFERENCE=<dir>)")


@pytest.fixture(scope="module")
def probes(tmp_path_factory):
    d = tmp_path_factory.mktemp("refmodels")
    out = {}
    for mode in ("reference", "installed"):          # reference first: it writes the state_dicts the other loads
        js = d / f"{mode}.json"
        res = subprocess.run([sys.executable, os.path.join(HERE, "ref_harness.py"), mode, str(js), str(d)],
                             capture_output=True, text=True, cwd=str(d), timeout=900)
        assert res.returncode == 0, res.stderr[-3000:]
        out[mode] = json.loads(js.read_text())
    return out


@needs_reference
@pytest.mark.parametrize("name", list(H.MODELS))
def test_model_builds_on_dropin_modules(probes, name):
    ref, ours = probes["reference"][name], probes["installed"][name]
    assert ours["keys"] == ref["keys"]                                   # same keys, same order, same shapes
    assert ours["strict_load"] == [[], []]                               # load_state_dict(strict=True) of a reference build
    # every attention module of the installed build is ours, none is the reference's
    att = [c for c in ours["attention_classes"] if "Attention" in c.split(".")[-1] and not c.startswith("model.")]
    assert att and all(c.startswith("multimodal_neuroimage_b200.modules.") for c in att), att
    assert len(att) == len([c for c in ref["attention_classes"] if not c.startswith("model.")])


@needs_reference
def test_star_exports_cover_the_reference():
    """`model.py` takes everything it uses from `from modules.X import *` (model.py:15,18): every public name of a
    reference module must exist in ours (VERDICT r1: trunc_normal_, Upsample, UpsampleOneStep, np, F were missing)."""
    code = r"""
import importlib, json, sys
sys.path.insert(0, %r); sys.path.insert(0, %r); sys.path.append(%r)
out = {}
for name in ["swin_v2_module", "swinfusion_module", "crossmodal_transformer", "multihead_attention", "position_embedding"]:
    ref = importlib.import_module("modules." + name)
    ours = importlib.import_module("multimodal_neuroimage_b200.modules." + name)
    out[name] = sorted(n for n in dir(ref) if not n.startswith("_") and not hasattr(ours, n))
print(json.dumps(out))
""" % (os.path.join(HERE, "golden", "_shims"), H.ROOT, H.REF)
    res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert res.returncode == 0, res.stderr[-2000:]
    missing = json.loads(res.stdout.strip().splitlines()[-1])
    missing["multihead_attention"] = [n for n in missing["multihead_attention"] if n != "sys"]   # an unused import there
    assert all(not v for v in missing.values()), missing


def test_install_serves_the_dropin_modules():
    """install() registers our modules under the reference's `modules.*` names, so the imports of model.py
    (model.py:8,15,18) bind our classes, and it rebinds the classes of a `model` module imported before it."""
    inst = importlib.import_module("multimodal_neuroimage_b200.install")
    names = ["modules", "model"] + [f"modules.{n}" for n in inst._NAMES]
    saved = {k: sys.modules[k] for k in names if k in sys.modules}
    for k in names:
        sys.modules.pop(k, None)
    try:
        early = types.ModuleType("model")               # a `model` imported before install(): the reference's classes
        early.SwinTransformerBlock = early.Cross_SwinTransformerBlock = early.TransformerEncoder = type("Theirs", (), {})
        sys.modules["model"] = early
        inst.install()
        ours = {n: importlib.import_module(f"multimodal_neuroimage_b200.modules.{n}") for n in inst._NAMES}
        assert all(sys.modules[f"modules.{n}"] is m for n, m in ours.items())
        ns = {}
        exec("from modules.swin_v2_module import *\nfrom modules.swinfusion_module import *\n"
             "from modules.crossmodal_transformer import TransformerEncoder", ns)
        v2, fu, cm = ours["swin_v2_module"], ours["swinfusion_module"], ours["crossmodal_transformer"]
        assert ns["SwinTransformerBlock"] is v2.SwinTransformerBlock and ns["BasicLayer"] is v2.BasicLayer
        assert ns["Cross_SwinTransformerBlock"] is fu.Cross_SwinTransformerBlock
        assert ns["TransformerEncoder"] is cm.TransformerEncoder
        assert early.SwinTransformerBlock is v2.SwinTransformerBlock
        assert early.Cross_SwinTransformerBlock is fu.Cross_SwinTransformerBlock
        assert early.TransformerEncoder is cm.TransformerEncoder
    finally:
        for k in names:
            sys.modules.pop(k, None)
        sys.modules.update(saved)


def test_upsample_modules_match_reference_layout():
    sf = importlib.import_module("multimodal_neuroimage_b200.modules.swinfusion_module")
    up = sf.Upsample(4, 8)
    assert [type(m).__name__ for m in up] == ["Conv2d", "PixelShuffle", "Conv2d", "PixelShuffle"]
    assert up[0].weight.shape == (32, 8, 3, 3)
    assert [type(m).__name__ for m in sf.Upsample(3, 8)] == ["Conv2d", "PixelShuffle"]
    with pytest.raises(ValueError):
        sf.Upsample(5, 8)
    one = sf.UpsampleOneStep(2, 12, 1, input_resolution=(84, 84))
    assert one[0].weight.shape == (4, 12, 3, 3) and one.flops() == 84 * 84 * 12 * 3 * 9
