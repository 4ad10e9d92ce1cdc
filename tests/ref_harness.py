"""Harness for driving the UNMODIFIED reference (the checkout MMN_REFERENCE names, read-only) from tests and
fixture generators: import-time stubs for the packages the reference imports but this image
lacks, the three shims of SURVEY.md 8c, and `main.py`'s own default arguments per phase.

Two modes, chosen before anything of the reference is imported:
  reference   the reference's `modules/*` (needs the `timm` shim of tests/golden/_shims)
  installed   `multimodal_neuroimage_b200.install()` first: the reference's model.py / trainer.py
              / main.py then run on the drop-in modules (what a user of the reference does)

Run as a script it is the probe the CPU tests launch in a subprocess (one mode per process:
the two module sets cannot coexist under the same `modules.*` names):
    python tests/ref_harness.py <reference|installed> <out.json> [state_dict dir]
"""
from __future__ import annotations

import importlib
import json
import os
import sys
import types

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
REF = os.environ.get("MMN_REFERENCE", "")

# model class -> (phase whose `_phaseN` flags configure it, extra command line) -- main.py:209-332, utils.py:95-128
MODELS = {
    "Transformer_Net_Cross_Attention": ("2", ["--fmri_type", "divided_frequency"]),
    "SwinTransformerV2": ("3", []),
    # phase 5's own default patch size (4, main.py:298) gives a 21x21 token grid that window 6 does not divide: the
    # reference itself fails in SwinTransformerBlock_fusion.calculate_mask with it; 7 is the un-suffixed default (main.py:199)
    "Func_Struct_Cross": ("5", ["--fmri_type", "divided_frequency", "--patch_size_phase5", "7"]),
    "SwinFusion": ("6", []),
}


def reference_available() -> bool:
    return bool(REF) and os.path.isfile(os.path.join(REF, "model.py"))


class _Stub(types.ModuleType):
    """A module whose every attribute is another stub (and callable): enough for `import x` / `from x import y`."""

    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)
        m = _Stub(self.__name__ + "." + name)
        setattr(self, name, m)
        return m

    def __call__(self, *a, **k):
        return self


def stub_missing_packages():
    import pandas  # noqa: F401  (must import before `pytz` is stubbed: pandas probes it as an optional dependency)
    for name in ["nibabel", "nitime", "nitime.timeseries", "nitime.analysis", "nitime.viz", "optuna", "pytz", "skimage",
                 "skimage.transform", "torchaudio", "torchaudio.functional", "xgboost", "dill"]:
        try:
            importlib.import_module(name)
        except Exception:
            sys.modules[name] = _Stub(name)


def enter(mode: str):
    """Put the reference on sys.path in `mode` and return its `model` module."""
    import torch
    assert mode in ("reference", "installed")
    if ROOT not in sys.path:
        sys.path.insert(0, ROOT)
    stub_missing_packages()
    os.environ.setdefault("WANDB_MODE", "disabled")
    if mode == "reference":
        sys.path.insert(0, os.path.join(HERE, "golden", "_shims"))           # timm.models.layers (3 symbols)
        orig = torch.Tensor.get_device                                         # swin_v2_module.py:154 on CPU (SURVEY F5)
        torch.Tensor.get_device = lambda self: (self.device if not self.is_cuda else orig(self))
    else:
        import multimodal_neuroimage_b200 as pkg
        pkg.install()
    if REF not in sys.path:
        sys.path.append(REF)
    model = importlib.import_module("model")
    # transformers >= 5: Transformer_Block.init_weights re-enters itself through post_init (SURVEY.md 8c shim 3)
    tb = model.Transformer_Block
    if not getattr(tb, "_mmn_guarded", False):
        orig_init = tb.init_weights
        base_init = model.BertPreTrainedModel.init_weights

        def guarded(self, *a, **k):
            if getattr(self, "_mmn_in_init", False):
                return base_init(self, *a, **k)
            self._mmn_in_init = True
            try:
                return self.post_init()
            finally:
                self._mmn_in_init = False
        tb.init_weights = guarded
        tb._mmn_guarded = True
        del orig_init
    return model


def default_kwargs(phase: str, extra=()):
    """The kwargs dict `main.run_phase` hands to Trainer and every model (main.py:340-357): argparse defaults of
    `get_arguments` with the active phase's `_phaseN` suffix stripped (utils.py:144-151)."""
    main = importlib.import_module("main")
    utils = importlib.import_module("utils")
    argv = sys.argv
    sys.argv = ["main.py", "--step", phase] + list(extra)
    try:
        args = main.get_arguments("/tmp/mmn_ref_base")
    finally:
        sys.argv = argv
    kw = utils.sort_args(phase, vars(args))
    kw.pop("wandb_key", None)                  # SURVEY F11: never carry the hard-coded key anywhere
    return kw


def build_model(model_mod, name: str, seed: int = 0):
    import torch
    phase, extra = MODELS[name]
    kw = default_kwargs(phase, extra)
    torch.manual_seed(seed)
    return getattr(model_mod, name)(**kw), kw


def _probe(mode: str, out_json: str, sd_dir: str | None):
    import torch
    model = enter(mode)
    report = {}
    for name in MODELS:
        m, _ = build_model(model, name)
        sd = m.state_dict()
        entry = {"keys": {k: list(v.shape) for k, v in sd.items()},
                 "attention_classes": sorted({type(x).__module__ + "." + type(x).__name__ for x in m.modules()
                                              if "Attention" in type(x).__name__ and "Bert" not in type(x).__name__})}
        if sd_dir:
            path = os.path.join(sd_dir, name + ".pth")
            if mode == "reference":
                torch.save(sd, path)
            elif os.path.exists(path):
                ref_sd = torch.load(path)
                res = m.load_state_dict(ref_sd, strict=True)
                entry["strict_load"] = [list(res.missing_keys), list(res.unexpected_keys)]
                # the partial loader the trainer uses for transfer (model.py:90-108)
                m.load_partial_state_dict(ref_sd, load_cls_embedding=True)
        report[name] = entry
    with open(out_json, "w") as f:
        json.dump(report, f)


if __name__ == "__main__":
    _probe(sys.argv[1], sys.argv[2], sys.argv[3] if len(sys.argv) > 3 else None)
