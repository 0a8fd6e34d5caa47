"""Import the UNMODIFIED reference model from the checkout of the original project that
VSR_REFERENCE_ROOT names.  The original is not part of this repository: without that variable
``available()`` is False and its callers skip (the stored golden vectors keep the comparison).

The reference constructor opens four JSON files relative to the CWD
(models/controllable_captioning.py:25-34), so it is constructed from a temp
directory holding those fixture files.
"""
import contextlib
import importlib
import json
import os
import sys
import tempfile

REFERENCE_ROOT = os.environ.get("VSR_REFERENCE_ROOT", "")


def available() -> bool:
    return bool(REFERENCE_ROOT) and os.path.isfile(os.path.join(REFERENCE_ROOT, "models", "controllable_captioning.py"))


@contextlib.contextmanager
def _cwd_with_tables(verb_table=None):
    old = os.getcwd()
    with tempfile.TemporaryDirectory() as tmp:
        for sub, names in (("coco", ("verb_2_vob_all_refine.json", "verb_2_vob.json")),
                           ("flickr", ("verb_2_vob_all_refine_flickr.json", "verb_2_vob_flickr.json"))):
            os.makedirs(os.path.join(tmp, "datasets", sub))
            for nm in names:
                with open(os.path.join(tmp, "datasets", sub, nm), "w") as f:
                    json.dump(verb_table or {}, f)
        os.chdir(tmp)
        try:
            yield tmp
        finally:
            os.chdir(old)


def reference_models():
    """Return the reference's ``models`` package (imported under its own name)."""
    assert available()
    # our drop-in package is also called ``models``; make sure the reference's wins here
    saved = {k: v for k, v in sys.modules.items() if k == "models" or k.startswith("models.")}
    for k in saved:
        del sys.modules[k]
    sys.path.insert(0, REFERENCE_ROOT)
    try:
        mod = importlib.import_module("models")
        ref = {k: v for k, v in sys.modules.items() if k == "models" or k.startswith("models.")}
    finally:
        sys.path.remove(REFERENCE_ROOT)
        for k in list(sys.modules):
            if k == "models" or k.startswith("models."):
                del sys.modules[k]
        sys.modules.update(saved)
    mod._ref_modules = ref
    return mod


def build_reference_model(dims: dict, seed=1234, verb_table=None, dataset="coco"):
    """Construct the reference ControllableCaptioningModel with ``torch.manual_seed(seed)``."""
    import torch
    mods = reference_models()
    with _cwd_with_tables(verb_table):
        # the class body does ``from models import _CaptioningModel`` at import time only
        if seed is not None:
            torch.manual_seed(seed)
        m = mods.ControllableCaptioningModel(
            dims["seq_len"], dims["vocab_size"], dims["bos_idx"],
            det_feat_size=dims["det_feat_size"], input_encoding_size=dims["input_encoding_size"],
            rnn_size=dims["rnn_size"], att_size=dims["att_size"],
            h2_first_lstm=dims["h2_first_lstm"], img_second_lstm=dims["img_second_lstm"],
            dataset=dataset)
    return m.eval()
