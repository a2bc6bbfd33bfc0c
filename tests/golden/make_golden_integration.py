"""Record how AutoGPTQ's own construction path builds QuantLinear modules, for tests/test_integration_reference.py.

    python tests/golden/make_golden_integration.py /path/to/AutoGPTQ      # a source checkout of the original project

Imports the original ``auto_gptq/modeling/_utils.py`` unmodified by file path (``accelerate`` is replaced by a stub and
the package ``__init__``s, which pull in the whole model zoo, by namespace stand-ins), then:

* runs its ``make_quant`` (_utils.py:69-148) on the tiny Llama of the test with the backend flags ``from_quantized``
  passes, ``dynamically_import_QuantLinear`` rebound by ``autogptq_b200.patch_auto_gptq()`` and wrapped in a recorder:
  it records the selection call, every constructor call (positional and keyword arguments), the ``device``
  attribute it sets and the ``.to()`` call;
* runs its ``autogptq_post_init`` (_utils.py:380-513) on one probe module per ``QUANT_TYPE`` of the original project's
  QuantLinear classes and on one of ours, and records which types it acts on.

Writes tests/golden/ref_make_quant.json.  Nothing here is imported by the product or the tests.
"""
import ast
import glob
import importlib
import importlib.machinery
import json
import os
import sys
import types

import torch
import torch.nn as nn

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", ".."))

MAKE_QUANT_FLAGS = dict(use_triton=False, disable_exllama=True, disable_exllamav2=False, use_cuda_fp16=True,
                        desc_act=False, trainable=False)


def import_reference_utils(ref):
    """auto_gptq.modeling._utils of the original project, unmodified, without running the package __init__s."""
    pkg_root = os.path.join(ref, "auto_gptq")
    acc = types.ModuleType("accelerate")
    acc.__path__ = []
    acc.__spec__ = importlib.machinery.ModuleSpec("accelerate", None, is_package=True)
    acc_utils = types.ModuleType("accelerate.utils")
    acc_utils.__spec__ = importlib.machinery.ModuleSpec("accelerate.utils", None)
    acc.utils = acc_utils
    sys.modules["accelerate"], sys.modules["accelerate.utils"] = acc, acc_utils
    for pkg, sub in (("auto_gptq", ""), ("auto_gptq.modeling", "modeling"), ("auto_gptq.utils", "utils"),
                     ("auto_gptq.nn_modules", "nn_modules"), ("auto_gptq.nn_modules.qlinear", "nn_modules/qlinear")):
        m = types.ModuleType(pkg)
        m.__path__ = [os.path.join(pkg_root, sub)] if sub else [pkg_root]
        sys.modules[pkg] = m
    return importlib.import_module("auto_gptq.modeling._utils")


def reference_quant_types(ref):
    """The QUANT_TYPE class attributes of the original project's QuantLinear classes (read from the sources)."""
    types_ = set()
    for path in glob.glob(os.path.join(ref, "auto_gptq", "nn_modules", "qlinear", "*.py")):
        for node in ast.walk(ast.parse(open(path).read())):
            if isinstance(node, ast.Assign) and any(getattr(t, "id", None) == "QUANT_TYPE" for t in node.targets):
                types_.add(ast.literal_eval(node.value))
    return sorted(types_)


def main(ref):
    import autogptq_b200
    from autogptq_b200 import QuantLinear
    from tests.test_integration_reference import _quant_names, _tiny_llama

    model = _tiny_llama()                      # imports transformers before the accelerate stand-in exists
    U = import_reference_utils(ref)
    autogptq_b200.patch_auto_gptq()
    selections, built = [], {}

    class Recorded(QuantLinear):
        def __init__(self, *args, **kwargs):
            super().__init__(*args, **kwargs)
            built[id(self)] = {"args": list(args), "kwargs": {k: str(v) if isinstance(v, torch.dtype) else v
                                                              for k, v in kwargs.items()}, "to": []}

        def to(self, *args, **kwargs):
            built[id(self)]["to"].append([str(a) for a in args])
            return super().to(*args, **kwargs)

    select = U.dynamically_import_QuantLinear

    def recording_select(*args, **kwargs):
        assert not args, "make_quant selects by keyword"
        selections.append(kwargs)
        assert select(**kwargs) is QuantLinear
        return Recorded

    U.dynamically_import_QuantLinear = recording_select
    names = _quant_names(model)
    U.make_quant(model, names, 4, 128, **MAKE_QUANT_FLAGS)
    mods = dict(model.named_modules())
    layers = []
    for n in names:
        rec = built[id(mods[n])]
        layers.append({"name": n, **rec, "device": str(mods[n].__dict__["device"])})

    acts_on = []
    for qt in reference_quant_types(ref) + [QuantLinear.QUANT_TYPE]:
        probe = nn.Module()                    # no qweight, no post_init: any handling of it raises
        probe.QUANT_TYPE = qt
        holder = nn.Sequential(probe)
        try:
            assert U.autogptq_post_init(holder, use_act_order=False) is holder
        except (AttributeError, ImportError, TypeError):
            acts_on.append(qt)
    assert QuantLinear.QUANT_TYPE not in acts_on

    out = {"make_quant": {"bits": 4, "group_size": 128, **MAKE_QUANT_FLAGS}, "selections": selections,
           "layers": layers, "post_init_acts_on": acts_on}
    path = os.path.join(HERE, "ref_make_quant.json")
    with open(path, "w") as f:
        json.dump(out, f, indent=1)
        f.write("\n")
    print("wrote", path, f"({len(layers)} layers, post_init acts on {acts_on})")


if __name__ == "__main__":
    main(sys.argv[1])
