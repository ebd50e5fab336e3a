#!/usr/bin/env python
"""Record tests/golden/shim_reference.json from the UNMODIFIED reference (needs its source tree, imported as in
make_golden.py): build gptqmodel_b200.reference_shim's class on the reference base `GPTQQuantLinear`, construct it the
way `create_quant_module` does (gptqmodel/utils/model.py:630-647), and run the reference's own discovery walk over it.
Also records the reference's constructor / validate() signatures and the SUPPORTS_* attributes its base classes leave
to the kernel, which tests/test_reference_shim.py's stand-in hierarchy must restate.

    python tests/golden/check_shim.py
"""
import inspect
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, HERE)

import make_golden  # noqa: E402  (stub finder + namespace shells for the reference package)

make_golden.import_reference()

import torch  # noqa: E402
from gptqmodel.adapter.adapter import Lora  # noqa: E402
from gptqmodel.models._const import DEVICE, PLATFORM  # noqa: E402
from gptqmodel.nn_modules.qlinear import BaseQuantLinear, GPTQQuantLinear, GroupedQuantLinear  # noqa: E402
from gptqmodel.quantization import FORMAT, METHOD  # noqa: E402
from gptqmodel.utils.backend import BACKEND  # noqa: E402

from gptqmodel_b200.reference_shim import make_reference_kernel  # noqa: E402

out = {}
# a maintainer adds BACKEND.GPTQ_B200; any existing member serves the purpose of the check
backend = getattr(BACKEND, "GPTQ_B200", None) or BACKEND.GPTQ_MARLIN
B200Linear = make_reference_kernel(GPTQQuantLinear, backend=backend, methods=[METHOD.GPTQ],
                                   formats={FORMAT.GPTQ: 120, FORMAT.GPTQ_V2: 120, FORMAT.GPTQ_P: 120}, adapters=[Lora],
                                   devices=[DEVICE.CUDA], platforms=[PLATFORM.LINUX])
out["mro"] = [c.__name__ for c in B200Linear.__mro__][:6]
B200Linear.verify_supports_params()
out["verify_supports_params"] = True

# the reference's discovery walk (utils/importer.py:110-127), restated on the reference's own root class
seen, kernels = set(), []


def walk(cls):
    for sub in cls.__subclasses__():
        if sub in seen:
            continue
        seen.add(sub)
        walk(sub)
        if "SUPPORTS_FORMATS" in sub.__dict__ and getattr(sub, "SUPPORTS_BACKEND_SELECTION", True):
            kernels.append(sub)


walk(BaseQuantLinear)
out["discovered"] = B200Linear in kernels
ranked = sorted((k for k in kernels if FORMAT.GPTQ in (k.SUPPORTS_FORMATS or {})),
                key=lambda k: k.SUPPORTS_FORMATS[FORMAT.GPTQ], reverse=True)
out["top_for_gptq"] = ranked[0].__name__ if ranked else None

# validate(): no CUDA device here -> NotImplementedError ("try the next kernel"), never a TypeError
B200Linear.cached_validate_once.cache_clear()
ok, err = B200Linear.validate(bits=4, group_size=128, desc_act=False, sym=True, in_features=256, out_features=128,
                              pack_dtype=torch.int32, dtype=torch.float16)
out["validate_without_gpu"] = [ok, type(err).__name__ if err else None]

# construct exactly like create_quant_module (validate_once patched: the container has no GPU)
B200Linear.validate_once = classmethod(lambda cls: (True, None))
B200Linear.cached_validate_once.cache_clear()
m = B200Linear(bits=4, group_size=128, desc_act=False, sym=True, in_features=256, out_features=128,
               pack_dtype=torch.int32, bias=True, dtype=torch.float16, name="model.layers.0.self_attn.q_proj",
               lm_head_name="lm_head", backend=backend, register_buffers=True, adapter=None)
out["constructed"] = True
out["shapes"] = {k: list(getattr(m, k).shape) for k in ("qweight", "qzeros", "scales", "g_idx", "bias")}
out["qzeros_format_initial"] = m.qzero_format()
out["isinstance_base"] = isinstance(m, GPTQQuantLinear) and isinstance(m, BaseQuantLinear)
out["state_dict_keys"] = sorted(m.state_dict().keys())
out["name"] = m.name
out["n_list_buffers"] = len(m.list_buffers())
bad = None
try:
    B200Linear(bits=16, group_size=128, desc_act=False, sym=True, in_features=256, out_features=128,
               pack_dtype=torch.int32, bias=False, backend=backend, adapter=None)
except NotImplementedError:
    bad = "NotImplementedError"
except Exception as e:  # noqa: BLE001
    bad = type(e).__name__
out["bits16"] = bad
# 3-bit continuous and planar 5-bit (format gptq_p) modules: checkpoint-shaped buffers, 4- / 8-bit kernel container
m3 = B200Linear(bits=3, group_size=128, desc_act=False, sym=True, in_features=256, out_features=128,
                pack_dtype=torch.int32, bias=False, backend=backend, adapter=None, register_buffers=True)
m5 = B200Linear(bits=5, group_size=64, desc_act=False, sym=False, in_features=256, out_features=128,
                pack_dtype=torch.int32, bias=False, backend=backend, adapter=None, register_buffers=True,
                format=FORMAT.GPTQ_P)
out["bits3"] = dict(qweight=list(m3.qweight.shape), qzeros=list(m3.qzeros.shape), kbits=m3.kbits, planar=bool(m3.planar))
out["bits5"] = dict(qweight=list(m5.qweight.shape), qzeros=list(m5.qzeros.shape), kbits=m5.kbits, planar=bool(m5.planar))


def signature(fn):
    return [[p.name, p.kind.name, None if p.default is inspect.Parameter.empty else repr(p.default)]
            for p in inspect.signature(fn).parameters.values()]


interface = {
    "signatures": {"BaseQuantLinear.__init__": signature(BaseQuantLinear.__init__),
                   "GPTQQuantLinear.__init__": signature(GPTQQuantLinear.__init__),
                   "BaseQuantLinear.validate": signature(BaseQuantLinear.validate)},
    "required_supports": {c.__name__: sorted(n for n, v in vars(c).items() if n.startswith("SUPPORTS") and v is None)
                          for c in (BaseQuantLinear, GroupedQuantLinear)},
}
with open(os.path.join(HERE, "shim_reference.json"), "w") as f:
    json.dump({"source": "ModelCloud/GPTQModel gptqmodel/nn_modules/qlinear/__init__.py, recorded by "
                         "tests/golden/check_shim.py", "interface": interface, "shim": out}, f, indent=1, sort_keys=True)
    f.write("\n")
print("wrote shim_reference.json")
