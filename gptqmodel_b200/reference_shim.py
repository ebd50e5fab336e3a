"""Reference-side binding: build the QuantLinear class a maintainer registers inside ModelCloud/GPTQModel.

The reference discovers kernels by walking `BaseQuantLinear.__subclasses__()` for classes that define `SUPPORTS_FORMATS`
in their own `__dict__` (gptqmodel/utils/importer.py:110-127), ranks them by the integer priority in `SUPPORTS_FORMATS`
(:182-233) and instantiates the winner with the keyword arguments of `create_quant_module`
(gptqmodel/utils/model.py:630-647) — which go through `GPTQQuantLinear.__init__` (qlinear/__init__.py:727-760:
`bits, group_size, desc_act, sym, in_features, out_features, bias, pack_dtype, backend, adapter, name, register_buffers,
..., dtype, format, **kwargs`), `PackedGroupedQuantLinear`, `GroupedQuantLinear` and `BaseQuantLinear.__init__`
(:102-194: deep-copies the adapter, runs `cls.validate(...)`).

`make_reference_kernel(GPTQQuantLinear, ...)` returns `class B200Linear(B200KernelMixin, GPTQQuantLinear)`:
  * `__init__` initialises the REFERENCE base explicitly with every argument it requires (no cooperative
    `super().__init__()` from the kernel mixin — the round-1 shim raised TypeError exactly there) and then calls
    `B200KernelMixin._b200_setup` for the kernel-side state and the checkpoint-shaped Parameters;
  * `validate()` / `_validate()` stay the reference's own (they read the `SUPPORTS_*` lists, which therefore hold the
    reference's enum members), `validate_once()` adds the device / library check;
  * `post_init()` / `forward()` / `dequantize_weight()` / `list_buffers()` come from the mixin; `post_init()` ends in the
    base's `post_init()` (adapter initialisation, qlinear/__init__.py:224-234).
The file a maintainer adds is shown in INTEGRATION.md §2; tests/test_reference_shim.py builds the class against a
stand-in hierarchy with the reference's exact constructor signatures and compares it with what the same class did on the
unmodified reference classes (recorded in tests/golden/shim_reference.json).
"""
from __future__ import annotations

from typing import Optional, Tuple

import torch

from .qlinear import B200KernelMixin


def make_reference_kernel(base_cls, *, backend, methods, formats, adapters, devices, platforms,
                          class_name: str = "B200Linear", quant_type: str = "b200"):
    """base_cls: the reference's `GPTQQuantLinear`; the other arguments are the reference's enum members, e.g.
    backend=BACKEND.GPTQ_B200, methods=[METHOD.GPTQ], formats={FORMAT.GPTQ: 110, FORMAT.GPTQ_V2: 110},
    adapters=[Lora], devices=[DEVICE.CUDA], platforms=[PLATFORM.LINUX]."""

    class _B200Linear(B200KernelMixin, base_cls):
        SUPPORTS_BACKENDS = [backend]
        SUPPORTS_METHODS = list(methods)
        SUPPORTS_FORMATS = dict(formats)   # > Swordfish 101 / Machete 100 / Marlin 90 wins auto-selection on CUDA
        SUPPORTS_BITS = [2, 3, 4, 5, 6, 7, 8]  # 2 / 3 and planar 5 / 6 / 7 are widened exactly to 4 / 8-bit fields (layouts.py)
        SUPPORTS_GROUP_SIZE = [-1, 32, 64, 128]
        SUPPORTS_DESC_ACT = [True, False]
        SUPPORTS_SYM = [True, False]
        SUPPORTS_SHARDS = True
        SUPPORTS_TRAINING = False
        SUPPORTS_AUTO_PADDING = False
        SUPPORTS_IN_FEATURES_DIVISIBLE_BY = [64]
        SUPPORTS_OUT_FEATURES_DIVISIBLE_BY = [32]
        SUPPORTS_PACK_DTYPES = [torch.int32]
        SUPPORTS_ADAPTERS = list(adapters)
        SUPPORTS_DEVICES = list(devices)
        SUPPORTS_PLATFORM = list(platforms)
        SUPPORTS_DTYPES = [torch.float16, torch.bfloat16]
        REQUIRES_FORMAT_V2 = True
        QUANT_TYPE = quant_type

        def __init__(self, bits: int, group_size: int, desc_act: bool, sym: bool, in_features: int, out_features: int,
                     bias: bool = False, pack_dtype: torch.dtype = torch.int32, adapter=None,
                     register_buffers: bool = True, **kwargs):
            kwargs.setdefault("backend", backend)
            # the reference base: nn.Module.__init__, adapter deep copy, validate(), bookkeeping attributes; it must NOT
            # register its own buffers (Marlin / Swordfish pass register_buffers=False the same way, swordfish.py:84-106)
            base_cls.__init__(self, bits=bits, group_size=group_size, desc_act=desc_act, sym=sym,
                              in_features=in_features, out_features=out_features, bias=bias, pack_dtype=pack_dtype,
                              adapter=adapter, register_buffers=False, **kwargs)
            self._b200_setup(bits, group_size, desc_act, sym, in_features, out_features, bias=bias,
                             pack_dtype=pack_dtype, adapter=adapter, register_buffers=register_buffers,
                             name=kwargs.get("name"), dtype=kwargs.get("dtype"), format=kwargs.get("format"))

        @classmethod
        def validate_once(cls) -> Tuple[bool, Optional[Exception]]:
            if not torch.cuda.is_available():
                return False, NotImplementedError(f"{cls.__name__} needs a CUDA device")
            major, minor = torch.cuda.get_device_capability()
            if major != 10:
                return False, NotImplementedError(f"{cls.__name__} is built for sm_100a only, found sm_{major}{minor}")
            return True, None

    _B200Linear.__name__ = _B200Linear.__qualname__ = class_name
    return _B200Linear
