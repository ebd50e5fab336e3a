"""The reference-side binding (gptqmodel_b200/reference_shim.py, INTEGRATION.md §2) constructs and is discoverable.

VERDICT r01 weak #9: the round-1 shim `class B200Linear(_Impl, GPTQQuantLinear)` raised TypeError because the kernel
class called a cooperative `super().__init__()` with no arguments.  Two checks:
  1. against a STAND-IN hierarchy that restates the reference's constructor signatures (qlinear/__init__.py:102-194,
     664-692, 727-760), its `validate()` plumbing (:257-332) and the discovery walk + priority ranking of
     utils/importer.py:110-127,182-233 — runs everywhere;
  2. against the UNMODIFIED reference classes, as recorded by tests/golden/check_shim.py in
     tests/golden/shim_reference.json: the stand-in must restate the recorded signatures, and the shim built on it must
     give the results the shim gave on the reference's own classes.
"""
import copy
import inspect
import json
import os
from typing import Optional

import pytest
import torch
import torch.nn as nn

from gptqmodel_b200.qlinear import B200KernelMixin, B200QuantLinear
from gptqmodel_b200.reference_shim import make_reference_kernel

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ---- stand-in for the reference's base classes: same constructor signatures, same validate() flow ------------------
class StandInBase(nn.Module):  # BaseQuantLinear, qlinear/__init__.py:73-194
    SUPPORTS_BACKENDS = None
    SUPPORTS_BACKEND_SELECTION = True
    SUPPORTS_METHODS = None
    SUPPORTS_FORMATS = None
    SUPPORTS_BITS = None
    SUPPORTS_SHARDS = None
    SUPPORTS_TRAINING = None
    SUPPORTS_AUTO_PADDING = None
    SUPPORTS_IN_FEATURES_DIVISIBLE_BY = None
    SUPPORTS_OUT_FEATURES_DIVISIBLE_BY = None
    SUPPORTS_PACK_DTYPES = None
    SUPPORTS_ADAPTERS = None
    SUPPORTS_DEVICES = None
    SUPPORTS_PLATFORM = None
    SUPPORTS_DTYPES = None
    REQUIRES_FORMAT_V2 = False
    post_init_calls = 0

    def __init__(self, bits: int, in_features: int, out_features: int, bias: bool, backend, adapter, name: str = None,
                 register_buffers: bool = False, register_buffers_in_features: int = None,
                 register_buffers_out_features: int = None, dtype: Optional[torch.dtype] = None,
                 validate_kwargs=None, **kwargs):
        super().__init__()
        self.name = name or f"{self.__class__.__module__}.{self.__class__.__qualname__}"
        self.in_features, self.out_features, self.bits, self.backend = in_features, out_features, bits, backend
        self.adapter = copy.deepcopy(adapter)
        args = {"bits": bits, "in_features": in_features, "out_features": out_features, "dtype": dtype, "adapter": adapter}
        if validate_kwargs:
            args.update(validate_kwargs)
        _, err = self.validate(**args)
        if err:
            raise err
        if register_buffers and bias:
            self.register_buffer("bias", torch.zeros(out_features, dtype=torch.float16))

    def post_init(self):
        type(self).post_init_calls += 1

    @classmethod
    def validate_once(cls):
        return True, None

    @classmethod
    def validate(cls, bits, group_size=-1, desc_act=False, sym=True, in_features=None, out_features=None,
                 pack_dtype=None, dtype=None, dynamic=None, device=None, trainable=None, adapter=None):
        ok, err = cls.validate_once()
        if not ok:
            return False, err
        # verify_supports_params (:300-332): every SUPPORTS_* that is None in the root must be set in the class's OWN dict
        missing = [n for n, v in StandInBase.__dict__.items()
                   if n.startswith("SUPPORTS") and v is None and n not in cls.__dict__]
        if missing:
            raise ValueError(f"{cls.__name__} these SUPPORTS variables are not overridden: {missing}")
        if adapter is not None and adapter.__class__ not in cls.SUPPORTS_ADAPTERS:
            return False, NotImplementedError("adapter")
        if pack_dtype not in cls.SUPPORTS_PACK_DTYPES:
            return False, NotImplementedError(f"pack_dtype {pack_dtype}")
        if dtype is not None and dtype not in cls.SUPPORTS_DTYPES:
            return False, NotImplementedError("dtype")
        if bits not in cls.SUPPORTS_BITS:
            return False, NotImplementedError("bits")
        if group_size not in cls.SUPPORTS_GROUP_SIZE:
            return False, NotImplementedError("group_size")
        if in_features is not None and any(in_features % d for d in cls.SUPPORTS_IN_FEATURES_DIVISIBLE_BY):
            return False, NotImplementedError("in_features")
        if out_features is not None and any(out_features % d for d in cls.SUPPORTS_OUT_FEATURES_DIVISIBLE_BY):
            return False, NotImplementedError("out_features")
        return True, None


class StandInGrouped(StandInBase):  # GroupedQuantLinear / PackedGroupedQuantLinear (:520-692)
    SUPPORTS_GROUP_SIZE = None
    SUPPORTS_DESC_ACT = None
    SUPPORTS_SYM = None

    def __init__(self, bits, group_size, desc_act, sym, in_features, out_features, bias, pack_dtype, backend, adapter,
                 **kwargs):
        super().__init__(bits=bits, in_features=in_features, out_features=out_features, bias=bias, backend=backend,
                         adapter=adapter, validate_kwargs={"group_size": group_size, "desc_act": desc_act, "sym": sym,
                                                           "pack_dtype": pack_dtype}, **kwargs)
        self.group_size = group_size if group_size != -1 else in_features
        self.desc_act, self.sym, self.pack_dtype = desc_act, sym, pack_dtype


class StandInGPTQ(StandInGrouped):  # GPTQQuantLinear (:727-760): all of these are REQUIRED positionally / by keyword
    def __init__(self, bits: int, group_size: int, desc_act: bool, sym: bool, in_features: int, out_features: int,
                 bias: bool, pack_dtype: torch.dtype, backend, adapter, name: str = None, register_buffers: bool = False,
                 register_buffers_in_features: int = None, register_buffers_out_features: int = None,
                 dtype: Optional[torch.dtype] = None, format=None, **kwargs):
        super().__init__(bits=bits, group_size=group_size, desc_act=desc_act, sym=sym, in_features=in_features,
                         out_features=out_features, bias=bias, pack_dtype=pack_dtype, backend=backend, adapter=adapter,
                         name=name, register_buffers=False, dtype=dtype, **kwargs)
        self.format = format
        self._qzeros_format = 1
        assert not register_buffers, "kernels that own their buffers pass register_buffers=False (swordfish.py:84-106)"


class OtherKernel(StandInGPTQ):  # a competing kernel with Swordfish's priority
    SUPPORTS_FORMATS = {"gptq": 101}
    SUPPORTS_BACKENDS = ["swordfish"]


def _discover(root):
    """utils/importer.py:110-127 + the priority sort of :182-233."""
    seen, kernels = set(), []

    def walk(cls):
        for sub in cls.__subclasses__():
            if sub in seen:
                continue
            seen.add(sub)
            walk(sub)
            if "SUPPORTS_FORMATS" in sub.__dict__ and getattr(sub, "SUPPORTS_BACKEND_SELECTION", True):
                kernels.append(sub)
    walk(root)
    return kernels


def _make():
    return make_reference_kernel(StandInGPTQ, backend="gptq_b200", methods=["gptq"], formats={"gptq": 120, "gptq_v2": 120},
                                 adapters=[], devices=["cuda"], platforms=["linux"])


def test_shim_constructs_on_the_reference_signature_and_is_discovered():
    cls = _make()
    cls.validate_once = classmethod(lambda c: (True, None))  # no GPU in the CPU suite
    assert [c.__name__ for c in cls.__mro__[:3]] == ["B200Linear", "B200KernelMixin", "StandInGPTQ"]
    # exactly the keyword set of create_quant_module (utils/model.py:630-647)
    m = cls(bits=4, group_size=128, desc_act=False, sym=True, in_features=256, out_features=128,
            pack_dtype=torch.int32, bias=True, dtype=torch.float16, name="model.layers.0.mlp.down_proj",
            lm_head_name="lm_head", backend="gptq_b200", register_buffers=True, adapter=None)
    assert isinstance(m, StandInGPTQ) and isinstance(m, B200KernelMixin) and not isinstance(m, B200QuantLinear)
    assert m.qweight.shape == (32, 128) and m.qzeros.shape == (2, 16) and m.scales.shape == (2, 128)
    assert m.g_idx.shape == (256,) and m.bias.shape == (128,)
    assert sorted(m.state_dict()) == ["bias", "g_idx", "qweight", "qzeros", "scales"]
    assert m.name == "model.layers.0.mlp.down_proj" and m.backend == "gptq_b200"
    assert m.qzero_format() == 1                     # the reference base's initial value survives the kernel setup
    m.convert_gptq_v1_to_v2()
    assert m.qzero_format() == 2 and int(m.qzeros[0, 0]) == 0x11111111
    assert len(m.list_buffers()) == 5
    # discovery + ranking: found by the __subclasses__ walk, wins FORMAT.GPTQ over the priority-101 kernel
    kernels = _discover(StandInBase)
    assert cls in kernels and OtherKernel in kernels
    ranked = sorted((k for k in kernels if "gptq" in k.SUPPORTS_FORMATS), key=lambda k: k.SUPPORTS_FORMATS["gptq"],
                    reverse=True)
    assert ranked[0] is cls
    # group_size -1 (per-channel) and no bias
    m2 = cls(bits=8, group_size=-1, desc_act=True, sym=False, in_features=128, out_features=64,
             pack_dtype=torch.int32, bias=False, backend="gptq_b200", adapter=None)
    assert m2.group_size == 128 and m2.qzeros.shape == (1, 16) and m2.bias is None


def test_shim_reports_unsupported_configs_as_not_implemented():
    cls = _make()
    cls.validate_once = classmethod(lambda c: (True, None))
    for bad in (dict(bits=16), dict(group_size=48), dict(in_features=100), dict(out_features=40),
                dict(pack_dtype=torch.int16)):
        kw = dict(bits=4, group_size=128, desc_act=False, sym=True, in_features=256, out_features=128,
                  pack_dtype=torch.int32, bias=False, backend="gptq_b200", adapter=None)
        kw.update(bad)
        with pytest.raises(NotImplementedError):   # "try the next kernel" (utils/model.py:703-707)
            cls(**kw)
    # without a CUDA device the environment check answers (False, NotImplementedError), it never raises
    fresh = _make()
    if not torch.cuda.is_available():
        ok, err = fresh.validate_once()
        assert not ok and isinstance(err, NotImplementedError)
        with pytest.raises(NotImplementedError):
            fresh(bits=4, group_size=128, desc_act=False, sym=True, in_features=256, out_features=128,
                  pack_dtype=torch.int32, bias=False, backend="gptq_b200", adapter=None)


def test_standalone_class_still_has_the_whole_contract():
    for name in ("post_init", "forward", "dequantize_weight", "list_buffers", "pack_block", "qzero_format",
                 "convert_gptq_v1_to_v2", "from_checkpoint_tensors", "validate", "validate_once", "validate_device"):
        assert hasattr(B200QuantLinear, name), name
    m = B200QuantLinear(bits=4, group_size=64, desc_act=False, sym=True, in_features=128, out_features=64, bias=True)
    assert m.qzero_format() == 2 and m.qzeros.shape == (2, 8)


def _signature(fn):
    return [[p.name, p.kind.name, None if p.default is inspect.Parameter.empty else repr(p.default)]
            for p in inspect.signature(fn).parameters.values()]


def _probe(cls, monkeypatch):
    """tests/golden/check_shim.py's checks, on `cls` built over the stand-in hierarchy."""
    out = {"mro": [c.__name__ for c in cls.__mro__][:6]}
    kernels = _discover(StandInBase)
    out["discovered"] = cls in kernels
    ranked = sorted((k for k in kernels if "gptq" in (k.SUPPORTS_FORMATS or {})), key=lambda k: k.SUPPORTS_FORMATS["gptq"],
                    reverse=True)
    out["top_for_gptq"] = ranked[0].__name__ if ranked else None
    with monkeypatch.context() as mp:  # the reference run had no CUDA device
        mp.setattr(torch.cuda, "is_available", lambda: False)
        ok, err = cls.validate(bits=4, group_size=128, desc_act=False, sym=True, in_features=256, out_features=128,
                               pack_dtype=torch.int32, dtype=torch.float16)
    out["validate_without_gpu"] = [ok, type(err).__name__ if err else None]
    cls.validate_once = classmethod(lambda c: (True, None))
    out["verify_supports_params"] = cls.validate(bits=4, pack_dtype=torch.int32) == (True, None)  # raises on a missing SUPPORTS_*
    m = cls(bits=4, group_size=128, desc_act=False, sym=True, in_features=256, out_features=128, pack_dtype=torch.int32,
            bias=True, dtype=torch.float16, name="model.layers.0.self_attn.q_proj", lm_head_name="lm_head",
            backend="gptq_b200", register_buffers=True, adapter=None)
    out["constructed"] = True
    out["shapes"] = {k: list(getattr(m, k).shape) for k in ("qweight", "qzeros", "scales", "g_idx", "bias")}
    out["qzeros_format_initial"] = m.qzero_format()
    out["isinstance_base"] = isinstance(m, StandInGPTQ) and isinstance(m, StandInBase)
    out["state_dict_keys"] = sorted(m.state_dict().keys())
    out["name"] = m.name
    out["n_list_buffers"] = len(m.list_buffers())
    try:
        cls(bits=16, group_size=128, desc_act=False, sym=True, in_features=256, out_features=128, pack_dtype=torch.int32,
            bias=False, backend="gptq_b200", adapter=None)
        out["bits16"] = None
    except Exception as e:  # noqa: BLE001
        out["bits16"] = type(e).__name__
    m3 = cls(bits=3, group_size=128, desc_act=False, sym=True, in_features=256, out_features=128, pack_dtype=torch.int32,
             bias=False, backend="gptq_b200", adapter=None, register_buffers=True)
    m5 = cls(bits=5, group_size=64, desc_act=False, sym=False, in_features=256, out_features=128, pack_dtype=torch.int32,
             bias=False, backend="gptq_b200", adapter=None, register_buffers=True, format="gptq_p")
    out["bits3"] = dict(qweight=list(m3.qweight.shape), qzeros=list(m3.qzeros.shape), kbits=m3.kbits, planar=bool(m3.planar))
    out["bits5"] = dict(qweight=list(m5.qweight.shape), qzeros=list(m5.qzeros.shape), kbits=m5.kbits, planar=bool(m5.planar))
    return out


def test_shim_against_the_unmodified_reference_classes(monkeypatch):
    with open(os.path.join(ROOT, "tests", "golden", "shim_reference.json")) as f:
        golden = json.load(f)
    # the stand-in still restates the reference's interface
    sigs = golden["interface"]["signatures"]
    assert _signature(StandInBase.__init__) == sigs["BaseQuantLinear.__init__"]
    assert _signature(StandInGPTQ.__init__) == sigs["GPTQQuantLinear.__init__"]
    assert _signature(StandInBase.validate) == sigs["BaseQuantLinear.validate"]
    required = golden["interface"]["required_supports"]
    for stand_in, name in ((StandInBase, "BaseQuantLinear"), (StandInGrouped, "GroupedQuantLinear")):
        assert sorted(n for n, v in vars(stand_in).items() if n.startswith("SUPPORTS") and v is None) == required[name]
    # what the shim did on the reference's own classes
    out = golden["shim"]
    assert out["mro"][:3] == ["B200Linear", "B200KernelMixin", "GPTQQuantLinear"]
    assert out["verify_supports_params"] and out["discovered"] and out["constructed"] and out["isinstance_base"]
    assert out["top_for_gptq"] == "B200Linear"
    assert out["validate_without_gpu"] == [False, "NotImplementedError"]
    assert out["shapes"] == {"qweight": [32, 128], "qzeros": [2, 16], "scales": [2, 128], "g_idx": [256], "bias": [128]}
    assert out["qzeros_format_initial"] == 1 and out["bits16"] == "NotImplementedError"
    assert out["bits3"] == dict(qweight=[24, 128], qzeros=[2, 12], kbits=4, planar=False)
    assert out["bits5"] == dict(qweight=[40, 128], qzeros=[4, 20], kbits=8, planar=True)
    assert out["state_dict_keys"] == ["bias", "g_idx", "qweight", "qzeros", "scales"]
    # ... and the same shim over the stand-in does the same
    got = _probe(_make(), monkeypatch)
    assert got["mro"][:3] == ["B200Linear", "B200KernelMixin", "StandInGPTQ"]
    assert {k: v for k, v in got.items() if k != "mro"} == {k: v for k, v in out.items() if k != "mro"}
