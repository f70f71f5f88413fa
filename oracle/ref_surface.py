"""Recorded attribute surface of mbrl-lib objects, so that tests can check the duck-typed boundary without mbrl-lib.

``record`` (run by ``oracle/gen_golden.py`` on the imported reference) walks an object -- an ``nn.Module`` tree, a
plain object, a callable -- and keeps what the object *exposes*: class names, public attributes with plain values,
parameter / buffer / tensor shapes and dtypes, child modules in order, a callable's module and name.  ``rebuild``
turns such a record back into an object that has exactly those attributes and nothing else: classes of the recorded
names, zero tensors of the recorded shapes (on the device asked for), indexable / iterable ``nn.Sequential``
stand-ins, and functions carrying the recorded ``__module__`` / ``__name__``.  Code that reads the rebuilt object
reads the same attribute paths it would read on the real one; an attribute the real object lacks is missing here too.
"""
from __future__ import annotations

import types

import torch

_PLAIN = (bool, int, float, str, type(None))


def _tensor(t):
    return {"tensor": list(t.shape), "dtype": str(t.dtype).replace("torch.", "")}


def record(obj):
    if isinstance(obj, torch.Tensor):
        return _tensor(obj)
    if isinstance(obj, _PLAIN):
        return obj
    if isinstance(obj, torch.device):
        return {"device": str(obj)}
    if isinstance(obj, (list, tuple)):
        return {"list": [record(v) for v in obj]}
    cls = type(obj)
    if isinstance(obj, (types.FunctionType, types.BuiltinFunctionType, types.MethodType)):
        return {"callable": obj.__name__, "module": obj.__module__ or ""}
    out = {"class": cls.__name__, "class_module": cls.__module__, "attrs": {}}
    if isinstance(obj, torch.nn.Module):
        out["sequence"] = isinstance(obj, torch.nn.Sequential)
        for k, v in vars(obj).items():
            if not k.startswith("_"):
                out["attrs"][k] = record(v)
        for group in (obj._parameters, obj._buffers, obj._modules):
            for k, v in group.items():
                out["attrs"][k] = None if v is None else record(v)
    else:
        for k, v in vars(obj).items():
            if not k.startswith("_"):
                out["attrs"][k] = record(v)
    return out


def _stand_in_function(name, module):
    def fn(*args, **kwargs):
        raise RuntimeError(f"stand-in for {module}.{name}: only its identity was recorded")

    fn.__name__ = fn.__qualname__ = name
    fn.__module__ = module
    return fn


def rebuild(rec, device="cpu"):
    if isinstance(rec, _PLAIN):
        return rec
    if "tensor" in rec:
        return torch.zeros(rec["tensor"], dtype=getattr(torch, rec["dtype"]), device=device)
    if "device" in rec:
        return torch.device(device)
    if "list" in rec:
        return [rebuild(v, device) for v in rec["list"]]
    if "callable" in rec:
        return _stand_in_function(rec["callable"], rec["module"])
    ns = {"__module__": rec["class_module"]}
    if rec.get("sequence"):
        ns["__getitem__"] = lambda self, i: list(self._children)[i]
        ns["__iter__"] = lambda self: iter(self._children)
        ns["__len__"] = lambda self: len(self._children)
    obj = type(rec["class"], (), ns)()
    for k, v in rec["attrs"].items():
        setattr(obj, k, rebuild(v, device))
    if rec.get("sequence"):  # nn.Sequential names its children "0", "1", ...
        obj._children = [getattr(obj, k) for k in sorted((k for k in rec["attrs"] if k.isdigit()), key=int)]
    return obj
