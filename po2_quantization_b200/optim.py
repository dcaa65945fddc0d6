"""The parameter update of the QAT step (reference train.py:54-56 ``optim.SGD(model.parameters(), lr, momentum,
weight_decay)``, train.py:92 ``optimizer.step()``) as ONE launch per 96 parameter tensors.

``SGD`` is a ``torch.optim.SGD`` subclass: same constructor, ``param_groups``, ``state`` (``momentum_buffer``),
``state_dict`` and LR-scheduler behaviour; only ``step()`` differs for parameters that are fp32 CUDA tensors --
torch's foreach path issues 14 launches for ResNet-56's 171 parameters, ``po2_sgd_step`` two, with the same
roundings (bit-identical parameters, tests/test_models_gpu.py).  Everything else (CPU tensors, other dtypes,
Nesterov, dampening, maximize, sparse gradients, tensors of 2^31 or more elements) is handed to
``torch.optim.SGD.step``.  CUDA-graph capturable like the
stock optimizer with a float ``lr`` (the value is baked into the captured launch)."""
import ctypes

import torch

from . import _lib, ops


SGD_MAX_NUMEL = 2**31 - 1     # po2_sgd_step indexes a tensor in 32 bits and refuses larger ones (PO2_E_SIZE)


class SGD(torch.optim.SGD):
    @torch.no_grad()
    def step(self, closure=None):
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        rest = []
        for group in self.param_groups:
            ours = (group["dampening"] == 0 and not group["nesterov"] and not group["maximize"]
                    and not isinstance(group["lr"], torch.Tensor))
            todo = {}
            for p in group["params"]:
                g = p.grad
                if g is None:
                    continue
                taken = (ours and p.is_cuda and p.dtype == torch.float32 and g.dtype == torch.float32 and not g.is_sparse
                         and p.is_contiguous() and g.is_contiguous() and g.device == p.device)
                if not (taken and p.numel() <= SGD_MAX_NUMEL):
                    if taken:                     # the size is the only reason: a kernel-eligible tensor leaves it
                        ops.note_library_path("sgd:size", f"optim.SGD hands a parameter of {p.numel()} elements to "
                                              "torch.optim.SGD.step (po2_sgd_step takes up to 2^31 - 1)")
                    rest.append(p)
                    continue
                first = "momentum_buffer" not in self.state[p] or self.state[p]["momentum_buffer"] is None
                todo.setdefault((p.device, first), []).append(p)
            for (dev, first), ps in todo.items():
                mom = float(group["momentum"])
                if mom != 0.0 and first:
                    for p in ps:
                        self.state[p]["momentum_buffer"] = torch.empty_like(p.grad, memory_format=torch.contiguous_format)
                n = len(ps)
                arr = ctypes.c_void_p * n
                pp = arr(*[p.data_ptr() for p in ps])
                gg = arr(*[p.grad.data_ptr() for p in ps])
                bb = arr(*[self.state[p]["momentum_buffer"].data_ptr() for p in ps]) if mom != 0.0 else None
                nn_ = (ctypes.c_longlong * n)(*[p.numel() for p in ps])
                lib = _lib.load()
                per = int(lib.po2_sgd_max_tensors_per_launch())
                with torch.cuda.device(dev):
                    ops.LAUNCHES += (n + per - 1) // per
                    _lib.check(lib.po2_sgd_step(pp, gg, bb, nn_, n, float(group["lr"]), mom, float(group["weight_decay"]),
                                                int(first), ops._stream_ptr(dev)), "po2_sgd_step")
                # the kernel wrote through raw pointers: tell autograd (and everything keyed on Tensor._version, like
                # the weight prefetch that re-quantizes only changed weights) that these tensors changed in place
                torch.autograd.graph.increment_version(ps)
                if mom != 0.0:
                    torch.autograd.graph.increment_version([self.state[p]["momentum_buffer"] for p in ps])
        if rest:
            # hand what the kernel does not take to the stock implementation: hide the gradients that are done
            keep = set(id(p) for p in rest)
            hidden = []
            for group in self.param_groups:
                for p in group["params"]:
                    if p.grad is not None and id(p) not in keep:
                        hidden.append((p, p.grad))
                        p.grad = None
            try:
                super().step()
            finally:
                for p, g in hidden:
                    p.grad = g
        return loss
