"""Executor + execution state stack: runs the lowered units and makes BPTT over snapshots work.

Semantics kept from ``stgraph/compiler/executor.py:29-106,187-445`` (STGraph's contribution over
Seastar; SURVEY.md section 2 #8, section 5 "sequence length"):

* per call: bind inputs (``restart``), run the forward units; every group of consecutive
  compiled units is ONE ``torch.autograd.Function`` application
  (``KernelWrapperTorch.apply(executor, uid, kernel_args, rets, *tensors)``, ``executor.py:328-346``);
* ``forward_cb`` launches the kernels, then pushes on a LIFO stack **only the tensors some
  backward unit reads** plus the graph's current timestamp (``executor.py:348-367``) -- not a copy
  of the graph;
* ``backward_cb`` reads the top of the stack, asks a ``DynamicGraph`` to rewind to that timestamp
  (``executor.py:385-387`` -> ``dynamic_graph.py:110-128``), allocates gradients, launches the
  backward units, pops (``executor.py:369-426``).

What changed: launches go through the C ABI on torch's current stream (the reference packs
ctypes pointers for ``cuLaunchKernel`` on the NULL stream, ``execution_unit.py:359-372``); outputs
that a kernel overwrites completely are allocated uninitialised instead of zero-filled.
"""
from __future__ import annotations

import ctypes
from collections import deque

import torch

from .. import _lib, kernels
from .lowering import lower_unit
from .registry import torch_eval
from .utils import ValType, is_const_scalar


class Stack:
    def __init__(self):
        self.content = deque()

    def push(self, val):
        self.content.append(val)

    def pop(self):
        self.content.pop()

    def top(self):
        return self.content[-1]

    def __len__(self):
        return len(self.content)


class ExeState:
    """Tensors of the call in flight + the LIFO stacks that outlive it until backward."""

    def __init__(self):
        self.tensor_map_stack = Stack()       # one dict {var id: tensor} per forward call, for backward
        self.graph_timestamp_stack = Stack()  # timestamp of the snapshot each forward call ran on
        self.current_tensor_map = {}

    def reset(self, input_map):
        self.current_tensor_map = dict(input_map)

    def track_tensor(self, key, val):
        self.current_tensor_map[key] = val

    def clear_current_tensor_state(self):
        self.current_tensor_map = {}


class MergedUnit:
    """Consecutive units of the same kind (``executor.py:109-185``)."""

    def __init__(self, units):
        self.units = list(units)

    def compiled(self):
        return self.units[-1].compiled

    def joint_inputs(self):
        produced = set()
        for u in self.units:
            produced |= u.tmps
        out = []
        for u in self.units:
            for a in u.unit_args():
                if a not in produced and a not in out:
                    out.append(a)
        return out

    def joint_rets(self):
        out = []
        for u in self.units:
            for r in u.unit_rets():
                if r not in out:
                    out.append(r)
        return out

    def __iter__(self):
        return iter(self.units)


def _is_dynamic(graph):
    return hasattr(graph, "get_backward_graph") and hasattr(graph, "current_timestamp")


class Executor:
    def __init__(self, graph, forward_exec_units, backward_exec_units, grad_in, grad_out, rets):
        self.forward_exec_units = self.merge_units(forward_exec_units)
        self.bulist = list(backward_exec_units)
        self.grad_in = grad_in            # forward output Var -> Var of its incoming gradient
        self.grad_out = grad_out          # forward input Var  -> Var of the gradient to return
        self._rets = list(rets)
        self.ts = ExeState()
        self.new_zeros = None
        self.new_empty = None
        self.raw_ptr = None
        self.graph = graph
        self.num_nodes = graph.get_num_nodes()
        self.num_edges = graph.get_num_edges()
        for mu in self.forward_exec_units:
            for u in mu:
                if u.compiled:
                    lower_unit(u)
        for u in self.bulist:
            if u.compiled:
                lower_unit(u)
        # forward tensors the backward units read: saved on the state stack, nothing else is kept
        bwd_produced = set()
        for u in self.bulist:
            bwd_produced |= u.tmps
        grad_in_vars = set(self.grad_in.values())
        self.saved_for_backward = []
        for u in self.bulist:
            for a in u.unit_args():
                if a not in bwd_produced and a not in grad_in_vars and a.id not in self.saved_for_backward:
                    self.saved_for_backward.append(a.id)

    @staticmethod
    def merge_units(units):
        assert len(units) > 0, "empty execution unit list"
        grouped = [MergedUnit([units[0]])]
        for u in units[1:]:
            if u.compiled == grouped[-1].compiled():
                grouped[-1].units.append(u)
            else:
                grouped.append(MergedUnit([u]))
        return grouped

    # -- callbacks installed by the backend (backend/callback.py) ---------------------
    def set_raw_ptr_cb(self, cb):
        self.raw_ptr = cb

    def set_new_zeros_cb(self, cb):
        self.new_zeros = cb

    def set_new_empty_cb(self, cb):
        self.new_empty = cb

    def restart(self, input_map, graph=None):
        self.ts.reset(input_map)
        if graph is not None:
            self.graph = graph
            self.num_nodes = graph.get_num_nodes()
            self.num_edges = graph.get_num_edges()

    # -- forward ----------------------------------------------------------------------
    def execute(self, FuncWrapper):
        for uid, mu in enumerate(self.forward_exec_units):
            if mu.compiled():
                self.execute_compiled(uid, FuncWrapper)
            else:
                self.execute_prog(mu.units, self.ts.current_tensor_map)
        ret = tuple(self.ts.current_tensor_map[r.id] for r in self._rets)
        self.ts.clear_current_tensor_state()
        return ret

    def _alloc(self, var, zero, like_map, dtype=None):
        lead = self.num_edges if var.is_edgevar() else self.num_nodes
        size = [lead] + list(var.var_shape)
        fn = self.new_zeros if (zero or self.new_empty is None) else self.new_empty
        dev = var.device
        if dev is None or (isinstance(dev, torch.device) and dev.type != "cuda"):
            dev = next(iter(like_map.values())).device
        return fn(size=size, dtype=var.var_dtype if dtype is None else dtype, device=dev, requires_grad=False)

    def _alloc_unit_outputs(self, unit, tensor_map):
        needs_zero = set()
        written = set()
        for la in unit.launches:
            needs_zero |= la.needs_zero
            written |= set(la.writes)
            # A scaled sum over bf16 / fp16 rows writes rows of that type.  The traced program cannot say so: it types
            # ``h * norm`` by promotion (fp32) and a gradient by its first operand, so the output takes x's dtype here.
            if la.kind == "scaled_sum" and la.out.id not in tensor_map:
                x = tensor_map.get(la.x.id)
                if x is not None and x.dtype in kernels.H16_DTYPES:
                    tensor_map[la.out.id] = self._alloc(la.out, False, tensor_map, dtype=x.dtype)
        for var in unit.unit_rets():
            if var.id not in tensor_map:
                tensor_map[var.id] = self._alloc(var, var in needs_zero or var not in written, tensor_map)

    def execute_compiled(self, uid, FuncWrapper):
        mu = self.forward_exec_units[uid]
        inputs = mu.joint_inputs()
        rets = mu.joint_rets()
        for unit in mu:
            self._alloc_unit_outputs(unit, self.ts.current_tensor_map)
        kernel_arg_list = [[v.id for v in u.kernel_args()] for u in mu]
        in_tensors = [self.ts.current_tensor_map[v.id] for v in inputs]
        # The state stacks are popped by backward_cb only: push when a backward can follow (the reference pushes on
        # every call, executor.py:377-380, so inference / validation loops grow its stacks without bound).
        self._will_backward = torch.is_grad_enabled() and any(isinstance(t, torch.Tensor) and t.requires_grad
                                                              for t in in_tensors)
        ret_tensors = FuncWrapper.apply(self, uid, kernel_arg_list, rets, *in_tensors)
        # only tensors returned by the Function carry grad_fn: re-track them (executor.py:343-346)
        for var, t in zip(rets, ret_tensors):
            self.ts.track_tensor(var.id, t)

    def run_launch(self, la, tensor_map, graph):
        view = graph.fwd_view() if la.center == ValType.DEST else graph.bwd_view()
        if la.kind == "scaled_sum":
            get = lambda v: None if v is None else tensor_map[v.id].detach()
            flat = lambda t: None if t is None else t.reshape(-1)
            csr = graph._forward_graph if la.center == ValType.DEST else graph._backward_graph
            if getattr(csr, "pack_enabled", False):     # static graph: packed {col, scale} array, built on first use
                kernels.agg_scaled_sum_graph(csr, get(la.x), flat(get(la.ns)), flat(get(la.es)), flat(get(la.rs)),
                                             out=tensor_map[la.out.id])
            else:
                kernels.agg_scaled_sum(view, get(la.x), flat(get(la.ns)), flat(get(la.es)), flat(get(la.rs)),
                                       out=tensor_map[la.out.id])
            return
        ptrs = (ctypes.c_void_p * _lib.VM_MAX_TENSORS)()
        for i, v in enumerate(la.tensor_vars):
            t = tensor_map[v.id]
            if not t.is_contiguous():
                t = t.contiguous()
                tensor_map[v.id] = t
            if t.dtype != torch.float32:
                raise TypeError(f"vertex-program tensors must be float32 (got {t.dtype} for {v.id})")
            ptrs[i] = self.raw_ptr(t) if self.raw_ptr is not None else ctypes.c_void_p(t.data_ptr())
        _lib.call("stg_vm_run_f32", ctypes.byref(view), ctypes.byref(la.program), ptrs, _lib.current_stream_ptr())
        kernels.launch_count += 1

    def forward_cb(self, uid, kernel_args, rets, tensor_list):
        """Called by ``KernelWrapper.forward``: launch, then save what backward needs + the timestamp."""
        mu = self.forward_exec_units[uid]
        tm = self.ts.current_tensor_map
        for unit in mu:
            for la in unit.launches:
                self.run_launch(la, tm, self.graph)
        if getattr(self, "_will_backward", True):
            self.ts.tensor_map_stack.push({k: tm[k] for k in self.saved_for_backward if k in tm})
            if _is_dynamic(self.graph):
                self.ts.graph_timestamp_stack.push(self.graph.current_timestamp)
        return tuple(tm[r.id] for r in rets)

    # -- backward ---------------------------------------------------------------------
    def backward_cb(self, kid, grad_list):
        """Called by ``KernelWrapper.backward`` with one gradient (or None) per forward ret."""
        mu = self.forward_exec_units[kid]
        inputs = mu.joint_inputs()
        rets = mu.joint_rets()
        tensor_map = dict(self.ts.tensor_map_stack.top())
        if _is_dynamic(self.graph):
            self.graph.get_backward_graph(self.ts.graph_timestamp_stack.top())
        self.num_nodes = self.graph.get_num_nodes()
        self.num_edges = self.graph.get_num_edges()
        for var, g in zip(rets, grad_list):
            gv = self.grad_in.get(var)
            if gv is None:
                continue
            if g is None:
                g = self._alloc(gv, True, tensor_map)
            elif not g.is_contiguous():
                g = g.contiguous()
            tensor_map[gv.id] = g
        for bu in self.bulist:
            if bu.compiled:
                self._alloc_unit_outputs(bu, tensor_map)
                for la in bu.launches:
                    self.run_launch(la, tensor_map, self.graph)
            else:
                self.execute_prog([bu], tensor_map)
        out = []
        for v in inputs:
            g = self.grad_out.get(v)
            out.append(tensor_map[g.id] if g is not None and g.id in tensor_map else None)
        self.ts.tensor_map_stack.pop()
        if _is_dynamic(self.graph):
            self.ts.graph_timestamp_stack.pop()
        return tuple(out)

    def execute_prog(self, units, tensor_map):
        """Uncompiled (node-wise) units run statement by statement through torch (``executor.py:428-445``)."""
        for unit in units:
            for stmt in unit.program:
                args = [tensor_map[a.id] if not is_const_scalar(a) else a for a in stmt.args]
                tensor_map[stmt.ret.id] = torch_eval(stmt, args)
