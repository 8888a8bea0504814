"""CUDA-graph replay of a fixed call sequence through the library's capture entry points
(irs_graph_begin / end / update_smoothing / launch, csrc/api.cu).

Whatever `enqueue()` submits to the current stream — staging copies and kernels of one iRS-LQR descent,
or of one (sample-sharded) linearization — is run eagerly twice (workspaces get allocated and warm),
captured on the third call of the same key and replayed from then on: one launch instead of ~8 API calls.
Before every replay the accumulate nodes are re-parameterised (seed, iteration, sigma).  Everything else a
captured kernel reads must be a function of the key or live in device memory (the epoch of the fused peer
exchange does).  IRS_CUDA_GRAPH=0 forces eager launches.
"""
import ctypes
import os

import torch

from . import _device, _lib

USE_GRAPHS = os.environ.get("IRS_CUDA_GRAPH", "1") != "0"


class GraphRunner:
    """lib: the library whose entry points the captured sequence calls (the accumulate node is looked up
    in that library's capture state)."""

    def __init__(self, lib=_lib.MAIN):
        self._lib = lib
        self._slots = {}

    def reset(self):
        for slot in self._slots.values():
            if slot[1] is not None:
                self._lib.call("irs_graph_destroy", slot[1])
        self._slots = {}

    def run(self, name, key, enqueue, update=None):
        """key None: the sequence cannot be replayed (run eagerly).  update(handle): re-parameterise the
        captured accumulate kernels before a replay."""
        if key is None or not USE_GRAPHS:
            enqueue()
            return
        key = (name,) + tuple(key)
        slot = self._slots.get(name)
        if slot is None or slot[0] != key:
            if slot is not None and slot[1] is not None:
                self._lib.call("irs_graph_destroy", slot[1])
            self._slots[name] = [key, None, 1]        # key, graph handle, eager calls so far
            enqueue()
            return
        if slot[1] is None:
            if slot[2] < 2:                           # let every workspace be allocated and warm first
                slot[2] += 1
                enqueue()
                return
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                self._lib.call("irs_graph_begin", side.cuda_stream)
                handle = ctypes.c_void_p()
                try:
                    enqueue()
                except BaseException:
                    # end the capture (a stream must not stay in capture mode), drop the partial graph and
                    # let the ORIGINAL exception propagate
                    try:
                        self._lib.call("irs_graph_end", side.cuda_stream, ctypes.byref(handle))
                        self._lib.call("irs_graph_destroy", handle)
                    except _lib.IrsCudaError:
                        pass
                    raise
                self._lib.call("irs_graph_end", side.cuda_stream, ctypes.byref(handle))
            slot[1] = handle
        if update is not None:
            update(slot[1])
        self._lib.call("irs_graph_launch", slot[1], _device.stream_ptr())
