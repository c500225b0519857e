"""CUDA-graph plumbing for the hot path: capture a step with torch, then instantiate it so that every kernel node
keeps its own launch priority (cudaGraphInstantiateFlagUseNodePriority).

Why: one training step has two independent branches -- the patchifier (FPS -> kNN/Group, latency-bound, small) and
the loss (Chamfer forward/backward, FMA-bound, fills every SM for two waves and leaves ~13 % of the SM-time idle in
its last wave).  With equal priorities the block scheduler interleaves the branches and the step costs the SUM of
the kernels; with the loss branch at high priority the patchifier's CTAs are dispatched only when no Chamfer CTA is
waiting, i.e. into the holes of the last wave.  torch.cuda.CUDAGraph instantiates with flags=0 (node priorities
ignored), so the captured graph is re-instantiated here through the CUDA driver API (cuda-python).

Plumbing only: no computation happens in this module.
"""
import torch


def _check(res):
    err = res[0]
    if int(err) != 0:
        raise RuntimeError("CUDA driver call failed: %s" % (err,))
    return res[1] if len(res) == 2 else res[1:]


class PriorityGraph:
    """with g.capture(): <enqueue the step>   ...   g.replay()

    `low_priority` lists substrings of kernel names that go to the lowest launch priority; every other kernel node
    gets the highest.  Memset / memcpy nodes have no priority."""

    def __init__(self, low_priority=("fps_", "knn_", "gather_")):
        self.low = tuple(low_priority)
        self.graph = torch.cuda.CUDAGraph(keep_graph=True)
        self.exec = None
        self.assigned = {}

    def capture(self, **kw):
        return torch.cuda.graph(self.graph, **kw)

    def instantiate(self):
        from cuda.bindings import driver as drv

        _check(drv.cuInit(0))
        raw = drv.CUgraph(int(self.graph.raw_cuda_graph()))
        _, n = _check(drv.cuGraphGetNodes(raw, 0))
        nodes, n = _check(drv.cuGraphGetNodes(raw, n))
        lo, hi = _check(drv.cuCtxGetStreamPriorityRange())  # (least, greatest): numerically lower = more urgent
        for node in nodes[:n]:
            if _check(drv.cuGraphNodeGetType(node)) != drv.CUgraphNodeType.CU_GRAPH_NODE_TYPE_KERNEL:
                continue
            params = _check(drv.cuGraphKernelNodeGetParams(node))
            name = _check(drv.cuFuncGetName(params.func))
            name = name.decode() if isinstance(name, bytes) else str(name)
            prio = lo if any(s in name for s in self.low) else hi
            val = drv.CUkernelNodeAttrValue()
            val.priority = prio
            _check(drv.cuGraphKernelNodeSetAttribute(node, drv.CUlaunchAttributeID.CU_LAUNCH_ATTRIBUTE_PRIORITY, val))
            self.assigned[name] = prio
        flags = drv.CUgraphInstantiate_flags.CUDA_GRAPH_INSTANTIATE_FLAG_USE_NODE_PRIORITY
        self.exec = _check(drv.cuGraphInstantiate(raw, int(flags)))
        self._launch, self._stream_t = drv.cuGraphLaunch, drv.CUstream
        return self

    def replay(self):
        if self.exec is None:
            self.instantiate()
        err, = self._launch(self.exec, self._stream_t(torch.cuda.current_stream().cuda_stream))
        if int(err) != 0:
            raise RuntimeError("cuGraphLaunch failed: %s" % (err,))
