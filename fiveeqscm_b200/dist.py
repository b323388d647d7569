"""Multi-GPU plumbing: shard the member axis, reduce the summary statistics (SURVEY.md 8e).

Members are independent, so ranks never exchange data during the integration.  The only
collective is at the end: integer histogram counts are summed (bitwise independent of the GPU
count), moment sums are summed, and min/max are reduced with MAX over [max, -min].
Works over any torch.distributed backend (nccl on the B200 box, gloo in the CPU tests).
"""
from __future__ import annotations

import math


def shard_bounds(n_member: int, world_size: int, rank: int, align: int = 128):
    """Contiguous member block of `rank`: [lo, hi).  Block edges are multiples of `align`
    (a CTA's worth of members) except the last one, so no rank runs a ragged CTA but the last."""
    if world_size < 1 or not (0 <= rank < world_size):
        raise ValueError("bad rank / world_size")
    blocks = (n_member + align - 1) // align
    lo_b = (blocks * rank) // world_size
    hi_b = (blocks * (rank + 1)) // world_size
    return min(lo_b * align, n_member), min(hi_b * align, n_member)


def allreduce_stats(hist, moments, group=None):
    """In-place all-reduce of (hist int64 [..., n_t][bins], moments float64 [..., n_t][4]; leading axes are
    statistics groups) across ranks, as TWO
    collectives: one SUM over [counts as float64 | sum T | sum T^2] (integer counts below 2^53 add
    exactly in any order, so the reduced histogram is bitwise independent of the GPU count) and one
    MAX over [max T, -min T].  Generic torch version (any backend, CPU or CUDA tensors);
    :class:`StatsReducer` is the device fast path that packs inside the library and overlaps.
    Weighted statistics (``stat_weight=``) reduce the same way: the counts are integer weight totals, exact as long
    as each rank's total stays <= 2^32 - 1 (and so the reduced one far below 2^53)."""
    import torch
    import torch.distributed as dist
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size(group) == 1:
        return hist, moments
    bins = hist.shape[-1]
    h2, m2 = hist.reshape(-1, bins), moments.reshape(-1, moments.shape[-1])
    sums = torch.cat([h2.to(torch.float64), m2[:, 0:2]], dim=1).contiguous()
    ext = torch.stack([m2[:, 3], -m2[:, 2]], dim=1).contiguous()
    dist.all_reduce(sums, op=dist.ReduceOp.SUM, group=group)
    dist.all_reduce(ext, op=dist.ReduceOp.MAX, group=group)
    hist.copy_(sums[:, :bins].to(torch.int64).reshape(hist.shape))
    red = torch.stack([sums[:, bins], sums[:, bins + 1], -ext[:, 1], ext[:, 0]], dim=1)   # sum, sumsq, min, max
    moments.copy_(red.reshape(moments.shape))
    return hist, moments


class StatsReducer:
    """Cross-GPU reduction of a :class:`DevicePlan`'s statistics (SURVEY.md 8e): the only collective of
    the path.  ``submit()`` (after ``plan.stats_pass()``) folds the private copies straight into the
    packed layout (``ufair_stats_finalize_packed``), then -- on a side stream, so that it overlaps the
    next block's integration -- runs ONE all-reduce SUM and ONE all-reduce MAX over NCCL / NVLink and
    unpacks into ``plan.result.hist`` / ``.moments``.  ``wait()`` makes the current stream wait for
    the last reduction submitted.  With one rank it is just the plain finalize."""

    def __init__(self, plan, group=None, depth: int = 2):
        import torch
        import torch.distributed as dist
        self.plan, self.group = plan, group
        self.world = dist.get_world_size(group) if (dist.is_available() and dist.is_initialized()) else 1
        self._k = 0
        self._rows = math.prod(plan.stats.lead_shape(plan.n_out)) if plan.stats is not None else 0
        if self.world > 1 and plan.stats is not None:
            rows, bins = self._rows, plan.stats.bins
            dev = plan.device
            self._sums = [torch.empty(rows, bins + 2, dtype=torch.float64, device=dev) for _ in range(depth)]
            self._ext = [torch.empty(rows, 2, dtype=torch.float64, device=dev) for _ in range(depth)]
            self._ready = [torch.cuda.Event() for _ in range(depth)]
            self._done = [None] * depth
            self._stream = torch.cuda.Stream(device=dev)

    def submit(self):
        import ctypes as C

        import torch
        import torch.distributed as dist

        from . import _abi
        plan = self.plan
        if plan.stats is None:
            return
        if self.world == 1:
            plan.finalize_stats()
            return
        k = self._k % len(self._sums)
        self._k += 1
        main = torch.cuda.current_stream(plan.device)
        if self._done[k] is not None:
            main.wait_event(self._done[k])       # the reduction that last used buffer k has drained
        L, r = _abi.lib(), plan.result
        _abi.check(L.ufair_stats_finalize_packed(C.byref(plan.desc), self._sums[k].data_ptr(), self._ext[k].data_ptr(),
                                                 main.cuda_stream))
        self._ready[k].record(main)
        with torch.cuda.stream(self._stream):
            self._stream.wait_event(self._ready[k])
            dist.all_reduce(self._sums[k], op=dist.ReduceOp.SUM, group=self.group)
            dist.all_reduce(self._ext[k], op=dist.ReduceOp.MAX, group=self.group)
            _abi.check(L.ufair_stats_unpack(self._sums[k].data_ptr(), self._ext[k].data_ptr(), self._rows, plan.stats.bins,
                                            r.hist.data_ptr(), r.moments.data_ptr(), self._stream.cuda_stream))
            ev = torch.cuda.Event()
            ev.record(self._stream)
        self._done[k] = ev
        self._last = ev

    def wait(self):
        import torch
        if self.world > 1 and getattr(self, "_last", None) is not None:
            torch.cuda.current_stream(self.plan.device).wait_event(self._last)


def _parse_cpulist(text: str):
    cpus = set()
    for part in text.strip().split(","):
        if not part:
            continue
        lo, _, hi = part.partition("-")
        cpus.update(range(int(lo), int(hi or lo) + 1))
    return cpus


def numa_cpus_of_gpu(pci_domain: int, pci_bus: int, pci_device: int, sysfs: str = "/sys"):
    """(numa node, CPUs of that node) for the GPU at PCI domain:bus:device, read from sysfs;
    (-1, empty set) when the platform does not say (single-socket hosts report node -1)."""
    import os
    bdf = "%04x:%02x:%02x.0" % (pci_domain, pci_bus, pci_device)
    try:
        node = int(open(os.path.join(sysfs, "bus/pci/devices", bdf, "numa_node")).read().strip())
        if node < 0:
            return -1, set()
        return node, _parse_cpulist(open(os.path.join(sysfs, "devices/system/node/node%d/cpulist" % node)).read())
    except (OSError, ValueError):
        return -1, set()


def bind_rank_to_cpus(local_rank: int, world_size: int):
    """One process per GPU: give each rank its own cores BEFORE it allocates page-locked host buffers.
    Where sysfs names the GPU's NUMA node (multi-socket hosts) the rank is bound to that node's CPUs;
    where it does not but the host has several memory nodes, the CPUs this process may run on are split
    evenly over the ranks (contiguous blocks follow the node order); a single-node host is left alone.
    Returns dict(node, cpus, how)."""
    import os
    out = bind_to_gpu_numa_node(local_rank)
    if out["cpus"]:
        out["how"] = "numa node of the GPU (sysfs)"
        return out
    try:
        nodes = [d for d in os.listdir("/sys/devices/system/node") if d.startswith("node") and d[4:].isdigit()]
    except OSError:
        nodes = []
    if len(nodes) <= 1:   # one memory node (the round-2 B200 boxes are single-node KVM guests): nothing to gain
        return dict(node=out["node"], cpus=0, how="single NUMA node: left unchanged")
    try:
        allowed = sorted(os.sched_getaffinity(0))
        per = len(allowed) // max(world_size, 1)
        if world_size > 1 and per >= 1:
            mine = set(allowed[local_rank * per:(local_rank + 1) * per])
            os.sched_setaffinity(0, mine)
            return dict(node=out["node"], cpus=len(mine), how="even split of the %d allowed CPUs over %d ranks" % (len(allowed), world_size))
    except (AttributeError, OSError):
        pass
    return dict(node=out["node"], cpus=0, how="unchanged")


def bind_to_gpu_numa_node(device_index: int):
    """One process per GPU on a multi-socket host: run this rank on the CPUs of the NUMA node its
    GPU hangs off, BEFORE allocating page-locked host buffers (first touch then places them on that
    node), so the host pipeline's H2D / D2H copies do not cross the socket interconnect.
    Returns dict(node, cpus) describing what was done (cpus == 0: left unchanged)."""
    import os

    import torch
    p = torch.cuda.get_device_properties(device_index)
    node, cpus = numa_cpus_of_gpu(p.pci_domain_id, p.pci_bus_id, p.pci_device_id)
    try:
        allowed = os.sched_getaffinity(0) & cpus
        if allowed:
            os.sched_setaffinity(0, allowed)
            return dict(node=node, cpus=len(allowed))
    except (AttributeError, OSError):
        pass
    return dict(node=node, cpus=0)
