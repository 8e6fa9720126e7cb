"""Input pipeline: the weight-independent front of the hot path, one batch ahead, on a side stream.

Host to device copy, hard voxelization (K1), MeanVFE (K2) and the index / rulebook builds of every level (K3/K4) depend on
the points only.  They also hold every host synchronisation of the path (the voxel count and the active-set size of each
strided convolution size the tensors that follow).  Run in-line, each of those waits for the whole stream, i.e. for the
previous batch's backward pass, and the GPU then idles while the host catches up.  `InputPipeline` runs that front for
batch i+1 on a high-priority side stream while the backbone of batch i executes on the main stream: the host waits only
for the small front kernels, and the forward pass that follows contains no index kernels and no synchronisation.

This is the role the reference gives its DataLoader workers (voxelization ahead of the training step,
pcdet/datasets/processor/data_processor.py L115-143 under torch DataLoader prefetch); here it is a CUDA stream.

    pipe = InputPipeline(vfe, backbone, device)
    nxt = pipe.submit({"points": pts, "point_frame_offsets": offs, "batch_size": B})
    for ...:
        batch_dict = pipe.consume(nxt)             # main stream waits for the front of this batch (event, no host sync)
        loss = head(backbone(batch_dict)) ...      # launches only
        nxt = pipe.submit(next_batch)              # overlaps with the kernels queued above
"""
from collections import deque

import torch


class _Handle:
    def __init__(self, batch_dict, ready, tensors):
        self.batch_dict, self.ready, self.tensors = batch_dict, ready, tensors


class InputPipeline:
    def __init__(self, vfe, backbone, device, reserve_bytes=8 << 30, preprocess=None):
        """preprocess: optional callable batch_dict -> batch_dict run on the side stream after the inputs are staged and
        before the VFE, e.g. the device augmentations and point pre-steps `lambda bd: pp.forward(aug.forward(bd))`.  Run
        before submit() instead, those would sit on the main stream behind the previous batch's backward pass."""
        self.vfe, self.backbone, self.preprocess = vfe, backbone, preprocess
        self.device = torch.device(device)
        lo, hi = torch.cuda.Stream.priority_range()      # (lowest, highest): highest is the numerically smaller one
        self.stream = torch.cuda.Stream(self.device, priority=hi)
        self._started = deque()     # main-stream events, one per consume(): "the batch before this one has finished"
        if reserve_bytes:
            # the caching allocator keeps one pool per stream: give the side stream its blocks up front so that row
            # counts that differ from batch to batch never reach cudaMalloc (which synchronises the device)
            with torch.cuda.stream(self.stream):
                block = torch.empty(int(reserve_bytes), dtype=torch.uint8, device=self.device)
                del block

    def submit(self, batch_dict, inputs_pending=True):
        """Starts the front of the path for `batch_dict` on the side stream.  `points` / `point_frame_offsets` may be
        pinned host tensors (copied here, asynchronously) or device tensors.  inputs_pending: device inputs may still
        be being written by work queued on the current stream, so the side stream waits for it; pass False for inputs
        that are already complete (then the front starts at once, next to whatever the main stream is running)."""
        # Bound the run-ahead: the front has no dependency on the main stream, so without this the host (throttled only
        # by the front's own small syncs) queues several steps ahead of the GPU, every queued batch keeps its ~0.5 GB of
        # tables alive, the side pool runs dry and torch falls back to cudaMalloc, which stalls for as long as the queue
        # in front of it (measured: 20-90 ms).  Waiting for the start of the batch consumed last keeps one full batch
        # queued on the main stream (the GPU never idles) and at most three batches' tables alive.
        while len(self._started) > 1:
            self._started.popleft()
        if self._started:
            self._started[0].synchronize()
        if inputs_pending and any(torch.is_tensor(v) and v.is_cuda for v in batch_dict.values()):
            self.stream.wait_stream(torch.cuda.current_stream(self.device))
        bd = dict(batch_dict)
        with torch.cuda.stream(self.stream), torch.no_grad():
            staged = []
            for key in ("points", "point_frame_offsets", "voxels", "voxel_coords", "voxel_num_points"):
                t = bd.get(key)
                if torch.is_tensor(t):
                    if not t.is_cuda:
                        t = t.to(self.device, non_blocking=True)
                        staged.append(t)
                    bd[key] = t
            before = set(id(v) for v in bd.values() if torch.is_tensor(v))
            if self.preprocess is not None:
                bd = self.preprocess(bd)
            bd = self.vfe(bd)
            plan = None
            if bd.get("voxel_coords_canonical", False):
                # (voxels that arrive in another row order, e.g. voxelized on the host, are put in canonical order by the
                # backbone's first layer together with their features: nothing to plan ahead without the features)
                plan = self.backbone.plan_geometry(bd["voxel_coords"], int(bd["batch_size"]), canonical=True)
                bd["spconv_geometry"] = plan
            ready = torch.cuda.Event()
            ready.record(self.stream)
        tensors = staged + [v for v in bd.values() if torch.is_tensor(v) and id(v) not in before]
        if plan is not None:
            tensors += plan.tensors()
        return _Handle(bd, ready, tensors)

    def consume(self, handle):
        """Makes the current stream wait for the front of that batch and hands over its batch_dict."""
        main = torch.cuda.current_stream(self.device)
        started = torch.cuda.Event()
        started.record(main)           # completes when everything queued before this batch (the previous batch) is done
        self._started.append(started)
        main.wait_event(handle.ready)
        for t in handle.tensors:
            t.record_stream(main)      # allocated on the side stream's pool, read by main-stream kernels from now on
        return handle.batch_dict
