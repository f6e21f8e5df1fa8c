"""Device-resident orchestration of the inference hot path for a batch of images:

    RPN head outputs (cls, regr) + conv features
      -> decode + sanitize + validity + top-k          (K-a, proposals.cu)
      -> greedy NMS 0.7 -> max_boxes                   (K-b, nms.cu)
      -> the reference's 64-RoI batching/padding rule  (pad_rois, boxes.cu)
      -> RoI layer (crop + bilinear resize, or max)    (K-d, roi.cu)

which replaces `DetTrainingManager.get_det_inputs` + the RoI-layer half of `detector.predict` in
`voc_dets.get_dets` (det_util.py:136-158, voc_dets.py:37-49, custom_layers.py:35-56) without the
reference's per-image GPU->host->GPU round trips.  Inputs may be host numpy arrays (staged through
pinned memory, the drop-in case) or CUDA tensors (stay on the device).  Images are independent:
the batch dimension maps to grid.y / one CTA per image.
"""
import numpy as np
import torch

from . import ops
from .runtime import get_context
from .shared_constants import DEFAULT_ANCHORS


class ProposalRoiPipeline:
    def __init__(self, anchor_dims=DEFAULT_ANCHORS, stride=16, pre_nms_topk=8000, nms_thresh=0.7, max_boxes=300,
                 num_rois=64, pool_size=7, mode="resize", device=None, h2d_chunk=8):
        self.anchor_dims = np.asarray(anchor_dims)
        self.stride, self.k, self.thresh, self.max_boxes = stride, pre_nms_topk, nms_thresh, max_boxes
        self.num_rois, self.pool_size, self.mode = num_rois, pool_size, mode
        self.ctx = get_context(device)
        self.h2d_chunk = h2d_chunk
        self._copy_stream = None
        self._dev = {}
        self._host = {}

    # -- staging ----------------------------------------------------------------------------------
    def _stage_out(self, name, t):
        pin = self._host.get(name)
        if pin is None or pin.shape != t.shape or pin.dtype != t.dtype:
            pin = self._host[name] = torch.empty(t.shape, dtype=t.dtype).pin_memory()
        pin.copy_(t, non_blocking=True)
        return pin

    # -- the call a user makes ----------------------------------------------------------------------
    def run_device(self, cls, regr, feat, extents=None):
        """CUDA tensors in, CUDA tensors out; nothing synchronises.
        cls (B,R,C,A), regr (B,R,C,4A), feat (B,R,C,Cf) ->
        rois (B,max_boxes,4) i16, scores (B,max_boxes) f32, count (B,) i32,
        padded_rois (B,M,4) i16, pooled (B,M,P,P,Cf) f32 [, argmax in max mode].
        `extents` (B,2) i32 (rows, cols) on the device: a padded batch of differently sized maps (ops.pad_batch).  The
        proposals are sanitized against each image's own map, so the RoI layer reads no padding and every image's result
        equals the call on its own map."""
        rois, scores, count = ops.proposals(regr, cls, self.anchor_dims, self.stride, self.k, self.thresh,
                                            self.max_boxes, extents=extents)
        padded, _ = ops.pad_rois(rois, count, self.num_rois)
        pooled = ops.roi_forward(feat, padded, self.pool_size, self.mode)
        return rois, scores, count, padded, pooled

    def capture(self, cls, regr, feat, extents=None):
        """CUDA-graph capture of `run_device` for fixed shapes (SURVEY 8f-1): returns a `GraphedRun` whose call copies
        new inputs into the captured buffers and replays decode -> top-k -> NMS -> pad -> RoI layer as ONE graph
        launch (5 kernels, no per-kernel Python/ctypes/launch overhead -- what matters at batch 1).  Captured with
        `extents`, the extents are an input of the graph too: one graph serves every mix of sizes up to the padded
        shape."""
        return GraphedRun(self, cls, regr, feat, extents)

    def __call__(self, cls, regr, feat, on_device=None):
        """Host (or device) arrays in; returns (rois, scores, count) as numpy on the host -- what
        `get_det_inputs` hands back in the reference -- plus the pooled features as a CUDA tensor
        ((pooled, argmax) in max mode), which stay on the device for the detector head exactly like the RoI layer's output inside the
        reference's TF graph.  `on_device(rois, scores, count)` (optional) is invoked with the device
        tensors before the read-back, e.g. to enqueue the multi-GPU all-gather of the final RoIs.

        Host inputs are uploaded in chunks of `h2d_chunk` images on a copy stream while the kernels of
        the previous chunk run (images are independent, so chunking does not change any result); one
        stream synchronisation at the end.  `feat` may already be a CUDA tensor while cls / regr are host arrays (a GPU
        backbone next to a host-side RPN head): it is then used in place and only the small head outputs are uploaded.

        A list of per-image host arrays cls (R_b,C_b,A), regr (R_b,C_b,4A) and feat (R_b,C_b,Cf) is a batch of differently
        sized images: only each image's valid region is uploaded into the padded device buffers, and the batch runs as one
        padded batch with extents (a CUDA tensor `feat` must then already be the padded (B,R,C,Cf) batch)."""
        host_in = isinstance(cls, (list, tuple)) or not (isinstance(cls, torch.Tensor) and cls.is_cuda)
        if not host_in:
            rois, scores, count, padded, pooled = self.run_device(cls, regr, feat)
        else:
            rois, scores, count, padded, pooled = self._run_chunked(cls, regr, feat)
        if on_device is not None:
            on_device(rois, scores, count)
        h_rois, h_scores, h_count = (self._stage_out("rois", rois), self._stage_out("scores", scores),
                                     self._stage_out("count", count))
        torch.cuda.current_stream(self.ctx.device).synchronize()
        # fresh arrays like the reference's get_det_inputs (det_util.py:158): the pinned staging buffers are reused by
        # the next call and must not alias what the caller keeps (a few KB per image)
        return h_rois.numpy().copy(), h_scores.numpy().copy(), h_count.numpy().copy(), pooled

    def _pinned(self, name, x):
        t = x if isinstance(x, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32))
        if t.dtype != torch.float32 or not t.is_contiguous():
            t = t.to(torch.float32).contiguous()
        if t.is_pinned():
            return t
        pin = self._host.get(name)
        if pin is None or pin.shape != t.shape:
            pin = self._host[name] = torch.empty(t.shape, dtype=torch.float32).pin_memory()
        pin.copy_(t)
        return pin

    def _device_buffer(self, name, shape, dtype):
        buf = self._dev.get(name)
        if buf is None or buf.shape != torch.Size(shape) or buf.dtype != dtype:
            buf = self._dev[name] = torch.empty(shape, dtype=dtype, device=self.ctx.device)
        return buf

    def _pinned_ragged(self, name, arrays):
        """per-image host arrays -> views of one pinned staging buffer, each image's valid region back to back"""
        ts = [torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32)) if not isinstance(x, torch.Tensor)
              else x.to(torch.float32).contiguous() for x in arrays]
        total = sum(t.numel() for t in ts)
        pin = self._host.get(name)
        if pin is None or pin.dim() != 1 or pin.numel() < total:
            pin = self._host[name] = torch.empty(max(total, 1), dtype=torch.float32).pin_memory()
        views, off = [], 0
        for t in ts:
            v = pin[off:off + t.numel()].view(t.shape)
            v.copy_(t)
            views.append(v)
            off += t.numel()
        return views

    def _run_chunked(self, cls, regr, feat):
        dev = self.ctx.device
        feat_on_device = isinstance(feat, torch.Tensor) and feat.is_cuda     # a GPU backbone hands its features over as is
        extents = None
        if isinstance(cls, (list, tuple)):                                   # differently sized images
            if len(regr) != len(cls) or (not feat_on_device and len(feat) != len(cls)):
                raise ValueError("cls, regr and feat must list the same images")
            ext = np.array([tuple(x.shape[:2]) for x in cls], np.int32).reshape(-1, 2)
            rows, cols = (int(v) for v in ext.max(axis=0))
            if feat_on_device:
                rows, cols = feat.shape[1], feat.shape[2]
            srcs = {"cls": self._pinned_ragged("cls", cls), "regr": self._pinned_ragged("regr", regr)}
            if not feat_on_device:
                srcs["feat"] = self._pinned_ragged("feat", feat)
            b = len(cls)
            bufs = {k: self._device_buffer(k, (b, rows, cols, v[0].shape[2]), torch.float32) for k, v in srcs.items()}
            extents = self.ctx.to_device(ext)
        else:
            srcs = {"cls": self._pinned("cls", cls), "regr": self._pinned("regr", regr)}
            if not feat_on_device:
                srcs["feat"] = self._pinned("feat", feat)
            b = srcs["cls"].shape[0]
            bufs = {k: self._device_buffer(k, v.shape, torch.float32) for k, v in srcs.items()}
        if feat_on_device:
            bufs["feat"] = feat if feat.dtype == torch.float32 and feat.is_contiguous() else feat.float().contiguous()
        m = -(-self.max_boxes // self.num_rois) * self.num_rois
        rois = self._device_buffer("o_rois", (b, self.max_boxes, 4), torch.int16)
        scores = self._device_buffer("o_scores", (b, self.max_boxes), torch.float32)
        count = self._device_buffer("o_count", (b,), torch.int32)
        padded = self._device_buffer("o_padded", (b, m, 4), torch.int16)
        rows = self._device_buffer("o_rows", (b,), torch.int32)
        pooled = torch.empty((b, m, self.pool_size, self.pool_size, bufs["feat"].shape[3]), dtype=torch.float32, device=dev)
        argmax = torch.empty(pooled.shape, dtype=torch.int32, device=dev) if self.mode == "max" else None
        if self._copy_stream is None:
            self._copy_stream = torch.cuda.Stream(device=dev)
        cur = torch.cuda.current_stream(dev)
        self._copy_stream.wait_stream(cur)            # the previous call's kernels no longer read the buffers
        events = []
        # chunked upload hides the 10 MB/image feature copy behind the kernels; with the features already on the device
        # only 0.4 MB/image of head outputs moves: a few large chunks keep that copy off the critical path without paying
        # the small-batch latency of the proposal kernels
        step = max(16, -(-b // 4)) if feat_on_device else max(1, int(self.h2d_chunk))
        with torch.cuda.stream(self._copy_stream):
            for lo in range(0, b, step):
                hi = min(b, lo + step)
                for k in srcs:
                    if extents is None:
                        bufs[k][lo:hi].copy_(srcs[k][lo:hi], non_blocking=True)
                    else:                                 # the valid region only; the padding is never read
                        for i in range(lo, hi):
                            r, c = srcs[k][i].shape[:2]
                            bufs[k][i, :r, :c].copy_(srcs[k][i], non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(self._copy_stream)
                events.append((lo, hi, ev))
        for lo, hi, ev in events:
            cur.wait_event(ev)
            ops.proposals(bufs["regr"][lo:hi], bufs["cls"][lo:hi], self.anchor_dims, self.stride, self.k, self.thresh,
                          self.max_boxes, out=(rois[lo:hi], scores[lo:hi], count[lo:hi]),
                          extents=None if extents is None else extents[lo:hi])
            ops.pad_rois(rois[lo:hi], count[lo:hi], self.num_rois, out=(padded[lo:hi], rows[lo:hi]))
            ops.roi_forward(bufs["feat"][lo:hi], padded[lo:hi], self.pool_size, self.mode, out=pooled[lo:hi],
                            argmax_out=None if argmax is None else argmax[lo:hi])
        return rois, scores, count, padded, (pooled if argmax is None else (pooled, argmax))

    @staticmethod
    def h2d_bytes(cls, regr, feat):
        """bytes uploaded per call; features that already live on the device are not counted"""
        on_dev = isinstance(feat, torch.Tensor) and feat.is_cuda
        return 4 * (int(np.prod(cls.shape)) + int(np.prod(regr.shape)) + (0 if on_dev else int(np.prod(feat.shape))))

    def d2h_bytes(self, batch):
        return batch * (self.max_boxes * 8 + self.max_boxes * 4 + 4)


class GraphedRun:
    """One captured `ProposalRoiPipeline.run_device` call.  The graph runs on a private C-ABI handle: its scratch arena
    is sized by two eager warm-up runs and can never be moved by other calls, so the device pointers baked into the
    graph stay valid.  Outputs are the captured tensors (overwritten by every replay)."""

    def __init__(self, pipe, cls, regr, feat, extents=None):
        from .runtime import Context, use_context
        dev = pipe.ctx.device
        self.inputs = tuple(torch.empty_like(t, device=dev).copy_(t) for t in (cls, regr, feat) +
                            (() if extents is None else (extents,)))
        self._ctx = Context(dev.index)
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with use_context(self._ctx), torch.cuda.stream(side):
            for _ in range(2):                       # grows the private arena to its final size (merge on 2nd call)
                pipe.run_device(*self.inputs)
            side.synchronize()
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph, stream=side):
                self.outputs = pipe.run_device(*self.inputs)
        torch.cuda.current_stream(dev).wait_stream(side)

    def __call__(self, cls=None, regr=None, feat=None, extents=None):
        """Replays the graph (after copying any given CUDA tensor into the captured input of the same shape).  New
        `extents` need a graph captured with extents."""
        if extents is not None and len(self.inputs) < 4:
            raise ValueError("this graph was captured without extents")
        for dst, src in zip(self.inputs, (cls, regr, feat, extents)):
            if src is not None and src.data_ptr() != dst.data_ptr():
                dst.copy_(src, non_blocking=True)
        self.graph.replay()
        return self.outputs


def _padded_inputs(cls, regr, feat, extents):
    """lists of per-image arrays -> padded batches + extents (ops.pad_batch); anything else passes through"""
    if not isinstance(cls, (list, tuple)):
        if extents is not None and not isinstance(extents, torch.Tensor):
            extents = get_context().to_device(np.asarray(extents, np.int32).reshape(-1, 2))
        return cls, regr, feat, extents
    cls, extents = ops.pad_batch(cls)
    regr, _ = ops.pad_batch(regr, pad_to=cls.shape[1:3])
    feat = feat if isinstance(feat, torch.Tensor) and feat.is_cuda else ops.pad_batch(feat, pad_to=cls.shape[1:3])[0]
    return cls.float(), regr.float(), feat.float(), extents


class DetectionPipeline(ProposalRoiPipeline):
    """Whole inference hot path of `voc_dets.get_dets` (voc_dets.py:20-88) for a BATCH of images, device-resident:

        RPN head outputs -> proposals -> 64-RoI padding -> RoI layer -> detector head (caller's callable)
                         -> per-class post-processing (arg-max class, float64 decode, NMS 0.5, rescale)

    `detector_head(pooled (B,M,P,P,C) f32, rois (B,M,4) i16) -> (out_cls (B,M,K) f32, out_reg (B,M,4(K-1)) f32)` runs on
    CUDA tensors (the dense layers are not part of this package).  Rows past the reference's padded length
    (`ceil(n_rois/64)*64`) are ignored, so results equal per-image `get_dets` calls.  With torch.distributed initialised,
    `gather=True` all-gathers the fixed-size detection buffers of every rank (the path's only collective)."""

    def __init__(self, detector_head, class_mapping, det_threshold=0.0, det_nms_thresh=0.5, det_max_boxes=2000, **kwargs):
        super().__init__(**kwargs)
        self.detector_head = detector_head
        self.class_mapping = class_mapping
        self.det_threshold, self.det_nms_thresh, self.det_max_boxes = det_threshold, det_nms_thresh, det_max_boxes

    def detect_device(self, cls, regr, feat, resize_ratios, gather=False, extents=None):
        """CUDA tensors in -> (det_boxes (B,M,4) i32, det_probs (B,M) f32, det_cls (B,M) i32, det_count (B,) i32).
        `extents` (B,2) i32 on the device: a padded batch of differently sized maps, as in `run_device`."""
        rois, scores, count = ops.proposals(regr, cls, self.anchor_dims, self.stride, self.k, self.thresh, self.max_boxes,
                                            extents=extents)
        padded, rows = ops.pad_rois(rois, count, self.num_rois)
        pooled = ops.roi_forward(feat, padded, self.pool_size, self.mode)
        out_cls, out_reg = self.detector_head(pooled if self.mode == "resize" else pooled[0], padded)
        ratios = resize_ratios if isinstance(resize_ratios, torch.Tensor) else \
            self.ctx.to_device(np.asarray(resize_ratios, dtype=np.float64))
        dets = ops.det_postprocess(padded, out_cls.contiguous(), out_reg.contiguous(), ratios, self.class_mapping['bg'],
                                   self.stride, self.det_threshold, self.det_nms_thresh, self.det_max_boxes, n_rows=rows)
        if gather:
            from . import parallel
            packed, counts = parallel.pack_detections(*dets)
            return parallel.all_gather_detections(packed, counts)
        return dets

    def detect(self, cls, regr, feat, resize_ratios, extents=None):
        """Host or device arrays in -> per image the reference's list of {'bbox', 'cls_name', 'prob'} dicts.  Lists of
        per-image (R_b,C_b,X) arrays are a batch of differently sized images (padded with ops.pad_batch)."""
        cls, regr, feat, extents = _padded_inputs(cls, regr, feat, extents)
        dev_in = [x if (isinstance(x, torch.Tensor) and x.is_cuda) else self.ctx.to_device(x, np.float32) for x in (cls, regr, feat)]
        boxes, probs, dcls, count = (self.ctx.to_host(t) for t in self.detect_device(*dev_in, resize_ratios,
                                                                                   extents=extents))
        names = {v: k for k, v in self.class_mapping.items()}
        return [[{'bbox': boxes[b, i].astype(np.int64), 'cls_name': names[int(dcls[b, i])], 'prob': probs[b, i]}
                 for i in range(int(count[b]))] for b in range(len(count))]


class DetTrainingPipeline:
    """Detector-training inputs of `DetTrainingManager.get_training_input` (det_util.py:63-133) for a BATCH of images,
    device-resident:

        RPN head outputs -> proposals (top-k 12000, NMS 0.7 -> 2000) -> RoI x GT labelling (eligible >= 0.1, positive
        >= 0.5, one-hot classes, class-specific regression targets) -> 64-RoI mini-batch (<= 25 % positives)
        [-> RoI layer on the sampled RoIs]

    By default only the mini-batch draw runs on the host: it replays `det_util._get_det_samples` with numpy's legacy
    global RNG, image by image in batch order, so the result equals calling the reference-shaped manager on each image in
    turn (one D2H of the positive flags and counts, one H2D of the B x 64 sample rows).  Given a `state`
    (ops.sampler_state) the draw runs on the device with a counter-based RNG instead (same rule, different stream).  An
    image without an eligible RoI (the reference returns 4 x None) gets zero rows and `has_rois[b] = False`."""

    def __init__(self, class_mapping, anchor_dims=DEFAULT_ANCHORS, stride=16, num_rois=64, pre_nms_topk=12000,
                 nms_thresh=0.7, max_boxes=2000, pool_size=7, mode="resize", device=None):
        if class_mapping['bg'] != len(class_mapping) - 1:
            raise NotImplementedError("'bg' must be the last class index (the reference assumes it too: det_util.py:120)")
        self.class_mapping, self.anchor_dims = class_mapping, np.asarray(anchor_dims)
        self.stride, self.num_rois, self.k, self.thresh, self.max_boxes = stride, num_rois, pre_nms_topk, nms_thresh, max_boxes
        self.pool_size, self.mode = pool_size, mode
        self.ctx = get_context(device)
        self._pinned = {}

    def _pin(self, key, shape, dtype):
        buf = self._pinned.get(key)
        if buf is None or buf.shape != torch.Size(shape) or buf.dtype != dtype:
            buf = self._pinned[key] = torch.empty(tuple(shape), dtype=dtype).pin_memory()
        return buf

    def ground_truth(self, images):
        """list of images -> (gt (B,Gmax,4) f64 feature units, gt_cls (B,Gmax) i32, n_gt (B,) i32) on the device."""
        from .det_util import _gt_feature_boxes
        per = [_gt_feature_boxes(img, self.class_mapping, self.stride) for img in images]
        g_max = max(len(g) for g, _ in per)
        gt = np.zeros((len(per), g_max, 4), np.float64)
        gt_cls = np.zeros((len(per), g_max), np.int32)
        for b, (g, c) in enumerate(per):
            gt[b, :len(g)], gt_cls[b, :len(c)] = g, c
        n_gt = np.array([len(g) for g, _ in per], np.int32)
        return self.ctx.to_device(gt), self.ctx.to_device(gt_cls), self.ctx.to_device(n_gt)

    def targets(self, cls, regr, gt, gt_cls, n_gt, chunk=32, extents=None, state=None):
        """CUDA tensors in -> (rois (B,S,4) i16, y_class_num (B,S,K) i32, y_transform (B,S,8(K-1)) f32) on the device and
        has_rois (B,) bool on the host.  The batch is enqueued in chunks of `chunk` images; the host draws the
        mini-batches of chunk i (in image order, so the RNG stream is the per-image one) while the GPU is still
        labelling chunks i+1..  `extents` (B,2) i32 on the device: a padded batch of differently sized maps.

        With `state` (ops.sampler_state) the mini-batches are drawn on the device instead (ops.sample_det: the same rule,
        a counter-based RNG stream): nothing returns to the host, has_rois is a CUDA bool tensor, the call can be
        captured in a CUDA graph, and image b's draw depends on (seed, offset + b) only, so not on `chunk`.  The
        state's offset advances by B."""
        b, dev = cls.shape[0], self.ctx.device
        stream = torch.cuda.current_stream(dev)
        staged = []
        for lo in range(0, b, chunk):
            hi = min(b, lo + chunk)
            rois, _, count = ops.proposals(regr[lo:hi], cls[lo:hi], self.anchor_dims, self.stride, self.k, self.thresh,
                                           self.max_boxes, extents=None if extents is None else extents[lo:hi])
            l_rois, y_cls, y_tr, _, m = ops.label_rois(rois, gt[lo:hi], gt_cls[lo:hi], n_gt[lo:hi],
                                                       len(self.class_mapping), n_roi=count)
            found_d = (y_cls[:, :, -1] == 0).to(torch.uint8)                      # positives = not background
            if state is not None:
                index, has = ops.sample_det(found_d, m, self.num_rois, state)
                staged.append(ops.gather_det_samples(l_rois, y_cls, y_tr, index) + (has,))
                continue
            found_h = self._pin(("found", lo), found_d.shape, torch.uint8)     # cached: cudaHostAlloc costs ~0.1 ms
            m_h = self._pin(("m", lo), m.shape, m.dtype)
            found_h.copy_(found_d, non_blocking=True)
            m_h.copy_(m, non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(stream)
            staged.append((l_rois, y_cls, y_tr, found_h, m_h, ev))
        if state is not None:
            return tuple(torch.cat([o[j] for o in staged]) for j in range(4))
        from .det_util import _get_det_samples
        outs, has = [], []
        for l_rois, y_cls, y_tr, found_h, m_h, ev in staged:
            ev.synchronize()
            found, m_host = found_h.numpy(), m_h.numpy()
            index = np.full((len(m_host), self.num_rois), -1, np.int32)
            for i, mb in enumerate(m_host.tolist()):                               # RNG draws in image order
                if mb > 0:
                    index[i] = _get_det_samples(found[i, :mb] == 1, self.num_rois)
            index_h = self._pin(("index", len(outs)), index.shape, torch.int32)
            index_h.copy_(torch.from_numpy(index))
            outs.append(ops.gather_det_samples(l_rois, y_cls, y_tr, index_h.to(dev, non_blocking=True)))
            has.append(m_host > 0)
        rois, y_cls, y_tr = (torch.cat([o[j] for o in outs]) for j in range(3))
        return rois, y_cls, y_tr, np.concatenate(has)

    def __call__(self, cls, regr, feat, images, extents=None, state=None):
        """Host or device arrays + the images' ground truth -> (rois, y_class_num, y_transform, pooled, has_rois):
        the detector's training inputs and the RoI layer's output on the sampled RoIs (CUDA tensors).  Lists of
        per-image (R_b,C_b,X) arrays, or padded arrays with `extents`, are a batch of differently sized images; the
        sampled RoIs lie inside each image's own map, so the RoI layer reads no padding.  `state`
        (ops.sampler_state): mini-batches drawn on the device, see `targets`."""
        cls, regr, feat, extents = _padded_inputs(cls, regr, feat, extents)
        dev_in = [x if (isinstance(x, torch.Tensor) and x.is_cuda) else self.ctx.to_device(x, np.float32) for x in (cls, regr, feat)]
        rois, y_cls, y_tr, has = self.targets(dev_in[0], dev_in[1], *self.ground_truth(images), extents=extents,
                                              state=state)
        pooled = ops.roi_forward(dev_in[2], rois, self.pool_size, self.mode)
        return rois, y_cls, y_tr, pooled, has
