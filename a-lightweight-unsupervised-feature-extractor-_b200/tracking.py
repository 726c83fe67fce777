"""GPU-resident tracker with the reference's surface (model/mainTracking.py).

* ``Tracking``            - drop-in for the reference class: ``Tracking().update(obj)`` returns
                            ``(matches_tid, unmatched_track_ids, unmatched_dets)`` (mainTracking.py:450-610).
* ``MultiStreamTracker``  - the same association step for S independent video streams per launch
                            (the batching the reference lacks; SURVEY.md section 8e/8f).

All state (Kalman filters, EMA embeddings, history banks, ages) lives on the device inside a
``b200_tracker`` handle; one ``update`` is one host->device copy of the detections, five kernels and
one device->host copy of a small result table.  There is no CPU fallback.
"""
import ctypes
from typing import Any, Dict, List, Optional

import numpy as np
import torch
import yaml

from . import _lib, cost as cost_ops, kalman as kalman_ops

# mainTracking.py:55-96 -- defaults used when a key is missing from the YAML `tracker` block.
CODE_DEFAULTS = dict(
    init_conf_min=0.5, hist_max=10, emb_top_k=5, app_tau=0.07, eps=1e-12, w_app=1.0, w_bbox=0.3, w_conf=0.2,
    alpha=1.0, beta=0.5, unmatch_cost=10.0, cost_max=50.0, max_age=30, ema_alpha=0.9, conf_update_min=0.55,
    cost_update_max=30.0, maha_thr=9.49, lost_reid_after=60, reid_sim_min=0.6)

# model/conf/conf.yaml:2-24 -- the tracker block the reference ships.
SHIPPED_CONF = dict(
    init_conf_min=0.5, hist_max=30, emb_top_k=5, app_tau=0.07, eps=1e-12, w_app=1.0, w_bbox=0.3, w_conf=0.2,
    alpha=1.0, beta=0.5, unmatch_cost=10.0, cost_max=50.0, max_age=120, ema_alpha=0.9, conf_update_min=0.55,
    cost_update_max=30.0, maha_thr=9.49, lost_reid_after=50, reid_sim_min=0.6, reid_only_cost_max=0.4)

R_NMATCH, R_NUT, R_NUD, R_NLIVE, R_NEXT, R_STATUS, R_M1, R_M2, R_HDR = range(9)


def load_conf(path: str) -> Dict[str, Any]:
    """mainTracking.py:11-13."""
    with open(path, "r", encoding="utf-8") as f:
        return yaml.safe_load(f)


def resolve_conf(tcfg: Dict[str, Any]) -> Dict[str, Any]:
    """Applies the reference's per-key defaults and the reid_only_cost_max rule (:92-96)."""
    c = dict(CODE_DEFAULTS)
    c.update({k: v for k, v in tcfg.items() if v is not None})
    if "reid_only_cost_max" not in tcfg:
        c["reid_only_cost_max"] = 1.0 - float(c["reid_sim_min"])
    for k in ("hist_max", "emb_top_k", "max_age", "lost_reid_after"):
        c[k] = int(c[k])
    return c


def _c_conf(c):
    s = _lib.tracker_conf()
    for name, _ in _lib.tracker_conf._fields_:
        setattr(s, name, c[name])
    return s


class MultiStreamTracker:
    """S independent trackers stepped by the same kernel launches.

    Detections are passed as dense host arrays padded to ``max_dets`` per stream:
    ``n_det[S]`` (-1 = stream idle, 0 = empty frame), ``boxes[S,max_dets,4]`` float64 xyxy,
    ``confs[S,max_dets]`` float64, ``embs[S,max_dets,128]`` float32, ``frame_ids[S]``.
    ``step_device`` takes the same layout on the device; ``step_detections`` takes the detector's rows and the
    encoder's embeddings on the device as they come, with a stream index per row.
    """

    def __init__(self, n_streams: int, conf: Optional[Dict[str, Any]] = None, max_tracks: int = 256,
                 max_dets: int = 128, device=None, auto_grow: bool = True):
        if not torch.cuda.is_available():
            raise _lib.B200Error("no CUDA device: this package has no CPU path")
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.conf = resolve_conf(SHIPPED_CONF if conf is None else conf)
        self.S, self.auto_grow = int(n_streams), bool(auto_grow)
        self._h = ctypes.c_void_p()
        self._create(int(max_tracks), int(max_dets))
        self.n_live = np.zeros(self.S, dtype=np.int64)
        self._n_live_stale = False                 # set by device-side steps and step-by-step methods: n_live is out of date
        self._pending = []                         # StepHandles of step_async calls whose result has not been collected
        self._pending_births = np.zeros(self.S, dtype=np.int64)

    def n_live_now(self) -> np.ndarray:
        """Live tracks per stream as of the work queued so far (re-read from the device after device-side steps)."""
        self.drain()
        if self._n_live_stale:
            n = np.zeros(self.S, np.int32)
            with torch.cuda.device(self.device):
                _lib.check(_lib.lib().b200_tracker_live_counts(self._h, n.ctypes.data_as(ctypes.c_void_p), None,
                                                               _lib.stream_ptr(self.device)))
            self.n_live[:] = n
            self._n_live_stale = False
        return self.n_live

    def _create(self, max_tracks, max_dets):
        h = ctypes.c_void_p()
        cc = _c_conf(self.conf)
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().b200_tracker_create(ctypes.byref(h), self.S, max_tracks, max_dets, ctypes.byref(cc)))
        self._h, self.max_tracks, self.max_dets = h, max_tracks, max_dets
        self.stride = _lib.lib().b200_tracker_result_stride(h)

    def grow(self, max_tracks: Optional[int] = None, max_dets: Optional[int] = None):
        """Migrates every stream's state into a handle with larger capacities, on the device: ``state_dict()`` -> a new
        handle -> import.  If the larger handle cannot be created the tracker is left as it was.  Live counts do not
        change.  A CUDA graph captured before a growth holds the old handle's buffers: capture it again."""
        self.drain()
        sd = self.state_dict()
        old = (self._h, self.max_tracks, self.max_dets, self.stride)
        self._create(max(self.max_tracks, int(max_tracks or 0)), max(self.max_dets, int(max_dets or 0)))
        try:
            status = self._import(sd, None)            # reads the status back: the import has completed
            bad = np.nonzero(status)[0]
            if len(bad):
                raise _lib.B200Error("grow: stream %d failed to migrate (status %d)" % (bad[0], status[bad[0]]))
        except BaseException:
            _lib.lib().b200_tracker_destroy(self._h)
            self._h, self.max_tracks, self.max_dets, self.stride = old
            raise
        _lib.lib().b200_tracker_destroy(old[0])

    # -- device-side state images (b200_tracker_state, layout _lib.STATE_LAYOUT) ----------------------------------
    def _stream_index(self, streams, what, distinct):
        """-> (host int64 indices, device int32 tensor, or None for every stream in order)."""
        if streams is None:
            return np.arange(self.S), None
        idx = np.asarray(streams.cpu() if isinstance(streams, torch.Tensor) else streams, dtype=np.int64).reshape(-1)
        if len(idx) and (idx.min() < 0 or idx.max() >= self.S):
            raise ValueError("%s: stream index out of range [0, %d)" % (what, self.S))
        if distinct and len(np.unique(idx)) != len(idx):
            raise ValueError("%s: duplicate stream index" % what)
        return idx, torch.as_tensor(idx, dtype=torch.int32).to(self.device)

    def _new_image(self, rows: int, cap: int) -> Dict[str, torch.Tensor]:
        dims = dict(cap=cap, hist_max=self.conf["hist_max"])
        return {n: torch.zeros((rows,) + tuple(dims.get(k, k) for k in shape), dtype=getattr(torch, dt), device=self.device)
                for n, dt, shape in _lib.STATE_LAYOUT}

    @staticmethod
    def _c_image(sd):
        im = _lib.tracker_state()
        for n, _, _ in _lib.STATE_LAYOUT:
            setattr(im, n, sd[n].data_ptr())
        im.n_rows, im.cap, im.hist_max = sd["n_live"].shape[0], sd["ids"].shape[1], sd["bank"].shape[2]
        return im

    def _import(self, sd, dev_idx, read_status=True):
        """b200_tracker_import_device on the current stream; returns the per-row status (synchronises) or None."""
        status = torch.empty(sd["n_live"].shape[0], dtype=torch.int32, device=self.device) if read_status else None
        im = self._c_image(sd)
        with torch.cuda.device(self.device):
            rc = _lib.lib().b200_tracker_import_device(self._h, _lib.ptr(dev_idx), ctypes.byref(im), _lib.ptr(status),
                                                       _lib.stream_ptr(self.device))
        _lib.check(rc)
        return status.cpu().numpy() if read_status else None

    def state_dict(self, streams=None) -> Dict[str, torch.Tensor]:
        """The state of ``streams`` (a list or tensor of stream indices; None = every stream, in order) as device tensors,
        one row per stream: ``n_live`` / ``next_id`` [R] int32 and the live tracks of each row in ascending track id,
        in ``export``'s layout with ``cap = max_tracks`` slots per row (``ids`` [R, cap], ``bank`` [R, cap, hist_max,
        128], ...; slots past ``n_live`` are zero).  Asynchronous on the current stream, no read-back: ``torch.save``
        it, ``load_state_dict`` it into another tracker, or capture it in a CUDA graph."""
        self.drain()
        idx, dev_idx = self._stream_index(streams, "state_dict", distinct=False)
        sd = self._new_image(len(idx), self.max_tracks)
        if len(idx):
            im = self._c_image(sd)
            with torch.cuda.device(self.device):
                rc = _lib.lib().b200_tracker_export_device(self._h, _lib.ptr(dev_idx), ctypes.byref(im), None,
                                                           _lib.stream_ptr(self.device))
            _lib.check(rc)
        return sd

    def load_state_dict(self, sd: Dict[str, torch.Tensor], streams=None):
        """Replaces the state of ``streams`` (distinct indices; None = every stream, in order) by the rows of ``sd``, an
        image as ``state_dict`` returns it (any ``cap``, tensors on any device).  The image carries state, not
        configuration: hyper-parameters stay this tracker's own, and ``hist_max`` must be equal (ValueError).  A row with
        more than ``max_tracks`` tracks grows the handle (``auto_grow``) or raises B200Error before anything changes.  A
        malformed row raises B200Error naming its stream; the other rows are applied."""
        self.drain()
        want = {n: (getattr(torch, dt), shape) for n, dt, shape in _lib.STATE_LAYOUT}
        if set(sd) != set(want):
            raise ValueError("load_state_dict: keys must be %s" % sorted(want))
        sd = {n: torch.as_tensor(v) for n, v in sd.items()}
        for n, (dt, _) in want.items():
            if sd[n].dtype != dt:
                raise TypeError("load_state_dict: %s must be %s, got %s" % (n, dt, sd[n].dtype))
        if sd["ids"].dim() != 2 or sd["bank"].dim() != 4:
            raise ValueError("load_state_dict: ids must be [R, cap] and bank [R, cap, hist_max, 128]")
        R, cap, H = sd["ids"].shape[0], sd["ids"].shape[1], sd["bank"].shape[2]
        if H != self.conf["hist_max"]:
            raise ValueError("load_state_dict: image hist_max %d, tracker hist_max %d" % (H, self.conf["hist_max"]))
        dims = dict(cap=cap, hist_max=H)
        for n, (_, shape) in want.items():
            if tuple(sd[n].shape) != (R,) + tuple(dims.get(k, k) for k in shape):
                raise ValueError("load_state_dict: %s has shape %s, inconsistent with ids %s" % (n, tuple(sd[n].shape), (R, cap)))
        if streams is None and R != self.S:
            raise ValueError("load_state_dict: %d rows for %d streams (pass streams=)" % (R, self.S))
        idx, dev_idx = self._stream_index(streams, "load_state_dict", distinct=True)
        if len(idx) != R:
            raise ValueError("load_state_dict: %d rows, %d stream indices" % (R, len(idx)))
        if R == 0:
            return
        n = sd["n_live"].cpu().numpy().astype(np.int64)
        if int(n.max()) > self.max_tracks:
            if not self.auto_grow:
                raise _lib.B200Error("load_state_dict: %d tracks exceed max_tracks=%d; construct the tracker with a "
                                     "larger max_tracks" % (int(n.max()), self.max_tracks))
            self.grow(max_tracks=max(int(n.max()), 2 * self.max_tracks))
        sd = {k: v.to(self.device).contiguous() for k, v in sd.items()}
        status = self._import(sd, dev_idx)
        ok = status == 0
        self.n_live[idx[ok]] = n[ok]
        bad = np.nonzero(~ok)[0]
        if len(bad):
            r = bad[0]
            raise _lib.B200Error("load_state_dict: stream %d not loaded: %s" % (
                idx[r], {_lib.EINVAL: "malformed image row", _lib.ECAPACITY: "more tracks than slots"}.get(
                    int(status[r]), "status %d" % status[r])))

    def import_state(self, stream: int, snap: Dict[str, np.ndarray]):
        """Inverse of ``export`` for one stream."""
        n = len(snap["ids"])
        c = lambda k, dt: np.ascontiguousarray(snap[k], dtype=dt)  # noqa: E731
        arrs = [c("ids", np.int32), c("x", np.float64), c("P", np.float64), c("stage", np.uint8), c("ema", np.float32),
                c("bank", np.float32), c("bank_len", np.int32), c("miss", np.int32), c("age", np.int32),
                c("last_bbox", np.float64), c("last_conf", np.float64), c("last_cost", np.float64)]
        with torch.cuda.device(self.device):
            rc = _lib.lib().b200_tracker_import(self._h, int(stream), n, *[a.ctypes.data_as(ctypes.c_void_p) for a in arrs],
                                                int(snap["next_id"]), _lib.stream_ptr(self.device))
        _lib.check(rc)
        self.n_live[stream] = n

    def close(self):
        """Frees the device state (b200_tracker_destroy)."""
        if getattr(self, "_h", None) is not None and self._h:
            _lib.lib().b200_tracker_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def reset(self, streams=None):
        """Back to the state of ``Tracking.__init__`` (mainTracking.py:45-96): no tracks, next id 0.  None: every
        stream; a list of distinct stream indices: only those (a camera's video ended and a new one starts in the same
        stream), the others untouched.  Asynchronous on the current stream."""
        if streams is None:
            with torch.cuda.device(self.device):
                _lib.check(_lib.lib().b200_tracker_reset(self._h, _lib.stream_ptr(self.device)))
            self.n_live[:] = 0
            return
        self.drain()
        idx, dev_idx = self._stream_index(streams, "reset", distinct=True)
        if len(idx):
            self._import(self._new_image(len(idx), 1), dev_idx, read_status=False)   # empty rows: cannot fail
            self.n_live[idx] = 0

    # -- one frame-step for every stream, host arrays in, host result table out -------------------
    def step(self, n_det, boxes, confs, embs, frame_ids) -> np.ndarray:
        """One ``Tracking.update`` (mainTracking.py:450-610) for every stream from host arrays padded to ``max_dets``:
        n_det [S], boxes [S,max_dets,4] float64 xyxy, confs [S,max_dets] float64, embs [S,max_dets,128] float32,
        frame_ids [S].  Returns the int32 result table [S, stride] (``decode`` turns a row into the reference's
        return value); raises ValueError where scipy would (NaN / infeasible cost matrix, hung.py:28)."""
        self.drain()                                   # earlier asynchronous steps first (their results stay on their handles)
        n_det, boxes, confs, embs, frame_ids = self._prepare(n_det, boxes, confs, embs, frame_ids, False)
        res = np.zeros((self.S, self.stride), dtype=np.int32)
        p = lambda a: a.ctypes.data_as(ctypes.c_void_p)  # noqa: E731
        with torch.cuda.device(self.device):           # synchronous entry point: copies and kernels on one stream
            rc = _lib.lib().b200_tracker_step_host(self._h, p(n_det), p(boxes), p(confs), p(embs), p(frame_ids), p(res),
                                                   _lib.stream_ptr(self.device))
        _lib.check(rc)
        err = self._read_result(res, current=True)
        if err is not None:
            raise err
        return res

    def step_async(self, n_det, boxes, confs, embs, frame_ids, *, pinned: bool = False) -> "StepHandle":
        """``step`` without the wait: uploads the detections, queues the step and the download of the result table on the
        current CUDA stream and returns at once; ``handle.result()`` blocks until THAT step is on the host and returns
        (or raises) exactly what ``step`` would.  The reference's consumer is a queue (tracking.py:329): a caller can
        queue frame t+1 before it looks at the result of frame t.  At most four steps may be pending; results must be
        collected in order.

        ``pinned=True``: ``boxes`` / ``confs`` / ``embs`` are page-locked arrays of the exact dtype and shape (numpy views
        of ``torch.empty(..., pin_memory=True)``, or tensors) that the caller leaves untouched until the result is
        collected; they are uploaded by DMA from where they are instead of through the handle's staging ring."""
        n_det, boxes, confs, embs, frame_ids = self._prepare(n_det, boxes, confs, embs, frame_ids, pinned)
        if len(self._pending) >= 4:
            raise _lib.B200Error("step_async: four steps are already pending; collect their results first")
        p = lambda a: a.ctypes.data_as(ctypes.c_void_p)  # noqa: E731
        ticket = ctypes.c_int64(-1)
        fn = _lib.lib().b200_tracker_step_pinned_async if pinned else _lib.lib().b200_tracker_step_host_async
        with torch.cuda.device(self.device):
            rc = fn(self._h, p(n_det), p(boxes), p(confs), p(embs), p(frame_ids), ctypes.byref(ticket),
                    _lib.stream_ptr(self.device))
        _lib.check(rc)
        h = StepHandle(self, int(ticket.value), np.maximum(n_det, 0).astype(np.int64))
        h._keep = (boxes, confs, embs) if pinned else None     # the DMA reads these after this call returns
        self._pending.append(h)
        self._pending_births = self._pending_births + h._births
        return h

    def _prepare(self, n_det, boxes, confs, embs, frame_ids, pinned):
        """Argument conversion and the capacity check shared by ``step`` and ``step_async``."""
        n_det = np.ascontiguousarray(n_det, dtype=np.int32).reshape(self.S)
        frame_ids = np.ascontiguousarray(frame_ids, dtype=np.int32).reshape(self.S)
        if pinned:
            arrs = []
            for a, dt, shape in ((boxes, np.float64, (self.S, self.max_dets, 4)), (confs, np.float64, (self.S, self.max_dets)),
                                 (embs, np.float32, (self.S, self.max_dets, 128))):
                a = a.numpy() if isinstance(a, torch.Tensor) else a
                if not (isinstance(a, np.ndarray) and a.dtype == dt and a.shape == shape and a.flags.c_contiguous):
                    raise TypeError("step_async(pinned=True): arrays must be C-contiguous %s of shape %s" % (np.dtype(dt), shape))
                arrs.append(a)
            boxes, confs, embs = arrs
        else:
            boxes = np.ascontiguousarray(boxes, dtype=np.float64).reshape(self.S, self.max_dets, 4)
            confs = np.ascontiguousarray(confs, dtype=np.float64).reshape(self.S, self.max_dets)
            embs = np.ascontiguousarray(embs, dtype=np.float32).reshape(self.S, self.max_dets, 128)
        self._reserve_tracks(n_det)
        return n_det, boxes, confs, embs, frame_ids

    def _reserve_tracks(self, n_det):
        """Grows the handle (raises with ``auto_grow=False``) unless live tracks + ``n_det`` fit in ``max_tracks``, where
        every pending step may have added all of its detections."""
        if self._n_live_stale:                         # device-side calls may have created tracks the host has not counted
            self.n_live_now()
        bound = self.n_live + self._pending_births + np.maximum(n_det, 0)
        while int(bound.max()) > self.max_tracks and self._pending:     # collect the oldest results until the bound fits
            self._pending[0]._collect()
            bound = self.n_live + self._pending_births + np.maximum(n_det, 0)
        if int(bound.max()) > self.max_tracks:         # the reference is unbounded: migrate to a larger handle
            if not self.auto_grow:
                raise _lib.B200Error("tracker capacity: live tracks + detections could exceed max_tracks=%d; "
                                     "construct the tracker with a larger max_tracks" % self.max_tracks)
            self.grow(max_tracks=max(int(bound.max()), 2 * self.max_tracks))

    def _read_result(self, res: np.ndarray, current: bool) -> Optional[Exception]:
        """Takes a collected result table (live counts, ``last_result``); returns the exception the step raises, or None."""
        self.n_live[:] = res[:, R_NLIVE]
        if current:                                    # nothing was queued after this step: the live counts are exact
            self._n_live_stale = False
        # A failing stream does not lose the others: the table (handle.table; last_result = the most recently collected
        # one) is complete before anything is raised, and the failing stream's state is what the reference leaves behind
        # when scipy raises (predict only).
        self.last_result = res
        bad = np.nonzero(res[:, R_STATUS])[0]
        if not len(bad):
            return None
        st = int(res[bad[0], R_STATUS])
        if st == _lib.ENUMERIC:
            return ValueError("matrix contains invalid numeric entries (stream %d)" % bad[0])
        if st == _lib.EINFEASIBLE:
            return ValueError("cost matrix is infeasible (stream %d)" % bad[0])
        if st == _lib.ECAPACITY:
            return _lib.B200Error(
                "tracker capacity exceeded on stream %d: births were dropped because live tracks + detections "
                "exceeded max_tracks=%d (device-side steps do not grow the handle; call grow() or construct with a "
                "larger max_tracks)" % (bad[0], self.max_tracks))
        return _lib.B200Error("tracker step failed on stream %d with status %d" % (bad[0], st))

    def drain(self):
        """Waits for every pending ``step_async`` (their results stay available on their handles)."""
        for h in list(self._pending):
            h._collect()

    # -- device-resident inputs, asynchronous on the current stream (no read-back) ------------------
    def step_device(self, n_det: torch.Tensor, boxes: torch.Tensor, confs: torch.Tensor, embs: torch.Tensor,
                    frame_ids: torch.Tensor, result: Optional[torch.Tensor] = None) -> torch.Tensor:
        """The same step with device-resident inputs, asynchronous on the current stream, no read-back (SURVEY 8f-1:
        the reference rebuilds host lists every frame, tracking.py:315-324).  The per-stream status is in column
        R_STATUS of the returned table."""
        for t, dt in ((n_det, torch.int32), (boxes, torch.float64), (confs, torch.float64), (embs, torch.float32),
                      (frame_ids, torch.int32)):
            _lib.require_cuda(t, "input")
            if t.dtype != dt or not t.is_contiguous():
                raise TypeError("step_device: wrong dtype or non-contiguous input")
        if result is None:
            result = torch.empty((self.S, self.stride), dtype=torch.int32, device=self.device)
        with torch.cuda.device(self.device):
            rc = _lib.lib().b200_tracker_step(self._h, _lib.ptr(n_det), _lib.ptr(boxes), _lib.ptr(confs), _lib.ptr(embs),
                                              _lib.ptr(frame_ids), _lib.ptr(result), _lib.stream_ptr(self.device))
        _lib.check(rc)
        self._n_live_stale = True
        return result

    def step_detections(self, boxes: torch.Tensor, confs: torch.Tensor, embs: torch.Tensor, frame_ids: torch.Tensor,
                        stream_index: Optional[torch.Tensor] = None, *, active: Optional[torch.Tensor] = None,
                        result: Optional[torch.Tensor] = None, track_of_det: Optional[torch.Tensor] = None):
        """``step_device`` fed with what a detector and an encoder produce, without the host round trip the reference
        makes (tracking.py:315-324) and without padding on the caller's side (b200_tracker_step_packed).

        ``boxes`` [K, >=4] (first four columns x1, y1, x2, y2) and ``confs`` [K]: float32 or float16, both the same;
        views such as ``dets[:, :4]`` and ``dets[:, 4]`` of the detector's [K, 6] rows are read in place.  ``embs``
        [K, 128] contiguous, float32 or float16.  ``stream_index`` int32 [K] (e.g. ROI Align's batch index), or None:
        every detection belongs to stream 0; a detection with an index outside [0, S) is ignored.  ``active`` int32 [S]
        or None: 0 leaves that stream idle this step (state untouched, like n_det = -1).  ``frame_ids`` int32 [S].
        All on the device.  Half values are widened exactly, so they give what ``update()`` gives for the same values.

        The j-th detection of stream s in input order is det_idx j of that stream in the result table.  Returns
        ``(result, track_of_det)``: the table ``step_device`` returns, and int32 [K] holding the track id each detection
        was matched to in this step, -1 otherwise.  Asynchronous on the current stream, no read-back, capturable in a
        CUDA graph.  A stream with more than ``max_dets`` detections is not stepped and gets ECAPACITY in its R_STATUS
        column (K <= max_dets rules that out); otherwise capacity is ``step_device``'s precondition."""
        if boxes.dim() != 2 or boxes.shape[1] < 4:
            raise ValueError("step_detections: boxes must be [K, >=4]")
        K = boxes.shape[0]
        if confs.dim() != 1 or confs.shape[0] != K or embs.dim() != 2 or embs.shape != (K, 128):
            raise ValueError("step_detections: confs must be [K] and embs [K, 128] for K = %d boxes" % K)
        if frame_ids.shape != (self.S,):
            raise ValueError("step_detections: frame_ids must be [%d]" % self.S)
        dtypes = {torch.float32: _lib.DTYPE_F32, torch.float16: _lib.DTYPE_F16}
        if boxes.dtype not in dtypes or confs.dtype != boxes.dtype or embs.dtype not in dtypes:
            raise TypeError("step_detections: boxes / confs must be float32 or float16 (the same), embs float32 or float16")
        if (K > 0 and (boxes.stride(1) != 1 or not embs.is_contiguous())) or (K > 1 and boxes.stride(0) < 4):
            raise TypeError("step_detections: boxes need unit column stride and embs must be contiguous")
        ints = [(frame_ids, "frame_ids")]
        if stream_index is not None:
            if stream_index.shape != (K,):
                raise ValueError("step_detections: stream_index must be [K]")
            ints.append((stream_index, "stream_index"))
        if active is not None:
            if active.shape != (self.S,):
                raise ValueError("step_detections: active must be [%d]" % self.S)
            ints.append((active, "active"))
        if result is None:
            result = torch.empty((self.S, self.stride), dtype=torch.int32, device=self.device)
        elif result.shape != (self.S, self.stride):
            raise ValueError("step_detections: result must be [%d, %d]" % (self.S, self.stride))
        if track_of_det is None:
            track_of_det = torch.empty((K,), dtype=torch.int32, device=self.device)
        elif track_of_det.shape != (K,):
            raise ValueError("step_detections: track_of_det must be [K]")
        ints += [(result, "result"), (track_of_det, "track_of_det")]
        for t, name in [(boxes, "boxes"), (confs, "confs"), (embs, "embs")] + ints:
            _lib.require_cuda(t, name)
        for t, name in ints:
            if t.dtype != torch.int32 or not t.is_contiguous():
                raise TypeError("step_detections: %s must be a contiguous int32 tensor" % name)
        box_stride = boxes.stride(0) if K > 1 else 4
        conf_stride = confs.stride(0) if K > 1 else 1
        with torch.cuda.device(self.device):
            rc = _lib.lib().b200_tracker_step_packed(
                self._h, K, _lib.ptr(boxes), box_stride, _lib.ptr(confs), conf_stride, dtypes[boxes.dtype], _lib.ptr(embs),
                dtypes[embs.dtype], _lib.ptr(stream_index), _lib.ptr(active), _lib.ptr(frame_ids), _lib.ptr(result),
                _lib.ptr(track_of_det), _lib.stream_ptr(self.device))
        _lib.check(rc)
        self._n_live_stale = True
        return result, track_of_det

    def decode(self, row: np.ndarray):
        """Result-table row -> (matches_tid, unmatched_track_ids, unmatched_dets) as Tracking.update returns."""
        MD, MT = self.max_dets, self.max_tracks
        nm, nut, nud = int(row[R_NMATCH]), int(row[R_NUT]), int(row[R_NUD])
        m = row[R_HDR:R_HDR + 2 * nm].reshape(nm, 2)
        ut = row[R_HDR + 2 * MD:R_HDR + 2 * MD + nut]
        ud = row[R_HDR + 2 * MD + MT:R_HDR + 2 * MD + MT + nud]
        return list(map(tuple, m.tolist())), ut.tolist(), ud.tolist()

    def export(self, stream: int = 0) -> Dict[str, np.ndarray]:
        """Copies one stream's live tracks (ascending track id) to host arrays."""
        MT, H = self.max_tracks, self.conf["hist_max"]
        out = dict(ids=np.zeros(MT, np.int32), x=np.zeros((MT, 8)), P=np.zeros((MT, 8, 8)), stage=np.zeros(MT, np.uint8),
                   ema=np.zeros((MT, 128), np.float32), bank=np.zeros((MT, H, 128), np.float32),
                   bank_len=np.zeros(MT, np.int32), miss=np.zeros(MT, np.int32), age=np.zeros(MT, np.int32),
                   last_bbox=np.zeros((MT, 4)), last_conf=np.zeros(MT), last_cost=np.zeros(MT))
        nxt = ctypes.c_int32(0)
        p = lambda a: a.ctypes.data_as(ctypes.c_void_p)  # noqa: E731
        with torch.cuda.device(self.device):
            n = _lib.lib().b200_tracker_export(
                self._h, int(stream), p(out["ids"]), p(out["x"]), p(out["P"]), p(out["stage"]), p(out["ema"]),
                p(out["bank"]), p(out["bank_len"]), p(out["miss"]), p(out["age"]), p(out["last_bbox"]),
                p(out["last_conf"]), p(out["last_cost"]), ctypes.byref(nxt), _lib.stream_ptr(self.device))
        if n < 0:
            _lib.check(n)
        out = {k: v[:n] for k, v in out.items()}
        out["next_id"] = int(nxt.value)
        return out


class StepHandle:
    """A queued ``MultiStreamTracker.step_async``; ``result()`` is what ``step`` would have returned."""

    def __init__(self, ms: MultiStreamTracker, ticket: int, births: np.ndarray):
        self._ms, self._ticket, self._births = ms, ticket, births
        self._res, self._error = None, None
        self.table = None                              # the step's result table once collected, also when result() raises

    def _collect(self):
        ms = self._ms
        if self._res is not None or self._error is not None:
            return
        if not ms._pending or ms._pending[0] is not self:
            for h in list(ms._pending):                # results come back in queue order
                if h is self:
                    break
                h._collect()
        res = np.zeros((ms.S, ms.stride), dtype=np.int32)
        with torch.cuda.device(ms.device):
            rc = _lib.lib().b200_tracker_step_result(ms._h, self._ticket, res.ctypes.data_as(ctypes.c_void_p))
        ms._pending.remove(self)
        ms._pending_births = ms._pending_births - self._births
        try:
            _lib.check(rc)
        except Exception as exc:                       # noqa: BLE001
            self._error = exc
            return
        self._res = self.table = res
        self._error = ms._read_result(res, current=False)

    def done(self) -> bool:
        return self._res is not None or self._error is not None

    def result(self) -> np.ndarray:
        self._collect()
        if self._error is not None:
            raise self._error
        return self._res


class TrackView:
    """Read-only host snapshot of one track (TrackState + TrackMemory, mainTracking.py:15-42)."""

    def __init__(self, snap, i):
        self.track_id = int(snap["ids"][i])
        self.miss_count = int(snap["miss"][i])
        self.age = int(snap["age"][i])
        self.state = "ACTIVE" if self.miss_count == 0 else "LOST"
        st = int(snap["stage"][i])
        self.x = snap["x"][i].reshape(8, 1) if st >= 2 else snap["x"][i].reshape(8, 1).astype(np.float32)
        self.P = snap["P"][i] if st >= 1 else snap["P"][i].astype(np.float32)
        self.encoder_feat = snap["ema"][i]
        n = int(snap["bank_len"][i])
        self.feat_historical = [snap["bank"][i, t] for t in range(n)]
        self.last_bbox = tuple(float(v) for v in snap["last_bbox"][i])
        self.last_conf = float(snap["last_conf"][i])
        c = float(snap["last_cost"][i])
        self.last_match_cost = None if np.isnan(c) else c


class Tracking:
    """Drop-in for the reference's ``Tracking`` (model/mainTracking.py:45).

    ``Tracking()`` reads ``model/conf/conf.yaml`` relative to the working directory exactly like the
    reference (:47); pass ``conf=`` (a tracker block) to skip the file.  ``max_tracks`` / ``max_dets``
    are initial capacities of the device-side state: like the reference the tracker is unbounded, a step
    that would not fit migrates the state into a larger handle first (``auto_grow=False`` raises instead).
    """

    def __init__(self, conf_path: str = "model/conf/conf.yaml", *, conf: Optional[Dict[str, Any]] = None,
                 max_tracks: int = 512, max_dets: int = 256, device=None, auto_grow: bool = True):
        if conf is None:
            full = load_conf(conf_path)
            if "tracker" not in full:
                raise KeyError("Missing 'tracker' section in YAML config.")
            conf = full["tracker"]
        self._ms = MultiStreamTracker(1, conf, max_tracks, max_dets, device, auto_grow)
        c = self._ms.conf
        for k, v in c.items():                       # same attribute names as the reference (:55-96)
            setattr(self, "tau" if k == "app_tau" else k, v)
        MD = self._ms.max_dets
        self._boxes = np.zeros((1, MD, 4), np.float64)
        self._confs = np.zeros((1, MD), np.float64)
        self._embs = np.zeros((1, MD, 128), np.float32)
        self._snap = None
        self._frame_dev = None                       # update_tensors: the frame id on the device

    @property
    def device(self):
        return self._ms.device

    # -- the call the pipeline makes (tracking.py:326) ---------------------------------------------
    def update(self, obj: Dict):
        """``Tracking.update`` (mainTracking.py:450-610): obj = {embs, bboxes, confs, input_hw, frame_id} ->
        (matches [(track_id, det_idx)], unmatched track ids, unmatched det indices), same order, same ValueErrors
        (:457-462, :267-268)."""
        det_embs = obj.get("embs", []) or []
        det_boxes = obj.get("bboxes", []) or []
        det_confs = obj.get("confs", []) or []
        input_hw = obj.get("input_hw", None)
        frame_id = obj.get("frame_id", None)
        if input_hw is None:
            raise ValueError("obj['input_hw'] is required")
        if frame_id is None:
            raise ValueError("obj['frame_id'] is required")
        if not (len(det_embs) == len(det_boxes) == len(det_confs)):
            raise ValueError("Length mismatch: embs/bboxes/confs must have same length")
        N = len(det_boxes)
        if N:
            try:                                   # equal-length vectors: one C-level conversion
                e = np.asarray(det_embs, dtype=np.float32).reshape(N, -1)
            except ValueError:                     # ragged input: per-vector conversion, then the reference's error
                e = None
            if e is None or e.shape[1] != 128:
                shapes = sorted({np.asarray(v).size for v in det_embs})
                raise ValueError(f"det_embs must be 128D, got sizes {shapes}")
            return self.update_arrays(np.asarray(det_boxes, dtype=np.float64), np.asarray(det_confs, dtype=np.float64),
                                      e, int(frame_id))
        return self.update_arrays(np.zeros((0, 4)), np.zeros((0,)), np.zeros((0, 128), np.float32), int(frame_id))

    def update_arrays(self, boxes: np.ndarray, confs: np.ndarray, embs: np.ndarray, frame_id: int):
        """Array form of ``update``: boxes [N,4] float64 xyxy, confs [N], embs [N,128] float32."""
        N = boxes.shape[0]
        self._reserve_dets(N)
        self._fit_buffers()
        self._boxes[0, :N] = boxes
        self._confs[0, :N] = confs
        self._embs[0, :N] = embs
        res = self._ms.step([N], self._boxes, self._confs, self._embs, [frame_id])
        self._snap = None
        return self._ms.decode(res[0])

    def update_tensors(self, boxes: torch.Tensor, confs: torch.Tensor, embs: torch.Tensor, frame_id: int):
        """``update`` fed from the detector's and the encoder's device tensors instead of host lists
        (tracking.py:315-324 copies them to the host): ``boxes`` [N, >=4] (e.g. ``dets[:, :4]`` of the detector's
        [N, 6] rows, read in place), ``confs`` [N] (e.g. ``dets[:, 4]``), both float32 or both float16, ``embs`` [N, 128]
        float32 or float16.  Returns what ``update`` returns for the same values, with the same errors and the same
        automatic growth; float16 inputs give exactly what ``update`` gives for their values, because both widen them
        exactly.  The inputs stay on the device; the only device -> host copy is the small result table."""
        ms = self._ms
        if boxes.dim() != 2 or confs.dim() != 1 or embs.dim() != 2 or not (boxes.shape[0] == confs.shape[0] == embs.shape[0]):
            raise ValueError("Length mismatch: embs/bboxes/confs must have same length")
        if embs.shape[1] != 128:
            raise ValueError(f"det_embs must be 128D, got sizes [{embs.shape[1]}]")
        N = boxes.shape[0]
        self._reserve_dets(N)
        ms._reserve_tracks([N])
        if self._frame_dev is None:
            self._frame_dev = torch.empty((1,), dtype=torch.int32, device=self.device)
        self._frame_dev.fill_(int(frame_id))
        table, _ = ms.step_detections(boxes, confs, embs, self._frame_dev)
        res = table.cpu().numpy()
        self._snap = None
        err = ms._read_result(res, current=True)
        if err is not None:
            raise err
        return ms.decode(res[0])

    def _fit_buffers(self):
        MD = self._ms.max_dets
        if self._boxes.shape[1] != MD:                 # the handle has grown (here or in one of the step-by-step methods)
            self._boxes, self._confs = np.zeros((1, MD, 4), np.float64), np.zeros((1, MD), np.float64)
            self._embs = np.zeros((1, MD, 128), np.float32)

    def state_dict(self) -> Dict[str, torch.Tensor]:
        """The tracker's state as device tensors (``MultiStreamTracker.state_dict`` of its one stream): ``torch.save`` it
        and ``load_state_dict`` it into a fresh ``Tracking`` to continue the video where it stopped."""
        return self._ms.state_dict()

    def load_state_dict(self, sd: Dict[str, torch.Tensor]):
        """Restores a ``state_dict`` (one row).  Hyper-parameters stay this tracker's own; ``hist_max`` must match."""
        self._snap = None
        self._ms.load_state_dict(sd)
        self._fit_buffers()

    def _reserve_dets(self, n: int):
        """Grows the handle's ``max_dets`` to hold ``n`` detections (raises instead with ``auto_grow=False``)."""
        if n > self._ms.max_dets:
            if not self._ms.auto_grow:
                raise ValueError("%d detections exceed max_dets=%d" % (n, self._ms.max_dets))
            self._ms.grow(max_dets=max(n, 2 * self._ms.max_dets))

    # -- the reference's methods one by one (mainTracking.py:340-448), on the device state -----------
    def _dets(self, det_embs, det_boxes, det_confs):
        n = len(det_boxes)
        if not (len(det_embs) == n == len(det_confs)):
            raise ValueError("Length mismatch: embs/bboxes/confs must have same length")
        if n > self._ms.max_dets:
            self._ms.grow(max_dets=max(n, 2 * self._ms.max_dets))
        e = np.zeros((n, 128), np.float32)
        for j, v in enumerate(det_embs):
            v = np.asarray(v, dtype=np.float32).reshape(-1)
            if v.shape[0] != 128:
                raise ValueError(f"emb must be shape (128,), got {v.shape}")
            e[j] = v
        return (n, np.ascontiguousarray(np.asarray(det_boxes, dtype=np.float64).reshape(n, 4)),
                np.ascontiguousarray(np.asarray(det_confs, dtype=np.float64).reshape(n)), e)

    def _op(self, name, *args):
        p = lambda a: a.ctypes.data_as(ctypes.c_void_p) if isinstance(a, np.ndarray) else a  # noqa: E731
        with torch.cuda.device(self.device):
            rc = getattr(_lib.lib(), name)(self._ms._h, 0, *[p(a) for a in args], _lib.stream_ptr(self.device))
        self._snap = None
        self._ms._n_live_stale = True
        return rc

    def predict_all(self):
        """mainTracking.py:340-345: Kalman predict of every track; ``last_bbox`` becomes the predicted box."""
        _lib.check(self._op("b200_tracker_predict_all"))

    def mark_missed(self, track_ids: List[int]):
        """mainTracking.py:347-355 (ids that are not live are skipped)."""
        ids = np.ascontiguousarray(np.asarray(list(track_ids), dtype=np.int32))
        _lib.check(self._op("b200_tracker_mark_missed", ids, len(ids)))

    def purge_dead(self):
        """mainTracking.py:357-360: drops tracks whose miss_count exceeds max_age."""
        _lib.check(self._op("b200_tracker_purge_dead"))

    def create_new_tracks(self, det_ids, det_embs, det_boxes, det_confs, frame_id):
        """mainTracking.py:362-373: one new track per listed detection with conf >= init_conf_min, ids in list order."""
        ids = np.ascontiguousarray(np.asarray(list(det_ids), dtype=np.int32))
        if len(ids) == 0:
            return
        n, boxes, confs, embs = self._dets(det_embs, det_boxes, det_confs)
        if int((confs[ids] >= self.init_conf_min).sum()) + int(self._ms.n_live_now()[0]) > self._ms.max_tracks:
            self._ms.grow(max_tracks=2 * self._ms.max_tracks + len(ids))
        rc = self._op("b200_tracker_create_tracks", ids, len(ids), boxes, confs, embs, n, int(frame_id))
        if rc < 0:
            _lib.check(rc)

    def update_matched(self, matches, row_to_tid, det_embs, det_boxes, det_confs, frame_id, C_total_np, *,
                       ema_alpha=0.9, conf_update_min=0.55, cost_update_max=50.0, maha_thr=9.49):
        """mainTracking.py:375-448: Kalman update + bookkeeping for every (row, det) match and, behind the
        confidence / cost / posterior-Mahalanobis gates, the EMA embedding and history-bank update."""
        matches = list(matches)
        if not matches:
            return
        try:
            tids = np.array([row_to_tid[r] for r, _ in matches], dtype=np.int32)
        except IndexError as exc:
            raise IndexError("update_matched: match row outside row_to_tid") from exc
        dets = np.array([j for _, j in matches], dtype=np.int32)
        C = np.asarray(C_total_np)
        costs = np.ascontiguousarray(np.array([C[r, j] for r, j in matches], dtype=np.float64).astype(np.float32))
        if not np.array_equal(costs.astype(np.float64), np.array([float(C[r, j]) for r, j in matches])):
            raise TypeError("update_matched: C_total_np must hold float32-representable costs (the reference passes float32)")
        n, boxes, confs, embs = self._dets(det_embs, det_boxes, det_confs)
        if len(dets) and (dets.min() < 0 or dets.max() >= n):
            raise IndexError("update_matched: detection index out of range")       # the reference: det_boxes[det_j] at :393
        rc = self._op("b200_tracker_update_matched", tids, dets, costs, len(matches), boxes, confs, embs, n, int(frame_id),
                      float(ema_alpha), float(conf_update_min), float(cost_update_max), float(maha_thr))
        _lib.check(rc, {_lib.EINVAL: KeyError})             # a track id that is not live: self.tracks[tid] at :390

    # -- state inspection ---------------------------------------------------------------------------
    def snapshot(self) -> Dict[str, np.ndarray]:
        """Host copy of the live tracks in ascending id order: the fields of TrackMemory / TrackState
        (mainTracking.py:15-42) plus the Kalman state."""
        if self._snap is None:
            self._snap = self._ms.export(0)
        return self._snap

    @property
    def tracks(self) -> Dict[int, TrackView]:
        """Read-only view shaped like the reference's ``self.tracks`` dict (mainTracking.py:45-46, :15-42)."""
        s = self.snapshot()
        return {int(s["ids"][i]): TrackView(s, i) for i in range(len(s["ids"]))}

    @property
    def next_id(self) -> int:
        """The id the next new track gets (mainTracking.py:371-372)."""
        return self.snapshot()["next_id"]

    def _rows(self, row_to_tid):
        s = self.snapshot()
        pos = {int(t): i for i, t in enumerate(s["ids"])}
        return s, [pos[int(t)] for t in row_to_tid]

    # -- operator-level queries over the device state (read-only) -----------------------------------
    @torch.no_grad()
    def build_C_app_topk(self, *, row_to_tid: List[int], det_embs: List[np.ndarray], device=None, topk: int = 5,
                         use_topk_mean: bool = True, fallback_to_ema: bool = True) -> torch.Tensor:
        """mainTracking.py:141-211."""
        M, N = len(row_to_tid), len(det_embs)
        if M == 0 or N == 0:
            return torch.zeros((M, N), device=self.device)
        s, rows = self._rows(row_to_tid)
        det = torch.from_numpy(np.stack([np.asarray(e, dtype=np.float32).reshape(-1) for e in det_embs])).to(self.device)
        bank = torch.from_numpy(s["bank"][rows]).to(self.device)
        lens = torch.from_numpy(s["bank_len"][rows]).to(self.device)
        fb = torch.from_numpy(s["ema"][rows]).to(self.device) if fallback_to_ema else None
        return cost_ops.app_cost_topk(bank, lens, det, topk=topk, use_topk_mean=use_topk_mean, fallback=fb)

    @torch.no_grad()
    def cal_cost(self, *, row_to_tid, det_embs, det_boxes, det_confs, input_hw, device=None, assign=None):
        """mainTracking.py:213-303."""
        s, rows = self._rows(row_to_tid)
        for e in det_embs:
            if np.asarray(e).reshape(-1).shape[0] != 128:
                raise ValueError("det_embs must be 128D")
        C_app = self.build_C_app_topk(row_to_tid=row_to_tid, det_embs=det_embs, topk=self.emb_top_k)
        return cost_ops.cal_cost(C_app=C_app, boxes_prev=s["last_bbox"][rows].tolist(), boxes_cur=det_boxes,
                                 input_hw=input_hw, conf_prev=s["last_conf"][rows].tolist(), conf_cur=det_confs,
                                 w_app=self.w_app, w_bbox=self.w_bbox, w_conf=self.w_conf, alpha=self.alpha,
                                 beta=self.beta, assign=assign, unmatch_cost=self.unmatch_cost)

    def apply_kalman_gating(self, C_total_np: np.ndarray, row_to_tid: List[int], det_boxes, *, maha_thr: float = 13.28,
                            INF: float = 1e9) -> np.ndarray:
        """mainTracking.py:306-338: gates ``C_total_np`` in place and returns it."""
        M, N = C_total_np.shape
        if M == 0 or N == 0:
            return C_total_np
        s, rows = self._rows(row_to_tid)
        bk = kalman_ops.BatchedKalman.__new__(kalman_ops.BatchedKalman)
        bk.device, bk.M = self.device, M
        bk.x = torch.from_numpy(s["x"][rows]).to(self.device)
        bk.P = torch.from_numpy(s["P"][rows]).to(self.device)
        bk.stage = torch.from_numpy(s["stage"][rows]).to(self.device)
        bk.r = torch.ones(4, dtype=torch.float32, device=self.device)
        d2 = bk.maha(det_boxes).cpu().numpy()
        C_total_np[d2 > float(maha_thr)] = float(INF)
        return C_total_np
