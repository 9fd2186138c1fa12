"""Drop-in for the reference's pipelines.py: nst() (8-110) and mask_and_crop_iris() (112-166).

nst() keeps the reference signature and return structure.  The closure evaluation (VGG-19 forward,
losses, backward to the image) is ONE call of libisx's fused driver and the L-BFGS iteration is one
call of isx_lbfgs_tick; all optimiser scalars stay on the device, so the loop runs without host
synchronisation except one flag read-back every `max_iter` evaluations."""
from __future__ import annotations

import ctypes
import math
import numbers
from typing import List, Optional, Sequence, Tuple, Union

import torch

from . import _lib
from .engine import (CONV_LEVEL, LbfgsConfig, NstEngine, gram_of, mask_pyramid, masked_gram_of, masked_stats_of,
                     stats_of)
from .vgg import VGG19

last_info: dict = {}


def _prep_images(img: torch.Tensor, device) -> Tuple[torch.Tensor, bool]:
    unbatched = img.dim() == 3
    if unbatched:
        img = img[None]
    return img.detach().to(device, torch.float32).contiguous(), unbatched


def _norm_mask(mask: torch.Tensor, B: int, H: int, W: int, name: str, dev) -> torch.Tensor:
    """Mask argument -> [Bm,H,W] on the device with Bm in {1, B}; anything else is a ValueError (never a silent
    broadcast).  Accepted: (H,W), (Bm,H,W), (Bm,1,H,W)."""
    m = mask.to(dev)
    if m.dim() == 2:
        m = m[None]
    elif m.dim() == 4:
        if m.shape[1] != 1:
            raise ValueError("%s must have one channel, got shape %s" % (name, tuple(mask.shape)))
        m = m[:, 0]
    elif m.dim() != 3:
        raise ValueError("%s must be (H,W), (B,H,W) or (B,1,H,W), got shape %s" % (name, tuple(mask.shape)))
    if m.shape[0] not in (1, B) or tuple(m.shape[-2:]) != (H, W):
        raise ValueError("%s of shape %s does not match a batch of %d %dx%d images (batch must be 1 or %d)"
                         % (name, tuple(mask.shape), B, H, W, B))
    return m


def _is_scalar(w) -> bool:
    return isinstance(w, numbers.Real) or (torch.is_tensor(w) and w.dim() == 0)


def _problem_layout(c_img, s_img, c_loss_weight, s_loss_weight, independent, problem_size, streams):
    """Images per problem g of an nst() call, or None for the two layouts without per-problem weights (the whole batch
    as one problem, or one problem per image with `independent`).  Checks everything on the host, before any device
    work: B % g, the weight vector lengths (P = B / g), the style batch (1, P or B) and the option combinations."""
    B = c_img.shape[0] if c_img.dim() == 4 else 1
    vectors = not (_is_scalar(c_loss_weight) and _is_scalar(s_loss_weight))
    if problem_size is None:
        if not vectors:
            return None
        g = 1 if independent else B       # a weight vector with the default layouts: one weight per problem
    else:
        g = int(problem_size)
        if g < 1 or g != problem_size or B % g:
            raise ValueError("problem_size %r must divide the batch of %d images" % (problem_size, B))
        if independent and g > 1:
            raise ValueError("independent=True means problem_size=1, got problem_size=%d" % g)
    P = B // g
    for name, w in (("c_loss_weight", c_loss_weight), ("s_loss_weight", s_loss_weight)):
        if not _is_scalar(w):
            t = torch.as_tensor(w)
            if t.dim() != 1 or t.numel() != P:
                raise ValueError("%s must be a scalar or a 1-D sequence of %d weights (one per problem), got shape %s"
                                 % (name, P, tuple(t.shape)))
    Bs = s_img.shape[0] if s_img.dim() == 4 else 1
    if Bs not in (1, P, B):
        raise ValueError("style batch %d must be 1, %d (one per problem) or %d (one per image)" % (Bs, P, B))
    if streams > 1 and g > 1:
        raise ValueError("streams > 1 needs one problem per image; problem_size=%d couples %d images" % (g, g))
    return g


def _ranged_layout(c_img, s_img, c_loss_weight, s_loss_weight, independent, problem_size, problem_sizes, streams):
    """The problem sizes (g_0, ..., g_{P-1}) of an nst(problem_sizes=...) call as a list of ints.  Checks everything on the
    host, before any device work: every g_p an integer >= 1, their sum B, the weight vector lengths (P), the style batch
    (1, P or B) and the options that cannot be combined with it."""
    B = c_img.shape[0] if c_img.dim() == 4 else 1
    if problem_size is not None:
        raise ValueError("pass problem_size (equal problems) or problem_sizes, not both")
    if independent:
        raise ValueError("independent=True is problem_sizes=[1] * B; it cannot be combined with problem_sizes")
    if streams > 1:
        raise ValueError("streams > 1 needs one problem per image; it cannot be combined with problem_sizes")
    sizes = list(problem_sizes.tolist() if torch.is_tensor(problem_sizes) else problem_sizes)
    for g in sizes:
        if isinstance(g, bool) or not isinstance(g, numbers.Integral) or g < 1:
            raise ValueError("problem_sizes must be integers >= 1, got %r" % (sizes,))
    sizes = [int(g) for g in sizes]
    if sum(sizes) != B:
        raise ValueError("problem_sizes %r sum to %d, not to the batch of %d images" % (sizes, sum(sizes), B))
    P = len(sizes)
    for name, w in (("c_loss_weight", c_loss_weight), ("s_loss_weight", s_loss_weight)):
        if not _is_scalar(w):
            t = torch.as_tensor(w)
            if t.dim() != 1 or t.numel() != P:
                raise ValueError("%s must be a scalar or a 1-D sequence of %d weights (one per problem), got shape %s"
                                 % (name, P, tuple(t.shape)))
    Bs = s_img.shape[0] if s_img.dim() == 4 else 1
    if Bs not in (1, P, B):
        raise ValueError("style batch %d must be 1, %d (one per problem) or %d (one per image)" % (Bs, P, B))
    return sizes


def _weight_vector(w, P: int, dev) -> torch.Tensor:
    """alpha or beta as a device float64 [P] tensor (a scalar is the same weight for every problem)."""
    if _is_scalar(w):
        return torch.full((P,), float(w), device=dev, dtype=torch.float64)
    return torch.as_tensor(w).detach().to(dev, torch.float64).reshape(P).contiguous()


class NstJob:
    """Device-resident state of one nst() call: targets, L-BFGS buffers, the evaluation engine.
    `tick()` = one closure evaluation (pipelines.py:80-101) + one L-BFGS iteration for the whole batch.
    problem_size g (validated by _problem_layout): B / g coupled problems with per-problem weights; None: one problem,
    or one per image with `independent`, with scalar weights.  problem_sizes (validated by _ranged_layout): problems of
    those sizes, one after the other, with per-problem weights."""

    def __init__(self, c_img, s_img, vgg, dev, clone_content=True, BN_loss=True, c_loss_weight=1.0,
                 s_loss_weight=1.0, lr=1.0, epochs=200, independent=False, history_size=100, x_init=None,
                 history_dtype=torch.float32, c_mask=None, s_mask=None, lbfgs_stream=None, problem_size=None,
                 problem_sizes=None):
        c_img, c_unbatched = _prep_images(c_img, dev)
        # optional second stream for the L-BFGS passes of every tick (NstJobGroup: a low-priority stream, so that the
        # HBM-bound history passes of this sub-batch run beside the tensor-bound convolutions of another one)
        self.aux = lbfgs_stream
        self._lbfgs_done = None
        s_img, s_unbatched = _prep_images(s_img, dev)
        self.c_unbatched = c_unbatched
        if clone_content:
            x = c_img.clone()
        elif x_init is not None:
            x = x_init.detach().to(dev, torch.float32).clone()
        else:
            x = torch.rand(c_img.shape).to(dev)  # pipelines.py:54
        self.x = x.contiguous()
        B, xc, H, W = self.x.shape
        packed = vgg.packed(dev)
        cc, sc = vgg.content_convs, vgg.style_convs
        self.independent = independent
        self.epochs = int(epochs)
        ranged = problem_sizes is not None
        problems = problem_size is not None or ranged
        P = len(problem_sizes) if ranged else B // problem_size if problems else (B if independent else 1)
        if problems:   # the weights live on the device; the scalar weights of the configs are not read
            self.c_w, self.s_w = _weight_vector(c_loss_weight, P, dev), _weight_vector(s_loss_weight, P, dev)
            c_loss_weight = s_loss_weight = math.nan

        # ---- targets (pipelines.py:62-68) ----
        levels = [CONV_LEVEL[i] for i in sc]
        cmask_b = 0
        if c_mask is not None:
            c_mask = _norm_mask(c_mask, B, H, W, "c_mask", dev)
            cmask_b = c_mask.shape[0]
        # an UNBATCHED content image (the notebook's call) makes utils.GramMatrix divide the prediction's Gram by H*W
        # only (utils.py:253-254); the target keeps its own normaliser (s_unbatched below), exactly like the reference
        eng = NstEngine(packed, B, H, W, xc, cc, sc, style_mode=1 if BN_loss else 0, c_weight=c_loss_weight,
                        s_weight=s_loss_weight, coupled=not independent, style_mask_b=cmask_b,
                        pred_unbatched=c_unbatched)
        if ranged:
            eng.set_problem_ranges([sum(problem_sizes[:p]) for p in range(P + 1)], self.c_w, self.s_w)
        elif problems:
            eng.set_problems(B // P, self.c_w, self.s_w)
        if cmask_b:
            eng.set_style_masks(mask_pyramid(c_mask, levels))
        eng.forward(c_img)
        eng.set_content_targets([eng.tap(i) for i in cc])
        Bs, xs, Hs, Ws = s_img.shape
        if (Bs, xs, Hs, Ws) == (B, xc, H, W):
            eng.forward(s_img)
            s_feats = [eng.tap_view(i) for i in sc]   # consumed below, before the engine runs again
        else:
            if Bs not in ((1, P, B) if problems else (1, B)):
                raise ValueError("style batch %d must be 1 or %d" % (Bs, B))
            seng = NstEngine(packed, Bs, Hs, Ws, xs, cc, sc)
            seng.forward(s_img)
            s_feats = [seng.tap_view(i) for i in sc]
        if BN_loss:
            if s_mask is not None:  # mask-weighted BN loss: targets are the statistics of the style features times the style's mask
                s_mask = _norm_mask(s_mask, Bs, Hs, Ws, "s_mask", dev)
                st = [masked_stats_of(f, m) for f, m in zip(s_feats, mask_pyramid(s_mask, levels))]
            else:
                st = [stats_of(f) for f in s_feats]
            eng.set_bn_targets([m for m, _ in st], [s for _, s in st])
        else:
            # unbatched style image (…2020.py:103-104): GramMatrix divides by H*W only (SURVEY note N3)
            inv = [1.0 / (f.shape[1] * f.shape[2]) if s_unbatched else None for f in s_feats]
            if s_mask is not None:  # row G': targets are Gram matrices of the style features weighted by the style's mask
                s_mask = _norm_mask(s_mask, Bs, Hs, Ws, "s_mask", dev)
                eng.set_gram_targets([masked_gram_of(f, m, n) for f, m, n in zip(s_feats, mask_pyramid(s_mask, levels), inv)])
            else:
                eng.set_gram_targets([gram_of(f, n) for f, n in zip(s_feats, inv)])
        del s_feats
        seng = None
        self.eng = eng

        # ---- optimiser (pipelines.py:59): torch.optim.LBFGS([x], lr) defaults ----
        self.problems, self.ranged = problems, ranged
        self.n_img = xc * H * W
        # N: floats of the largest problem (the grid and the scratch of the L-BFGS passes)
        self.P, self.ipp, self.N = P, B // P, (max(problem_sizes) * self.n_img if ranged else self.x.numel() // P)
        # one (y, s) pair per iteration, so a short job never needs all 100 slots
        hist = max(1, min(int(history_size), self.epochs + 20))
        if history_dtype not in (torch.float32, torch.bfloat16):
            raise ValueError("history_dtype must be torch.float32 (reference) or torch.bfloat16")
        self.cfg = LbfgsConfig(epochs=self.epochs, max_iter=20, max_eval=25, history=hist,
                               history_bf16=int(history_dtype == torch.bfloat16), reserved_=0, lr=float(lr),
                               tolerance_grad=1e-7, tolerance_change=1e-9, c_weight=float(c_loss_weight),
                               s_weight=float(s_loss_weight))
        self.max_ticks = self.epochs + 20
        M1 = hist + 1
        N = self.N
        self.state = torch.empty(_lib.call_i64("isx_lbfgs_state_bytes", P), device=dev, dtype=torch.uint8)
        self.mats = torch.zeros(_lib.call_i64("isx_lbfgs_mats_bytes", P, hist), device=dev, dtype=torch.uint8)
        self.scratch = torch.empty(_lib.call_i64("isx_lbfgs_scratch_bytes", P, _lib.i64(N), hist), device=dev,
                                   dtype=torch.uint8)
        if ranged:   # problem p's block starts at M1 * first_p * n_img: with equal sizes the (P, M1, N) layout below
            self.Sh = torch.empty(M1 * B * self.n_img, device=dev, dtype=history_dtype)
            self.Yh = torch.empty(M1 * B * self.n_img, device=dev, dtype=history_dtype)
        else:
            self.Sh = torch.empty(P, M1, N, device=dev, dtype=history_dtype)
            self.Yh = torch.empty(P, M1, N, device=dev, dtype=history_dtype)
        self.grad = torch.empty_like(self.x)
        self.grad_prev = torch.empty_like(self.x)
        self.hist_c = torch.zeros(self.max_ticks, P, device=dev, dtype=torch.float64)
        self.hist_s = torch.zeros(self.max_ticks, P, device=dev, dtype=torch.float64)
        self.done = torch.zeros(P, device=dev, dtype=torch.int32)
        self.ticks = 0
        self._graph = None
        _lib.call("isx_lbfgs_init", self.state, P, _lib.stream_ptr())
        _lib.call("isx_clamp01", self.x, _lib.i64(self.x.numel()), _lib.stream_ptr())  # pipelines.py:82 (first closure)

    def _lbfgs(self):
        if self.ranged:
            _lib.call("isx_lbfgs_tick_ranges", self.x, self.grad, self.grad_prev, self.Sh, self.Yh, self.state, self.mats,
                      self.scratch, self.eng.loss_c, self.eng.loss_s, ctypes.byref(self.eng.ranges), self.x.shape[0],
                      _lib.i64(self.n_img), ctypes.byref(self.cfg), self.hist_c, self.hist_s, self.ticks,
                      _lib.stream_ptr())
            return
        if self.problems:
            _lib.call("isx_lbfgs_tick_problems", self.x, self.grad, self.grad_prev, self.Sh, self.Yh, self.state, self.mats,
                      self.scratch, self.eng.loss_c, self.eng.loss_s, self.ipp, self.P, _lib.i64(self.N),
                      ctypes.byref(self.cfg), self.c_w, self.s_w, self.hist_c, self.hist_s, self.ticks, _lib.stream_ptr())
            return
        _lib.call("isx_lbfgs_tick", self.x, self.grad, self.grad_prev, self.Sh, self.Yh, self.state, self.mats,
                  self.scratch, self.eng.loss_c, self.eng.loss_s, self.ipp, self.P, _lib.i64(self.N),
                  ctypes.byref(self.cfg), self.hist_c, self.hist_s, self.ticks, _lib.stream_ptr())

    def _tick_body(self):
        self.eng.eval(self.x, self.grad)
        self._lbfgs()

    def sync_lbfgs(self):
        """Make the current stream wait for the L-BFGS passes issued on the auxiliary stream (no-op without one)."""
        if self._lbfgs_done is not None:
            torch.cuda.current_stream().wait_event(self._lbfgs_done)

    def tick(self):
        if self._graph is not None:
            self._graph.replay()
        elif self.aux is None:
            self._tick_body()
        else:
            main = torch.cuda.current_stream()
            self.sync_lbfgs()                      # x of this evaluation = the previous tick's update
            self.eng.eval(self.x, self.grad)
            ev = torch.cuda.Event()
            ev.record(main)
            with torch.cuda.stream(self.aux):
                self.aux.wait_event(ev)
                self._lbfgs()
                self._lbfgs_done = torch.cuda.Event()
                self._lbfgs_done.record(self.aux)
        self.ticks += 1

    def enable_graph(self):
        """Capture one tick (~45 kernel launches, all parameters tick-invariant, no host synchronisation) in a CUDA
        graph and replay it from then on -- removes the launch gaps that dominate small batches."""
        if self._graph is not None:
            return
        self.tick()  # eager first tick: function attributes, driver entry points, allocator warm-up
        torch.cuda.current_stream().synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            self._tick_body()
        self._graph = g

    def evals_done(self):
        """Per-problem evaluation counts (0 while a problem is still running); one small D2H read."""
        self.sync_lbfgs()
        _lib.call("isx_lbfgs_done_flags", self.state, self.P, self.done, _lib.stream_ptr())
        return self.done.cpu()

    def history_counts(self):
        """Per-problem number of (y, s) pairs currently in the L-BFGS ring (one small D2H read)."""
        out = torch.zeros(self.P, device=self.x.device, dtype=torch.int32)
        self.sync_lbfgs()
        _lib.call("isx_lbfgs_history_counts", self.state, self.P, out, _lib.stream_ptr())
        return out.cpu()

    def finish(self):
        evals = self.evals_done()      # (waits for the auxiliary stream)
        n_evals = int(evals.max().item()) if bool((evals > 0).all().item()) else self.ticks
        hc = self.hist_c[:n_evals].cpu()
        hs = self.hist_s[:n_evals].cpu()
        for p_, e_ in enumerate(evals.tolist()):  # a problem that finished early keeps its last logged losses
            if 0 < e_ < n_evals:
                hc[e_:, p_] = hc[e_ - 1, p_]
                hs[e_:, p_] = hs[e_ - 1, p_]
        x = self.x.detach()
        _lib.call("isx_clamp01", x, _lib.i64(x.numel()), _lib.stream_ptr())  # pipelines.py:108-109
        return x, n_evals, evals, hc, hs


class NstJobGroup:
    """`streams` sub-batches of an independent-problems job, each an NstJob on its own CUDA stream.  Ticks of the
    sub-jobs are issued round-robin, so the HBM-bound L-BFGS passes of one sub-batch overlap the tensor-core
    convolutions of another (the two kernel families stress different units)."""

    def __init__(self, c_img, s_img, vgg, dev, streams=2, overlap=False, **kw):
        if not kw.get("independent", False):
            raise ValueError("multi-stream execution needs independent=True (one problem per image)")
        B = c_img.shape[0]
        n = max(1, min(int(streams), B))
        bounds = [(B * i) // n for i in range(n + 1)]
        main = torch.cuda.current_stream(dev)
        # overlap: evaluations on HIGH-priority streams, the L-BFGS passes of each sub-batch on its own LOW-priority
        # stream; with isx_set_option("smem_reserve_kb") the streaming CTAs are resident beside the persistent conv CTAs
        self.streams = [torch.cuda.Stream(dev, priority=-1 if overlap else 0) for _ in range(n)]
        self.aux = [torch.cuda.Stream(dev, priority=0) if overlap else None for _ in range(n)]
        self.jobs: List[NstJob] = []
        x_init = kw.pop("x_init", None)
        c_mask, s_mask = kw.pop("c_mask", None), kw.pop("s_mask", None)
        s_batched = s_img.dim() == 4 and s_img.shape[0] == B and B > 1

        def part(m, lo, hi, batched):  # per-image masks follow their images into the sub-batch
            if m is None or m.dim() < 3 or m.shape[0] == 1 or not batched:
                return m
            return m[lo:hi]

        weights = {k: kw.pop(k) for k in ("c_loss_weight", "s_loss_weight") if k in kw}

        for i, st in enumerate(self.streams):
            lo, hi = bounds[i], bounds[i + 1]
            st.wait_stream(main)
            with torch.cuda.stream(st):
                si = s_img[lo:hi] if s_batched else s_img
                xi = x_init[lo:hi] if x_init is not None else None
                wi = {k: w if _is_scalar(w) else w[lo:hi] for k, w in weights.items()}   # per-image weights follow their images
                self.jobs.append(NstJob(c_img[lo:hi], si, vgg, dev, x_init=xi, c_mask=part(c_mask, lo, hi, True),
                                        s_mask=part(s_mask, lo, hi, s_batched), lbfgs_stream=self.aux[i], **wi, **kw))
        self.max_ticks = self.jobs[0].max_ticks
        self.epochs = self.jobs[0].epochs
        self.P = B

    @property
    def ticks(self):
        return self.jobs[0].ticks

    def tick(self):
        for job, st in zip(self.jobs, self.streams):
            with torch.cuda.stream(st):
                job.tick()

    def join(self, dev):
        main = torch.cuda.current_stream(dev)
        for st, ax in zip(self.streams, self.aux):
            main.wait_stream(st)
            if ax is not None:
                main.wait_stream(ax)

    def fork(self, dev):
        main = torch.cuda.current_stream(dev)
        for st, ax in zip(self.streams, self.aux):
            st.wait_stream(main)
            if ax is not None:
                ax.wait_stream(main)

    def evals_done(self):
        outs = []
        for job, st in zip(self.jobs, self.streams):
            with torch.cuda.stream(st):
                outs.append(job.evals_done())
        return torch.cat(outs)

    def finish(self):
        xs, hcs, hss, evs = [], [], [], []
        n_evals = 0
        for job, st in zip(self.jobs, self.streams):
            with torch.cuda.stream(st):
                x, n, ev, hc, hs = job.finish()
            xs.append(x); evs.append(ev); hcs.append(hc); hss.append(hs)
            n_evals = max(n_evals, n)
        pad = lambda h: torch.cat([h, h[-1:].expand(n_evals - h.shape[0], -1)]) if h.shape[0] < n_evals else h
        dev = xs[0].device
        self.join(dev)
        return (torch.cat(xs), n_evals, torch.cat(evs), torch.cat([pad(h) for h in hcs], dim=1),
                torch.cat([pad(h) for h in hss], dim=1))


class _HistoryWriter:
    """x_hist without stalling the optimisation loop (SURVEY K11; the reference does a blocking
    `x.detach().cpu()` per evaluation, pipelines.py:93).  Per kept evaluation: a device-to-device snapshot of x on
    the compute stream (x is overwritten by the L-BFGS update of the same tick), then a device-to-host copy on a
    side stream, ordered by events only -- the host never synchronises inside the loop.
      * small histories (<= ISX_XHIST_PINNED_GB, default 8 GiB in total): every entry is its own pinned host tensor
        (torch's caching host allocator recycles the blocks across calls) and is the D2H destination;
      * larger ones: a ring of pinned slots drained into ordinary (pageable) tensors by a worker thread.
    `finish()` is the only synchronisation point."""

    SLOTS = 3

    def __init__(self, shape, n_entries, dev):
        import os
        import threading

        self.dev, self.shape = dev, tuple(shape)
        nbytes = 4
        for d in self.shape:
            nbytes *= d
        limit = float(os.environ.get("ISX_XHIST_PINNED_GB", "8")) * (1 << 30)
        self.direct = nbytes * max(1, n_entries) <= limit
        self.copy_stream = torch.cuda.Stream(dev)
        self.dslots = [torch.empty(self.shape, device=dev, dtype=torch.float32) for _ in range(self.SLOTS)]
        self.d2h_done = [None] * self.SLOTS          # event on copy_stream: device slot j may be overwritten
        self.entries = []
        self.k = 0
        if not self.direct:
            self.pslots = [torch.empty(self.shape, dtype=torch.float32).pin_memory() for _ in range(self.SLOTS)]
            self.free = [threading.Event() for _ in range(self.SLOTS)]
            for f in self.free:
                f.set()
            self.queue = []
            self.cv = threading.Condition()
            self.closed = False
            self.error = None
            self.worker = threading.Thread(target=self._drain, daemon=True)
            self.worker.start()

    def _drain(self):
        try:
            while True:
                with self.cv:
                    while not self.queue and not self.closed:
                        self.cv.wait()
                    if not self.queue:
                        return
                    j, ev, dst = self.queue.pop(0)
                ev.synchronize()
                dst.copy_(self.pslots[j])
                self.free[j].set()
        except Exception as e:  # surfaced by finish()
            self.error = e
            for f in self.free:
                f.set()

    def snapshot(self, x: torch.Tensor):
        """Record the current x (called on the compute stream right before the evaluation that consumes it)."""
        j = self.k % self.SLOTS
        self.k += 1
        main = torch.cuda.current_stream(self.dev)
        if self.d2h_done[j] is not None:
            main.wait_event(self.d2h_done[j])
        self.dslots[j].copy_(x.view(self.shape), non_blocking=True)
        snap = torch.cuda.Event()
        snap.record(main)
        if self.direct:
            dst = torch.empty(self.shape, dtype=torch.float32, pin_memory=True)
        else:
            self.free[j].wait()       # back-pressure only when the host drains slower than the GPU produces
            if self.error is not None:
                raise self.error
            self.free[j].clear()
            dst = self.pslots[j]
        with torch.cuda.stream(self.copy_stream):
            self.copy_stream.wait_event(snap)
            dst.copy_(self.dslots[j], non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(self.copy_stream)
        self.d2h_done[j] = ev
        if self.direct:
            self.entries.append(dst)
        else:
            out = torch.empty(self.shape, dtype=torch.float32)
            self.entries.append(out)
            with self.cv:
                self.queue.append((j, ev, out))
                self.cv.notify()

    def finish(self, keep: int):
        self.copy_stream.synchronize()
        if not self.direct:
            with self.cv:
                self.closed = True
                self.cv.notify()
            self.worker.join()
            if self.error is not None:
                raise self.error
        return self.entries[:keep]


def nst(c_img: torch.Tensor,
        s_img: torch.Tensor,
        clone_content: bool = True,
        BN_loss: bool = True,
        c_loss_weight: Union[float, Sequence[float], torch.Tensor] = 1,
        s_loss_weight: Union[float, Sequence[float], torch.Tensor] = 1,
        lr: float = 1,
        epochs: int = 200,
        vgg: torch.nn.Module = None,
        use_tqdm: bool = True,
        device: str = 'cuda:0',
        *,
        independent: bool = False,
        x_hist_stride: int = 1,
        history_size: int = 100,
        x_init: Optional[torch.Tensor] = None,
        history_dtype: torch.dtype = torch.float32,
        streams: int = 1,
        overlap: bool = False,
        cuda_graph: Optional[bool] = None,
        c_mask: Optional[torch.Tensor] = None,
        s_mask: Optional[torch.Tensor] = None,
        problem_size: Optional[int] = None,
        problem_sizes: Optional[Sequence[int]] = None,
        ) -> tuple[torch.Tensor, list, list, list]:
    """Neural style transfer pipeline (pipelines.py:8-110).

    Reference arguments and returns are unchanged.  Extensions (keyword-only):
      independent   False: the batch is ONE L-BFGS problem exactly like the reference (shared history,
                    content loss averaged over the batch, SURVEY.md F6).  True: every image is its own
                    problem (== calling the reference once per image with B=1); this is what shards.
      problem_size  g: the batch is B / g problems, images [p*g, (p+1)*g) forming problem p, each exactly the
                    reference's nst() on those g images (content loss averaged over them, style loss summed, its own
                    L-BFGS history and exit tests), all advancing in one device job.  c_loss_weight / s_loss_weight may
                    then be sequences or 1-D tensors of P = B / g weights (a scalar = the same for every problem; a
                    weight sequence without problem_size means one weight per problem of the default layout).  The
                    style batch is 1 (shared), P (one per problem) or B (one per image).  problem_size=B is the
                    default layout, problem_size=1 is independent=True; independent=True with problem_size > 1 and
                    streams > 1 with problem_size > 1 raise ValueError.
      problem_sizes (g_0, ..., g_{P-1}), integers >= 1 summing to B: problems of unequal size, problem p being the images
                    [g_0 + ... + g_{p-1}, g_0 + ... + g_p), each exactly the reference's nst() on its images, like
                    problem_size (weights, style batch 1 / P / B and outputs as there).  [g] * P is problem_size=g, [B]
                    the default layout and [1] * B independent=True, bit for bit.  It cannot be combined with
                    problem_size, independent=True or streams > 1 (ValueError).
      x_hist_stride keep every k-th evaluated image in x_hist (1 = reference behaviour, 0 = none).
      history_size  L-BFGS history (torch default 100).
      x_init        replaces torch.rand (pipelines.py:54) when clone_content is False.
      streams       > 1 (with independent=True): split the batch into that many sub-batches on separate CUDA
                    streams so L-BFGS passes (HBM-bound) overlap convolutions (tensor-bound) of another sub-batch.
      overlap       (with streams > 1) run each sub-batch's L-BFGS passes on a low-priority stream of its own so that they are
                    resident beside the persistent conv CTAs of the other sub-batches (needs the conv kernels to leave some
                    shared memory free: _lib.call("isx_set_option", b"smem_reserve_kb", 16)).
      c_mask/s_mask iris masks [B|1,1,H,W] of the content / style frames: the style loss then compares the statistics of the
                    MASK-WEIGHTED features F * m_l -- GramMatrix(F * m_l) or, with BN_loss, mean / std of F * m_l --, m_l = the
                    mask average-pooled to layer l (row G' of SURVEY.md §8a; the reference only has the dormant hooks
                    vgg.py:84-85 / pipelines.py:83).  All-ones masks == the plain losses.
      cuda_graph    replay each tick from a captured CUDA graph.  Off by default: a tick has no host synchronisation,
                    so eager launches already queue ahead of the GPU; capture + instantiation (~0.25 s) only pays off
                    for very long single-image jobs (measured, profiles/r01_README.md).
      history_dtype torch.float32 (the reference's optimiser state) or torch.bfloat16: the (s, y) history is then
                    stored in bf16, halving the HBM traffic and footprint of the L-BFGS passes (opt-in).
    c_loss_hist / s_loss_hist hold one float per closure evaluation, aggregated over the batch the way
    the reference's batched losses are (content: mean over images, style: sum over images); per-image
    values are left in `pipelines.last_info`.  With several problems the histories are the mean (content) and the sum
    (style) over problems, and last_info['c_loss_per_problem'] / ['s_loss_per_problem'] ([evals, P]) hold each
    problem's own."""
    if problem_sizes is not None:
        problem_sizes = _ranged_layout(c_img, s_img, c_loss_weight, s_loss_weight, independent, problem_size,
                                       problem_sizes, streams)
    else:
        problem_size = _problem_layout(c_img, s_img, c_loss_weight, s_loss_weight, independent, problem_size, streams)
    if problem_size == 1:
        independent = True
    dev = torch.device(device)
    if dev.type != 'cuda':
        raise _lib.IsxError("iris_b200.nst runs on a CUDA B200 only (device=%r); there is no CPU fallback" % (device,))
    if dev.index is None:
        dev = torch.device('cuda', torch.cuda.current_device())
    if vgg is None:
        vgg = VGG19()
    vgg.to(dev)
    with torch.cuda.device(dev), torch.no_grad():
        kw = dict(clone_content=clone_content, BN_loss=BN_loss, c_loss_weight=c_loss_weight,
                  s_loss_weight=s_loss_weight, lr=lr, epochs=epochs, independent=independent,
                  history_size=history_size, x_init=x_init, history_dtype=history_dtype, c_mask=c_mask, s_mask=s_mask,
                  problem_size=problem_size, problem_sizes=problem_sizes)
        if streams > 1 and independent and c_img.dim() == 4 and c_img.shape[0] > 1:
            c_dev, _ = _prep_images(c_img, dev)
            s_dev = s_img.detach().to(dev, torch.float32)
            job = NstJobGroup(c_dev, s_dev, vgg, dev, streams=streams, overlap=overlap, **kw)
        else:
            job = NstJob(c_img, s_img, vgg, dev, **kw)
        B_all = c_img.shape[0] if c_img.dim() == 4 else 1
        hist = None
        if x_hist_stride:
            n_keep = (job.max_ticks + x_hist_stride - 1) // x_hist_stride
            shape = tuple(c_img.shape[-3:]) if c_img.dim() == 3 else (B_all,) + tuple(c_img.shape[-3:])
            hist = _HistoryWriter(shape, n_keep, dev)
        group = isinstance(job, NstJobGroup)

        def snapshot():
            if group:     # sub-batches live on their own streams: gather their images on the caller's stream
                job.join(dev)
                hist.snapshot(torch.cat([j.x for j in job.jobs]))
                job.fork(dev)
            else:
                hist.snapshot(job.x)

        if cuda_graph and not group:
            if hist is not None:
                snapshot()            # image of the eager first evaluation
            job.enable_graph()
        pbar = None
        if use_tqdm:
            import tqdm
            pbar = tqdm.tqdm(total=epochs)
        while job.ticks < job.max_ticks:
            if hist is not None and job.ticks % x_hist_stride == 0:
                snapshot()            # pipelines.py:93, without the host synchronisation
            job.tick()
            if pbar is not None:
                pbar.update(1)
            if job.ticks >= job.epochs:
                # `while current_epoch[0] < epochs` (pipelines.py:79): no problem can finish before `epochs` evaluations,
                # so the host never synchronises before that; afterwards it polls the device flags every tick (a problem
                # whose optimizer.step exited early -- lbfgs.py:370-374,463,511-526 -- overshoots by up to 19).
                if bool((job.evals_done() > 0).all().item()):
                    break
        if pbar is not None:
            pbar.close()
        x, n_evals, evals, hc, hs = job.finish()
        x_hist: List[torch.Tensor] = []
        if hist is not None:
            x_hist = hist.finish((n_evals + x_hist_stride - 1) // x_hist_stride)
        if c_img.dim() == 3:          # unbatched content image: the reference returns (3,H,W) (pipelines.py:52,110)
            x = x[0]
        per_problem = independent or problem_size is not None or problem_sizes is not None
        c_loss_hist = (hc.mean(dim=1) if per_problem else hc[:, 0]).tolist()
        s_loss_hist = (hs.sum(dim=1) if per_problem else hs[:, 0]).tolist()
        last_info.clear()
        last_info.update(ticks=job.ticks, evals=n_evals, evals_per_problem=evals, c_loss_per_image=hc,
                         s_loss_per_image=hs, c_loss_per_problem=hc, s_loss_per_problem=hs, problems=job.P)
    return x, x_hist, c_loss_hist, s_loss_hist


def mask_and_crop_iris(x: torch.Tensor,
                       ritnet: torch.nn.Module = None,
                       glint_threshold: float = 0.8,
                       area_threshold: int = 500,
                       connectivity: int = 2,
                       device: str = 'cuda:0',
                       *,
                       seg: Optional[torch.Tensor] = None,
                       ) -> tuple[torch.Tensor, torch.Tensor, int, int, int, int]:
    """pipelines.py:112-166: m = (ritnet(x) == 2) * (x <= glint_threshold); x*m; trim to the bbox of the nonzero
    pixels; repeat to 3 channels.  `ritnet`: any callable returning the (1,H,W) label map -- iris_b200.RITnet (the
    segmenter on the device), the reference's RITnet, ... -- default = iris_b200.RITnet() like pipelines.py:133-135; or
    pass the label map itself as `seg`.  int64 and uint8 label maps are read as they are (e.g. from
    `iris_b200.RITnet(label_dtype=torch.uint8)`); other integer dtypes are widened to int64.
    Returns (x (3,h,w) fp32, m (1,h,w) bool, x_min, y_min, x_max, y_max) like the reference."""
    from .utils import _bbox_of

    x = x.to(device)
    if seg is None:
        if ritnet is None:
            from .ritnet import RITnet

            ritnet = RITnet()  # pipelines.py:133-135: the default loads models/weights/ritnet_pretrained.pkl
        if hasattr(ritnet, "to"):
            ritnet.to(device)
        seg = ritnet(x)
    bbox, mask, xm = _bbox_of(x[None], seg=seg.reshape(1, *x.shape), label=2, threshold=glint_threshold,
                              want_mask=True, want_masked=True)
    x_min, y_min, x_max, y_max = bbox[0].tolist()
    if x_max < 0:
        raise RuntimeError("mask_and_crop_iris: empty iris mask (the reference fails in min() of an empty tensor)")
    xc = xm[0][:, x_min: x_max + 1, y_min: y_max + 1]
    mc = mask[0][:, x_min: x_max + 1, y_min: y_max + 1].bool()
    return xc.repeat(3, 1, 1), mc, x_min, y_min, x_max, y_max


def iris_masks_and_bboxes(frames: torch.Tensor, segs: torch.Tensor, glint_threshold: float = 0.8, label: int = 2):
    """Batched form of the mask recipe (data_preprocessing.py:164-185, …2020.py:79-100): frames [B,1,H,W],
    label maps [B,1,H,W] (int64 or uint8 read as they are, other integer dtypes widened to int64) -> (mask uint8 [B,1,H,W],
    bbox int32 [B,4]) in one kernel launch."""
    from .utils import _bbox_of

    bbox, mask, _ = _bbox_of(frames, seg=segs, label=label, threshold=glint_threshold, want_mask=True)
    return mask, bbox


def crop_resize_irises(frames: torch.Tensor, masks: torch.Tensor, bboxes: torch.Tensor, size=(224, 224)):
    """…2019.py:66-79: (frame * mask)[bbox] -> Resize(size) (bilinear, antialias) -> repeat to 3 channels, for the whole
    batch in ONE launch (isx_crop_resize_masked: the mask multiply happens on the source taps inside the kernel).
    frames [B,1,H,W] fp32, masks uint8 [B,1,H,W], bboxes int32 [B,4]."""
    if not frames.is_cuda:
        raise _lib.IsxError("iris_b200 needs CUDA tensors (B200); there is no CPU path")
    B, _, H, W = frames.shape
    # zero-initialised: a frame WITHOUT iris pixels (bbox sentinel row_max = -1) yields an all-zero crop, never
    # uninitialised memory; callers that must skip such frames test `bboxes[:, 2] < 0` (mask_and_crop_iris raises)
    out = torch.zeros(B, 3, size[0], size[1], device=frames.device, dtype=torch.float32)
    with torch.cuda.device(frames.device):
        _lib.call("isx_crop_resize_masked", frames.detach().to(torch.float32).contiguous(),
                  masks.to(torch.uint8).contiguous(), bboxes.to(torch.int32).contiguous(), out, 3, size[0], size[1], B, H, W,
                  _lib.stream_ptr())
    return out


def composite_irises(frames: torch.Tensor, new_irises: torch.Tensor, masks: torch.Tensor, bboxes: torch.Tensor):
    """…2019.py:111-130 / …2020.py:121-139 for the whole batch, in place on `frames` [B,1,H,W]:
    rgb_to_grayscale(new) -> Resize(bbox shape) -> * mask[bbox] -> frame[bbox] = frame[bbox] * ~mask + new."""
    if not frames.is_cuda:
        raise _lib.IsxError("iris_b200 needs CUDA tensors (B200); there is no CPU path")
    assert frames.is_contiguous() and frames.dtype == torch.float32
    B, _, H, W = frames.shape
    new = new_irises.detach().to(frames.device, torch.float32).contiguous()
    with torch.cuda.device(frames.device):
        _lib.call("isx_composite", new, new.shape[1], new.shape[2], new.shape[3], frames,
                  masks.to(torch.uint8).contiguous(), bboxes.to(torch.int32).contiguous(), B, H, W, _lib.stream_ptr())
    return frames
