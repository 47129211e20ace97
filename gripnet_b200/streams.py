"""Fork / join of side streams inside one training step.

At pose-0 size a step is ~70 kernels of 3-50 us, most of them latency-bound at 10-30 %
occupancy (``profiles/r01_v4_ncu_full_summary.csv``), and about half of the summed kernel time
is OFF the critical path: weight / bias gradients (``X^T dY``, column sums), the decoder's
``dw`` next to its ``dz``, the negative edges' decoder next to the positive ones.  A ``Branch``
sends such kernels to a side stream so they overlap the dependency chain; when the step is
captured (``capture.py``) the fork / join events become parallel branches of the CUDA graph.

Rules that keep this safe with PyTorch's caching allocator (which only orders reuse of a block on
the stream that allocated it):

* torch's *current* stream is never switched: every tensor is still allocated on the caller's
  stream; only the kernels launched inside ``with branch(...)`` go to the side stream
  (``graph._stream()`` honours the override);
* every entry into the branch re-forks: the side stream waits for everything enqueued on the
  caller's stream so far, so a block the allocator recycled is no longer in use there;
* every tensor a side kernel reads or scratches — the ones passed to ``branch(...)`` and all
  temporaries allocated while the branch is active (``keep``) — is held until ``join()``, after which the
  caller's stream is ordered behind the side work and normal stream-ordered reuse is safe again;
* results are allocated by the caller (on its stream) and must not be consumed before ``join()``.

Branches nest (a branch created inside ``with other:`` forks off that side stream and hands its
temporaries to the parent on ``join``).  No collective / peer exchange is ever issued inside a branch: a
partitioned (multi-GPU) run branches only for work that stays on the GPU (parameter gradients when their reduction
is deferred to the end of the step, index structures, weight images).

A branch may be joined by its CONSUMER instead of where it was forked: ``pipelines.PoseModel`` forks the build of
the decoder backward's index structures before the first kernel of a step and hands the branch to
``ops.DistMultPair``, whose backward joins it; ``ops.RelPrologue`` does the same for the relational layer's
parameter-only work.  A branch that is dropped un-joined joins itself first (``__del__``), so the temporaries it
holds are never released under running side work.  ``background=True`` puts a branch on a default-priority stream,
below the high-priority stream the step's dependency chain is captured on (``capture.CapturedStep``).
"""
import threading

import torch

# Stream priorities: the kernels of the step's dependency chain (and the branches that are joined straight back into
# it) run on high-priority streams, parameter-gradient / structure-build branches ("background") on default-priority
# ones, so a chain kernel that becomes ready while a wide weight-gradient kernel is in flight gets the next free SM
# slots.  A captured graph keeps the priority of the stream each kernel was captured on.
CHAIN_PRIORITY = -1
_N_SIDE = 8
_tls = threading.local()
_pools = {}
_pool_lock = threading.Lock()


def override():
    """The torch.cuda.Stream kernels are redirected to, or None."""
    return getattr(_tls, "side", None)


def effective_stream():
    s = override()
    return s if s is not None else torch.cuda.current_stream()


def keep(*tensors):
    """Hold temporaries of a side-stream launch until the active branch joins (no-op otherwise)."""
    b = getattr(_tls, "branch", None)
    if b is not None:
        b._keep.extend(t for t in tensors if t is not None)


def _next_side(device, avoid=None, background=False):
    idx = device.index if device.index is not None else torch.cuda.current_device()
    prio = 0 if background else CHAIN_PRIORITY
    with _pool_lock:
        pool = _pools.get((idx, prio))
        if pool is None:
            pool = _pools[(idx, prio)] = [[torch.cuda.Stream(device=idx, priority=prio) for _ in range(_N_SIDE)], 0]
        for _ in range(_N_SIDE):
            pool[1] = (pool[1] + 1) % _N_SIDE
            if avoid is None or pool[0][pool[1]].cuda_stream != avoid.cuda_stream:
                break
        return pool[0][pool[1]]


class Branch:
    """One side stream forked off the caller's stream.

        br = Branch()
        out = torch.empty(...)                  # allocated by the caller
        with br(x, y):                          # x, y: tensors the side kernels read
            launch_kernels(x, y, out)           # -> side stream
        ...                                     # the caller's stream carries on
        br.join()                               # before `out` is consumed / returned
    """

    def __init__(self, enabled=True, background=False):
        """``background``: work nothing on the step's dependency chain waits for soon (parameter gradients, index
        structures of the backward, weight images): default-priority stream, below the chain's."""
        self.enabled = bool(enabled)
        self._keep = []
        self._dirty = False
        self._args = ()
        self._parent = getattr(_tls, "branch", None)     # created inside another branch: nested fork
        if self.enabled:
            self.main = effective_stream()
            self.side = _next_side(self.main.device, avoid=self.main, background=background)

    def __call__(self, *tensors):
        self._args = tensors
        return self

    def __enter__(self):
        if not self.enabled:
            return self
        self._keep.extend(t for t in self._args if t is not None)
        self._args = ()
        ev = torch.cuda.Event()
        ev.record(self.main)
        self.side.wait_event(ev)
        self._prev = (getattr(_tls, "side", None), getattr(_tls, "branch", None))
        _tls.side, _tls.branch = self.side, self
        self._dirty = True
        return self

    def __exit__(self, *exc):
        if self.enabled:
            _tls.side, _tls.branch = self._prev
        return False

    def join(self, deferrable=False):
        """Order the caller's stream behind the side work.  ``deferrable``: the results are parameter gradients
        that nothing reads before the backward pass ends (the caller has checked that autograd will only STORE
        them): the join is postponed to an autograd-engine callback that runs when the whole backward pass is
        done, so the dependency chain of the step never waits for weight-gradient kernels."""
        if deferrable and self.enabled and self._dirty and self._parent is None and _defer(self):
            return
        self._join_now()

    def _join_now(self):
        if self.enabled and self._dirty:
            ev = torch.cuda.Event()
            ev.record(self.side)
            self.main.wait_event(ev)
            self._dirty = False
        if self._parent is not None:
            # only the parent's side stream is ordered behind this branch so far: the temporaries stay
            # alive until the parent joins the stream that allocated them
            self._parent._keep.extend(self._keep)
        self._keep.clear()

    def __del__(self):
        # a branch handed to a consumer that never ran (e.g. the structure branch of a decoder whose backward was
        # never called): order the caller's stream behind the side work BEFORE the held temporaries are released
        try:
            if self.enabled and self._dirty:
                self._join_now()
        except Exception:          # interpreter / CUDA context shutting down
            pass


# ---- joins deferred to the end of the autograd backward pass -------------------------------------------------
_deferred = []
_deferred_lock = threading.Lock()
_callback_queued = [False]


def _drain_deferred():
    with _deferred_lock:
        items = list(_deferred)
        _deferred.clear()
        _callback_queued[0] = False
    for b in items:
        b._join_now()


def _defer(branch):
    """Queue ``branch`` for the end-of-backward callback; False when no backward pass is running."""
    with _deferred_lock:
        need_cb = not _callback_queued[0]
        if need_cb:
            try:
                torch.autograd.Variable._execution_engine.queue_callback(_drain_deferred)
            except RuntimeError:          # not inside a backward pass
                return False
            _callback_queued[0] = True
        _deferred.append(branch)
    return True


def grads_only_stored(params, needs):
    """True when every parameter of ``params`` that needs a gradient is a leaf whose ``.grad`` is still None:
    autograd's AccumulateGrad will then just keep the tensor it is handed (no kernel reads it), so the kernels
    that produce it may still be running on a side stream when ``backward()`` returns to the engine."""
    for p, need in zip(params, needs):
        if not need or p is None:
            continue
        if not p.is_leaf or p.grad is not None:
            return False
    return True
