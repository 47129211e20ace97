"""Host-side trace of the layer stacks, no GPU needed: run GcnStack / RgcnStack forward + backward of the tree ROOT
on CPU tensors against a stand-in library, stand-in streams and a stand-in partition context (world 2, rank 1, with
and without halo plans and deferred reduction), and log every library call (name, non-pointer arguments, stream),
every side-stream pick, fork and join, every slot-buffer allocation, gather and gradient reduction.

    python profiles/stack_host_trace.py ROOT OUT.json        # one tree
    python profiles/stack_host_trace.py --compare A.json B.json

The kernels do not run: the trace shows what the host code asks for, in which order and on which stream."""
import json
import os
import sys

if sys.argv[1] == "--compare":
    def cases(path):
        out, cur = {}, None
        for e in json.load(open(path)):
            if e[0] == "case":
                cur = out[e[1]] = []
            else:
                cur.append(e)
        return out
    A, B = cases(sys.argv[2]), cases(sys.argv[3])
    for name in A:
        slots = [e for e in A[name] if e[0] == "slot_buffer"] == [e for e in B[name] if e[0] == "slot_buffer"]
        rest = [e for e in A[name] if e[0] != "slot_buffer"] == [e for e in B[name] if e[0] != "slot_buffer"]
        print(f"{name:48s} slot allocations {'same' if slots else 'DIFFER'}, "
              f"{'identical' if A[name] == B[name] else 'same apart from slot positions' if rest else 'DIFFER'}")
    sys.exit(0)
root, out = os.path.abspath(sys.argv[1]), sys.argv[2]
sys.path.insert(0, root)
import torch  # noqa: E402

import gripnet_b200  # noqa: E402,F401
from gripnet_b200 import _lib, ops, streams  # noqa: E402

assert os.path.dirname(ops.__file__) == os.path.join(root, "gripnet_b200")
LOG = []


class FakeStream:
    def __init__(self, i):
        self.id = self.cuda_stream = i
        self.device = torch.device("cpu")

    def wait_event(self, ev):
        LOG.append(("wait", self.id, ev.src))


class FakeEvent:
    def record(self, s):
        self.src = s.id


MAIN = FakeStream(0)
_sides = [0]


def next_side(device, avoid=None, background=False):
    _sides[0] += 1
    LOG.append(("side", _sides[0], background))
    return FakeStream(_sides[0])


def norm(a):
    if isinstance(a, int) and abs(a) >= 1 << 20:
        return "P"
    if a is None or isinstance(a, (int, float, str, bool)):
        return a
    return type(a).__name__


class FakeLib:
    def __getattr__(self, name):
        def f(*args):
            if name.endswith("workspace_bytes"):
                return 0
            LOG.append((name, ops._stream(), [norm(a) for a in args if not (isinstance(a, int) and abs(a) >= 1 << 20)]))
            return 0
        return f


fake = FakeLib()
_lib.load = lambda: fake
torch.cuda.Event = FakeEvent
streams.effective_stream = lambda: streams.override() or MAIN
streams._next_side = next_side
ops._stream = lambda: (streams.override() or MAIN).id
ops.require_cuda = lambda t, name, dtype=None: t


class Csr:
    ref = None

    def partial(self, f):
        return None


class Halo:
    def __init__(self, rows):
        self.rows = rows


class Dctx:
    def __init__(self, world, rank, defer):
        self.world, self.rank, self.defer_grad_reduce = world, rank, defer

    def slot_buffer(self, rows, f, like, uniform=True):
        LOG.append(("slot_buffer", rows, f, uniform))
        return torch.empty((rows, f))

    def all_gather_slots(self, full):
        LOG.append(("all_gather", tuple(full.shape)))

    def halo_gather(self, full, plan):
        LOG.append(("halo_gather", tuple(full.shape)))

    def reduce_param_grad_(self, t):
        LOG.append(("reduce", tuple(t.shape), ops._stream()))


class GcnG:
    def __init__(self, n_src, n_dst, dctx=None, halo=False):
        self.n_src, self.n_dst, self.fwd, self.bwd = n_src, n_dst, Csr(), Csr()
        if dctx is not None:
            self.ctx, self.b_src, self.b_dst = dctx, n_src + 1, n_dst + 1
            self.fwd_halo = Halo(n_src + 7) if halo else None
            self.bwd_halo = Halo(n_dst + 5) if halo else None


class RgcnG:
    def __init__(self, n, r, dctx=None):
        self.n_nodes, self.n_rel, self.fwd, self.bwd = n, r, Csr(), Csr()
        self.inv_cnt = torch.ones(n)
        if dctx is not None:
            self.ctx, self.b = dctx, n + 2


def p(*shape, grad=True):
    return torch.randn(*shape).requires_grad_(grad)


def run(name, fn):
    LOG.append(("case", name))
    _sides[0] = 0
    torch.manual_seed(0)
    fn()


def gcn(g, dims, relu, catout, bias=True, x_grad=True, bias_grad=True):
    params = []
    for k, f in zip(dims[:-1], dims[1:]):
        params += [p(k, f), p(f, grad=bias_grad) if bias else None]
    x = p(g.n_src, dims[0], grad=x_grad)
    y = ops.GcnStack.apply(x, g, relu, catout, *params)
    y.backward(torch.randn_like(y))


def rgcn(g, dims, relu, catout, bias=False, x_grad=True, nb=3):
    params = []
    for k, f in zip(dims[:-1], dims[1:]):
        params += [p(nb, k, f), p(g.n_rel, nb), p(k, f), p(f) if bias else None]
    x = p(g.n_nodes, dims[0], grad=x_grad)
    y = ops.RgcnStack.apply(x, g, relu, catout, *params)
    y.backward(torch.randn_like(y))


for x_grad in (True, False):
    run(f"gcn catout x_grad={x_grad}", lambda: gcn(GcnG(50, 50), [8, 16, 12, 8], (True,) * 3, True, x_grad=x_grad))
    run(f"gcn plain mixed relu x_grad={x_grad}",
        lambda: gcn(GcnG(50, 50), [8, 16, 12], (True, False), False, x_grad=x_grad))
    run(f"gcn inter x_grad={x_grad}", lambda: gcn(GcnG(40, 30), [8, 16], (True,), False, x_grad=x_grad))
    run(f"gcn no bias x_grad={x_grad}", lambda: gcn(GcnG(50, 50), [8, 16, 12], (True, True), True, bias=False,
                                                   x_grad=x_grad))
    run(f"rgcn catout x_grad={x_grad}", lambda: rgcn(RgcnG(40, 4), [8, 16, 12], (True, True), True, x_grad=x_grad))
    run(f"rgcn plain x_grad={x_grad}", lambda: rgcn(RgcnG(40, 4), [8, 16, 12], (True, False), False, x_grad=x_grad))
    for defer in (True, False):
        for halo in (True, False):
            run(f"dist gcn catout defer={defer} halo={halo} x_grad={x_grad}",
                lambda: gcn(GcnG(50, 50, Dctx(2, 1, defer), halo), [8, 16, 12, 8], (True,) * 3, True, x_grad=x_grad))
            run(f"dist gcn inter defer={defer} halo={halo} x_grad={x_grad}",
                lambda: gcn(GcnG(40, 30, Dctx(2, 1, defer), halo), [8, 16], (False,), False, x_grad=x_grad))
        run(f"dist rgcn catout defer={defer} x_grad={x_grad}",
            lambda: rgcn(RgcnG(40, 4, Dctx(2, 1, defer)), [8, 16, 12], (True, True), True, x_grad=x_grad))
        run(f"dist rgcn plain defer={defer} x_grad={x_grad}",
            lambda: rgcn(RgcnG(40, 4, Dctx(2, 1, defer)), [8, 16, 12], (True, False), False, x_grad=x_grad))
run("gcn frozen bias", lambda: gcn(GcnG(50, 50), [8, 16, 12], (True, True), True, bias_grad=False))
run("rgcn with bias", lambda: rgcn(RgcnG(40, 4), [8, 16, 12], (True, True), True, bias=True))
json.dump(LOG, open(out, "w"))
print(len(LOG), "entries")
