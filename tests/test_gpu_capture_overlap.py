"""Flat fake-quant launches captured into a CUDA graph as independent of their predecessor.

Inside a stream capture, a per-tensor forward or backward whose only dependency is the previous flat launch of the
library, and which reads nothing that launch writes, loads its qparams and first tile before griddepcontrol.wait.
`dlmcq_capture_overlap_count()` reports how many launches were captured that way.  Every chain below is launched
eagerly once, then captured, replayed with its outputs poisoned with NaN, and compared bit for bit with the eager
results.  The dependent chains must count 0: their second launch reads what the first one writes (or the first
launch is not its only dependency), and it reads the region its predecessor writes last, so a load hoisted above the
wait would meet data that is not written yet.  Replays run once; nothing here loops."""
import ctypes as C
import math

import pytest
import torch

import bench
from tests.golden_io import bits_equal, first_mismatch

pytestmark = pytest.mark.gpu

N_A = 1 << 24            # elements the first launch of a chain writes
N_B = 1 << 22            # elements the second launch reads
VEC = 4                  # fp32 elements in one 16-byte vector


def lib():
    from dlmc_quant_b200 import _lib
    return _lib, _lib.lib()


def overlap_count():
    return lib()[1].dlmcq_capture_overlap_count()


def stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


class Q:
    """qparams of one per-tensor AFFINE 4-bit quantizer (the benchmark's activation form)."""

    def __init__(self, scale, n):
        L, _ = lib()
        dev = torch.device("cuda")
        self.scale = torch.tensor([scale], dtype=torch.float32, device=dev)
        self.off = torch.tensor([-0.25], dtype=torch.float32, device=dev)
        self.qp = L.QParams(L.FORM_AFFINE, 0, 15, 1 / math.sqrt(n * 15), self.scale.data_ptr(), self.off.data_ptr())


def fwd(x, y, q):
    L, h = lib()
    lay = L.Layout(1, 1, x.numel(), L.F32)
    L.check(h.dlmcq_fq_forward(x.data_ptr(), y.data_ptr(), None, C.byref(lay), C.byref(q.qp), stream()))


def bwd_deferred(x, dy, dx, q, partials):
    L, h = lib()
    lay = L.Layout(1, 1, x.numel(), L.F32)
    L.check(h.dlmcq_fq_backward_partials(x.data_ptr(), dy.data_ptr(), dx.data_ptr(), C.byref(lay), C.byref(q.qp),
                                         partials.data_ptr(), stream()))


def bwd(x, dy, dx, dscale, q, ws):
    L, h = lib()
    lay = L.Layout(1, 1, x.numel(), L.F32)
    L.check(h.dlmcq_fq_backward(x.data_ptr(), dy.data_ptr(), dx.data_ptr(), dscale.data_ptr(), None, C.byref(lay),
                                C.byref(q.qp), ws.data_ptr(), ws.numel(), stream()))


def randn(n, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.randn(n, generator=g, device="cuda") * 3


def check_chain(inputs, outputs, chain, expect):
    """inputs: tensors restored before every run; outputs: tensors poisoned with NaN before every run."""
    saved = [t.clone() for t in inputs]

    def reset():
        for t, s in zip(inputs, saved):
            t.copy_(s)
        for t in outputs:
            t.fill_(float("nan"))

    reset()
    chain()
    torch.cuda.synchronize()
    eager = [t.clone() for t in outputs]
    assert all(not torch.isnan(e).all() for e in eager)
    overlap_count()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        chain()
    assert overlap_count() == expect
    reset()
    torch.cuda.synchronize()
    graph.replay()
    torch.cuda.synchronize()
    for i, (e, t) in enumerate(zip(eager, outputs)):
        assert bits_equal(e, t), f"output {i}: {first_mismatch(e, t)}"


# --------------------------------------------------------------------------------------
def test_bench_step_overlaps_53_of_54_launches_per_graph():
    """bench.Workload's three graphs: 53 forwards and 53 backwards are independent of their predecessor (the first
    launch of each graph has none; finalize_many and the grouped weight kernels never count).  The replayed step is
    bitwise equal to the same step launched eagerly."""
    wl = bench.Workload(16, torch.device("cuda"), 2333)
    outs = [wl.dscale] + [a[k] for a in wl.acts for k in ("y", "dx")] + [w[k] for w in wl.wts for k in ("y", "dx")]
    wl.fwd_acts(); wl.bwd_acts(); wl.weights()
    torch.cuda.synchronize()
    eager = [t.clone() for t in outs]
    overlap_count()
    wl.capture()
    assert overlap_count() == 106
    for t in outs:
        t.fill_(float("nan"))
    wl.deferred.partials.fill_(float("nan"))
    torch.cuda.synchronize()
    wl.g_fwd.replay(); wl.g_bwd.replay(); wl.g_wt.replay()
    torch.cuda.synchronize()
    for i, (e, t) in enumerate(zip(eager, outs)):
        assert bits_equal(e, t), f"bench output {i}: {first_mismatch(e, t)}"


def two_forwards(a_x, a_y, b_x, b_y):
    qa, qb = Q(0.5, a_x.numel()), Q(0.375, b_x.numel())

    def chain():
        fwd(a_x, a_y, qa)
        fwd(b_x, b_y, qb)
    return chain


def test_dependent_reads_predecessor_output():
    """B's x is the last quarter of A's y."""
    a_x, a_y, b_y = randn(N_A, 1), torch.empty(N_A, device="cuda"), torch.empty(N_B, device="cuda")
    check_chain([a_x], [a_y, b_y], two_forwards(a_x, a_y, a_y[N_A - N_B:], b_y), 0)


@pytest.mark.parametrize("end", ["head", "tail"])
def test_dependent_one_vector_overlap(end):
    """B's x shares exactly one 16-byte vector with A's y: its first vector is A's last, or its last is A's first."""
    buf = randn(N_A + N_B, 2)
    if end == "head":
        a_y, b_x = buf[:N_A], buf[N_A - VEC:N_A - VEC + N_B]
    else:
        b_x, a_y = buf[:N_B], buf[N_B - VEC:N_B - VEC + N_A]
    a_x, b_y = randn(N_A, 3), torch.empty(N_B, device="cuda")
    check_chain([a_x, buf], [b_y], two_forwards(a_x, a_y, b_x, b_y), 0)


def test_dependent_reads_predecessor_dx():
    """A is a deferred backward; B's x is the tail of A's dx."""
    a_x, a_dy = randn(N_A, 4), randn(N_A, 5)
    a_dx, b_y = torch.empty(N_A, device="cuda"), torch.empty(N_B, device="cuda")
    L, h = lib()
    parts = torch.empty(h.dlmcq_fq_partials_floats(), device="cuda")
    qa, qb = Q(0.5, N_A), Q(0.375, N_B)
    b_x = a_dx[N_A - N_B:]

    def chain():
        bwd_deferred(a_x, a_dy, a_dx, qa, parts)
        fwd(b_x, b_y, qb)
    check_chain([a_x, a_dy], [a_dx, b_y], chain, 0)


def test_dependent_in_place_forward_then_read():
    """A fake-quantises x in place (y is x); B reads the tail of x."""
    a_x, b_y = randn(N_A, 6), torch.empty(N_B, device="cuda")
    check_chain([a_x], [b_y], two_forwards(a_x, a_x, a_x[N_A - N_B:], b_y), 0)


def test_dependent_shared_workspace():
    """Two in-kernel-finalised backwards on disjoint tensors that share one workspace (ticket counter, partials)."""
    L, h = lib()
    ws = torch.zeros(h.dlmcq_workspace_bytes(None), dtype=torch.uint8, device="cuda")
    a_x, a_dy, b_x, b_dy = randn(N_A, 7), randn(N_A, 8), randn(N_B, 9), randn(N_B, 10)
    a_dx, b_dx = torch.empty(N_A, device="cuda"), torch.empty(N_B, device="cuda")
    ds = torch.empty(2, device="cuda")
    qa, qb = Q(0.5, N_A), Q(0.375, N_B)

    def chain():
        bwd(a_x, a_dy, a_dx, ds[0:1], qa, ws)
        bwd(b_x, b_dy, b_dx, ds[1:2], qb, ws)
    check_chain([a_x, a_dy, b_x, b_dy], [a_dx, b_dx, ds], chain, 0)


def test_dependent_torch_kernel_between():
    """A writes y, a torch kernel negates it in place, B reads its tail: B's predecessor is not a flat launch."""
    a_x, a_y, b_y = randn(N_A, 11), torch.empty(N_A, device="cuda"), torch.empty(N_B, device="cuda")
    qa, qb = Q(0.5, N_A), Q(0.375, N_B)

    def chain():
        fwd(a_x, a_y, qa)
        a_y.mul_(-1)
        fwd(a_y[N_A - N_B:], b_y, qb)
    check_chain([a_x], [a_y, b_y], chain, 0)


def test_dependent_fork_join():
    """A on the capturing stream, C (disjoint from everything else) on a forked stream; after the join B has two
    dependencies, the last flat launch recorded is C, and B reads the tail of A's y."""
    a_x, c_x = randn(N_A, 12), randn(N_B, 13)
    a_y, c_y, b_y = (torch.empty(n, device="cuda") for n in (N_A, N_B, N_B))
    qa, qb, qc = Q(0.5, N_A), Q(0.375, N_B), Q(0.25, N_B)
    side = torch.cuda.Stream()

    def chain():
        main = torch.cuda.current_stream()
        side.wait_stream(main)
        fwd(a_x, a_y, qa)
        with torch.cuda.stream(side):
            fwd(c_x, c_y, qc)
        main.wait_stream(side)
        fwd(a_y[N_A - N_B:], b_y, qb)
    check_chain([a_x, c_x], [a_y, c_y, b_y], chain, 0)


def test_independent_adjacent_buffers():
    """A's y ends exactly where B's x begins: disjoint, so B is captured as independent."""
    buf = randn(N_A + N_B, 14)
    a_x, b_y = randn(N_A, 15), torch.empty(N_B, device="cuda")
    check_chain([a_x, buf], [b_y], two_forwards(a_x, buf[:N_A], buf[N_A:], b_y), 1)


def test_independent_writes_predecessor_input():
    """A is a deferred backward, whose capped grid walks x tile by tile and reaches the tail last; B writes the tail
    of A's x.  B reads nothing A writes, so it is independent, and its stores must still wait for A to finish."""
    a_x, a_dy, b_x = randn(N_A, 16), randn(N_A, 17), randn(N_B, 18)
    a_dx = torch.empty(N_A, device="cuda")
    L, h = lib()
    parts = torch.empty(h.dlmcq_fq_partials_floats(), device="cuda")
    qa, qb = Q(0.5, N_A), Q(0.375, N_B)

    def chain():
        bwd_deferred(a_x, a_dy, a_dx, qa, parts)
        fwd(b_x, a_x[N_A - N_B:], qb)
    check_chain([a_x, a_dy, b_x], [a_dx], chain, 1)
