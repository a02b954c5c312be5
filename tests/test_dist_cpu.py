"""The N>1 host logic on CPU with the gloo backend, world_size 2: sharding, the max-over-ranks
timing reduction and the whole-job throughput aggregation that bench.py uses."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

from voicesplit_b200 import dist as vdist


def test_shard_covers_batch_exactly():
    for gb in (1, 2, 7, 256, 2048):
        for world in (1, 2, 3, 8):
            spans = [vdist.shard(gb, r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == gb
            assert all(spans[i][1] == spans[i + 1][0] for i in range(world - 1))
            sizes = [b - a for a, b in spans]
            assert max(sizes) - min(sizes) <= 1


def _worker(rank, world, port, out):
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank), MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    d = vdist.init("gloo")
    assert d is not None and d.get_world_size() == world
    a, b = vdist.shard(257, rank, world)
    local_ms = 100.0 + 50.0 * rank            # rank 1 is the slow one
    thr, ms = vdist.aggregate_throughput(b - a, local_ms, d)
    d.barrier()
    if rank == 0:
        out.put((thr, ms))
    d.destroy_process_group()


def test_two_rank_gloo_aggregation():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    thr, ms = q.get(timeout=120)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert ms == pytest.approx(150.0)                  # max over ranks, not the mean
    assert thr == pytest.approx(257 / 0.150)           # all utterances / slowest rank


def _grad_worker(rank, world, port, out):
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank), MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    d = vdist.init("gloo")
    torch.manual_seed(0)
    params = [torch.nn.Parameter(torch.zeros(5, 3)), torch.nn.Parameter(torch.zeros(7))]
    for i, p in enumerate(params):
        p.grad = torch.full_like(p, float(rank + 1) * (i + 1))          # rank-dependent gradients
    n = vdist.allreduce_gradients(params, d)
    if rank == 0:
        out.put((n, [p.grad.clone() for p in params]))
    d.barrier()
    d.destroy_process_group()


def test_flat_gradient_allreduce_averages_over_ranks():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_grad_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    n, grads = q.get(timeout=120)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert n == 22
    assert torch.allclose(grads[0], torch.full((5, 3), 1.5)) and torch.allclose(grads[1], torch.full((7,), 3.0))


def _reference_checks():
    # outputs of the unmodified reference SiSNR_With_Pit, written by tests/golden/make_reference_checks_golden.py
    return np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_checks.npz"))


def test_si_snr_matches_reference_formula():
    """voicesplit_b200/losses.py against the reference criterion."""
    from voicesplit_b200.losses import si_snr_with_pit
    torch.manual_seed(1)
    est, src = torch.randn(3, 1, 500), torch.randn(3, 1, 500)
    lengths = torch.tensor([500, 321, 77])
    mine = si_snr_with_pit(est.clone(), src.clone(), lengths)
    assert torch.isfinite(mine)
    ref = torch.tensor(_reference_checks()["sisnr_c1.loss"])
    assert torch.allclose(mine, ref, atol=1e-5)


class _FakeFlatModule:
    """Stands in for a MaskEstimator after its backward: .grad tensors are views of ONE flat buffer (no GPU needed)."""

    def __init__(self, rank):
        self.flat = torch.arange(10, dtype=torch.float32) * (rank + 1)
        self.params = [torch.nn.Parameter(torch.zeros(2, 3)), torch.nn.Parameter(torch.zeros(4))]
        self.params[0].grad = self.flat[0:6].view(2, 3)
        self.params[1].grad = self.flat[6:10]
        self._dp_pending = None

    def parameters(self):
        return iter(self.params)

    def flat_gradient(self):
        return self.flat


def _flat_worker(rank, world, port, overlap, out):
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank), MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    d = vdist.init("gloo")
    m = _FakeFlatModule(rank)
    if overlap:     # what MaskEstimator._dp_stage does mid-backward: the tail of the buffer is already being reduced
        m._dp_pending = (m.flat, 6, vdist.reduce_flat(m.flat[6:], d, async_op=True))
    n = vdist.allreduce_gradients(m, d)
    if rank == 0:
        out.put((n, m.flat.tolist(), m.params[0].grad.data_ptr() == m.flat.data_ptr(), m._dp_pending is None))
    d.barrier()
    d.destroy_process_group()


@pytest.mark.parametrize("overlap", [False, True])
def test_flat_buffer_fast_path_reduces_in_place(overlap):
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_flat_worker, args=(r, 2, port, overlap, q)) for r in range(2)]
    for p in procs:
        p.start()
    n, flat, aliased, pending = q.get(timeout=120)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert n == 10 and aliased and pending
    assert torch.allclose(torch.tensor(flat), torch.arange(10, dtype=torch.float32) * 1.5)     # mean of (1x, 2x), every element exactly once


@pytest.mark.parametrize("C", [2, 3])
def test_general_pit_matches_the_live_reference_with_gradients(C):
    """C > 1 sources (the permutation search the reference carries but its training never uses, generic_utils.py:443-474): loss and
    d(loss)/d(estimate) of losses.si_snr_with_pit against the unmodified SiSNR_With_Pit (its loss and gradient on these inputs are
    stored by tests/golden/make_reference_checks_golden.py)."""
    from voicesplit_b200.losses import si_snr_with_pit
    g = torch.Generator().manual_seed(7 + C)
    src = torch.randn(4, C, 400, generator=g)
    mix = torch.randn(4, C, C, generator=g) * 0.3 + torch.eye(C)[torch.randperm(C, generator=g)]      # estimates = permuted, leaky sources
    est0 = torch.einsum("bij,bjl->bil", mix, src) + 0.1 * torch.randn(4, C, 400, generator=g)
    lengths = torch.tensor([400, 399, 123, 57])
    a = est0.clone().requires_grad_(True)
    mine = si_snr_with_pit(a, src.clone(), lengths)
    z = _reference_checks()
    ref, ref_grad = torch.tensor(z[f"sisnr_c{C}.loss"]), torch.from_numpy(z[f"sisnr_c{C}.grad"])
    assert torch.allclose(mine, ref, atol=1e-5), (float(mine), float(ref))
    mine.backward()
    assert torch.allclose(a.grad, ref_grad, atol=1e-6 + 1e-4 * float(ref_grad.abs().max()))
