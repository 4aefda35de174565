"""Two-GPU tests (skipped on a single-GPU box): the gradient exchange folded into the optimizer kernel over NVLink peer
memory (bnn_adam_kl_step_peers + bnn_peer_barrier, training.ElboTrainer(exchange='peer')) against the NCCL all-reduce of
the flat gradient buffer (exchange='flat') — same parameters after three steps, bit-identical across ranks — and the
data x sample grid against a single process that evaluates all samples of both batch slices."""
import os
import socket
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, results):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    device = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=device)
    try:
        sys.path.insert(0, ROOT)
        import bench
        import bayesianneuralnetworks_b200 as bnn
        from bayesianneuralnetworks_b200.training import ElboTrainer
        bnn.set_precision("fp32")
        S, B = 4, 32
        finals = {}
        for mode in ("peer", "peer2hop", "flat", "bucketed"):
            two_hop, mode = mode == "peer2hop", "peer" if mode == "peer2hop" else mode
            torch.manual_seed(0)
            model = bench.build_model("c2", S).to(device)            # S = global samples; grid 1 data x 2 sample groups
            initial = torch.cat([p.detach().flatten() for p in model.parameters()]).clone()
            trainer = ElboTrainer(model, 10, lr=1e-2, graph=(mode != "bucketed"), exchange=mode, sample_groups=2)
            assert trainer.exchange == mode and (trainer.data_index, trainer.sample_index) == (0, rank)
            if two_hop:          # the exchange of more than two ranks (bnn_peer_average: reduce-scatter + all-gather in place)
                trainer.opt.two_hop_above = 1
            gen = torch.Generator().manual_seed(7)
            x, y = bench.synthetic_batch("c2", B, gen)
            x, y = x.to(device), y.to(device)
            # injected eps (the same in every mode; each rank draws for ITS two samples of the four)
            ge = torch.Generator().manual_seed(100 + rank)
            eps = {w: torch.randn((S // world,) + tuple(w.shape), generator=ge).to(device)
                   for w in model.modules() if isinstance(w, bnn.nn.WeightNormal)}
            with bnn.injected_eps(eps):
                if trainer.use_graph:
                    trainer.capture(x, y)                             # three eager steps
                else:
                    for _ in range(3):
                        trainer.step(x, y)
                for _ in range(2):
                    loss = trainer.step(x, y)
            torch.cuda.synchronize()
            finals["peer2hop" if two_hop else mode] = torch.cat([p.detach().flatten() for p in model.parameters()]).clone()
            assert torch.isfinite(loss)
            trainer.release()
            del trainer, model
        # every rank holds the same parameters (the peer kernel sums the ranks in a fixed order: bit-identical)
        gathered = [torch.empty_like(finals["peer"]) for _ in range(world)]
        dist.all_gather(gathered, finals["peer"])
        assert torch.equal(gathered[0], gathered[1]), "ranks diverged under the peer exchange"
        # the two-hop kernel on its own: in-place average of the ranks' flat buffers == NCCL's average of the same
        # values, bit for bit with two ranks (one addition and an exact halving), on a length that is not a multiple of 4
        from bayesianneuralnetworks_b200 import _C, parallel
        pg = parallel.PeerGradients(100003, device)
        vals = torch.randn(100003, generator=torch.Generator().manual_seed(50 + rank)).to(device)
        for _ in range(2):
            pg.flat.copy_(vals)
            ref = vals.clone()
            dist.all_reduce(ref, op=dist.ReduceOp.AVG)
            pg.barrier()
            _C.peer_average(pg.bases, pg.rank, pg.flat.numel(), device)
            pg.barrier()
            torch.cuda.synchronize()
            assert torch.equal(pg.flat, ref), "bnn_peer_average differs from the all-reduce average"
        # and they are the parameters the NCCL exchanges produce.  The summation order differs, i.e. the gradients differ by
        # rounding; Adam's first steps are lr * g / |g|, so an element whose gradient is at rounding level can take a full
        # step the other way (max deviation ~ lr) — the measure is the relative L2 error of the whole update and the 99th
        # percentile of the element deviations
        for other in ("flat", "bucketed", "peer2hop"):
            diff = (finals["peer"] - finals[other]).abs()
            upd = (finals[other] - initial).norm()
            assert float(diff.norm() / upd) < 2e-2 and float(diff.flatten().quantile(0.99)) < 1e-4, (
                other, float(diff.norm() / upd), float(diff.flatten().quantile(0.99)), float(diff.max()))
        results[rank] = "ok"
    finally:
        dist.destroy_process_group()


def test_peer_memory_gradient_exchange_matches_nccl_on_two_gpus():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    import torch.multiprocessing as mp
    world, port = 2, _free_port()
    with mp.Manager() as m:
        results = m.dict()
        mp.spawn(_worker, args=(world, port, results), nprocs=world, join=True)
        assert dict(results) == {0: "ok", 1: "ok"}
