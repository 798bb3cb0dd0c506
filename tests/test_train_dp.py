"""Data-parallel LoRA step on CPU with two real processes over gloo (config 5 is 4 x B200 data parallel): every rank runs
LoraTrainer through the torch test double on ITS shard of the records; one all-reduce of the gradient arena must give the
step a single process computes on the union of the records (token-mean over the global batch)."""
import os
import socket

import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import lora as ol


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _install_double():
    from chatts_b200 import _cabi
    from tests.cabi_double import TorchDouble
    dbl = TorchDouble()
    _cabi.get_context = lambda device=None: dbl
    torch.cuda.is_available = lambda: True
    torch.cuda.current_device = lambda: 0
    torch.Tensor.pin_memory = lambda self: self
    return dbl


def _run(records, group_world):
    from chatts_b200.train import LoraTrainer, encode_records
    from tests.test_host_train import _build
    cfg, sd, model, proc = _build(_install_double(), True)
    tr = LoraTrainer(model, r=8, lora_alpha=16, seed=7, init_b_std=0.05, lr=1e-2, max_grad_norm=0.5)
    batch = encode_records(proc, records, eos_token_id=cfg.eos_token_id)
    p_init = tr.p.clone()
    loss = float(tr.train_step(batch)[0])
    return loss, tr.g.clone(), tr.p.clone(), float(tr.norm_out[0]), p_init


def _worker(rank, world, port, ret):
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from chatts_b200.train import shard_records
    from tests.test_host_train import RECORDS
    ret[rank] = _run(shard_records(RECORDS, rank, world), world)
    dist.destroy_process_group()


def test_two_ranks_equal_one_process_on_the_union():
    world = 2
    mgr = mp.Manager()
    ret = mgr.dict()
    mp.spawn(_worker, args=(world, _free_port(), ret), nprocs=world, join=True)
    from chatts_b200.train import shard_records
    from tests.test_host_train import RECORDS
    # the union in the order the ranks saw it (rank 0: records 0, 2; rank 1: record 1)
    union = shard_records(RECORDS, 0, 2) + shard_records(RECORDS, 1, 2)
    loss, g, p, norm, _ = _run(union, 1)
    (l0, g0, p0, n0, p0_init), (l1, g1, p1, n1, _) = ret[0], ret[1]
    assert torch.equal(g0, g1) and torch.equal(p0, p1) and l0 == l1            # every rank holds the same step
    assert abs(l0 - loss) < 2e-3 * abs(loss), (l0, loss)
    rel = float((g0 - g).abs().max() / g.abs().max())
    assert rel < 2e-2, rel                                                       # bf16 forward on differently padded batches
    assert abs(n0 - norm) < 2e-2 * norm
    # the ranks' step is AdamW of the all-reduced gradient, clipped to 0.5 ...
    pe, _, _ = ol.adamw_update(p0_init, g0 * min(1.0, 0.5 / (n0 + 1e-6)), torch.zeros_like(p0), torch.zeros_like(p0), 1, lr=1e-2)
    assert torch.allclose(p0, pe, atol=1e-6, rtol=1e-5)
    # ... and the single process's step wherever the gradient is resolved.  The first Adam step moves every element by ~lr * sign(g): where
    # |g| lies within the two gradients' disagreement (whose size follows the host's thread count) the sign may differ, up to 2 lr apart
    resolved = g.abs() > (g0 - g).abs().max()
    assert float(resolved.float().mean()) > 0.9
    assert float((p0 - p)[resolved].abs().max()) < 2e-3 and float((p0 - p).abs().max()) < 2e-2      # lr = 1e-2, Adam step magnitude ~lr
