"""Data-parallel training on >= 2 GPUs (NCCL): the all-reduced gradient of TXLTrainer equals the oracle's gradient on the
concatenated batch, and every rank holds the same weights after the Adam step.  Self-skips on a one-GPU box; the driver's scaling
run and `bench.py --gpus N` exercise the same code path (`train.comm` in the bench record)."""
import os
import socket

import pytest
import torch
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu
V = 324


def _worker(rank, world, port, wire, q):
    os.environ.update(RANK=str(rank), LOCAL_RANK=str(rank), WORLD_SIZE=str(world), MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    import torch.distributed as dist
    from deepmusicgeneration_b200 import sharding
    from deepmusicgeneration_b200.model import get_language_model
    from deepmusicgeneration_b200.training import TXLTrainer
    from oracle import train as otrain
    from oracle import txl
    try:
        sharding.init_distributed(backend='nccl')
        torch.cuda.set_device(rank)
        bptt, per = 128, 2
        cfg = dict(txl.default_config(), n_layers=6, d_model=128, n_heads=2, d_head=64, d_inner=256, mem_len=bptt, ctx_len=bptt,
                   encode_position=False, mask_steps=1)
        # train mode draws rand_window_mask on the host (p = 0.2 of a k = 0 window even with mask_steps = 1): pin both sides to (1, 1)
        txl.rand_window_mask = lambda x_len, m_len, device, **kw: txl.window_mask(x_len, device, m_len, size=(1, 1))
        torch.manual_seed(0)
        om = txl.get_language_model(V, cfg, drop_mult=0.).train()
        pm = get_language_model(V, cfg, dtype='bf16', device=rank, max_batch=per, max_seq=bptt, keep_hidden=False, init=False)
        pm.load_state_dict(om.state_dict())
        tr = TXLTrainer(pm, per, bptt, cfg, drop_mult=0., distributed=True, wire=wire, bucket_layers=1)
        assert len(tr.buckets) >= 3
        g = torch.Generator().manual_seed(5)
        lo, hi = rank * per, (rank + 1) * per
        om.reset(); tr.reset()
        opt = otrain.AdamTrueWD(otrain.unique_params(om), eps=1e-3)
        worst, worst_at = 0., None
        for s in range(2):                                         # the second step runs over a warm memory
            x = torch.randint(0, V, (world * per, bptt), generator=g)
            y = torch.randint(0, V, (world * per, bptt), generator=g)
            ref = otrain.train_step(om, x, y, opt, 1e-3, wd=0.01, clip=0.5)         # the reference step on the WHOLE batch
            tr.forward(x[lo:hi], y[lo:hi], None, mask_size=(1, 1))
            tr.backward()                                          # all-reduce (SUM) inside
            got = tr.grads()
            refg = {n: p.grad for n, p in om.state_dict(keep_vars=True).items() if getattr(p, 'grad', None) is not None}
            for name, gsum in got.items():
                r = refg.get(name, refg.get('1.decoder.weight') if name == '0.encoder.weight' else None)
                assert r is not None, name
                e = ((gsum / world - r.reshape(gsum.shape)).norm() / r.norm().clamp_min(1e-20)).item()
                if e > worst: worst, worst_at = e, (s, name)
            tr.optimizer_step(1e-3, betas=(0.9, 0.99), eps=1e-3, wd=0.01, clip=0.5)
            gn = tr.losses()['grad_norm']
            assert abs(gn - ref['grad_norm']) < 4e-2 * ref['grad_norm'], (s, gn, ref['grad_norm'])
        sd = pm.state_dict()
        digest = torch.stack([v.double().sum() for _, v in sorted(sd.items())]).cuda()
        both = [torch.empty_like(digest) for _ in range(world)]
        dist.all_gather(both, digest)
        same = all(torch.equal(both[0], b) for b in both)
        comm = tr.profile_comm(lambda: (tr.forward(x[lo:hi], y[lo:hi], None, mask_size=(1, 1)), tr.backward()), reps=1)
        tr.close()
        q.put((rank, worst, same, (comm['bytes_per_step'], worst_at), None))
    except Exception as e:                                         # surface the failure in the parent
        import traceback
        q.put((rank, None, None, None, traceback.format_exc()))
    finally:
        sharding.finalize()


@pytest.mark.parametrize('wire', ['bf16', 'f32'])
def test_two_rank_allreduced_gradient_equals_oracle_on_concatenated_batch(wire):
    if torch.cuda.device_count() < 2:
        pytest.skip('needs 2 GPUs')
    s = socket.socket(); s.bind(('127.0.0.1', 0)); port = s.getsockname()[1]; s.close()
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, wire, q)) for r in range(2)]
    for p in procs: p.start()
    res = [q.get(timeout=600) for _ in procs]
    for p in procs: p.join(timeout=120)
    for rank, worst, same, nbytes, err in res:
        assert err is None, err
        print(f'rank {rank}: wire {wire}, worst gradient rel err vs oracle (whole batch) {worst:.3e} at {nbytes[1]}, {nbytes[0]} bytes exchanged per step, same weights {same}')
        assert worst < 2.5e-2 and same
