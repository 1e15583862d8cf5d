"""GPU, needs >= 2 devices (skipped on a single-GPU box): a batch sharded by image over two processes / two GPUs.

The two-kernel sharded step (Npos and loss sums exchanged by stores into peer memory over NVLink from inside the mining
kernel) must return the GLOBAL losses of the full batch and, on every rank, exactly the gradient slice a single GPU
computes for the full batch.  The NCCL route (Losses.process_group) must agree as well."""
import os

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

from objectdetection_ssd_b200 import synth
from oracle import ssd_oracle as O

pytestmark = [pytest.mark.gpu,
              pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")]

B_TOTAL, SEED = 12, 95


def _worker(rank, world, port, q):
    import torch.distributed as dist
    from objectdetection_ssd_b200.ctx import SSDHeadContext
    from objectdetection_ssd_b200.dist import shard_range
    from objectdetection_ssd_b200.head import MultiboxHead, multibox_loss
    from objectdetection_ssd_b200.priors import make_priors
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        pri = make_priors()
        P = pri.shape[0]
        gb, gc = synth.make_gt(SEED, B_TOTAL)
        loc, conf = synth.make_head(SEED, B_TOTAL, P)
        lo, hi = shard_range(rank, world, B_TOTAL)
        B = hi - lo
        gx, gcl, off = synth.pack_gt(gb[lo:hi], gc[lo:hi])
        d = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
        tl, tc, tgx, tgc, toff = d(loc[lo:hi]), d(conf[lo:hi]), d(gx), d(gcl), d(off)
        # --- peer-memory route: two kernels, no NCCL in the step
        ctx = SSDHeadContext(pri.numpy(), max_batch=B, device=rank)
        handles = [None] * world
        dist.all_gather_object(handles, ctx.xchg_export())
        ctx.xchg_import(handles, rank)
        dist.barrier()
        sums = torch.empty(2, dtype=torch.float64, device=dev)
        losses = torch.empty(2, device=dev)
        gl, gcf = torch.empty_like(tl), torch.empty_like(tc)
        st = torch.cuda.current_stream(dev).cuda_stream
        for _ in range(3):                                   # several steps: sequence numbers / parity slots
            ctx.loss_dev(tl.data_ptr(), tc.data_ptr(), tgx.data_ptr(), tgc.data_ptr(), toff.data_ptr(), B, int(off[-1]),
                         sums.data_ptr(), losses.data_ptr(), gl.data_ptr(), gcf.data_ptr(), st)
        torch.cuda.synchronize()
        assert not ctx.xchg_error()
        # --- the same sharded step on the six per-level tensors (ssdhead_multibox_step_levels_sharded)
        from objectdetection_ssd_b200 import _lib as L
        counts, s0 = (5776, 2166, 600, 150, 36, 4), 0
        lv = L.Levels()
        lv.num_levels = len(counts)
        keep = []
        for i, n in enumerate(counts):
            lc, cc = tl[:, s0:s0 + n].contiguous(), tc[:, s0:s0 + n].contiguous()
            glv, gcv = torch.empty_like(lc), torch.empty_like(cc)
            keep.append((lc, cc, glv, gcv))
            lv.count[i] = n
            lv.loc[i], lv.conf[i], lv.grad_loc[i], lv.grad_conf[i] = lc.data_ptr(), cc.data_ptr(), glv.data_ptr(), gcv.data_ptr()
            s0 += n
        sums_lv = torch.empty(2, dtype=torch.float64, device=dev)
        losses_lv = torch.empty(2, device=dev)
        ctx.loss_levels_dev(lv, tgx.data_ptr(), tgc.data_ptr(), toff.data_ptr(), B, int(off[-1]),
                            sums_lv.data_ptr(), losses_lv.data_ptr(), st)
        torch.cuda.synchronize()
        assert not ctx.xchg_error()
        assert torch.equal(losses_lv, losses) and torch.equal(sums_lv, sums), (losses_lv, losses)
        assert torch.equal(torch.cat([k[2] for k in keep], 1), gl) and torch.equal(torch.cat([k[3] for k in keep], 1), gcf)
        # --- the host-buffer steps on the same exchange (xchg_npos_kernel, sum_chunks_xchg_kernel): dense gradients
        # into page-locked and into pageable buffers, then packed rows scattered back to dense
        from objectdetection_ssd_b200.ctx import SparseRows
        from objectdetection_ssd_b200.pinned import pinned_empty
        host = {}
        for pinned in (True, False):
            alloc = pinned_empty if pinned else (lambda shape, dt=np.float32: np.empty(shape, dt))
            hl, hc = alloc(tl.shape), alloc(tc.shape)
            hl[...] = loc[lo:hi]
            hc[...] = conf[lo:hi]
            hgl, hgc = alloc(tl.shape), alloc(tc.shape)
            lh = ctx.loss_host(hl, hc, gx, gcl, off, hgl, hgc)
            host["pinned" if pinned else "pageable"] = (np.array(lh, np.float32), hgl.copy(), hgc.copy())
        rows = SparseRows(B, cap=4096)
        ls = ctx.loss_host_sparse(np.ascontiguousarray(loc[lo:hi]), np.ascontiguousarray(conf[lo:hi]), gx, gcl, off, rows)
        sgl, sgc = rows.scatter(P)
        host["sparse"] = (np.array(ls, np.float32), sgl, sgc)
        assert not ctx.xchg_error()
        # --- three steps with resident gradient tensors, the first one fresh
        rgl, rgc = torch.empty_like(tl), torch.empty_like(tc)
        sums_res, losses_res = torch.empty(2, dtype=torch.float64, device=dev), torch.empty(2, device=dev)
        for i in range(3):
            ctx.loss_dev_resident(tl.data_ptr(), tc.data_ptr(), tgx.data_ptr(), tgc.data_ptr(), toff.data_ptr(), B,
                                  int(off[-1]), sums_res.data_ptr(), losses_res.data_ptr(), rgl.data_ptr(), rgc.data_ptr(), st,
                                  fresh=(i == 0))
        torch.cuda.synchronize()
        assert not ctx.xchg_error()
        host["resident"] = (losses_res.cpu().numpy(), rgl.cpu().numpy(), rgc.cpu().numpy())
        # --- NCCL route through the drop-in surface
        head = MultiboxHead(pri, dev)
        l2 = tl.clone().requires_grad_(True)
        c2 = tc.clone().requires_grad_(True)
        a, b = multibox_loss(head, l2, c2, [torch.from_numpy(x) for x in gb[lo:hi]], [torch.from_numpy(x) for x in gc[lo:hi]],
                             group=dist.group.WORLD)
        (a + b).backward()
        torch.cuda.synchronize()
        q.put((rank, lo, hi, losses.cpu().numpy(), sums.cpu().numpy(), gl.cpu().numpy(), gcf.cpu().numpy(),
               np.array([a.item(), b.item()]), l2.grad.cpu().numpy(), c2.grad.cpu().numpy(), host))
        ctx.close()
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(600)
def test_two_gpu_sharded_step_equals_full_batch():
    from objectdetection_ssd_b200.head import MultiboxHead, PackedGT
    from objectdetection_ssd_b200.priors import make_priors
    world, port = 2, 29641 + os.getpid() % 500
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = sorted([q.get(timeout=500) for _ in range(world)], key=lambda r: r[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    # single-GPU full batch = the reference of the sharded runs; the oracle pins it
    pri = make_priors()
    gb, gc = synth.make_gt(SEED, B_TOTAL)
    loc, conf = synth.make_head(SEED, B_TOTAL, pri.shape[0])
    tb = [torch.from_numpy(b) for b in gb]
    tc = [torch.from_numpy(c) for c in gc]
    head = MultiboxHead(pri, "cuda:0")
    full = head.loss(torch.from_numpy(loc).cuda(), torch.from_numpy(conf).cuda(), PackedGT(tb, tc, head.dev), with_grads=True)
    torch.cuda.synchronize()
    ref = O.multibox_loss(torch.from_numpy(loc), torch.from_numpy(conf), tb, tc, pri)
    fl = full["losses"].cpu().numpy()
    assert abs(fl[0] - ref["loc_loss"].item()) <= 1e-5 * ref["loc_loss"].item()
    for rank, lo, hi, losses, sums, gl, gcf, nccl_losses, ngl, ngc, host in res:
        assert np.allclose(losses, fl, rtol=1e-6), (rank, losses, fl)                     # global losses on every rank
        assert np.allclose(sums, full["sums"].cpu().numpy(), rtol=1e-9)
        assert np.array_equal(gcf, full["grad_conf"][lo:hi].cpu().numpy())                # exact gradient slices
        assert np.array_equal(gl, full["grad_loc"][lo:hi].cpu().numpy())
        assert np.allclose(nccl_losses, fl, rtol=1e-6)
        assert np.array_equal(ngc, gcf) and np.array_equal(ngl, gl)
        # host-buffer and resident steps after xchg_import: exact gradient slices; the host path sums per chunk, so its
        # losses agree with the full batch's to rounding
        for name, (hl, hgl, hgc) in host.items():
            assert np.array_equal(hgl, gl) and np.array_equal(hgc, gcf), (rank, name)
            assert np.allclose(hl, fl, rtol=1e-6, atol=0), (rank, name, hl, fl)
    assert np.array_equal(res[0][3], res[1][3]), "both ranks must hold bit-identical global losses"
    for name in res[0][10]:                             # sum_chunks_xchg_kernel folds in rank order on every rank
        assert np.array_equal(res[0][10][name][0], res[1][10][name][0]), name
