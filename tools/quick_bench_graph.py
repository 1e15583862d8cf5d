"""Developer timing of the training-head step captured into a CUDA graph (StaticHead) against the eager calls.

Per batch size (32 and 256 by default), one JSON line with:
  eager_ssd_ms      (a) Losses.ssd() + backward() from host gt lists, host clock per step (ends in a synchronise)
  graph_step_ms     (b) StaticHead.load_packed() of collate_gt output + replay of the captured loss + backward, host clock
  graph_gpu_ms      (c) CUDA-event time per step of (b)
  ctx_eager_gpu_ms      CUDA-event time per step of eager SSDHeadContext.loss_dev (device gts)
  ctx_graph_gpu_ms      CUDA-event time per replay of a graph holding only SSDHeadContext.loss_dev (sumG = capacity):
                        the same two kernels, so the difference to ctx_eager_gpu_ms is what capture does to the
                        programmatic overlap of the streaming and mining kernels
The event timings alternate three times.  Every step reads the same loc / conf (at batch 32 they stay in L2).  The card
name and power limit are printed with the numbers.

    python tools/quick_bench_graph.py [--batches 32 256] [--steps 200]
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from objectdetection_ssd_b200 import Losses, synth  # noqa: E402
from objectdetection_ssd_b200.collate import collate_gt  # noqa: E402
from objectdetection_ssd_b200.ctx import SSDHeadContext  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[torch.cuda.current_device()] if q.returncode == 0 else torch.cuda.get_device_name()


def host_ms(fn, steps):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(steps):
        fn(i)
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3 / steps


def gpu_ms(fn, steps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for i in range(steps):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def run(B, steps, max_per_image=16):
    pri = Losses.ancs_xywh
    P = pri.shape[0]
    nb = 8
    lists = []
    for k in range(nb):
        gb, gc = synth.make_gt(50 + k, B, 1, max_per_image)
        lists.append(([torch.from_numpy(b) for b in gb], [torch.from_numpy(c) for c in gc]))
    packed = [collate_gt(b, c) for b, c in lists]
    l0, c0 = (torch.from_numpy(a).cuda() for a in synth.make_head(50, B, P))
    loc, conf = l0.clone().requires_grad_(), c0.clone().requires_grad_()

    def eager(i):
        tb, tc = lists[i % nb]
        loc.grad = conf.grad = None
        a, b = Losses.ssd((loc, conf), tc, tb)
        (a + b).backward()

    sh = Losses.StaticHead(pri, B, max_per_image * B, "cuda")
    sh.load_packed(*packed[0])

    def step():
        loc.grad = conf.grad = None
        a, b = sh.loss(loc, conf)
        (a + b).backward()

    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        step()
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        step()

    def replay(i):
        sh.load_packed(*packed[i % nb])
        g.replay()

    # the context's device step, eager and captured (sumG = capacity), on device copies of the same gts
    cap = max_per_image * B
    ctx_e = SSDHeadContext(pri.numpy(), max_batch=B, max_total_gt=cap)
    ctx_g = SSDHeadContext(pri.numpy(), max_batch=B, max_total_gt=cap)
    dev = [tuple(torch.from_numpy(a).cuda() for a in p) for p in packed]
    sums, losses = torch.empty(2, dtype=torch.float64, device="cuda"), torch.empty(2, device="cuda")
    gl, gcf = torch.empty_like(l0), torch.empty_like(c0)
    st = torch.cuda.current_stream().cuda_stream
    gx_s = torch.zeros(cap, 4, device="cuda")
    gc_s = torch.zeros(cap, device="cuda")
    off_s = dev[0][2].clone()
    n0 = int(dev[0][2][-1])
    gx_s[:n0].copy_(dev[0][0])
    gc_s[:n0].copy_(dev[0][1])

    def ctx_eager(i):
        gx, gcl, off = dev[i % nb]
        ctx_e.loss_dev(l0.data_ptr(), c0.data_ptr(), gx.data_ptr(), gcl.data_ptr(), off.data_ptr(), B, int(gx.shape[0]),
                       sums.data_ptr(), losses.data_ptr(), gl.data_ptr(), gcf.data_ptr(), st)

    def ctx_step():
        ctx_g.loss_dev(l0.data_ptr(), c0.data_ptr(), gx_s.data_ptr(), gc_s.data_ptr(), off_s.data_ptr(), B, cap,
                       sums.data_ptr(), losses.data_ptr(), gl.data_ptr(), gcf.data_ptr(),
                       torch.cuda.current_stream().cuda_stream)

    ctx_step()
    torch.cuda.synchronize()
    g2 = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g2):
        ctx_step()

    for fn in (eager, replay, ctx_eager, lambda i: g2.replay()):
        for i in range(10):
            fn(i)
    r = dict(B=B, steps=steps, gts_per_image=f"1..{max_per_image}", capacity=cap,
             eager_ssd_ms=round(host_ms(eager, steps), 4), graph_step_ms=round(host_ms(replay, steps), 4),
             graph_gpu_ms=[], ctx_eager_gpu_ms=[], ctx_graph_gpu_ms=[])
    for _ in range(3):
        r["graph_gpu_ms"].append(round(gpu_ms(replay, steps), 4))
        r["ctx_eager_gpu_ms"].append(round(gpu_ms(ctx_eager, steps), 4))
        r["ctx_graph_gpu_ms"].append(round(gpu_ms(lambda i: g2.replay(), steps), 4))
    del g, g2
    ctx_e.close()
    ctx_g.close()
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", type=int, nargs="+", default=[32, 256])
    ap.add_argument("--steps", type=int, default=200)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("quick_bench_graph.py needs a CUDA device")
    gpu = card()
    for B in args.batches:
        r = run(B, args.steps)
        r["gpu"] = gpu
        print(json.dumps(r), flush=True)


if __name__ == "__main__":
    main()
