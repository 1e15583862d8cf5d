"""Developer timing loop for detect on the outputs of a trained head (tests/test_gpu_detect_trained.py's generator:
margins 10 / 17 / 25 / 40, a large object and a multi-object image with thousands of scores at exactly 1.0, images with
few candidates).  Both routes forced through SSDHEAD_DETECT_SHORTLIST, batches 64 / 128 / 256, min_score 0.01,
top_k 200; prints the step time of each and the short-list route's fallback count (images listed twice).

    python tools/quick_bench_detect_trained.py [steps]
"""
import ctypes
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from objectdetection_ssd_b200 import _lib
from objectdetection_ssd_b200.head import MultiboxHead
from tests.test_gpu_detect_trained import KINDS, trained_batch


def run(B, shortlist, steps=50, warm=5, top_k=200, min_score=0.01):
    pri, loc, conf, _ = trained_batch(3000, KINDS * (B // len(KINDS)))
    P = pri.shape[0]
    head = MultiboxHead(pri, "cuda")
    lib = _lib.load()
    loc, conf = loc.cuda().contiguous(), conf.cuda().contiguous()
    ob = torch.empty(B, top_k, 4, device="cuda"); op = torch.empty(B, top_k, device="cuda")
    oc = torch.empty(B, top_k, dtype=torch.int32, device="cuda"); oi = torch.empty_like(oc)
    on = torch.empty(B, dtype=torch.int32, device="cuda")
    ws = torch.zeros(int(lib.ssdhead_workspace_bytes(_lib.WS_DETECT, B, P, 21, 0)), dtype=torch.uint8, device="cuda")
    st = torch.cuda.current_stream().cuda_stream
    os.environ["SSDHEAD_DETECT_SHORTLIST"] = "1" if shortlist else "0"

    def step():
        return lib.ssdhead_detect(loc.data_ptr(), conf.data_ptr(), head.pri_cxcywh.data_ptr(), B, P, 21, min_score, 0.45,
                                  top_k, None, 0, ob.data_ptr(), op.data_ptr(), oc.data_ptr(), oi.data_ptr(),
                                  on.data_ptr(), ws.data_ptr(), ws.numel(), st)
    for _ in range(warm):
        _lib.check(step(), "ssdhead_detect")
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    nfb = ctypes.c_int32(-1)
    _lib.check(lib.ssdhead_detect_fallbacks(ws.data_ptr(), ws.numel(), B, P, 21, 0, ctypes.addressof(nfb), st),
               "ssdhead_detect_fallbacks")
    print(json.dumps(dict(B=B, route="shortlist" if shortlist else "exhaustive", fallbacks=nfb.value,
                          step_us=round(e0.elapsed_time(e1) / steps * 1e3, 1), kept=on.sum().item())))


if __name__ == "__main__":
    steps = int(sys.argv[1]) if len(sys.argv) > 1 else 50
    print(torch.cuda.get_device_name())
    for B in (64, 128, 256):
        for rep in range(2):                      # alternate the routes twice
            for shortlist in (True, False):
                run(B, shortlist, steps)
    os.environ.pop("SSDHEAD_DETECT_SHORTLIST", None)
