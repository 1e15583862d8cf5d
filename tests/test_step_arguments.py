"""CPU: the return code of every loss entry point for calls with exactly one bad argument.

Each entry point gets a call whose arguments are all acceptable (fake, 16-byte aligned device addresses), and then that
call with one fault: a null required pointer, a negative or unsupported size, a pointer 4 bytes off a 16-byte
boundary, a workspace one byte short, a bad exchange argument or a bad level table.  The faulty calls must be refused
with the documented code before anything touches the device.  The acceptable call must get past every check: with no
device visible its first CUDA call fails, so it returns a positive CUDA error code.

Every call runs in a subprocess that sees no CUDA device, so a check that moved behind a launch shows up as a positive
code here, never as a kernel launched on a fake address.
"""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

BADARG, UNSUPPORTED, WORKSPACE, ALIGN = -1, -2, -3, -4
ACCEPTED = "accepted"                      # passes every check: a positive CUDA error code without a device

# argument names in the order of include/ssdhead.h
STEP_HEAD = ["loc", "conf", "gt_xyxy", "gt_cls", "gt_off", "pri_xyxy", "pri_cxcywh",
             "B", "P", "C", "sumG", "neg_ratio", "pos_iou", "sums", "losses", "grad_loc", "grad_conf",
             "cls_u8", "best_prior", "npos"]
XCHG = ["R", "rank", "seq", "peers", "xchg_local", "err_flag"]
LEVELS_HEAD = ["levels", "gt_xyxy", "gt_cls", "gt_off", "pri_xyxy", "pri_cxcywh",
               "B", "P", "C", "sumG", "neg_ratio", "pos_iou", "sums", "losses", "cls_u8", "best_prior", "npos",
               "ws_loss", "ws_loss_bytes", "ws_match", "ws_match_bytes"]
MINE_HEAD = ["loc", "conf", "gt_xyxy", "gt_cls", "gt_off", "pri_xyxy", "pri_cxcywh", "best_prior", "npos", "npos_norm",
             "cls_u8", "B", "P", "C", "neg_ratio", "pos_iou", "sums", "losses"]
WS_PAIR = ["ws_loss", "ws_loss_bytes", "ws_match", "ws_match_bytes"]
CTX_HEAD = ["ctx", "loc", "conf", "gt_xyxy", "gt_cls", "gt_off", "B", "sumG", "neg_ratio", "pos_iou", "sums", "losses"]

ENTRY_POINTS = {
    "ssdhead_ce_match_stream": ["conf", "gt_xyxy", "gt_cls", "gt_off", "pri_xyxy", "B", "P", "C", "sumG", "pos_iou",
                                "ce", "grad_loc", "grad_conf", "cls_u8", "best_prior", "npos", *WS_PAIR,
                                "run_finalizer", "stream"],
    "ssdhead_multibox_step": [*STEP_HEAD, "mined_mask", "ce", *WS_PAIR, "stream"],
    "ssdhead_multibox_step_sharded": [*STEP_HEAD, *WS_PAIR, *XCHG, "stream"],
    "ssdhead_multibox_step_resident": [*STEP_HEAD, *WS_PAIR, "ws_rows", "ws_rows_bytes", *XCHG, "stream"],
    "ssdhead_multibox_step_levels": [*LEVELS_HEAD, "stream"],
    "ssdhead_multibox_step_levels_sharded": [*LEVELS_HEAD, *XCHG, "stream"],
    "ssdhead_mine": [*MINE_HEAD, "grad_loc", "grad_conf", "mined_mask", "ce", "ws_loss", "ws_loss_bytes", "stream"],
    "ssdhead_mine_sparse": [*MINE_HEAD, "row_cap", "row_cnt", "row_idx", "grad_conf_rows", "grad_loc_rows",
                            "ws_loss", "ws_loss_bytes", "stream"],
    "ssdhead_ctx_multibox_loss_dev": [*CTX_HEAD, "grad_loc", "grad_conf", "stream"],
    "ssdhead_ctx_multibox_loss_dev_resident": [*CTX_HEAD, "grad_loc", "grad_conf", "fresh", "stream"],
    "ssdhead_ctx_multibox_loss_levels_dev": [*CTX_HEAD[:1], "levels", *CTX_HEAD[3:], "stream"],
}

SIZES = {"B", "P", "C", "sumG", "neg_ratio", "pos_iou", "run_finalizer", "R", "rank", "seq", "row_cap", "fresh",
         "ws_loss_bytes", "ws_match_bytes", "ws_rows_bytes"}
LEVEL_COUNTS = [5776, 2166, 600, 150, 36, 4]          # SSD300: P = 8732


def required_pointers(entry):
    """Pointers whose absence the entry point refuses (with sumG > 0)."""
    optional = {"ce", "mined_mask", "stream", "peers", "xchg_local", "err_flag"}     # exchange pointers: R > 1 only
    if entry != "ssdhead_multibox_step_resident":
        optional |= {"grad_loc", "grad_conf"}
    if entry.startswith("ssdhead_mine"):
        optional |= {"gt_xyxy", "gt_cls", "best_prior"}
    return [a for a in ENTRY_POINTS[entry] if a not in SIZES and a not in optional]


def aligned_pointers(entry):
    """Pointers the entry point requires 16-byte aligned.  conf and grad_conf are not among them: rows of 84 bytes
    take the plain-load path when unaligned."""
    by_entry = {
        "ssdhead_ce_match_stream": ["gt_xyxy", "pri_xyxy", "grad_loc", "ws_loss", "ws_match"],
        "ssdhead_multibox_step": ["loc", "gt_xyxy", "pri_xyxy", "pri_cxcywh", "grad_loc", "ws_loss", "ws_match"],
        "ssdhead_mine": ["loc", "gt_xyxy", "pri_xyxy", "pri_cxcywh", "grad_loc", "ws_loss"],
        "ssdhead_multibox_step_levels": ["gt_xyxy", "pri_xyxy", "pri_cxcywh", "ws_loss", "ws_match",
                                         "level_loc", "level_grad_loc"],
    }
    by_entry["ssdhead_multibox_step_sharded"] = by_entry["ssdhead_multibox_step"]
    by_entry["ssdhead_multibox_step_resident"] = by_entry["ssdhead_multibox_step"] + ["ws_rows"]
    by_entry["ssdhead_multibox_step_levels_sharded"] = by_entry["ssdhead_multibox_step_levels"]
    by_entry["ssdhead_mine_sparse"] = ["loc", "gt_xyxy", "pri_xyxy", "pri_cxcywh", "grad_loc_rows", "ws_loss"]
    return by_entry.get(entry, [])


def cases(entry):
    """(name, overrides, expected) for the acceptable call and each one-fault call of `entry`."""
    args = ENTRY_POINTS[entry]
    if entry.startswith("ssdhead_ctx_"):
        return [("null context", {}, BADARG)]           # every other argument is acceptable
    out = [("valid", {}, ACCEPTED), ("B=0", {"B": 0}, 0)]
    for p in required_pointers(entry):
        out.append((f"null {p}", {p: None}, BADARG))
    if "grad_loc" in args and entry != "ssdhead_multibox_step_resident":
        out.append(("grad_loc without grad_conf", {"grad_conf": None}, BADARG))
    out.append(("B<0", {"B": -1}, BADARG))
    if "neg_ratio" in args:
        out.append(("neg_ratio<0", {"neg_ratio": -1}, BADARG))
    out.append(("C=20", {"C": 20}, UNSUPPORTED))
    out.append(("P past the loss limit", {"P": "P_max+1"}, UNSUPPORTED))
    for p in aligned_pointers(entry):
        out.append((f"unaligned {p}", {p: "+4"}, ALIGN))
    if "conf" in args:
        out.append(("unaligned conf", {"conf": "+4"}, ACCEPTED))
    for ws in ("ws_loss_bytes", "ws_match_bytes", "ws_rows_bytes"):
        if ws in args:
            out.append((f"{ws} one byte short", {ws: "-1"}, WORKSPACE))
    if "R" in args:
        resident = entry == "ssdhead_multibox_step_resident"
        out += [("R=0", {"R": 0}, BADARG), ("R=17", {"R": 17}, BADARG),
                ("rank=R", {"rank": "R"}, BADARG), ("R=2 rank=2", {"R": 2, "rank": 2}, BADARG),
                ("R=1 seq=0", {"R": 1, "seq": 0}, ACCEPTED if resident else BADARG),
                ("R=2 seq=0", {"R": 2, "seq": 0}, BADARG),
                ("R=2 without peers", {"R": 2, "peers": None}, BADARG),
                ("R=2 without exchange buffer", {"R": 2, "xchg_local": None}, BADARG),
                ("R=2 without error flag", {"R": 2, "err_flag": None}, BADARG),
                ("R=2", {"R": 2}, ACCEPTED), ("R=16 rank=15", {"R": 16, "rank": 15}, ACCEPTED)]
    if "levels" in args:
        out += [("levels do not sum to P", {"level_counts": LEVEL_COUNTS[:-1] + [5]}, BADARG),
                ("num_levels=0", {"num_levels": 0}, BADARG),
                ("num_levels=9", {"num_levels": 9}, BADARG),
                ("a level of 0 priors", {"level_counts": [5776, 2166, 600, 186, 0, 4]}, BADARG),
                ("a level without conf", {"level_null": "conf"}, BADARG),
                ("a level without loc", {"level_null": "loc"}, BADARG),
                ("grads on some levels", {"level_grads": 3}, BADARG),
                ("a level with grad_conf only", {"level_null": "grad_loc"}, BADARG),
                ("forward-only levels", {"level_grads": 0}, ACCEPTED),
                ("unaligned level conf", {"level_conf": "+4"}, ACCEPTED)]
    if entry == "ssdhead_mine_sparse":
        out.append(("row_cap=0", {"row_cap": 0}, BADARG))
    if entry == "ssdhead_mine":
        out.append(("forward only", {"grad_loc": None, "grad_conf": None}, ACCEPTED))
    # an empty batch: which checks still run before it returns 0
    out.append(("B=0 unaligned ws_loss", {"B": 0, "ws_loss": "+4"}, 0))
    if "loc" in args:
        flat_step = entry.startswith("ssdhead_multibox_step")
        out.append(("B=0 unaligned loc", {"B": 0, "loc": "+4"}, ALIGN if flat_step else 0))
    if "levels" in args:
        out += [("B=0 unaligned pri_cxcywh", {"B": 0, "pri_cxcywh": "+4"}, 0),
                ("B=0 a level without tensors", {"B": 0, "level_null": "conf"}, 0),
                ("B=0 levels do not sum to P", {"B": 0, "level_counts": LEVEL_COUNTS[:-1] + [5]}, 0),
                ("B=0 without levels", {"B": 0, "levels": None}, BADARG),
                ("B=0 num_levels=0", {"B": 0, "num_levels": 0}, BADARG)]
    return out


CHILD = r"""
import ctypes as C, json, sys
from objectdetection_ssd_b200 import _lib
from tests.test_step_arguments import ENTRY_POINTS, LEVEL_COUNTS, cases
lib = _lib.load()
entry = sys.argv[1]
B, P, sumG = 4, sum(LEVEL_COUNTS), 10
lo, hi = P, 1 << 16                          # largest P the loss workspace query accepts
while hi - lo > 1:
    mid = (lo + hi) // 2
    lo, hi = (mid, hi) if lib.ssdhead_workspace_bytes(_lib.WS_LOSS, B, mid, 21, 0) else (lo, mid)
P_max = lo
addr = [0x7f0000000000]
def fake():
    addr[0] += 1 << 24
    return addr[0]
results = []
for name, ov, _ in cases(entry):
    v = {"B": B, "P": P, "C": 21, "sumG": sumG, "neg_ratio": 3, "pos_iou": 0.5, "run_finalizer": 1,
         "R": 1, "rank": 0, "seq": 1, "row_cap": 64, "fresh": 0, "stream": None, "ce": None, "mined_mask": None,
         "ctx": None}
    if "R" in ENTRY_POINTS[entry] and entry.endswith("_sharded"):
        v["R"] = 2
    v.update({k: x for k, x in ov.items() if k in ("B", "P", "C", "R", "rank", "seq", "neg_ratio", "row_cap")})
    if v["P"] == "P_max+1":
        v["P"] = P_max + 1
    if v["rank"] == "R":
        v["rank"] = v["R"]
    Bq, Pq = max(v["B"], 0), v["P"]
    v["ws_loss_bytes"] = lib.ssdhead_workspace_bytes(_lib.WS_LOSS, Bq, Pq, 21, 0) or (1 << 40)
    v["ws_match_bytes"] = lib.ssdhead_workspace_bytes(_lib.WS_MATCH, Bq, Pq, 21, sumG)
    v["ws_rows_bytes"] = lib.ssdhead_workspace_bytes(_lib.WS_ROWS, Bq, Pq, 21, 0)
    counts = ov.get("level_counts", LEVEL_COUNTS if Pq == P else LEVEL_COUNTS[:-1] + [LEVEL_COUNTS[-1] + Pq - P])
    lv = _lib.Levels()
    lv.num_levels = ov.get("num_levels", len(counts))
    ng = ov.get("level_grads", len(counts))
    for l, n in enumerate(counts):
        lv.count[l] = n
        lv.conf[l], lv.loc[l] = fake(), fake()
        if l < ng:
            lv.grad_conf[l], lv.grad_loc[l] = fake(), fake()
    for key, field in (("level_loc", "loc"), ("level_grad_loc", "grad_loc"), ("level_conf", "conf")):
        if key in ov:
            getattr(lv, field)[1] += 4
    if "level_null" in ov:
        getattr(lv, ov["level_null"])[2] = None
    v["levels"] = C.addressof(lv)
    call = []
    for a in ENTRY_POINTS[entry]:
        x = v[a] if a in v else fake()
        o = ov.get(a)
        if a in ov and o is None:
            x = None
        elif o == "+4":
            x += 4
        elif o == "-1":
            x -= 1
        call.append(x)
    rc = getattr(lib, entry)(*call)
    results.append([name, rc])
print(json.dumps(results))
"""


@pytest.mark.parametrize("entry", sorted(ENTRY_POINTS))
def test_one_fault_calls_get_the_documented_code(entry):
    res = subprocess.run([sys.executable, "-c", CHILD, entry], capture_output=True, text=True, cwd=ROOT,
                         env=dict(os.environ, CUDA_VISIBLE_DEVICES=""), timeout=300)
    assert res.returncode == 0, res.stderr
    got = dict(json.loads(res.stdout.strip().splitlines()[-1]))
    expected = {name: want for name, _, want in cases(entry)}
    assert set(got) == set(expected)
    wrong = {name: (got[name], want) for name, want in expected.items()
             if not (got[name] > 0 if want == ACCEPTED else got[name] == want)}
    assert not wrong, f"{entry}: case -> (returned, expected) {wrong}"
