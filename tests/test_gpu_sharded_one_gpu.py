"""The image-sharded training step on ONE GPU: the R ranks of a sharded batch run one after another on one stream.

The sharded mining kernel of rank r publishes its positive count and its two loss sums by storing them into the
exchange buffer of every rank (its own included), and it waits only for words in its OWN buffer (csrc/loss.cu,
mine_body).  So the ranks can run in turn, each on its own buffer, once the words of the ranks that have not run yet
are written into that buffer beforehand (the "prefill").  What a rank publishes does not depend on the other ranks: its
own positive count, and its loss sums before normalisation - what the plain single-GPU step returns for the same shard.
With the right words no wait spins; every wait is bounded anyway (it sets err_flag and continues), so nothing here can
hang, and every step asserts err_flag == 0.

Exchange buffer layout (csrc/common.cuh:250-252): XCHG_WORDS = 2 * 4 * 16 int64 words,
    slot(seq, what, q) = ((seq & 1) * 4 + what) * 16 + q
    what = 0: seq << 32 | npos_q      what = 1, 2: bits of rank q's float64 sum_l1, sum_ce      what = 3: seq
After a step every buffer must hold exactly the words of all R ranks for that step, in the slots of its parity, next to
the previous step's words in the other parity: the test keeps that table and compares every buffer with it, which also
checks that the prefilled words (taken from the plain step) are the bits the sharded ranks store.

Each rank's outputs are compared bit for bit with its slice of the full batch on one GPU; the full batch itself is
pinned to the float64 reference of test_gpu_trained_regime.py, and the sharded sums must lie within the same budget.
The NCCL route (head.loss with a process group) and the two-halves API of the context run here too, with a test-local
all-reduce.  The one thing that needs two processes - opening another process's IPC handle - stays in
test_gpu_sharded.py.
"""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from objectdetection_ssd_b200 import _lib
from objectdetection_ssd_b200.dist import shard_range
from tests import helpers as H
from tests.test_gpu_trained_regime import CASES, EPS, case_inputs, check_against_references, same_bits

C = 21
XCHG_MAX_R = 16
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LEVEL_COUNTS = (5776, 2166, 600, 150, 36, 4)


def slot(seq, what, q):
    """Index of word `what` of rank q for step `seq` in an exchange buffer (csrc/common.cuh:252)."""
    return ((seq & 1) * 4 + what) * XCHG_MAX_R + q


def f64_bits(x):
    return int(np.array([x], np.float64).view(np.int64)[0])


def test_slot_formula_matches_the_source():
    """The layout restated above is the one csrc/common.cuh defines."""
    with open(os.path.join(ROOT, "objectdetection_ssd_b200", "csrc", "common.cuh")) as f:
        src = f.read()
    assert re.search(r"constexpr int XCHG_MAX_R = 16;", src)
    assert re.search(r"constexpr int XCHG_WORDS = 2 \* 4 \* XCHG_MAX_R;", src)
    assert "return ((int)(seq & 1u) * 4 + what) * XCHG_MAX_R + rank;" in src
    assert sorted(slot(s, w, q) for s in (1, 2) for w in range(4) for q in range(16)) == list(range(128))


# ----------------------------------------------------------------------------------------------------------- harness
def _lib_():
    return _lib.load()


def _st():
    return torch.cuda.current_stream().cuda_stream


def _head(pri):
    from objectdetection_ssd_b200.head import MultiboxHead
    return MultiboxHead(pri, "cuda")


def _gt(head, tb, tc):
    from objectdetection_ssd_b200.head import PackedGT
    return PackedGT(tb, tc, head.dev)


def cpu(o):
    return {k: v.cpu() for k, v in o.items() if torch.is_tensor(v)}


class Emulation:
    """R ranks on one GPU: per rank an exchange buffer (int64 words, zeroed once, reused across steps) and an int32
    err_flag; one device table of the R buffer addresses, indexed by rank, shared by all ranks."""

    def __init__(self, R):
        self.R = R
        self.nwords = int(_lib_().ssdhead_xchg_bytes()) // 8
        assert self.nwords == 2 * 4 * XCHG_MAX_R
        self.xchg = [torch.zeros(self.nwords, dtype=torch.int64, device="cuda") for _ in range(R)]
        self.err = [torch.zeros(1, dtype=torch.int32, device="cuda") for _ in range(R)]
        self.peers = torch.tensor([b.data_ptr() for b in self.xchg], dtype=torch.int64, device="cuda")
        self.table = np.zeros((R, self.nwords), np.int64)      # what every buffer must hold
        self.seq = 0

    def xargs(self, rank):
        """The trailing arguments of the sharded entry points for `rank` at the current step."""
        return (self.R, rank, self.seq, self.peers.data_ptr(), self.xchg[rank].data_ptr(), self.err[rank].data_ptr(), _st())

    def step(self, plains, launch, prefill=None):
        """One step: `plains[q]` = (own count, sums [2] float64) of rank q from the plain step on its shard; `launch(r)`
        enqueues rank r and returns its outputs.  Before rank r, the words of every rank q > r go into r's buffer
        (`prefill`, if given, replaces that list of (q, words) pairs).  Checks err_flag and the full word table of
        every buffer; returns the ranks' outputs on the host."""
        self.seq += 1
        seq = self.seq
        words = [((seq << 32) | int(n), f64_bits(float(s[0])), f64_bits(float(s[1])), seq) for n, s in plains]
        outs = []
        ranks = range(self.R) if prefill is None else [0]
        for r in ranks:
            pre = [(q, words[q]) for q in range(r + 1, self.R)] if prefill is None else prefill(words)
            for q, w in pre:
                for what in range(4):
                    self.xchg[r][slot(seq, what, q)] = w[what]
            outs.append(launch(r))
        torch.cuda.synchronize()
        for r in ranks:
            assert int(self.err[r].item()) == 0, f"rank {r}: a wait for a peer expired"
        if prefill is None:
            for b in range(self.R):
                for q in range(self.R):
                    for what in range(4):
                        self.table[b, slot(seq, what, q)] = words[q][what]
                got = self.xchg[b].cpu().numpy()
                bad = np.nonzero(got != self.table[b])[0]
                assert bad.size == 0, (f"step {seq}: exchange buffer of rank {b} differs from the word table at slots "
                                       f"{bad.tolist()[:8]}: {got[bad][:8].tolist()} vs {self.table[b][bad][:8].tolist()}")
        return [cpu(o) for o in outs]


class Shard:
    """Rank r's slice of a batch: device inputs, packed gts, its range and gt offsets in the full batch."""

    def __init__(self, head, loc, conf, tb, tc, r, R):
        self.lo, self.hi = shard_range(r, R, int(loc.shape[0]))
        self.B = self.hi - self.lo
        self.loc = loc[self.lo:self.hi].cuda().contiguous()
        self.conf = conf[self.lo:self.hi].cuda().contiguous()
        self.gt = _gt(head, tb[self.lo:self.hi], tc[self.lo:self.hi])
        counts = [int(b.shape[0]) for b in tb]
        self.g0, self.g1 = sum(counts[:self.lo]), sum(counts[:self.hi])


def plain_step(head, sh):
    """ssdhead_multibox_step on the shard alone: the count and the sums that rank publishes."""
    o = head.loss(sh.loc, sh.conf, sh.gt, with_grads=True)
    return o


def _outputs(head, sh, grads=True):
    o = dict(sums=torch.empty(2, dtype=torch.float64, device="cuda"), losses=torch.empty(2, device="cuda"),
             **{k: v for k, v in head._match_outputs(sh.gt, False).items() if v is not None})
    if grads:
        o["grad_loc"], o["grad_conf"] = torch.empty_like(sh.loc), torch.empty_like(sh.conf)
    return o


def _ws(head, sh):
    ws = head._workspace(_lib.WS_LOSS, sh.B, 0)
    wm = head._workspace(_lib.WS_MATCH, sh.B, sh.gt.sumG)
    return ws, wm


def sharded_flat(head, sh, xargs):
    """ssdhead_multibox_step_sharded for one rank."""
    o = _outputs(head, sh)
    ws, wm = _ws(head, sh)
    _lib.check(_lib_().ssdhead_multibox_step_sharded(
        sh.loc.data_ptr(), sh.conf.data_ptr(), sh.gt.boxes.data_ptr(), sh.gt.classes.data_ptr(), sh.gt.off.data_ptr(),
        head.pri_xyxy.data_ptr(), head.pri_cxcywh.data_ptr(), sh.B, head.P, C, sh.gt.sumG, 3, 0.5,
        o["sums"].data_ptr(), o["losses"].data_ptr(), o["grad_loc"].data_ptr(), o["grad_conf"].data_ptr(),
        o["cls_u8"].data_ptr(), o["best_prior"].data_ptr(), o["npos"].data_ptr(),
        ws.data_ptr(), ws.numel(), wm.data_ptr(), wm.numel(), *xargs), "ssdhead_multibox_step_sharded")
    return o


def level_bounds(P):
    counts = LEVEL_COUNTS if P == sum(LEVEL_COUNTS) else (P // 2, P - P // 2)
    return list(zip(np.cumsum((0,) + counts)[:-1], np.cumsum(counts)))


def levels_struct(loc, conf, P):
    """The six per-level tensors (and their gradients) of flat [B,P,*] tensors; returns (struct, kept tensors)."""
    st = _lib.Levels()
    keep = []
    bounds = level_bounds(P)
    st.num_levels = len(bounds)
    for i, (a, b) in enumerate(bounds):
        lc, cc = loc[:, a:b].contiguous(), conf[:, a:b].contiguous()
        gl, gc = torch.empty_like(lc), torch.empty_like(cc)
        keep.append((lc, cc, gl, gc))
        st.count[i] = int(b - a)
        st.loc[i], st.conf[i], st.grad_loc[i], st.grad_conf[i] = lc.data_ptr(), cc.data_ptr(), gl.data_ptr(), gc.data_ptr()
    return st, keep


def sharded_levels(head, sh, xargs):
    """ssdhead_multibox_step_levels_sharded for one rank; gradients concatenated back to [B,P,*]."""
    o = _outputs(head, sh, grads=False)
    st, keep = levels_struct(sh.loc, sh.conf, head.P)
    ws, wm = _ws(head, sh)
    _lib.check(_lib_().ssdhead_multibox_step_levels_sharded(
        ctypes.addressof(st), sh.gt.boxes.data_ptr(), sh.gt.classes.data_ptr(), sh.gt.off.data_ptr(),
        head.pri_xyxy.data_ptr(), head.pri_cxcywh.data_ptr(), sh.B, head.P, C, sh.gt.sumG, 3, 0.5,
        o["sums"].data_ptr(), o["losses"].data_ptr(), o["cls_u8"].data_ptr(), o["best_prior"].data_ptr(),
        o["npos"].data_ptr(), ws.data_ptr(), ws.numel(), wm.data_ptr(), wm.numel(), *xargs),
        "ssdhead_multibox_step_levels_sharded")
    o["grad_loc"] = torch.cat([k[2] for k in keep], 1)
    o["grad_conf"] = torch.cat([k[3] for k in keep], 1)
    return o


class Resident:
    """A rank's resident gradient tensors and rows workspace, for up to maxB images, zero-filled once."""

    def __init__(self, head, maxB):
        self.gl = torch.zeros(maxB, head.P, 4, device="cuda")
        self.gc = torch.zeros(maxB, head.P, C, device="cuda")
        n = int(_lib_().ssdhead_workspace_bytes(_lib.WS_ROWS, maxB, head.P, C, 0))
        self.rows = torch.zeros(n, dtype=torch.uint8, device="cuda")


def sharded_resident(head, sh, res, xargs):
    """ssdhead_multibox_step_resident with R > 1 for one rank; the gradients are views of the resident tensors."""
    o = _outputs(head, sh, grads=False)
    ws, wm = _ws(head, sh)
    _lib.check(_lib_().ssdhead_multibox_step_resident(
        sh.loc.data_ptr(), sh.conf.data_ptr(), sh.gt.boxes.data_ptr(), sh.gt.classes.data_ptr(), sh.gt.off.data_ptr(),
        head.pri_xyxy.data_ptr(), head.pri_cxcywh.data_ptr(), sh.B, head.P, C, sh.gt.sumG, 3, 0.5,
        o["sums"].data_ptr(), o["losses"].data_ptr(), res.gl.data_ptr(), res.gc.data_ptr(),
        o["cls_u8"].data_ptr(), o["best_prior"].data_ptr(), o["npos"].data_ptr(),
        ws.data_ptr(), ws.numel(), wm.data_ptr(), wm.numel(), res.rows.data_ptr(), res.rows.numel(), *xargs),
        "ssdhead_multibox_step_resident")
    o["grad_loc"], o["grad_conf"] = res.gl[:sh.B].clone(), res.gc[:sh.B].clone()
    return o


# ----------------------------------------------------------------------------------------------------------- checks
def full_batch(head, loc, conf, tb, tc):
    """The single-GPU step on the whole batch, with the taps."""
    o = head.loss(loc.cuda().contiguous(), conf.cuda().contiguous(), _gt(head, tb, tc), with_grads=True, taps=True)
    return cpu(o)


def compare_rank(o, full, sh, what=""):
    """Rank outputs `o` against the shard's slice of the full batch: gradients, class map, per-image counts and the
    shard's best priors bit for bit; npos[B] is the rank's own count."""
    lo, hi, B = sh.lo, sh.hi, sh.B
    assert same_bits(o["grad_loc"], full["grad_loc"][lo:hi]), f"{what}grad_loc differs from the full-batch slice"
    assert same_bits(o["grad_conf"], full["grad_conf"][lo:hi]), f"{what}grad_conf differs from the full-batch slice"
    assert torch.equal(o["cls_u8"], full["cls_u8"][lo:hi]), f"{what}class map"
    assert torch.equal(o["npos"][:B], full["npos"][lo:hi]), f"{what}positives per image"
    assert int(o["npos"][B]) == int(full["npos"][lo:hi].sum()), f"{what}npos[B] is not the rank's own count"
    assert torch.equal(o["best_prior"][:sh.g1 - sh.g0], full["best_prior"][sh.g0:sh.g1]), f"{what}best priors"


def fold(plains):
    """The float64 sums every rank must return: 0.0 + s_0 + s_1 + ... in rank order."""
    a, c = 0.0, 0.0
    for _, s in plains:
        a += float(s[0])
        c += float(s[1])
    return a, c


def check_global(outs, plains, N):
    """sums and losses identical in bits on every rank: the rank-order fold and its fp32 quotients by the global N."""
    a, c = fold(plains)
    want_s = torch.tensor([a, c], dtype=torch.float64)
    want_l = torch.tensor([np.float32(a / (4.0 * N)), np.float32(c / N)], dtype=torch.float32)
    for r, o in enumerate(outs):
        assert same_bits(o["sums"], want_s), (r, o["sums"].tolist(), [a, c])
        assert same_bits(o["losses"], want_l), (r, o["losses"].tolist(), want_l.tolist())


def pin_full_batch(pri, loc, conf, tb, tc, full):
    """The full batch against the float64 reference (check_against_references); returns the budgets of its two sums:
    (float64 L1, its budget), (float64 sum of the CE taps over positives and mined rows, its budget)."""
    _, r, ref, mined = check_against_references(pri, loc, conf, tb, tc, full)
    l1 = r["sums"][0]
    b1 = EPS * (0.5 * np.abs(r["dl"]) + 4.0 * np.abs(r["tgt"])).sum() + 1e-12 * l1
    sel = ref["pos"].numpy() | mined.numpy()
    tap_sum = full["ce"].double().numpy()[sel].sum()
    return (l1, b1), (tap_sum, 1e-12 * abs(tap_sum))


def run_sharded_case(pri, loc, conf, tb, tc, R, em=None, heads=None, plain=None, pin=True):
    """One batch through the emulated ranks; every check of the module.  Returns (rank outputs, full batch, shards)."""
    plain = plain or _head(pri)
    heads = heads or [_head(pri) for _ in range(R)]
    em = em or Emulation(R)
    full = full_batch(plain, loc, conf, tb, tc)
    shards = [Shard(plain, loc, conf, tb, tc, r, R) for r in range(R)]
    pl = [cpu(plain_step(plain, sh)) for sh in shards]
    plains = [(int(p["npos"][sh.B]), p["sums"]) for p, sh in zip(pl, shards)]
    outs = em.step(plains, lambda r: sharded_flat(heads[r], shards[r], em.xargs(r)))
    for r, (o, sh) in enumerate(zip(outs, shards)):
        compare_rank(o, full, sh, f"rank {r}: ")
    N = int(full["npos"][loc.shape[0]])
    assert sum(n for n, _ in plains) == N
    check_global(outs, plains, N)
    if pin:
        (l1, b1), (s1, b2) = pin_full_batch(pri, loc, conf, tb, tc, full)
        s = outs[0]["sums"]
        assert abs(float(s[0]) - l1) <= b1, (float(s[0]), l1, b1)
        assert abs(float(s[1]) - s1) <= b2, (float(s[1]), s1, b2)
    return outs, full, shards, plains


# ----------------------------------------------------------------------------------------------------------- tests
SHAPES = [(12, 2), (37, 3), (16, 16), (64, 8), (256, 2)]


@pytest.mark.gpu
@pytest.mark.parametrize("B_total,R", SHAPES)
def test_sharded_equals_full_batch(B_total, R):
    """Ordinary heads; uneven shards (37 over 3), one image per rank at the largest R, a full-size batch."""
    pri = H.priors()
    loc, conf, tb, tc = H.train_inputs(400 + B_total, B_total, pri.shape[0])
    run_sharded_case(pri, loc, conf, tb, tc, R)


@pytest.mark.gpu
@pytest.mark.parametrize("name", CASES)
def test_sharded_trained_head_equals_full_batch(name):
    """The trained-head families of test_gpu_trained_regime.py (zero-CE ties, radix selection, +-1e4 rows, bf16
    logits), 7 images over 3 ranks."""
    pri, loc, conf, tb, tc = case_inputs(name, B=7)
    run_sharded_case(pri, loc, conf, tb, tc, 3)


@pytest.mark.gpu
def test_sharded_stress_ssd512_100_gts():
    """SSD512 priors, 100 gts per image (the seeded cull of the fused match is on), 8 images over 4 ranks."""
    pri = H.priors("ssd512")
    loc, conf, tb, tc = H.train_inputs(512, 8, pri.shape[0], 100, 100)
    run_sharded_case(pri, loc, conf, tb, tc, 4)


@pytest.mark.gpu
def test_sharded_several_steps_reuse_both_parity_slots():
    """Four steps (seq 1-4) on the same buffers, a different batch and different shard sizes each step: both parity
    slots are reused while the words of the step before last are still in them."""
    pri = H.priors()
    R = 3
    em, heads, plain = Emulation(R), [_head(pri) for _ in range(R)], _head(pri)
    for i, B_total in enumerate((12, 7, 20, 5)):
        loc, conf, tb, tc = H.train_inputs(600 + i, B_total, pri.shape[0])
        run_sharded_case(pri, loc, conf, tb, tc, R, em=em, heads=heads, plain=plain)
    assert em.seq == 4


@pytest.mark.gpu
@pytest.mark.parametrize("B_total,R", [(12, 2), (37, 3)])
def test_levels_sharded_equals_flat_sharded(B_total, R):
    """ssdhead_multibox_step_levels_sharded on the six SSD300 level tensors gives the bits of the flat sharded step."""
    pri = H.priors()
    loc, conf, tb, tc = H.train_inputs(700 + B_total, B_total, pri.shape[0])
    em, heads, plain = Emulation(R), [_head(pri) for _ in range(R)], _head(pri)
    flat, full, shards, plains = run_sharded_case(pri, loc, conf, tb, tc, R, em=em, heads=heads, plain=plain, pin=False)
    lv = em.step(plains, lambda r: sharded_levels(heads[r], shards[r], em.xargs(r)))
    for r, (a, b) in enumerate(zip(lv, flat)):
        for key in ("sums", "losses", "grad_loc", "grad_conf"):
            assert same_bits(a[key], b[key]), f"rank {r}: {key}"
        for key in ("cls_u8", "npos"):
            assert torch.equal(a[key], b[key]), f"rank {r}: {key}"
        assert torch.equal(a["best_prior"][:shards[r].g1 - shards[r].g0], b["best_prior"][:shards[r].g1 - shards[r].g0])


@pytest.mark.gpu
def test_resident_sharded_equals_dense_sharded():
    """ssdhead_multibox_step_resident with R = 2 over a plan with a smaller batch after a larger one and repeated
    inputs: after every step the first B images of each rank's resident tensors hold the bits of the dense sharded
    step (the rows of images beyond B stay listed until those images return, include/ssdhead.h)."""
    pri = H.priors()
    R = 2
    plan = [(12, 0), (6, 1), (6, 1), (12, 2), (12, 2), (10, 3)]        # (images, input seed)
    maxB = max(shard_range(0, R, b)[1] for b, _ in plan)
    heads, res_heads, plain = [_head(pri) for _ in range(R)], [_head(pri) for _ in range(R)], _head(pri)
    em_dense, em_res = Emulation(R), Emulation(R)
    res = [Resident(plain, maxB) for _ in range(R)]
    for B_total, seed in plan:
        loc, conf, tb, tc = H.train_inputs(800 + seed, B_total, pri.shape[0])
        dense, full, shards, plains = run_sharded_case(pri, loc, conf, tb, tc, R, em=em_dense, heads=heads, plain=plain,
                                                       pin=False)
        outs = em_res.step(plains, lambda r: sharded_resident(res_heads[r], shards[r], res[r], em_res.xargs(r)))
        for r, (a, b) in enumerate(zip(outs, dense)):
            for key in ("sums", "losses", "grad_loc", "grad_conf"):
                assert same_bits(a[key], b[key]), f"B={B_total} seed {seed} rank {r}: {key}"
            for key in ("cls_u8", "npos"):
                assert torch.equal(a[key], b[key]), f"B={B_total} seed {seed} rank {r}: {key}"


@pytest.mark.gpu
def test_one_rank_through_the_sharded_entry_points_is_the_plain_step():
    """R = 1 through ssdhead_multibox_step_sharded and _levels_sharded: the bits of ssdhead_multibox_step."""
    pri = H.priors()
    loc, conf, tb, tc = H.train_inputs(901, 9, pri.shape[0])
    head, plain = _head(pri), _head(pri)
    sh = Shard(plain, loc, conf, tb, tc, 0, 1)
    want = cpu(plain_step(plain, sh))
    em = Emulation(1)
    em.seq = 1
    flat = cpu(sharded_flat(head, sh, em.xargs(0)))
    lv = cpu(sharded_levels(head, sh, em.xargs(0)))
    torch.cuda.synchronize()
    assert int(em.err[0].item()) == 0
    for got in (flat, lv):
        for key in ("sums", "losses", "grad_loc", "grad_conf"):
            assert same_bits(got[key], want[key]), key
        for key in ("cls_u8", "npos", "best_prior"):
            assert torch.equal(got[key], want[key]), key


@pytest.mark.gpu
def test_wrong_prefilled_count_is_detected():
    """The comparison can fail: rank 0 of two runs alone with rank 1's count prefilled one too high.  The word is
    well-formed (err_flag stays 0), so rank 0 normalises by N + 1: its gradients and losses must differ from the
    full-batch slices, and compare_rank / check_global must say so."""
    pri = H.priors()
    loc, conf, tb, tc = H.train_inputs(902, 12, pri.shape[0])
    R = 2
    plain, head = _head(pri), _head(pri)
    full = full_batch(plain, loc, conf, tb, tc)
    shards = [Shard(plain, loc, conf, tb, tc, r, R) for r in range(R)]
    pl = [cpu(plain_step(plain, sh)) for sh in shards]
    plains = [(int(p["npos"][sh.B]), p["sums"]) for p, sh in zip(pl, shards)]
    em = Emulation(R)

    def wrong(words):
        w = list(words[1])
        w[0] += 1                                   # seq << 32 | (npos_1 + 1)
        return [(1, tuple(w))]

    outs = em.step(plains, lambda r: sharded_flat(head, shards[r], em.xargs(r)), prefill=wrong)
    N = int(full["npos"][12])
    assert int(outs[0]["npos"][shards[0].B]) == plains[0][0]
    assert not same_bits(outs[0]["grad_conf"], full["grad_conf"][:shards[0].B])
    with pytest.raises(AssertionError, match="grad_loc|grad_conf"):
        compare_rank(outs[0], full, shards[0])
    with pytest.raises(AssertionError):
        check_global(outs, plains, N)
    # normalised by N + 1, everything else as the right step
    a, c = fold(plains)
    assert same_bits(outs[0]["losses"], torch.tensor([np.float32(a / (4.0 * (N + 1))), np.float32(c / (N + 1))]))


# ----------------------------------------------------------------------------------------------------------- NCCL route
class _Group:
    """Sentinel process group of the test-local all-reduce."""


def _fake_all_reduce(monkeypatch, sentinel, N, plain_sums, fold_sums):
    """torch.distributed.all_reduce for the group `sentinel`: the int32 count becomes the global N; the float64 sums
    must arrive as this rank's plain-step sums (bit for bit) and become the rank-order fold.  plain_sums: a one-item
    list, set per rank."""
    import torch.distributed as dist
    calls = []

    def fake(t, op=None, group=None, async_op=False):
        assert group is sentinel and op == dist.ReduceOp.SUM
        if t.dtype == torch.int32:
            t.fill_(N)
        else:
            assert t.dtype == torch.float64
            assert same_bits(t.cpu(), plain_sums[0]), ("sums handed to the all-reduce", t.tolist(), plain_sums[0].tolist())
            t.copy_(torch.tensor(fold_sums, dtype=torch.float64))
        calls.append(t.dtype)

    monkeypatch.setattr(dist, "all_reduce", fake)
    return calls


@pytest.mark.gpu
@pytest.mark.parametrize("B_total,R", [(12, 2), (37, 3)])
def test_nccl_route_with_a_local_all_reduce(monkeypatch, B_total, R):
    """head.loss(group=...) (ssdhead_ce_match_stream, ssdhead_mine with the global count, ssdhead_finish_loss): taps,
    class map, counts and gradients are the full-batch slices, losses the fp32 quotients of the fold; then
    multibox_loss(group=...) with upstream gradients 0.75 and 3.0 scales the slices exactly (ssdhead_scale_grads)."""
    import torch.distributed as dist
    if not dist.is_available():
        pytest.skip("torch.distributed is not built")
    from objectdetection_ssd_b200.head import multibox_loss
    pri = H.priors()
    loc, conf, tb, tc = H.train_inputs(1000 + B_total, B_total, pri.shape[0])
    plain = _head(pri)
    full = full_batch(plain, loc, conf, tb, tc)
    shards = [Shard(plain, loc, conf, tb, tc, r, R) for r in range(R)]
    pl = [cpu(plain_step(plain, sh)) for sh in shards]
    plains = [(int(p["npos"][sh.B]), p["sums"]) for p, sh in zip(pl, shards)]
    N = int(full["npos"][B_total])
    a, c = fold(plains)
    want_l = torch.tensor([np.float32(a / (4.0 * N)), np.float32(c / N)])
    G = _Group()
    cur = [None]
    calls = _fake_all_reduce(monkeypatch, G, N, cur, (a, c))
    P = pri.shape[0]
    for r, sh in enumerate(shards):
        head = _head(pri)
        cur[0] = plains[r][1]
        o = cpu(head.loss(sh.loc, sh.conf, sh.gt, with_grads=True, taps=True, group=G))
        assert calls[-2:] == [torch.int32, torch.float64]
        compare_rank(o, full, sh, f"rank {r}: ")
        assert same_bits(o["ce"], full["ce"][sh.lo:sh.hi]), f"rank {r}: CE taps"
        assert torch.equal(H.unpack_mask(o["mined_mask"], P), H.unpack_mask(full["mined_mask"][sh.lo:sh.hi], P))
        assert same_bits(o["sums"], torch.tensor([a, c], dtype=torch.float64))
        assert same_bits(o["losses"], want_l), (o["losses"].tolist(), want_l.tolist())
        # the drop-in surface with non-unit upstream gradients
        lt = sh.loc.clone().requires_grad_(True)
        ct = sh.conf.clone().requires_grad_(True)
        l1, l2 = multibox_loss(head, lt, ct, tb[sh.lo:sh.hi], tc[sh.lo:sh.hi], group=G)
        assert same_bits(torch.stack([l1.detach(), l2.detach()]).cpu(), want_l)
        (0.75 * l1 + 3.0 * l2).backward()
        assert same_bits(lt.grad.cpu(), full["grad_loc"][sh.lo:sh.hi] * np.float32(0.75)), f"rank {r}: scaled grad_loc"
        assert same_bits(ct.grad.cpu(), full["grad_conf"][sh.lo:sh.hi] * np.float32(3.0)), f"rank {r}: scaled grad_conf"


class _DevInt32:
    """A device int32 the library owns, seen by torch without a copy (__cuda_array_interface__)."""

    def __init__(self, ptr):
        self.__cuda_array_interface__ = dict(shape=(1,), typestr="<i4", data=(int(ptr), False), version=2, strides=None)


@pytest.mark.gpu
def test_context_begin_end_halves():
    """SSDHeadContext.loss_begin / loss_end, one context per rank: the R counts begin hands back summed into one device
    int32 for end, the sums folded and finished with finish_loss - gradients are the full-batch slices and losses the
    peer route's in bits; end without a global count is the plain step on the shard alone."""
    from objectdetection_ssd_b200.ctx import SSDHeadContext
    pri = H.priors()
    B_total, R = 13, 3
    loc, conf, tb, tc = H.train_inputs(1100, B_total, pri.shape[0])
    plain = _head(pri)
    peer, full, shards, plains = run_sharded_case(pri, loc, conf, tb, tc, R, plain=plain, pin=False)
    st = _st()
    ctxs = [SSDHeadContext(pri.numpy(), max_batch=sh.B) for sh in shards]
    grads = [(torch.empty_like(sh.loc), torch.empty_like(sh.conf)) for sh in shards]
    counts = []
    for ctx, sh, (gl, gc) in zip(ctxs, shards, grads):
        ptr = ctx.loss_begin(sh.conf.data_ptr(), sh.gt.boxes.data_ptr(), sh.gt.classes.data_ptr(), sh.gt.off.data_ptr(),
                             sh.B, sh.gt.sumG, gl.data_ptr(), gc.data_ptr(), st)
        counts.append(torch.as_tensor(_DevInt32(ptr), device="cuda"))
    total = torch.zeros(1, dtype=torch.int32, device="cuda")
    for n in counts:
        total += n
    sums = [torch.empty(2, dtype=torch.float64, device="cuda") for _ in shards]
    losses = [torch.empty(2, device="cuda") for _ in shards]
    for ctx, sh, (gl, gc), s, l in zip(ctxs, shards, grads, sums, losses):
        ctx.loss_end(sh.loc.data_ptr(), sh.conf.data_ptr(), sh.gt.boxes.data_ptr(), sh.gt.classes.data_ptr(),
                     sh.gt.off.data_ptr(), sh.B, total.data_ptr(), s.data_ptr(), l.data_ptr(), gl.data_ptr(),
                     gc.data_ptr(), st)
    torch.cuda.synchronize()
    assert int(total.item()) == int(full["npos"][B_total])
    a, c = 0.0, 0.0
    for r, s in enumerate(sums):
        assert same_bits(s.cpu(), plains[r][1]), f"rank {r}: end's sums are not the plain step's"
        a += float(s[0])
        c += float(s[1])
    folded = torch.tensor([a, c], dtype=torch.float64, device="cuda")
    for r, (ctx, sh, (gl, gc)) in enumerate(zip(ctxs, shards, grads)):
        fin = torch.empty(2, device="cuda")
        ctx.finish_loss(folded.data_ptr(), total.data_ptr(), fin.data_ptr(), st)
        torch.cuda.synchronize()
        assert same_bits(gl.cpu(), full["grad_loc"][sh.lo:sh.hi]), f"rank {r}: grad_loc"
        assert same_bits(gc.cpu(), full["grad_conf"][sh.lo:sh.hi]), f"rank {r}: grad_conf"
        assert same_bits(fin.cpu(), peer[r]["losses"]), f"rank {r}: losses differ from the peer route's"
    # end with npos_norm = None: normalised by the rank's own count - the plain step on the shard alone
    for r, (ctx, sh) in enumerate(zip(ctxs, shards)):
        gl, gc = torch.empty_like(sh.loc), torch.empty_like(sh.conf)
        s, l = torch.empty(2, dtype=torch.float64, device="cuda"), torch.empty(2, device="cuda")
        ctx.loss_begin(sh.conf.data_ptr(), sh.gt.boxes.data_ptr(), sh.gt.classes.data_ptr(), sh.gt.off.data_ptr(),
                       sh.B, sh.gt.sumG, gl.data_ptr(), gc.data_ptr(), st)
        ctx.loss_end(sh.loc.data_ptr(), sh.conf.data_ptr(), sh.gt.boxes.data_ptr(), sh.gt.classes.data_ptr(),
                     sh.gt.off.data_ptr(), sh.B, None, s.data_ptr(), l.data_ptr(), gl.data_ptr(), gc.data_ptr(), st)
        want = cpu(plain_step(plain, sh))
        torch.cuda.synchronize()
        assert same_bits(s.cpu(), want["sums"]) and same_bits(l.cpu(), want["losses"]), f"rank {r}: local losses"
        assert same_bits(gl.cpu(), want["grad_loc"]) and same_bits(gc.cpu(), want["grad_conf"]), f"rank {r}: local grads"
    for ctx in ctxs:
        ctx.close()


# ----------------------------------------------------------------------------------------------------------- refusal
B_PAST = 300          # more images than 2 CTAs x 148 SMs of a B200 hold co-resident (test_gpu_fullsize.py)


def _fresh_ws(pri, B, sumG):
    lib = _lib_()
    P = pri.shape[0]
    ws = torch.zeros(int(lib.ssdhead_workspace_bytes(_lib.WS_LOSS, B, P, C, 0)), dtype=torch.uint8, device="cuda")
    wm = torch.zeros(int(lib.ssdhead_workspace_bytes(_lib.WS_MATCH, B, P, C, sumG)), dtype=torch.uint8, device="cuda")
    return ws, wm


def _plain_call(head, sh, ws, wm):
    o = _outputs(head, sh)
    _lib.check(_lib_().ssdhead_multibox_step(
        sh.loc.data_ptr(), sh.conf.data_ptr(), sh.gt.boxes.data_ptr(), sh.gt.classes.data_ptr(), sh.gt.off.data_ptr(),
        head.pri_xyxy.data_ptr(), head.pri_cxcywh.data_ptr(), sh.B, head.P, C, sh.gt.sumG, 3, 0.5,
        o["sums"].data_ptr(), o["losses"].data_ptr(), o["grad_loc"].data_ptr(), o["grad_conf"].data_ptr(),
        o["cls_u8"].data_ptr(), o["best_prior"].data_ptr(), o["npos"].data_ptr(), None, None,
        ws.data_ptr(), ws.numel(), wm.data_ptr(), wm.numel(), _st()), "ssdhead_multibox_step")
    return o


@pytest.mark.gpu
@pytest.mark.parametrize("entry", ["flat", "levels", "resident"])
def test_oversized_sharded_batch_is_refused_before_any_launch(entry):
    """B = 300 does not fit the co-resident grid the sharded mining kernel needs: every sharded entry point returns
    SSDHEAD_E_UNSUPPORTED before it launches anything - workspaces still zero, gradients untouched - and the next
    plain step on the same workspaces gives the bits of a step on fresh ones."""
    pri = H.priors()
    P = pri.shape[0]
    loc, conf, tb, tc = H.train_inputs(75, B_PAST, P)
    head = _head(pri)
    sh = Shard(head, loc, conf, tb, tc, 0, 1)
    lib = _lib_()
    # precondition: the plain step at this size takes the three-kernel route
    ws0, wm0 = _fresh_ws(pri, B_PAST, sh.gt.sumG)
    n0 = _lib.launch_count()
    want = cpu(_plain_call(head, sh, ws0, wm0))
    assert _lib.launch_count() - n0 == 3, "B = 300 should take the three-kernel route on one GPU"
    del ws0, wm0

    em = Emulation(2)
    em.seq = 1
    ws, wm = _fresh_ws(pri, B_PAST, sh.gt.sumG)
    o = _outputs(head, sh, grads=False)
    SENT = 7.25
    gl = torch.full_like(sh.loc, SENT)
    gc = torch.full_like(sh.conf, SENT)
    args_mid = (head.pri_xyxy.data_ptr(), head.pri_cxcywh.data_ptr(), B_PAST, P, C, sh.gt.sumG, 3, 0.5,
                o["sums"].data_ptr(), o["losses"].data_ptr())
    gts = (sh.gt.boxes.data_ptr(), sh.gt.classes.data_ptr(), sh.gt.off.data_ptr())
    match = (o["cls_u8"].data_ptr(), o["best_prior"].data_ptr(), o["npos"].data_ptr())
    wss = (ws.data_ptr(), ws.numel(), wm.data_ptr(), wm.numel())
    keep = None
    n0 = _lib.launch_count()
    if entry == "flat":
        rc = lib.ssdhead_multibox_step_sharded(sh.loc.data_ptr(), sh.conf.data_ptr(), *gts, *args_mid,
                                               gl.data_ptr(), gc.data_ptr(), *match, *wss, *em.xargs(0))
    elif entry == "levels":
        st, keep = levels_struct(sh.loc, sh.conf, P)
        for lc, cc, glv, gcv in keep:
            glv.fill_(SENT)
            gcv.fill_(SENT)
        rc = lib.ssdhead_multibox_step_levels_sharded(ctypes.addressof(st), *gts, *args_mid, *match, *wss, *em.xargs(0))
    else:
        rows = torch.zeros(int(lib.ssdhead_workspace_bytes(_lib.WS_ROWS, B_PAST, P, C, 0)), dtype=torch.uint8,
                           device="cuda")
        rc = lib.ssdhead_multibox_step_resident(sh.loc.data_ptr(), sh.conf.data_ptr(), *gts, *args_mid,
                                                gl.data_ptr(), gc.data_ptr(), *match, *wss, rows.data_ptr(), rows.numel(),
                                                *em.xargs(0))
    torch.cuda.synchronize()
    assert rc == _lib.E_UNSUPPORTED, rc
    assert _lib.launch_count() == n0, f"{_lib.launch_count() - n0} kernels launched before the refusal"
    assert int(wm.count_nonzero()) == 0, "the match workspace is no longer zero"
    assert int(ws.count_nonzero()) == 0, "the loss workspace is no longer zero"
    for g in ([gl, gc] if keep is None else [t for k in keep for t in k[2:]]):
        assert bool((g == SENT).all()), "a gradient tensor was written"
    assert int(em.err[0].item()) == 0 and int(em.xchg[0].count_nonzero()) == 0
    # the same workspaces carry on as fresh ones
    got = cpu(_plain_call(head, sh, ws, wm))
    for key in ("sums", "losses", "grad_loc", "grad_conf"):
        assert same_bits(got[key], want[key]), f"{key} of the next plain step differs from a step on fresh workspaces"
    for key in ("cls_u8", "npos", "best_prior"):
        assert torch.equal(got[key], want[key]), f"{key} of the next plain step differs from a step on fresh workspaces"
