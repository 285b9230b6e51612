"""ReconstructReply receiving (handle_msg_reconstruct_reply, crossword/messages.rs:634-722, rspaxos/messages.rs:519-594)
batched on the device: absorb the replied shards, walk the execution bar, reconstruct_data of the walked instances.

`literal_stream` below restates the handler per reply entry, in arrival order; it is the oracle the device call is
compared with.  It is test code: it uses the CPU oracle's reconstruct (oracle/ss_oracle.c) for the decode and never
calls the product.  CPU tests pin it against a model of the batched semantics (absorb all, walk once, decode); GPU
tests compare ss_reconstruct_reply_dev with it, bit for bit."""
import numpy as np
import pytest
import torch

DEV = "cuda:0"
NO_INST = 0xFFFFFFFF
NULL, PREPARING, ACCEPTING, COMMITTED, EXECUTED = range(5)     # Status, declaration order
SENTINEL = 0xEE


def _bits(m):
    return [j for j in range(32) if (m >> j) & 1]


def _popc(m):
    return bin(int(m)).count("1")


class Case:
    """A follower's window: planes uint8 [T, G*W, ss] (padded slot ds = round_up(L,16), then a sentinel gap up to ss),
    status / bal / present per row, exec bar per group, and replies (row, ballot, mask, shards uint8 [popc(mask), ds])."""

    def __init__(self, d, p, G, W, data_len, gap=32):
        self.d, self.p, self.T, self.G, self.W, self.n = d, p, d + p, G, W, G * W
        self.data_len = data_len
        self.L = (data_len + d - 1) // d
        self.ds = (self.L + 15) // 16 * 16
        self.ss = self.ds + gap
        self.planes = np.full((self.T, self.n, self.ss), SENTINEL, dtype=np.uint8)
        self.status = np.full(self.n, COMMITTED, dtype=np.uint8)
        self.bal = np.ones(self.n, dtype=np.uint64)
        self.present = np.zeros(self.n, dtype=np.uint32)
        self.bar = np.zeros(G, dtype=np.uint32)
        self.replies = []

    def copy(self):
        c = Case.__new__(Case)
        c.__dict__.update(self.__dict__)
        for k in ("planes", "status", "bal", "present", "bar"):
            setattr(c, k, getattr(self, k).copy())
        c.replies = list(self.replies)
        return c

    def hold(self, r, j, shard):
        """the row holds shard j (L bytes, zero padding up to the slot)"""
        self.planes[j, r, :self.ds] = 0
        self.planes[j, r, :self.L] = shard[:self.L]
        self.present[r] |= np.uint32(1 << j)


def codewords(oracle, d, p, n, data_len, rng):
    """n consistent codewords: uint8 [n, T, L] (data shards = the split payload, parity = the oracle's encode)"""
    L = (data_len + d - 1) // d
    out = np.zeros((n, d + p, L), dtype=np.uint8)
    payload = rng.integers(0, 256, (n, data_len), dtype=np.uint8)
    for r in range(n):
        out[r, :d] = oracle.cw_split(payload[r].tobytes(), d)
        shards = [out[r, j].copy() for j in range(d + p)]
        assert oracle.rs_encode(d, p, shards) == 0
        for j in range(d, d + p):
            out[r, j] = shards[j]
    return out, payload


def _reply_shards(case, cw_row, mask):
    s = np.zeros((_popc(mask), case.ds), dtype=np.uint8)
    for k, j in enumerate(_bits(mask)):
        s[k, :case.L] = cw_row[j]
    return s


def settled_case(oracle, rng, d, p, G, W, data_len, dup_rate=0.3):
    """Random state that satisfies the batched call's preconditions: the instance at each bar is not ready on entry, and
    every reply for a row carries shards of that row's one codeword.  Includes duplicates, stale ballots, Executed and
    Null instances, replies for Accepting instances, out-of-window entries and malformed masks."""
    c = Case(d, p, G, W, data_len)
    T = c.T
    cw, _ = codewords(oracle, d, p, c.n, data_len, rng)
    c.status = rng.choice([NULL, ACCEPTING, COMMITTED, EXECUTED], size=c.n, p=[0.03, 0.07, 0.82, 0.08]).astype(np.uint8)
    c.bal = rng.integers(1, 4, c.n).astype(np.uint64)
    for r in range(c.n):
        for j in rng.choice(T, size=int(rng.integers(0, d)), replace=False):     # at most d-1 shards held on entry
            c.hold(r, int(j), cw[r, int(j)])
    c.bar = rng.integers(0, W + 1, G).astype(np.uint32)
    c.bar[0] = 0
    for g in range(G):                             # rows below the bar were executed with their data in place
        for s in range(int(c.bar[g])):
            r = g * W + s
            c.status[r] = max(int(c.status[r]), COMMITTED)
            for j in range(d):
                if not (int(c.present[r]) >> j) & 1:
                    c.hold(r, j, cw[r, j])
    for r in range(c.n):
        for _ in range(int(rng.integers(1, 4))):
            mask = int(rng.integers(1, 1 << T))
            ballot = int(c.bal[r]) + int(rng.choice([-1, 0, 0, 0, 1]))
            c.replies.append((r, ballot, mask, _reply_shards(c, cw[r], mask)))
            if rng.random() < dup_rate:            # the same shards again, from another peer
                c.replies.append((r, ballot + int(rng.integers(0, 2)), mask, _reply_shards(c, cw[r], mask)))
    for _ in range(max(4, c.n // 20)):
        mask = int(rng.integers(1, 1 << T))
        junk = rng.integers(0, 256, (_popc(mask), c.ds), dtype=np.uint8)
        c.replies.append((NO_INST, 9, mask, junk))                  # slot below start_slot / outside the window
    r = int(rng.integers(0, c.n))
    bad = (1 << T) | 1                                              # names shard T: malformed, dropped whole
    c.replies.append((r, int(c.bal[r]) + 1, bad, rng.integers(0, 256, (2, c.ds), dtype=np.uint8)))
    order = rng.permutation(len(c.replies))
    c.replies = [c.replies[i] for i in order]
    return c, cw


def _decode_row(oracle, c, r):
    """reconstruct_data (rscoding.rs:512-520 -> the crate's reconstruct_data) of row r, in place"""
    shards = [c.planes[j, r, :c.L].copy() if (int(c.present[r]) >> j) & 1 else None for j in range(c.T)]
    assert oracle.rs_reconstruct(c.d, c.p, shards, True) == 0
    for j in range(c.d):
        if not (int(c.present[r]) >> j) & 1:
            c.planes[j, r, :c.ds] = 0
            c.planes[j, r, :c.L] = shards[j]
    c.present[r] |= np.uint32((1 << c.d) - 1)


def _eligible(c, r, ballot, mask):
    return r != NO_INST and r < c.n and (mask >> c.T) == 0 and c.status[r] < EXECUTED and ballot >= int(c.bal[r])


def literal_stream(oracle, c):
    """handle_msg_reconstruct_reply applied per (slot, (ballot, reqs_cw)) entry in arrival order, in place on c.
    Returns submit [G]: bit s = instance s was handed to execution."""
    submit = np.zeros(c.G, dtype=np.uint64)
    for r, ballot, mask, shards in c.replies:
        if r == NO_INST or r >= c.n:
            continue                               # slot < self.start_slot (crossword/messages.rs:641-643)
        if mask >> c.T:
            continue                               # not a codeword of this code: no such frame decodes
        # if inst.status < Status::Executed && ballot >= inst.bal (crossword/messages.rs:667, rspaxos/messages.rs:542)
        if not (c.status[r] < EXECUTED and ballot >= int(c.bal[r])):
            continue
        # inst.reqs_cw.absorb_other(reqs_cw): shard i is taken only where self.shards[i] is None (rscoding.rs:336-342)
        for k, j in enumerate(_bits(mask)):
            if not (int(c.present[r]) >> j) & 1:
                c.planes[j, r, :c.ds] = shards[k]
                c.present[r] |= np.uint32(1 << j)
        g, s = divmod(r, c.W)
        if s == int(c.bar[g]):                     # if slot == self.commit_bar (crossword/messages.rs:670)
            while int(c.bar[g]) < c.W:
                r2 = g * c.W + int(c.bar[g])
                # status < Committed || avail_shards() < num_data_shards() -> break (:674-679)
                if c.status[r2] < COMMITTED or _popc(c.present[r2]) < c.d:
                    break
                if _popc(int(c.present[r2]) & ((1 << c.d) - 1)) < c.d:
                    _decode_row(oracle, c, r2)     # reconstruct_data(Some(&self.rs_coder)) (:681-687)
                submit[g] |= np.uint64(1 << int(c.bar[g]))
                c.bar[g] += 1
    return submit


def batched_model(oracle, c):
    """What ss_reconstruct_reply_dev computes: absorb every reply (first copy of a shard wins), walk each bar once,
    then decode the walked rows that lack data shards.  In place on c; returns (submit, taken)."""
    taken = np.zeros(len(c.replies), dtype=np.uint32)
    for i, (r, ballot, mask, shards) in enumerate(c.replies):
        if not _eligible(c, r, ballot, mask):
            continue
        won = mask & ~int(c.present[r])
        for k, j in enumerate(_bits(mask)):
            if (won >> j) & 1:
                c.planes[j, r, :c.ds] = shards[k]
        c.present[r] |= np.uint32(won)
        taken[i] = won
    submit = np.zeros(c.G, dtype=np.uint64)
    marked = []
    for g in range(c.G):
        while int(c.bar[g]) < c.W:
            r = g * c.W + int(c.bar[g])
            if c.status[r] < COMMITTED or _popc(c.present[r]) < c.d:
                break
            if _popc(int(c.present[r]) & ((1 << c.d) - 1)) < c.d:
                marked.append(r)
            submit[g] |= np.uint64(1 << int(c.bar[g]))
            c.bar[g] += 1
    for r in marked:
        _decode_row(oracle, c, r)
    return submit, taken


def _same_state(a, b):
    assert (a.present == b.present).all()
    assert (a.bar == b.bar).all()
    assert (a.planes == b.planes).all()


# ---------------------------------------------------------------------------------------------
# CPU: the literal handler and the batched semantics agree on settled inputs; each filter alone
# ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("d,p,data_len", [(3, 2, 100), (6, 4, 61), (2, 1, 33)])
def test_literal_equals_batched_on_settled_inputs(oracle, d, p, data_len):
    rng = np.random.default_rng(d * 100 + data_len)
    for trial in range(3):
        base, _ = settled_case(oracle, rng, d, p, 5, 12, data_len)
        want = base.copy()
        want_submit, _ = batched_model(oracle, want)
        assert want_submit.any() and (want.bar > base.bar).any()          # the walk moved somewhere
        for perm in range(4):
            c = base.copy()
            c.replies = [base.replies[i] for i in rng.permutation(len(base.replies))]
            submit = literal_stream(oracle, c)
            assert (submit == want_submit).all(), (trial, perm)
            _same_state(c, want)


def _one_reply_case(oracle, status, inst_bal, ballot):
    """RS(3,2), one group of 4 instances, bar at 0, row 0 holding shard 0; one reply with shards {1, 2} for row 0."""
    rng = np.random.default_rng(5)
    c = Case(3, 2, 1, 4, 48)
    cw, _ = codewords(oracle, 3, 2, c.n, 48, rng)
    c.status[0] = status
    c.bal[0] = inst_bal
    c.hold(0, 0, cw[0, 0])
    c.replies = [(0, ballot, 0b110, _reply_shards(c, cw[0], 0b110))]
    return c, cw


def _both(oracle, c):
    a, b = c.copy(), c.copy()
    sa = literal_stream(oracle, a)
    sb, taken = batched_model(oracle, b)
    assert (sa == sb).all()
    _same_state(a, b)
    return a, sa, taken


def test_filter_outdated_slot(oracle):
    c, _ = _one_reply_case(oracle, COMMITTED, 1, 1)
    c.replies = [(NO_INST, 1, m, s) for _, _, m, s in c.replies]          # slot < start_slot
    a, submit, taken = _both(oracle, c)
    assert a.present[0] == 1 and submit[0] == 0 and a.bar[0] == 0 and taken[0] == 0
    assert (a.planes == c.planes).all()


def test_filter_executed(oracle):
    c, _ = _one_reply_case(oracle, EXECUTED, 1, 1)
    a, submit, taken = _both(oracle, c)
    assert a.present[0] == 1 and taken[0] == 0 and (a.planes == c.planes).all()
    assert submit[0] == 0 and a.bar[0] == 0                                # Executed with one shard is not ready


def test_filter_stale_ballot(oracle):
    c, _ = _one_reply_case(oracle, COMMITTED, 5, 4)
    a, submit, taken = _both(oracle, c)
    assert a.present[0] == 1 and taken[0] == 0 and submit[0] == 0 and (a.planes == c.planes).all()
    c, cw = _one_reply_case(oracle, COMMITTED, 5, 5)                      # ballot == inst.bal is taken
    a, submit, taken = _both(oracle, c)
    assert a.present[0] == 0b111 and taken[0] == 0b110 and submit[0] == 1 and a.bar[0] == 1
    assert (a.planes[1, 0, :c.L] == cw[0, 1]).all()


def test_accepting_is_absorbed_not_walked(oracle):
    """the handler's debug_assert!(status >= Committed) does not filter in a release build (crossword/messages.rs:651-654)"""
    c, cw = _one_reply_case(oracle, ACCEPTING, 1, 1)
    a, submit, taken = _both(oracle, c)
    assert a.present[0] == 0b111 and taken[0] == 0b110
    assert (a.planes[2, 0, :c.L] == cw[0, 2]).all()
    assert submit[0] == 0 and a.bar[0] == 0


def test_walk_decodes_with_parity(oracle):
    """a row holding only parity-heavy shards is reconstructed when the bar passes it; the bar stops at the next
    instance that is not ready"""
    rng = np.random.default_rng(9)
    c = Case(3, 2, 1, 4, 50)
    cw, payload = codewords(oracle, 3, 2, c.n, 50, rng)
    c.hold(0, 3, cw[0, 3])
    c.hold(1, 0, cw[1, 0]); c.hold(1, 1, cw[1, 1]); c.hold(1, 2, cw[1, 2])
    c.replies = [(0, 1, 0b10001, _reply_shards(c, cw[0], 0b10001))]
    a, submit, taken = _both(oracle, c)
    assert submit[0] == 0b11 and a.bar[0] == 2 and a.present[0] == 0b11111
    assert a.planes[:3, 0, :c.L].reshape(-1)[:50].tobytes() == payload[0].tobytes()
    assert (a.planes[1:3, 0, c.L:c.ds] == 0).all()                        # regenerated slots: zero padding


# ---------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------
def _t(a):
    a = np.ascontiguousarray(a)
    if a.dtype == np.uint64:
        a = a.view(np.int64)
    elif a.dtype == np.uint32:
        a = a.view(np.int32)
    return torch.from_numpy(a).to(DEV)


def _pack(c, rng):
    """the replies as one buffer in serve's layout, with unused 16-byte multiples between replies"""
    off, at = [], 0
    for _, _, mask, shards in c.replies:
        off.append(at)
        at += shards.shape[0] * c.ds + 16 * int(rng.integers(0, 3))
    buf = np.full(at + 16, 0x33, dtype=np.uint8)
    for o, (_, _, _, shards) in zip(off, c.replies):
        buf[o:o + shards.size] = shards.reshape(-1)
    inst = np.array([r for r, _, _, _ in c.replies], dtype=np.uint32)
    ballot = np.array([b for _, b, _, _ in c.replies], dtype=np.uint64)
    mask = np.array([m for _, _, m, _ in c.replies], dtype=np.uint32)
    return buf, np.array(off, dtype=np.uint64), mask, inst, ballot


def _run_gpu(rs, c, rng):
    buf, off, mask, inst, ballot = _pack(c, rng)
    planes = _t(c.planes)
    present, bar = _t(c.present), _t(c.bar)
    submit, taken = rs.reconstruct_reply(planes, c.data_len, c.W, _t(c.status), _t(c.bal), present, bar, _t(buf), _t(off),
                                         _t(mask), _t(inst), _t(ballot))
    torch.cuda.synchronize()
    out = c.copy()
    out.planes = planes.cpu().numpy()
    out.present = present.cpu().numpy().view(np.uint32)
    out.bar = bar.cpu().numpy().view(np.uint32)
    return out, submit.cpu().numpy().view(np.uint64), taken.cpu().numpy().view(np.uint32)


def _check_taken(c0, taken):
    """per row the taken masks are disjoint, lie inside eligible replies' masks and together are the new bits the
    absorb step set"""
    union = np.zeros(c0.n, dtype=np.uint32)
    for i, (r, ballot, mask, _) in enumerate(c0.replies):
        t = int(taken[i])
        if not _eligible(c0, r, ballot, mask):
            assert t == 0, i
            continue
        assert t & ~mask == 0 and t & int(c0.present[r]) == 0, i
        assert t & int(union[r]) == 0, i
        union[r] |= np.uint32(t)
    return union


@pytest.mark.gpu
@pytest.mark.parametrize("d,p,data_len,W", [(3, 2, 4096, 64), (3, 2, 18, 64), (3, 2, 1000, 64), (2, 1, 1000, 40),
                                            (4, 3, 1000, 64), (6, 4, 1000, 64)])
def test_reply_matches_oracle(ctx, oracle, d, p, data_len, W):
    from summerset_b200.api import ReedSolomon
    rng = np.random.default_rng(d * 7 + data_len + W)
    rs = ReedSolomon(ctx, d, p)
    G = 24
    c0, _ = settled_case(oracle, rng, d, p, G, W, data_len)
    got, submit, taken = _run_gpu(rs, c0, rng)
    want = c0.copy()
    want_submit = literal_stream(oracle, want)
    assert (submit == want_submit).all()
    assert (got.bar == want.bar).all()
    assert (got.present == want.present).all()
    assert (got.planes == want.planes).all()               # every data and parity slot, and the sentinel gaps
    union = _check_taken(c0, taken)
    model = c0.copy()
    _, want_taken = batched_model(oracle, model)
    absorbed = np.zeros(c0.n, dtype=np.uint32)
    for i, (r, _, _, _) in enumerate(c0.replies):
        if want_taken[i]:
            absorbed[r] |= want_taken[i]
    assert (union == absorbed).all()
    assert int(want_submit.astype(bool).sum()) > G // 3


@pytest.mark.gpu
def test_reply_disagreeing_duplicates(ctx, oracle):
    """replies for one slot that carry different bytes for the same shard: every absorbed slot is exactly one candidate's
    shard, whole; the decode of a walked row is consistent with the shards that were absorbed"""
    from summerset_b200.api import ReedSolomon
    rng = np.random.default_rng(77)
    d, p, G, W, data_len = 3, 2, 8, 64, 1000
    rs = ReedSolomon(ctx, d, p)
    c0 = Case(d, p, G, W, data_len)
    for r in range(c0.n):
        if rng.random() < 0.5:
            c0.hold(r, int(rng.integers(0, 5)), rng.integers(0, 256, c0.L, dtype=np.uint8))
        for _ in range(int(rng.integers(1, 5))):
            mask = int(rng.integers(1, 32))
            c0.replies.append((r, 1, mask, rng.integers(0, 256, (_popc(mask), c0.ds), dtype=np.uint8)))
    c0.replies = [c0.replies[i] for i in rng.permutation(len(c0.replies))]
    got, submit, taken = _run_gpu(rs, c0, rng)
    union = _check_taken(c0, taken)
    for i, (r, _, mask, shards) in enumerate(c0.replies):
        for k, j in enumerate(_bits(mask)):
            if (int(taken[i]) >> j) & 1:
                assert (got.planes[j, r, :c0.ds] == shards[k]).all(), (i, j)
    dmask = (1 << d) - 1
    for r in range(c0.n):
        held = int(c0.present[r]) | int(union[r])
        g, s = divmod(r, W)
        walked = (int(submit[g]) >> s) & 1
        assert int(got.present[r]) == (held | dmask if walked else held)
        ref = c0.copy()
        ref.planes[:, r] = got.planes[:, r]
        ref.present[r] = held
        if walked and (held & dmask) != dmask:
            _decode_row(oracle, ref, r)
        for j in range(c0.T):
            if not (held >> j) & 1 and not (walked and j < d):
                assert (got.planes[j, r] == SENTINEL).all()          # never written
        assert (got.planes[:, r] == ref.planes[:, r]).all(), r
        assert (got.planes[:, r, c0.ds:] == SENTINEL).all()
    assert submit.any()


@pytest.mark.gpu
def test_crossword_round_trip_plan_serve_reply(ctx, oracle):
    """Crossword n=5, RS(6,4), two shards per replica: encode, follower `me` keeps its assigned shards, plan the
    Reconstruct requests (ss_gossip_plan_dev), serve each target from that peer's shards (ss_reconstruct_serve_dev),
    apply every peer's reply (ss_reconstruct_reply_dev).  Every walked instance holds its payload again; the bar stops
    at the first instance that is not committed."""
    from summerset_b200 import _lib
    from summerset_b200.api import ReedSolomon, crossword_brr_assignment, _ptr
    rng = np.random.default_rng(3)
    n_rep, d, p, W, G, data_len, me, leader = 5, 6, 4, 64, 8, 3000, 2, 0
    T = d + p
    policies = [crossword_brr_assignment(n_rep, T, 2)]
    rs = ReedSolomon(ctx, d, p)
    n = G * W
    L = (data_len + d - 1) // d
    ds = (L + 15) // 16 * 16
    stride = (data_len + 15) // 16 * 16
    payload = rng.integers(0, 256, (n, stride), dtype=np.uint8)
    full = torch.zeros((T, n, ds), dtype=torch.uint8, device=DEV)
    check = _lib.check
    check(rs.lib.ss_rs_encode_uniform_dev(rs.h, _ptr(_t(payload)), stride, data_len, n, full[d].data_ptr(), n * ds, ds,
                                          _lib.SS_RS_OUT_PADDED16 | 2))              # | SS_RS_EMIT_DATA
    mine = policies[0][me]
    planes = torch.full((T, n, ds), SENTINEL, dtype=torch.uint8, device=DEV)
    for j in _bits(mine):
        planes[j] = full[j]
    present = torch.full((n,), mine, dtype=torch.int32, device=DEV)
    status = np.full(n, COMMITTED, dtype=np.uint8)
    stop = rng.integers(0, W + 1, G)
    stop[0], stop[1] = W, 0
    for g in range(G):
        if stop[g] < W:
            status[g * W + stop[g]] = ACCEPTING
    rows = np.nonzero(status == COMMITTED)[0].astype(np.uint32)
    N = rows.size
    targets, excl = ctx.gossip_plan(me, n_rep, d, torch.full((N,), leader, dtype=torch.uint8, device=DEV),
                                    present[torch.from_numpy(rows.astype(np.int64)).to(DEV)],
                                    torch.zeros(N, dtype=torch.uint8, device=DEV), policies, (1 << n_rep) - 1)
    targets = targets.cpu().numpy()
    bar = torch.zeros(G, dtype=torch.int32, device=DEV)
    bal = torch.ones(n, dtype=torch.int64, device=DEV)
    submit = np.zeros(G, dtype=np.uint64)
    served = 0
    for q in range(n_rep):
        sel = np.nonzero((targets >> q) & 1)[0]
        if sel.size == 0:
            continue
        req_rows = rows[sel]
        held = np.full(sel.size, policies[0][q], dtype=np.uint32)
        off = (np.arange(sel.size, dtype=np.uint64) * np.uint64(_popc(policies[0][q]) * ds))
        mask, out = ctx.reconstruct_serve(full, L, _t(req_rows), _t(held), excl[q][torch.from_numpy(sel).to(DEV)].contiguous(),
                                          torch.full((sel.size,), COMMITTED, dtype=torch.uint8, device=DEV), _t(off),
                                          int(off[-1]) + _popc(policies[0][q]) * ds)
        s, _ = rs.reconstruct_reply(planes, data_len, W, _t(status), bal, present, bar, out, _t(off), mask, _t(req_rows),
                                    torch.ones(sel.size, dtype=torch.int64, device=DEV), want_taken=False)
        submit |= s.cpu().numpy().view(np.uint64)
        served += 1
    torch.cuda.synchronize()
    assert served == 2                                          # two peers cover the six data shards
    bar = bar.cpu().numpy()
    assert (bar == stop).all()
    pl = planes.cpu().numpy()
    for g in range(G):
        assert int(submit[g]) == (1 << int(stop[g])) - 1
        for s in range(int(stop[g])):
            r = g * W + s
            assert pl[:d, r, :L].reshape(-1)[:data_len].tobytes() == payload[r, :data_len].tobytes(), r
    pres = present.cpu().numpy().view(np.uint32)
    assert all(_popc(pres[r]) >= d for r in rows)


@pytest.mark.gpu
def test_reply_argument_errors_and_empty_batch(ctx):
    from summerset_b200 import _lib
    from summerset_b200.api import ReedSolomon, _ptr
    rs = ReedSolomon(ctx, 3, 2)
    G, W, data_len = 2, 8, 100
    L = 34
    ds = 48
    n = G * W
    planes = torch.zeros((5, n, ds), dtype=torch.uint8, device=DEV)
    st = torch.full((n,), COMMITTED, dtype=torch.uint8, device=DEV)
    bal = torch.zeros(n, dtype=torch.int64, device=DEV)
    present = torch.full((n,), 1, dtype=torch.int32, device=DEV)
    bar = torch.zeros(G, dtype=torch.int32, device=DEV)
    buf = torch.zeros(4 * ds, dtype=torch.uint8, device=DEV)
    off = torch.zeros(1, dtype=torch.int64, device=DEV)
    mask = torch.full((1,), 0b110, dtype=torch.int32, device=DEV)
    inst = torch.zeros(1, dtype=torch.int32, device=DEV)
    rb = torch.zeros(1, dtype=torch.int64, device=DEV)
    submit = torch.full((G,), -7, dtype=torch.int64, device=DEV)

    def call(coder=rs.h, pl=planes.data_ptr(), ps=n * ds, ss=ds, dl=data_len, ng=G, w=W, buf_ptr=buf.data_ptr(), nr=1,
             sub=submit.data_ptr()):
        return rs.lib.ss_reconstruct_reply_dev(coder, pl, ps, ss, dl, ng, w, _ptr(st), _ptr(bal), _ptr(present), _ptr(bar),
                                               buf_ptr, _ptr(off), _ptr(mask), _ptr(inst), _ptr(rb), nr, sub, None)

    E = _lib.SS_ERR_INVALID_ARG
    assert call(coder=None) == E
    assert call(sub=None) == E and call(buf_ptr=None) == E
    assert call(pl=planes.data_ptr() + 8) == E and call(buf_ptr=buf.data_ptr() + 4) == E and call(ss=ds + 8) == E
    assert call(ps=n * ds + 1) == E
    assert call(ss=32) == E                                     # shorter than round_up(L, 16) = 48
    assert call(w=0) == E and call(w=65) == E and call(ng=0) == E and call(dl=0) == E
    big = ReedSolomon(ctx, 9, 4)                                # d+p = 13: no uniform reconstruct
    assert call(coder=big.h) == _lib.SS_ERR_UNSUPPORTED
    launches = ctx.launches
    assert call(nr=0, buf_ptr=None) == _lib.SS_OK               # empty batch: nothing launched, nothing written
    torch.cuda.synchronize()
    assert ctx.launches == launches
    assert (submit.cpu() == -7).all() and (present.cpu() == 1).all() and (bar.cpu() == 0).all()
    assert call() == _lib.SS_OK                                 # the same arguments are fine
    torch.cuda.synchronize()
    assert ctx.launches == launches + 3
    assert (present.cpu()[0] == 0b111) and int(bar.cpu()[0]) == 1 and int(submit.cpu()[0]) == 1
