"""Python host side over the C ABI (include/summerset_b200.h).

PyTorch is used only for device memory and streams.  The classes mirror the reference's names and
error behaviour for this path so tests read like the reference's own:

  ReedSolomon   <- reed_solomon_erasure::galois_8::ReedSolomon as used by src/utils/rscoding.rs
  Bitmap        <- src/utils/bitmap.rs
  RSCodeword    <- src/utils/rscoding.rs (payload = opaque serialized bytes)

plus the batched device-resident calls (tally_planes, encode_uniform, ...), which are what a
batched multi-group engine drives every step.  Nothing here computes shard bytes or tallies on the
CPU: every such call goes through libsummerset_b200.so and raises SummersetError if that fails.
"""
from __future__ import annotations

import ctypes as C
from typing import Iterable, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _lib
from ._lib import SummersetError, check

SS_RS_OUT_PADDED16 = _lib.SS_RS_OUT_PADDED16


def _ptr(t: Optional[torch.Tensor]) -> int:
    return 0 if t is None else t.data_ptr()


def round_up(x: int, a: int) -> int:
    return (x + a - 1) // a * a


def cw_slot_pitch(L):
    """SS_CW_SLOT_PITCH of include/summerset_b200.h: bytes between the slots of one codeword in a Crossword replica log
    (shard length rounded up to 32; works on ints and numpy arrays)."""
    return (L + 31) // 32 * 32


def shard_len(data_len: int, d: int) -> int:
    """rscoding.rs:177-181"""
    return data_len // d if data_len % d == 0 else data_len // d + 1


class Context:
    """A device context bound to torch's CURRENT stream on `device` at creation time."""

    def __init__(self, device: int = 0, own_stream: bool = False):
        self.lib = _lib.load()
        self.device = int(device)
        h = C.c_void_p()
        if own_stream:
            check(self.lib.ss_ctx_create(self.device, C.byref(h)))
        else:
            if not torch.cuda.is_available():
                # let the library produce its own loud error (no CPU fallback)
                check(self.lib.ss_ctx_create(self.device, C.byref(h)))
            with torch.cuda.device(self.device):
                stream = torch.cuda.current_stream().cuda_stream
            check(self.lib.ss_ctx_create_on_stream(self.device, C.c_void_p(stream), C.byref(h)))
        self.h = h

    def sync(self) -> None:
        check(self.lib.ss_ctx_sync(self.h))

    @property
    def launches(self) -> int:
        return int(self.lib.ss_ctx_launch_count(self.h))

    @property
    def sm_count(self) -> int:
        return int(self.lib.ss_ctx_sm_count(self.h))

    def close(self) -> None:
        if getattr(self, "h", None) is not None and self.h:
            self.lib.ss_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- raw device buffers + cross-process peer memory ----------------------------------------------
    def dev_alloc(self, nbytes: int) -> "DevBuffer":
        p = C.c_void_p()
        check(self.lib.ss_dev_alloc(self.h, nbytes, C.byref(p)))
        return DevBuffer(self, p.value, nbytes, owned=True)

    def ipc_export(self, buf: "DevBuffer") -> bytes:
        h = (C.c_uint8 * 64)()
        check(self.lib.ss_ipc_export(self.h, buf.ptr, h))
        return bytes(h)

    def ipc_open(self, handle: bytes, nbytes: int) -> "DevBuffer":
        h = (C.c_uint8 * 64).from_buffer_copy(handle)
        p = C.c_void_p()
        check(self.lib.ss_ipc_open(self.h, h, C.byref(p)))
        return DevBuffer(self, p.value, nbytes, owned=False)

    def copy_d2d(self, dst_ptr: int, src_ptr: int, nbytes: int) -> None:
        check(self.lib.ss_copy_d2d(self.h, dst_ptr, src_ptr, nbytes))

    def flags_signal(self, sync: "StepSync") -> None:
        check(self.lib.ss_flags_signal_dev(self.h, C.byref(sync.c)))

    def flags_wait(self, sync: "StepSync") -> None:
        check(self.lib.ss_flags_wait_dev(self.h, C.byref(sync.c)))

    def event_create(self) -> int:
        ev = C.c_void_p()
        check(self.lib.ss_event_create(self.h, C.byref(ev)))
        return ev.value

    def event_destroy(self, ev: int) -> None:
        check(self.lib.ss_event_destroy(self.h, ev))

    def event_record(self, ev: int) -> None:
        check(self.lib.ss_event_record(self.h, ev))

    def event_wait(self, ev: int) -> None:
        check(self.lib.ss_event_wait(self.h, ev))

    def device_status(self) -> int:
        """Reads and clears the device status word (bit 0: a step-flag wait timed out); synchronises the stream."""
        st = C.c_uint32(0)
        check(self.lib.ss_ctx_device_status(self.h, C.byref(st)))
        return int(st.value)

    def follower_ack(self, ack_src: torch.Tensor, ack_dst: Sequence[int], sync: Optional["StepSync"] = None) -> None:
        """ack_src int64 [R, G] on the GPU; ack_dst: R raw device pointers (0 = skip) into the leaders' ack buffers."""
        assert ack_src.is_cuda and ack_src.dtype == torch.int64 and ack_src.is_contiguous() and ack_src.dim() == 2
        R, G = ack_src.shape
        arr = (C.c_void_p * R)(*[p if p else None for p in ack_dst])
        check(self.lib.ss_follower_ack_dev(self.h, _ptr(ack_src), arr, R, G, C.byref(sync.c) if sync else None))

    # ---- tallies -------------------------------------------------------------------------------
    def tally_planes(self, planes: torch.Tensor, threshold: int, want_bar: bool = True,
                     committed: Optional[torch.Tensor] = None, commit_bar: Optional[torch.Tensor] = None):
        """planes: int64 [R, G] on the GPU (bit s of planes[r, g] = replica r acked slot s)."""
        assert planes.is_cuda and planes.dtype == torch.int64 and planes.is_contiguous() and planes.dim() == 2
        R, G = planes.shape
        if committed is None:
            committed = torch.empty(G, dtype=torch.int64, device=planes.device)
        if want_bar and commit_bar is None:
            commit_bar = torch.empty(G, dtype=torch.int32, device=planes.device)
        check(self.lib.ss_tally_planes_dev(self.h, _ptr(planes), R, G, threshold, _ptr(committed),
                                           _ptr(commit_bar) if want_bar else 0))
        return committed, (commit_bar if want_bar else None)

    def tally_planes_host(self, planes: np.ndarray, threshold: int):
        """HOST buffers through ss_tally_planes (copies inside)."""
        planes = np.ascontiguousarray(planes, dtype=np.uint64)
        R, G = planes.shape
        committed = np.empty(G, dtype=np.uint64)
        bar = np.empty(G, dtype=np.uint32)
        check(self.lib.ss_tally_planes(self.h, planes.ctypes.data, R, G, threshold, committed.ctypes.data,
                                       bar.ctypes.data))
        return committed, bar

    def tally_masks(self, masks: torch.Tensor, threshold: int) -> torch.Tensor:
        """masks: uint8 or int16 [n] on the GPU, one accept_acks Bitmap per instance."""
        assert masks.is_cuda and masks.is_contiguous() and masks.dim() == 1
        mb = {torch.uint8: 1, torch.int16: 2}[masks.dtype]
        n = masks.numel()
        out = torch.empty((n + 63) // 64, dtype=torch.int64, device=masks.device)
        check(self.lib.ss_tally_masks_dev(self.h, _ptr(masks), mb, n, threshold, _ptr(out)))
        return out

    def ack_ingest(self, rec_group, rec_slot, rec_peer, rec_ballot, bal_prepared, inst_bal, accepting,
                   n_replicas: int, planes: torch.Tensor) -> None:
        G = bal_prepared.numel()
        assert planes.shape == (n_replicas, G) and planes.dtype == torch.int64
        assert rec_group.dtype == torch.int32 and rec_slot.dtype == torch.uint8 and rec_peer.dtype == torch.uint8
        assert rec_ballot.dtype == torch.int64 and inst_bal.numel() == G * 64
        check(self.lib.ss_ack_ingest_dev(self.h, _ptr(rec_group), _ptr(rec_slot), _ptr(rec_peer), _ptr(rec_ballot),
                                         rec_group.numel(), _ptr(bal_prepared), _ptr(inst_bal), _ptr(accepting),
                                         n_replicas, G, _ptr(planes)))

    def tally_crossword(self, masks: torch.Tensor, policy_idx: torch.Tensor, policies: Sequence[Sequence[int]],
                        total_shards: int, data_shards: int, majority: int, fault_tolerance: int,
                        balanced: bool) -> torch.Tensor:
        assert masks.is_cuda and policy_idx.is_cuda and policy_idx.dtype == torch.uint8
        mb = {torch.uint8: 1, torch.int16: 2}[masks.dtype]
        pol = np.ascontiguousarray(np.array(policies, dtype=np.uint32))
        K, n_rep = pol.shape
        n = masks.numel()
        out = torch.empty((n + 63) // 64, dtype=torch.int64, device=masks.device)
        check(self.lib.ss_tally_crossword_dev(self.h, _ptr(masks), mb, _ptr(policy_idx), n, pol.ctypes.data, K, n_rep,
                                              total_shards, data_shards, majority, fault_tolerance,
                                              1 if balanced else 0, _ptr(out)))
        return out

    def raft_commit_scan(self, match: torch.Tensor, last_commit: torch.Tensor, log_end: torch.Tensor,
                         curr_term: torch.Tensor, terms: torch.Tensor, threshold: int,
                         out: Optional[torch.Tensor] = None, window_overflow: Optional[torch.Tensor] = None) -> torch.Tensor:
        """match int32 [P, G]; terms int32 [G, W]; everything on the GPU.  window_overflow: optional int32 [1] counter of
        groups whose candidate range exceeded W (their result is a lower bound)."""
        assert match.dtype == torch.int32 and terms.dtype == torch.int32 and match.is_contiguous() and terms.is_contiguous()
        P, G = match.shape
        W = terms.shape[1]
        if out is None:
            out = torch.empty(G, dtype=torch.int32, device=match.device)
        check(self.lib.ss_raft_commit_scan_dev(self.h, _ptr(match), P, G, _ptr(last_commit), _ptr(log_end),
                                               _ptr(curr_term), _ptr(terms), W, threshold, _ptr(out), _ptr(window_overflow)))
        return out


class StepSync:
    """Host-side builder of an ss_step_sync: wait until every flag of `wait_flags` (a LOCAL device array of n_wait u64
    counters) is >= wait_value, and store signal_value to each pointer of `signal_ptrs` (local or peer) afterwards."""

    def __init__(self, wait_flags_ptr: int = 0, n_wait: int = 0, wait_value: int = 0,
                 signal_ptrs: Sequence[int] = (), signal_value: int = 0):
        self._sig = (C.c_void_p * max(1, len(signal_ptrs)))(*signal_ptrs)
        self.c = _lib.StepSync(C.c_void_p(wait_flags_ptr or None), n_wait, max(0, wait_value),
                               C.cast(self._sig, C.POINTER(C.c_void_p)), len(signal_ptrs), signal_value)


def _ctx_extras():
    def raft_kth_match(self, match: torch.Tensor, k: int) -> torch.Tensor:
        """k-th largest peer match per group (CRaft shadow_last_commit with k = threshold - 1)."""
        assert match.dtype == torch.int32 and match.is_contiguous()
        P, G = match.shape
        out = torch.empty(G, dtype=torch.int32, device=match.device)
        check(self.lib.ss_raft_kth_match_dev(self.h, _ptr(match), P, G, k, _ptr(out)))
        return out

    def prepare_merge(self, vote_bal: torch.Tensor, vote_mask: torch.Tensor, acks_cnt: torch.Tensor, data_shards: int,
                      population: int, fault_tolerance: int):
        """vote_bal int64 [R, N], vote_mask int32 [R, N] (0 = no vote), acks_cnt uint8 [N]."""
        assert vote_bal.dtype == torch.int64 and vote_mask.dtype == torch.int32 and acks_cnt.dtype == torch.uint8
        R, N = vote_bal.shape
        dev = vote_bal.device
        max_bal = torch.empty(N, dtype=torch.int64, device=dev)
        merged = torch.empty(N, dtype=torch.int32, device=dev)
        action = torch.empty(N, dtype=torch.uint8, device=dev)
        check(self.lib.ss_prepare_merge_dev(self.h, _ptr(vote_bal), _ptr(vote_mask), R, N, _ptr(acks_cnt), data_shards,
                                            population, fault_tolerance, _ptr(max_bal), _ptr(merged), _ptr(action)))
        return max_bal, merged, action

    def frame_accept_batch(self, shard_plane: torch.Tensor, shard_idx: int, d: int, p: int, data_len: int, slot: torch.Tensor,
                           ballot: torch.Tensor, msg_variant: int = 2):
        """shard_plane uint8 [n, shard_stride]; returns (out uint8 [n, frame_stride], frame_off int64 [n], frame_len int32 [n])."""
        n, ss = shard_plane.shape
        L = shard_len(data_len, d)
        stride = round_up(L + 96 + d + p, 16)
        dev = shard_plane.device
        out = torch.full((n, stride), 0xA5, dtype=torch.uint8, device=dev)   # the C ABI does not require a zeroed buffer
        off = torch.empty(n, dtype=torch.int64, device=dev)
        ln = torch.empty(n, dtype=torch.int32, device=dev)
        check(self.lib.ss_frame_accept_batch_dev(self.h, _ptr(shard_plane), ss, shard_idx, d, p, data_len, msg_variant,
                                                 _ptr(slot), _ptr(ballot), n, _ptr(out), stride, _ptr(off), _ptr(ln)))
        return out, off, ln

    def gossip_plan(self, me: int, population: int, data_shards: int, src_peer: torch.Tensor, avail: torch.Tensor,
                    policy_idx: torch.Tensor, policies: Sequence[Sequence[int]], peer_alive: int):
        """returns (targets int32 [N], excl int32 [population, N]); excl rows of unselected peers stay -1."""
        assert src_peer.dtype == torch.uint8 and avail.dtype == torch.int32 and policy_idx.dtype == torch.uint8
        pol = np.ascontiguousarray(np.array(policies, dtype=np.uint32))
        N = avail.numel()
        targets = torch.empty(N, dtype=torch.int32, device=avail.device)
        excl = torch.full((population, N), -1, dtype=torch.int32, device=avail.device)
        check(self.lib.ss_gossip_plan_dev(self.h, me, population, data_shards, _ptr(src_peer), _ptr(avail), _ptr(policy_idx),
                                          pol.ctypes.data, pol.shape[0], peer_alive, N, _ptr(targets), _ptr(excl)))
        return targets, excl

    def frame_accept_pack(self, shard_planes: torch.Tensor, data_len: int, d: int, p: int, policies: Sequence[Sequence[int]],
                          policy_idx: Optional[torch.Tensor], peer: int, slot: torch.Tensor, ballot: torch.Tensor, kind: int = 0,
                          msg_variant: int = 2, with_assignment: bool = False, max_shards: Optional[int] = None,
                          frame_stride: Optional[int] = None):
        """General Accept / WAL AcceptData packer.  shard_planes uint8 [d+p, n, shard_stride]; policies [K][population] shard
        bitmasks.  Returns (out uint8 [n, frame_stride], frame_off int64 [n], frame_len int32 [n])."""
        T, n, ss = shard_planes.shape
        assert T == d + p and shard_planes.is_contiguous()
        pol = np.ascontiguousarray(np.array(policies, dtype=np.uint32))
        dev = shard_planes.device
        pol_dev = torch.from_numpy(pol.view(np.int32)).to(dev)
        spec = _lib.FrameSpec(kind, msg_variant, d, p, data_len, pol.shape[1], 1 if with_assignment else 0, T)
        stride = frame_stride or int(self.lib.ss_frame_accept_max_len(C.byref(spec), max_shards if max_shards is not None else T))
        out = torch.full((n, stride), 0xA5, dtype=torch.uint8, device=dev)       # the C ABI does not require a zeroed buffer
        off = torch.empty(n, dtype=torch.int64, device=dev)
        ln = torch.empty(n, dtype=torch.int32, device=dev)
        check(self.lib.ss_frame_accept_pack_dev(self.h, C.byref(spec), _ptr(shard_planes), n * ss, ss, _ptr(pol_dev), pol.shape[0],
                                                _ptr(policy_idx), peer, _ptr(slot), _ptr(ballot), n, _ptr(out), stride, _ptr(off), _ptr(ln)))
        return out, off, ln

    def accept_reply_parse(self, buf: torch.Tensor, frame_off: torch.Tensor, frame_group: torch.Tensor, frame_peer: torch.Tensor,
                           window_base: torch.Tensor, reply_variant: int = 3, with_size: bool = False):
        """AcceptReply frames -> (rec_group int32, rec_slot uint8, rec_peer uint8, rec_ballot int64, rec_kind int32)."""
        assert buf.dtype == torch.uint8 and frame_off.dtype == torch.int64 and frame_group.dtype == torch.int32
        assert frame_peer.dtype == torch.uint8 and window_base.dtype == torch.int64
        n, dev = frame_off.numel(), buf.device
        rg = torch.empty(n, dtype=torch.int32, device=dev); rs_ = torch.empty(n, dtype=torch.uint8, device=dev)
        rp = torch.empty(n, dtype=torch.uint8, device=dev); rb = torch.empty(n, dtype=torch.int64, device=dev)
        rk = torch.empty(n, dtype=torch.int32, device=dev)
        check(self.lib.ss_accept_reply_parse_dev(self.h, _ptr(buf), buf.numel(), _ptr(frame_off), _ptr(frame_group), _ptr(frame_peer),
                                                 _ptr(window_base), n, window_base.numel(), reply_variant, 1 if with_size else 0,
                                                 _ptr(rg), _ptr(rs_), _ptr(rp), _ptr(rb), _ptr(rk)))
        return rg, rs_, rp, rb, rk

    def wal_commit_pack(self, newly: torch.Tensor, window_base: torch.Tensor, capacity: int, commit_variant: int = 2):
        """newly int64 [G] -> (entries uint8 [capacity, 24], entry_group int32, entry_len int32, n_entries int64 [1])."""
        dev = newly.device
        entries = torch.zeros((capacity, 24), dtype=torch.uint8, device=dev)
        eg = torch.empty(capacity, dtype=torch.int32, device=dev); el = torch.empty(capacity, dtype=torch.int32, device=dev)
        cnt = torch.zeros(1, dtype=torch.int64, device=dev)
        check(self.lib.ss_wal_commit_pack_dev(self.h, _ptr(newly), _ptr(window_base), newly.numel(), commit_variant, _ptr(entries),
                                              _ptr(eg), _ptr(el), capacity, _ptr(cnt)))
        return entries, eg, el, cnt

    def reconstruct_serve(self, shard_planes: torch.Tensor, shard_len_: int, req_group: torch.Tensor, req_held: torch.Tensor,
                          req_excl: torch.Tensor, req_status: torch.Tensor, reply_off: torch.Tensor, out_bytes: int):
        """shard_planes uint8 [T, n, shard_stride].  Returns (reply_mask int32 [R], out uint8 [out_bytes])."""
        T, n, ss = shard_planes.shape
        dev = shard_planes.device
        mask = torch.empty(req_group.numel(), dtype=torch.int32, device=dev)
        out = torch.full((out_bytes,), 0x77, dtype=torch.uint8, device=dev)
        check(self.lib.ss_reconstruct_serve_dev(self.h, _ptr(shard_planes), n * ss, ss, T, shard_len_, _ptr(req_group), _ptr(req_held),
                                                _ptr(req_excl), _ptr(req_status), _ptr(reply_off), req_group.numel(), _ptr(mask), _ptr(out)))
        return mask, out

    Context.frame_accept_pack = frame_accept_pack
    Context.accept_reply_parse = accept_reply_parse
    Context.wal_commit_pack = wal_commit_pack
    Context.reconstruct_serve = reconstruct_serve
    Context.gossip_plan = gossip_plan
    Context.frame_accept_batch = frame_accept_batch
    Context.raft_kth_match = raft_kth_match
    Context.prepare_merge = prepare_merge


_ctx_extras()


def craft_threshold(majority: int, fault_tolerance: int, full_copy_mode: bool) -> int:
    """craft/messages.rs:300-308"""
    return majority if full_copy_mode else majority + fault_tolerance


def crossword_brr_assignment(population: int, total_shards: int, shards_per_replica: int) -> list:
    """Balanced round-robin shard assignment policy of Crossword (crossword/mod.rs:866-888): replica r is assigned
    shards ((r*dj)..(r*dj+spr)).map(|i| i % T) with dj = T / n; returned as one bitmask of shard indices per replica.
    Host-side policy table handed to ss_tally_crossword_dev / ss_crossword_distribute_dev (nothing here touches data)."""
    dj = total_shards // population
    out = []
    for r in range(population):
        m = 0
        for i in range(r * dj, r * dj + shards_per_replica):
            m |= 1 << (i % total_shards)
        out.append(m)
    return out


class DevBuffer:
    """A raw device allocation from ss_dev_alloc (or a peer GPU's buffer opened through CUDA IPC).
    Exposes __cuda_array_interface__ so `torch.as_tensor(buf, device=...)` views it without a copy."""

    def __init__(self, ctx: "Context", ptr: int, nbytes: int, owned: bool):
        self.ctx, self.ptr, self.nbytes, self.owned = ctx, ptr, nbytes, owned
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 2}

    def tensor(self) -> torch.Tensor:
        return torch.as_tensor(self, device=torch.device("cuda", self.ctx.device))

    def free(self) -> None:
        if self.ptr:
            if self.owned:
                self.ctx.lib.ss_dev_free(self.ctx.h, self.ptr)
            else:
                self.ctx.lib.ss_ipc_close(self.ctx.h, self.ptr)
            self.ptr = 0


class ReedSolomon:
    """GPU-backed stand-in for `reed_solomon_erasure::galois_8::ReedSolomon`."""

    def __init__(self, ctx: Context, data_shards: int, parity_shards: int):
        self.ctx = ctx
        self.lib = ctx.lib
        h = C.c_void_p()
        check(self.lib.ss_rs_coder_create(ctx.h, data_shards, parity_shards, C.byref(h)))
        self.h = h
        self.d, self.p = data_shards, parity_shards

    def close(self) -> None:
        if getattr(self, "h", None) is not None and self.h:
            self.lib.ss_rs_coder_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def data_shard_count(self) -> int:
        return int(self.lib.ss_rs_data_shard_count(self.h))

    def parity_shard_count(self) -> int:
        return int(self.lib.ss_rs_parity_shard_count(self.h))

    def total_shard_count(self) -> int:
        return int(self.lib.ss_rs_total_shard_count(self.h))

    def matrix(self) -> np.ndarray:
        m = np.zeros((self.d + self.p, self.d), dtype=np.uint8)
        check(self.lib.ss_rs_coder_matrix(self.h, m.ctypes.data))
        return m

    def set_variant(self, v: int) -> None:
        check(self.lib.ss_rs_set_variant(self.h, v))

    def last_kernel(self) -> str:
        return self.lib.ss_rs_last_kernel(self.h).decode()

    # ---- single codeword, host slices (crate API) ---------------------------------------------
    @staticmethod
    def _ptr_array(shards: Sequence[np.ndarray]):
        return (C.c_void_p * len(shards))(*[s.ctypes.data for s in shards])

    def encode(self, shards: List[np.ndarray]) -> None:
        """shards: d+p uint8 arrays of equal length; the last p are overwritten with parity."""
        if len(shards) == 0:
            raise SummersetError(_lib.SS_ERR_TOO_FEW_SHARDS, "too few shards")
        L = len(shards[0])
        if any(len(s) != L for s in shards):
            raise SummersetError(_lib.SS_ERR_INCORRECT_SHARD_SIZE, "incorrect shard size")
        check(self.lib.ss_rs_encode(self.h, self._ptr_array(shards), len(shards), L))

    def _reconstruct(self, shards: List[Optional[np.ndarray]], data_only: bool) -> None:
        sizes = {len(s) for s in shards if s is not None}
        if len(sizes) > 1:
            raise SummersetError(_lib.SS_ERR_INCORRECT_SHARD_SIZE, "incorrect shard size")
        L = sizes.pop() if sizes else 0
        present = np.array([0 if s is None else 1 for s in shards], dtype=np.uint8)
        bufs = [s if s is not None else np.zeros(max(L, 1), dtype=np.uint8) for s in shards]
        fn = self.lib.ss_rs_reconstruct_data if data_only else self.lib.ss_rs_reconstruct
        if L == 0 and len(shards) == self.d + self.p:
            raise SummersetError(_lib.SS_ERR_TOO_FEW_SHARDS_PRESENT, "too few shards present")
        check(fn(self.h, self._ptr_array(bufs), present.ctypes.data, len(shards), L))
        for i in range(len(shards)):
            if shards[i] is None and present[i]:
                shards[i] = bufs[i]

    def reconstruct(self, shards: List[Optional[np.ndarray]]) -> None:
        self._reconstruct(shards, False)

    def reconstruct_data(self, shards: List[Optional[np.ndarray]]) -> None:
        self._reconstruct(shards, True)

    def verify(self, shards: List[np.ndarray]) -> bool:
        L = len(shards[0]) if shards else 0
        if any(len(s) != L for s in shards):
            raise SummersetError(_lib.SS_ERR_INCORRECT_SHARD_SIZE, "incorrect shard size")
        ok = C.c_int(0)
        check(self.lib.ss_rs_verify(self.h, self._ptr_array(shards), len(shards), L, C.byref(ok)))
        return bool(ok.value)

    # ---- batched, device-resident --------------------------------------------------------------
    def parity_layout(self, data_len: int, n: int) -> Tuple[int, int, int]:
        """(L, shard_stride, plane_stride) of the padded-16 parity layout for uniform codewords."""
        L = shard_len(data_len, self.d)
        ds = round_up(L, 16)
        return L, ds, ds * n

    def encode_uniform(self, data: torch.Tensor, data_len: int, parity: Optional[torch.Tensor] = None,
                       data_stride: Optional[int] = None) -> torch.Tensor:
        """data: uint8 [n, data_stride] on the GPU, codeword g = data[g, :data_len].
        Returns parity uint8 [p, n, round_up(L,16)] (bytes past L are zero)."""
        assert data.is_cuda and data.dtype == torch.uint8 and data.is_contiguous()
        n = data.shape[0]
        stride = data.shape[1] if data_stride is None else data_stride
        L, ds, ps = self.parity_layout(data_len, n)
        if parity is None:
            parity = torch.empty((self.p, n, ds), dtype=torch.uint8, device=data.device)
        check(self.lib.ss_rs_encode_uniform_dev(self.h, _ptr(data), stride, data_len, n, _ptr(parity), ps, ds,
                                                SS_RS_OUT_PADDED16))
        return parity

    def encode_batch(self, data: torch.Tensor, data_off: torch.Tensor, data_len: torch.Tensor, parity: torch.Tensor,
                     plane_stride: int, par_off: torch.Tensor, padded: bool = True) -> None:
        assert data.is_cuda and data_off.dtype == torch.int64 and data_len.dtype == torch.int32 and par_off.dtype == torch.int64
        check(self.lib.ss_rs_encode_batch_dev(self.h, _ptr(data), _ptr(data_off), _ptr(data_len), data_len.numel(),
                                              _ptr(parity), plane_stride, _ptr(par_off),
                                              SS_RS_OUT_PADDED16 if padded else 0))

    def reconstruct_batch(self, shards: torch.Tensor, plane_stride: int, off: torch.Tensor, data_len: torch.Tensor,
                          present: torch.Tensor, data_only: bool, padded: bool = True) -> torch.Tensor:
        assert shards.is_cuda and off.dtype == torch.int64 and data_len.dtype == torch.int32 and present.dtype == torch.int32
        n = data_len.numel()
        status = torch.empty(n, dtype=torch.int32, device=shards.device)
        check(self.lib.ss_rs_reconstruct_batch_dev(self.h, _ptr(shards), plane_stride, _ptr(off), _ptr(data_len),
                                                   _ptr(present), n, 1 if data_only else 0, _ptr(status),
                                                   SS_RS_OUT_PADDED16 if padded else 0))
        return status

    def reconstruct_uniform(self, shards: torch.Tensor, data_len: int, present: torch.Tensor, data_only: bool) -> torch.Tensor:
        """shards uint8 [d+p, n, shard_stride] (padded-16 slots); present int32 [n].  Regenerates in place; returns status."""
        assert shards.is_cuda and shards.dtype == torch.uint8 and shards.is_contiguous() and shards.dim() == 3
        assert present.dtype == torch.int32 and present.numel() == shards.shape[1]
        t, n, ss = shards.shape
        assert t == self.d + self.p
        status = torch.empty(n, dtype=torch.int32, device=shards.device)
        check(self.lib.ss_rs_reconstruct_uniform_dev(self.h, _ptr(shards), n * ss, ss, data_len, _ptr(present), n,
                                                     1 if data_only else 0, _ptr(status)))
        return status

    def reconstruct_reply(self, shards: torch.Tensor, data_len: int, window: int, inst_status: torch.Tensor,
                          inst_bal: torch.Tensor, present: torch.Tensor, exec_bar: torch.Tensor, reply_buf: torch.Tensor,
                          reply_off: torch.Tensor, reply_mask: torch.Tensor, reply_inst: torch.Tensor,
                          reply_ballot: torch.Tensor, want_taken: bool = True):
        """ReconstructReply receiving for G groups of `window` instances (ss_reconstruct_reply_dev).  shards uint8
        [d+p, G*window, shard_stride] (padded-16 slots), inst_status uint8 / inst_bal int64 / present int32 [G*window],
        exec_bar int32 [G]; present and exec_bar are updated in place.  Replies in the layout reconstruct_serve writes:
        reply_buf uint8, reply_off int64, reply_mask int32, reply_inst int32 (-1 = skip), reply_ballot int64.
        Returns (submit int64 [G], taken int32 [R] or None)."""
        assert shards.is_cuda and shards.dtype == torch.uint8 and shards.is_contiguous() and shards.dim() == 3
        t, n, ss = shards.shape
        assert t == self.d + self.p and n % window == 0
        assert inst_status.dtype == torch.uint8 and inst_bal.dtype == torch.int64 and present.dtype == torch.int32
        assert exec_bar.dtype == torch.int32 and reply_buf.dtype == torch.uint8 and reply_off.dtype == torch.int64
        assert reply_mask.dtype == torch.int32 and reply_inst.dtype == torch.int32 and reply_ballot.dtype == torch.int64
        G, R = n // window, reply_off.numel()
        assert present.numel() == n and inst_status.numel() == n and inst_bal.numel() == n and exec_bar.numel() == G
        # the call writes every entry of both, except that an empty batch launches nothing
        submit = (torch.empty if R else torch.zeros)(G, dtype=torch.int64, device=shards.device)
        taken = torch.empty(R, dtype=torch.int32, device=shards.device) if want_taken else None
        check(self.lib.ss_reconstruct_reply_dev(self.h, _ptr(shards), n * ss, ss, data_len, G, window, _ptr(inst_status),
                                                _ptr(inst_bal), _ptr(present), _ptr(exec_bar), _ptr(reply_buf),
                                                _ptr(reply_off), _ptr(reply_mask), _ptr(reply_inst), _ptr(reply_ballot),
                                                R, _ptr(submit), _ptr(taken)))
        return submit, taken

    def accept_step_fused(self, data: torch.Tensor, data_len: int, parity: torch.Tensor, planes: torch.Tensor,
                          threshold: int, committed: torch.Tensor, commit_bar: Optional[torch.Tensor]) -> None:
        """BASELINE config 3 step: RS-encode n groups' request batches + tally their ack windows, one launch."""
        n = data.shape[0]
        R, G = planes.shape
        assert G == n
        L, ds, ps = self.parity_layout(data_len, n)
        check(self.lib.ss_accept_step_fused_dev(self.h, _ptr(data), data.shape[1], data_len, n, _ptr(parity), ps, ds,
                                                SS_RS_OUT_PADDED16, _ptr(planes), R, threshold, _ptr(committed),
                                                _ptr(commit_bar)))

    def accept_step_replicate(self, data: torch.Tensor, data_len: int, shard_planes: Sequence[int], shard_stride: int,
                              planes: Optional[torch.Tensor], threshold: int, committed: Optional[torch.Tensor],
                              commit_bar: Optional[torch.Tensor], sync: Optional["StepSync"] = None) -> None:
        """Multi-GPU accept step: encode + tally + write every shard plane to its (local or peer) destination.
        shard_planes: d+p raw device pointers (ints).  sync: step flags (tally waits, followers are signalled)."""
        arr = (C.c_void_p * len(shard_planes))(*shard_planes)
        n = data.shape[0]
        R = planes.shape[0] if planes is not None else 0
        check(self.lib.ss_accept_step_replicate_dev(self.h, _ptr(data), data.shape[1], data_len, n, arr, shard_stride,
                                                    _ptr(planes), R, threshold, _ptr(committed), _ptr(commit_bar),
                                                    C.byref(sync.c) if sync else None))

    def crossword_distribute(self, data: torch.Tensor, data_off: torch.Tensor, data_len: torch.Tensor, spr: torch.Tensor,
                             rep_off: torch.Tensor, replica_logs: Sequence[int]) -> None:
        """Crossword: encode the ragged batch and write replica r's spr[g] shards {(r*dj + k) mod T} into replica_logs[r]
        (len(replica_logs) = population; T = d + p must be a multiple of it) at rep_off[g] + k * cw_slot_pitch(L_g)."""
        assert data_off.dtype == torch.int64 and data_len.dtype == torch.int32 and spr.dtype == torch.uint8 and rep_off.dtype == torch.int64
        arr = (C.c_void_p * len(replica_logs))(*replica_logs)
        check(self.lib.ss_crossword_distribute_dev(self.h, _ptr(data), _ptr(data_off), _ptr(data_len), _ptr(spr),
                                                   _ptr(rep_off), data_len.numel(), arr, len(replica_logs)))

    def accept_step_fused_host(self, data: np.ndarray, data_len: int, parity: np.ndarray, planes: np.ndarray,
                               threshold: int, committed: np.ndarray, commit_bar: Optional[np.ndarray]) -> None:
        """HOST buffers through ss_accept_step_fused: data uint8 [n, stride]; parity uint8 [p, n, shard_stride];
        planes uint64 [R, n]; committed uint64 [n]; commit_bar uint32 [n] or None."""
        assert data.dtype == np.uint8 and parity.dtype == np.uint8 and data.flags.c_contiguous and parity.flags.c_contiguous
        assert planes.dtype == np.uint64 and planes.flags.c_contiguous and committed.dtype == np.uint64
        n, stride = data.shape
        p, n2, ss = parity.shape
        R, G = planes.shape
        assert p == self.p and n2 == n and G == n and committed.shape == (n,)
        check(self.lib.ss_accept_step_fused(self.h, data.ctypes.data, stride, data_len, n, parity.ctypes.data, n * ss, ss,
                                            planes.ctypes.data, R, threshold, committed.ctypes.data,
                                            commit_bar.ctypes.data if commit_bar is not None else None))

    def encode_uniform_host(self, data: np.ndarray, data_len: int, parity: np.ndarray) -> None:
        """HOST buffers through ss_rs_encode_uniform: data uint8 [n, stride]; parity uint8 [p, n, shard_stride]."""
        assert data.dtype == np.uint8 and parity.dtype == np.uint8 and data.flags.c_contiguous and parity.flags.c_contiguous
        n, stride = data.shape
        p, n2, ss = parity.shape
        assert p == self.p and n2 == n
        check(self.lib.ss_rs_encode_uniform(self.h, data.ctypes.data, stride, data_len, n, parity.ctypes.data,
                                            n * ss, ss))


# =================================================================================================
# Host-side mirrors of the reference's helper types (pure host logic; no shard arithmetic here)
# =================================================================================================
class Bitmap:
    """Mirror of src/utils/bitmap.rs: compact u8-id -> bool map."""

    def __init__(self, size: int, ones: bool = False):
        if size == 0:
            raise AssertionError(f"invalid bitmap size {size}")     # bitmap.rs:64 (panics)
        if not (0 < size <= 255):
            raise ValueError("size must fit u8")
        self._size = size
        self._bits = (1 << size) - 1 if ones else 0

    @classmethod
    def from_indices(cls, size: int, ones: Iterable[int]) -> "Bitmap":
        """From<(u8, Vec<u8>)> / From<(u8, Range<u8>)> (bitmap.rs:151-185); out-of-range index panics there."""
        b = cls(size, False)
        for i in ones:
            b.set(i, True)
        return b

    def set(self, idx: int, flag: bool) -> None:
        if idx >= self._size or idx < 0:
            raise SummersetError(_lib.SS_ERR_INVALID_INDEX, f"index {idx} out of bound")   # bitmap.rs:76-81
        if flag:
            self._bits |= 1 << idx
        else:
            self._bits &= ~(1 << idx)

    def get(self, idx: int) -> bool:
        if idx >= self._size or idx < 0:
            raise SummersetError(_lib.SS_ERR_INVALID_INDEX, f"index {idx} out of bound")   # bitmap.rs:89-94
        return bool((self._bits >> idx) & 1)

    def size(self) -> int:
        return self._size

    def count(self) -> int:
        return bin(self._bits).count("1")

    def flip(self) -> None:
        self._bits ^= (1 << self._size) - 1

    def union(self, other: "Bitmap") -> None:
        if self._size != other._size:
            raise SummersetError(_lib.SS_ERR_INVALID_ARG, f"unioning sizes mismatch: {self._size} != {other._size}")
        self._bits |= other._bits

    def clear(self) -> None:
        self._bits = 0

    def iter(self):
        return ((i, bool((self._bits >> i) & 1)) for i in range(self._size))

    def __iter__(self):
        return self.iter()

    def __eq__(self, other):
        return isinstance(other, Bitmap) and self._size == other._size and self._bits == other._bits

    def __repr__(self):
        return "{" + str(self._size) + "; [" + ", ".join(str(i) for i, f in self.iter() if f) + "]}"

    def to_mask(self) -> int:
        return self._bits

    def encode(self) -> bytes:
        """bincode 2 `standard()` of Bitmap (bitmap.rs:20-30): bit length, then the usize block slice."""
        nblocks = (self._size + 63) // 64
        out = bytearray(bincode_varint(self._size)) + bytearray(bincode_varint(nblocks))
        for b in range(nblocks):
            out += bincode_varint((self._bits >> (64 * b)) & ((1 << 64) - 1))
        return bytes(out)


def bincode_varint(v: int) -> bytes:
    """bincode 2 standard-config unsigned varint."""
    if v < 251:
        return bytes([v])
    if v < 1 << 16:
        return bytes([251]) + v.to_bytes(2, "little")
    if v < 1 << 32:
        return bytes([252]) + v.to_bytes(4, "little")
    return bytes([253]) + v.to_bytes(8, "little")


def bincode_string(s: str) -> bytes:
    """bincode 2 standard-config String / newtype-of-String: varint byte length + UTF-8."""
    b = s.encode("utf-8")
    return bincode_varint(len(b)) + b


class RSCodeword:
    """Mirror of src/utils/rscoding.rs `RSCodeword<T>` with T = an already-serialized byte string."""

    def __init__(self, d: int, p: int, data_len: int, shard_len_: int, shards: List[Optional[np.ndarray]],
                 data_copy: Optional[bytes]):
        self.num_data_shards_, self.num_parity_shards_ = d, p
        self.data_len_, self.shard_len_ = data_len, shard_len_
        self.shards = shards
        self.data_copy = data_copy

    # rscoding.rs:165-220
    @classmethod
    def _internal_new(cls, data_copy, data_bytes: Optional[bytes], data_len: int, d: int, p: int) -> "RSCodeword":
        if d == 0:
            raise SummersetError(_lib.SS_ERR_TOO_FEW_DATA_SHARDS, "num_data_shards is zero")
        L = shard_len(data_len, d)
        if data_bytes is not None:
            padded = np.zeros(L * d, dtype=np.uint8)
            padded[:data_len] = np.frombuffer(data_bytes, dtype=np.uint8)
            shards: List[Optional[np.ndarray]] = [padded[i * L:(i + 1) * L] for i in range(d)]
            shards += [None] * p
        else:
            shards = [None] * (d + p)
        return cls(d, p, data_len, L, shards, data_copy)

    @classmethod
    def from_data(cls, data: bytes, d: int, p: int) -> "RSCodeword":
        return cls._internal_new(data, data, len(data), d, p)

    @classmethod
    def from_null(cls, d: int, p: int) -> "RSCodeword":
        return cls._internal_new(None, None, 0, d, p)

    def subset_copy(self, subset: Bitmap, copy_data: bool) -> "RSCodeword":
        if self.data_len_ == 0:
            raise SummersetError(_lib.SS_ERR_INVALID_ARG, "codeword is null")
        shards: List[Optional[np.ndarray]] = [None] * self.num_shards()
        for i, flag in subset.iter():
            if not flag:
                continue
            if i >= len(shards):
                raise SummersetError(_lib.SS_ERR_INVALID_INDEX, f"shard index {i} out-of-bound")
            shards[i] = None if self.shards[i] is None else self.shards[i].copy()
        return RSCodeword(self.num_data_shards_, self.num_parity_shards_, self.data_len_, self.shard_len_, shards,
                          self.data_copy if copy_data else None)

    def absorb_other(self, other: "RSCodeword") -> None:
        if self.num_data_shards_ != other.num_data_shards_:
            raise SummersetError(_lib.SS_ERR_INVALID_ARG, "num_data_shards mismatch")
        if self.num_parity_shards_ != other.num_parity_shards_:
            raise SummersetError(_lib.SS_ERR_INVALID_ARG, "num_parity_shards mismatch")
        if self.data_len_ != 0 and self.data_len_ != other.data_len_:
            raise SummersetError(_lib.SS_ERR_INVALID_ARG, "data_len mismatch")
        if self.shard_len_ != 0 and self.shard_len_ != other.shard_len_:
            raise SummersetError(_lib.SS_ERR_INVALID_ARG, "shard_len mismatch")
        if self.data_len_ == 0:
            self.data_len_, self.shard_len_ = other.data_len_, other.shard_len_
        for i in range(len(other.shards)):
            if other.shards[i] is not None and self.shards[i] is None:
                self.shards[i] = other.shards[i]
                other.shards[i] = None

    def num_data_shards(self) -> int: return self.num_data_shards_
    def num_parity_shards(self) -> int: return self.num_parity_shards_
    def num_shards(self) -> int: return len(self.shards)
    def avail_data_shards(self) -> int: return sum(s is not None for s in self.shards[:self.num_data_shards_])
    def avail_parity_shards(self) -> int: return sum(s is not None for s in self.shards[self.num_data_shards_:])
    def avail_shards(self) -> int: return sum(s is not None for s in self.shards)
    def data_len(self) -> int: return self.data_len_
    def shard_len(self) -> int: return self.shard_len_

    def avail_shards_map(self) -> Bitmap:
        return Bitmap.from_indices(self.num_shards(), [i for i, s in enumerate(self.shards) if s is not None])

    def _splits_match(self, rs: ReedSolomon) -> None:
        if rs.data_shard_count() != self.num_data_shards_:
            raise SummersetError(_lib.SS_ERR_INVALID_ARG, "num_data_shards mismatch")
        if rs.parity_shard_count() != self.num_parity_shards_:
            raise SummersetError(_lib.SS_ERR_INVALID_ARG, "num_parity_shards mismatch")

    def compute_parity(self, rs: Optional[ReedSolomon]) -> None:            # rscoding.rs:447-486
        if self.data_len_ == 0:
            raise SummersetError(_lib.SS_ERR_INVALID_ARG, "codeword is null")
        if self.num_parity_shards_ == 0:
            return
        if rs is None:
            raise SummersetError(_lib.SS_ERR_INVALID_ARG, "ReedSolomon coder is None")
        self._splits_match(rs)
        if self.avail_data_shards() < self.num_data_shards_:
            raise SummersetError(_lib.SS_ERR_INVALID_ARG, "not all data shards present")
        for i in range(self.num_data_shards_, len(self.shards)):
            if self.shards[i] is None:
                self.shards[i] = np.zeros(self.shard_len_, dtype=np.uint8)
        bufs = [np.ascontiguousarray(s) for s in self.shards]
        rs.encode(bufs)
        self.shards = bufs

    def _reconstruct(self, rs: Optional[ReedSolomon], data_only: bool) -> None:   # rscoding.rs:490-520
        if self.data_len_ == 0:
            raise SummersetError(_lib.SS_ERR_INVALID_ARG, "codeword is null")
        if self.num_parity_shards_ == 0:
            if self.avail_data_shards() == self.num_data_shards_:
                return
            raise SummersetError(_lib.SS_ERR_INVALID_ARG, "insufficient data shards")
        if rs is None:
            raise SummersetError(_lib.SS_ERR_INVALID_ARG, "ReedSolomon coder is None")
        self._splits_match(rs)
        bufs = [None if s is None else np.ascontiguousarray(s) for s in self.shards]
        if data_only:
            rs.reconstruct_data(bufs)
        else:
            rs.reconstruct(bufs)
        self.shards = bufs

    def reconstruct_all(self, rs: Optional[ReedSolomon]) -> None:
        self._reconstruct(rs, False)

    def reconstruct_data(self, rs: Optional[ReedSolomon]) -> None:
        self._reconstruct(rs, True)

    def verify_parity(self, rs: Optional[ReedSolomon]) -> bool:             # rscoding.rs:542-576
        if self.data_len_ == 0:
            raise SummersetError(_lib.SS_ERR_INVALID_ARG, "codeword is null")
        if self.num_parity_shards_ == 0:
            if self.avail_data_shards() == self.num_data_shards_:
                return True
            raise SummersetError(_lib.SS_ERR_INVALID_ARG, "not all shards present")
        if rs is None:
            raise SummersetError(_lib.SS_ERR_INVALID_ARG, "ReedSolomon is None")
        self._splits_match(rs)
        if self.avail_shards() < self.num_shards():
            raise SummersetError(_lib.SS_ERR_INVALID_ARG, "not all shards present")
        return rs.verify([np.ascontiguousarray(s) for s in self.shards])

    def get_data(self) -> bytes:                                            # rscoding.rs:581-606
        if self.data_len_ == 0:
            raise SummersetError(_lib.SS_ERR_INVALID_ARG, "codeword is null")
        if self.avail_data_shards() < self.num_data_shards_:
            raise SummersetError(_lib.SS_ERR_INVALID_ARG, "not all data shards present")
        if self.data_copy is None:
            cat = np.concatenate(self.shards[:self.num_data_shards_])      # ShardsReader, rscoding.rs:649-682
            self.data_copy = cat[:self.data_len_].tobytes()
        return self.data_copy
