/*
 * summerset_b200.h -- C ABI of libsummerset_b200.so
 *
 * The B200 (sm_100a) implementation of Summerset's quorum-tally + Reed-Solomon hot path.
 * Plain C: pointers and sizes only, no torch / C++ types.  This is the boundary a Rust
 * `extern "C"` block (INTEGRATION.md) binds; the GenericReplica / SmrProtocol surface
 * (src/server/replica.rs:15-42, src/protocols/mod.rs:118-215) is untouched by it.
 *
 * The reference has no FFI for this path (SURVEY.md 8b).  Each entry point states the reference
 * interface it replaces (path:line relative to the reference tree, josehu07/summerset @ 1daf80aa).
 *
 * Conventions
 *   - Ownership: the caller owns every buffer.  The library never frees or retains caller
 *     memory (rscoding.rs:479-484, :515-517 -- encode/reconstruct mutate caller slices in place).
 *   - Errors: `int` return, 0 = ok, negative = error.  Codes -1..-13 mirror the variants of
 *     `reed_solomon_erasure::Error`, which the reference converts into `SummersetError(String)`
 *     (src/utils/error.rs:6-14,59); ss_last_error() gives the message text for that conversion.
 *   - Threading: every call may come from a different OS thread (the replica's run() task
 *     migrates across tokio worker threads, summerset_server/src/main.rs:45-47,133-137).  No
 *     thread-local CUDA state is assumed: each call binds its handle's device.  Calls on ONE
 *     handle must be serialised by the caller (the reference calls from a single task).
 *   - `_dev` entry points take DEVICE pointers and are asynchronous on the context's stream;
 *     the others take HOST pointers, copy in/out and return when the result is in host memory.
 *   - No CPU fallback: every compute entry point fails with SS_ERR_NO_DEVICE / SS_ERR_CUDA when
 *     no sm_100 device is usable.
 */
#ifndef SUMMERSET_B200_H
#define SUMMERSET_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SS_VERSION 200 /* 0.2.0: engine, step flags, wire formats, uniform reconstruct; several round-1 signatures gained a parameter */

/* ---- error codes ---------------------------------------------------------------------------
 * -1..-13: reed_solomon_erasure::Error variants in declaration order. */
enum {
    SS_OK = 0,
    SS_ERR_TOO_FEW_SHARDS = -1,
    SS_ERR_TOO_MANY_SHARDS = -2,
    SS_ERR_TOO_FEW_DATA_SHARDS = -3,
    SS_ERR_TOO_MANY_DATA_SHARDS = -4,
    SS_ERR_TOO_FEW_PARITY_SHARDS = -5,
    SS_ERR_TOO_MANY_PARITY_SHARDS = -6,
    SS_ERR_TOO_FEW_BUFFER_SHARDS = -7,
    SS_ERR_TOO_MANY_BUFFER_SHARDS = -8,
    SS_ERR_INCORRECT_SHARD_SIZE = -9,
    SS_ERR_TOO_FEW_SHARDS_PRESENT = -10,
    SS_ERR_EMPTY_SHARD = -11,
    SS_ERR_INVALID_SHARD_FLAGS = -12,
    SS_ERR_INVALID_INDEX = -13,
    /* library-level */
    SS_ERR_INVALID_ARG = -20,
    SS_ERR_UNSUPPORTED = -21,
    SS_ERR_OUT_OF_MEMORY = -22,
    SS_ERR_NO_DEVICE = -30,   /* no CUDA device / not sm_100: there is NO CPU fallback */
    SS_ERR_CUDA = -31
};

typedef struct ss_ctx ss_ctx;           /* device + stream + scratch */
typedef struct ss_rs_coder ss_rs_coder; /* replaces reed_solomon_erasure::galois_8::ReedSolomon */

int ss_version(void);
/* Text of the most recent error raised on the CALLING thread (one buffer per OS thread; the pointer stays valid until
 * the next failing call on that thread).  Read it right after the failing call, before yielding: two replicas driven
 * from two tokio worker threads never see each other's text.  Maps to SummersetError::msg (src/utils/error.rs:6-14). */
const char *ss_last_error(void);
const char *ss_strerror(int code);

/* ---- context ------------------------------------------------------------------------------- */
/* Creates a context on `device` with its own non-blocking stream. */
int ss_ctx_create(int device, ss_ctx **out);
/* Same, but launches on a caller-owned cudaStream_t (e.g. torch's current stream). */
int ss_ctx_create_on_stream(int device, void *cuda_stream, ss_ctx **out);
/* Coders / engines created on a context keep it alive: destroying the context before them only marks it closed and the
 * last handle's destroy call frees it (either order is safe). */
int ss_ctx_destroy(ss_ctx *ctx);
int ss_ctx_sync(ss_ctx *ctx);               /* cudaStreamSynchronize on the context's stream */
void *ss_ctx_stream(ss_ctx *ctx);           /* the cudaStream_t */
int ss_ctx_sm_count(ss_ctx *ctx);
/* number of kernels this context has launched so far (bench.py's gpu_launches claim) */
uint64_t ss_ctx_launch_count(ss_ctx *ctx);

/* device / pinned-host memory helpers for non-CUDA callers (Rust shim) */
int ss_dev_alloc(ss_ctx *ctx, size_t bytes, void **dptr);
int ss_dev_free(ss_ctx *ctx, void *dptr);
int ss_dev_memset(ss_ctx *ctx, void *dptr, int value, size_t bytes);      /* async */
int ss_host_alloc(ss_ctx *ctx, size_t bytes, void **hptr);                /* pinned */
/* write-combined pinned memory: for buffers the CPU only WRITES and the GPU reads (payload staging); faster H2D on
 * some hosts, very slow for CPU reads */
int ss_host_alloc_wc(ss_ctx *ctx, size_t bytes, void **hptr);
int ss_host_free(ss_ctx *ctx, void *hptr);
int ss_copy_h2d(ss_ctx *ctx, void *dst_dev, const void *src_host, size_t bytes); /* async */
int ss_copy_d2h(ss_ctx *ctx, void *dst_host, const void *src_dev, size_t bytes); /* async */

int ss_copy_d2d(ss_ctx *ctx, void *dst_dev, const void *src_dev, size_t bytes);  /* async; dst/src may be peer memory */

/* ---- cross-process peer memory (one process per GPU, NVLink) ---------------------------------
 * ss_ipc_export gives a 64-byte handle for a buffer obtained from ss_dev_alloc; another process on the same
 * box turns it into a device pointer with ss_ipc_open (peer access is enabled on first use).  The pointers
 * can be passed to ss_accept_step_replicate_dev / ss_copy_d2d: kernels then store straight into the peer
 * GPU's HBM over NVLink -- the replacement for TransportHub::send_msg of a shard (server/transport.rs:258-345,
 * rspaxos/request.rs:127-142) when the simulated replicas of a group live on the GPUs of one box. */
#define SS_IPC_HANDLE_BYTES 64
int ss_ipc_export(ss_ctx *ctx, void *dptr, uint8_t handle[SS_IPC_HANDLE_BYTES]);
int ss_ipc_open(ss_ctx *ctx, const uint8_t handle[SS_IPC_HANDLE_BYTES], void **dptr);
int ss_ipc_close(ss_ctx *ctx, void *dptr);

/* ---- Reed-Solomon coder --------------------------------------------------------------------
 * Replaces ReedSolomon::new(d, p) (constructors at rspaxos/mod.rs:606, crossword/mod.rs:827,
 * craft/mod.rs:534, benches/rse_bench.rs:51).  GF(2^8) poly 0x11D; systematic matrix
 * M = vandermonde(d+p, d) * inverse(top d x d) -- bit-identical to the crate's.
 * Errors: d == 0 -> TOO_FEW_DATA_SHARDS, p == 0 -> TOO_FEW_PARITY_SHARDS, d+p > 256 ->
 * TOO_MANY_SHARDS (the crate's behaviour; Summerset special-cases p == 0 before touching the
 * coder, rscoding.rs:454-456,498-507).  Batched kernels need d <= 32, p <= 8, d+p <= 32. */
int ss_rs_coder_create(ss_ctx *ctx, int data_shards, int parity_shards, ss_rs_coder **out);
int ss_rs_coder_destroy(ss_rs_coder *coder);
int ss_rs_data_shard_count(const ss_rs_coder *coder);    /* rscoding.rs:428 */
int ss_rs_parity_shard_count(const ss_rs_coder *coder);  /* rscoding.rs:434 */
int ss_rs_total_shard_count(const ss_rs_coder *coder);
/* copies the (d+p) x d coding matrix, row-major, into out */
int ss_rs_coder_matrix(const ss_rs_coder *coder, uint8_t *out);

/* -- one codeword, HOST slices: the four crate methods RSCodeword calls ----------------------
 * shards: n_shards (= d+p) pointers to shard_len bytes each.
 * ss_rs_encode            replaces rs.encode(slices)             (rscoding.rs:484)
 * ss_rs_reconstruct       replaces rs.reconstruct(&mut shards)   (rscoding.rs:517)
 * ss_rs_reconstruct_data  replaces rs.reconstruct_data(..)       (rscoding.rs:515)
 * ss_rs_verify            replaces rs.verify(&slices)            (rscoding.rs:575)
 * present[j] != 0 <=> shards[j] is Some(..); missing entries must still point at a
 * shard_len-byte buffer to fill (the crate allocates it; here the caller does).  On success
 * present[] is updated for the regenerated shards.  Fewer than d present ->
 * SS_ERR_TOO_FEW_SHARDS_PRESENT and no output is written (never partial). */
int ss_rs_encode(ss_rs_coder *coder, uint8_t *const *shards, size_t n_shards, size_t shard_len);
int ss_rs_reconstruct(ss_rs_coder *coder, uint8_t *const *shards, uint8_t *present,
                      size_t n_shards, size_t shard_len);
int ss_rs_reconstruct_data(ss_rs_coder *coder, uint8_t *const *shards, uint8_t *present,
                           size_t n_shards, size_t shard_len);
int ss_rs_verify(ss_rs_coder *coder, const uint8_t *const *shards, size_t n_shards,
                 size_t shard_len, int *ok);

/* -- batched, device-resident log of codewords ------------------------------------------------
 * Codeword g: payload bytes data[data_off[g] .. +data_len[g]) = the bincode-serialised request
 * batch RSCodeword::from_data produces (rscoding.rs:223-243).  Geometry is the reference's
 * (rscoding.rs:177-199): L_g = ceil(data_len/d); data shard i = payload bytes [i*L, (i+1)*L),
 * zero-padded past data_len; a contiguous split, so data shards are VIEWS of the payload.
 * Parity shard j of codeword g is written to parity[j*plane_stride + par_off[g] .. +L_g).
 * One launch = RSCodeword::from_data's split + compute_parity (rspaxos/request.rs:72-77,
 * crossword/request.rs:82-87) for n codewords; plane j is at the same time the packed
 * per-destination send buffer subset_copy builds one codeword at a time (rscoding.rs:255-293,
 * rspaxos/request.rs:127-142).  data_len[g] == 0 (null codeword) is skipped.
 *
 * flags:
 *   SS_RS_OUT_PADDED16  every parity slot starts 16-byte aligned and has capacity
 *                       round_up(L_g,16); bytes [L_g, round_up) are written as zeros.  This is
 *                       the fast path (128-bit stores).  Without it stores are byte-exact.
 *                       16-byte alignment is what correctness needs; where the layout is yours to choose,
 *                       prefer 32-byte multiples for par_off / shard_stride: write-heavy kernels lose ~7 %
 *                       when rows start in the middle of a DRAM sector (see SS_CW_SLOT_PITCH).
 *   SS_RS_EMIT_DATA     `parity` is plane d of a (d+p)-plane shard store with the same plane_stride:
 *                       the kernel ALSO copies data shard i into plane i (parity - (d-i)*plane_stride),
 *                       so all d+p planes are packed per-destination send buffers after one pass.
 * The payload arena must be a CUDA allocation (the kernel issues aligned 16-byte loads that may
 * cover up to 15 bytes either side of a payload, inside the allocation's 256-byte granule). */
#define SS_RS_OUT_PADDED16 1u
#define SS_RS_EMIT_DATA 2u
int ss_rs_encode_batch_dev(ss_rs_coder *coder, const uint8_t *data, const uint64_t *data_off,
                           const uint32_t *data_len, uint64_t n, uint8_t *parity,
                           uint64_t plane_stride, const uint64_t *par_off, uint32_t flags);
/* uniform geometry: data_off[g] = g*data_stride, data_len[g] = data_len, par_off[g] = g*shard_stride */
int ss_rs_encode_uniform_dev(ss_rs_coder *coder, const uint8_t *data, uint64_t data_stride,
                             uint32_t data_len, uint64_t n, uint8_t *parity,
                             uint64_t plane_stride, uint64_t shard_stride, uint32_t flags);

/* Batched reconstruct (rscoding.rs:490-537 over n codewords; callers rspaxos/durability.rs:146-159,
 * crossword/durability.rs:163-179).  Shard j of codeword g lives at
 * shards[j*plane_stride + off[g] .. +L_g), L_g = ceil(data_len[g]/d).  present[g] bit j =
 * shard j available.  Missing DATA shards are regenerated in place (and missing parity too when
 * data_only == 0).  status[g] = 0, SS_ERR_TOO_FEW_SHARDS_PRESENT (nothing written for g), or
 * SS_ERR_INVALID_ARG for a null codeword (data_len == 0; rscoding.rs:495-497). */
int ss_rs_reconstruct_batch_dev(ss_rs_coder *coder, uint8_t *shards, uint64_t plane_stride,
                                const uint64_t *off, const uint32_t *data_len,
                                const uint32_t *present, uint64_t n, int data_only,
                                int32_t *status, uint32_t flags);

/* uniform geometry: every codeword has data_len bytes and its shard j sits at shards + j*plane_stride + g*shard_stride
 * (16-byte aligned slots of capacity round_up(L,16), the layout ss_rs_encode_uniform_dev writes with
 * SS_RS_OUT_PADDED16; regenerated shards get zero padding).  For RS(3,2) -- every 5-replica deployment -- this runs
 * the pattern-specialised row kernel (compile-time decode rows per present mask); other codes go through the kernels of
 * the ragged call.  status as above. */
int ss_rs_reconstruct_uniform_dev(ss_rs_coder *coder, uint8_t *shards, uint64_t plane_stride, uint64_t shard_stride,
                                  uint32_t data_len, const uint32_t *present, uint64_t n, int data_only,
                                  int32_t *status);

/* host-buffer forms of the two batch calls (H2D, kernel, D2H inside; chunked + overlapped) */
int ss_rs_encode_uniform(ss_rs_coder *coder, const uint8_t *data, uint64_t data_stride,
                         uint32_t data_len, uint64_t n, uint8_t *parity, uint64_t plane_stride,
                         uint64_t shard_stride);

/* ---- quorum tallies ------------------------------------------------------------------------
 * Bit-plane form.  planes[r*G + g] bit s = a VALID AcceptReply from replica r for slot s of
 * group g (the leader's own WAL ack is one of the planes, multipaxos/durability.rs:99-103).
 * committed[g] bit s = (count of set planes >= threshold) -- the end state of
 * handle_msg_accept_reply on that ack set (multipaxos/messages.rs:404-413 with
 * threshold = quorum_cnt; rspaxos/messages.rs:438-440 with majority + fault_tolerance).
 * commit_bar[g] (may be NULL) = length of the committed prefix of the 64-slot window
 * (multipaxos/durability.rs:161-170).  R <= 16. */
int ss_tally_planes_dev(ss_ctx *ctx, const uint64_t *planes, uint32_t n_replicas, uint64_t n_groups,
                        uint32_t threshold, uint64_t *committed, uint32_t *commit_bar);
int ss_tally_planes(ss_ctx *ctx, const uint64_t *planes, uint32_t n_replicas, uint64_t n_groups,
                    uint32_t threshold, uint64_t *committed, uint32_t *commit_bar);

/* Per-instance vote-mask form: masks[i] = the instance's accept_acks Bitmap (bit r = replica r,
 * src/utils/bitmap.rs:17; LeaderBookkeeping.accept_acks, multipaxos/mod.rs:181-197), one
 * mask_bytes-wide (1 or 2) little-endian integer per instance.  commit_bits word i/64 bit i%64 =
 * Bitmap::count() >= threshold (bitmap.rs:111-113). */
int ss_tally_masks_dev(ss_ctx *ctx, const void *masks, uint32_t mask_bytes, uint64_t n_instances,
                       uint32_t threshold, uint64_t *commit_bits);

/* Ack ingest: applies the filters of handle_msg_accept_reply to a record stream and ORs the
 * surviving acks into the planes (multipaxos/messages.rs:388 ballot == bal_prepared;
 * :394-399 status == Accepting && ballot >= inst.bal; :404-406 duplicates are idempotent).
 * accepting[g] bit s = instance (g,s) is in Status::Accepting; inst_bal[g*64+s] its ballot.
 * Records with peer >= n_replicas or slot >= 64 are dropped (Bitmap::get -> Err, bitmap.rs:89-97). */
int ss_ack_ingest_dev(ss_ctx *ctx, const uint32_t *rec_group, const uint8_t *rec_slot,
                      const uint8_t *rec_peer, const uint64_t *rec_ballot, uint64_t n_records,
                      const uint64_t *bal_prepared, const uint64_t *inst_bal,
                      const uint64_t *accepting, uint32_t n_replicas, uint64_t n_groups,
                      uint64_t *planes);

/* Crossword commit predicate (crossword/messages.rs:15-62 coverage_under_faults, :535-542).
 * policies[k*n_replicas + r] = shard bitmask (over T = total_shards ids) replica r holds under
 * assignment policy k (Instance.assignment, crossword/mod.rs:260; balanced round-robin policies
 * crossword/mod.rs:866-888, or the single init_assignment when unbalanced, adaptive.rs:129-131).
 * policy_idx[i] selects instance i's policy; masks[i] = which replicas acked.
 * balanced != 0 uses the reference's closed form (:28-33), else the subset enumeration (:35-61).
 * commit iff #acks >= majority && coverage >= data_shards.  n_replicas <= 12, n_policies <= 16. */
int ss_tally_crossword_dev(ss_ctx *ctx, const void *masks, uint32_t mask_bytes,
                           const uint8_t *policy_idx, uint64_t n_instances,
                           const uint32_t *policies_host, uint32_t n_policies, uint32_t n_replicas,
                           uint32_t total_shards, uint32_t data_shards, uint32_t majority,
                           uint32_t fault_tolerance, int balanced, uint64_t *commit_bits);

/* Raft / CRaft match-index commit scan (raft/messages.rs:256-275; craft/messages.rs:288-314).
 * match[p*G + g] for the n_peers = population-1 peers (self excluded, raft/mod.rs:560-562);
 * entries last_commit+1 .. log_end-1 of group g have terms terms[g*window + (slot-last_commit-1)]
 * (log_end - last_commit - 1 <= window).  new_commit[g] = the LAST slot in that range with
 * term == curr_term and 1 + #{p: match[p] >= slot} >= threshold, else last_commit[g].
 * threshold = quorum_cnt (Raft), majority+f or majority (CRaft full-copy).
 * window_overflow (device u32, may be NULL): incremented once per group whose candidate range exceeds `window`
 * entries (precondition violated); for such a group new_commit is a lower bound of the reference's result (candidates
 * beyond the window cannot be examined) and the host should rescan it with a larger window. */
int ss_raft_commit_scan_dev(ss_ctx *ctx, const uint32_t *match, uint32_t n_peers, uint64_t n_groups,
                            const uint32_t *last_commit, const uint32_t *log_end,
                            const uint32_t *curr_term, const uint32_t *terms, uint32_t window,
                            uint32_t threshold, uint32_t *new_commit, uint32_t *window_overflow);

/* k-th largest peer match per group.  k = threshold - 1 gives CRaft's shadow_last_commit
 * (craft/messages.rs:677-690: match slots sorted descending, element [threshold-2], threshold =
 * majority + fault_tolerance, or majority in full-copy mode); k = n_peers gives the bound of Raft's
 * last_snap scan (raft/messages.rs:298-309: every server has the entry). */
int ss_raft_kth_match_dev(ss_ctx *ctx, const uint32_t *match, uint32_t n_peers, uint64_t n_groups, uint32_t k,
                          uint32_t *out);

/* Prepare-phase shard merge + decision for n_instances recovering instances (leader fail-over;
 * rspaxos/messages.rs:182-259, crossword/messages.rs:233-312).  vote_bal[r*N+i] / vote_mask[r*N+i] = the
 * (ballot, shards carried) of replica r's PrepareReply vote for instance i; vote_mask == 0 means "no vote".
 * merged[i] = shard set inst.reqs_cw ends with (shards voted at the highest ballot; max_bal[i] that ballot;
 * order-independent because absorb_other only adds).  action[i]: bit0 USE (>= data_shards shards), bit1 NULL
 * request batch (fewer, but acks_cnt[i] >= population - fault_tolerance), 0 = not yet; bit2 reconstruct_data
 * needed; bit3 compute_parity needed (avail shards < POPULATION, as the reference compares).  The regeneration
 * itself is ss_rs_reconstruct_batch_dev(present = merged, data_only = 0). */
#define SS_PM_USE 1u
#define SS_PM_NULL 2u
#define SS_PM_RECONSTRUCT 4u
#define SS_PM_PARITY 8u
int ss_prepare_merge_dev(ss_ctx *ctx, const uint64_t *vote_bal, const uint32_t *vote_mask, uint32_t n_replicas,
                         uint64_t n_instances, const uint8_t *acks_cnt, uint32_t data_shards, uint32_t population,
                         uint32_t fault_tolerance, uint64_t *max_bal, uint32_t *merged, uint8_t *action);

/* ---- fused accept step (BASELINE config 3: RSPaxos encode + quorum) -------------------------
 * ONE kernel launch that, for n_groups groups: RS-encodes each group's new request batch
 * (as ss_rs_encode_uniform_dev) and tallies the group's 64-slot ack window
 * (as ss_tally_planes_dev). */
int ss_accept_step_fused_dev(ss_rs_coder *coder, const uint8_t *data, uint64_t data_stride,
                             uint32_t data_len, uint64_t n_groups, uint8_t *parity,
                             uint64_t plane_stride, uint64_t shard_stride, uint32_t flags,
                             const uint64_t *planes, uint32_t n_replicas, uint32_t threshold,
                             uint64_t *committed, uint32_t *commit_bar);

/* ---- step flags: cross-GPU ordering without host synchronisation ---------------------------------------------
 * A flag is a u64 step counter in device memory (ss_dev_alloc + ss_dev_memset 0; exported to peers with
 * ss_ipc_export).  Calls that take an ss_step_sync
 *   - first wait (on the device, inside the kernel) until every wait_flags[i] >= wait_value -- wait_flags is a device
 *     array in LOCAL memory that peers write into;
 *   - after all of the call's stores are visible system-wide, store signal_value to every *signal_flags[i]
 *     (st.release.sys) -- signal_flags is a HOST array of device pointers into local or peer memory.
 * This replaces the per-step stream barrier + ack copies a host would otherwise need: a follower's kernel starts when
 * the leader's shards have landed, the leader's next tally starts when the followers' acks have landed
 * (rspaxos/request.rs:127-142 -> rspaxos/durability.rs:101-118 -> rspaxos/messages.rs:395-465, with NVLink stores in
 * place of TransportHub messages).  Waits are bounded (2 s): on time-out bit 0 of ss_ctx_device_status is set and the
 * kernel proceeds.  n_wait, n_signal <= 32; either part may be empty; a NULL ss_step_sync means no ordering. */
typedef struct ss_step_sync {
    const uint64_t *wait_flags;
    uint32_t n_wait;
    uint64_t wait_value;
    uint64_t *const *signal_flags;
    uint32_t n_signal;
    uint64_t signal_value;
} ss_step_sync;
/* the two halves of an ss_step_sync as stand-alone stream operations (one-warp kernels on the context's stream) */
int ss_flags_wait_dev(ss_ctx *ctx, const ss_step_sync *sync);
int ss_flags_signal_dev(ss_ctx *ctx, const ss_step_sync *sync);
/* Stream-ordering between TWO contexts of one process (e.g. a compute context and a copy context whose
 * ss_copy_d2d pushes run on the copy engines while the next step computes): an event recorded on one context's stream
 * can be waited for by another's (cudaEventRecord / cudaStreamWaitEvent). */
int ss_event_create(ss_ctx *ctx, void **event);
int ss_event_destroy(ss_ctx *ctx, void *event);
int ss_event_record(ss_ctx *ctx, void *event);
int ss_event_wait(ss_ctx *ctx, void *event);
/* reads (and clears) the context's device status word; synchronises the context's stream */
#define SS_DEV_STATUS_FLAG_TIMEOUT 1u
#define SS_DEV_STATUS_FRAME_OVERFLOW 4u   /* ss_frame_accept_pack_dev: a frame did not fit frame_stride */
int ss_ctx_device_status(ss_ctx *ctx, uint32_t *status);

/* Fused encode + tally + REPLICATE (the multi-GPU accept step): as ss_accept_step_fused_dev, but shard j of the
 * local groups (data shards included) is written to shard_planes[j] + g*shard_stride, where each shard_planes[j]
 * is a device pointer into LOCAL memory or into a PEER GPU's memory (ss_ipc_open): the encode kernel itself
 * delivers every replica's shard over NVLink -- no pack pass, no separate collective.  shard_planes is a HOST
 * array of d+p pointers; every target slot is 16-byte aligned with capacity round_up(L,16).  Any code with d <= 8
 * data shards (every Summerset cluster code; others are specialised at run time), 16-byte-aligned uniform payloads of
 * any length (SS_ERR_UNSUPPORTED otherwise).  sync (may be NULL): the tally waits for
 * sync->wait_flags (the followers' ack flags) and the followers are signalled when every shard has landed. */
int ss_accept_step_replicate_dev(ss_rs_coder *coder, const uint8_t *data, uint64_t data_stride, uint32_t data_len,
                                 uint64_t n_groups, uint8_t *const *shard_planes, uint64_t shard_stride,
                                 const uint64_t *planes, uint32_t n_replicas, uint32_t threshold,
                                 uint64_t *committed, uint32_t *commit_bar, const ss_step_sync *sync);

/* Host-buffer form of the fused accept step (the call a host without device-resident state makes): payloads, ack
 * planes, parity planes, commit words and commit_bar are HOST arrays with the layouts of ss_accept_step_fused_dev;
 * chunks of groups are uploaded, run through the ONE fused kernel and downloaded with copy and compute overlapped
 * (three staging buffers on separate copy streams).  Returns when every result is in host memory.  Pinned host
 * buffers (ss_host_alloc) are needed for the overlap. */
int ss_accept_step_fused(ss_rs_coder *coder, const uint8_t *data, uint64_t data_stride, uint32_t data_len,
                         uint64_t n_groups, uint8_t *parity, uint64_t plane_stride, uint64_t shard_stride,
                         const uint64_t *planes, uint32_t n_replicas, uint32_t threshold, uint64_t *committed,
                         uint32_t *commit_bar);

/* The simulated followers' side of the step (rspaxos/durability.rs:101-118: log the Accept, reply): once the leaders'
 * shards have landed (sync->wait_flags), ack plane r -- ack_src[r*n_groups .. +n_groups), this GPU's followers' ack
 * bits for the groups they follow -- is stored to ack_dst[r] (n_groups words in the leader GPU's memory, local or
 * peer; a NULL entry is skipped), then the leaders are signalled.  ack_dst is a HOST array of n_replicas pointers. */
int ss_follower_ack_dev(ss_ctx *ctx, const uint64_t *ack_src, uint64_t *const *ack_dst, uint32_t n_replicas,
                        uint64_t n_groups, const ss_step_sync *sync);

/* Crossword encode + distribute (BASELINE config 4; crossword/request.rs:82-87,137-185): RS-encodes a ragged batch with
 * the coder's (d, T-d) code and writes, for every codeword g, the spr[g] shards the balanced round-robin assignment gives
 * replica r -- shards {(r*dj + k) mod T : k < spr[g]}, dj = T / n_replicas (crossword/mod.rs:866-888) -- into
 * replica_logs[r] at rep_off[g] + k*SS_CW_SLOT_PITCH(L_g), k = 0..spr-1 (bytes past L_g zero; the pitch is L_g rounded up
 * to 32 bytes so that every slot of a log built from 32-byte aligned offsets starts on a DRAM sector: with a 16-byte
 * pitch the same kernel is 7 % slower, profiles/r02_distribute_variants.txt).  replica_logs is a HOST array
 * of n_replicas device pointers, local or peer (ss_ipc_open): the kernel's stores are the shard transfer.  Per codeword
 * (n-1)*spr*L_g bytes cross to other replicas, as in the reference.  Any code with d <= 8 and T a multiple of
 * n_replicas <= 16 (crossword/mod.rs:805-830); n = 5 with RS(3,2) runs the hand-specialised kernel. */
#define SS_CW_SLOT_PITCH(L) ((((uint64_t)(L)) + 31u) & ~(uint64_t)31u)
int ss_crossword_distribute_dev(ss_rs_coder *coder, const uint8_t *data, const uint64_t *data_off,
                                const uint32_t *data_len, const uint8_t *spr, const uint64_t *rep_off,
                                uint64_t n, uint8_t *const *replica_logs, uint32_t n_replicas);

/* Accept-frame packer (the step after the path, SURVEY 8f-2): for n uniform codewords, builds the byte frames an
 * unmodified Summerset peer reads off its TCP connection -- 8-byte big-endian body length (utils/safetcp.rs:30-88)
 * + bincode(PeerMessage::Msg { msg: PeerMsg::Accept { slot, ballot, reqs_cw } }) (server/transport.rs:37-40,
 * rspaxos/mod.rs:283-288) where reqs_cw = the codeword holding only shard `shard_idx` (what subset_copy builds for
 * that peer, rspaxos/request.rs:127-142), encoded per utils/rscoding.rs:54-71 with data_copy = None.
 * shard_plane: shard `shard_idx` of codeword g at shard_plane + g*shard_stride.  Frame g is written inside
 * out[g*frame_stride .. (g+1)*frame_stride) at frame_off[g] (so that the shard bytes are 16-byte aligned) and is
 * frame_len[g] bytes long.  frame_stride: multiple of 16, >= shard_len + 96 + d + p.  msg_variant = the index of
 * the Accept variant in the protocol's PeerMsg enum (2 for RSPaxos).  This is the single-shard fast path (the shard
 * is copied with aligned 128-bit accesses on both sides); ss_frame_accept_pack_dev is the general packer.  bincode
 * layout from knowledge of the crate: unpinned against the reference (it cannot run here); tested byte for byte against
 * the oracle's independent C encoder (oracle/ss_wire.c). */
int ss_frame_accept_batch_dev(ss_ctx *ctx, const uint8_t *shard_plane, uint64_t shard_stride, uint32_t shard_idx,
                              uint32_t data_shards, uint32_t parity_shards, uint32_t data_len, uint32_t msg_variant,
                              const uint64_t *slot, const uint64_t *ballot, uint64_t n, uint8_t *out,
                              uint64_t frame_stride, uint64_t *frame_off, uint32_t *frame_len);

/* ---- wire / WAL formats on the device (SURVEY 8f-2) -------------------------------------------------------------
 * General Accept packer: for n codewords and ONE destination, builds either the frames an unmodified Summerset peer
 * reads off its TCP connection -- 8-byte big-endian body length (utils/safetcp.rs:30-88) + bincode(PeerMessage::Msg {
 * msg: PeerMsg::Accept { slot, ballot, reqs_cw [, assignment] } }) (server/transport.rs:37-40, rspaxos/mod.rs:283-288,
 * crossword/mod.rs:356-362) -- or the records StorageHub appends -- 8-byte big-endian length (server/storage.rs:333-337)
 * + bincode(WalEntry::AcceptData { slot, ballot, reqs_cw }) (rspaxos/mod.rs:219-228).  reqs_cw carries exactly the shards
 * policies[policy_idx[g]][peer] names (what subset_copy(.., false) builds for that peer: one shard in RSPaxos,
 * rspaxos/request.rs:127-142; spr shards in Crossword, crossword/request.rs:164-185), data_copy None, encoded per
 * utils/rscoding.rs:43-72; with_assignment appends assignment: Vec<Bitmap> = that policy row (utils/bitmap.rs:20-30).
 * policies: DEVICE array [n_policies][population] of shard bitmasks; policy_idx: device [n] or NULL (policy 0).
 * Frame g is written inside out[g*frame_stride ..) at frame_off[g] (placed so that its first shard's bytes are 16-byte
 * aligned) and is frame_len[g] bytes long; frame_stride >= ss_frame_accept_max_len(spec, max shards per frame) -- a
 * frame that would not fit its slot is not written: frame_len[g] = 0 and bit 2 of ss_ctx_device_status is set.
 * bincode layout from knowledge of the crate: unpinned against the reference; tested byte for byte against the oracle's
 * independent C encoder (oracle/ss_wire.c), and decode(encode(x)) == x. */
#define SS_FRAME_PEER_ACCEPT 0u
#define SS_FRAME_WAL_ACCEPT_DATA 1u
typedef struct ss_frame_spec {
    uint32_t kind;             /* SS_FRAME_PEER_ACCEPT / SS_FRAME_WAL_ACCEPT_DATA */
    uint32_t msg_variant;      /* index of Accept in the protocol's PeerMsg enum (2), or of AcceptData in WalEntry (1) */
    uint32_t data_shards, parity_shards, data_len;
    uint32_t population;       /* replicas (columns of the policy table) */
    uint32_t with_assignment;  /* Crossword Accept: append assignment: Vec<Bitmap> */
    uint32_t assign_size;      /* bit length of each assignment Bitmap (= rs_total_shards) */
} ss_frame_spec;
uint64_t ss_frame_accept_max_len(const ss_frame_spec *spec, uint32_t max_shards_per_frame);
int ss_frame_accept_pack_dev(ss_ctx *ctx, const ss_frame_spec *spec, const uint8_t *shard_planes, uint64_t plane_stride,
                             uint64_t shard_stride, const uint32_t *policies, uint32_t n_policies,
                             const uint8_t *policy_idx, uint32_t peer, const uint64_t *slot, const uint64_t *ballot,
                             uint64_t n, uint8_t *out, uint64_t frame_stride, uint64_t *frame_off, uint32_t *frame_len);

/* AcceptReply frames -> ack records.  buf holds frames as read off the peers' connections (8-byte big-endian length +
 * body each); frame i starts at frame_off[i], came from replica frame_peer[i] of group frame_group[i].  A well-formed
 * PeerMessage::Msg{PeerMsg::AcceptReply{slot, ballot}} (rspaxos/mod.rs:290-291; with_size: crossword's
 * {slot, ballot, size, reply_ts}, crossword/mod.rs:365-373) yields rec_kind[i] = reply_variant and the record
 * (group, slot - window_base[group], peer, ballot) in the layout ss_ack_ingest_dev / ss_engine_ingest take; slots below
 * the group's window base (`slot < start_slot`, messages.rs:377) or beyond the 64-slot window get rec_slot = 0xff, which
 * the ingest kernel drops.  Other messages: rec_kind = their PeerMsg variant index (0x80000000 | k for the
 * PeerMessage variants LeaseMsg / Leave / LeaveReply) -- the host handles them; malformed: SS_FRAME_KIND_MALFORMED. */
#define SS_FRAME_KIND_MALFORMED 0xffffffffu
int ss_accept_reply_parse_dev(ss_ctx *ctx, const uint8_t *buf, uint64_t buf_len, const uint64_t *frame_off,
                              const uint32_t *frame_group, const uint8_t *frame_peer, const uint64_t *window_base,
                              uint64_t n_frames, uint64_t n_groups, uint32_t reply_variant, int with_size,
                              uint32_t *rec_group, uint8_t *rec_slot, uint8_t *rec_peer, uint64_t *rec_ballot,
                              uint32_t *rec_kind);

/* WalEntry::CommitSlot { slot } records (rspaxos/mod.rs:231; commit_variant = 2) for every instance that committed in a
 * tick: newly[g] bit s (ss_engine_tick's output) -> one 24-byte cell in `entries` holding the 8-byte big-endian length
 * + bincode record of absolute slot window_base[g] + s, with entry_group / entry_len beside it.  *n_entries (device u64)
 * = number of records; cells beyond `capacity` are counted but not written.  Cell order is unspecified (every group
 * has its own WAL; the host routes by entry_group). */
int ss_wal_commit_pack_dev(ss_ctx *ctx, const uint64_t *newly, const uint64_t *window_base, uint64_t n_groups,
                           uint32_t commit_variant, uint8_t *entries, uint32_t *entry_group, uint32_t *entry_len,
                           uint64_t capacity, uint64_t *n_entries);

/* Reconstruct serving (SURVEY 8f-4; crossword/messages.rs:577-632, rspaxos/messages.rs:468-517) for n_requests
 * (slot, exclude) pairs of a Reconstruct message: request i concerns the instance of group req_group[i] whose shards sit
 * in shard_planes (shard j at shard_planes + j*plane_stride + req_group[i]*shard_stride), of which this replica holds
 * req_held[i]; req_status[i] is the instance's Status (>= 2 = Accepting).  reply_mask[i] = held & flip(exclude) -- 0 when
 * the status is below Accepting or nothing is left, in which case the slot gets no entry in the reply -- and the
 * selected shards are copied in index order, each in a round_up(shard_len,16)-byte slot, to out + reply_off[i]
 * (16-byte aligned offsets). */
int ss_reconstruct_serve_dev(ss_ctx *ctx, const uint8_t *shard_planes, uint64_t plane_stride, uint64_t shard_stride,
                             uint32_t total_shards, uint32_t shard_len, const uint32_t *req_group,
                             const uint32_t *req_held, const uint32_t *req_excl, const uint8_t *req_status,
                             const uint64_t *reply_off, uint64_t n_requests, uint32_t *reply_mask, uint8_t *out);

/* Reconstruct replies, receiving side (SURVEY 8f-4; handle_msg_reconstruct_reply, crossword/messages.rs:634-722,
 * rspaxos/messages.rs:519-594), batched over a follower's window of instances.  Instance row r = g*window + s (group g,
 * window slot s, window <= 64); its shard j sits at shard_planes + j*plane_stride + r*shard_stride in 16-byte aligned
 * slots of capacity round_up(L,16), L = ceil(data_len/d) -- the geometry of ss_rs_reconstruct_uniform_dev.
 * inst_status[r]: Status in declaration order (0 Null .. 2 Accepting, 3 Committed, 4 Executed); inst_bal[r]: Instance.bal;
 * present[r] (in/out): bit j = shard j held (avail_shards_map); exec_bar[g] (in/out): the handler's commit_bar, relative
 * to the window.  Reply i has the layout ss_reconstruct_serve_dev writes: the shards of reply_mask[i] in index order, one
 * round_up(L,16)-byte slot each, at reply_buf + reply_off[i] (16-byte aligned offsets), so serve's output on one GPU,
 * copied or read over NVLink, is this call's input on another.  reply_inst[i] = row of the instance, 0xffffffff (or any
 * row >= n_groups*window) for a slot below start_slot or outside the window: skipped (crossword/messages.rs:641-643);
 * reply_ballot[i] = the replier's ballot.  Three kernels on the context's stream:
 *   absorb  reply i is taken when inst_status < Executed && reply_ballot >= inst_bal (crossword/messages.rs:667,
 *           rspaxos/messages.rs:542; as in the release build, Accepting instances are absorbed too).  absorb_other
 *           (rscoding.rs:296-345) fills empty slots only: every shard missing from present is claimed by exactly one reply
 *           (atomicOr on present[r]) and its whole padded slot is copied; taken[i] (may be NULL) = the bits reply i won.
 *           A mask with bits >= d+p is malformed network input: the reply is dropped whole (taken 0).
 *   walk    per group from exec_bar[g]: advance while s < window, status >= Committed and popcount(present) >= d
 *           (crossword/messages.rs:670-688, rspaxos/messages.rs:545-560).  submit[g] bit s = instance s passed (written for
 *           every group); passed instances with fewer than d data shards are marked for decode and their present gains the
 *           data bits.
 *   decode  reconstruct_data of the marked rows (ss_rs_reconstruct_uniform_dev's kernels; RS(3,2) gets its row kernel).
 * Not done here: setting Executed (the reference does it only for an empty ReqBatch, which takes the payload -- a host
 * decision) and bincode ReconstructReply frames.
 * Batched vs per-message: the reference walks only when a reply lands exactly on commit_bar, decoding at that moment;
 * this call absorbs the whole batch, walks once, then decodes.  The end states (present, exec_bar, submit, data bytes)
 * are the same when (1) on entry the instance at each bar is not ready (not both Committed and holding >= d shards) --
 * the walk leaves every bar in that state, so it holds from call to call -- and (2) every reply for a slot at a ballot
 * >= inst.bal carries shards of the same codeword, which Paxos safety gives for committed instances.  Which of several
 * replies carrying the same missing shard wins it (taken) is unspecified.
 * Errors: SS_ERR_INVALID_ARG for null buffers, window 0 or > 64, n_groups 0, data_len 0, misaligned planes / reply_buf /
 * strides, shard_stride < round_up(L,16); SS_ERR_UNSUPPORTED when d+p > 12.  n_replies == 0: SS_OK, nothing launched and
 * no output written. */
int ss_reconstruct_reply_dev(ss_rs_coder *coder, uint8_t *shard_planes, uint64_t plane_stride, uint64_t shard_stride,
                             uint32_t data_len, uint64_t n_groups, uint32_t window, const uint8_t *inst_status,
                             const uint64_t *inst_bal, uint32_t *present, uint32_t *exec_bar, const uint8_t *reply_buf,
                             const uint64_t *reply_off, const uint32_t *reply_mask, const uint32_t *reply_inst,
                             const uint64_t *reply_ballot, uint64_t n_replies, uint64_t *submit, uint32_t *taken);

/* Crossword follower gossip planning (SURVEY 8f-4; crossword/gossiping.rs:35-84 gossip_targets_excl) for
 * n_instances committed-but-incomplete instances of replica `me`: walking peers me+1, me+2, ... (mod population) and
 * skipping the instance's source peer (src_peer[i]) and peers absent from `peer_alive`, a peer is selected when its
 * assigned shards (policies[policy_idx[i]][peer], as in ss_tally_crossword_dev) include one not yet held/asked for;
 * excl[peer*N + i] = the availability map at that moment (what the Reconstruct message tells the peer to leave out,
 * crossword/messages.rs:577-632); the walk stops once data_shards shards are covered.  targets[i] = selected peers.
 * excl entries of unselected peers are left untouched. */
int ss_gossip_plan_dev(ss_ctx *ctx, uint32_t me, uint32_t population, uint32_t data_shards, const uint8_t *src_peer,
                       const uint32_t *avail, const uint8_t *policy_idx, const uint32_t *policies_host,
                       uint32_t n_policies, uint32_t peer_alive, uint64_t n_instances, uint32_t *targets, uint32_t *excl);

/* ---- batched multi-group consensus engine ----------------------------------------------------------------------
 * The leader-side state of n_groups independent replica groups (64-slot instance window each) lives in HBM as a
 * struct of arrays; the host drives all groups together, once per event-loop turn:
 *   ss_engine_propose   one new instance per group at window position `slot`: RS-encode the request batches into the
 *                       shard planes (per-peer packed send buffers) and enter Status::Accepting under the group's
 *                       prepared ballot with an empty ack set   (multipaxos/request.rs:112-221,
 *                       rspaxos/request.rs:72-142, crossword/request.rs:82-185)
 *   ss_engine_ingest    a batch of AcceptReply records through handle_msg_accept_reply's filters
 *                       (multipaxos/messages.rs:377-409, rspaxos/messages.rs:402-437, crossword/messages.rs:489-530)
 *   ss_engine_tick      ONE kernel: commit decision of every Accepting instance (MultiPaxos quorum_cnt,
 *                       multipaxos/messages.rs:412-413; RSPaxos majority + fault_tolerance, rspaxos/messages.rs:438-440;
 *                       Crossword #acks >= majority && coverage_under_faults >= d, crossword/messages.rs:535-542),
 *                       committed |= newly, accepting &= ~newly, commit_bar = committed prefix
 *                       (multipaxos/durability.rs:161-170)
 * Raft / CRaft engines keep match_slot / next_slot / log terms instead: ss_engine_raft_append (the leader appends
 * entries in its term), ss_engine_raft_ingest (successful AppendEntriesReply, raft/messages.rs:243-252) and
 * ss_engine_tick (commit scan raft/messages.rs:254-275,295 with quorum_cnt -- CRaft: majority + fault_tolerance,
 * craft/messages.rs:300-308 -- and last_snap, raft/messages.rs:298-309).  Conflict replies, elections, heartbeats,
 * durability and execution stay in the host's event loop (out of scope, SURVEY.md 2b).
 * All array arguments are DEVICE pointers; calls are asynchronous on the context's stream. */
typedef struct ss_engine ss_engine;
#define SS_PROTO_MULTIPAXOS 0u
#define SS_PROTO_RSPAXOS 1u
#define SS_PROTO_CROSSWORD 2u
#define SS_PROTO_RAFT 3u
#define SS_PROTO_CRAFT 4u
typedef struct ss_engine_config {
    uint32_t protocol;          /* SS_PROTO_* */
    uint32_t population;        /* n <= 12 */
    uint32_t fault_tolerance;   /* f <= n - majority (rspaxos/mod.rs:599-605); ignored by MultiPaxos / Raft */
    uint32_t data_len;          /* bytes of every request batch (RS-coded protocols) */
    uint32_t rs_total_shards;   /* Crossword: T (0 = n; must be a multiple of n, crossword/mod.rs:805-830) */
    uint32_t rs_data_shards;    /* Crossword: d (0 = majority) */
    uint32_t keep_slots;        /* depth of the shard store: proposals of slot s live in store s % keep_slots (0 = 1) */
    uint32_t raft_window;       /* Raft: uncommitted-tail capacity per group, power of two (0 = 64) */
} ss_engine_config;
/* device pointers into the engine's state (valid until ss_engine_destroy), for hosts that read results in place or
 * install state (recovery, tests).  Arrays a protocol does not use are NULL. */
typedef struct ss_engine_view {
    uint64_t n_groups;
    uint32_t population, threshold, data_shards, total_shards, shard_len, shard_stride, raft_window, pad0;
    uint64_t plane_stride;      /* bytes between shard planes of one proposal */
    uint64_t slot_stride;       /* bytes between the shard stores of consecutive keep slots */
    uint64_t *planes;           /* [n][G]  valid-ack bit-planes */
    uint64_t *bal_prepared;     /* [G] */
    uint64_t *inst_bal;         /* [G*64] */
    uint64_t *accepting;        /* [G]  bit s = Status::Accepting */
    uint64_t *committed;        /* [G]  bit s = Status::Committed */
    uint32_t *commit_bar;       /* [G] */
    uint8_t *shards;            /* [keep][T][G][shard_stride] */
    uint8_t *policy_idx;        /* Crossword [G*64]: assignment policy of each instance */
    uint32_t *match, *next_slot;/* Raft [n-1][G] */
    uint32_t *last_commit, *log_end, *curr_term, *last_snap;   /* Raft [G] */
    uint32_t *terms;            /* Raft [G][raft_window]: term of slot s at index s & (raft_window-1) */
} ss_engine_view;
int ss_engine_create(ss_ctx *ctx, const ss_engine_config *cfg, uint64_t n_groups, ss_engine **out);
int ss_engine_destroy(ss_engine *engine);
int ss_engine_view_get(ss_engine *engine, ss_engine_view *view);
/* bal_prepared of every group (become_a_leader ... handle_msg_prepare_reply, outside this path) */
int ss_engine_set_prepared_ballots(ss_engine *engine, const uint64_t *ballots);
/* Crossword: the assignment policies instances may use (policies_host[k*n + r] = shard bitmask of replica r, as
 * ss_tally_crossword_dev) and whether the balanced closed form applies (crossword/mod.rs:849-850) */
int ss_engine_set_policies(ss_engine *engine, const uint32_t *policies_host, uint32_t n_policies, int balanced);
/* payloads: request batch of group g at payloads + g*payload_stride (data_len bytes; NULL for MultiPaxos).  policy:
 * Crossword only, [G] policy index of the new instance (NULL = 0).  *shard_planes (may be NULL) receives the base of
 * this proposal's T shard planes: shard j of group g at base + j*plane_stride + g*shard_stride. */
int ss_engine_propose(ss_engine *engine, uint32_t slot, const uint8_t *payloads, uint64_t payload_stride,
                      const uint8_t *policy, uint8_t **shard_planes);
int ss_engine_ingest(ss_engine *engine, const uint32_t *rec_group, const uint8_t *rec_slot, const uint8_t *rec_peer,
                     const uint64_t *rec_ballot, uint64_t n_records);
/* newly (may be NULL): [G] bit s = instance s committed in THIS tick (what the host logs as WalEntry::CommitSlot) */
int ss_engine_tick(ss_engine *engine, uint64_t *newly);
/* Raft: n_new[g] entries appended by the leader in curr_term[g]; exceeding raft_window uncommitted entries sets bit 1
 * of ss_ctx_device_status and leaves that group unchanged */
#define SS_DEV_STATUS_RAFT_WINDOW_FULL 2u
int ss_engine_raft_append(ss_engine *engine, const uint32_t *n_new);
int ss_engine_raft_ingest(ss_engine *engine, const uint32_t *rec_group, const uint8_t *rec_peer,
                          const uint32_t *rec_end_slot, uint64_t n_records);

/* ---- tuning / introspection (bench + tests) ------------------------------------------------ */
/* Tuning knob for experiments (profiles/r01_row_kernel_sweep.txt); 0 = the measured-best defaults.
 *   bits 0-3  kernel choice / register budget: 1 = flat one-column-per-thread RS(3,2) kernel instead of the row kernel,
 *             5 = bit-plane generic kernels instead of the Horner ones, 8 = global-table Horner reconstruct instead of the
 *             shared-memory small-code kernel; 3 / 6 / 7 = 32 / 64 / 56-register builds of the row kernel (default 40)
 *   bit 4     row kernel: contiguous chunk of codewords per CTA instead of grid-stride
 *   bits 5-7  row kernel waves of CTAs per resident set: {64 (default), 1, 32, 4, 16, 256, 128, 8}
 *   bits 8-9  cache operator of the plane stores in replicate mode: .cs (default), write-back, .cg, .wt
 *   bit 10    row kernel: fixed instead of rotating warp -> column-block assignment
 *   ss_crossword_distribute_dev, bits 0-3: 6 / 7 = a warp takes runs of 8 / 4 codewords from a shared counter and pools the
 *             short ones into shared passes (3.3x on batches of sub-KB payloads, 1-2 % behind on mixed sizes), 4 = the
 *             general (any code) kernel also for RS(3,2) / n = 5
 *   d <= 8 codes other than RS(3,2) (horner_encode_row_kernel / horner_encode_packed_kernel):
 *   bits 0-3  1 = flat kernel; 2 / 3 / 4 = 48 / 64 / 80-register builds of the row layout (default by width)
 *   bit 11    run-time coefficient masks even when the matrix is one of the compile-time cluster codes
 *   bit 13    never / bit 14 always use the packed layout (m codewords side by side per CTA, tail columns apart)
 *   bit 15    software-pipelined packed loop also for shards that are not 16-byte aligned
 *   bit 16    small-code reconstruct kernel: two columns per lane and pass (80 registers) instead of one (64)
 *   bit 17    no run-time specialisation: codes without a compile-time table use the run-time-mask kernels */
int ss_rs_set_variant(ss_rs_coder *coder, int variant);
/* Codes without a compile-time table (anything but the cluster codes RS(2,1) RS(3,1) RS(3,2) RS(4,2) RS(4,3) RS(5,4)) with
 * d <= 8 get their row / packed encode kernels specialised at run time by NVRTC for the coder's own parity rows (once
 * per coder, on the first batched encode).  ss_rs_jit_status tells what happened; if libnvrtc is unavailable the coder
 * keeps the run-time-mask kernels.  ss_jit_selftest compiles the kernels for RS(d,p) without a GPU and returns the
 * CUBIN size (> 0) or a negative error code with the compiler log in `log`. */
const char *ss_rs_jit_status(const ss_rs_coder *coder);
long ss_jit_selftest(int data_shards, int parity_shards, char *log, size_t log_cap);
/* name of the kernel the last batch call on this coder launched (static string) */
const char *ss_rs_last_kernel(const ss_rs_coder *coder);

#ifdef __cplusplus
}
#endif
#endif /* SUMMERSET_B200_H */
