// wire_kernels.cu -- the steps either side of the hot path (SURVEY 8f-2, 8f-4), batched on the device so that what the
// kernels produce can be handed to an unmodified TransportHub / StorageHub, and what those deliver can feed the kernels:
//
//   frame_pack_kernel           PeerMessage::Msg{PeerMsg::Accept{slot, ballot, reqs_cw[, assignment]}} frames for one
//                               destination peer, or WalEntry::AcceptData{slot, ballot, reqs_cw} records -- 8-byte
//                               big-endian length (utils/safetcp.rs:30-88, server/storage.rs:333-337) + bincode body, the
//                               codeword carrying exactly the shards of the peer's assignment (subset_copy(.., false),
//                               rspaxos/request.rs:127-142, crossword/request.rs:164-185; encoding utils/rscoding.rs:43-72,
//                               assignment Vec<Bitmap> utils/bitmap.rs:20-30)
//   accept_reply_parse_kernel   AcceptReply frames -> (group, window slot, peer, ballot) records for ss_ack_ingest_dev /
//                               ss_engine_ingest (rspaxos/mod.rs:290-291, crossword/mod.rs:365-373)
//   wal_commit_pack_kernel      newly committed instances -> WalEntry::CommitSlot{slot} records (rspaxos/mod.rs:231)
//   reconstruct_serve_kernel    Reconstruct serving: reply shards = held & flip(exclude) per requested instance, packed
//                               (crossword/messages.rs:577-632, rspaxos/messages.rs:468-517)
//   reconstruct_absorb_kernel   ReconstructReply receiving: the replied shards a row lacks, claimed with atomicOr on its
//   reconstruct_walk_kernel     present mask and copied into the shard planes; then the execution-bar walk per group
//                               (crossword/messages.rs:634-722, rspaxos/messages.rs:519-594); reconstruct_data of the
//                               walked rows runs through the uniform reconstruct kernels
//
// bincode 2 standard config facts are from knowledge of the crate (unpinned against the reference, DESIGN.md section 4);
// every kernel is tested byte for byte against oracle/ss_wire.c.
#include "device_common.cuh"
#include "ss_internal.hpp"

namespace ssb {

constexpr int kWireThreads = 256;

__device__ __forceinline__ int wv_put(uint8_t *p, uint64_t v) {
    if (v < 251ull) { p[0] = static_cast<uint8_t>(v); return 1; }
    int nb; uint8_t tag;
    if (v < (1ull << 16)) { nb = 2; tag = 251; }
    else if (v < (1ull << 32)) { nb = 4; tag = 252; }
    else { nb = 8; tag = 253; }
    p[0] = tag;
    for (int i = 0; i < nb; ++i) p[1 + i] = static_cast<uint8_t>(v >> (8 * i));
    return 1 + nb;
}
__device__ __forceinline__ int wv_len(uint64_t v) { return v < 251ull ? 1 : v < (1ull << 16) ? 3 : v < (1ull << 32) ? 5 : 9; }

// returns bytes consumed (0: truncated or not a u64 varint)
__device__ __forceinline__ uint32_t wv_get(const uint8_t *p, uint64_t avail, uint64_t &v) {
    if (avail < 1) return 0;
    const uint8_t t = p[0];
    if (t < 251) { v = t; return 1; }
    const uint32_t nb = t == 251 ? 2u : t == 252 ? 4u : t == 253 ? 8u : 0u;
    if (nb == 0u || avail < 1u + nb) return 0;
    uint64_t x = 0;
    for (uint32_t i = 0; i < nb; ++i) x |= static_cast<uint64_t>(p[1 + i]) << (8 * i);
    v = x;
    return 1u + nb;
}

// warp-cooperative copy of n bytes: src 16-byte aligned (a padded shard slot), dst at any alignment
__device__ __forceinline__ void warp_copy_bytes(uint8_t *dst, const uint8_t *__restrict__ src, uint32_t n, uint32_t lane) {
    uint32_t head = (16u - (static_cast<uint32_t>(reinterpret_cast<uintptr_t>(dst)) & 15u)) & 15u;
    if (head > n) head = n;
    if (lane < head) dst[lane] = src[lane];
    const uint32_t nvec = (n - head) >> 4;
    for (uint32_t v = lane; v < nvec; v += 32u) {
        // aligned 16-byte destination vector <- the (generally misaligned) 16 source bytes that belong there
        const uint4 x = head == 0u ? dev::ldg128(src + v * 16u) : dev::load16(src + head + v * 16u, 16);
        dev::stg128_cs(dst + head + v * 16u, x);
    }
    const uint32_t done = head + nvec * 16u, rem = n - done;
    if (lane < rem) dst[done + lane] = src[done + lane];
}

struct PackArgs {
    const uint8_t *planes;          // shard j of codeword g at planes + j*plane_stride + g*shard_stride (16-byte aligned slots)
    uint64_t plane_stride, shard_stride;
    uint32_t d, p, data_len, L;
    uint32_t kind;                  // SS_FRAME_PEER_ACCEPT / SS_FRAME_WAL_ACCEPT_DATA
    uint32_t variant;
    const uint32_t *policies;       // [n_policies][population] shard bitmasks
    const uint8_t *policy_idx;      // [n] or nullptr (policy 0)
    uint32_t n_policies, population, peer;
    uint32_t with_assignment, assign_size;
    const uint64_t *slot, *ballot;
    uint64_t n;
    uint8_t *out;
    uint64_t frame_stride;
    uint64_t *frame_off;
    uint32_t *frame_len;
    uint32_t *status;               // context's device status word
};

__global__ void __launch_bounds__(kWireThreads) frame_pack_kernel(const __grid_constant__ PackArgs A) {
    const uint32_t lane = threadIdx.x & 31u;
    const uint64_t warp = (static_cast<uint64_t>(blockIdx.x) * kWireThreads + threadIdx.x) >> 5;
    const uint64_t nwarps = (static_cast<uint64_t>(gridDim.x) * kWireThreads) >> 5;
    const uint32_t T = A.d + A.p;
    for (uint64_t g = warp; g < A.n; g += nwarps) {
        uint32_t k = A.policy_idx != nullptr ? A.policy_idx[g] : 0u;
        if (k >= A.n_policies) k = 0u;
        const uint32_t *pol = A.policies + static_cast<uint64_t>(k) * A.population;
        const uint32_t mask = __ldg(pol + A.peer) & (T >= 32u ? 0xffffffffu : ((1u << T) - 1u));
        // fixed fields (every lane builds them; at most 41 bytes)
        uint8_t hdr[44];
        int h = 0;
        if (A.kind == SS_FRAME_PEER_ACCEPT) hdr[h++] = 0;                       // PeerMessage::Msg
        h += wv_put(hdr + h, A.variant);
        h += wv_put(hdr + h, __ldg(A.slot + g));
        h += wv_put(hdr + h, __ldg(A.ballot + g));
        hdr[h++] = static_cast<uint8_t>(A.d);
        hdr[h++] = static_cast<uint8_t>(A.p);
        h += wv_put(hdr + h, A.data_len);
        h += wv_put(hdr + h, A.L);
        h += wv_put(hdr + h, T);
        const uint32_t some_len = 1u + static_cast<uint32_t>(wv_len(A.L));       // Some tag + byte length
        // bytes before the first carried shard's payload decide the padding that makes that payload 16-byte aligned
        const uint32_t first = mask ? static_cast<uint32_t>(__ffs(mask) - 1) : T;
        const uint32_t pre = 8u + static_cast<uint32_t>(h) + first + (mask ? some_len : 0u);
        const uint32_t pad = (16u - (pre & 15u)) & 15u;
        // the frame must fit its slot: its length is known before a byte is written
        uint32_t asg_len = 0;
        if (A.with_assignment) {
            const uint32_t nblocks = (A.assign_size + 63u) / 64u;
            asg_len = static_cast<uint32_t>(wv_len(A.population));
            for (uint32_t r = 0; r < A.population; ++r)
                asg_len += static_cast<uint32_t>(wv_len(A.assign_size) + wv_len(nblocks) + wv_len(pol[r])) + (nblocks > 1u ? nblocks - 1u : 0u);
        }
        const uint32_t carried = static_cast<uint32_t>(__popc(mask));
        const uint64_t need = static_cast<uint64_t>(pad) + 8u + static_cast<uint32_t>(h) + (T - carried) +
                              static_cast<uint64_t>(carried) * (some_len + A.L) + 1u + asg_len;
        if (need > A.frame_stride) {
            if (lane == 0u) {
                A.frame_off[g] = g * A.frame_stride;
                A.frame_len[g] = 0;                                              // nothing written for this codeword
                atomicOr(A.status, 4u);                                          // SS_DEV_STATUS_FRAME_OVERFLOW
            }
            continue;
        }
        uint8_t *f = A.out + g * A.frame_stride + pad;
        for (uint32_t i = lane; i < static_cast<uint32_t>(h); i += 32u) f[8u + i] = hdr[i];
        uint32_t at = 8u + static_cast<uint32_t>(h);                             // running offset inside the frame
        for (uint32_t j = 0; j < T; ++j) {
            if (!((mask >> j) & 1u)) {
                if (lane == 0u) f[at] = 0;                                       // None
                at += 1u;
                continue;
            }
            if (lane == 0u) { f[at] = 1; wv_put(f + at + 1u, A.L); }             // Some(bytes): tag, length
            at += some_len;
            warp_copy_bytes(f + at, A.planes + static_cast<uint64_t>(j) * A.plane_stride + g * A.shard_stride, A.L, lane);
            at += A.L;
        }
        if (lane == 0u) f[at] = 0;                                               // data_copy: None
        at += 1u;
        if (A.with_assignment) {                                                 // assignment: Vec<Bitmap>
            uint32_t w = at;
            if (lane == 0u) {
                w += wv_put(f + w, A.population);
                const uint32_t nblocks = (A.assign_size + 63u) / 64u;
                for (uint32_t r = 0; r < A.population; ++r) {
                    w += wv_put(f + w, A.assign_size);
                    w += wv_put(f + w, nblocks);
                    for (uint32_t b = 0; b < nblocks; ++b) w += wv_put(f + w, b == 0u ? pol[r] : 0u);
                }
            }
            at = __shfl_sync(0xffffffffu, w, 0);
        }
        const uint64_t body = at - 8u;
        if (lane < 8u) f[lane] = static_cast<uint8_t>(body >> (8u * (7u - lane)));
        if (lane == 0u) {
            A.frame_off[g] = g * A.frame_stride + pad;
            A.frame_len[g] = at;
        }
    }
}

struct ParseArgs {
    const uint8_t *buf;
    uint64_t buf_len;
    const uint64_t *frame_off;
    const uint32_t *frame_group;
    const uint8_t *frame_peer;
    const uint64_t *window_base;    // [G]: absolute slot of window position 0 (start_slot of the group's in-memory log)
    uint64_t n_frames, G;
    uint32_t reply_variant, with_size;
    uint32_t *rec_group;
    uint8_t *rec_slot, *rec_peer;
    uint64_t *rec_ballot;
    uint32_t *rec_kind;
};

// one frame per thread: these frames are a dozen bytes; the work is the varint walk
__global__ void __launch_bounds__(kWireThreads) accept_reply_parse_kernel(const __grid_constant__ ParseArgs A) {
    const uint64_t stride = static_cast<uint64_t>(gridDim.x) * kWireThreads;
    for (uint64_t i = static_cast<uint64_t>(blockIdx.x) * kWireThreads + threadIdx.x; i < A.n_frames; i += stride) {
        uint32_t kind = SS_FRAME_KIND_MALFORMED;
        uint8_t wslot = 0xff;
        uint64_t ballot = 0;
        const uint32_t grp = A.frame_group[i];
        const uint64_t off = A.frame_off[i];
        do {
            if (off + 8u > A.buf_len) break;
            const uint8_t *fr = A.buf + off;
            uint64_t len = 0;
            for (int b = 0; b < 8; ++b) len = (len << 8) | fr[b];
            if (len > A.buf_len - off - 8u) break;
            const uint8_t *b = fr + 8;
            uint64_t n = 0, v = 0, slot = 0;
            uint32_t c;
            if (!(c = wv_get(b + n, len - n, v))) break;
            n += c;
            if (v != 0u) { kind = 0x80000000u | static_cast<uint32_t>(v); break; }   // LeaseMsg / Leave / LeaveReply
            if (!(c = wv_get(b + n, len - n, v))) break;
            n += c;
            if (v != A.reply_variant) { kind = static_cast<uint32_t>(v); break; }    // another PeerMsg: the host's business
            if (!(c = wv_get(b + n, len - n, slot))) break;
            n += c;
            if (!(c = wv_get(b + n, len - n, ballot))) break;
            n += c;
            if (A.with_size) {                                                        // crossword: size, reply_ts
                if (!(c = wv_get(b + n, len - n, v))) break;
                n += c;
                if (n >= len) break;
                const uint8_t tag = b[n++];
                if (tag == 1) {
                    if (!(c = wv_get(b + n, len - n, v))) break;
                    n += c;
                    if (!(c = wv_get(b + n, len - n, v))) break;
                    n += c;
                } else if (tag != 0) break;
            }
            if (n != len) break;
            kind = A.reply_variant;
            // `slot < start_slot` is ignored by the handler (messages.rs:377); beyond the window cannot be an instance
            if (grp < A.G) {
                const uint64_t base = A.window_base[grp];
                if (slot >= base && slot - base < 64u) wslot = static_cast<uint8_t>(slot - base);
            }
        } while (false);
        A.rec_group[i] = grp;
        A.rec_slot[i] = wslot;                        // 0xff: dropped by the ingest kernel (slot >= 64)
        A.rec_peer[i] = A.frame_peer[i];
        A.rec_ballot[i] = ballot;
        A.rec_kind[i] = kind;
    }
}

// newly committed instances -> CommitSlot records (24-byte cells: the record is at most 8 + 1 + 9 bytes)
__global__ void __launch_bounds__(kWireThreads)
wal_commit_pack_kernel(const uint64_t *__restrict__ newly, const uint64_t *__restrict__ window_base, uint64_t G, uint32_t variant,
                       uint8_t *__restrict__ entries, uint32_t *__restrict__ entry_group, uint32_t *__restrict__ entry_len,
                       uint64_t capacity, unsigned long long *counter) {
    const uint64_t stride = static_cast<uint64_t>(gridDim.x) * kWireThreads;
    for (uint64_t g = static_cast<uint64_t>(blockIdx.x) * kWireThreads + threadIdx.x; g < G; g += stride) {
        uint64_t w = __ldg(newly + g);
        if (w == 0ull) continue;
        const unsigned long long first = atomicAdd(counter, static_cast<unsigned long long>(__popcll(w)));
        uint64_t e = first;
        while (w) {
            const int s = __ffsll(static_cast<long long>(w)) - 1;
            w &= w - 1ull;
            if (e < capacity) {
                uint8_t *cell = entries + e * 24u;
                int n = 0;
                n += wv_put(cell + 8 + n, variant);
                n += wv_put(cell + 8 + n, window_base[g] + static_cast<uint64_t>(s));
                for (int b = 0; b < 8; ++b) cell[b] = b == 7 ? static_cast<uint8_t>(n) : 0;
                entry_group[e] = static_cast<uint32_t>(g);
                entry_len[e] = static_cast<uint32_t>(8 + n);
            }
            ++e;
        }
    }
}

struct ServeArgs {
    const uint8_t *planes;
    uint64_t plane_stride, shard_stride;
    uint32_t T, L;
    const uint32_t *req_group, *req_held, *req_excl;
    const uint8_t *req_status;
    const uint64_t *reply_off;
    uint64_t n;
    uint32_t *reply_mask;
    uint8_t *out;
};

// a warp per request: reply = held & flip(exclude) when the instance is at least Accepting; the selected shards are
// copied back to back (padded slots) at reply_off[i]
__global__ void __launch_bounds__(kWireThreads) reconstruct_serve_kernel(const __grid_constant__ ServeArgs A) {
    const uint32_t lane = threadIdx.x & 31u;
    const uint64_t warp = (static_cast<uint64_t>(blockIdx.x) * kWireThreads + threadIdx.x) >> 5;
    const uint64_t nwarps = (static_cast<uint64_t>(gridDim.x) * kWireThreads) >> 5;
    const uint32_t all = A.T >= 32u ? 0xffffffffu : ((1u << A.T) - 1u);
    const uint32_t vpc = (A.L + 15u) >> 4;
    for (uint64_t i = warp; i < A.n; i += nwarps) {
        uint32_t m = 0;
        if (A.req_status[i] >= 2u)                                       // Status::Accepting (messages.rs:606-608)
            m = __ldg(A.req_held + i) & ~__ldg(A.req_excl + i) & all;    // subset.flip(); subset_copy(&subset, false)
        if (lane == 0u) A.reply_mask[i] = m;                             // 0: no entry in the reply (:611-613)
        if (m == 0u) continue;
        const uint64_t g = __ldg(A.req_group + i);
        uint8_t *dst = A.out + __ldg(A.reply_off + i);
        uint32_t rem = m;
        while (rem) {
            const uint32_t j = static_cast<uint32_t>(__ffs(rem) - 1);
            rem &= rem - 1u;
            const uint8_t *src = A.planes + static_cast<uint64_t>(j) * A.plane_stride + g * A.shard_stride;
            for (uint32_t v = lane; v < vpc; v += 32u) dev::stg128_cs(dst + v * 16u, dev::ldg128(src + v * 16u));
            dst += static_cast<uint64_t>(vpc) * 16u;
        }
    }
}

struct AbsorbArgs {
    uint8_t *planes;
    uint64_t plane_stride, shard_stride;
    uint32_t all, vpc;                  // all: the T shard bits; vpc: 16-byte vectors per padded shard slot
    uint64_t n_rows;
    const uint8_t *inst_status;
    const uint64_t *inst_bal;
    uint32_t *present;
    const uint8_t *buf;
    const uint64_t *reply_off;
    const uint32_t *reply_mask, *reply_inst;
    const uint64_t *reply_ballot;
    uint64_t n;
    uint32_t *taken;                    // may be null
};

// a warp per reply: handle_msg_reconstruct_reply's filter (crossword/messages.rs:667, rspaxos/messages.rs:542), then
// absorb_other (rscoding.rs:336-342): only shards the row does not hold yet are written.  The atomicOr on present[r]
// hands every missing slot to exactly one reply, so two replies' bytes never mix in a slot.
__global__ void __launch_bounds__(kWireThreads) reconstruct_absorb_kernel(const __grid_constant__ AbsorbArgs A) {
    const uint32_t lane = threadIdx.x & 31u;
    const uint64_t warp = (static_cast<uint64_t>(blockIdx.x) * kWireThreads + threadIdx.x) >> 5;
    const uint64_t nwarps = (static_cast<uint64_t>(gridDim.x) * kWireThreads) >> 5;
    for (uint64_t i = warp; i < A.n; i += nwarps) {
        uint32_t won = 0u, m = 0u, r = 0u;
        if (lane == 0u) {
            r = __ldg(A.reply_inst + i);
            m = __ldg(A.reply_mask + i);
            // r out of range (0xffffffff: slot < start_slot or beyond the window, messages.rs:641-643) and masks naming
            // shards >= T (malformed) are dropped whole
            if (r < A.n_rows && (m & ~A.all) == 0u && __ldg(A.inst_status + r) < 4u &&      // Status::Executed
                __ldg(A.reply_ballot + i) >= __ldg(A.inst_bal + r))
                won = m & ~atomicOr(A.present + r, m);
            if (A.taken != nullptr) A.taken[i] = won;
        }
        won = __shfl_sync(0xffffffffu, won, 0);
        if (won == 0u) continue;
        m = __shfl_sync(0xffffffffu, m, 0);
        r = __shfl_sync(0xffffffffu, r, 0);
        const uint64_t slot_bytes = static_cast<uint64_t>(A.vpc) * 16u;
        const uint8_t *src0 = A.buf + __ldg(A.reply_off + i);
        uint8_t *dst0 = A.planes + static_cast<uint64_t>(r) * A.shard_stride;
        while (won) {
            const uint32_t j = static_cast<uint32_t>(__ffs(won) - 1);
            won &= won - 1u;
            // the reply carries its shards in index order, one padded slot each (the layout reconstruct_serve_kernel writes)
            const uint8_t *src = src0 + static_cast<uint64_t>(__popc(m & ((1u << j) - 1u))) * slot_bytes;
            uint8_t *dst = dst0 + static_cast<uint64_t>(j) * A.plane_stride;
            // four loads in flight per lane before their stores: one at a time leaves HBM latency exposed
            for (uint32_t base = 0; base < A.vpc; base += 128u) {
                uint4 x[4];
#pragma unroll
                for (uint32_t k = 0; k < 4u; ++k) {
                    const uint32_t v = base + lane + 32u * k;
                    if (v < A.vpc) x[k] = dev::ldg128(src + v * 16u);
                }
#pragma unroll
                for (uint32_t k = 0; k < 4u; ++k) {
                    const uint32_t v = base + lane + 32u * k;
                    if (v < A.vpc) dev::stg128_cs(dst + v * 16u, x[k]);
                }
            }
        }
    }
}

struct WalkArgs {
    const uint8_t *inst_status;
    uint32_t *present;
    uint32_t *exec_bar;
    uint64_t *submit;
    uint32_t *dec_present;              // [n_rows] present mask the decode kernel sees: all ones = intact, nothing to do
    uint64_t G;
    uint32_t W, d, all, dmask;
};

// a warp per group, two window slots per lane: the execution-bar walk of handle_msg_reconstruct_reply
// (crossword/messages.rs:670-688, rspaxos/messages.rs:545-560) once over the absorbed state
__global__ void __launch_bounds__(kWireThreads) reconstruct_walk_kernel(const __grid_constant__ WalkArgs A) {
    const uint32_t lane = threadIdx.x & 31u;
    const uint64_t warp = (static_cast<uint64_t>(blockIdx.x) * kWireThreads + threadIdx.x) >> 5;
    const uint64_t nwarps = (static_cast<uint64_t>(gridDim.x) * kWireThreads) >> 5;
    for (uint64_t g = warp; g < A.G; g += nwarps) {
        const uint64_t row0 = g * A.W;
        uint32_t pm[2] = {0u, 0u};
        bool ready[2] = {false, false};
#pragma unroll
        for (uint32_t h = 0; h < 2u; ++h) {
            const uint32_t s = lane + 32u * h;
            if (s < A.W) {
                pm[h] = A.present[row0 + s];
                // status >= Committed and avail_shards() >= d
                ready[h] = __ldg(A.inst_status + row0 + s) >= 3u && static_cast<uint32_t>(__popc(pm[h] & A.all)) >= A.d;
            }
        }
        const uint64_t rdy = static_cast<uint64_t>(__ballot_sync(0xffffffffu, ready[0])) |
                             (static_cast<uint64_t>(__ballot_sync(0xffffffffu, ready[1])) << 32);
        const uint32_t bar = A.exec_bar[g];
        uint64_t pass = 0ull;
        uint32_t len = 0u;
        if (bar < A.W) {
            const uint64_t x = ~(rdy >> bar);          // slots >= W are never ready, so the run ends inside the window
            len = x ? static_cast<uint32_t>(__ffsll(static_cast<long long>(x)) - 1) : 64u;
            pass = (len >= 64u ? ~0ull : ((1ull << len) - 1ull)) << bar;
        }
#pragma unroll
        for (uint32_t h = 0; h < 2u; ++h) {
            const uint32_t s = lane + 32u * h;
            if (s >= A.W) continue;
            // passed with fewer than d data shards: reconstruct_data, after which the row holds every data shard
            const bool decode = ((pass >> s) & 1ull) && (pm[h] & A.dmask) != A.dmask;
            A.dec_present[row0 + s] = decode ? (pm[h] & A.all) : 0xffffffffu;
            if (decode) A.present[row0 + s] = pm[h] | A.dmask;
        }
        if (lane == 0u) {
            A.submit[g] = pass;
            A.exec_bar[g] = bar + len;
        }
    }
}

static inline uint32_t wire_grid(ss_ctx *ctx, uint64_t items, uint32_t per_cta) {
    uint64_t ctas = (items + per_cta - 1) / per_cta;
    const uint64_t cap = static_cast<uint64_t>(ctx->sm_count) * 8ull * 8ull;
    if (ctas > cap) ctas = cap;
    if (ctas == 0) ctas = 1;
    return static_cast<uint32_t>(ctas);
}

}  // namespace ssb

using namespace ssb;

extern "C" {

uint64_t ss_frame_accept_max_len(const ss_frame_spec *s, uint32_t max_shards_per_frame) {
    if (s == nullptr) return 0;
    const uint64_t T = uint64_t(s->data_shards) + s->parity_shards;
    const uint64_t L = s->data_shards ? (uint64_t(s->data_len) + s->data_shards - 1) / s->data_shards : 0;
    uint64_t n = 8 + 44 + T + uint64_t(max_shards_per_frame) * (5 + L) + 1;
    if (s->with_assignment) n += 5 + uint64_t(s->population) * (5 + 5 + 9);
    return (n + 15 + 15) & ~uint64_t(15);            // + the alignment pad, rounded up to the stride granule
}

int ss_frame_accept_pack_dev(ss_ctx *ctx, const ss_frame_spec *s, const uint8_t *shard_planes, uint64_t plane_stride,
                             uint64_t shard_stride, const uint32_t *policies, uint32_t n_policies, const uint8_t *policy_idx,
                             uint32_t peer, const uint64_t *slot, const uint64_t *ballot, uint64_t n, uint8_t *out,
                             uint64_t frame_stride, uint64_t *frame_off, uint32_t *frame_len) {
    if (ctx == nullptr || s == nullptr) return set_error(SS_ERR_INVALID_ARG, "null context or spec");
    SS_TRY(ctx_bind(ctx));
    if (n == 0) return SS_OK;
    if (!shard_planes || !policies || !slot || !ballot || !out || !frame_off || !frame_len) return set_error(SS_ERR_INVALID_ARG, "null buffer");
    const uint32_t T = s->data_shards + s->parity_shards;
    if (s->data_shards == 0 || T > 32) return set_error(SS_ERR_INVALID_ARG, "shard counts must satisfy 1 <= d, d+p <= 32");
    if (s->kind != SS_FRAME_PEER_ACCEPT && s->kind != SS_FRAME_WAL_ACCEPT_DATA) return set_error(SS_ERR_INVALID_ARG, "unknown frame kind %u", s->kind);
    if (s->data_len == 0) return set_error(SS_ERR_INVALID_ARG, "null codeword cannot be framed");
    if (s->population == 0 || s->population > 32 || peer >= s->population || n_policies == 0)
        return set_error(SS_ERR_INVALID_ARG, "bad population / peer / policy table");
    if (s->with_assignment && (s->assign_size == 0 || s->assign_size > 64)) return set_error(SS_ERR_INVALID_ARG, "assignment bitmaps must have 1..64 bits");
    if ((frame_stride & 15u) || ((reinterpret_cast<uintptr_t>(out) | reinterpret_cast<uintptr_t>(shard_planes) | plane_stride | shard_stride) & 15u))
        return set_error(SS_ERR_INVALID_ARG, "frame_stride, buffers and strides must be 16-byte aligned");
    PackArgs A;
    A.status = ctx->dev_status;     // a frame that does not fit frame_stride is skipped (frame_len 0) and reported there
    A.planes = shard_planes; A.plane_stride = plane_stride; A.shard_stride = shard_stride;
    A.d = s->data_shards; A.p = s->parity_shards; A.data_len = s->data_len; A.L = (s->data_len + s->data_shards - 1) / s->data_shards;
    A.kind = s->kind; A.variant = s->msg_variant; A.policies = policies; A.policy_idx = policy_idx; A.n_policies = n_policies;
    A.population = s->population; A.peer = peer; A.with_assignment = s->with_assignment; A.assign_size = s->assign_size;
    A.slot = slot; A.ballot = ballot; A.n = n; A.out = out; A.frame_stride = frame_stride; A.frame_off = frame_off; A.frame_len = frame_len;
    if (shard_stride < ((uint64_t(A.L) + 15) & ~uint64_t(15))) return set_error(SS_ERR_INVALID_ARG, "shard_stride shorter than a padded shard");
    frame_pack_kernel<<<wire_grid(ctx, n, kWireThreads / 32), kWireThreads, 0, ctx->stream>>>(A);
    SS_CUDA(cudaGetLastError());
    ctx->launches++;
    return SS_OK;
}

int ss_accept_reply_parse_dev(ss_ctx *ctx, const uint8_t *buf, uint64_t buf_len, const uint64_t *frame_off, const uint32_t *frame_group,
                              const uint8_t *frame_peer, const uint64_t *window_base, uint64_t n_frames, uint64_t n_groups,
                              uint32_t reply_variant, int with_size, uint32_t *rec_group, uint8_t *rec_slot, uint8_t *rec_peer,
                              uint64_t *rec_ballot, uint32_t *rec_kind) {
    if (ctx == nullptr) return set_error(SS_ERR_INVALID_ARG, "null context");
    SS_TRY(ctx_bind(ctx));
    if (n_frames == 0) return SS_OK;
    if (!buf || !frame_off || !frame_group || !frame_peer || !window_base || !rec_group || !rec_slot || !rec_peer || !rec_ballot || !rec_kind)
        return set_error(SS_ERR_INVALID_ARG, "null buffer");
    ParseArgs A;
    A.buf = buf; A.buf_len = buf_len; A.frame_off = frame_off; A.frame_group = frame_group; A.frame_peer = frame_peer;
    A.window_base = window_base; A.n_frames = n_frames; A.G = n_groups; A.reply_variant = reply_variant; A.with_size = with_size ? 1u : 0u;
    A.rec_group = rec_group; A.rec_slot = rec_slot; A.rec_peer = rec_peer; A.rec_ballot = rec_ballot; A.rec_kind = rec_kind;
    accept_reply_parse_kernel<<<wire_grid(ctx, n_frames, kWireThreads), kWireThreads, 0, ctx->stream>>>(A);
    SS_CUDA(cudaGetLastError());
    ctx->launches++;
    return SS_OK;
}

int ss_wal_commit_pack_dev(ss_ctx *ctx, const uint64_t *newly, const uint64_t *window_base, uint64_t n_groups, uint32_t commit_variant,
                           uint8_t *entries, uint32_t *entry_group, uint32_t *entry_len, uint64_t capacity, uint64_t *n_entries) {
    if (ctx == nullptr) return set_error(SS_ERR_INVALID_ARG, "null context");
    SS_TRY(ctx_bind(ctx));
    if (!newly || !window_base || !entries || !entry_group || !entry_len || !n_entries) return set_error(SS_ERR_INVALID_ARG, "null buffer");
    SS_CUDA(cudaMemsetAsync(n_entries, 0, 8, ctx->stream));
    if (n_groups == 0) return SS_OK;
    wal_commit_pack_kernel<<<wire_grid(ctx, n_groups, kWireThreads), kWireThreads, 0, ctx->stream>>>(
        newly, window_base, n_groups, commit_variant, entries, entry_group, entry_len, capacity, reinterpret_cast<unsigned long long *>(n_entries));
    SS_CUDA(cudaGetLastError());
    ctx->launches++;
    return SS_OK;
}

int ss_reconstruct_serve_dev(ss_ctx *ctx, const uint8_t *shard_planes, uint64_t plane_stride, uint64_t shard_stride, uint32_t total_shards,
                             uint32_t shard_len, const uint32_t *req_group, const uint32_t *req_held, const uint32_t *req_excl,
                             const uint8_t *req_status, const uint64_t *reply_off, uint64_t n_requests, uint32_t *reply_mask, uint8_t *out) {
    if (ctx == nullptr) return set_error(SS_ERR_INVALID_ARG, "null context");
    SS_TRY(ctx_bind(ctx));
    if (n_requests == 0) return SS_OK;
    if (!shard_planes || !req_group || !req_held || !req_excl || !req_status || !reply_off || !reply_mask || !out)
        return set_error(SS_ERR_INVALID_ARG, "null buffer");
    if (total_shards == 0 || total_shards > 32 || shard_len == 0) return set_error(SS_ERR_INVALID_ARG, "bad shard geometry");
    if (((reinterpret_cast<uintptr_t>(shard_planes) | reinterpret_cast<uintptr_t>(out) | plane_stride | shard_stride) & 15u) ||
        shard_stride < ((uint64_t(shard_len) + 15) & ~uint64_t(15)))
        return set_error(SS_ERR_INVALID_ARG, "reconstruct serving needs 16-byte aligned, padded shard slots");
    ServeArgs A;
    A.planes = shard_planes; A.plane_stride = plane_stride; A.shard_stride = shard_stride; A.T = total_shards; A.L = shard_len;
    A.req_group = req_group; A.req_held = req_held; A.req_excl = req_excl; A.req_status = req_status; A.reply_off = reply_off;
    A.n = n_requests; A.reply_mask = reply_mask; A.out = out;
    reconstruct_serve_kernel<<<wire_grid(ctx, n_requests, kWireThreads / 32), kWireThreads, 0, ctx->stream>>>(A);
    SS_CUDA(cudaGetLastError());
    ctx->launches++;
    return SS_OK;
}

int ss_reconstruct_reply_dev(ss_rs_coder *coder, uint8_t *shard_planes, uint64_t plane_stride, uint64_t shard_stride,
                             uint32_t data_len, uint64_t n_groups, uint32_t window, const uint8_t *inst_status,
                             const uint64_t *inst_bal, uint32_t *present, uint32_t *exec_bar, const uint8_t *reply_buf,
                             const uint64_t *reply_off, const uint32_t *reply_mask, const uint32_t *reply_inst,
                             const uint64_t *reply_ballot, uint64_t n_replies, uint64_t *submit, uint32_t *taken) {
    if (coder == nullptr) return set_error(SS_ERR_INVALID_ARG, "null coder");
    ss_ctx *ctx = coder->ctx;
    SS_TRY(ctx_bind(ctx));
    if (n_replies == 0) return SS_OK;
    if (!shard_planes || !inst_status || !inst_bal || !present || !exec_bar || !reply_buf || !reply_off || !reply_mask ||
        !reply_inst || !reply_ballot || !submit)
        return set_error(SS_ERR_INVALID_ARG, "null buffer");
    if (window == 0 || window > 64) return set_error(SS_ERR_INVALID_ARG, "window must be 1..64 instances");
    // row indices are u32 with 0xffffffff reserved for "no instance"
    if (n_groups == 0 || n_groups > 0xfffffffeull / window) return set_error(SS_ERR_INVALID_ARG, "n_groups * window must be 1..2^32-2");
    if (data_len == 0) return set_error(SS_ERR_INVALID_ARG, "null codewords cannot be reconstructed (rscoding.rs:495-497)");
    if (!coder->batch_ok || !coder->dec_ok)
        return set_error(SS_ERR_UNSUPPORTED, "batched reconstruct needs d+p <= 12 (coder is %d,%d)", coder->d, coder->p);
    const uint32_t d = static_cast<uint32_t>(coder->d), T = d + static_cast<uint32_t>(coder->p);
    const uint32_t L = (data_len + d - 1u) / d, vpc = (L + 15u) >> 4;
    if (((reinterpret_cast<uintptr_t>(shard_planes) | reinterpret_cast<uintptr_t>(reply_buf) | plane_stride | shard_stride) & 15u) ||
        shard_stride < static_cast<uint64_t>(vpc) * 16u)
        return set_error(SS_ERR_INVALID_ARG, "reconstruct replies need 16-byte aligned, padded shard slots (shard_stride >= round_up(L,16))");
    const uint64_t n = n_groups * window;
    // scratch: [0, keep) stays free for launch_rs_reconstruct_uniform's own offsets (n*12 + 256 bytes for codes other than
    // RS(3,2)); then the decode kernel's present masks and its per-row status, which nobody reads
    const uint64_t keep = (n * 12u + 256u + 255u) & ~uint64_t(255);
    void *scr = nullptr;
    SS_TRY(ctx_scratch(ctx, keep + n * 8u, &scr));
    uint32_t *dec_present = reinterpret_cast<uint32_t *>(static_cast<uint8_t *>(scr) + keep);
    int32_t *dec_status = reinterpret_cast<int32_t *>(dec_present + n);

    AbsorbArgs A;
    A.planes = shard_planes; A.plane_stride = plane_stride; A.shard_stride = shard_stride;
    A.all = (1u << T) - 1u; A.vpc = vpc; A.n_rows = n;
    A.inst_status = inst_status; A.inst_bal = inst_bal; A.present = present;
    A.buf = reply_buf; A.reply_off = reply_off; A.reply_mask = reply_mask; A.reply_inst = reply_inst; A.reply_ballot = reply_ballot;
    A.n = n_replies; A.taken = taken;
    reconstruct_absorb_kernel<<<wire_grid(ctx, n_replies, kWireThreads / 32), kWireThreads, 0, ctx->stream>>>(A);
    SS_CUDA(cudaGetLastError());
    ctx->launches++;

    WalkArgs W;
    W.inst_status = inst_status; W.present = present; W.exec_bar = exec_bar; W.submit = submit; W.dec_present = dec_present;
    W.G = n_groups; W.W = window; W.d = d; W.all = A.all; W.dmask = (1u << d) - 1u;
    reconstruct_walk_kernel<<<wire_grid(ctx, n_groups, kWireThreads / 32), kWireThreads, 0, ctx->stream>>>(W);
    SS_CUDA(cudaGetLastError());
    ctx->launches++;

    // reconstruct_data for the rows the walk marked; every other row reads as intact
    return launch_rs_reconstruct_uniform(coder, shard_planes, plane_stride, shard_stride, data_len, dec_present, n, 1, dec_status);
}

}  // extern "C"
