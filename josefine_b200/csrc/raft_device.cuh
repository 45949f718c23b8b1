// raft_device.cuh -- device-side Chained-Raft replica state machine (sm_100a).
//
// One lane owns one replica.  A CTA is GROUPS_PER_CTA(=32) consecutive groups x R
// replicas; warp w holds replica index w of those 32 groups, so every state
// plane [replica][group] is read with one coalesced 128-bit load per lane and a
// warp normally executes ONE role's code path (all leaders or all followers).
// A launch fuses n ticks: replica state stays in registers, the CTA's mailboxes
// and a block-table cache live in shared memory (struct Local), ticks are
// separated by __syncthreads() only (groups never interact).
//
// Behaviour follows josefine src/raft (file:line cited per function, paths
// relative to the reference).  Data layout and control structure are ours.
#pragma once
#include <stdint.h>

#include "jr_cuda.h"

#include "../../include/josefine_raft_abi.h"

namespace jr {

constexpr uint32_t ABSENT = 0xFFFFFFFFu;     // block table: no such key
constexpr uint32_t TO_PEERS = 0u;            // Address::Peers
constexpr uint32_t TO_CLIENT = 0xFFFFu;      // Address::Client
constexpr uint32_t GROUPS_PER_CTA = 32;

// phases of one dense launch
enum : uint32_t {
  PH_RESET_OUT = 1u << 0,  // start a new outbox (count = 0)
  PH_RESET_FSM = 1u << 1,  // start a new Instruction FIFO
  PH_DRAIN = 1u << 2,      // apply peer mail of the previous step
  PH_PROPOSE = 1u << 3,    // dense + synthetic proposals
  PH_TICK = 1u << 4        // Command::Tick
};

// Mailbox unit (16 B): x = kind[0:4) | flag[4] | aux[8:16) | to[16:32); y,z = term / token; w = block id.
// AppendEntries: header (aux = n_blocks); its block units {id, next, token} follow inline (flag = 0)
// or sit at slot w of the same mailbox (flag = 1: an earlier AppendEntries of this tick carried the same run).
__host__ __device__ inline uint32_t unit_hdr(uint32_t kind, uint32_t flag, uint32_t aux, uint32_t to) {
  return (kind & 15u) | ((flag & 1u) << 4) | ((aux & 255u) << 8) | (to << 16);
}

struct Dev {
  uint4 *p0, *p1, *p2, *p3, *pr;   // state planes, [plane][replica][group]
  uint32_t* mk;                    // max block id present
  uint4* qt;                       // queued client requests [q][replica][group]
  uint4* dg;                       // stream digests {msg, fsm}
  uint2* cn;                       // stream counts {msgs, fsm}
  uint32_t* cnext;                 // block table: next pointer, [id & capm][replica][group] (a window of ids, see tb)
  unsigned long long* ctok;        // block table: payload token
  uint32_t* tb;                    // [group]: window floor -- ids below it were truncated (jr_truncate, deviation D7)
  uint4* ob[2];                    // mailboxes [unit][replica][group], double buffered
  uint32_t* oc[2];                 // units used per replica
  uint4* fs;                       // Instruction-stream records (jr_fsm_record, 2 x uint4 each) [2*rec + half][replica][group]
  uint4* fr;                       // raw Instructions of the running launch [unit][replica][group], Fr units (scratch of fsm_flush)
  uint2* fc;                       // {records stored since the last drain, Instructions emitted since the last drain}
  uint32_t* fq;                    // raw Instructions in d.fr handed from one part of a split launch to the next
  uint32_t G, Gp, R, cap, capm, U, F, Fr, flags;   // cap: ids a window may span; capm: table rows - 1 (power of two >= cap)
  uint32_t emin, emax, hb;
  uint32_t Us, W;                  // shared-memory mailbox units per replica, table-cache entries (power of 2)
  uint32_t use_index;              // receivers use the delivery index (else scan whole mailboxes)
  uint32_t resident;               // bit r: replica index r is hosted here (others are inert, see jr_config)
  uint32_t* hunf;                  // mapped HOST word: the epoch of the last launch in which sym2_kernel left a group to step_kernel
  uint32_t* hscat;                 // mapped HOST word: the epoch of the last launch in which some CTA saw leaders on >= 2 replica indices
  uint32_t* scatter;               // [0] set by a launch when some CTA has leaders on >= 2 replica indices;
                                   // [1] task ticket counter of the running step launch (both zeroed per launch)
  uint32_t* done;                  // [CTA-sized group block]: epoch + parts finished (split launches, see step_kernel)
  unsigned long long* prof;        // JR_PROFILE builds: cycle counters [role 3][slot 16] x {cycles, count}
  uint64_t seed, goff;
};

// Per-lane view of the CTA's shared memory.  Us == 0 / W == 0 (sparse inject
// kernel) means "no staging": every access goes to global memory.
struct Local {
  uint4* in;        // mailbox units of the previous tick   [unit][replica][lane]
  uint4* out;       // mailbox units written this tick
  uint32_t* cin;    // units used, previous tick            [replica][lane]
  uint32_t* cout;
  uint4* tc;        // block-table cache {id, next, token}  [id & (W-1)][replica][lane]
  // Delivery index: bit u of mk[receiver][sender][lane] = unit u of the sender's
  // mailbox is a header addressed to that receiver (or to Peers).  MK_SCAN = the
  // sender emitted a header at slot >= MK_SLOTS: scan its whole mailbox instead.
  uint16_t* mk_in;
  uint16_t* mk_out;
  uint32_t Us, W, lane;
};
constexpr uint32_t MK_SCAN = 0x8000u;   // delivery masks are 16 bits: slots 0..14 + this flag
constexpr uint32_t MK_SLOTS = 15u;

struct StepParams {
  uint64_t now;
  uint64_t step_index;
  uint32_t phases;               // phases of the FIRST tick; later ticks are RESET_OUT|DRAIN|PROPOSE|TICK
  uint32_t n_synth;
  uint32_t n_ticks;              // ticks fused in this launch (>= 1)
  uint32_t dt;                   // ms between fused ticks
  int cur;                       // outbox written by the first tick; 1-cur is read
  const jr_proposal* proposals;  // device, G entries for the first tick, or null
  uint32_t prop_stride;          // entries from one tick's proposals to the next (0: first tick only)
  // Split launch: the n_ticks of every 32-group block are cut into n_parts consecutive runs, one CTA each
  // (grid = n_blocks * n_parts).  Finer tasks fill the last wave of CTAs; see step_kernel.
  uint32_t n_parts = 1, part_ticks = 0, n_blocks = 0, epoch = 0;
  uint32_t trunc = 0, trunc_margin = 0;   // jr_set_auto_truncate: this launch ends with jr_truncate(trunc_margin)
  uint32_t ticket_base = 0;      // value of the ticket counter when this launch starts (every CTA of a split launch takes exactly one)
  // Symmetric-group fold (sym_fold.cuh): set when sym2_kernel ran in front of this launch.  symdone[g] = 1: group g's
  // whole launch has been applied already; symblk[b] = 1: that holds for all 32 groups of block b.
  const uint8_t* symdone = nullptr;
  const uint8_t* symblk = nullptr;
  // jr_run_token_runs: the dense proposal of tick k is computed instead of loaded: runs[g] = {base lo, hi, stride lo, hi},
  // token = base + (tok_tick + k) * stride (base 0: none), node = route[g].  Excludes `proposals`.
  const uint4* tok_runs = nullptr;
  const uint32_t* tok_route = nullptr;
  uint32_t tok_tick = 0;
};

__host__ __device__ inline uint64_t mix64(uint64_t x) {
  x += 0x9e3779b97f4a7c15ull;
  x = (x ^ (x >> 30)) * 0xbf58476d1ce4e5b9ull;
  x = (x ^ (x >> 27)) * 0x94d049bb133111ebull;
  return x ^ (x >> 31);
}
__host__ __device__ inline uint64_t fold(uint64_t h, uint64_t w) { return mix64(h ^ w); }

// Deviation D2 (normative text in the ABI header).
__host__ __device__ inline uint32_t election_timeout_draw(uint64_t seed, uint64_t group, uint32_t node,
                                                          uint32_t draw, uint32_t mn, uint32_t mx) {
  uint64_t x = mix64(seed ^ 0x6a09e667f3bcc908ull);
  x = mix64(x + group);
  x = mix64(x + (((uint64_t)node << 32) | draw));
  return mn + (uint32_t)(((x >> 32) * (uint64_t)(mx - mn)) >> 32);
}

__host__ __device__ inline uint64_t synth_token(uint64_t step_index, uint32_t i, uint64_t g_global) {
  return ((step_index * 8 + i + 1) << 32) | (g_global & 0xffffffffull);
}

// A decoded command as the handlers see it.  Blocks come either from mailbox
// units (strided) or from a host jr_msg copied to the device.
struct Cmd {
  uint32_t kind, flag, node_id, nblk;
  uint32_t block;          // head / commit / block id; for ClientRequest: client address (kind<<16 | id)
  uint64_t term;           // term; for ClientRequest / ClientResponse: the request token (D5)
  uint64_t last_term;      // VoteRequest only
  uint32_t blk_s, blk_at;  // mailbox: sender index and slot of the first block unit
  const jr_msg* host_msg;  // injected command (blocks are read from it) or null
};

#ifdef JR_DEVICE_CODE

// Stream digest of one Message (normative: DESIGN.md "Digests").  Kept out of
// line: it is only live with JR_F_STREAM_DIGEST and would otherwise be inlined
// at every send site.
__device__ __noinline__ uint64_t digest_message_fn(uint64_t h, uint32_t kind, uint32_t to, uint32_t flag,
                                                   uint32_t nblk, uint32_t node_id, uint64_t t,
                                                   uint64_t last_term, uint64_t block, uint64_t token,
                                                   uint32_t addr) {
  uint32_t to_kind = to == TO_PEERS ? JR_ADDR_PEERS : (to == TO_CLIENT ? JR_ADDR_CLIENT : JR_ADDR_PEER);
  uint32_t to_id = to_kind == JR_ADDR_PEER ? to : 0u;
  h = fold(h, (uint64_t)kind | ((uint64_t)to_kind << 8) | ((uint64_t)(flag & 1u) << 16) |
                  ((uint64_t)nblk << 24) | ((uint64_t)to_id << 32));
  h = fold(h, node_id);
  h = fold(h, t);
  h = fold(h, last_term);
  h = fold(h, block);
  h = fold(h, token);
  h = fold(h, (uint64_t)(addr >> 16) | ((uint64_t)(addr & 0xffffu) << 8));
  return h;
}

__device__ __noinline__ uint64_t digest_send_fn(uint64_t h, uint32_t self, uint32_t kind, uint32_t to,
                                                uint32_t flag, uint32_t aux, uint64_t t, uint32_t w,
                                                uint32_t* n_out) {
  uint32_t n = 1;
  switch (kind) {
    case JR_CMD_VOTE_REQUEST:
      n = aux;
      for (uint32_t k = 0; k < aux; ++k) h = digest_message_fn(h, kind, to, 0, 0, self, t, t, w, 0, 0);
      break;
    case JR_CMD_VOTE_RESPONSE: h = digest_message_fn(h, kind, to, flag, 0, self, t, 0, 0, 0, 0); break;
    case JR_CMD_APPEND_RESPONSE: h = digest_message_fn(h, kind, to, flag, 0, self, t, 0, w, 0, 0); break;
    case JR_CMD_HEARTBEAT: h = digest_message_fn(h, kind, to, 0, 0, self, t, 0, w, 0, 0); break;
    case JR_CMD_HEARTBEAT_RESPONSE: h = digest_message_fn(h, kind, to, flag, 0, 0, 0, 0, w, 0, 0); break;
    case JR_CMD_CLIENT_REQUEST: h = digest_message_fn(h, kind, to, 0, 0, 0, 0, 0, 0, t, w); break;
    default: h = digest_message_fn(h, kind, to, 0, 0, 0, 0, 0, 0, t, 0); break;  // ClientResponse
  }
  *n_out = n;
  return h;
}

__device__ __noinline__ uint64_t digest_fsm_fn(uint64_t h, bool notify, uint32_t bid, uint32_t next_or_addr,
                                               uint64_t tok) {
  if (notify) {
    h = fold(h, (uint64_t)JR_FSM_NOTIFY | ((uint64_t)(next_or_addr >> 16) << 8) |
                    ((uint64_t)(next_or_addr & 0xffffu) << 32));
    h = fold(h, bid);
    h = fold(h, 0);
  } else {
    h = fold(h, (uint64_t)JR_FSM_APPLY);
    h = fold(h, bid);
    h = fold(h, next_or_addr);
  }
  return fold(h, tok);
}

#ifdef JR_PROFILE
// Phase profiler (tools/phase_profile.py): lane 0 of a warp attributes clock64() deltas
// to (role, slot).  Slots 0..11 = time inside apply for that Command kind, 12 = whole
// tick, 13 = waiting at the per-tick barrier, 14 = fetch (next_cmd), 15 = tick bookkeeping.
// per-warp accumulators live in static shared memory and are flushed once per launch
__device__ __forceinline__ unsigned long long* jr_prof_smem() {
  __shared__ unsigned long long acc[8 * 3 * 16 * 2];
  return acc;
}
#define JR_PROF_T0(var) long long var = clock64()
#define JR_PROF_ADD(role, slot, var) do { long long _n = clock64(); if ((threadIdx.x & 31u) == 0) { unsigned long long* _p = jr_prof_smem() + (((threadIdx.x >> 5) * 3 + (role)) * 16 + (slot)) * 2; _p[0] += (unsigned long long)(_n - var); _p[1] += 1ull; } var = clock64(); } while (0)
#else
#define JR_PROF_T0(var) do { } while (0)
#define JR_PROF_ADD(role, slot, var) do { } while (0)
#endif


// ---------------------------------------------------------------------------------------------
// Instruction-stream encoder (fsm_tx, fsm.rs:19-29).  A replica's Instructions leave the device
// run-length encoded as jr_fsm_record (32 B, layout normative in the ABI header):
//   APPLY run   blocks id0, id0+1, ... whose `next` is id-1 and whose tokens form an arithmetic
//               progression (count == 1: any block, `next` explicit)
//   NOTIFY run  block ids id0, id0+1, ... for Address::Client, tokens in arithmetic progression
//               (count == 1: any client address)
//   PATTERN     which positions of the replica's stream are Notify (bit = 1); positions no PATTERN
//               record covers are Apply.  Applies and Notifies each keep their own order, so the
//               three together reproduce the stream exactly.
// The state machine itself only appends the raw Instruction (16 B) to the replica's scratch FIFO
// d.fr -- one store, no state beyond a counter.  The encoding runs in fsm_flush, once per launch
// (and when the scratch FIFO fills up), where the open runs can live in registers because nothing
// of the Replica is live in that function: the hot loop pays no registers and no shared memory.
constexpr uint32_t FSR_APPLY = 0u, FSR_NOTIFY = 1u, FSR_PATTERN = 2u;
constexpr uint32_t FSR_CLIENT = (uint32_t)JR_ADDR_CLIENT << 16;
constexpr uint32_t FS_MAX_RUN = 0xffffffu;   // the record's count field is 24 bits
constexpr uint32_t FS_PATTERN_BITS = 160u;   // Instructions one PATTERN record covers
constexpr uint32_t FS_NOTIFY_BIT = 0x80000000u;   // raw entry: x = block id | this; y = next / client address; z,w = token

struct FsmOut {       // where one replica's records go
  uint4* slot0;       // d.fs + rg
  size_t plane;       // R * Gp
  uint32_t F, g, r;
  uint32_t mask = 0;  // APPLY records stand for every node whose bit (id - 1) is set (symmetric followers, sym_fold.cuh)
};

struct FsmRun {       // an open run: next id expected, elements so far, last token, stride (count 1: lo word = next / address)
  uint32_t next_id, count;
  uint64_t last, stride;
};

__device__ __forceinline__ uint32_t fsm_put_record(uint32_t nrec, const FsmOut& o, uint32_t kind, uint32_t count, uint32_t id0,
                                                   uint32_t addr, uint64_t tok0, uint64_t stride) {
  if (nrec < o.F) {
    o.slot0[(size_t)(2 * nrec) * o.plane] = make_uint4(o.g, kind | (o.r << 2) | (count << 8), id0, addr);
    o.slot0[(size_t)(2 * nrec + 1) * o.plane] =
        make_uint4((uint32_t)tok0, (uint32_t)(tok0 >> 32), (uint32_t)stride, (uint32_t)(stride >> 32));
  }
  return nrec + 1;  // past F: counted, not stored (the drain reports JR_E_CAPACITY; consensus is not affected)
}

__device__ __forceinline__ uint32_t fsm_close_run(uint32_t nrec, const FsmOut& o, bool notify, const FsmRun& run) {
  const uint32_t c = run.count;
  if (!c) return nrec;
  const uint64_t tok0 = c > 1 ? run.last - (uint64_t)(c - 1) * run.stride : run.last;
  const uint32_t addr = notify ? (c > 1 ? FSR_CLIENT : (uint32_t)run.stride) : o.mask;
  return fsm_put_record(nrec, o, notify ? FSR_NOTIFY : FSR_APPLY, c, run.next_id - c, addr, tok0,
                        (notify && c == 1) ? 0ull : run.stride);
}

// Streaming encoder of one replica's Instruction stream: fsm_flush feeds it the raw FIFO of a launch; the symmetric-group
// fold (sym_fold.cuh) feeds it every Instruction as it is produced, with this state parked in shared memory in between.
struct FsmEnc {
  uint32_t nrec, seq;        // records / Instructions since the last drain
  // pattern window: FS_PATTERN_BITS Instructions per PATTERN record (bits 0-63 in tok0, 64-127 in stride, 128-159 in addr);
  // a window starts where the previous launch stopped (wseq) and is closed when full or when the launch ends
  uint32_t wseq, pb2;
  uint64_t pb0, pb1;
  FsmRun ra, rn;             // the open APPLY / NOTIFY run
};

__device__ __forceinline__ void fsm_enc_begin(FsmEnc& s, uint2 c) {
  s.nrec = c.x; s.seq = s.wseq = c.y;
  s.pb0 = s.pb1 = 0; s.pb2 = 0;
  s.ra = FsmRun{0, 0, 0, 0};
  s.rn = FsmRun{0, 0, 0, 0};
}

template <bool NOTIFY>
__device__ __forceinline__ void fsm_enc_push(FsmEnc& s, const FsmOut& o, uint32_t bid, uint32_t nxa, uint64_t tok) {
  if (NOTIFY) {
    const uint32_t b = s.seq - s.wseq;
    if (b < 64u) s.pb0 |= 1ull << b;
    else if (b < 128u) s.pb1 |= 1ull << (b - 64u);
    else s.pb2 |= 1u << (b - 128u);
  }
  ++s.seq;
  if (s.seq - s.wseq == FS_PATTERN_BITS) {   // the pattern window is complete
    if (s.pb0 | s.pb1 | s.pb2) s.nrec = fsm_put_record(s.nrec, o, FSR_PATTERN, FS_PATTERN_BITS, s.wseq, s.pb2, s.pb0, s.pb1);
    s.pb0 = s.pb1 = 0; s.pb2 = 0;
    s.wseq = s.seq;
  }
  FsmRun& run = NOTIFY ? s.rn : s.ra;   // (picked at compile time: both runs stay in registers)
  if (run.count) {
    const uint64_t step = tok - run.last;
    bool ok = bid == run.next_id && run.count < FS_MAX_RUN;
    if (NOTIFY) ok = ok && nxa == FSR_CLIENT && (run.count > 1u || (uint32_t)run.stride == FSR_CLIENT);
    else ok = ok && nxa == bid - 1u && (run.count > 1u || (uint32_t)run.stride == bid - 2u);   // count 1: its own `next` must be regular too
    if (ok && run.count > 1u) ok = step == run.stride;
    if (ok) {
      if (run.count == 1u) run.stride = step;
      run.next_id = bid + 1u;
      run.count += 1u;
      run.last = tok;
      return;
    }
    s.nrec = fsm_close_run(s.nrec, o, NOTIFY, run);
  }
  run = FsmRun{bid + 1u, 1u, tok, (uint64_t)nxa};   // count 1: Apply keeps the block's `next`, Notify the client address
}

// Close the open runs and the pattern window; returns the replica's new {records, Instructions} counters.
__device__ __forceinline__ uint2 fsm_enc_end(FsmEnc& s, const FsmOut& o) {
  s.nrec = fsm_close_run(s.nrec, o, false, s.ra);
  s.nrec = fsm_close_run(s.nrec, o, true, s.rn);
  if (s.pb0 | s.pb1 | s.pb2) s.nrec = fsm_put_record(s.nrec, o, FSR_PATTERN, s.seq - s.wseq, s.wseq, s.pb2, s.pb0, s.pb1);
  return make_uint2(s.nrec, s.seq);
}

// Encode the n_raw raw Instructions of this replica (raw0[u * plane], u < min(n_raw, Fr)) behind what d.fc says was
// emitted before them.  Raw entries beyond Fr were never stored: they count as dropped records.
__device__ __noinline__ void fsm_flush(const uint4* raw0, uint32_t n_raw, uint32_t Fr, FsmOut o, uint2* fc) {
  FsmEnc s;
  fsm_enc_begin(s, *fc);
  const uint32_t n = n_raw < Fr ? n_raw : Fr;
  constexpr uint32_t AHEAD = 8;   // entries are independent loads (L2 / DRAM): fetch a batch, then encode it
  for (uint32_t u0 = 0; u0 < n; u0 += AHEAD) {
    uint4 buf[AHEAD];
#pragma unroll
    for (uint32_t j = 0; j < AHEAD; ++j)
      if (u0 + j < n) buf[j] = __ldcg(raw0 + (size_t)(u0 + j) * o.plane);
#pragma unroll
    for (uint32_t j = 0; j < AHEAD; ++j) {
      if (u0 + j >= n) break;
      const uint4 e = buf[j];
      const uint32_t bid = e.x & ~FS_NOTIFY_BIT;
      const uint64_t tok = (uint64_t)e.z | ((uint64_t)e.w << 32);
      if (e.x & FS_NOTIFY_BIT) fsm_enc_push<true>(s, o, bid, e.y, tok);
      else fsm_enc_push<false>(s, o, bid, e.y, tok);
    }
  }
  uint2 c = fsm_enc_end(s, o);
  if (n_raw > Fr) c.x = (c.x > o.F ? c.x : o.F) + (n_raw - Fr);   // lost Instructions: the drain must say so
  *fc = c;
}

template <int R, bool SORTED = false>
struct Replica {
  const Dev& d;
  const Local& L;
  const uint32_t r, g;   // replica index (node id - 1), local group
  const size_t rg;       // r * Gp + g
  const size_t plane;    // R * Gp
  uint64_t now;
  int cur;
  uint32_t ocnt0;        // units already in the outbox when this launch started (continuation launches)
  // ---- State (mod.rs:271-287) + role state + Chain scalars (chain.rs:99-104)
  uint64_t term, etime, hbtime;
  uint32_t voted, etimeout, draws, head, commit, idgen, maxkey, tbase;
  uint32_t role, fault, prmask, nq, dead, ckey;
  // Role-exclusive state shares registers: a Leader's progress heads ph[0..R), a Candidate's vote masks and a
  // Follower's leader_id are never live together (every transition below re-initialises what the new role reads).
  uint32_t ph[R < 3 ? 3 : R];
#define seen ph[0]
#define granted ph[1]
#define leader ph[2]
  // ---- output cursors
  uint32_t ocnt, fcnt;   // units in the outbox; raw Instructions in d.fr since the last fsm_flush
  // (the stream digests and counts of JR_F_STREAM_DIGEST stay in d.dg / d.cn: a test feature must not cost the
  //  product kernel six registers)
  uint32_t mko[R];       // delivery index of this tick's outbox, one mask per receiver (see Local::mk_out)

  __device__ __forceinline__ Replica(const Dev& dv, const Local& lv, uint32_t r_, uint32_t g_)
      : d(dv), L(lv), r(r_), g(g_), rg((size_t)r_ * dv.Gp + g_), plane((size_t)R * dv.Gp) {}

  __device__ __forceinline__ uint32_t id() const { return r + 1; }
  __device__ __forceinline__ bool live() const { return !dead && fault == 0; }
  __device__ __forceinline__ bool digest_on() const { return d.flags & JR_F_STREAM_DIGEST; }

  // ------------------------------------------------------------------ load/store
  __device__ __forceinline__ void load(bool reset_out, bool reset_fsm, bool continues = false) {
    uint4 a = d.p0[rg], b = d.p1[rg], c = d.p2[rg];
    term = (uint64_t)a.x | ((uint64_t)a.y << 32); voted = a.z;
    etime = (uint64_t)b.x | ((uint64_t)b.y << 32); etimeout = b.z; draws = b.w;
    head = c.x; commit = c.y; idgen = c.z;
    uint32_t m = c.w;
    role = m & 255u; fault = (m >> 8) & 255u; prmask = (m >> 16) & 255u;
    nq = (m >> 24) & 7u; dead = (m >> 27) & 1u; ckey = (m >> 28) & 1u;
    maxkey = d.mk[rg];
    tbase = d.tb[g];
    hbtime = 0;
#pragma unroll
    for (int i = 0; i < (R < 3 ? 3 : R); ++i) ph[i] = 0;
    leader = a.w;   // Follower.leader_id (0 for the other roles)
    if (role != JR_ROLE_FOLLOWER) {
      uint4 e = d.p3[rg];
      hbtime = (uint64_t)e.x | ((uint64_t)e.y << 32); seen = e.z; granted = e.w;
      if (role == JR_ROLE_LEADER) {
#pragma unroll
        for (int q = 0; q < (R + 3) / 4; ++q) {
          uint4 v = d.pr[(size_t)q * plane + rg];
          if (q * 4 + 0 < R) ph[q * 4 + 0] = v.x;
          if (q * 4 + 1 < R) ph[q * 4 + 1] = v.y;
          if (q * 4 + 2 < R) ph[q * 4 + 2] = v.z;
          if (q * 4 + 3 < R) ph[q * 4 + 3] = v.w;
        }
      }
    }
    ocnt = reset_out ? 0u : d.oc[cur][rg];
    ocnt0 = ocnt;
    fcnt = (continues && (d.flags & JR_F_CAPTURE_FSM)) ? d.fq[rg] : 0u;   // a later part of a split launch appends to the same raw FIFO
    if (reset_fsm && (d.flags & JR_F_CAPTURE_FSM)) d.fc[rg] = make_uint2(0u, 0u);
  }

  __device__ __forceinline__ void store(bool last_part = true) {
    d.p0[rg] = make_uint4((uint32_t)term, (uint32_t)(term >> 32), voted, role == JR_ROLE_FOLLOWER ? leader : 0u);
    d.p1[rg] = make_uint4((uint32_t)etime, (uint32_t)(etime >> 32), etimeout, draws);
    uint32_t m = role | (fault << 8) | (prmask << 16) | (nq << 24) | (dead << 27) | (ckey << 28);
    d.p2[rg] = make_uint4(head, commit, idgen, m);
    d.mk[rg] = maxkey;
    if (role != JR_ROLE_FOLLOWER) {
      d.p3[rg] = make_uint4((uint32_t)hbtime, (uint32_t)(hbtime >> 32), role == JR_ROLE_CANDIDATE ? seen : 0u,
                            role == JR_ROLE_CANDIDATE ? granted : 0u);
      if (role == JR_ROLE_LEADER) {
#pragma unroll
        for (int q = 0; q < (R + 3) / 4; ++q) {
          uint4 v = make_uint4(0, 0, 0, 0);
          if (q * 4 + 0 < R) v.x = ph[q * 4 + 0];
          if (q * 4 + 1 < R) v.y = ph[q * 4 + 1];
          if (q * 4 + 2 < R) v.z = ph[q * 4 + 2];
          if (q * 4 + 3 < R) v.w = ph[q * 4 + 3];
          d.pr[(size_t)q * plane + rg] = v;
        }
      }
    }
    // the last tick's mailbox lives in shared memory: publish it for the next launch / capture
    const uint32_t staged = ocnt < L.Us ? ocnt : L.Us;
    for (uint32_t u = ocnt0; u < staged; ++u)
      d.ob[cur][((size_t)u * R + r) * d.Gp + g] = L.out[(u * R + r) * 32 + L.lane];
    d.oc[cur][rg] = ocnt;
    if (last_part) fsm_flush_now();                       // the launch's Instructions become records once, at its end
    else if (d.flags & JR_F_CAPTURE_FSM) d.fq[rg] = fcnt;
  }

  // ------------------------------------------------------------------ block table (chain.rs)
  // The table holds the ids of a window [tbase, tbase + cap): row = id & capm.  Ids below the floor were
  // truncated (jr_truncate, deviation D7) and read as absent; ids at or past the end cannot be stored.
  __device__ __forceinline__ size_t tix(uint32_t bid) const { return (size_t)(bid & d.capm) * plane + rg; }
  __device__ __forceinline__ bool in_window(uint32_t bid) const { return bid - tbase < d.cap && bid < FS_NOTIFY_BIT; }   // (ids < 2^31, D4)
  // Block table reads go through a direct-mapped, write-through cache in shared
  // memory (tag = id).  Only this lane writes its own table, so the cache is
  // coherent for the whole launch; it is rebuilt at launch start.
  __device__ __forceinline__ uint4* tc_slot(uint32_t bid) const {
    return L.tc + (((bid & (L.W - 1)) * R + r) * 32 + L.lane);
  }
  __device__ __forceinline__ void tbl_fetch(uint32_t bid, uint32_t& next, uint64_t& tok) const {
    if (L.W) {
      const uint4 e = *tc_slot(bid);
      if (e.x == bid) { next = e.y; tok = (uint64_t)e.z | ((uint64_t)e.w << 32); return; }
    }
    if (!in_window(bid)) { next = ABSENT; tok = 0; return; }
    next = d.cnext[tix(bid)];   // both loads issue together: one latency
    tok = d.ctok[tix(bid)];
    if (L.W) *tc_slot(bid) = make_uint4(bid, next, (uint32_t)tok, (uint32_t)(tok >> 32));
  }
  __device__ __forceinline__ uint32_t tbl_next(uint32_t bid) const {
    uint32_t n; uint64_t t;
    tbl_fetch(bid, n, t);
    return n;
  }
  __device__ __forceinline__ uint64_t tbl_tok(uint32_t bid) const {
    uint32_t n; uint64_t t;
    tbl_fetch(bid, n, t);
    return t;
  }
  // chain.rs:155-157
  __device__ __forceinline__ bool has(uint32_t bid) const { return tbl_next(bid) != ABSENT; }
  __device__ __forceinline__ void tbl_put(uint32_t bid, uint32_t next, uint64_t tok) {
    d.cnext[tix(bid)] = next;
    d.ctok[tix(bid)] = tok;
    if (L.W) *tc_slot(bid) = make_uint4(bid, next, (uint32_t)tok, (uint32_t)(tok >> 32));
    if (bid > maxkey) maxkey = bid;
  }
  // Launch start: invalidate, then pull the table tail (the blocks the steady state touches).
  // The loads of a batch are independent and issued together: this runs once per task, in front of
  // every tick, and a task is short when a launch is split (step_kernel).
  __device__ __forceinline__ void tc_prefetch() const {
    if (!L.W) return;
    for (uint32_t k = 0; k < L.W; ++k) L.tc[(k * R + r) * 32 + L.lane] = make_uint4(0xFFFFFFFFu, ABSENT, 0, 0);
    if (maxkey < tbase) return;            // (a silenced replica the window has moved past)
    const uint32_t span = maxkey - tbase;  // ids tbase..maxkey are the part of the window that may hold blocks
    for (uint32_t k0 = 0; k0 < L.W && k0 <= span; k0 += 4) {
      uint32_t n[4];
      uint64_t t[4];
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (k0 + j < L.W && k0 + j <= span) {
          n[j] = d.cnext[tix(maxkey - k0 - j)];
          t[j] = d.ctok[tix(maxkey - k0 - j)];
        }
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (k0 + j < L.W && k0 + j <= span)
          *tc_slot(maxkey - k0 - j) = make_uint4(maxkey - k0 - j, n[j], (uint32_t)t[j], (uint32_t)(t[j] >> 32));
    }
  }
  // Launch start: copy this lane's own previous-tick outbox into the shared mailbox.
  __device__ __forceinline__ void stage_inbox(bool deliver) const {
    if (!L.cin) return;
    const int prv = 1 - cur;
    const uint32_t cnt = deliver ? d.oc[prv][rg] : 0u;
    L.cin[r * 32 + L.lane] = cnt;
    const uint32_t n = cnt < L.Us ? cnt : L.Us;
    for (uint32_t u0 = 0; u0 < n; u0 += 4) {  // coherent loads: a split launch hands mailboxes over inside a kernel
      uint4 v[4];
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (u0 + j < n) v[j] = __ldcg(d.ob[prv] + ((size_t)(u0 + j) * R + r) * d.Gp + g);
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (u0 + j < n) L.in[((u0 + j) * R + r) * 32 + L.lane] = v[j];
    }
    // the delivery index is derived data: rebuild it from the units just staged
    uint32_t m[R];
#pragma unroll
    for (int t = 0; t < R; ++t) m[t] = 0;
    for (uint32_t u = 0; u < cnt;) {
      const uint4 h = u < L.Us ? L.in[(u * R + r) * 32 + L.lane] : __ldcg(d.ob[prv] + ((size_t)u * R + r) * d.Gp + g);
      const uint32_t kind = h.x & 15u, aux = (h.x >> 8) & 255u, to = h.x >> 16;
      const uint32_t bit = u < MK_SLOTS ? (1u << u) : MK_SCAN;
      const bool noop = kind == JR_CMD_HEARTBEAT_RESPONSE && (((h.x >> 4) & 1u) || h.w == 0);
      if (!noop || bit == MK_SCAN) {
#pragma unroll
        for (int t = 0; t < R; ++t)
          if (to == TO_PEERS || to == (uint32_t)t + 1u) m[t] |= bit;
      }
      u += 1u + ((kind == JR_CMD_APPEND_ENTRIES && !((h.x >> 4) & 1u)) ? aux : 0u);
    }
#pragma unroll
    for (int t = 0; t < R; ++t) L.mk_in[(t * R + r) * 32 + L.lane] = (uint16_t)m[t];
  }
  // chain.rs:160-175; returns false on fault
  __device__ __forceinline__ bool chain_append(uint64_t tok, uint32_t& out_id) {
    uint32_t bid = idgen++;  // fetch_add precedes the assert
    if (!(bid > head)) { fault = JR_FAULT_APPEND_ID_NOT_GT_HEAD; return false; }
    if (!in_window(bid)) { fault = JR_FAULT_ENGINE_CHAIN_CAPACITY; return false; }
    tbl_put(bid, head, tok);
    head = bid;
    out_id = bid;
    return true;
  }
  // chain.rs:178-192
  __device__ __forceinline__ bool chain_extend(uint32_t bid, uint32_t next, uint64_t tok) {
    if (!has(next)) { fault = JR_FAULT_EXTEND_PARENT_MISSING; return false; }
    if (!in_window(bid)) { fault = JR_FAULT_ENGINE_CHAIN_CAPACITY; return false; }
    tbl_put(bid, next, tok);
    head = bid;
    return true;
  }
  // chain.rs:195-205
  __device__ __forceinline__ bool chain_commit(uint32_t bid) {
    if (!has(bid)) { fault = JR_FAULT_COMMIT_BLOCK_MISSING; return false; }
    ckey = 1;  // db.insert("commit", ..)
    commit = bid;
    return true;
  }

  // ------------------------------------------------------------------ outputs
  __device__ __forceinline__ bool put_unit(uint32_t slot, uint4 v) {
    if (slot >= d.U) { fault = JR_FAULT_ENGINE_MAILBOX_OVERFLOW; return false; }
    if (slot < L.Us) L.out[(slot * R + r) * 32 + L.lane] = v;
    else d.ob[cur][((size_t)slot * R + r) * d.Gp + g] = v;
    return true;
  }
  __device__ __forceinline__ uint4 own_unit(uint32_t slot) const {  // read back what this lane emitted
    if (slot < L.Us) return L.out[(slot * R + r) * 32 + L.lane];
    return d.ob[cur][((size_t)slot * R + r) * d.Gp + g];
  }
  // unit `u` of sender `s_` in the previous tick's mailbox
  __device__ __forceinline__ uint4 inbox_unit(uint32_t s_, uint32_t u) const {
    if (u < L.Us) return L.in[(u * R + s_) * 32 + L.lane];
    return __ldcg(d.ob[1 - cur] + ((size_t)u * R + s_) * d.Gp + g);  // spilled unit: L2, never a stale L1 line
  }

  __device__ __forceinline__ void mark(uint32_t to, uint32_t slot) {
    const uint32_t bit = slot < MK_SLOTS ? (1u << slot) : MK_SCAN;
#pragma unroll
    for (int t = 0; t < R; ++t)
      if (to == TO_PEERS || to == (uint32_t)t + 1u) mko[t] |= bit;
  }
  __device__ __forceinline__ void clear_marks() {
#pragma unroll
    for (int t = 0; t < R; ++t) mko[t] = 0;
  }
  __device__ __forceinline__ void publish_marks() const {
    if (!L.mk_out) return;
#pragma unroll
    for (int t = 0; t < R; ++t) L.mk_out[(t * R + r) * 32 + L.lane] = (uint16_t)mko[t];
  }

  // mod.rs:390-400 for every single-unit command.
  __device__ __forceinline__ void send(uint32_t kind, uint32_t to, uint32_t flag, uint32_t aux, uint64_t t, uint32_t w) {
    if (!put_unit(ocnt, make_uint4(unit_hdr(kind, flag, aux, to), (uint32_t)t, (uint32_t)(t >> 32), w))) return;
    // HeartbeatResponse{has_committed || commit == 0} changes nothing in any role
    // (follower.rs:61, candidate.rs:193, leader.rs:227): emitted, but not indexed for dispatch.
    if (!(kind == JR_CMD_HEARTBEAT_RESPONSE && (flag || w == 0))) mark(to, ocnt);
    ++ocnt;
    if (digest_on()) {
      uint32_t n;
      uint4 v = d.dg[rg];
      const uint64_t h = digest_send_fn((uint64_t)v.x | ((uint64_t)v.y << 32), id(), kind, to, flag, aux, t, w, &n);
      v.x = (uint32_t)h; v.y = (uint32_t)(h >> 32);
      d.dg[rg] = v;
      d.cn[rg].x += n;
    }
  }

  __device__ __forceinline__ FsmOut fsm_out() const { return FsmOut{d.fs + rg, plane, d.F, g, r}; }
  // Encode what sits in the raw FIFO (launch end; tick end when it is nearly full).
  __device__ __forceinline__ void fsm_flush_now() {
    if ((d.flags & JR_F_CAPTURE_FSM) && fcnt) {
      fsm_flush(d.fr + rg, fcnt, d.Fr, fsm_out(), d.fc + rg);
      fcnt = 0;
    }
  }
  // fsm_tx.send(Instruction) (fsm.rs:19-29)
  __device__ __forceinline__ void fsm_emit(bool notify, uint32_t bid, uint32_t next_or_addr, uint64_t tok) {
    if (d.flags & JR_F_CAPTURE_FSM) {
      if (fcnt < d.Fr)
        d.fr[(size_t)fcnt * plane + rg] =
            make_uint4(bid | (notify ? FS_NOTIFY_BIT : 0u), next_or_addr, (uint32_t)tok, (uint32_t)(tok >> 32));
      ++fcnt;
    }
    if (digest_on()) {
      uint4 v = d.dg[rg];
      const uint64_t h = digest_fsm_fn((uint64_t)v.z | ((uint64_t)v.w << 32), notify, bid, next_or_addr, tok);
      v.z = (uint32_t)h; v.w = (uint32_t)(h >> 32);
      d.dg[rg] = v;
      d.cn[rg].y += 1u;
    }
  }

  // ------------------------------------------------------------------ mod.rs
  // mod.rs:352-357 (Instant::elapsed saturates)
  __device__ __forceinline__ bool needs_election() const {
    uint64_t el = now >= etime ? now - etime : 0;
    return el > (uint64_t)etimeout;
  }
  // mod.rs:360-365 + Role::term (follower.rs:27-29, candidate.rs:161-163, leader.rs:33-35)
  __device__ __forceinline__ bool set_term(uint64_t t) {
    voted = 0;
    term = t;
    if (role == JR_ROLE_FOLLOWER) leader = 0;
    else if (role == JR_ROLE_CANDIDATE) seen = granted = 0;
    else { fault = JR_FAULT_LEADER_TERM_UNIMPLEMENTED; return false; }
    return true;
  }
  // follower.rs:103-113 (D2)
  __device__ __forceinline__ void set_election_timeout() {
    etimeout = election_timeout_draw(d.seed, d.goff + g, id(), draws++, d.emin, d.emax);
    etime = now;
  }

  // ------------------------------------------------------------------ queue (follower.rs:23, candidate.rs:20)
  __device__ __forceinline__ bool queue_push(uint64_t tok, uint32_t addr) {
    if (nq >= JR_CLIENT_QUEUE_CAP) { fault = JR_FAULT_ENGINE_QUEUE_OVERFLOW; return false; }
    d.qt[(size_t)nq * plane + rg] = make_uint4((uint32_t)tok, (uint32_t)(tok >> 32), addr, 0);
    ++nq;
    return true;
  }

  // ------------------------------------------------------------------ election.rs
  __device__ __forceinline__ void vote(uint32_t from, bool v) {  // election.rs:33-35, last write wins
    uint32_t bit = 1u << ((from - 1) & 31u);
    seen |= bit;
    granted = v ? (granted | bit) : (granted & ~bit);
  }
  // election.rs:37-73: 0 Elected, 1 Voting, 2 Defeated
  __device__ __forceinline__ int election_status() const {
    const int q = (R == 1) ? 0 : (R / 2 + 1);
    int votes = __popc(granted), total = __popc(seen);
    if (votes >= q) return 0;
    if (total - votes == q) return 2;
    return 1;
  }

  // ------------------------------------------------------------------ progress.rs
  __device__ __forceinline__ uint32_t get_ph(uint32_t i) const {
    uint32_t v = 0;
#pragma unroll
    for (int k = 0; k < R; ++k) if (k == (int)i) v = ph[k];
    return v;
  }
  // progress.rs:42-46,76-94,133-140
  __device__ __forceinline__ bool progress_advance(uint32_t node, uint32_t bid) {
    if (node < 1 || node > (uint32_t)R) { fault = JR_FAULT_PROGRESS_UNKNOWN_NODE; return false; }
    uint32_t i = node - 1;
    bool inc = false;
#pragma unroll
    for (int k = 0; k < R; ++k)
      if (k == (int)i && ph[k] < bid) { ph[k] = bid; inc = true; }
    prmask = inc ? (prmask | (1u << i)) : (prmask & ~(1u << i));  // Replicate iff incremented
    return true;
  }
  // progress.rs:48-60: heads sorted descending, element [R/2]
  __device__ __forceinline__ uint32_t committed_index() const {
    uint32_t v[R];
#pragma unroll
    for (int i = 0; i < R; ++i) v[i] = ph[i];
#pragma unroll
    for (int i = 0; i < R; ++i)
#pragma unroll
      for (int j = 0; j + 1 < R - i; ++j) {
        uint32_t a = v[j], b = v[j + 1];
        v[j] = max(a, b);
        v[j + 1] = min(a, b);
      }
    return v[R / 2];
  }

  // ------------------------------------------------------------------ transitions
  __device__ __forceinline__ void become_candidate() {  // follower.rs:285-304
    seen = granted = 0;
    nq = 0;      // Candidate { queued_reqs: Vec::new() }
    leader = 0;
    role = JR_ROLE_CANDIDATE;
  }
  __device__ __forceinline__ void candidate_to_follower() {  // candidate.rs:198-214
    leader = 0;
    role = JR_ROLE_FOLLOWER;
  }
  __device__ __forceinline__ void candidate_to_leader() {  // candidate.rs:216-238
#pragma unroll
    for (int i = 0; i < R; ++i) ph[i] = 0;
    prmask = 0;
    hbtime = now;
    nq = 0;
    role = JR_ROLE_LEADER;
  }

  // ------------------------------------------------------------------ follower.rs
  __device__ __forceinline__ void cmd_block(const Cmd& c, uint32_t k, uint32_t& bid, uint32_t& next, uint64_t& tok) const {
    if (c.host_msg) {
      bid = (uint32_t)c.host_msg->blocks[k].id;
      next = (uint32_t)c.host_msg->blocks[k].next;
      tok = c.host_msg->blocks[k].data;
    } else {
      uint4 u = inbox_unit(c.blk_s, c.blk_at + k);
      bid = u.x; next = u.y; tok = (uint64_t)u.z | ((uint64_t)u.w << 32);
    }
  }

  __device__ __forceinline__ void follower_append_entries(const Cmd& c) {  // follower.rs:130-176
    uint32_t ldr = c.node_id;
    if (voted == 0 && c.term >= term) {
      set_term(c.term);
      etime = now;  // timer restarted, timeout kept
      leader = ldr;
      voted = ldr;
    }
    if (voted != 0 && voted != ldr && c.term < term) { fault = JR_FAULT_AE_STALE_LEADER; return; }
    if (c.nblk) {
      for (uint32_t k = 0; k < c.nblk; ++k) {
        uint32_t bid, next; uint64_t tok;
        cmd_block(c, k, bid, next, tok);
        if (!chain_extend(bid, next, tok)) return;  // Err -> `?` -> node stops
      }
      send(JR_CMD_APPEND_RESPONSE, ldr, 1, 0, term, head);
    }
  }

  __device__ __forceinline__ void follower_heartbeat(const Cmd& c) {  // follower.rs:178-217
    uint32_t ldr = c.node_id;
    set_election_timeout();
    set_term(c.term);  // unconditional
    leader = ldr;
    voted = ldr;
    for (uint32_t q = 0; q < nq; ++q) {  // follower.rs:190-197
      uint4 e = d.qt[(size_t)q * plane + rg];
      send(JR_CMD_CLIENT_REQUEST, ldr, 0, 0, (uint64_t)e.x | ((uint64_t)e.y << 32), e.z);
      if (fault) return;
    }
    nq = 0;
    bool hasc = has(c.block);
    if (hasc && c.block > commit) {
      uint32_t prev = commit;
      chain_commit(c.block);
      for (uint32_t b = max(prev, tbase); b < c.block; ++b) {  // range(prev..commit), key order (nothing below the floor)
        uint32_t nx; uint64_t tk;
        tbl_fetch(b, nx, tk);
        if (nx != ABSENT) { fsm_emit(false, b, nx, tk); if (fault) return; }
      }
    }
    send(JR_CMD_HEARTBEAT_RESPONSE, ldr, hasc ? 1 : 0, 0, 0, commit);
  }

  __device__ __forceinline__ void follower_vote_request(const Cmd& c) {  // follower.rs:97-101,219-246
    bool can = !(voted != 0 || term > c.last_term || commit > c.block);
    send(JR_CMD_VOTE_RESPONSE, c.node_id, can ? 1 : 0, 0, term, 0);
    if (fault) return;
    if (can) voted = c.node_id;
  }

  __device__ __forceinline__ void follower_client_request(uint64_t tok) {  // follower.rs:258-269
    uint32_t addr = ((uint32_t)JR_ADDR_PEER << 16) | id();  // req.address = Peer(self.id)
    if (leader != 0) send(JR_CMD_CLIENT_REQUEST, leader, 0, 0, tok, addr);
    else queue_push(tok, addr);
  }

  // ------------------------------------------------------------------ candidate.rs
  // candidate.rs:91-113.  Returns through state: may become Leader (+ heartbeat) or Follower.
  __device__ __forceinline__ void candidate_vote_response(uint32_t from, bool g_) {
    vote(from, g_);
    int st = election_status();
    if (st == 0) {  // elect(): Raft::from(self) then heartbeat()
      candidate_to_leader();
      heartbeat();
    } else if (st == 2) {
      voted = 0;
      candidate_to_follower();
    }
  }

  __device__ __forceinline__ void candidate_vote_request(const Cmd& c) {  // candidate.rs:71-88
    if (c.term > term) {
      set_term(c.term);
      candidate_to_follower();
      return;
    }
    send(JR_CMD_VOTE_RESPONSE, c.node_id, 0, 0, term, 0);
  }

  __device__ __forceinline__ void candidate_heartbeat(const Cmd& c) {  // candidate.rs:137-157
    bool hasc = has(c.block);
    uint32_t own = commit;
    set_term(c.term);
    voted = c.node_id;
    candidate_to_follower();
    send(JR_CMD_HEARTBEAT_RESPONSE, c.node_id, hasc ? 1 : 0, 0, 0, own);
  }

  // ------------------------------------------------------------------ leader.rs
  __device__ __forceinline__ void heartbeat() {  // leader.rs:44-51
    send(JR_CMD_HEARTBEAT, TO_PEERS, 0, 0, term, commit);
  }

  __device__ __forceinline__ void leader_commit() {  // leader.rs:87-99
    // committed_index() is element [R/2] of the heads sorted descending; it exceeds
    // `commit` iff at least R/2+1 heads do.  Count first, sort only when it matters.
    int above = 0;
#pragma unroll
    for (int i = 0; i < R; ++i) above += ph[i] > commit ? 1 : 0;
    if (above < R / 2 + 1) return;
    uint32_t q = committed_index();
    if (q > commit) {
      uint32_t prev = commit;
      if (!chain_commit(q)) return;
      bool first = true;
      for (uint32_t b = max(prev, tbase); b <= q; ++b) {  // range(prev..=new).skip(1), key order (nothing below the floor)
        uint32_t nx; uint64_t tk;
        tbl_fetch(b, nx, tk);
        if (nx == ABSENT) continue;
        if (first) { first = false; continue; }
        fsm_emit(false, b, nx, tk);
        if (fault) return;
      }
    }
  }

  // leader.rs:124-174.  Probe: range(head..).nth(1); Replicate: range(head..).skip(1).take(5).
  __device__ __forceinline__ void replicate() {
    // Peers with the same progress head and mode get the same blocks (the steady
    // state: all of them).  The key-order scan runs once per distinct
    // (head, mode); repeats copy the block units already sitting in the outbox.
    uint32_t memo_head = 0xFFFFFFFFu, memo_take = 0, memo_first = 0, memo_nb = 0;
    JR_PROF_T0(tr);
    bool first_done = false;
    (void)first_done;
    uint32_t first_peer = 0xFFFFFFFFu;  // SORTED: the peer whose block run was scanned up front
    if constexpr (SORTED) {
      // Role-sorted warps hold leaders with DIFFERENT replica indices, so "the first peer" differs
      // per lane (index 1 for replica 0, else 0).  Scan its block run here, for all lanes at once;
      // the loop below then only writes headers.  Mailbox layout is identical to the plain path:
      // the first peer's header goes to slot ocnt, its blocks follow inline.
      if (R > 1) {
        first_peer = r == 0 ? 1u : 0u;
        const uint32_t take = (prmask >> first_peer) & 1u ? JR_MAX_AE_BLOCKS : 1u;
        const uint32_t head0 = get_ph(first_peer);
        uint32_t bid = max(head0, tbase), pulled = 0, nb = 0;
        while (pulled < 1 + take) {
          uint32_t nx = ABSENT; uint64_t tok = 0;
          while (bid <= maxkey) {
            tbl_fetch(bid, nx, tok);
            if (nx != ABSENT) break;
            ++bid;
          }
          if (bid > maxkey) {
            if ((d.flags & JR_F_SLED_COMMIT_KEY_STRICT) && ckey) { fault = JR_FAULT_RANGE_COMMIT_KEY; return; }
            break;
          }
          if (pulled >= 1) {
            if (!put_unit(ocnt + 1 + nb, make_uint4(bid, nx, (uint32_t)tok, (uint32_t)(tok >> 32)))) return;
            ++nb;
          }
          ++pulled;
          ++bid;
        }
        memo_head = head0; memo_take = take; memo_first = ocnt + 1; memo_nb = nb;
      }
    }
#pragma unroll
    for (int p = 0; p < R; ++p) {
      if (p == (int)r) continue;  // config.nodes holds peers only
#ifdef JR_PROFILE
      if (first_done) { JR_PROF_ADD(JR_ROLE_LEADER, 2, tr); first_done = false; }
#endif
      const uint32_t take = (prmask >> p) & 1u ? JR_MAX_AE_BLOCKS : 1u;
      uint32_t nb = 0, first = ocnt + 1;
      bool ref = false;
      if (ph[p] == memo_head && take == memo_take) {
        nb = memo_nb;       // same blocks as an earlier peer: point at that run
        first = memo_first;
        ref = (uint32_t)p != first_peer;  // (the peer scanned up front owns the inline run)
      } else {
        uint32_t bid = max(ph[p], tbase), pulled = 0;
        while (pulled < 1 + take) {
          uint32_t nx = ABSENT; uint64_t tok = 0;
          while (bid <= maxkey) {
            tbl_fetch(bid, nx, tok);
            if (nx != ABSENT) break;
            ++bid;
          }
          if (bid > maxkey) {
            // sled would now yield the "commit" key and bincode panics (D6)
            if ((d.flags & JR_F_SLED_COMMIT_KEY_STRICT) && ckey) { fault = JR_FAULT_RANGE_COMMIT_KEY; return; }
            break;
          }
          if (pulled >= 1) {
            if (!put_unit(ocnt + 1 + nb, make_uint4(bid, nx, (uint32_t)tok, (uint32_t)(tok >> 32)))) return;
            ++nb;
          }
          ++pulled;
          ++bid;
        }
        memo_head = ph[p]; memo_take = take; memo_first = ocnt + 1; memo_nb = nb;
#ifdef JR_PROFILE
        first_done = true;
#endif
      }
      if (!put_unit(ocnt, make_uint4(unit_hdr(JR_CMD_APPEND_ENTRIES, ref ? 1u : 0u, nb, p + 1), (uint32_t)term,
                                     (uint32_t)(term >> 32), first)))
        return;
      mko[p] |= ocnt < MK_SLOTS ? (1u << ocnt) : MK_SCAN;
      if (digest_on()) {
        uint4 v = d.dg[rg];
        uint64_t h = digest_message_fn((uint64_t)v.x | ((uint64_t)v.y << 32), JR_CMD_APPEND_ENTRIES, p + 1, 0, nb, id(), term, 0, 0, 0, 0);
        d.cn[rg].x += 1u;
        for (uint32_t k = 0; k < nb; ++k) {
          uint4 u = own_unit(first + k);
          h = fold(h, u.x);
          h = fold(h, u.y);
          h = fold(h, (uint64_t)u.z | ((uint64_t)u.w << 32));
        }
        v.x = (uint32_t)h; v.y = (uint32_t)(h >> 32);
        d.dg[rg] = v;
      }
      ocnt += ref ? 1u : 1u + nb;
    }
    JR_PROF_ADD(JR_ROLE_LEADER, 3, tr);
  }

  // ------------------------------------------------------------------ Apply::apply (mod.rs:471-479)
  // The state machine is split by role.  A Leader never changes role (leader.rs
  // has no transition out; a higher term panics, leader.rs:33-35), so once a
  // replica is Leader the rest of its tick runs in the leader loop; Follower and
  // Candidate share the other one.  Each handler is instantiated exactly once.
  // The heavy continuations the reference reaches from several places are shared
  // tails:
  //   timeout tail   = Raft<Follower>::apply_timeout -> seek_election (follower.rs:248-256, candidate.rs:24-45)
  //   advance tail   = ReplicationProgress::advance + Leader::commit (leader.rs:211-219, also 191-196)
  //   replicate tail = Leader::replicate (leader.rs:124-174, reached from 228 and 242)
  __device__ __forceinline__ void apply_fc(const Cmd& c) {  // follower.rs:38-63, candidate.rs:170-196
    bool t_timeout = false;
    if (role == JR_ROLE_FOLLOWER) {
      switch (c.kind) {
        case JR_CMD_TICK: t_timeout = needs_election(); break;  // follower.rs:121-128
        case JR_CMD_TIMEOUT: t_timeout = true; break;
        case JR_CMD_APPEND_ENTRIES: follower_append_entries(c); break;
        case JR_CMD_HEARTBEAT: follower_heartbeat(c); break;
        case JR_CMD_VOTE_REQUEST: follower_vote_request(c); break;
        case JR_CMD_CLIENT_REQUEST: follower_client_request(c.term); break;
        case JR_CMD_CLIENT_RESPONSE: send(JR_CMD_CLIENT_RESPONSE, TO_CLIENT, 0, 0, c.term, 0); break;  // follower.rs:271-282
        default: break;
      }
    } else {
      switch (c.kind) {
        case JR_CMD_TICK:  // candidate.rs:48-68
          if (needs_election()) {
            if (election_status() == 0) { fault = JR_FAULT_CANDIDATE_TICK_ELECTED; break; }
            voted = 0;
            candidate_to_follower();
            t_timeout = true;  // raft.apply(Command::Timeout) as a Follower
          }
          break;
        case JR_CMD_VOTE_REQUEST: candidate_vote_request(c); break;
        case JR_CMD_VOTE_RESPONSE: candidate_vote_response(c.node_id, c.flag != 0); break;
        case JR_CMD_APPEND_ENTRIES: if (c.term >= term) candidate_to_follower(); break;  // candidate.rs:116-134
        case JR_CMD_HEARTBEAT: candidate_heartbeat(c); break;
        case JR_CMD_CLIENT_REQUEST: queue_push(c.term, c.block); break;
        default: break;
      }
    }
    if (fault) return;
    if (t_timeout && voted == 0) {  // follower.rs:248-256
      set_election_timeout();
      become_candidate();
      // seek_election, candidate.rs:24-45
      voted = id();
      term += 1;
      // N-1 broadcasts of the same VoteRequest: one unit with aux = copies
      if (R > 1) send(JR_CMD_VOTE_REQUEST, TO_PEERS, 0, R - 1, term, head);
      if (fault) return;
      candidate_vote_response(id(), true);
    }
  }

  __device__ __forceinline__ void apply_leader(const Cmd& c) {  // leader.rs:248-266
    bool t_replicate = false, t_advance = false;
    uint32_t adv_node = 0, adv_block = 0;
    switch (c.kind) {
      case JR_CMD_APPEND_RESPONSE: t_advance = true; adv_node = c.node_id; adv_block = c.block; break;  // leader.rs:211-219
      case JR_CMD_HEARTBEAT_RESPONSE: t_replicate = !c.flag && c.block > 0; break;                     // leader.rs:222-231
      case JR_CMD_TICK: {  // leader.rs:234-245
        uint64_t el = now >= hbtime ? now - hbtime : 0;
        if (el > (uint64_t)d.hb) {
          heartbeat();
          hbtime = now;
        }
        t_replicate = true;
        break;
      }
      case JR_CMD_CLIENT_REQUEST: {  // leader.rs:177-197
        uint32_t bid;
        if (!chain_append(c.term, bid)) break;
        fsm_emit(true, bid, c.block, c.term);
        t_advance = true; adv_node = id(); adv_block = head;  // self AppendResponse
        break;
      }
      case JR_CMD_APPEND_ENTRIES: if (c.term > term) set_term(c.term); break;  // leader.rs:200-208
      default: break;
    }
    if (fault) return;
    if (t_advance) {
      if (progress_advance(adv_node, adv_block)) leader_commit();
    }
    if (t_replicate && !fault) replicate();
  }

  // Sparse / injected commands (inject kernel): pick the loop by current role.
  __device__ __forceinline__ void apply(const Cmd& c) {
    if (!live()) return;
    if (role == JR_ROLE_LEADER) apply_leader(c);
    else apply_fc(c);
  }

  // ------------------------------------------------------------------ the step schedule (jr_step_args)
  // One tick of this replica: peer mail (ascending sender, FIFO per sender) ->
  // dense proposal -> synthetic proposals -> Tick.  The three trailing sources
  // are virtual senders R, R+1, R+2.  `Pos` is the resumable position in that
  // schedule, so the follower/candidate loop can hand over to the leader loop in
  // the middle of a tick (the moment an election is won).
  struct Pos {
    uint32_t pend;   // peers (0..R-1) that still have something for me
    uint32_t s;      // sender being drained
    uint32_t idx;    // indexed delivery: my headers of sender s still to visit (0 = none)
    uint32_t u, cnt; // scan delivery (index overflow, or a virtual sender): units u..cnt of sender s
    uint32_t reps;   // copies of the current VoteRequest unit still to apply ...
    uint32_t rep_at; // ... and its slot (the unit is re-read, so no Cmd has to stay alive)
    uint32_t tail, tail_i;  // trailing schedule entries: see next_tail
  };

  // Which senders have mail for me this tick: one shared-memory read per peer, up front.
  __device__ __forceinline__ void plan_tick(Pos& k, const StepParams& p) const {
    k.pend = 0; k.s = 0; k.idx = 0; k.u = 0; k.cnt = 0; k.reps = 0; k.rep_at = 0;
    if (p.phases & PH_DRAIN) {
#pragma unroll
      for (int s_ = 0; s_ < R; ++s_)
        if (d.use_index ? (uint32_t)L.mk_in[(r * R + s_) * 32 + L.lane] : L.cin[s_ * 32 + L.lane]) k.pend |= 1u << s_;
      k.pend &= ~(1u << r);  // never my own mailbox
    }
    k.tail = 0;
  }

  // The trailing schedule entries need no mailbox: dense proposal (stage 0), synthetic
  // proposals to a Leader (stage 1, `tail_i` counts them), Tick (stage 2).
  __device__ __forceinline__ bool next_tail(Pos& k, const StepParams& p, Cmd& c) const {
    const uint32_t me = id();
    c.flag = 0; c.node_id = 0; c.nblk = 0; c.last_term = 0; c.blk_s = 0; c.blk_at = 0;
    if (k.tail == 0) {  // event_loop client arm, server.rs:156-160
      k.tail = 1;
      k.tail_i = 0;
      if ((p.phases & PH_PROPOSE) && (p.proposals || p.tok_runs) && g < d.G) {
        uint4 pr;
        if (p.tok_runs) {   // run-length input: the token is base + tick * stride
          const uint4 rn = __ldg(p.tok_runs + g);
          const uint64_t base = (uint64_t)rn.x | ((uint64_t)rn.y << 32);
          const uint64_t tok = base + (uint64_t)p.tok_tick * ((uint64_t)rn.z | ((uint64_t)rn.w << 32));
          pr = make_uint4((uint32_t)tok, (uint32_t)(tok >> 32), base ? __ldg(p.tok_route + g) : 0u, 0u);
        } else {
          pr = __ldg(reinterpret_cast<const uint4*>(p.proposals) + g);
        }
        if (pr.z == me) {
          c.kind = JR_CMD_CLIENT_REQUEST; c.block = (uint32_t)JR_ADDR_CLIENT << 16;
          c.term = (uint64_t)pr.x | ((uint64_t)pr.y << 32);
          return true;
        }
      }
    }
    if (k.tail == 1) {
      if ((p.phases & PH_PROPOSE) && k.tail_i < p.n_synth && role == JR_ROLE_LEADER) {
        c.kind = JR_CMD_CLIENT_REQUEST; c.block = (uint32_t)JR_ADDR_CLIENT << 16;
        c.term = synth_token(p.step_index, k.tail_i, d.goff + g);
        ++k.tail_i;
        return true;
      }
      k.tail = 2;
    }
    if (k.tail == 2) {
      k.tail = 3;
      if (p.phases & PH_TICK) { c.kind = JR_CMD_TICK; c.block = 0; c.term = 0; return true; }
    }
    return false;
  }

  // Next command addressed to this replica, or false when the schedule is exhausted.
  __device__ __forceinline__ bool next_cmd(Pos& k, const StepParams& p, Cmd& c) {
    const uint32_t me = id();
    uint4 h;
    uint32_t at = 0;
    bool again = false;
    for (;;) {
      if (k.reps) {  // another copy of the same VoteRequest broadcast: re-read the unit
        --k.reps;
        at = k.rep_at;
        h = inbox_unit(k.s, at);
        again = true;
        break;
      }
      if (k.idx) {  // indexed delivery: jump to my next header of sender s
        at = (uint32_t)__ffs((int)k.idx) - 1u;
        k.idx &= k.idx - 1u;
        h = inbox_unit(k.s, at);
        break;
      }
      if (k.u < k.cnt) {  // scan delivery (the sender's index overflowed)
        at = k.u;
        h = inbox_unit(k.s, k.u);
        const uint32_t k0 = h.x & 15u, to = h.x >> 16;
        k.u += 1u + ((k0 == JR_CMD_APPEND_ENTRIES && !((h.x >> 4) & 1u)) ? ((h.x >> 8) & 255u) : 0u);
        if (to != TO_PEERS && to != me) continue;
        break;
      }
      if (!k.pend) return next_tail(k, p, c);  // peers exhausted: proposals, then Tick
      k.s = (uint32_t)__ffs((int)k.pend) - 1u;
      k.pend &= k.pend - 1u;
      k.u = 0; k.cnt = 0;
      const uint32_t m = d.use_index ? L.mk_in[(r * R + k.s) * 32 + L.lane] : MK_SCAN;
      if (m & MK_SCAN) k.cnt = L.cin[k.s * 32 + L.lane];
      else k.idx = m;
    }
    const uint32_t kind = h.x & 15u, aux = (h.x >> 8) & 255u;
    c.kind = kind; c.flag = (h.x >> 4) & 1u; c.node_id = k.s + 1; c.nblk = aux; c.block = h.w;
    c.term = (uint64_t)h.y | ((uint64_t)h.z << 32); c.last_term = c.term;
    c.blk_s = k.s;
    c.blk_at = (kind == JR_CMD_APPEND_ENTRIES && c.flag) ? h.w : at + 1;
    // N-1 identical VoteRequest broadcasts travel as one unit (candidate.rs:30-37)
    if (!again && kind == JR_CMD_VOTE_REQUEST && aux > 1u) { k.reps = aux - 1u; k.rep_at = at; }
    return true;
  }

  __device__ __forceinline__ void run_step(const StepParams& p) {
    Pos k;
    plan_tick(k, p);
    Cmd c;
    c.host_msg = nullptr;
    bool more = live();
    while (more) {
      JR_PROF_T0(tp);
      if (role == JR_ROLE_LEADER) {
        // Steady-state fast drain: a peer whose only dispatchable mail is ONE AppendResponse
        // (its HeartbeatResponse{has} is a no-op and not indexed).  Same effect as the generic
        // path below -- ReplicationProgress::advance + Leader::commit, leader.rs:211-219 --
        // without the generic fetch/dispatch.  Senders are taken in ascending order and the
        // drain stops at the first one that does not fit, so delivery order is unchanged.
        if (d.use_index && k.idx == 0 && k.u >= k.cnt && k.reps == 0) {
          const uint32_t real = k.pend & ((1u << R) - 1u);
          // all peers' delivery masks, then all candidate units: independent loads, one latency each
          uint32_t m[R], w[R];
#pragma unroll
          for (int s_ = 0; s_ < R; ++s_) m[s_] = ((real >> s_) & 1u) ? L.mk_in[(r * R + s_) * 32 + L.lane] : 0u;
          uint32_t okm = 0;
#pragma unroll
          for (int s_ = 0; s_ < R; ++s_) {
            const bool single = m[s_] != 0u && !(m[s_] & MK_SCAN) && !(m[s_] & (m[s_] - 1u));
            uint4 h = make_uint4(0, 0, 0, 0);
            if (single) h = inbox_unit(s_, (uint32_t)__ffs((int)m[s_]) - 1u);
            w[s_] = h.w;
            if (single && (h.x & 15u) == JR_CMD_APPEND_RESPONSE) okm |= 1u << s_;
          }
          // ascending sender order: only the senders below the first one that does not fit
          JR_PROF_ADD(JR_ROLE_LEADER, 8, tp);   // profile: drain loads
          const uint32_t bad = real & ~okm;
          uint32_t elig = bad ? (okm & ((bad & (0u - bad)) - 1u)) : okm;
          int above = 0;
#pragma unroll
          for (int i = 0; i < R; ++i) above += ph[i] > commit ? 1 : 0;
          while (elig && live()) {
            bool trig = false;
#pragma unroll
            for (int s_ = 0; s_ < R; ++s_) {
              if (!trig && ((elig >> s_) & 1u)) {  // ReplicationProgress::advance, progress.rs:42-46,76-94,133-140
                const uint32_t v = w[s_];
                const bool inc = ph[s_] < v;
                if (inc && ph[s_] <= commit && v > commit) ++above;
                if (inc) ph[s_] = v;
                prmask = inc ? (prmask | (1u << s_)) : (prmask & ~(1u << s_));
                elig &= ~(1u << s_);
                k.pend &= ~(1u << s_);
                trig = above >= R / 2 + 1;  // committed_index() > commit: Leader::commit acts (leader.rs:87-99)
              }
            }
            if (trig) {
              JR_PROF_ADD(JR_ROLE_LEADER, 9, tp);  // profile: drain advances
              leader_commit();
              JR_PROF_ADD(JR_ROLE_LEADER, 1, tp);  // profile: Leader::commit
              above = 0;
#pragma unroll
              for (int i = 0; i < R; ++i) above += ph[i] > commit ? 1 : 0;
            }
          }
          JR_PROF_ADD(JR_ROLE_LEADER, 11, tp);
        }
        // leader loop: runs to the end of the tick
        while (live() && next_cmd(k, p, c)) {
          JR_PROF_ADD(JR_ROLE_LEADER, 14, tp);
          apply_leader(c);
          JR_PROF_ADD(JR_ROLE_LEADER, c.kind, tp);
        }
        more = false;
      } else {
        // follower / candidate loop: leaves when the replica wins an election
        more = false;
        while (live() && next_cmd(k, p, c)) {
          JR_PROF_ADD(JR_ROLE_FOLLOWER, 14, tp);
          apply_fc(c);
          JR_PROF_ADD(JR_ROLE_FOLLOWER, c.kind, tp);
          if (role == JR_ROLE_LEADER) { more = live(); break; }
        }
      }
    }
  }
};
#undef seen
#undef granted
#undef leader

#endif  // JR_DEVICE_CODE
}  // namespace jr
