// sym_fold.cuh -- the symmetric-group fold: a whole fused launch of a group in TWO lanes (sym2_kernel).
//
// In a healthy group every follower is in the same state: same term, same head and commit, the same mail from the
// leader in flight, and the leader holds the same progress entry for each of them.  R-1 replicas then make the same
// decisions on the same data, tick after tick.  This kernel exploits that symmetry exactly, not approximately:
// the leader's state and ONE follower state that stands for all R-1 followers, the mail between them in its canonical
// shapes (listed below), and the very handlers of raft_device.cuh -- restated here for scalar operands, each citing
// the same reference lines -- for all n ticks of the launch.  No mailboxes in HBM, no divergence between roles; what
// is left is the data that really has to move: the proposal tokens in, the block-table rows of every replica and the
// Instruction stream out.  sym2_kernel runs the two sides in two lanes of two warps (within a tick they only depend on
// the previous tick's mail), with the mail, the row caches and the Instruction encoders in shared memory and one
// barrier per tick.
//
// Exactness contract:
//   * It FIRST CHECKS that a group is symmetric, that its followers' tables agree over every id the launch can read,
//     and that its mail in flight has the canonical shapes (sym_enter); every other group is left to step_kernel
//     untouched.
//   * If anything outside the canonical evolution would happen during the launch (a fault, an election timer that
//     could fire, a HeartbeatResponse{has_committed: false}, a read below the compared rows, ...) the lane ABORTS
//     (tells the other lane through the mail, and both check the other's last mail after the last barrier): it has
//     only written block-table rows and Instruction records beyond the FIFO counters, which
//     step_kernel writes identically when it re-runs the group from the untouched state planes -- an abort costs time,
//     never correctness.
//   * On success the replicas' state planes, progress planes and the mailboxes of the last tick are written in the
//     exact unit layout step_kernel produces, and the Instruction streams leave through the same streaming encoder
//     fsm_flush uses (fsm_enc_push), fed as the Instructions are produced.
//   * Stream digests (JR_F_STREAM_DIGEST) need every Message in order, which this path never materialises: engines
//     created with that flag, or with JR_F_SLED_COMMIT_KEY_STRICT / JR_F_NO_SYMMETRIC_FOLD, never take it.
//     tests/test_sym_fold.py compares folded runs with step_kernel runs and with the oracle through everything else:
//     replica state, block tables, leader tables, Instruction streams -- scenario by scenario and over random scripts.
//
// Canonical mail (all that can be in flight in a symmetric group):
//   leader -> each follower, in this order:  [Heartbeat{term, commit}]  [AppendEntries{term, <= 5 blocks}]
//   each follower -> leader, in this order:  [HeartbeatResponse{commit, has}]  [AppendResponse{term, head}]
#pragma once
#include "raft_device.cuh"

namespace jr {
#ifdef JR_DEVICE_CODE

struct SymMail {
  uint32_t hb, hb_commit;                 // leader -> followers
  uint32_t ae, ae_nb, ae_id[JR_MAX_AE_BLOCKS];
  uint32_t mk;                            // the leader's largest block id when it sent this (which cache slots it may be rewriting)
  uint32_t hbr, hbr_commit, hbr_has;      // followers -> leader
  uint32_t ar, ar_head;
};

// Block-table rows the fold has touched recently, per lane, in SHARED memory: two direct-mapped caches (the leader's
// table, the followers' identical tables) of SYM_ROWS entries {id, next, token}, laid out [cache][slot][lane] so that a
// lane's access is one conflict-free 128-bit LDS/STS.  Everything a steady group reads was written a few ticks ago, so
// after the fill at entry no table READ leaves the SM (rows are still written through to HBM).  (A register shift
// register cost ~400 instructions per tick in compare/select chains; local-memory arrays were slower still.)
constexpr uint32_t SYM_ROWS = 8;
// The Instruction streams are encoded AS THEY ARE PRODUCED, by the same streaming encoder fsm_flush uses (fsm_enc_push):
// its state is parked in shared memory between two Instructions, [slot][lane] like the row caches.  (The raw FIFO +
// fsm_flush round trip of step_kernel cost this kernel a quarter of its instructions and half of its DRAM traffic.)
//   leader    e0 = {nrec, seq0, wseq, pb2}  e1 = {pb0, pb1}  e2 = {ra.next_id, ra.count, ra.last}
//             e3 = {ra.stride, rn.stride}   e4 = {rn.next_id, rn.count, rn.last}
//   followers f0 = {nrec, seq0, wseq, -}    f1 = {ra.next_id, ra.count, ra.last}   f2 = {ra.stride, -}   (no Notify: pb = 0)
// seq = seq0 + the lane's Instruction counter (lcnt / fcnt), which lives in a register anyway.
constexpr uint32_t SYM_ENC_L = 5, SYM_ENC_F = 3;
constexpr uint32_t SYM_SMEM_UNITS = 2 * SYM_ROWS + SYM_ENC_L + SYM_ENC_F;   // uint4 per lane
// TWO lanes per group, in two warps of the same CTA -- one runs the leader's handlers, the other the
// followers' -- because within a tick the two sides only depend on the mail of the PREVIOUS tick.  The kernel is latency
// bound with 3.5 warps per SM sub-partition; this doubles the warps and halves each warp's serial chain.  The mail goes
// through shared memory, double buffered, one __syncthreads() per tick:
//   leader -> followers   A = {hb | ae << 1 | nb << 4 | abort << 8 | ids << 9 | mode << 10, commit, leader's max key, id0 / progress head}
//                         B = {id1 .. id4}   (ids = 1: the AppendEntries' blocks are listed -- the mail sym_enter found in
//                         flight; ids = 0: the follower lane derives them, see replicate())
//   followers -> leader   C = {hbr | has << 1 | ar << 2 | abort << 8, hbr_commit, ar_head, -}
constexpr uint32_t SYM2_GROUPS = 64;                                        // groups per CTA: 128 threads
// CTAs per SM the launch bounds ask for: all 1,024 CTAs of 65,536 groups must be resident at once (a second wave would
// double the time), so 7 per SM on 148 SMs, which holds the kernel to 72 registers per thread.
constexpr int SYM2_MINCTAS = 7;
constexpr uint32_t SYM2_UNITS = SYM_SMEM_UNITS + 2 * 2 + 2 * 1;            // uint4 per group
constexpr uint32_t SYM2_ABORT = 1u << 8, SYM2_IDS = 1u << 9, SYM2_MODE = 1u << 10;

template <int R>
struct SymGroup {
  static constexpr uint32_t STRIDE = SYM2_GROUPS;   // columns of the CTA's per-group shared memory
  const Dev& d;
  const uint32_t g;
  const size_t plane;
  uint32_t L;                              // leader's replica index
  uint32_t F0;                             // lowest follower index: its block table stands for every follower's
  uint64_t term, hbtime, now;
  uint32_t head, commit, idgen, maxkey, ckey, ph_self, mode_self, ph_f, mode_f;   // leader
  uint32_t fhead, fcommit, fmaxkey, fckey;                                        // every follower
  uint32_t n_hb;                           // heartbeats the followers took in this launch
  uint64_t last_hb;
  uint32_t tbase;
  uint32_t flo;                            // lowest id whose row sym_enter found identical in every follower
  uint4* rows;                             // this lane's column of the CTA's row caches (see above)
  uint4* enc;                              // this lane's column of the encoder states (see above)
  uint32_t lcnt, fcnt;                     // raw Instructions emitted: leader / each follower
  uint32_t n_app;                          // most blocks the leader can append in one tick (dense + synthetic proposals)
  bool abort;
  bool share;                              // the followers' Instruction FIFOs are all empty: their records can be shared

  __device__ __forceinline__ SymGroup(const Dev& dv, uint32_t g_) : d(dv), g(g_), plane((size_t)R * dv.Gp) {}
  __device__ __forceinline__ size_t rg(uint32_t r) const { return (size_t)r * d.Gp + g; }
  __device__ __forceinline__ size_t row(uint32_t r, uint32_t bid) const { return (size_t)(bid & d.capm) * plane + rg(r); }
  __device__ __forceinline__ bool in_window(uint32_t bid) const { return bid - tbase < d.cap; }   // (sym_enter made sure ids stay below 2^31)
  __device__ __forceinline__ uint4& slot(uint32_t r, uint32_t bid) const { return rows[((r == L ? 0u : SYM_ROWS) + (bid % SYM_ROWS)) * STRIDE]; }
  __device__ __forceinline__ void cache_put(uint32_t r, uint32_t bid, uint32_t nx, uint64_t tk) const {
    slot(r, bid) = make_uint4(bid, nx, (uint32_t)tk, (uint32_t)(tk >> 32));
  }
  // r is the leader (its own table) or F0 (the followers' table)
  __device__ __forceinline__ void fetch(uint32_t r, uint32_t bid, uint32_t& next, uint64_t& tok) {
    if (!in_window(bid)) { next = ABSENT; tok = 0; return; }
    const uint4 e = slot(r, bid);
    if (e.x == bid) { next = e.y; tok = (uint64_t)e.z | ((uint64_t)e.w << 32); return; }
    next = __ldcg(d.cnext + row(r, bid));   // rows written earlier in this launch by this lane: read them at L2
    tok = __ldcg(d.ctok + row(r, bid));     // (a miss does not fill: a cache is only written at entry and by appends, see fetch_sent)
  }
  // Follower lane: a block the leader sent one tick ago, read from the LEADER's row cache, which the leader lane is
  // appending to right now.  Its appends of this tick are the ids (mk_sent, mk_sent + n_app]; a slot one of them maps to
  // is not read (the row is in global memory, written before the last barrier).  No other write happens to that cache
  // after entry, so every slot this reads is quiescent.
  __device__ __forceinline__ void fetch_sent(uint32_t bid, uint32_t mk_sent, uint32_t n_app, uint32_t& next, uint64_t& tok) {
    if (!in_window(bid)) { next = ABSENT; tok = 0; return; }
    if (bid + SYM_ROWS > mk_sent + n_app) {
      const uint4 e = slot(L, bid);
      if (e.x == bid) { next = e.y; tok = (uint64_t)e.z | ((uint64_t)e.w << 32); return; }
    }
    next = __ldcg(d.cnext + row(L, bid));
    tok = __ldcg(d.ctok + row(L, bid));
  }
  __device__ __forceinline__ void cache_clear(uint32_t first = 0, uint32_t n = 2 * SYM_ROWS) const {
#pragma unroll
    for (uint32_t k = 0; k < 2 * SYM_ROWS; ++k)
      if (k >= first && k < first + n) rows[k * STRIDE] = make_uint4(ABSENT, ABSENT, 0u, 0u);   // tag ABSENT matches no id
  }
  __device__ __forceinline__ void cache_fill(uint32_t r, uint32_t top) const {   // independent loads, issued together
    uint32_t nx[SYM_ROWS];
    uint64_t tk[SYM_ROWS];
#pragma unroll
    for (uint32_t j = 0; j < SYM_ROWS; ++j)
      if (j <= top && in_window(top - j)) {
        nx[j] = d.cnext[row(r, top - j)];
        tk[j] = d.ctok[row(r, top - j)];
      }
#pragma unroll
    for (uint32_t j = 0; j < SYM_ROWS; ++j)
      if (j <= top && in_window(top - j)) cache_put(r, top - j, nx[j], tk[j]);
  }
  __device__ __forceinline__ bool has(uint32_t r, uint32_t bid) {
    uint32_t n; uint64_t t;
    fetch(r, bid, n, t);
    return n != ABSENT;
  }
  // The followers' table, read through the lowest follower's: only rows sym_enter compared across followers (>= flo),
  // rows this launch wrote to all of them, or ids below the floor (absent everywhere) may be answered that way.
  __device__ __forceinline__ void fetch_f(uint32_t bid, uint32_t& next, uint64_t& tok) {
    if (in_window(bid) && bid < flo) { abort = true; next = ABSENT; tok = 0; return; }
    fetch(F0, bid, next, tok);
  }
  __device__ __forceinline__ bool has_f(uint32_t bid) {
    uint32_t n; uint64_t t;
    fetch_f(bid, n, t);
    return n != ABSENT;
  }

  // fsm_tx.send (fsm.rs:19-29)
  __device__ __forceinline__ uint4& eq(uint32_t k) const { return enc[k * STRIDE]; }
  __device__ __forceinline__ FsmOut leader_out() const { return FsmOut{d.fs + rg(L), plane, d.F, g, L}; }
  __device__ __forceinline__ FsmOut followers_out() const {   // one set of records for all followers: node mask in the APPLY records
    return FsmOut{d.fs + rg(F0), plane, d.F, g, F0, ((1u << R) - 1u) & ~(1u << L)};
  }
  __device__ __forceinline__ void enc_init_leader(uint2 leader_fc) const {
    eq(0) = make_uint4(leader_fc.x, leader_fc.y, leader_fc.y, 0u);
#pragma unroll
    for (uint32_t k = 1; k < SYM_ENC_L; ++k) eq(k) = make_uint4(0u, 0u, 0u, 0u);
  }
  __device__ __forceinline__ void enc_init_followers() const {
#pragma unroll
    for (uint32_t k = SYM_ENC_L; k < SYM_ENC_L + SYM_ENC_F; ++k) eq(k) = make_uint4(0u, 0u, 0u, 0u);
  }
  template <bool NOTIFY>
  __device__ __forceinline__ void emit_leader(uint32_t bid, uint32_t nxa, uint64_t tok) {
    if (!(d.flags & JR_F_CAPTURE_FSM)) return;
    if (lcnt >= d.Fr) { abort = true; return; }          // step_kernel's raw FIFO would overflow (it drops and counts): its business
    FsmEnc e;
    const uint4 q0 = eq(0);
    e.nrec = q0.x; e.seq = q0.y + lcnt; e.wseq = q0.z; e.pb2 = q0.w;
    ++lcnt;
    const bool window = NOTIFY || e.seq + 1u - e.wseq == FS_PATTERN_BITS;   // pattern words: read by a Notify and when the window closes
    uint4 q1 = make_uint4(0u, 0u, 0u, 0u);
    if (window) q1 = eq(1);
    e.pb0 = (uint64_t)q1.x | ((uint64_t)q1.y << 32);
    e.pb1 = (uint64_t)q1.z | ((uint64_t)q1.w << 32);
    const uint4 qr = eq(NOTIFY ? 4 : 2), qs = eq(3);
    FsmRun& run = NOTIFY ? e.rn : e.ra;
    run.next_id = qr.x; run.count = qr.y;
    run.last = (uint64_t)qr.z | ((uint64_t)qr.w << 32);
    run.stride = NOTIFY ? ((uint64_t)qs.z | ((uint64_t)qs.w << 32)) : ((uint64_t)qs.x | ((uint64_t)qs.y << 32));
    fsm_enc_push<NOTIFY>(e, leader_out(), bid, nxa, tok);
    if (e.nrec != q0.x || e.wseq != q0.z || e.pb2 != q0.w) eq(0) = make_uint4(e.nrec, q0.y, e.wseq, e.pb2);
    if (window) eq(1) = make_uint4((uint32_t)e.pb0, (uint32_t)(e.pb0 >> 32), (uint32_t)e.pb1, (uint32_t)(e.pb1 >> 32));
    eq(NOTIFY ? 4 : 2) = make_uint4(run.next_id, run.count, (uint32_t)run.last, (uint32_t)(run.last >> 32));
    uint2* st = reinterpret_cast<uint2*>(&eq(3)) + (NOTIFY ? 1 : 0);
    *st = make_uint2((uint32_t)run.stride, (uint32_t)(run.stride >> 32));
  }
  __device__ __forceinline__ uint2 leader_end() {          // close the leader's runs: its new {records, Instructions}
    FsmEnc e;
    const uint4 q0 = eq(0), q1 = eq(1), q2 = eq(2), q3 = eq(3), q4 = eq(4);
    e.nrec = q0.x; e.seq = q0.y + lcnt; e.wseq = q0.z; e.pb2 = q0.w;
    e.pb0 = (uint64_t)q1.x | ((uint64_t)q1.y << 32);
    e.pb1 = (uint64_t)q1.z | ((uint64_t)q1.w << 32);
    e.ra = FsmRun{q2.x, q2.y, (uint64_t)q2.z | ((uint64_t)q2.w << 32), (uint64_t)q3.x | ((uint64_t)q3.y << 32)};
    e.rn = FsmRun{q4.x, q4.y, (uint64_t)q4.z | ((uint64_t)q4.w << 32), (uint64_t)q3.z | ((uint64_t)q3.w << 32)};
    return fsm_enc_end(e, leader_out());
  }
  __device__ __forceinline__ void emit_followers(uint32_t bid, uint32_t next, uint64_t tok) {
    if (!(d.flags & JR_F_CAPTURE_FSM)) return;
    if (fcnt >= d.Fr) { abort = true; return; }
    if (share) {                                           // encoded once, for all followers
      FsmEnc e;
      const uint4 q0 = eq(SYM_ENC_L), q1 = eq(SYM_ENC_L + 1);
      const uint2 q2 = *reinterpret_cast<const uint2*>(&eq(SYM_ENC_L + 2));
      e.nrec = q0.x; e.seq = q0.y + fcnt; e.wseq = q0.z; e.pb2 = 0;
      e.pb0 = e.pb1 = 0;
      e.ra = FsmRun{q1.x, q1.y, (uint64_t)q1.z | ((uint64_t)q1.w << 32), (uint64_t)q2.x | ((uint64_t)q2.y << 32)};
      fsm_enc_push<false>(e, followers_out(), bid, next, tok);
      if (e.nrec != q0.x || e.wseq != q0.z) eq(SYM_ENC_L) = make_uint4(e.nrec, q0.y, e.wseq, 0u);
      eq(SYM_ENC_L + 1) = make_uint4(e.ra.next_id, e.ra.count, (uint32_t)e.ra.last, (uint32_t)(e.ra.last >> 32));
      *reinterpret_cast<uint2*>(&eq(SYM_ENC_L + 2)) = make_uint2((uint32_t)e.ra.stride, (uint32_t)(e.ra.stride >> 32));
    } else {                                               // followers with records pending: raw entries, fsm_flush at the end
      const uint4 e = make_uint4(bid, next, (uint32_t)tok, (uint32_t)(tok >> 32));
#pragma unroll
      for (int r = 0; r < R; ++r)
        if ((uint32_t)r != L) d.fr[(size_t)fcnt * plane + rg(r)] = e;
    }
    ++fcnt;
  }
  __device__ __forceinline__ uint2 followers_end() {
    FsmEnc e;
    const uint4 q0 = eq(SYM_ENC_L), q1 = eq(SYM_ENC_L + 1), q2 = eq(SYM_ENC_L + 2);
    e.nrec = q0.x; e.seq = q0.y + fcnt; e.wseq = q0.z; e.pb2 = 0;
    e.pb0 = e.pb1 = 0;
    e.ra = FsmRun{q1.x, q1.y, (uint64_t)q1.z | ((uint64_t)q1.w << 32), (uint64_t)q2.x | ((uint64_t)q2.y << 32)};
    e.rn = FsmRun{0, 0, 0, 0};
    return fsm_enc_end(e, followers_out());
  }

  // ---- leader (leader.rs) ------------------------------------------------------------------------------------
  // progress.rs:48-60 over {ph_self, n_new x v_new, (R-1-n_new) x v_old}: heads sorted descending, element [R/2]
  __device__ __forceinline__ uint32_t committed_index(uint32_t v_new, uint32_t n_new, uint32_t v_old) const {
    uint32_t v[R];
    v[0] = ph_self;
#pragma unroll
    for (int i = 1; i < R; ++i) v[i] = (uint32_t)i <= n_new ? v_new : v_old;
#pragma unroll
    for (int i = 0; i < R; ++i)
#pragma unroll
      for (int j = 0; j + 1 < R - i; ++j) {
        const uint32_t a = v[j], b = v[j + 1];
        v[j] = max(a, b);
        v[j + 1] = min(a, b);
      }
    return v[R / 2];
  }
  // leader.rs:87-99 with the current heads
  __device__ __forceinline__ void leader_commit(uint32_t v_new, uint32_t n_new, uint32_t v_old) {
    // committed_index() exceeds `commit` iff at least R/2+1 heads do: count first, sort only when it matters
    const uint32_t above = (ph_self > commit ? 1u : 0u) + (v_new > commit ? n_new : 0u) + (v_old > commit ? (uint32_t)(R - 1) - n_new : 0u);
    if (above < (uint32_t)(R / 2 + 1)) return;
    const uint32_t q = committed_index(v_new, n_new, v_old);
    if (q <= commit) return;
    if (!has(L, q)) { abort = true; return; }           // chain.rs:197-202 would panic
    const uint32_t prev = commit;
    ckey = 1;
    commit = q;
    bool first = true;
    for (uint32_t b = max(prev, tbase); b <= q; ++b) {   // range(prev..=new).skip(1), key order
      uint32_t nx; uint64_t tk;
      fetch(L, b, nx, tk);
      if (nx == ABSENT) continue;
      if (first) { first = false; continue; }
      emit_leader<false>(b, nx, tk);
    }
  }
  // leader.rs:177-197
  __device__ __forceinline__ void client_request(uint64_t tok) {
    const uint32_t bid = idgen++;
    if (!(bid > head) || !in_window(bid)) { abort = true; return; }   // chain.rs:163 / engine window: a fault -> step_kernel's business
    d.cnext[row(L, bid)] = head;
    d.ctok[row(L, bid)] = tok;
    cache_put(L, bid, head, tok);
    if (bid > maxkey) maxkey = bid;
    head = bid;
    emit_leader<true>(bid, FSR_CLIENT, tok);
    mode_self = ph_self < head ? 1u : 0u;               // progress.rs:76-94 on the leader's own entry
    if (ph_self < head) ph_self = head;
    leader_commit(ph_f, R - 1, ph_f);
  }

  __device__ __forceinline__ void leader_tick(const SymMail& in, SymMail& out, uint64_t dense_tok, uint32_t n_synth,
                                              uint64_t step_index) {
    // peer mail, ascending sender, FIFO per sender: every follower sent the same [HeartbeatResponse][AppendResponse]
    if (in.hbr && !in.hbr_has && in.hbr_commit > 0) { abort = true; return; }   // leader.rs:222-231 would replicate mid-drain
    if (in.ar) {
      const uint32_t old = ph_f, v = in.ar_head;
      const bool inc = old < v;                          // progress.rs:133-140, the same for every follower
      const uint32_t nw = inc ? v : old;
      for (uint32_t j = 1; j <= (uint32_t)(R - 1) && !abort; ++j) leader_commit(nw, j, old);   // leader.rs:211-219 after each response
      ph_f = nw;
      mode_f = inc ? 1u : 0u;
      if (abort) return;
    }
    // client arm, server.rs:156-160: the dense proposal, then the synthetic ones
    if (dense_tok) client_request(dense_tok);
    for (uint32_t i = 0; i < n_synth && !abort; ++i) client_request(synth_token(step_index, i, d.goff + g));
    if (abort) return;
    // Command::Tick, leader.rs:234-245
    const uint64_t el = now >= hbtime ? now - hbtime : 0;
    if (el > (uint64_t)d.hb) {
      out.hb = 1;
      out.hb_commit = commit;
      hbtime = now;
    }
    out.ae = 1;                                            // replicate() follows: one AppendEntries per peer
    out.mk = maxkey;
  }
  // replicate, leader.rs:124-174: Probe -> range(head..).nth(1); Replicate -> range(head..).skip(1).take(5), over the
  // leader's table as it stood when its largest key was `mk`.  Within the launch the FOLLOWER lane runs this scan at the
  // start of the next tick (follower_tick_view), from the {progress head, mode, max key} the leader lane put in its mail
  // -- the same rows, read through fetch_sent, the same blocks; it takes a sixth of the leader's chain off the critical
  // lane.  The leader lane runs it once itself, after the last tick, for the outbox the launch leaves behind.
  __device__ __forceinline__ void replicate(uint32_t phf, uint32_t modef, uint32_t mk, SymMail& out) {
    const uint32_t take = modef ? JR_MAX_AE_BLOCKS : 1u;
    uint32_t bid = max(phf, tbase), pulled = 0, nb = 0;
    while (pulled < 1 + take) {
      uint32_t nx = ABSENT; uint64_t tk = 0;
      while (bid <= mk) {
        fetch(L, bid, nx, tk);
        if (nx != ABSENT) break;
        ++bid;
      }
      if (bid > mk) break;
      if (pulled >= 1) out.ae_id[nb++] = bid;
      ++pulled;
      ++bid;
    }
    out.ae_nb = nb;
  }

  // ---- follower (follower.rs), once for all R-1 of them ----------------------------------------------------------
  __device__ __forceinline__ void follower_heartbeat(const SymMail& in, SymMail& out) {   // follower.rs:178-217
    ++n_hb;                                                // set_election_timeout: one RNG draw, timer restarted
    last_hb = now;
    const uint32_t c = in.hb_commit;
    const bool hasc = has_f(c);
    if (hasc && c > fcommit) {
      const uint32_t prev = fcommit;
      fckey = 1;
      fcommit = c;
      for (uint32_t b = max(prev, tbase); b < c; ++b) {    // range(prev..commit), key order
        uint32_t nx; uint64_t tk;
        fetch_f(b, nx, tk);
        if (nx != ABSENT) emit_followers(b, nx, tk);
      }
    }
    out.hbr = 1;
    out.hbr_commit = fcommit;
    out.hbr_has = hasc ? 1u : 0u;
  }
  // one block of an AppendEntries, applied by every follower (follower.rs:156-173 -> chain.rs:180-190)
  __device__ __forceinline__ void follower_extend(uint32_t bid, uint32_t nx, uint64_t tk) {
    if (nx == ABSENT || !has_f(nx) || !in_window(bid)) { abort = true; return; }   // chain.rs:180-185 Err / window: step_kernel's business
#pragma unroll
    for (int r = 0; r < R; ++r)
      if ((uint32_t)r != L) {
        d.cnext[row(r, bid)] = nx;
        d.ctok[row(r, bid)] = tk;
      }
    cache_put(F0, bid, nx, tk);
    if (bid > fmaxkey) fmaxkey = bid;
    fhead = bid;                                           // chain.rs:188-190: unconditionally
  }
  __device__ __forceinline__ void follower_tick(const SymMail& in, SymMail& out) {
    if (in.hb) follower_heartbeat(in, out);
    if (in.ae) {                                           // follower.rs:130-176 with voted_for == Some(leader)
      for (uint32_t k = 0; k < in.ae_nb && !abort; ++k) {
        const uint32_t bid = in.ae_id[k];
        uint32_t nx; uint64_t tk;
        fetch_sent(bid, in.mk, n_app, nx, tk);             // the block as the leader sent it
        follower_extend(bid, nx, tk);
      }
      if (abort) return;
      if (in.ae_nb) {
        out.ar = 1;
        out.ar_head = fhead;
      }
    }
    // Command::Tick: the election timer cannot have expired (sym_enter checked the bound)
  }
  // Follower lane: the same tick when the AppendEntries' blocks are not listed in the mail.  The leader's
  // replicate() (leader.rs:124-174: Probe -> range(head..).nth(1); Replicate -> range(head..).skip(1).take(5)) is run
  // HERE, over the leader's table as it stood when its largest key was `mk`, and each block it yields is applied on the
  // spot -- the same blocks in the same order as listing them first, without the list and without reading them twice.
  __device__ __forceinline__ void follower_tick_view(const SymMail& in, uint32_t phf, uint32_t modef, uint32_t mk, SymMail& out) {
    if (in.hb) follower_heartbeat(in, out);
    if (!in.ae || abort) return;
    const uint32_t take = modef ? JR_MAX_AE_BLOCKS : 1u;
    uint32_t bid = max(phf, tbase), pulled = 0, nb = 0;
    while (pulled < 1 + take) {
      uint32_t nx = ABSENT; uint64_t tk = 0;
      while (bid <= mk) {
        fetch_sent(bid, mk, n_app, nx, tk);
        if (nx != ABSENT) break;
        ++bid;
      }
      if (bid > mk) break;
      if (pulled >= 1) {
        follower_extend(bid, nx, tk);
        if (abort) return;
        ++nb;
      }
      ++pulled;
      ++bid;
    }
    if (nb) {
      out.ar = 1;
      out.ar_head = fhead;
    }
  }
};

// ---- entry: is the group symmetric, is its mail canonical? ---------------------------------------------------------
template <int R>
__device__ __forceinline__ bool sym_enter(SymGroup<R>& s, SymMail& m, const StepParams& p, int prv) {
  const Dev& d = s.d;
  if (s.g >= d.G) return false;
  // roles: one live leader, R-1 live followers of that leader
  uint32_t L = R, nlead = 0;
  uint4 p2[R];
#pragma unroll
  for (int r = 0; r < R; ++r) {
    p2[r] = d.p2[s.rg(r)];
    const uint32_t meta = p2[r].w;
    if (((meta >> 8) & 255u) || ((meta >> 27) & 1u)) return false;          // faulted or silenced
    if ((meta & 255u) == JR_ROLE_LEADER) { L = r; ++nlead; }
    else if ((meta & 255u) != JR_ROLE_FOLLOWER) return false;
    if ((meta >> 24) & 7u) return false;                                      // queued client requests
  }
  if (nlead != 1) return false;
  s.L = L;
  s.F0 = L == 0 ? 1u : 0u;
  const uint4 l0 = d.p0[s.rg(L)];
  s.term = (uint64_t)l0.x | ((uint64_t)l0.y << 32);
  s.tbase = d.tb[s.g];
  uint4 pl = p2[0], pf = p2[0];             // the leader's and the first follower's P2 (static selects: no local array)
  const uint32_t f0i = L == 0 ? 1u : 0u;
#pragma unroll
  for (int r = 0; r < R; ++r) {
    if ((uint32_t)r == L) pl = p2[r];
    if ((uint32_t)r == f0i) pf = p2[r];
  }
  s.head = pl.x; s.commit = pl.y; s.idgen = pl.z;
  s.ckey = (pl.w >> 28) & 1u;
  s.maxkey = d.mk[s.rg(L)];
  if (!(s.idgen > s.head)) return false;                                      // the next append would assert (chain.rs:163)
  const uint4 l3 = d.p3[s.rg(L)];
  s.hbtime = (uint64_t)l3.x | ((uint64_t)l3.y << 32);
  // followers: identical
  const uint32_t f0 = s.F0;
  s.fhead = pf.x; s.fcommit = pf.y; s.fckey = (pf.w >> 28) & 1u;
  s.fmaxkey = d.mk[s.rg(f0)];
  const uint64_t hbgap = ((uint64_t)d.hb / p.dt + 1) * p.dt;                 // ticks between two heartbeats, in ms
#pragma unroll
  for (int r = 0; r < R; ++r) {
    if ((uint32_t)r == L) continue;
    const uint4 a = d.p0[s.rg(r)];
    if (((uint64_t)a.x | ((uint64_t)a.y << 32)) != s.term || a.z != L + 1 || a.w != L + 1) return false;
    if (p2[r].x != s.fhead || p2[r].y != s.fcommit || ((p2[r].w >> 28) & 1u) != s.fckey) return false;
    if (d.mk[s.rg(r)] != s.fmaxkey) return false;
  }
  if ((uint64_t)d.emin <= hbgap || s.hbtime > p.now) return false;   // between two heartbeats no timer (>= emin) can fire
  // the leader's view of the followers: one progress entry value for all of them
  uint32_t ph[R];
#pragma unroll
  for (int q = 0; q < (R + 3) / 4; ++q) {
    const uint4 v = d.pr[(size_t)q * s.plane + s.rg(L)];
    if (q * 4 + 0 < R) ph[q * 4 + 0] = v.x;
    if (q * 4 + 1 < R) ph[q * 4 + 1] = v.y;
    if (q * 4 + 2 < R) ph[q * 4 + 2] = v.z;
    if (q * 4 + 3 < R) ph[q * 4 + 3] = v.w;
  }
  const uint32_t prmask = (pl.w >> 16) & 255u;
  s.ph_self = 0; s.ph_f = 0;
#pragma unroll
  for (int r = 0; r < R; ++r) {
    if ((uint32_t)r == L) s.ph_self = ph[r];
    if ((uint32_t)r == f0) s.ph_f = ph[r];
  }
  s.mode_self = (prmask >> L) & 1u;
  s.mode_f = (prmask >> f0) & 1u;
#pragma unroll
  for (int r = 0; r < R; ++r)
    if ((uint32_t)r != L && (ph[r] != s.ph_f || ((prmask >> r) & 1u) != s.mode_f)) return false;
  // Everything the launch reads of a follower's table lies in [flo, fmaxkey] (or is written by the launch itself):
  // the commit a heartbeat names (>= commit), the apply range (from fcommit), the parents of the blocks behind ph_f.
  // Those rows must be identical in every follower, because the lowest follower's table stands for all of them; a read
  // below flo that is not below the floor aborts the lane (fetch_f).  At most SYM_WINDOW ids, else step_kernel's business.
  constexpr uint32_t SYM_WINDOW = 16;
  const uint32_t top = min(s.maxkey, s.fmaxkey);
  const uint32_t lo_min = max(top > SYM_WINDOW - 1u ? top - (SYM_WINDOW - 1u) : 0u, s.tbase);   // (below the floor nobody holds anything)
  if (top < s.tbase || s.ph_f < lo_min || s.fcommit < lo_min || s.commit < lo_min || s.fhead < lo_min || s.fmaxkey > s.maxkey) return false;
  const uint32_t lo = min(min(s.ph_f, s.fcommit), min(s.commit, s.fhead));
  s.flo = lo;
  const uint64_t grow = (uint64_t)p.n_ticks * (1u + p.n_synth) + 2u;
  if ((uint64_t)s.maxkey + grow >= (uint64_t)s.tbase + d.cap || (uint64_t)s.maxkey + grow >= FS_NOTIFY_BIT) return false;
  {  // batches of independent loads, no exit in between: the latency of ~100 dependent loads was 14% of the kernel
    constexpr uint32_t B = 4;
    bool same = true;
    for (uint32_t b0 = lo; b0 <= s.fmaxkey && same; b0 += B) {
      uint32_t n0[B];
      unsigned long long t0[B];
#pragma unroll
      for (uint32_t j = 0; j < B; ++j) {
        const uint32_t b = min(b0 + j, s.fmaxkey);          // (the tail re-checks the last id: no divergent guards)
        n0[j] = d.cnext[s.row(f0, b)];
        t0[j] = d.ctok[s.row(f0, b)];
      }
#pragma unroll
      for (int r = 0; r < R; ++r) {
        if ((uint32_t)r == L || (uint32_t)r == f0) continue;
#pragma unroll
        for (uint32_t j = 0; j < B; ++j) {
          const uint32_t b = min(b0 + j, s.fmaxkey);
          const uint32_t n = d.cnext[s.row(r, b)];
          const unsigned long long t = d.ctok[s.row(r, b)];
          same = same && n == n0[j] && (n0[j] == ABSENT || t == t0[j]);
        }
      }
    }
    if (!same) return false;
  }
  // mail in flight (the previous tick's outboxes), delivered only with PH_DRAIN
  m = SymMail{};
  if (p.phases & PH_DRAIN) {
  {  // leader: [Heartbeat to Peers] then one AppendEntries per peer, ascending, all carrying the same run
    const uint32_t cnt = d.oc[prv][s.rg(L)];
    uint32_t u = 0;
    auto unit = [&](uint32_t k) { return d.ob[prv][((size_t)k * R + L) * d.Gp + s.g]; };
    if (cnt > (uint32_t)(1 + JR_MAX_AE_BLOCKS + R)) return false;
    if (u < cnt) {
      const uint4 h = unit(u);
      if ((h.x & 15u) == JR_CMD_HEARTBEAT) {
        if ((h.x >> 16) != TO_PEERS || ((uint64_t)h.y | ((uint64_t)h.z << 32)) != s.term) return false;
        m.hb = 1; m.hb_commit = h.w;
        ++u;
      }
    }
    if (u < cnt) {
      uint32_t first = 0;
      for (int r = 0; r < R; ++r) {
        if ((uint32_t)r == L) continue;
        if (u >= cnt) return false;
        const uint4 h = unit(u);
        if ((h.x & 15u) != JR_CMD_APPEND_ENTRIES || (h.x >> 16) != (uint32_t)r + 1u ||
            ((uint64_t)h.y | ((uint64_t)h.z << 32)) != s.term) return false;
        const uint32_t nb = (h.x >> 8) & 255u, ref = (h.x >> 4) & 1u;
        if (!m.ae) {                                        // the first peer carries the run inline
          if (ref || nb > JR_MAX_AE_BLOCKS || h.w != u + 1 || u + 1 + nb > cnt) return false;
          m.ae = 1; m.ae_nb = nb; first = u + 1;
          for (uint32_t k = 0; k < nb; ++k) {
            const uint4 bu = unit(first + k);
            uint32_t nx; uint64_t tk;
            s.fetch(L, bu.x, nx, tk);                       // the sim re-reads the block from the leader's table: must be what was sent
            if (nx != bu.y || tk != ((uint64_t)bu.z | ((uint64_t)bu.w << 32))) return false;
            m.ae_id[k] = bu.x;
          }
          u += 1 + nb;
        } else {                                            // the others point at it
          if (!ref || nb != m.ae_nb || h.w != first) return false;
          ++u;
        }
      }
    }
    if (u != cnt) return false;
  }
  {  // followers: [HeartbeatResponse][AppendResponse] to the leader, the same from each
    const uint32_t cnt = d.oc[prv][s.rg(f0)];
    if (cnt > 2) return false;
    uint4 want[2] = {make_uint4(0, 0, 0, 0), make_uint4(0, 0, 0, 0)};
    for (uint32_t u = 0; u < cnt; ++u) want[u] = d.ob[prv][((size_t)u * R + f0) * d.Gp + s.g];
#pragma unroll
    for (int r = 0; r < R; ++r) {
      if ((uint32_t)r == L || (uint32_t)r == f0) continue;
      if (d.oc[prv][s.rg(r)] != cnt) return false;
      for (uint32_t u = 0; u < cnt; ++u) {
        const uint4 v = d.ob[prv][((size_t)u * R + r) * d.Gp + s.g];
        if (v.x != want[u].x || v.y != want[u].y || v.z != want[u].z || v.w != want[u].w) return false;
      }
    }
    uint32_t u = 0;
    if (u < cnt && (want[u].x & 15u) == JR_CMD_HEARTBEAT_RESPONSE) {
      if ((want[u].x >> 16) != L + 1) return false;
      m.hbr = 1; m.hbr_has = (want[u].x >> 4) & 1u; m.hbr_commit = want[u].w;
      ++u;
    }
    if (u < cnt && (want[u].x & 15u) == JR_CMD_APPEND_RESPONSE) {
      if ((want[u].x >> 16) != L + 1 || ((uint64_t)want[u].y | ((uint64_t)want[u].z << 32)) != s.term) return false;
      m.ar = 1; m.ar_head = want[u].w;
      ++u;
    }
    if (u != cnt) return false;
  }
  }
  // Election timers (mod.rs:352-357): no follower may time out before the first heartbeat of this launch reaches it.
  // The leader heartbeats at the first tick with now - heartbeat_time > heartbeat_ms (leader.rs:78-84,237-240); the
  // follower takes it one tick later, before its own Tick.  (Afterwards the static bound above holds.)
  uint64_t t_arr = 0;
  if (!m.hb) {
    const uint64_t due = s.hbtime + (uint64_t)d.hb + 1;                     // smallest `now` that heartbeats
    t_arr = (due > p.now ? (due - p.now + p.dt - 1) / p.dt : 0) + 1;
  }
  const uint64_t checked = t_arr < p.n_ticks ? t_arr : p.n_ticks;           // ticks whose Tick runs on the old timer
  if (checked) {
    const uint64_t t_last = p.now + (checked - 1) * p.dt;
#pragma unroll
    for (int r = 0; r < R; ++r) {
      if ((uint32_t)r == L) continue;
      const uint4 b = d.p1[s.rg(r)];
      const uint64_t etime = (uint64_t)b.x | ((uint64_t)b.y << 32);
      if (t_last >= etime && t_last - etime > (uint64_t)b.z) return false;
    }
  }
  return true;
}

// ---- exit: write everything step_kernel would have left behind -------------------------------------------------------
template <int R>
__device__ __forceinline__ void sym_leave_leader(SymGroup<R>& s, const SymMail& last, int cur_last) {
  const Dev& d = s.d;
  const uint32_t L = s.L;
  {  // leader: P2, P3, progress planes, max key (P0 / P1 are untouched by a steady leader)
    const size_t i = s.rg(L);
    uint32_t prmask = 0;
#pragma unroll
    for (int r = 0; r < R; ++r) prmask |= (((uint32_t)r == L ? s.mode_self : s.mode_f) & 1u) << r;
    const uint32_t keep = d.p2[i].w & ~((255u << 16) | (1u << 28));
    d.p2[i] = make_uint4(s.head, s.commit, s.idgen, keep | (prmask << 16) | (s.ckey << 28));
    d.p3[i] = make_uint4((uint32_t)s.hbtime, (uint32_t)(s.hbtime >> 32), 0u, 0u);
#pragma unroll
    for (int q = 0; q < (R + 3) / 4; ++q) {
      uint32_t v[4] = {0, 0, 0, 0};
#pragma unroll
      for (int k = 0; k < 4; ++k)
        if (q * 4 + k < R) v[k] = (uint32_t)(q * 4 + k) == L ? s.ph_self : s.ph_f;
      d.pr[(size_t)q * s.plane + i] = make_uint4(v[0], v[1], v[2], v[3]);
    }
    d.mk[i] = s.maxkey;
    // outbox of the last tick: [Heartbeat][AppendEntries x (R-1): first inline, the rest pointing at its run]
    uint32_t u = 0;
    auto put = [&](uint32_t k, uint4 v) { d.ob[cur_last][((size_t)k * R + L) * d.Gp + s.g] = v; };
    if (last.hb) put(u++, make_uint4(unit_hdr(JR_CMD_HEARTBEAT, 0, 0, TO_PEERS), (uint32_t)s.term, (uint32_t)(s.term >> 32), last.hb_commit));
    if (last.ae) {
      uint32_t first = 0;
      bool have = false;
#pragma unroll
      for (int r = 0; r < R; ++r) {
        if ((uint32_t)r == L) continue;
        if (!have) {
          first = u + 1;
          put(u, make_uint4(unit_hdr(JR_CMD_APPEND_ENTRIES, 0, last.ae_nb, r + 1), (uint32_t)s.term, (uint32_t)(s.term >> 32), first));
          for (uint32_t k = 0; k < last.ae_nb; ++k) {
            uint32_t nx; uint64_t tk;
            s.fetch(L, last.ae_id[k], nx, tk);
            put(first + k, make_uint4(last.ae_id[k], nx, (uint32_t)tk, (uint32_t)(tk >> 32)));
          }
          u += 1 + last.ae_nb;
          have = true;
        } else {
          put(u++, make_uint4(unit_hdr(JR_CMD_APPEND_ENTRIES, 1, last.ae_nb, r + 1), (uint32_t)s.term, (uint32_t)(s.term >> 32), first));
        }
      }
    }
    d.oc[cur_last][i] = u;
    if ((d.flags & JR_F_CAPTURE_FSM) && s.lcnt) d.fc[i] = s.leader_end();
  }
}

template <int R>
__device__ __forceinline__ void sym_leave_followers(SymGroup<R>& s, const SymMail& last, int cur_last) {
  const Dev& d = s.d;
  const uint32_t L = s.L;
  // The followers emitted the same Instructions.  If none of them has anything pending since the last drain, ONE set of
  // records (in the lowest follower's FIFO, APPLY records carrying the mask of all followers) stands for all of them;
  // the others only advance their Instruction counters.  Otherwise every follower gets its own copy.
  const bool shared_records = s.share;
#pragma unroll
  for (int r = 0; r < R; ++r) {   // followers: P1 (timer, RNG), P2, max key, outbox
    if ((uint32_t)r == L) continue;
    const size_t i = s.rg(r);
    if (s.n_hb) {                  // follower.rs:103-113 per heartbeat: only the last draw is visible
      const uint4 b = d.p1[i];
      const uint32_t draws = b.w + s.n_hb;
      d.p1[i] = make_uint4((uint32_t)s.last_hb, (uint32_t)(s.last_hb >> 32),
                           election_timeout_draw(d.seed, d.goff + s.g, r + 1, draws - 1, d.emin, d.emax), draws);
    }
    const uint4 c = d.p2[i];
    d.p2[i] = make_uint4(s.fhead, s.fcommit, c.z, (c.w & ~(1u << 28)) | (s.fckey << 28));
    d.mk[i] = s.fmaxkey;
    uint32_t u = 0;
    if (last.hbr)
      d.ob[cur_last][((size_t)u++ * R + r) * d.Gp + s.g] =
          make_uint4(unit_hdr(JR_CMD_HEARTBEAT_RESPONSE, last.hbr_has, 0, L + 1), 0u, 0u, last.hbr_commit);
    if (last.ar)
      d.ob[cur_last][((size_t)u++ * R + r) * d.Gp + s.g] =
          make_uint4(unit_hdr(JR_CMD_APPEND_RESPONSE, 1, 0, L + 1), (uint32_t)s.term, (uint32_t)(s.term >> 32), last.ar_head);
    d.oc[cur_last][i] = u;
    if ((d.flags & JR_F_CAPTURE_FSM) && s.fcnt) {
      if (!shared_records) fsm_flush(d.fr + i, s.fcnt, d.Fr, FsmOut{d.fs + i, s.plane, d.F, s.g, (uint32_t)r}, d.fc + i);
      else if ((uint32_t)r == s.F0) d.fc[i] = s.followers_end();
      else d.fc[i] = make_uint2(0u, s.fcnt);               // counted here, carried by F0's masked records
    }
  }
}

// Two lanes per group (see SYM2_GROUPS above).  Both lanes run sym_enter on the same, still untouched planes and reach
// the same verdict; afterwards each keeps to its side: the leader lane owns the leader's table cache, encoder state,
// planes and outbox, the follower lane those of the followers.  Either side may abort: it says so in its mail, the
// other side sees it one barrier later, and after the last barrier both check the other's final mail, so a group is
// either left (by both) or not at all.
template <int R>
__global__ void __launch_bounds__(2 * SYM2_GROUPS, SYM2_MINCTAS) sym2_kernel(const Dev d, const StepParams p, uint8_t* symdone, uint8_t* symblk) {
  JR_DYN_SMEM(uint4, smem);
  // One __syncthreads() per tick for both warp pairs of the CTA.  (A named barrier per pair -- `bar.sync 0/1, 64`, the
  // pairs never need each other -- measured 3% SLOWER, twice; with a register operand for the id ptxas charges the CTA
  // all 16 barriers and only one CTA fits an SM.)
  auto pair_sync = [] { __syncthreads(); };
  constexpr uint32_t S = SYM2_GROUPS;
  const uint32_t w = threadIdx.x >> 5, lane = threadIdx.x & 31u;
  const bool lead = ((w ^ blockIdx.x) & 1u) == 0;          // roles alternate from CTA to CTA: no SM sub-partition gets leaders only
  const uint32_t gi = (w >> 1) * 32u + lane;               // group within the CTA
  const uint32_t g = blockIdx.x * S + gi;                  // (g >= Gp: sym_enter says no; the lane only keeps the barriers company)
  SymGroup<R> s(d, g);
  s.abort = false;
  s.lcnt = s.fcnt = 0;
  s.n_hb = 0;
  s.last_hb = 0;
  s.share = false;
  s.n_app = 1u + p.n_synth;
  s.rows = smem + gi;
  s.enc = smem + 2 * SYM_ROWS * S + gi;
  uint4* mail = smem + SYM_SMEM_UNITS * S + gi;            // [k * S]: k = 2 * buf + {0, 1} leader -> followers, 4 + buf followers -> leader
  s.cache_clear(lead ? 0u : SYM_ROWS, SYM_ROWS);
  const uint32_t blk = g / GROUPS_PER_CTA;                  // step_kernel's 32-group block of this warp pair
  if (lead && lane == 0 && g < d.Gp) symblk[blk] = 1;      // (cleared below by any lane whose group is not folded)
  pair_sync();
  SymMail a;
  bool dead = !sym_enter(s, a, p, 1 - p.cur);
  pair_sync();                                         // the other lane's sym_enter may still be reading this lane's (empty) cache
  if (!dead) {
    if (lead) {
      s.cache_fill(s.L, s.maxkey);
      s.enc_init_leader((d.flags & JR_F_CAPTURE_FSM) ? d.fc[s.rg(s.L)] : make_uint2(0u, 0u));
      // the mail in flight, where tick 0 looks for it
      mail[2 * S] = make_uint4(a.hb | (a.ae << 1) | (a.ae_nb << 4) | SYM2_IDS, a.hb_commit, s.maxkey, a.ae_id[0]);
      mail[3 * S] = make_uint4(a.ae_id[1], a.ae_id[2], a.ae_id[3], a.ae_id[4]);
    } else {
      s.cache_fill(s.F0, s.fmaxkey);
      s.enc_init_followers();
      s.share = (d.flags & JR_F_CAPTURE_FSM) != 0;
#pragma unroll
      for (int r = 0; r < R; ++r) {
        if ((uint32_t)r == s.L) continue;
        const uint2 c = d.fc[s.rg(r)];
        if (c.x | c.y) s.share = false;
      }
      mail[5 * S] = make_uint4(a.hbr | (a.hbr_has << 1) | (a.ar << 2), a.hbr_commit, a.ar_head, 0u);
    }
  }
  pair_sync();
  const jr_proposal* props = p.proposals;
  s.now = p.now;
  uint32_t cur = 0;                                        // mail buffer written this tick; 1 - cur is read
  for (uint32_t t = 0; t < p.n_ticks; ++t) {
    if (lead) {
      if (!dead) {
        const uint4 c = mail[(4 + (1 - cur)) * S];
        if (c.x & SYM2_ABORT) dead = true;
        else {
          SymMail in{}, out{};
          in.hbr = c.x & 1u; in.hbr_has = (c.x >> 1) & 1u; in.ar = (c.x >> 2) & 1u;
          in.hbr_commit = c.y; in.ar_head = c.z;
          uint64_t tok = 0;
          if ((p.phases & PH_PROPOSE) && (props || p.tok_runs)) {
            uint4 pr;
            if (p.tok_runs) {
              const uint4 rn = __ldg(p.tok_runs + g);
              const uint64_t base = (uint64_t)rn.x | ((uint64_t)rn.y << 32);
              const uint64_t tk = base + (uint64_t)(p.tok_tick + t) * ((uint64_t)rn.z | ((uint64_t)rn.w << 32));
              pr = make_uint4((uint32_t)tk, (uint32_t)(tk >> 32), base ? __ldg(p.tok_route + g) : 0u, 0u);
            } else {
              pr = __ldg(reinterpret_cast<const uint4*>(props + (size_t)t * p.prop_stride) + g);
            }
            if (pr.z == s.L + 1) tok = (uint64_t)pr.x | ((uint64_t)pr.y << 32);
            else if (pr.z != 0) s.abort = true;           // a proposal for a follower: proxied ClientRequest, not canonical
          }
          if (!s.abort) s.leader_tick(in, out, tok, (p.phases & PH_PROPOSE) ? p.n_synth : 0u, p.step_index + t);
          if (s.abort) dead = true;
          else {
            // (.y: the leader's commit -- what a Heartbeat of this tick carries, leader.rs:78-84; the last one also bounds the truncation)
            mail[(2 * cur) * S] = make_uint4(out.hb | (out.ae << 1) | (s.mode_f ? SYM2_MODE : 0u), s.commit, s.maxkey, s.ph_f);
          }
        }
      }
      if (dead) mail[(2 * cur) * S] = make_uint4(SYM2_ABORT, 0u, 0u, 0u);
    } else {
      if (!dead) {
        const uint4 ma = mail[(2 * (1 - cur)) * S];
        if (ma.x & SYM2_ABORT) dead = true;
        else {
          SymMail in{}, out{};
          in.hb = ma.x & 1u; in.ae = (ma.x >> 1) & 1u;
          in.hb_commit = ma.y; in.mk = ma.z;
          if (ma.x & SYM2_IDS) {                           // tick 0: the blocks sym_enter found in the leader's outbox
            const uint4 mb = mail[(2 * (1 - cur) + 1) * S];
            in.ae_nb = (ma.x >> 4) & 15u;
            in.ae_id[0] = ma.w; in.ae_id[1] = mb.x; in.ae_id[2] = mb.y; in.ae_id[3] = mb.z; in.ae_id[4] = mb.w;
            s.follower_tick(in, out);
          } else {
            s.follower_tick_view(in, ma.w, (ma.x & SYM2_MODE) ? 1u : 0u, ma.z, out);
          }
          if (s.abort) dead = true;
          else mail[(4 + cur) * S] = make_uint4(out.hbr | (out.hbr_has << 1) | (out.ar << 2), out.hbr_commit, out.ar_head, 0u);
        }
      }
      if (dead) mail[(4 + cur) * S] = make_uint4(SYM2_ABORT, 0u, 0u, 0u);
    }
    s.now += p.dt;
    pair_sync();
    cur ^= 1u;
  }
  const uint32_t lastb = cur ^ 1u;                         // the buffers the last tick wrote
  const uint4 la = mail[(2 * lastb) * S], lc = mail[(4 + lastb) * S];
  const bool ok = !dead && !((la.x | lc.x) & SYM2_ABORT);
  if (ok) {
    const int cur_last = p.cur ^ (int)((p.n_ticks - 1) & 1u);
    SymMail last{};
    if (lead) {
      last.hb = la.x & 1u; last.ae = (la.x >> 1) & 1u;
      last.hb_commit = la.y;
      if (last.ae) s.replicate(s.ph_f, s.mode_f, s.maxkey, last);   // what the last tick sent: the outbox it leaves behind
      sym_leave_leader(s, last, cur_last);
    } else {
      last.hbr = lc.x & 1u; last.hbr_has = (lc.x >> 1) & 1u; last.ar = (lc.x >> 2) & 1u;
      last.hbr_commit = lc.y; last.ar_head = lc.z;
      sym_leave_followers(s, last, cur_last);
    }
  }
  if (p.trunc) {   // jr_truncate(margin) for this group (truncate_kernel, engine.cu): every replica is live, the
    //              leader's commit after the last tick travels in its last mail
    pair_sync();   // the leader lane's sym_leave may still be reading rows this is about to blank
    if (ok && !lead) {
      const uint32_t lo = min(s.fcommit, la.y);
      const uint32_t floor = lo > p.trunc_margin ? lo - p.trunc_margin : 0u;
      if (floor > s.tbase) {
        for (uint32_t b = s.tbase; b < floor && b - s.tbase < d.cap; ++b)
#pragma unroll
          for (int r = 0; r < R; ++r) d.cnext[s.row(r, b)] = ABSENT;
        d.tb[g] = floor;
      }
    }
  }
  if (lead && g < d.Gp) {
    symdone[g] = ok ? 1 : 0;
    if (!ok) {
      symblk[blk] = 0;
      if (g < d.G) *(volatile uint32_t*)d.hunf = p.epoch;   // advisory, for the host's choice of the next step_kernel grid
    }
  }
}

#endif  // JR_DEVICE_CODE
}  // namespace jr
