// engine.cu -- kernels + C ABI of the B200 batched Chained-Raft engine.
//
// Build: nvcc -gencode arch=compute_100a,code=sm_100a (see __graft_entry__.build).
// No CPU fallback: without a CUDA device jr_engine_create returns JR_E_NO_DEVICE.
//
// Reference interfaces replaced are cited in include/josefine_raft_abi.h; the
// replica state machine is in raft_device.cuh.
#include <algorithm>
#include <atomic>
#include <chrono>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <condition_variable>
#include <mutex>
#include <new>
#include <thread>
#include <vector>

#include "raft_device.cuh"
#include "sym_fold.cuh"

using namespace jr;

// ============================================================================
// kernels
// ============================================================================

// n_ticks fused schedule steps for every replica.  CTA = 32 groups x R warps; warp w
// is replica w of those groups.  Replica state lives in registers for the whole
// launch; the mailboxes of the CTA's groups live in shared memory (double
// buffered, units beyond Us spill to the global mailbox); block-table reads go
// through a per-lane shared-memory cache.  Groups never interact, so the only
// synchronisation between ticks is __syncthreads().
// A split launch (p0.n_parts > 1) runs every block's ticks as n_parts consecutive tasks.  Tasks are taken by
// ticket, in launch order, so all part k-1 tasks are running or done before any part k task starts; a part k
// task waits for its block's part k-1 (release/acquire on d.done[block]) and then continues from the state
// and mailboxes that task stored -- exactly what the next launch would do.  The point is the last wave:
// 2048 equal tasks on 592 CTA slots take 4 rounds, 4096 half-length tasks take 7 half-rounds.
#ifdef JR_EMU
#ifdef JR_EMU_BREAK_HANDOFF  // negative control of tests/emu/tsan_split.cpp: the race detector must notice this
#define JR_EMU_HANDOFF_ACQUIRE __ATOMIC_RELAXED
#define JR_EMU_HANDOFF_RELEASE __ATOMIC_RELAXED
#else
#define JR_EMU_HANDOFF_ACQUIRE __ATOMIC_ACQUIRE
#define JR_EMU_HANDOFF_RELEASE __ATOMIC_RELEASE
#endif
#endif
__device__ __forceinline__ uint32_t ld_acquire_u32(const uint32_t* p) {
#ifdef JR_EMU
  return __atomic_load_n(p, JR_EMU_HANDOFF_ACQUIRE);
#else
  uint32_t v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
#endif
}
__device__ __forceinline__ void st_release_u32(uint32_t* p, uint32_t v) {
#ifdef JR_EMU
  __atomic_store_n(p, v, JR_EMU_HANDOFF_RELEASE);
#else
  asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
#endif
}

// Resident CTAs the register allocation must allow (the kernel is latency bound: occupancy is throughput).
// R = 5 (160 threads) holds 4 CTAs per SM at 96 registers, what ptxas picked on its own before the stream encoder
// was added; the other sizes keep their natural allocation.
constexpr int step_min_ctas(int R) { return (R == 4 || R == 5) ? 4 : 1; }

template <int R, bool SORTED>
__global__ void __launch_bounds__(32 * R, step_min_ctas(R)) step_kernel(const Dev d, const StepParams p0) {
  JR_DYN_SMEM(uint4, smem);
  const uint32_t w = threadIdx.x >> 5, lane = threadIdx.x & 31u;
  StepParams p = p0;
  uint32_t blk = blockIdx.x, part = 0;
  if (p0.n_parts > 1) {
    uint32_t* s_ticket = reinterpret_cast<uint32_t*>(smem);  // free until stage_inbox: fenced by the two barriers
    if (threadIdx.x == 0) *s_ticket = atomicAdd(d.scatter + 1, 1u) - p0.ticket_base;
    __syncthreads();
    const uint32_t ticket = *s_ticket;
    __syncthreads();
    part = ticket / p0.n_blocks;
    blk = ticket - part * p0.n_blocks;
    const uint32_t t0 = part * p0.part_ticks;  // host: (n_parts - 1) * part_ticks < n_ticks
    p.n_ticks = min(p0.part_ticks, p0.n_ticks - t0);
    p.now += (uint64_t)t0 * p0.dt;
    p.step_index += t0;
    p.cur ^= (int)(t0 & 1u);
    if (p.proposals) p.proposals += (size_t)t0 * p0.prop_stride;
    p.tok_tick += t0;
    if (part) {
      p.phases = PH_RESET_OUT | PH_DRAIN | PH_PROPOSE | PH_TICK;
      if (threadIdx.x == 0)
        while (ld_acquire_u32(d.done + blk) != p0.epoch + part) {}
      __syncthreads();
    }
  }
  if (p0.symblk && p0.symblk[blk]) {   // every group of this block was folded by sym2_kernel: only keep the hand-over chain alive
    if (p0.n_parts > 1 && part + 1 < p0.n_parts && threadIdx.x == 0) st_release_u32(d.done + blk, p0.epoch + part + 1);
    return;
  }
  const uint32_t g = blk * GROUPS_PER_CTA + lane;  // padded groups (g >= G) are real, unused replicas
  const bool folded = p0.symdone && p0.symdone[g];   // this lane's group is done: it idles through the barriers
  // Which replica of group g this thread steps.  Plain variant: replica index = warp index, so a
  // warp runs one role's code when the CTA's leaders share a replica index (and every branch on
  // `r` is provably warp-uniform).  SORTED variant, picked by the host when a previous launch saw
  // leaders on several indices: the group's live leader goes to warp 0, the others follow in
  // index order.  Pure scheduling -- state planes and mailboxes are indexed by replica.
  uint32_t r = w;
  if constexpr (SORTED) {
    uint32_t lead = R;
#pragma unroll
    for (int rr = 0; rr < R; ++rr) {
      const uint32_t m = d.p2[(size_t)rr * d.Gp + g].w;
      if (lead == (uint32_t)R && (m & 255u) == JR_ROLE_LEADER && ((m >> 8) & 255u) == 0 && !((m >> 27) & 1u)) lead = rr;
    }
    if (lead != (uint32_t)R) r = w == 0 ? lead : (w <= lead ? w - 1 : w);
  }
  const uint32_t box = d.Us * R * 32;
  Local L;
  L.in = smem;
  L.out = smem + box;
  L.tc = smem + 2 * box;
  L.cin = reinterpret_cast<uint32_t*>(smem + 2 * box + d.W * R * 32);
  L.cout = L.cin + R * 32;
  L.mk_in = reinterpret_cast<uint16_t*>(L.cout + R * 32);
  L.mk_out = L.mk_in + R * R * 32;
  L.Us = d.Us; L.W = d.W; L.lane = lane;
  Replica<R, SORTED> rep(d, L, r, g);
  rep.now = p.now;
  rep.cur = p.cur;
  rep.load(p.phases & PH_RESET_OUT, p.phases & PH_RESET_FSM, part != 0);
  if (folded) rep.dead = 1;   // never stepped, never stored
  rep.tc_prefetch();
  rep.stage_inbox(p.phases & PH_DRAIN);
#ifdef JR_PROFILE
  for (uint32_t i = threadIdx.x; i < 8 * 3 * 16 * 2; i += blockDim.x) jr_prof_smem()[i] = 0;
#endif
  __syncthreads();
  StepParams q = p;
  for (uint32_t t = 0;; ++t) {
    JR_PROF_T0(tt);
    const uint32_t prole = rep.role == JR_ROLE_LEADER ? JR_ROLE_LEADER : JR_ROLE_FOLLOWER;
    (void)prole;
    rep.clear_marks();
    rep.run_step(q);
    JR_PROF_ADD(prole, 12, tt);
    if (t + 1 == p.n_ticks) break;
    L.cout[r * 32 + lane] = rep.ocnt;
    rep.publish_marks();
    JR_PROF_ADD(prole, 15, tt);
    __syncthreads();
    JR_PROF_ADD(prole, 13, tt);
    // next tick: what was written becomes the inbox
    uint4* tb = L.in; L.in = L.out; L.out = tb;
    uint32_t* tcn = L.cin; L.cin = L.cout; L.cout = tcn;
    uint16_t* tmk = L.mk_in; L.mk_in = L.mk_out; L.mk_out = tmk;
    rep.cur ^= 1;
    rep.ocnt = 0;
    rep.ocnt0 = 0;
    rep.now += p.dt;
    q.now = rep.now;
    q.step_index += 1;
    q.phases = PH_RESET_OUT | PH_DRAIN | PH_PROPOSE | PH_TICK;
    q.proposals = (p.proposals && p.prop_stride) ? p.proposals + (size_t)(t + 1) * p.prop_stride : nullptr;
    q.tok_tick += 1;
  }
  if (!folded) rep.store(part + 1 >= p0.n_parts);
  {  // tell the host whether the next launch should sort: leaders on >= 2 replica indices in this CTA?
    uint32_t* lmask = reinterpret_cast<uint32_t*>(L.tc);  // the table cache is dead now; reuse one word of it
    __syncthreads();
    if (threadIdx.x == 0) *lmask = 0;
    __syncthreads();
    if (!folded && rep.role == JR_ROLE_LEADER && rep.live()) atomicOr(lmask, 1u << r);
    __syncthreads();
    if (threadIdx.x == 0 && (*lmask & (*lmask - 1u))) *(volatile uint32_t*)d.hscat = p0.epoch;   // advisory, read by the host a launch or two later
  }
  if (p0.n_parts > 1 && part + 1 < p0.n_parts) {  // hand the block over to its next part
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) st_release_u32(d.done + blk, p0.epoch + part + 1);
  }
#ifdef JR_PROFILE
  __syncthreads();
  if (d.prof)
    for (uint32_t i = threadIdx.x; i < R * 3 * 16 * 2; i += blockDim.x) {
      const unsigned long long v = jr_prof_smem()[i];
      if (v) atomicAdd(d.prof + (i % (3 * 16 * 2)), v);
    }
#endif
}

// Host-injected commands: one thread per distinct target replica, commands in
// array order.  targets[i] = {group, replica index, first, count}.  No staging.
template <int R>
__global__ void inject_kernel(const Dev d, const StepParams p, const jr_msg* msgs, const uint4* targets,
                              uint32_t n_targets) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  Local L;
  L.in = L.out = L.tc = nullptr; L.cin = L.cout = nullptr; L.mk_in = L.mk_out = nullptr; L.Us = 0; L.W = 0; L.lane = 0;
  if (i >= n_targets) return;
  const uint4 t = targets[i];
  Replica<R> rep(d, L, t.y, t.x);
  rep.now = p.now;
  rep.cur = p.cur;
  rep.load(false, false);
  for (uint32_t k = 0; k < t.w; ++k) {
    const jr_msg* m = msgs + t.z + k;
    Cmd c;
    c.kind = m->kind; c.flag = m->flag ? 1u : 0u; c.node_id = m->node_id; c.block = (uint32_t)m->block;
    c.nblk = m->n_blocks; c.term = m->term; c.last_term = m->last_term;
    if (m->kind == JR_CMD_CLIENT_REQUEST || m->kind == JR_CMD_CLIENT_RESPONSE) {  // Cmd aliases, see raft_device.cuh
      c.term = m->token;
      c.block = ((uint32_t)m->client_kind << 16) | (m->client_id & 0xffffu);
    }
    c.blk_s = 0; c.blk_at = 0; c.host_msg = m;
    rep.apply(c);
  }
  rep.store();
}

// RaftHandle::new for every replica (mod.rs:428-435; follower.rs:68-95; chain.rs:117-153).
__global__ void init_kernel(const Dev d) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t plane = (size_t)d.R * d.Gp;
  if (i >= plane) return;
  const uint32_t r = (uint32_t)(i / d.Gp), g = (uint32_t)(i % d.Gp);
  const uint32_t timeout = election_timeout_draw(d.seed, d.goff + g, r + 1, 0, d.emin, d.emax);
  d.p0[i] = make_uint4(0, 0, 0, 0);
  d.p1[i] = make_uint4(0, 0, timeout, 1);                 // init(): first draw, election_time = 0
  // head 0, commit 0, id_gen 1; a node this engine does not host is inert (the `dead` bit)
  d.p2[i] = make_uint4(0, 0, 1, JR_ROLE_FOLLOWER | (((d.resident >> r) & 1u) ? 0u : (1u << 27)));
  d.p3[i] = make_uint4(0, 0, 0, 0);
  d.mk[i] = 0;
  d.cnext[i] = 0;                                         // genesis block 0 -> 0 (chain.rs:139-153)
  d.ctok[i] = 0;
  d.oc[0][i] = 0;
  d.oc[1][i] = 0;
  d.fc[i] = make_uint2(0, 0);
  if (r == 0) d.tb[g] = 0;
  const uint64_t tag = mix64(((d.goff + g) << 8) | (r + 1));
  d.dg[i] = make_uint4((uint32_t)tag, (uint32_t)(tag >> 32), (uint32_t)tag, (uint32_t)(tag >> 32));
  d.cn[i] = make_uint2(0, 0);
}

// Chain::compact for every live replica (chain.rs:239-253).
__global__ void compact_kernel(const Dev d) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t plane = (size_t)d.R * d.Gp;
  if (i >= plane || (uint32_t)(i % d.Gp) >= d.G) return;
  const uint4 c = d.p2[i];
  const uint32_t meta = c.w;
  if (((meta >> 8) & 255u) != 0 || ((meta >> 27) & 1u)) return;  // faulted or dead
  bool have = false;
  uint32_t expect = 0;
  const uint32_t floor = d.tb[i % d.Gp];
  for (uint32_t b = c.y; b-- > floor;) {  // ids in [0, commit), descending; nothing is left below the floor (D7)
    if (b - floor >= d.cap) continue;    // (a commit past the window cannot exist: chain_commit needs the block)
    const uint32_t nx = d.cnext[(size_t)(b & d.capm) * plane + i];
    if (nx == ABSENT) continue;
    if (have && b != expect) d.cnext[(size_t)(b & d.capm) * plane + i] = ABSENT;
    expect = nx;  // even for a removed block
    have = true;
  }
}

// Adds every thread's v into *out (one atomic per CTA on the device).
__device__ inline void block_add(unsigned long long* out, uint64_t v, uint64_t* smem) {
#ifdef JR_EMU
  (void)smem;
  atomicAdd(out, (unsigned long long)v);
#else
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  if ((threadIdx.x & 31) == 0) smem[threadIdx.x >> 5] = v;
  __syncthreads();
  if (threadIdx.x < 32) {
    uint64_t t = threadIdx.x < (blockDim.x >> 5) ? smem[threadIdx.x] : 0;
    for (int o = 16; o > 0; o >>= 1) t += __shfl_down_sync(0xffffffffu, t, o);
    if (threadIdx.x == 0) atomicAdd(out, (unsigned long long)t);
  }
  __syncthreads();
#endif
}

// Normative state digest (DESIGN.md "Digests"); must equal jro_state_digest.
__global__ void state_digest_kernel(const Dev d, unsigned long long* out) {
  __shared__ uint64_t sm[32];
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t plane = (size_t)d.R * d.Gp;
  uint64_t h = 0;
  if (i < plane && (uint32_t)(i % d.Gp) < d.G) {
    const uint32_t r = (uint32_t)(i / d.Gp), g = (uint32_t)(i % d.Gp);
    const uint4 a = d.p0[i], b = d.p1[i], c = d.p2[i];
    const uint32_t role = c.w & 255u, fault = (c.w >> 8) & 255u, prmask = (c.w >> 16) & 255u;
    const uint32_t nq = (c.w >> 24) & 7u, dead = (c.w >> 27) & 1u;
    h = mix64(0x243f6a8885a308d3ull ^ (((d.goff + g) << 8) | (r + 1)));
    h = fold(h, (uint64_t)a.x | ((uint64_t)a.y << 32));
    h = fold(h, a.z);
    h = fold(h, (uint64_t)role | ((uint64_t)fault << 8) | ((uint64_t)(dead ? 0 : 1) << 16) | ((uint64_t)nq << 24));
    h = fold(h, (uint64_t)b.x | ((uint64_t)b.y << 32));
    h = fold(h, (uint64_t)b.z | ((uint64_t)b.w << 32));
    h = fold(h, c.x);
    h = fold(h, c.y);
    h = fold(h, c.z);
    if (role == JR_ROLE_FOLLOWER) h = fold(h, a.w);
    if (role == JR_ROLE_CANDIDATE) {
      const uint4 e = d.p3[i];
      h = fold(h, (uint64_t)e.z | ((uint64_t)e.w << 32));
    }
    if (role == JR_ROLE_LEADER) {
      const uint4 e = d.p3[i];
      h = fold(h, (uint64_t)e.x | ((uint64_t)e.y << 32));
      for (uint32_t k = 0; k < d.R; ++k) {
        const uint4 v = d.pr[(size_t)(k / 4) * plane + i];
        const uint32_t ph = (k & 3) == 0 ? v.x : (k & 3) == 1 ? v.y : (k & 3) == 2 ? v.z : v.w;
        h = fold(h, ph);
      }
      h = fold(h, prmask);
    }
    for (uint32_t q = 0; q < nq; ++q) {
      const uint4 e = d.qt[(size_t)q * plane + i];
      h = fold(h, (uint64_t)e.x | ((uint64_t)e.y << 32));
      h = fold(h, (uint64_t)(e.z >> 16) | ((uint64_t)(e.z & 0xffffu) << 8));
    }
    uint64_t chain = 0;
    const uint32_t mk = d.mk[i], floor = d.tb[g];
    for (uint32_t bid = floor; bid <= mk && bid - floor < d.cap; ++bid) {
      const uint32_t nx = d.cnext[(size_t)(bid & d.capm) * plane + i];
      if (nx == ABSENT) continue;
      const uint64_t tok = d.ctok[(size_t)(bid & d.capm) * plane + i];
      chain += mix64(mix64((uint64_t)bid + 0x13198a2e03707344ull) ^ ((uint64_t)nx * 0xa4093822299f31d1ull) ^ tok);
    }
    h = fold(h, chain);
  }
  block_add(out, h, sm);
}

// out[0..3] = sum msg digest, sum fsm digest, n msgs, n fsm; out[4] = faulted replicas
__global__ void stream_digest_kernel(const Dev d, unsigned long long* out) {
  __shared__ uint64_t sm[32];
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t plane = (size_t)d.R * d.Gp;
  uint64_t a = 0, b = 0, x = 0, y = 0, f = 0;
  if (i < plane && (uint32_t)(i % d.Gp) < d.G) {
    const uint4 v = d.dg[i];
    const uint2 n = d.cn[i];
    a = (uint64_t)v.x | ((uint64_t)v.y << 32);
    b = (uint64_t)v.z | ((uint64_t)v.w << 32);
    x = n.x;
    y = n.y;
    f = ((d.p2[i].w >> 8) & 255u) != 0;
  }
  block_add(out + 0, a, sm);
  block_add(out + 1, b, sm);
  block_add(out + 2, x, sm);
  block_add(out + 3, y, sm);
  block_add(out + 4, f, sm);
}

// Leader::write_state (leader.rs:101-121) for every group: the live leader with
// the highest (term, id).  One thread per group.
__global__ void leader_table_kernel(const Dev d, jr_leader_entry* out, uint32_t* route) {
  const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= d.G) return;
  jr_leader_entry e{0, 0, 0};
  for (uint32_t r = 0; r < d.R; ++r) {
    const size_t i = (size_t)r * d.Gp + g;
    const uint4 c = d.p2[i];
    const uint32_t role = c.w & 255u, fault = (c.w >> 8) & 255u, dead = (c.w >> 27) & 1u;
    if (role != JR_ROLE_LEADER || fault || dead) continue;
    const uint4 a = d.p0[i];
    const uint64_t term = (uint64_t)a.x | ((uint64_t)a.y << 32);
    if (e.leader_id == 0 || term >= e.term) {
      e.term = term;
      e.leader_id = r + 1;
      e.commit = c.y;
    }
  }
  out[g] = e;
  route[g] = e.leader_id;  // where jr_run_tokens sends this group's proposals until the next announce
}

// jr_run_tokens: tokens[k*G + g] -> jr_proposal{token, node = last announced leader of g}.  Pure streaming
// (8 B in, 16 B out per group-tick); the step kernel then reads the same dense layout jr_run_proposals stages.
__global__ void route_tokens_kernel(const unsigned long long* __restrict__ tokens, const uint32_t* __restrict__ route,
                                    jr_proposal* __restrict__ out, uint32_t G, size_t n) {
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const unsigned long long t = tokens[i];
    jr_proposal p;
    p.token = t;
    p.node = t ? route[i % G] : 0u;
    p.reserved = 0;
    out[i] = p;
  }
}

__global__ void kill_leaders_kernel(const Dev d, uint64_t base, uint32_t permille, unsigned long long* n_killed) {
  const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
  const bool pick = g < d.G && mix64(base + d.goff + g) % 1000 < permille;
  uint32_t killed = 0;
  for (uint32_t r = 0; r < d.R; ++r) {
    bool hit = false;
    if (pick) {
      const size_t i = (size_t)r * d.Gp + g;
      const uint32_t m = d.p2[i].w;
      hit = (m & 255u) == JR_ROLE_LEADER && ((m >> 8) & 255u) == 0 && ((m >> 27) & 1u) == 0;
      if (hit) d.p2[i].w = m | (1u << 27);
    }
#ifdef JR_EMU
    killed += hit ? 1u : 0u;
#else
    // warp-aggregated count: one vote per lane, popcount of the ballot, one atomic per warp
    const uint32_t votes = __ballot_sync(0xffffffffu, hit);
    if ((threadIdx.x & 31u) == 0) killed += (uint32_t)__popc(votes);
#endif
  }
  if (killed) atomicAdd(n_killed, (unsigned long long)killed);
}

__global__ void set_alive_kernel(const Dev d, uint32_t g, uint32_t r, int alive) {
  const size_t i = (size_t)r * d.Gp + g;
  uint32_t m = d.p2[i].w;
  d.p2[i].w = alive ? (m & ~(1u << 27)) : (m | (1u << 27));
}

// jr_query_many: thread k reads replica (groups[k], nodes[k] - 1)
__global__ void query_kernel(const Dev d, const uint32_t* groups, const uint32_t* nodes, uint32_t n, jr_replica_state* out) {
  const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const uint32_t g = groups[k], r = nodes[k] - 1u;
  jr_replica_state* o = out + k;
  const size_t plane = (size_t)d.R * d.Gp;
  const size_t i = (size_t)r * d.Gp + g;
  const uint4 a = d.p0[i], b = d.p1[i], c = d.p2[i], e = d.p3[i];
  jr_replica_state s;
  memset(&s, 0, sizeof s);
  s.current_term = (uint64_t)a.x | ((uint64_t)a.y << 32);
  s.voted_for = a.z;
  s.role = c.w & 255u;
  s.leader_id = s.role == JR_ROLE_FOLLOWER ? a.w : 0;
  s.election_time_ms = (uint64_t)b.x | ((uint64_t)b.y << 32);
  s.election_timeout_ms = b.z;
  s.rng_draws = b.w;
  s.head = c.x;
  s.commit = c.y;
  s.id_gen = c.z;
  s.max_key = d.mk[i];
  s.fault = (c.w >> 8) & 255u;
  s.alive = ((c.w >> 27) & 1u) ? 0 : 1;
  s.n_queued = (c.w >> 24) & 7u;
  if (s.role == JR_ROLE_LEADER) {
    s.heartbeat_time_ms = (uint64_t)e.x | ((uint64_t)e.y << 32);
    s.progress_replicate = (c.w >> 16) & 255u;
    for (uint32_t k = 0; k < d.R; ++k) {
      const uint4 v = d.pr[(size_t)(k / 4) * plane + i];
      s.progress_head[k] = (k & 3) == 0 ? v.x : (k & 3) == 1 ? v.y : (k & 3) == 2 ? v.z : v.w;
    }
  }
  if (s.role == JR_ROLE_CANDIDATE) {
    s.votes_seen = e.z;
    s.votes_granted = e.w;
  }
  s.chain_floor = d.tb[g];
  *o = s;
}

// jr_chain_read_many: request q = {group, node - 1, first id, output offset}; one CTA per request
__global__ void chain_read_kernel(const Dev d, const uint4* reqs, const uint32_t* counts, jr_block* out, uint8_t* present) {
  const uint32_t q = blockIdx.x;
  const uint4 rq = reqs[q];
  const uint32_t n = counts[q];
  const size_t plane = (size_t)d.R * d.Gp;
  const size_t i = (size_t)rq.y * d.Gp + rq.x;
  const uint32_t floor = d.tb[rq.x];
  for (uint32_t k = threadIdx.x; k < n; k += blockDim.x) {
    const uint64_t bid = (uint64_t)rq.z + k;
    uint32_t nx = ABSENT;
    if (bid >= floor && bid - floor < d.cap) nx = d.cnext[(size_t)((uint32_t)bid & d.capm) * plane + i];
    present[rq.w + k] = nx != ABSENT;
    out[rq.w + k] = jr_block{bid, nx != ABSENT ? nx : 0ull,
                             nx != ABSENT ? d.ctok[(size_t)((uint32_t)bid & d.capm) * plane + i] : 0ull};
  }
}

// jr_truncate (deviation D7).  One thread per group: new floor = min(commit over live replicas) - margin, never
// below the old one; every block below it leaves the table of EVERY replica of the group (rows are reused by
// the ids one window further up, so they must read as absent).
__global__ void truncate_kernel(const Dev d, uint32_t margin, const uint8_t* skip) {
  const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= d.Gp) return;
  if (skip && skip[g]) return;   // truncated by the lane that folded the group (sym2_kernel)
  const size_t plane = (size_t)d.R * d.Gp;
  const uint32_t old = d.tb[g];
  uint32_t lo = 0xFFFFFFFFu;
  for (uint32_t r = 0; r < d.R; ++r) {
    const uint4 c = d.p2[(size_t)r * d.Gp + g];
    if (((c.w >> 8) & 255u) != 0 || ((c.w >> 27) & 1u)) continue;  // faulted or silenced: not waited for
    lo = min(lo, c.y);
  }
  if (lo == 0xFFFFFFFFu) return;
  const uint32_t floor = lo > margin ? lo - margin : 0u;
  if (floor <= old) return;
  for (uint32_t b = old; b < floor && b - old < d.cap; ++b)
    for (uint32_t r = 0; r < d.R; ++r) d.cnext[(size_t)(b & d.capm) * plane + (size_t)r * d.Gp + g] = ABSENT;
  // a replica that was not waited for (silenced / faulted) may have lost every block it held: an empty table's largest key is 0
  for (uint32_t r = 0; r < d.R; ++r)
    if (d.mk[(size_t)r * d.Gp + g] < floor) d.mk[(size_t)r * d.Gp + g] = 0;
  d.tb[g] = floor;
}

// jr_node_restart: Chain::new over persisted blocks (chain.rs:117-137) + Raft::<Follower>::new (follower.rs:68-95)
// for one replica.  Single thread; `blocks` is device memory.
__global__ void node_restart_kernel(const Dev d, uint32_t g, uint32_t r, uint64_t now, const jr_block* blocks, uint32_t n,
                                    uint32_t commit, uint32_t ckey) {
  const size_t plane = (size_t)d.R * d.Gp;
  const size_t i = (size_t)r * d.Gp + g;
  const uint32_t floor = d.tb[g];
  for (uint32_t b = 0; b < d.cap; ++b) d.cnext[(size_t)((floor + b) & d.capm) * plane + i] = ABSENT;  // an empty sled tree
  uint32_t mk = 0;
  for (uint32_t k = 0; k < n; ++k) {   // host-validated: floor <= id < floor + cap
    const uint32_t bid = (uint32_t)blocks[k].id;
    d.cnext[(size_t)(bid & d.capm) * plane + i] = (uint32_t)blocks[k].next;
    d.ctok[(size_t)(bid & d.capm) * plane + i] = blocks[k].data;
    mk = max(mk, bid);
  }
  uint32_t idgen = commit;             // IdGenerator::new(commit), chain.rs:126
  if (commit == 0) {                   // chain.init(), chain.rs:139-153: id_gen.next() == 0, block 0 -> 0 inserted
    if (floor == 0) { d.cnext[i] = 0; d.ctok[i] = 0; }
    idgen = 1;
  }
  const uint32_t timeout = election_timeout_draw(d.seed, d.goff + g, r + 1, 0, d.emin, d.emax);
  d.p0[i] = make_uint4(0, 0, 0, 0);
  d.p1[i] = make_uint4((uint32_t)now, (uint32_t)(now >> 32), timeout, 1);
  d.p2[i] = make_uint4(commit, commit, idgen, JR_ROLE_FOLLOWER | ((ckey ? 1u : 0u) << 28));
  d.p3[i] = make_uint4(0, 0, 0, 0);
  d.mk[i] = mk;
  d.oc[0][i] = 0;
  d.oc[1][i] = 0;
}

// ---- Instruction-stream drain -----------------------------------------------------------------
// Records sit in per-replica FIFOs ([2*rec + half][replica][group]).  The drain packs them into one dense
// array in thread order i = replica * Gp + group -- sorted by (node, group), FIFO per replica -- with an exclusive
// scan over the per-replica counts, writes them to a device staging buffer and empties the FIFOs; the copy engine
// takes the batch to pinned host memory (fsm_records_enqueue).
constexpr uint32_t SCAN_THREADS = 1024;
struct FsmHeader {          // written by fsm_pack_kernel next to the records
  unsigned long long n_records, n_dropped, n_instructions;
  uint32_t node_offset[JR_MAX_REPLICAS + 1];
};

// Three small kernels (CTAs of T threads; the CPU emulation runs them with T = 1):
//   fsm_count_kernel  per-CTA sums of the replicas' record counts            -> part[3][n_ctas]
//   fsm_scan_kernel   one CTA: exclusive scan of those sums, batch totals     -> part[0] becomes CTA offsets, hdr
//   fsm_pack_kernel   CTA-local scan + CTA offset = each replica's position; copies its records, empties its FIFO
// Padded groups (g >= G) contribute nothing.
__device__ __forceinline__ uint32_t fsm_kept(const Dev& d, size_t i, uint2 c) {
  return (uint32_t)(i % d.Gp) < d.G ? min(c.x, d.F) : 0u;
}

__global__ void fsm_count_kernel(const Dev d, unsigned long long* part, uint32_t n_ctas) {
  __shared__ unsigned long long s[3][SCAN_THREADS / 32];
  const size_t plane = (size_t)d.R * d.Gp;
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  unsigned long long rec = 0, drop = 0, ins = 0;
  if (i < plane && (uint32_t)(i % d.Gp) < d.G) {
    const uint2 c = d.fc[i];
    rec = min(c.x, d.F);
    drop = c.x > d.F ? c.x - d.F : 0u;
    ins = c.y;
  }
#ifdef JR_EMU
  (void)s;
#else
  for (int o = 16; o > 0; o >>= 1) {
    rec += __shfl_down_sync(0xffffffffu, rec, o);
    drop += __shfl_down_sync(0xffffffffu, drop, o);
    ins += __shfl_down_sync(0xffffffffu, ins, o);
  }
  if ((threadIdx.x & 31) == 0) { s[0][threadIdx.x >> 5] = rec; s[1][threadIdx.x >> 5] = drop; s[2][threadIdx.x >> 5] = ins; }
  __syncthreads();
  if (threadIdx.x != 0) return;
  rec = drop = ins = 0;
  for (uint32_t w = 0; w < (blockDim.x + 31) / 32; ++w) { rec += s[0][w]; drop += s[1][w]; ins += s[2][w]; }
#endif
  part[blockIdx.x] = rec;
  part[n_ctas + blockIdx.x] = drop;
  part[2 * (size_t)n_ctas + blockIdx.x] = ins;
}

__global__ void fsm_scan_kernel(unsigned long long* part, uint32_t n_ctas, FsmHeader* hdr, uint32_t cap_records) {
  __shared__ unsigned long long s_sum[SCAN_THREADS];
  const uint32_t t = threadIdx.x, T = blockDim.x;
  const uint32_t per = (n_ctas + T - 1) / T;
  const uint32_t lo = min(n_ctas, per * t), hi = min(n_ctas, per * (t + 1));
  unsigned long long sum = 0, drop = 0, ins = 0;
  for (uint32_t k = lo; k < hi; ++k) { sum += part[k]; drop += part[n_ctas + k]; ins += part[2 * (size_t)n_ctas + k]; }
#ifdef JR_EMU
  s_sum[t] = sum;
  __syncthreads();
  if (t == 0) {
    unsigned long long run = 0;
    for (uint32_t k = 0; k < T; ++k) { const unsigned long long v = s_sum[k]; s_sum[k] = run; run += v; }
    hdr->n_records = min(run, (unsigned long long)cap_records);
    hdr->n_dropped = run > cap_records ? run - cap_records : 0ull;   // + the per-replica drops, added below
    hdr->n_instructions = 0;
  }
  __syncthreads();
#else
  {  // exclusive scan of the T per-thread sums: warp shuffles, then the warp totals (T <= 1024: one warp's worth)
    __shared__ unsigned long long s_warp[32];
    const uint32_t lane = t & 31u, w = t >> 5;
    unsigned long long inc = sum;
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned long long v = __shfl_up_sync(0xffffffffu, inc, o);
      if (lane >= (uint32_t)o) inc += v;
    }
    if (lane == 31) s_warp[w] = inc;
    __syncthreads();
    if (w == 0) {
      const unsigned long long mine = lane < (T + 31) / 32 ? s_warp[lane] : 0ull;
      unsigned long long wi = mine;
      for (int o = 1; o < 32; o <<= 1) {
        const unsigned long long v = __shfl_up_sync(0xffffffffu, wi, o);
        if (lane >= (uint32_t)o) wi += v;
      }
      s_warp[lane] = wi - mine;                           // exclusive prefix of the warp totals
      if (lane == 31) {
        hdr->n_records = min(wi, (unsigned long long)cap_records);
        hdr->n_dropped = wi > cap_records ? wi - cap_records : 0ull;   // + the per-replica drops, added below
        hdr->n_instructions = 0;
      }
    }
    __syncthreads();
    s_sum[t] = s_warp[w] + inc - sum;
  }
  __syncthreads();
#endif
#ifdef JR_EMU
  hdr->n_dropped += drop;
  hdr->n_instructions += ins;
#else
  if (drop) atomicAdd(&hdr->n_dropped, drop);
  if (ins) atomicAdd(&hdr->n_instructions, ins);
#endif
  unsigned long long at = s_sum[t];
  for (uint32_t k = lo; k < hi; ++k) { const unsigned long long v = part[k]; part[k] = at; at += v; }
}

// Thread i moves its replica's records to out[position ..] and empties the FIFO.  `out` may be mapped host memory.
__global__ void fsm_pack_kernel(const Dev d, const unsigned long long* part, FsmHeader* hdr, uint4* out, uint32_t cap_records) {
  __shared__ uint32_t s_warp[SCAN_THREADS / 32];
  const size_t plane = (size_t)d.R * d.Gp;
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const uint32_t n = i < plane ? fsm_kept(d, i, d.fc[i]) : 0u;
  // exclusive scan of n over the CTA
  uint32_t pre = 0;
#ifdef JR_EMU
  (void)s_warp;
#else
  const uint32_t lane = threadIdx.x & 31u, w = threadIdx.x >> 5;
  uint32_t inc = n;
  for (int o = 1; o < 32; o <<= 1) {
    const uint32_t v = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= (uint32_t)o) inc += v;
  }
  if (lane == 31) s_warp[w] = inc;
  __syncthreads();
  uint32_t base = 0;
  for (uint32_t k = 0; k < w; ++k) base += s_warp[k];
  pre = base + inc - n;
#endif
  const unsigned long long at64 = part[blockIdx.x] + pre;
  if (i < plane) {
    const uint32_t at = (uint32_t)min(at64, (unsigned long long)cap_records);
    for (uint32_t k = 0; k < n && at + k < cap_records; ++k) {
      out[(size_t)2 * (at + k)] = d.fs[(size_t)(2 * k) * plane + i];
      out[(size_t)2 * (at + k) + 1] = d.fs[(size_t)(2 * k + 1) * plane + i];
    }
    if (i % d.Gp == 0) hdr->node_offset[i / d.Gp] = at;
    if (i + 1 == plane) hdr->node_offset[d.R] = (uint32_t)min(at64 + n, (unsigned long long)cap_records);
    d.fc[i] = make_uint2(0, 0);
  }
}

__global__ void max_u32_kernel(const uint32_t* v, size_t n, uint32_t* out) {
  uint32_t m = 0;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    m = max(m, v[i]);
#ifndef JR_EMU
  for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_down_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0)
#endif
    atomicMax(out, m);
}

// ============================================================================
// host side
// ============================================================================

extern "C" { static jr_status stream_sums(jr_engine* e, uint64_t v[5]); }
static thread_local char g_err[512] = "";
static void set_err(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof g_err, fmt, ap);
  va_end(ap);
}

#define CK(call)                                                                      \
  do {                                                                                \
    cudaError_t _e = (call);                                                          \
    if (_e != cudaSuccess) {                                                          \
      set_err("%s:%d %s: %s", __FILE__, __LINE__, #call, cudaGetErrorString(_e));     \
      return JR_E_CUDA;                                                               \
    }                                                                                 \
  } while (0)

struct jr_engine {
  jr_config cfg;
  Dev d;
  cudaStream_t stream = nullptr;
  cudaStream_t own_stream = nullptr;
  volatile uint32_t* h_scatter = nullptr;  // pinned + mapped: epoch of the last launch that saw scattered leaders (written by the kernel)
  volatile uint32_t* h_unfolded = nullptr; // pinned + mapped: epoch of the last launch whose fold left some group to step_kernel (0: never)
  uint32_t ticket_sum = 0;                 // tickets taken so far (the counter is never reset: each launch gets its base)
  int force_sorted = 0;      // JR_STEP_VARIANT=sorted|plain pins the kernel variant (tests, A/B)
  uint64_t launches_sorted = 0, launches_total = 0, launches_split = 0;
  uint32_t slots = 0;        // CTAs of the step kernel the device holds at once (occupancy x SMs)
  uint32_t force_parts = 0;  // JR_PARTS=n pins the split (tests, A/B); 0 = choose_parts
  int cur = 0;               // outbox index the NEXT step writes
  uint64_t step_index = 0;
  std::vector<void*> allocs;
  // scratch
  unsigned long long* scratch = nullptr;  // 8 x u64 (device)
  jr_msg* inj_msgs = nullptr;             // device, grows
  uint4* inj_targets = nullptr;
  size_t inj_cap = 0;
  // Copy/compute overlap for the host-buffer path: proposals are staged H2D on `h2d`,
  // leader tables leave D2H on `d2h`, both double buffered and fenced with events, so the
  // copy-in of tick k+1, the kernels of tick k and the copy-out of tick k-1 run concurrently.
  static constexpr int NBUF = JR_STAGING_DEPTH;   // staging depth: a host may keep three steps in flight (copy-out, host fold and the next submit overlap)
  jr_proposal* prop[NBUF] = {nullptr, nullptr};         // device, G entries each
  jr_leader_entry* leaders[NBUF] = {nullptr, nullptr};  // device, G entries each
  cudaStream_t h2d = nullptr, d2h = nullptr;
  cudaEvent_t prop_ready[NBUF] = {nullptr, nullptr};    // H2D of prop[i] finished
  cudaEvent_t prop_free[NBUF] = {nullptr, nullptr};     // the kernel that read prop[i] finished
  cudaEvent_t tab_ready[NBUF] = {nullptr, nullptr};     // leader_table_kernel into leaders[i] finished
  cudaEvent_t tab_free[NBUF] = {nullptr, nullptr};      // D2H of leaders[i] finished
  bool prop_used[NBUF] = {false, false}, tab_used[NBUF] = {false, false};
  jr_proposal* batch[NBUF] = {nullptr, nullptr};        // device, batch_cap entries each (jr_run_proposals)
  size_t batch_cap[NBUF] = {0, 0};
  cudaEvent_t batch_ready[NBUF] = {nullptr, nullptr}, batch_free[NBUF] = {nullptr, nullptr};
  bool batch_used[NBUF] = {false, false};
  int batch_i = 0;
  unsigned long long* tokbuf[NBUF] = {nullptr, nullptr};  // device staging of jr_run_tokens input, tok_cap entries each
  size_t tok_cap[NBUF] = {0, 0};
  uint32_t* route = nullptr;              // device, G entries: leader_id of the last leader-table call (0 = none)
  int tab_pending[NBUF] = {0, 0};  // FIFO of leaders[] buffers whose copy-out has not been waited for
  int tab_npending = 0;
  int prop_i = 0, tab_i = 0;
  // scratch of the *_many introspection calls (device, grows)
  void* many_buf = nullptr;
  size_t many_cap = 0;
  // Instruction-stream drain (JR_F_CAPTURE_FSM): scan -> pack into stage[b] on the engine stream, then
  // the copy engine moves stage[b] into the pinned host buffer host[fsm_host_of[b]] on the d2h stream.
  // The host buffers rotate on their own, one more of them than stage buffers: with NBUF batches outstanding, the
  // async right after a wait must not land in the buffer that wait has just returned (it stays the caller's until
  // the NBUF-1'th async after the wait, include/josefine_raft_abi.h).
  static constexpr int NHOST = NBUF + 1;
  unsigned long long* fsm_part = nullptr;                     // device, 3 x (CTAs of the count/pack kernels): per-CTA sums -> offsets
  uint32_t fsm_cap = 0;                                       // records per batch
  uint4* fsm_stage[NBUF] = {nullptr, nullptr};                // device, 2 * fsm_cap uint4 each
  FsmHeader* fsm_stage_hdr[NBUF] = {nullptr, nullptr};        // device
  uint4* fsm_host[NHOST] = {nullptr, nullptr};                // pinned + mapped host
  int fsm_host_of[NBUF] = {0, 0};                             // host buffer the batch in stage[b] lands in
  int fsm_hi = 0;                                             // next host buffer
  FsmHeader* fsm_host_hdr[NBUF] = {nullptr, nullptr};         // pinned + mapped host
  cudaEvent_t fsm_packed[NBUF] = {nullptr, nullptr};          // pack into stage[b] finished (engine stream)
  cudaEvent_t fsm_landed[NBUF] = {nullptr, nullptr};          // copy of stage[b] to the host finished (d2h stream)
  size_t fsm_copied[NBUF] = {0, 0};                           // records of stage[b] the enqueued copy covers
  size_t fsm_last_records = 0;                                // size of the last batch taken (the next copy's guess)
  bool fsm_used[NBUF] = {false, false};
  int fsm_i = 0, fsm_pending[NBUF] = {0, 0}, fsm_npending = 0;
  std::mutex qmu;   // the two FIFOs of outstanding copy-outs (fsm_pending, tab_pending) and fsm_last_records: a second host thread may
                    // sit in jr_fsm_records_wait / jr_leader_table_wait while the first one keeps submitting
  // symmetric-group fold
  uint8_t* symdone = nullptr;   // device, Gp entries
  uint8_t* symblk = nullptr;    // device, Gp / 32 entries
  bool auto_trunc = false;      // jr_set_auto_truncate
  uint32_t auto_trunc_margin = 0;
  uint64_t launches_folded = 0;
  bool last_launch_folded = false;
};

template <typename T>
static jr_status dalloc(jr_engine* e, T** p, size_t n) {
  void* q = nullptr;
  cudaError_t err = cudaMalloc(&q, n * sizeof(T));
  if (err != cudaSuccess) {
    set_err("cudaMalloc(%zu bytes): %s", n * sizeof(T), cudaGetErrorString(err));
    return err == cudaErrorMemoryAllocation ? JR_E_NOMEM : JR_E_CUDA;
  }
  e->allocs.push_back(q);
  *p = (T*)q;
  return JR_OK;
}

#define DISPATCH_R(R_, CALL)           \
  switch (R_) {                        \
    case 1: { constexpr int RR = 1; CALL; } break; \
    case 2: { constexpr int RR = 2; CALL; } break; \
    case 3: { constexpr int RR = 3; CALL; } break; \
    case 4: { constexpr int RR = 4; CALL; } break; \
    case 5: { constexpr int RR = 5; CALL; } break; \
    case 6: { constexpr int RR = 6; CALL; } break; \
    case 7: { constexpr int RR = 7; CALL; } break; \
    default: { constexpr int RR = 8; CALL; } break; \
  }

template <int R>
static void launch_step_r(jr_engine* e, const StepParams& p, bool sorted, uint32_t grid, size_t smem) {
  auto kfn = sorted ? step_kernel<R, true> : step_kernel<R, false>;
  JR_LAUNCH_SMEM(kfn, grid, 32 * R, smem, e->stream, e->d, p);
}

template <int R>
static cudaError_t step_smem_attr_r(int smem) {
  cudaError_t a = cudaFuncSetAttribute(step_kernel<R, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
  if (a != cudaSuccess) return a;
  return cudaFuncSetAttribute(step_kernel<R, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
}

#ifndef JR_EMU
template <int R>
static cudaError_t step_occupancy_r(int* per_sm, int smem) {
  return cudaOccupancyMaxActiveBlocksPerMultiprocessor(per_sm, step_kernel<R, false>, 32 * R, (size_t)smem);
}
#endif

static size_t step_smem_bytes(const Dev& d) {
  return ((size_t)2 * d.Us + d.W) * d.R * 32 * sizeof(uint4) + (size_t)2 * d.R * 32 * sizeof(uint32_t) +
         (size_t)2 * d.R * d.R * 32 * sizeof(uint16_t);
}

// How many consecutive tasks to cut each block's ticks into: the fewest that minimise the number of
// rounds the CTA slots need, in units of a whole-launch task.  1 when the grid fits the slots anyway,
// when the launch is short, or when its first tick is not a whole tick (jr_step's split phases).
static uint32_t choose_parts(const jr_engine* e, const StepParams& p, uint32_t n_blocks) {
  const uint32_t whole = PH_RESET_OUT | PH_DRAIN | PH_TICK;
  if ((p.phases & whole) != whole || p.n_ticks < 2) return 1;
  if (e->force_parts) return std::min<uint32_t>(e->force_parts, p.n_ticks);
  if (!e->slots || n_blocks <= e->slots) return 1;
  uint32_t best = 1;
  double best_rounds = (double)((n_blocks + e->slots - 1) / e->slots);
  for (uint32_t n = 2; n <= 8 && p.n_ticks / n >= 8; n *= 2) {
    const double rounds = (double)(((size_t)n_blocks * n + e->slots - 1) / e->slots) / n;
    if (rounds < best_rounds * 0.97) { best = n; best_rounds = rounds; }
  }
  return best;
}

static jr_status launch_step_once(jr_engine* e, const StepParams& p_in);

// A capturing engine keeps every launch short enough for the raw Instruction FIFO (Fr entries per replica, encoded when
// the launch ends): at most Fr / 3 ticks per launch.  Consecutive launches are indistinguishable from one long launch.
static jr_status launch_step(jr_engine* e, const StepParams& p_in) {
  const uint32_t limit = (e->d.flags & JR_F_CAPTURE_FSM) ? std::max(1u, e->d.Fr / 3u) : 0xffffffffu;
  if (p_in.n_ticks <= limit) return launch_step_once(e, p_in);
  StepParams p = p_in;
  for (uint32_t done = 0; done < p_in.n_ticks;) {
    p.n_ticks = std::min(limit, p_in.n_ticks - done);
    p.trunc = (p_in.trunc && done + p.n_ticks == p_in.n_ticks) ? 1u : 0u;   // the call ends with ONE truncation
    jr_status st = launch_step_once(e, p);
    if (st != JR_OK) return st;
    done += p.n_ticks;
    p.now += (uint64_t)p.n_ticks * p.dt;
    p.step_index += p.n_ticks;
    p.cur ^= (int)(p.n_ticks & 1u);
    if (p.proposals) p.proposals += (size_t)p.n_ticks * p.prop_stride;
    p.tok_tick += p.n_ticks;
    p.phases = PH_RESET_OUT | PH_DRAIN | (p_in.phases & PH_PROPOSE) | PH_TICK;
  }
  return JR_OK;
}

template <int R>
static void launch_sym_r(jr_engine* e, const StepParams& p) {
  if constexpr (R >= 2)
    JR_LAUNCH_SMEM(sym2_kernel<R>, (e->d.Gp + SYM2_GROUPS - 1) / SYM2_GROUPS, 2 * SYM2_GROUPS,
                   (size_t)SYM2_UNITS * SYM2_GROUPS * sizeof(uint4), e->stream, e->d, p, e->symdone, e->symblk);
}

// May this launch be offered to the symmetric-group fold?  (Whether a GROUP takes it is sym_enter's decision.)
static bool fold_eligible(const jr_engine* e, const StepParams& p) {
  const Dev& d = e->d;
  const uint32_t whole = PH_RESET_OUT | PH_DRAIN | PH_TICK;
  if (d.flags & (JR_F_STREAM_DIGEST | JR_F_SLED_COMMIT_KEY_STRICT | JR_F_NO_SYMMETRIC_FOLD)) return false;
  if (d.R < 2 || d.U < d.R + 7 || d.resident != 0xffu || p.dt == 0) return false;
  if ((p.phases & ~(uint32_t)PH_PROPOSE) != whole || p.n_ticks < 2) return false;
  if (p.proposals && p.prop_stride != d.G) return false;
  return true;   // (tok_runs: always per-tick)
}

static jr_status launch_step_once(jr_engine* e, const StepParams& p_in) {
  const uint32_t n_blocks = e->d.Gp / GROUPS_PER_CTA;
  const size_t smem = step_smem_bytes(e->d);
  StepParams p = p_in;
  p.epoch = (uint32_t)(e->launches_total + 1) * 8u;
  if (fold_eligible(e, p)) {
    DISPATCH_R(e->cfg.n_replicas, (launch_sym_r<RR>(e, p)));
    CK(cudaGetLastError());
    p.symdone = e->symdone;
    p.symblk = e->symblk;
    e->launches_folded += 1;
  }
  e->last_launch_folded = p.symdone != nullptr;
  p.n_parts = choose_parts(e, p, n_blocks);
  // When the fold has been taking every group (no launch of the last two left one behind -- a hint the kernel stores in
  // mapped host memory), step_kernel's CTAs only look at symblk and return: do not cut them in parts, which would cost
  // each of them a ticket and two barriers first.  A wrong guess costs balance in that one launch, nothing else.
  if (p.symdone && e->h_unfolded && (*e->h_unfolded == 0 || p.epoch - *e->h_unfolded > 2u * 8u) && !e->force_parts)
    p.n_parts = 1;
  p.part_ticks = (p.n_ticks + p.n_parts - 1) / p.n_parts;
  p.n_parts = (p.n_ticks + p.part_ticks - 1) / p.part_ticks;  // no empty trailing part
  p.n_blocks = n_blocks;
  const uint32_t grid = n_blocks * p.n_parts;
  // Variant choice from the (possibly one launch stale) scatter flag: it only affects speed.
  // (the kernel stores its epoch into that mapped host word: no memset, no copy-back in the launch path)
  const bool sorted = e->force_sorted > 0 || (e->force_sorted == 0 && e->h_scatter && *e->h_scatter != 0 && p.epoch - *e->h_scatter <= 2u * 8u);
  p.ticket_base = e->ticket_sum;
  if (p.n_parts > 1) e->ticket_sum += grid;
  DISPATCH_R(e->cfg.n_replicas, (launch_step_r<RR>(e, p, sorted, grid, smem)));
  CK(cudaGetLastError());
  if (p.trunc) {   // sym2_kernel truncated the groups it folded
    JR_LAUNCH(truncate_kernel, (e->d.Gp + 127) / 128, 128, e->stream, e->d, p.trunc_margin, p.symdone);
    CK(cudaGetLastError());
  }
  e->launches_sorted += sorted ? 1 : 0;
  e->launches_split += p.n_parts > 1 ? 1 : 0;
  e->launches_total += 1;
  return JR_OK;
}

extern "C" {

#ifdef JR_EMU
// Marker of the TEST-ONLY host build (tests/emu): the package loader refuses a library that has it.
int jr_is_emulation(void) { return 1; }
#endif

const char* jr_last_error(void) { return g_err; }

void jr_config_default(jr_config* cfg, uint32_t n_groups, uint32_t n_replicas) {
  if (!cfg) return;
  memset(cfg, 0, sizeof *cfg);
  cfg->abi_version = JR_ABI_VERSION;
  cfg->n_groups = n_groups;
  cfg->n_replicas = n_replicas;
  cfg->election_min_ms = 500;   // mod.rs:318
  cfg->election_max_ms = 1000;  // mod.rs:319
  cfg->heartbeat_ms = 100;      // config.rs:104
  cfg->chain_capacity = 4096;
  cfg->mailbox_units = 64;
  cfg->fsm_units = 64;
}

uint32_t jr_election_timeout(uint64_t seed, uint64_t group, uint32_t node, uint32_t draw, uint32_t mn,
                             uint32_t mx) {
  return election_timeout_draw(seed, group, node, draw, mn, mx);
}

jr_status jr_engine_create(const jr_config* cfg, jr_engine** out) {
  if (!cfg || !out) return JR_E_INVAL;
  // RaftConfig::validate analogue (config.rs:60-84)
  if (cfg->abi_version != JR_ABI_VERSION) { set_err("abi_version mismatch"); return JR_E_INVAL; }
  if (cfg->n_replicas < 1 || cfg->n_replicas > JR_MAX_REPLICAS || cfg->n_groups < 1) { set_err("bad G/R"); return JR_E_INVAL; }
  if (cfg->election_max_ms <= cfg->election_min_ms) { set_err("empty election timeout range"); return JR_E_INVAL; }
  // RaftConfig::validate, config.rs:70-75 (the rules that have a counterpart here)
  if (cfg->heartbeat_ms < 5) { set_err("heartbeat timeout is too low"); return JR_E_INVAL; }
  if (cfg->election_min_ms < 5) { set_err("election timeout is too low"); return JR_E_INVAL; }
  if (cfg->chain_capacity < 2 || cfg->chain_capacity > 0x40000000u) { set_err("chain_capacity out of range"); return JR_E_INVAL; }
  if (cfg->mailbox_units < 8 || cfg->fsm_units < 1) { set_err("mailbox_units >= 8, fsm_units >= 1"); return JR_E_INVAL; }
  if (cfg->fsm_units > (1u << 20) || cfg->fsm_raw_units > (1u << 20) || (cfg->fsm_raw_units && cfg->fsm_raw_units < 32)) {
    set_err("fsm_units <= 2^20, 32 <= fsm_raw_units <= 2^20");
    return JR_E_INVAL;
  }
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    set_err("no CUDA device; this library has no CPU fallback");
    return JR_E_NO_DEVICE;
  }
  if (cfg->device < 0 || cfg->device >= ndev) { set_err("device ordinal %d out of range", cfg->device); return JR_E_INVAL; }
  CK(cudaSetDevice(cfg->device));
  jr_engine* e = new (std::nothrow) jr_engine();
  if (!e) return JR_E_NOMEM;
  e->cfg = *cfg;
  Dev& d = e->d;
  memset(&d, 0, sizeof d);
  d.G = cfg->n_groups;
  d.Gp = (cfg->n_groups + GROUPS_PER_CTA - 1) / GROUPS_PER_CTA * GROUPS_PER_CTA;
  d.R = cfg->n_replicas;
  d.cap = cfg->chain_capacity;
  d.capm = 1;
  while (d.capm < d.cap) d.capm <<= 1;   // table rows: the power of two >= cap, so row = id & capm
  d.capm -= 1;
  d.U = cfg->mailbox_units;
  d.F = cfg->fsm_units;
  d.Fr = cfg->fsm_raw_units ? cfg->fsm_raw_units : 192u;
  d.flags = cfg->flags;
  d.emin = cfg->election_min_ms;
  d.emax = cfg->election_max_ms;
  d.hb = cfg->heartbeat_ms;
  d.seed = cfg->seed;
  d.goff = cfg->group_offset;
  // shared-memory staging: Us mailbox units per replica per buffer, W table-cache entries
  d.Us = std::min<uint32_t>(cfg->mailbox_units, 6u);
  d.W = 4;
  d.use_index = getenv("JR_NO_INDEX") ? 0u : 1u;
  d.resident = cfg->resident_mask ? cfg->resident_mask : 0xffu;
  if (const char* ev = getenv("JR_SMEM_UNITS")) d.Us = std::min<uint32_t>(cfg->mailbox_units, (uint32_t)atoi(ev));
  if (const char* ev = getenv("JR_TABLE_CACHE")) { uint32_t w = (uint32_t)atoi(ev); d.W = (w & (w - 1)) ? 8 : w; }
  const size_t plane = (size_t)d.R * d.Gp;
  jr_status st = JR_OK;
#define A(ptr, n) if (st == JR_OK) st = dalloc(e, &(ptr), (n))
  A(d.p0, plane); A(d.p1, plane); A(d.p2, plane); A(d.p3, plane);
  A(d.pr, plane * ((d.R + 3) / 4));
  A(d.mk, plane);
  A(d.qt, plane * JR_CLIENT_QUEUE_CAP);
  A(d.dg, plane); A(d.cn, plane);
  A(d.cnext, plane * ((size_t)d.capm + 1));
  A(d.ctok, plane * ((size_t)d.capm + 1));
  A(d.ob[0], plane * (size_t)d.U); A(d.ob[1], plane * (size_t)d.U);
  A(d.oc[0], plane); A(d.oc[1], plane);
  A(d.fs, plane * (size_t)((d.flags & JR_F_CAPTURE_FSM) ? 2 * (size_t)d.F : 1));
  A(d.fc, plane);
  A(d.fq, plane);
  A(d.fr, plane * (size_t)((d.flags & JR_F_CAPTURE_FSM) ? d.Fr : 1));
  A(d.tb, d.Gp);
  A(e->symdone, d.Gp);
  A(e->symblk, d.Gp / GROUPS_PER_CTA);
  if (d.flags & JR_F_CAPTURE_FSM) {
    const size_t reps = (size_t)cfg->n_groups * cfg->n_replicas;   // default: 2 per replica, but never less than a small engine's whole FIFO space
    const size_t want = cfg->fsm_host_records ? cfg->fsm_host_records
                                              : std::max(3 * reps + 1024, std::min<size_t>(reps * cfg->fsm_units, 1u << 16));
    e->fsm_cap = (uint32_t)std::min<size_t>(want, 0x7fffffffu);
    A(e->fsm_part, 3 * plane);   // (sized for one-thread CTAs, which is what the CPU emulation launches)
    for (int i = 0; i < jr_engine::NBUF; ++i) { A(e->fsm_stage[i], 2 * (size_t)e->fsm_cap); A(e->fsm_stage_hdr[i], 1); }
  }
  A(e->scratch, 8);
  A(d.scatter, 2);
  A(d.done, d.Gp / GROUPS_PER_CTA);
#ifdef JR_PROFILE
  A(d.prof, 3 * 16 * 2);
#endif
  for (int i = 0; i < jr_engine::NBUF; ++i) { A(e->prop[i], d.G); A(e->leaders[i], d.G); }
  A(e->route, d.G);
#undef A
  if (st != JR_OK) { jr_engine_destroy(e); return st; }
  if (cudaStreamCreateWithFlags(&e->own_stream, cudaStreamNonBlocking) != cudaSuccess) {
    set_err("cudaStreamCreate failed");
    jr_engine_destroy(e);
    return JR_E_CUDA;
  }
  e->stream = e->own_stream;
  {
    bool ok = cudaStreamCreateWithFlags(&e->h2d, cudaStreamNonBlocking) == cudaSuccess &&
              cudaStreamCreateWithFlags(&e->d2h, cudaStreamNonBlocking) == cudaSuccess;
    for (int i = 0; ok && i < jr_engine::NBUF; ++i)
      ok = cudaEventCreateWithFlags(&e->prop_ready[i], cudaEventDisableTiming) == cudaSuccess &&
           cudaEventCreateWithFlags(&e->prop_free[i], cudaEventDisableTiming) == cudaSuccess &&
           cudaEventCreateWithFlags(&e->tab_ready[i], cudaEventDisableTiming) == cudaSuccess &&
           cudaEventCreateWithFlags(&e->tab_free[i], cudaEventDisableTiming) == cudaSuccess &&
           cudaEventCreateWithFlags(&e->batch_ready[i], cudaEventDisableTiming) == cudaSuccess &&
           cudaEventCreateWithFlags(&e->batch_free[i], cudaEventDisableTiming) == cudaSuccess &&
           cudaEventCreateWithFlags(&e->fsm_packed[i], cudaEventDisableTiming) == cudaSuccess &&
           cudaEventCreateWithFlags(&e->fsm_landed[i], cudaEventDisableTiming) == cudaSuccess;
    for (int i = 0; ok && e->fsm_cap && i < jr_engine::NHOST; ++i)   // the drain's landing buffers: pinned, device-visible
      ok = cudaHostAlloc((void**)&e->fsm_host[i], (size_t)e->fsm_cap * sizeof(jr_fsm_record), cudaHostAllocMapped) == cudaSuccess;
    for (int i = 0; ok && e->fsm_cap && i < jr_engine::NBUF; ++i)
      ok = cudaHostAlloc((void**)&e->fsm_host_hdr[i], sizeof(FsmHeader), cudaHostAllocMapped) == cudaSuccess;
    if (!ok) {
      set_err("copy streams / events could not be created");
      jr_engine_destroy(e);
      return JR_E_CUDA;
    }
  }
  {
    const int smem = (int)step_smem_bytes(d);
    cudaError_t aerr = cudaSuccess;
    DISPATCH_R(d.R, (aerr = step_smem_attr_r<RR>(smem)));
    if (aerr == cudaSuccess) aerr = cudaHostAlloc((void**)&e->h_scatter, sizeof(uint32_t), cudaHostAllocMapped);
    if (aerr == cudaSuccess) *e->h_scatter = 0;
    if (aerr == cudaSuccess) aerr = cudaHostGetDevicePointer((void**)&e->d.hscat, (void*)e->h_scatter, 0);
    if (aerr == cudaSuccess) aerr = cudaHostAlloc((void**)&e->h_unfolded, sizeof(uint32_t), cudaHostAllocMapped);
    if (aerr == cudaSuccess) *e->h_unfolded = 0;
    if (aerr == cudaSuccess) aerr = cudaHostGetDevicePointer((void**)&e->d.hunf, (void*)e->h_unfolded, 0);
    if (const char* ev = getenv("JR_PARTS")) e->force_parts = (uint32_t)std::min(std::max(atoi(ev), 0), 8);
#ifndef JR_EMU
    if (aerr == cudaSuccess) {
      int per_sm = 0, sms = 0;
      DISPATCH_R(d.R, (aerr = step_occupancy_r<RR>(&per_sm, smem)));
      if (aerr == cudaSuccess) aerr = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, cfg->device);
      e->slots = (uint32_t)(per_sm * sms);
    }
#endif
    if (const char* ev = getenv("JR_STEP_VARIANT")) e->force_sorted = !strcmp(ev, "sorted") ? 1 : (!strcmp(ev, "plain") ? -1 : 0);
    if (aerr != cudaSuccess) {
      set_err("step kernel needs %d bytes of shared memory: %s", smem, cudaGetErrorString(aerr));
      jr_engine_destroy(e);
      return JR_E_CUDA;
    }
  }
  if (jr_engine_reset(e) != JR_OK) {
    jr_engine_destroy(e);
    return JR_E_CUDA;
  }
  *out = e;
  return JR_OK;
}

#ifdef JR_PROFILE
// Profiling builds only (not part of the ABI): read and clear the phase counters.
jr_status jr_profile_read(jr_engine* e, unsigned long long* out96) {
  if (!e || !out96) return JR_E_INVAL;
  CK(cudaStreamSynchronize(e->stream));
  CK(cudaMemcpyAsync(out96, e->d.prof, 96 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, e->stream));
  CK(cudaMemsetAsync(e->d.prof, 0, 96 * sizeof(unsigned long long), e->stream));
  CK(cudaStreamSynchronize(e->stream));
  return JR_OK;
}
#endif

jr_status jr_engine_reset(jr_engine* e) {
  if (!e) return JR_E_INVAL;
  CK(cudaSetDevice(e->cfg.device));
  const Dev& d = e->d;
  const size_t plane = (size_t)d.R * d.Gp;
  // block tables start empty (all keys absent); pr / qt zero
  CK(cudaMemsetAsync(d.cnext, 0xFF, plane * ((size_t)d.capm + 1) * sizeof(uint32_t), e->stream));
  CK(cudaMemsetAsync(d.pr, 0, plane * ((d.R + 3) / 4) * sizeof(uint4), e->stream));
  CK(cudaMemsetAsync(d.qt, 0, plane * JR_CLIENT_QUEUE_CAP * sizeof(uint4), e->stream));
  CK(cudaMemsetAsync(e->route, 0, (size_t)d.G * sizeof(uint32_t), e->stream));  // no leader announced yet
  CK(cudaMemsetAsync(d.done, 0, (size_t)(d.Gp / GROUPS_PER_CTA) * sizeof(uint32_t), e->stream));
  CK(cudaMemsetAsync(d.scatter, 0, 2 * sizeof(uint32_t), e->stream));   // [1] = the ticket counter: from here on only launches move it,
  e->ticket_sum = 0;                                                     //       and each one is told where it stands (ticket_base)
  JR_LAUNCH(init_kernel, (unsigned)((plane + 255) / 256), 256, e->stream, d);
  CK(cudaGetLastError());
  CK(cudaStreamSynchronize(e->stream));
  e->cur = 0;
  e->step_index = 0;
  // (h_scatter keeps its last value: advisory only, and a reset is usually followed by the same workload)
#ifdef JR_PROFILE
  CK(cudaMemsetAsync(e->d.prof, 0, 96 * sizeof(unsigned long long), e->stream));
#endif
  return JR_OK;
}

void jr_engine_destroy(jr_engine* e) {
  if (!e) return;
  if (getenv("JR_DEBUG_VARIANT"))
    fprintf(stderr, "[jr] engine %p: %llu step launches, %llu role-sorted, %llu split, %llu offered to the fold; %u CTA slots\n",
            (void*)e, (unsigned long long)e->launches_total, (unsigned long long)e->launches_sorted,
            (unsigned long long)e->launches_split, (unsigned long long)e->launches_folded, e->slots);
  cudaSetDevice(e->cfg.device);
  if (e->stream) cudaStreamSynchronize(e->stream);
  for (void* p : e->allocs) cudaFree(p);
  if (e->inj_msgs) cudaFree(e->inj_msgs);
  if (e->inj_targets) cudaFree(e->inj_targets);
  if (e->many_buf) cudaFree(e->many_buf);
  if (e->h2d) { cudaStreamSynchronize(e->h2d); cudaStreamDestroy(e->h2d); }
  if (e->d2h) { cudaStreamSynchronize(e->d2h); cudaStreamDestroy(e->d2h); }
  for (int i = 0; i < jr_engine::NBUF; ++i) {
    if (e->prop_ready[i]) cudaEventDestroy(e->prop_ready[i]);
    if (e->prop_free[i]) cudaEventDestroy(e->prop_free[i]);
    if (e->tab_ready[i]) cudaEventDestroy(e->tab_ready[i]);
    if (e->tab_free[i]) cudaEventDestroy(e->tab_free[i]);
    if (e->batch_ready[i]) cudaEventDestroy(e->batch_ready[i]);
    if (e->batch_free[i]) cudaEventDestroy(e->batch_free[i]);
    if (e->fsm_packed[i]) cudaEventDestroy(e->fsm_packed[i]);
    if (e->fsm_landed[i]) cudaEventDestroy(e->fsm_landed[i]);
    if (e->fsm_host_hdr[i]) cudaFreeHost(e->fsm_host_hdr[i]);
    if (e->batch[i]) cudaFree(e->batch[i]);
    if (e->tokbuf[i]) cudaFree(e->tokbuf[i]);
  }
  for (int i = 0; i < jr_engine::NHOST; ++i)
    if (e->fsm_host[i]) cudaFreeHost(e->fsm_host[i]);
  if (e->h_scatter) cudaFreeHost((void*)e->h_scatter);
  if (e->h_unfolded) cudaFreeHost((void*)e->h_unfolded);
  if (e->own_stream) cudaStreamDestroy(e->own_stream);
  delete e;
}

jr_status jr_engine_set_stream(jr_engine* e, void* s) {
  if (!e) return JR_E_INVAL;
  CK(cudaStreamSynchronize(e->stream));
  e->stream = s ? (cudaStream_t)s : e->own_stream;
  return JR_OK;
}

jr_status jr_engine_sync(jr_engine* e) {
  if (!e) return JR_E_INVAL;
  CK(cudaStreamSynchronize(e->h2d));
  CK(cudaStreamSynchronize(e->stream));
  CK(cudaStreamSynchronize(e->d2h));
  return JR_OK;
}

// ---- capture: decode raw mailboxes / FIFOs on the host --------------------------------

static void decode_unit(const uint4& h, uint32_t group, uint32_t sender, const uint4* blocks, size_t stride,
                        std::vector<jr_msg>& out) {
  const uint32_t kind = h.x & 15u, flag = (h.x >> 4) & 1u, aux = (h.x >> 8) & 255u, to = h.x >> 16;
  jr_msg m;
  memset(&m, 0, sizeof m);
  m.group = group;
  m.from_kind = JR_ADDR_PEER;
  m.from_id = sender;
  m.to_kind = to == TO_PEERS ? JR_ADDR_PEERS : (to == TO_CLIENT ? JR_ADDR_CLIENT : JR_ADDR_PEER);
  m.to_id = m.to_kind == JR_ADDR_PEER ? to : 0;
  m.kind = (uint8_t)kind;
  const uint64_t t = (uint64_t)h.y | ((uint64_t)h.z << 32);
  uint32_t copies = 1;
  switch (kind) {
    case JR_CMD_VOTE_REQUEST: m.term = t; m.node_id = sender; m.last_term = t; m.block = h.w; copies = aux; break;
    case JR_CMD_VOTE_RESPONSE: m.term = t; m.node_id = sender; m.flag = flag; break;
    case JR_CMD_APPEND_ENTRIES:
      m.term = t; m.node_id = sender; m.n_blocks = (uint8_t)aux;
      for (uint32_t k = 0; k < aux && k < JR_MAX_AE_BLOCKS; ++k) {
        const uint4& b = blocks[(size_t)k * stride];
        m.blocks[k] = jr_block{b.x, b.y, (uint64_t)b.z | ((uint64_t)b.w << 32)};
      }
      break;
    case JR_CMD_APPEND_RESPONSE: m.node_id = sender; m.term = t; m.block = h.w; m.flag = flag; break;
    case JR_CMD_HEARTBEAT: m.term = t; m.block = h.w; m.node_id = sender; break;
    case JR_CMD_HEARTBEAT_RESPONSE: m.block = h.w; m.flag = flag; break;
    case JR_CMD_CLIENT_REQUEST: m.token = t; m.client_kind = (uint8_t)(h.w >> 16); m.client_id = h.w & 0xffffu; break;
    case JR_CMD_CLIENT_RESPONSE: m.token = t; break;
    default: break;
  }
  for (uint32_t k = 0; k < copies; ++k) out.push_back(m);
}

static jr_status device_max(jr_engine* e, const uint32_t* v, size_t n, uint32_t* out) {
  uint32_t* s = reinterpret_cast<uint32_t*>(e->scratch);
  CK(cudaMemsetAsync(s, 0, sizeof(uint32_t), e->stream));
  JR_LAUNCH(max_u32_kernel, 64, 256, e->stream, v, n, s);
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(out, s, sizeof(uint32_t), cudaMemcpyDeviceToHost, e->stream));
  CK(cudaStreamSynchronize(e->stream));
  return JR_OK;
}

static jr_status capture_messages(jr_engine* e, int buf, std::vector<jr_msg>& out) {
  const Dev& d = e->d;
  const size_t plane = (size_t)d.R * d.Gp;
  uint32_t mx = 0;
  jr_status st = device_max(e, d.oc[buf], plane, &mx);
  if (st != JR_OK) return st;
  std::vector<uint32_t> cnt(plane);
  CK(cudaMemcpyAsync(cnt.data(), d.oc[buf], plane * sizeof(uint32_t), cudaMemcpyDeviceToHost, e->stream));
  std::vector<uint4> units((size_t)mx * plane);
  if (mx) CK(cudaMemcpyAsync(units.data(), d.ob[buf], units.size() * sizeof(uint4), cudaMemcpyDeviceToHost, e->stream));
  CK(cudaStreamSynchronize(e->stream));
  for (uint32_t g = 0; g < d.G; ++g)
    for (uint32_t r = 0; r < d.R; ++r) {
      const size_t i = (size_t)r * d.Gp + g;
      for (uint32_t u = 0; u < cnt[i];) {
        const uint4& h = units[(size_t)u * plane + i];
        const uint32_t kind = h.x & 15u, aux = (h.x >> 8) & 255u;
        const bool ae = kind == JR_CMD_APPEND_ENTRIES, ref = ae && ((h.x >> 4) & 1u);
        const uint32_t span = 1 + ((ae && !ref) ? aux : 0u);
        const uint32_t first = ref ? h.w : u + 1;  // block run: inline, or shared with an earlier AppendEntries
        decode_unit(h, g, r + 1, (ae && aux) ? &units[(size_t)first * plane + i] : nullptr, plane, out);
        u += span;
      }
    }
  return JR_OK;
}

// ---- Instruction-stream drain -----------------------------------------------------------------

static jr_status fsm_records_enqueue(jr_engine* e) {
  const Dev& d = e->d;
  if (!(d.flags & JR_F_CAPTURE_FSM)) { set_err("engine created without JR_F_CAPTURE_FSM"); return JR_E_INVAL; }
  size_t last_records;
  {
    std::lock_guard<std::mutex> l(e->qmu);
    if (e->fsm_npending == jr_engine::NBUF) { set_err("%d batches outstanding: call jr_fsm_records_wait first", jr_engine::NBUF); return JR_E_INVAL; }
    last_records = e->fsm_last_records;
  }
  const int b = e->fsm_i, hb = e->fsm_hi;
  e->fsm_i = (b + 1) % jr_engine::NBUF;
  e->fsm_hi = (hb + 1) % jr_engine::NHOST;
  e->fsm_host_of[b] = hb;
  const size_t plane = (size_t)d.R * d.Gp;
  if (e->fsm_used[b]) CK(cudaStreamWaitEvent(e->stream, e->fsm_landed[b], 0));  // stage[b] has left the device
#ifdef JR_EMU
  const uint32_t T = 1, Ts = 1;
#else
  const uint32_t T = 256, Ts = SCAN_THREADS;
#endif
  const uint32_t n_ctas = (uint32_t)((plane + T - 1) / T);
  JR_LAUNCH(fsm_count_kernel, n_ctas, T, e->stream, d, e->fsm_part, n_ctas);
  CK(cudaGetLastError());
  JR_LAUNCH(fsm_scan_kernel, 1, Ts, e->stream, e->fsm_part, n_ctas, e->fsm_stage_hdr[b], e->fsm_cap);
  CK(cudaGetLastError());
  JR_LAUNCH(fsm_pack_kernel, n_ctas, T, e->stream, d, e->fsm_part, e->fsm_stage_hdr[b], e->fsm_stage[b], e->fsm_cap);
  CK(cudaGetLastError());
  CK(cudaEventRecord(e->fsm_packed[b], e->stream));
  CK(cudaStreamWaitEvent(e->d2h, e->fsm_packed[b], 0));
  // Copy engine, speculatively: the batch size is only known on the device, so copy as many records as the previous
  // batch held plus a margin; fsm_records_take fetches the rest in the (rare) case the batch turned out larger.
  // (A copy by the SMs would store to host memory through the LSUs the next step's kernel needs: that kernel is one wave
  // of CTAs, so the slowest SM sets its duration.  A DMA copy takes nothing from the SMs.)
  const size_t guess = std::min<size_t>(e->fsm_cap, std::max<size_t>(last_records + last_records / 8 + 1024, 16384));
  if (guess) CK(cudaMemcpyAsync(e->fsm_host[hb], e->fsm_stage[b], guess * sizeof(jr_fsm_record), cudaMemcpyDeviceToHost, e->d2h));
  CK(cudaMemcpyAsync(e->fsm_host_hdr[b], e->fsm_stage_hdr[b], sizeof(FsmHeader), cudaMemcpyDeviceToHost, e->d2h));
  e->fsm_copied[b] = guess;
  CK(cudaEventRecord(e->fsm_landed[b], e->d2h));
  e->fsm_used[b] = true;
  std::lock_guard<std::mutex> l(e->qmu);
  e->fsm_pending[e->fsm_npending++] = b;
  return JR_OK;
}

static jr_status fsm_records_take(jr_engine* e, const jr_fsm_record** recs, jr_fsm_batch* batch) {
  int b;
  {
    std::lock_guard<std::mutex> l(e->qmu);
    if (e->fsm_npending == 0) { set_err("no batch outstanding"); return JR_E_INVAL; }
    b = e->fsm_pending[0];   // (only this thread removes entries: the oldest stays b while the submitting thread appends)
  }
  uint4* host = e->fsm_host[e->fsm_host_of[b]];
  CK(cudaEventSynchronize(e->fsm_landed[b]));
  const FsmHeader h = *e->fsm_host_hdr[b];   // a copy: once stage[b] is released below, the next batch's header lands there
  if (h.n_records > e->fsm_copied[b]) {   // the speculative copy was short: fetch the tail now (stage[b] is still intact)
    const size_t have = e->fsm_copied[b];
    CK(cudaMemcpyAsync(reinterpret_cast<jr_fsm_record*>(host) + have, reinterpret_cast<const jr_fsm_record*>(e->fsm_stage[b]) + have,
                       ((size_t)h.n_records - have) * sizeof(jr_fsm_record), cudaMemcpyDeviceToHost, e->d2h));
    CK(cudaEventRecord(e->fsm_landed[b], e->d2h));
    CK(cudaEventSynchronize(e->fsm_landed[b]));
    e->fsm_copied[b] = h.n_records;
  }
  {
    // Only now is stage[b] free for the next jr_fsm_records_async: until the tail above had landed, a pack into it from
    // the submitting thread would have overwritten records not yet copied out.
    std::lock_guard<std::mutex> l(e->qmu);
    for (int k = 0; k + 1 < jr_engine::NBUF; ++k) e->fsm_pending[k] = e->fsm_pending[k + 1];
    --e->fsm_npending;
    e->fsm_last_records = h.n_records;
  }
  if (recs) *recs = reinterpret_cast<const jr_fsm_record*>(host);
  if (batch) {
    memset(batch, 0, sizeof *batch);
    batch->n_records = h.n_records;
    batch->n_dropped = h.n_dropped;
    batch->n_instructions = h.n_instructions;
    for (uint32_t r = 0; r <= JR_MAX_REPLICAS; ++r) batch->node_offset[r] = r <= e->d.R ? h.node_offset[r] : h.node_offset[e->d.R];
  }
  if (h.n_dropped) {
    set_err("%llu Instruction records were dropped (raise fsm_units / fsm_host_records, or drain more often)",
            (unsigned long long)h.n_dropped);
    return JR_E_CAPACITY;
  }
  return JR_OK;
}

// Synchronous drain into expanded Instructions (jr_step capture, jr_drain_fsm).
static jr_status capture_fsm(jr_engine* e, std::vector<jr_fsm_instr>& out) {
  const Dev& d = e->d;
  if (!(d.flags & JR_F_CAPTURE_FSM)) return JR_OK;
  if (e->fsm_npending) { set_err("jr_fsm_records_async batches are outstanding"); return JR_E_INVAL; }
  jr_status st = fsm_records_enqueue(e);
  if (st != JR_OK) return st;
  const jr_fsm_record* recs = nullptr;
  jr_fsm_batch batch;
  const jr_status took = fsm_records_take(e, &recs, &batch);
  if (took != JR_OK) return took;   // JR_E_CAPACITY: records are missing, so what is left cannot be expanded faithfully
  size_t n = 0;
  st = jr_fsm_expand(recs, batch.n_records, d.G, d.R, nullptr, 0, &n);
  if (st != JR_OK && st != JR_E_CAPACITY) return st;
  out.resize(n);
  if (n && (st = jr_fsm_expand(recs, batch.n_records, d.G, d.R, out.data(), n, &n)) != JR_OK) return st;
  return took;
}

// ---- jr_step ------------------------------------------------------------------------------

jr_status jr_step(jr_engine* e, jr_step_args* a) {
  if (!e || !a) return JR_E_INVAL;
  CK(cudaSetDevice(e->cfg.device));
  const Dev& d = e->d;
  const uint32_t R = d.R, G = d.G;
  if (a->n_synth > 8) { set_err("n_synth <= 8"); return JR_E_INVAL; }
  if ((a->out_msgs && !(d.flags & JR_F_CAPTURE_MESSAGES)) || (a->out_fsm && !(d.flags & JR_F_CAPTURE_FSM))) {
    set_err("output buffer given but capture flag not set at create");
    return JR_E_INVAL;
  }
  // ---- validate + bucket injected commands by target, stable
  std::vector<jr_msg> sorted;
  std::vector<uint4> targets;
  if (a->n_inject) {
    if (!a->inject) return JR_E_INVAL;
    std::vector<uint32_t> order(a->n_inject);
    for (size_t i = 0; i < a->n_inject; ++i) {
      const jr_msg& m = a->inject[i];
      if (m.group >= G || m.to_kind != JR_ADDR_PEER) { set_err("inject[%zu]: bad group / to_kind", i); return JR_E_INVAL; }
      if (m.to_id < 1 || m.to_id > R) return JR_E_UNKNOWN_NODE;
      if (m.node_id > JR_MAX_NODE_ID || m.from_id > JR_MAX_NODE_ID || m.client_id > JR_MAX_NODE_ID) return JR_E_INVAL;
      if (m.kind == JR_CMD_VOTE_RESPONSE && (m.node_id < 1 || m.node_id > 32)) return JR_E_UNKNOWN_NODE;
      if (m.n_blocks > JR_MAX_AE_BLOCKS) return JR_E_INVAL;
      if (m.block >= 0xffffffffull) { set_err("inject[%zu]: block id >= 2^32-1 (D4)", i); return JR_E_INVAL; }
      for (unsigned k = 0; k < m.n_blocks; ++k)
        if (m.blocks[k].id >= 0xffffffffull || m.blocks[k].next >= 0xffffffffull) return JR_E_INVAL;
      order[i] = (uint32_t)i;
    }
    std::stable_sort(order.begin(), order.end(), [&](uint32_t x, uint32_t y) {
      const jr_msg &p = a->inject[x], &q = a->inject[y];
      return p.group != q.group ? p.group < q.group : p.to_id < q.to_id;
    });
    sorted.reserve(a->n_inject);
    for (uint32_t idx : order) {
      const jr_msg& m = a->inject[idx];
      if (targets.empty() || targets.back().x != m.group || targets.back().y != m.to_id - 1)
        targets.push_back(make_uint4(m.group, m.to_id - 1, (uint32_t)sorted.size(), 0));
      targets.back().w++;
      sorted.push_back(m);
    }
  }
  if (a->proposals && !(a->flags & JR_STEP_TRUSTED_PROPOSALS))
    for (uint32_t g = 0; g < G; ++g)
      if (a->proposals[g].node > R) return JR_E_UNKNOWN_NODE;

  StepParams p;
  p.now = a->now_ms;
  p.step_index = e->step_index;
  p.n_synth = (a->flags & JR_STEP_SYNTH_PROPOSALS) ? a->n_synth : 0;
  p.cur = e->cur;
  p.n_ticks = 1;
  p.dt = 0;
  p.prop_stride = 0;
  p.proposals = nullptr;
  int staged = -1;
  if (a->proposals) {
    const int b = e->prop_i;
    e->prop_i = (b + 1) % jr_engine::NBUF;
    if (e->prop_used[b]) CK(cudaStreamWaitEvent(e->h2d, e->prop_free[b], 0));  // its last reader is done
    CK(cudaMemcpyAsync(e->prop[b], a->proposals, (size_t)G * sizeof(jr_proposal), cudaMemcpyHostToDevice, e->h2d));
    CK(cudaEventRecord(e->prop_ready[b], e->h2d));
    CK(cudaStreamWaitEvent(e->stream, e->prop_ready[b], 0));
    p.proposals = e->prop[b];
    staged = b;
  }
  const uint32_t ph_first = PH_RESET_OUT | PH_RESET_FSM | ((a->flags & JR_STEP_DELIVER) ? PH_DRAIN : 0u);
  const uint32_t ph_last = ((p.proposals || p.n_synth) ? PH_PROPOSE : 0u) | ((a->flags & JR_STEP_TICK) ? PH_TICK : 0u);
  jr_status st;
  if (targets.empty()) {
    p.phases = ph_first | ph_last;
    if ((st = launch_step(e, p)) != JR_OK) return st;
  } else {
    if (sorted.size() > e->inj_cap) {
      if (e->inj_msgs) cudaFree(e->inj_msgs);
      if (e->inj_targets) cudaFree(e->inj_targets);
      e->inj_msgs = nullptr; e->inj_targets = nullptr;
      e->inj_cap = std::max<size_t>(sorted.size() * 2, 64);
      CK(cudaMalloc(&e->inj_msgs, e->inj_cap * sizeof(jr_msg)));
      CK(cudaMalloc(&e->inj_targets, e->inj_cap * sizeof(uint4)));
    }
    CK(cudaMemcpyAsync(e->inj_msgs, sorted.data(), sorted.size() * sizeof(jr_msg), cudaMemcpyHostToDevice, e->stream));
    CK(cudaMemcpyAsync(e->inj_targets, targets.data(), targets.size() * sizeof(uint4), cudaMemcpyHostToDevice, e->stream));
    p.phases = ph_first;
    if ((st = launch_step(e, p)) != JR_OK) return st;
    const uint32_t nt = (uint32_t)targets.size();
    DISPATCH_R(R, (JR_LAUNCH(inject_kernel<RR>, (nt + 63) / 64, 64, e->stream, e->d, p, e->inj_msgs, e->inj_targets, nt)));
    CK(cudaGetLastError());
    if (ph_last) {
      p.phases = ph_last;
      if ((st = launch_step(e, p)) != JR_OK) return st;
    }
    CK(cudaStreamSynchronize(e->stream));  // `sorted` / `targets` are stack-owned host buffers
  }
  if (staged >= 0) {  // proposals buffer may be refilled once the kernels of this step are done
    CK(cudaEventRecord(e->prop_free[staged], e->stream));
    e->prop_used[staged] = true;
    CK(cudaEventSynchronize(e->prop_ready[staged]));  // a->proposals has been read: the caller may reuse it on return
  }
  const int written = e->cur;
  e->cur ^= 1;
  e->step_index++;

  // ---- capture (synchronises)
  a->n_msgs = 0;
  a->n_fsm = 0;
  bool ovf = false;
  if (a->out_msgs) {
    std::vector<jr_msg> msgs;
    if ((st = capture_messages(e, written, msgs)) != JR_OK) return st;
    a->n_msgs = msgs.size();
    memcpy(a->out_msgs, msgs.data(), std::min(msgs.size(), a->cap_msgs) * sizeof(jr_msg));
    ovf |= msgs.size() > a->cap_msgs;
  }
  if (a->out_fsm) {
    std::vector<jr_fsm_instr> fsm;
    st = capture_fsm(e, fsm);
    if (st != JR_OK && st != JR_E_CAPACITY) return st;
    a->n_fsm = fsm.size();
    memcpy(a->out_fsm, fsm.data(), std::min(fsm.size(), a->cap_fsm) * sizeof(jr_fsm_instr));
    ovf |= fsm.size() > a->cap_fsm || st == JR_E_CAPACITY;
  }
  if (a->flags & JR_STEP_REPORT_FAULTS) {
    uint64_t v[5];
    if ((st = stream_sums(e, v)) != JR_OK) return st;
    a->n_faulted = v[4];
  }
  return ovf ? JR_E_CAPACITY : JR_OK;
}

// One fused run of n_steps whole ticks from where the engine stands (jr_run and the batched calls).  `src` carries the
// proposal source only (n_synth, proposals / prop_stride or tok_runs / tok_route); everything else comes from the engine
// and the arguments.  Instructions accumulate until drained.  b >= 0: the batch slot the run reads, released once the
// run has finished with it.
static jr_status fused_run(jr_engine* e, const StepParams& src, uint64_t now0, uint32_t dt, uint32_t n_steps, int b) {
  StepParams p = src;
  p.now = now0;
  p.dt = dt;
  p.n_ticks = n_steps;
  p.step_index = e->step_index;
  p.cur = e->cur;
  p.phases = PH_RESET_OUT | PH_DRAIN | ((p.n_synth || p.proposals || p.tok_runs) ? PH_PROPOSE : 0u) | PH_TICK;
  p.trunc = e->auto_trunc ? 1u : 0u;
  p.trunc_margin = e->auto_trunc_margin;
  jr_status st = launch_step(e, p);
  if (st != JR_OK) return st;
  if (b >= 0) {
    CK(cudaEventRecord(e->batch_free[b], e->stream));
    e->batch_used[b] = true;
  }
  e->cur ^= (int)(n_steps & 1u);
  e->step_index += n_steps;
  return JR_OK;
}

jr_status jr_run(jr_engine* e, uint64_t now0, uint32_t dt, uint32_t n_steps, uint32_t n_synth) {
  if (!e) return JR_E_INVAL;
  if (n_synth > 8) { set_err("n_synth <= 8"); return JR_E_INVAL; }
  CK(cudaSetDevice(e->cfg.device));
  if (n_steps == 0) return JR_OK;
  StepParams src{};
  src.n_synth = n_synth;
  return fused_run(e, src, now0, dt, n_steps, -1);
}

// Grow batch[b] to n entries once its last reader is done; returns with the h2d stream fenced on that reader.
static jr_status batch_reserve(jr_engine* e, int b, size_t n) {
  if (e->batch_used[b]) CK(cudaStreamWaitEvent(e->h2d, e->batch_free[b], 0));  // its last reader is done
  if (n > e->batch_cap[b]) {
    if (e->batch_used[b]) CK(cudaEventSynchronize(e->batch_free[b]));
    if (e->batch[b]) cudaFree(e->batch[b]);
    e->batch[b] = nullptr;
    e->batch_cap[b] = 0;
    CK(cudaMalloc(&e->batch[b], n * sizeof(jr_proposal)));
    e->batch_cap[b] = n;
  }
  return JR_OK;
}

jr_status jr_run_proposals(jr_engine* e, uint64_t now0, uint32_t dt, uint32_t n_steps, const jr_proposal* proposals,
                           uint32_t flags) {
  if (!e || !proposals) return JR_E_INVAL;
  if (n_steps == 0) return JR_OK;
  CK(cudaSetDevice(e->cfg.device));
  const uint32_t G = e->d.G, R = e->d.R;
  const size_t n = (size_t)n_steps * G;
  if (!(flags & JR_STEP_TRUSTED_PROPOSALS))
    for (size_t i = 0; i < n; ++i)
      if (proposals[i].node > R) return JR_E_UNKNOWN_NODE;
  const int b = e->batch_i;
  e->batch_i = (b + 1) % jr_engine::NBUF;
  jr_status st = batch_reserve(e, b, n);
  if (st != JR_OK) return st;
  CK(cudaMemcpyAsync(e->batch[b], proposals, n * sizeof(jr_proposal), cudaMemcpyHostToDevice, e->h2d));
  CK(cudaEventRecord(e->batch_ready[b], e->h2d));
  CK(cudaStreamWaitEvent(e->stream, e->batch_ready[b], 0));
  StepParams src{};
  src.proposals = e->batch[b];
  src.prop_stride = G;
  return fused_run(e, src, now0, dt, n_steps, b);
}

jr_status jr_run_tokens(jr_engine* e, uint64_t now0, uint32_t dt, uint32_t n_steps, const uint64_t* tokens) {
  if (!e || !tokens) return JR_E_INVAL;
  if (n_steps == 0) return JR_OK;
  CK(cudaSetDevice(e->cfg.device));
  const uint32_t G = e->d.G;
  const size_t n = (size_t)n_steps * G;
  const int b = e->batch_i;
  e->batch_i = (b + 1) % jr_engine::NBUF;
  jr_status st = batch_reserve(e, b, n);  // batch_free[b] also covers tokbuf[b]: the routing kernel precedes the step
  if (st != JR_OK) return st;
  if (n > e->tok_cap[b]) {
    if (e->batch_used[b]) CK(cudaEventSynchronize(e->batch_free[b]));
    if (e->tokbuf[b]) cudaFree(e->tokbuf[b]);
    e->tokbuf[b] = nullptr;
    e->tok_cap[b] = 0;
    CK(cudaMalloc(&e->tokbuf[b], n * sizeof(unsigned long long)));
    e->tok_cap[b] = n;
  }
  CK(cudaMemcpyAsync(e->tokbuf[b], tokens, n * sizeof(unsigned long long), cudaMemcpyHostToDevice, e->h2d));
  CK(cudaEventRecord(e->batch_ready[b], e->h2d));
  CK(cudaStreamWaitEvent(e->stream, e->batch_ready[b], 0));
  // on the engine stream: ordered after the leader_table_kernel that last wrote `route`
  const unsigned blocks = (unsigned)std::min<size_t>((n + 255) / 256, (size_t)148 * 16);
  JR_LAUNCH(route_tokens_kernel, blocks, 256, e->stream, e->tokbuf[b], e->route, e->batch[b], G, n);
  CK(cudaGetLastError());
  StepParams src{};
  src.proposals = e->batch[b];
  src.prop_stride = G;
  return fused_run(e, src, now0, dt, n_steps, b);
}

jr_status jr_run_token_runs(jr_engine* e, uint64_t now0, uint32_t dt, uint32_t n_steps, const jr_token_run* runs) {
  if (!e || !runs) return JR_E_INVAL;
  if (n_steps == 0) return JR_OK;
  CK(cudaSetDevice(e->cfg.device));
  const uint32_t G = e->d.G;
  const int b = e->batch_i;
  e->batch_i = (b + 1) % jr_engine::NBUF;
  jr_status st = batch_reserve(e, b, G);   // batch[b] doubles as the staging buffer: G x 16 bytes
  if (st != JR_OK) return st;
  CK(cudaMemcpyAsync(e->batch[b], runs, (size_t)G * sizeof(jr_token_run), cudaMemcpyHostToDevice, e->h2d));
  CK(cudaEventRecord(e->batch_ready[b], e->h2d));
  CK(cudaStreamWaitEvent(e->stream, e->batch_ready[b], 0));
  StepParams src{};
  src.tok_runs = reinterpret_cast<const uint4*>(e->batch[b]);
  src.tok_route = e->route;    // on the engine stream: ordered after the leader_table_kernel that last wrote it
  return fused_run(e, src, now0, dt, n_steps, b);
}

jr_status jr_drain_fsm(jr_engine* e, jr_fsm_instr* out, size_t cap, size_t* n) {
  if (!e || !n) return JR_E_INVAL;
  CK(cudaSetDevice(e->cfg.device));
  if (!(e->d.flags & JR_F_CAPTURE_FSM)) { *n = 0; return JR_OK; }
  std::vector<jr_fsm_instr> fsm;
  jr_status st = capture_fsm(e, fsm);
  if (st != JR_OK && st != JR_E_CAPACITY) return st;
  *n = fsm.size();
  if (out) memcpy(out, fsm.data(), std::min(fsm.size(), cap) * sizeof(jr_fsm_instr));
  return ((out && fsm.size() > cap) || st == JR_E_CAPACITY) ? JR_E_CAPACITY : JR_OK;
}

jr_status jr_fsm_fold(const jr_fsm_record* recs, size_t n, uint32_t G, uint32_t R, uint32_t* applied_hi, uint64_t* totals) {
  if ((!recs && n) || !applied_hi || !totals || R < 1 || R > JR_MAX_REPLICAS) return JR_E_INVAL;
  uint64_t na = 0, nn = 0;
  for (size_t i = 0; i < n; ++i) {
    const jr_fsm_record& rc = recs[i];
    const uint32_t kind = JR_FSMR_KIND(rc.hdr), node = JR_FSMR_NODE(rc.hdr), count = JR_FSMR_COUNT(rc.hdr);
    if (rc.group >= G || node > R) return JR_E_INVAL;
    if (kind == JR_FSMR_APPLY) {
      if (rc.addr) {   // shared by the nodes of the mask
        if (rc.addr >> R) return JR_E_INVAL;
        for (uint32_t n = 0; n < R; ++n)
          if ((rc.addr >> n) & 1u) {
            uint32_t& hi = applied_hi[(size_t)n * G + rc.group];
            hi = std::max(hi, rc.id0 + count - 1);
            na += count;
          }
      } else {
        uint32_t& hi = applied_hi[(size_t)(node - 1) * G + rc.group];
        hi = std::max(hi, rc.id0 + count - 1);
        na += count;
      }
    } else if (kind == JR_FSMR_NOTIFY) {
      nn += count;
    }
  }
  totals[0] += na;
  totals[1] += nn;
  totals[2] += n;
  return JR_OK;
}

// jr_fsm_fold_mt: a small persistent pool (created on first use and deliberately never destroyed: its workers sleep on
// a condition variable for the life of the process).  A batch is sorted by (node, group); thread t folds the records of
// groups [G*t/T, G*(t+1)/T) of EVERY node section (found by binary search), so no two threads ever touch the same
// watermark -- masked records included, because all nodes of a group belong to the same thread -- and no atomics are
// needed.  A batch that is not sorted that way is folded on the calling thread.
namespace {
struct FoldJob {
  const jr_fsm_record* recs = nullptr;
  size_t n = 0;
  uint32_t G = 0, R = 0, parts = 0;
  uint32_t* applied = nullptr;
  size_t sec[JR_MAX_REPLICAS + 1];   // record index where node k+1's section starts
  uint64_t na[64], nn[64];
  int bad[64];
};
inline uint64_t rec_key(const jr_fsm_record& rc) { return ((uint64_t)JR_FSMR_NODE(rc.hdr) << 32) | rc.group; }
size_t lower_bound_key(const jr_fsm_record* recs, size_t lo, size_t hi, uint64_t key) {
  while (lo < hi) {
    const size_t mid = lo + (hi - lo) / 2;
    if (rec_key(recs[mid]) < key) lo = mid + 1;
    else hi = mid;
  }
  return lo;
}
void fold_slice(FoldJob& j, uint32_t t) {
  const uint32_t g_lo = (uint32_t)((uint64_t)j.G * t / j.parts), g_hi = (uint32_t)((uint64_t)j.G * (t + 1) / j.parts);
  uint64_t na = 0, nn = 0;
  for (uint32_t node = 1; node <= j.R; ++node) {
    const size_t lo = lower_bound_key(j.recs, j.sec[node - 1], j.sec[node], ((uint64_t)node << 32) | g_lo);
    const size_t hi = lower_bound_key(j.recs, lo, j.sec[node], ((uint64_t)node << 32) | g_hi);
    for (size_t i = lo; i < hi; ++i) {
      const jr_fsm_record& rc = j.recs[i];
      const uint32_t kind = JR_FSMR_KIND(rc.hdr), count = JR_FSMR_COUNT(rc.hdr);
      if (kind == JR_FSMR_APPLY) {
        if (rc.addr) {
          if (rc.addr >> j.R) { j.bad[t] = 1; return; }
          for (uint32_t k = 0; k < j.R; ++k)
            if ((rc.addr >> k) & 1u) {
              uint32_t& hi_w = j.applied[(size_t)k * j.G + rc.group];
              hi_w = std::max(hi_w, rc.id0 + count - 1);
              na += count;
            }
        } else {
          uint32_t& hi_w = j.applied[(size_t)(node - 1) * j.G + rc.group];
          hi_w = std::max(hi_w, rc.id0 + count - 1);
          na += count;
        }
      } else if (kind == JR_FSMR_NOTIFY) {
        nn += count;
      }
    }
  }
  j.na[t] = na;
  j.nn[t] = nn;
}
class FoldPool {
  // Workers SPIN for a little while after a job before they go to sleep: a host that folds a batch every few hundred
  // microseconds (bench.py's end-to-end leg) then never pays the futex wake-up of seven threads -- which took as long as
  // the fold itself.  A host that folds rarely finds them asleep on the condition variable, as before.
  static constexpr long long SPIN_NS = 2'000'000;
 public:
  static FoldPool& get() { static FoldPool* p = new FoldPool(); return *p; }   // leaked on purpose (see above)
  void run(FoldJob& j) {
    {
      std::lock_guard<std::mutex> l(m_);
      while (n_workers_ + 1 < j.parts) {   // worker k serves slice k + 1; the caller folds slice 0
        const uint32_t k = n_workers_++;
        std::thread th([this, k] { loop(k); });
        th.detach();
      }
      job_ = &j;
      left_.store(j.parts - 1, std::memory_order_relaxed);
      // one word says which job is current and how many slices it has: a worker decides from a single load
      state_.store(((state_.load(std::memory_order_relaxed) >> 8) + 1) << 8 | j.parts, std::memory_order_release);
    }
    if (sleepers_.load(std::memory_order_acquire)) cv_.notify_all();
    fold_slice(j, 0);
    const auto t0 = std::chrono::steady_clock::now();
    while (left_.load(std::memory_order_acquire) != 0) {
      if (std::chrono::steady_clock::now() - t0 > std::chrono::nanoseconds(SPIN_NS)) {
        std::unique_lock<std::mutex> l(m_);
        done_.wait(l, [this] { return left_.load(std::memory_order_acquire) == 0; });
        break;
      }
      cpu_relax();
    }
  }
 private:
  static void cpu_relax() {
#if defined(__x86_64__) || defined(__i386__)
    __builtin_ia32_pause();
#endif
  }
  void loop(uint32_t k) {
    uint64_t seen = 0;   // generation (state >> 8) this worker has dealt with
    for (;;) {
      uint64_t st = state_.load(std::memory_order_acquire);
      const auto t0 = std::chrono::steady_clock::now();
      while ((st >> 8) == seen) {
        if (std::chrono::steady_clock::now() - t0 > std::chrono::nanoseconds(SPIN_NS)) {
          std::unique_lock<std::mutex> l(m_);
          sleepers_.fetch_add(1, std::memory_order_acq_rel);
          cv_.wait(l, [&] { return (state_.load(std::memory_order_acquire) >> 8) != seen; });
          sleepers_.fetch_sub(1, std::memory_order_acq_rel);
        } else {
          cpu_relax();
        }
        st = state_.load(std::memory_order_acquire);
      }
      seen = st >> 8;
      if (k + 1 >= (uint32_t)(st & 255u)) continue;   // not one of this job's slices (and then job_ is not this worker's to touch)
      fold_slice(*job_, k + 1);                         // (run() cannot return, nor the next job start, before left_ reaches 0)
      if (left_.fetch_sub(1, std::memory_order_acq_rel) == 1) {
        std::lock_guard<std::mutex> l(m_);
        done_.notify_all();
      }
    }
  }
  std::mutex m_;
  std::condition_variable cv_, done_;
  uint32_t n_workers_ = 0;
  FoldJob* job_ = nullptr;
  std::atomic<uint32_t> left_{0}, sleepers_{0};
  std::atomic<uint64_t> state_{0};   // generation << 8 | slices of the current job
};
}  // namespace

jr_status jr_fsm_fold_mt(const jr_fsm_record* recs, size_t n, uint32_t G, uint32_t R, uint32_t* applied_hi, uint64_t* totals,
                         uint32_t n_threads) {
  if (n_threads <= 1 || n < 4096) return jr_fsm_fold(recs, n, G, R, applied_hi, totals);
  if ((!recs && n) || !applied_hi || !totals || R < 1 || R > JR_MAX_REPLICAS) return JR_E_INVAL;
  FoldJob j;
  j.recs = recs; j.n = n; j.G = G; j.R = R; j.applied = applied_hi;
  j.parts = std::min<uint32_t>(n_threads, 64);
  // node sections; then a cheap sortedness probe (a full check would cost as much as the fold)
  j.sec[0] = 0;
  for (uint32_t node = 1; node <= R; ++node) j.sec[node] = lower_bound_key(recs, j.sec[node - 1], n, (uint64_t)(node + 1) << 32);
  bool sorted = j.sec[R] == n && recs[n - 1].group < G;
  for (size_t probe = 1; sorted && probe < 64; ++probe) {
    const size_t i = n * probe / 64;
    sorted = i == 0 || rec_key(recs[i - 1]) <= rec_key(recs[i]);
  }
  if (!sorted) return jr_fsm_fold(recs, n, G, R, applied_hi, totals);
  static std::mutex* one_at_a_time = new std::mutex();
  std::lock_guard<std::mutex> guard(*one_at_a_time);
  for (uint32_t t = 0; t < j.parts; ++t) { j.na[t] = j.nn[t] = 0; j.bad[t] = 0; }
  FoldPool::get().run(j);
  for (uint32_t t = 0; t < j.parts; ++t) {
    if (j.bad[t]) return JR_E_INVAL;
    totals[0] += j.na[t];
    totals[1] += j.nn[t];
  }
  totals[2] += n;
  return JR_OK;
}

jr_status jr_fsm_records_async(jr_engine* e) {
  if (!e) return JR_E_INVAL;
  CK(cudaSetDevice(e->cfg.device));
  return fsm_records_enqueue(e);
}

jr_status jr_fsm_records_wait(jr_engine* e, const jr_fsm_record** records, jr_fsm_batch* batch) {
  if (!e) return JR_E_INVAL;
  CK(cudaSetDevice(e->cfg.device));   // (may be a consumer thread of its own: the device is per thread)
  return fsm_records_take(e, records, batch);
}

// Pure host code: records -> Instructions (include/josefine_raft_abi.h, jr_fsm_record).
jr_status jr_fsm_expand(const jr_fsm_record* recs, size_t n_records, uint32_t G, uint32_t R, jr_fsm_instr* out, size_t cap,
                        size_t* n_out) {
  if (!n_out || (!recs && n_records) || R < 1 || R > JR_MAX_REPLICAS || G < 1) return JR_E_INVAL;
  // stable counting sort of record indices by (group, node).  An APPLY record with a node mask (addr != 0: symmetric
  // followers share it) goes into the bucket of every node of the mask, in front of that node's own records: masked
  // records are only ever produced while the nodes' own streams are still empty.
  const size_t nb = (size_t)G * R;
  std::vector<uint32_t> start(nb + 1, 0u);
  auto masked = [&](const jr_fsm_record& rc) { return JR_FSMR_KIND(rc.hdr) == JR_FSMR_APPLY && rc.addr != 0; };
  for (size_t i = 0; i < n_records; ++i) {
    const uint32_t node = JR_FSMR_NODE(recs[i].hdr);
    if (recs[i].group >= G || node > R || JR_FSMR_KIND(recs[i].hdr) > JR_FSMR_PATTERN) return JR_E_INVAL;
    if (masked(recs[i])) {
      if (recs[i].addr >> R) return JR_E_INVAL;
      for (uint32_t n = 0; n < R; ++n)
        if ((recs[i].addr >> n) & 1u) ++start[(size_t)recs[i].group * R + n + 1];
    } else {
      ++start[(size_t)recs[i].group * R + (node - 1) + 1];
    }
  }
  for (size_t b = 0; b < nb; ++b) start[b + 1] += start[b];
  std::vector<uint32_t> order(start[nb]), fill(start.begin(), start.end() - 1);
  for (int pass = 0; pass < 2; ++pass)
    for (size_t i = 0; i < n_records; ++i) {
      if (masked(recs[i]) != (pass == 0)) continue;
      if (pass == 0) {
        for (uint32_t n = 0; n < R; ++n)
          if ((recs[i].addr >> n) & 1u) order[fill[(size_t)recs[i].group * R + n]++] = (uint32_t)i;
      } else {
        order[fill[(size_t)recs[i].group * R + (JR_FSMR_NODE(recs[i].hdr) - 1)]++] = (uint32_t)i;
      }
    }
  size_t k = 0;
  std::vector<uint64_t> is_notify;
  for (size_t b = 0; b < nb; ++b) {
    const uint32_t lo = start[b], hi = start[b + 1];
    if (lo == hi) continue;
    const uint32_t g = (uint32_t)(b / R), node = (uint32_t)(b % R) + 1;
    size_t n_apply = 0, n_note = 0;
    for (uint32_t j = lo; j < hi; ++j) {
      const jr_fsm_record& rc = recs[order[j]];
      if (JR_FSMR_KIND(rc.hdr) == JR_FSMR_APPLY) n_apply += JR_FSMR_COUNT(rc.hdr);
      else if (JR_FSMR_KIND(rc.hdr) == JR_FSMR_NOTIFY) n_note += JR_FSMR_COUNT(rc.hdr);
    }
    const size_t total = n_apply + n_note;
    is_notify.assign((total + 63) / 64, 0ull);
    size_t marked = 0;
    for (uint32_t j = lo; j < hi; ++j) {
      const jr_fsm_record& rc = recs[order[j]];
      if (JR_FSMR_KIND(rc.hdr) != JR_FSMR_PATTERN) continue;
      const uint32_t nbits = JR_FSMR_COUNT(rc.hdr);
      if (nbits > 160) return JR_E_INVAL;
      for (uint32_t bit = 0; bit < nbits; ++bit)
        if ((bit < 64 ? rc.tok0 >> bit : bit < 128 ? rc.stride >> (bit - 64) : (uint64_t)rc.addr >> (bit - 128)) & 1ull) {
          const size_t pos = (size_t)rc.id0 + bit;
          if (pos >= total || ((is_notify[pos >> 6] >> (pos & 63)) & 1ull)) return JR_E_INVAL;
          is_notify[pos >> 6] |= 1ull << (pos & 63);
          ++marked;
        }
    }
    if (marked != n_note) return JR_E_INVAL;
    // two cursors, one per kind, both in record order
    uint32_t ja = lo, jn = lo, ia = 0, in_ = 0;
    for (size_t pos = 0; pos < total; ++pos) {
      const bool note = (is_notify[pos >> 6] >> (pos & 63)) & 1ull;
      uint32_t& j = note ? jn : ja;
      uint32_t& i = note ? in_ : ia;
      const uint32_t want = note ? JR_FSMR_NOTIFY : JR_FSMR_APPLY;
      while (JR_FSMR_KIND(recs[order[j]].hdr) != want || i >= JR_FSMR_COUNT(recs[order[j]].hdr)) { ++j; i = 0; }
      const jr_fsm_record& rc = recs[order[j]];
      if (out && k < cap) {
        jr_fsm_instr f;
        memset(&f, 0, sizeof f);
        f.group = g;
        f.node = node;
        if (note) {
          f.kind = JR_FSM_NOTIFY;
          f.client_kind = (uint8_t)(rc.addr >> 16);
          f.client_id = rc.addr & 0xffffu;
          f.block = jr_block{(uint64_t)(rc.id0 + i), 0, rc.tok0 + (uint64_t)i * rc.stride};
        } else {
          f.kind = JR_FSM_APPLY;
          const uint32_t bid = rc.id0 + i;
          if (JR_FSMR_COUNT(rc.hdr) == 1) f.block = jr_block{bid, (uint32_t)rc.stride, rc.tok0};
          else f.block = jr_block{bid, bid - 1u, rc.tok0 + (uint64_t)i * rc.stride};
        }
        out[k] = f;
      }
      ++k;
      ++i;
    }
  }
  *n_out = k;
  return (out && k > cap) || (!out && k) ? JR_E_CAPACITY : JR_OK;
}

// ---- introspection ----------------------------------------------------------------------------

static jr_status many_reserve(jr_engine* e, size_t bytes) {
  if (bytes <= e->many_cap) return JR_OK;
  if (e->many_buf) cudaFree(e->many_buf);
  e->many_buf = nullptr;
  e->many_cap = 0;
  const size_t want = std::max<size_t>(bytes * 2, 4096);
  CK(cudaMalloc(&e->many_buf, want));
  e->many_cap = want;
  return JR_OK;
}

jr_status jr_query_many(jr_engine* e, const uint32_t* groups, const uint32_t* nodes, size_t n, jr_replica_state* out) {
  if (!e || !out || !groups || !nodes) return JR_E_INVAL;
  if (n == 0) return JR_OK;
  if (n > 0x7fffffffu) return JR_E_INVAL;
  for (size_t i = 0; i < n; ++i)
    if (groups[i] >= e->d.G || nodes[i] < 1 || nodes[i] > e->d.R) return JR_E_INVAL;
  CK(cudaSetDevice(e->cfg.device));
  const size_t idx = ((n * 2 * sizeof(uint32_t)) + 15) / 16 * 16;   // [groups][nodes] then the states
  jr_status st = many_reserve(e, idx + n * sizeof(jr_replica_state));
  if (st != JR_OK) return st;
  uint32_t* dg = (uint32_t*)e->many_buf;
  uint32_t* dn = dg + n;
  jr_replica_state* ds = (jr_replica_state*)((char*)e->many_buf + idx);
  CK(cudaMemcpyAsync(dg, groups, n * sizeof(uint32_t), cudaMemcpyHostToDevice, e->stream));
  CK(cudaMemcpyAsync(dn, nodes, n * sizeof(uint32_t), cudaMemcpyHostToDevice, e->stream));
  JR_LAUNCH(query_kernel, (unsigned)((n + 127) / 128), 128, e->stream, e->d, dg, dn, (uint32_t)n, ds);
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(out, ds, n * sizeof(jr_replica_state), cudaMemcpyDeviceToHost, e->stream));
  CK(cudaStreamSynchronize(e->stream));
  return JR_OK;
}

jr_status jr_query(jr_engine* e, uint32_t group, uint32_t node, jr_replica_state* out) {
  return jr_query_many(e, &group, &node, 1, out);
}

jr_status jr_chain_read_many(jr_engine* e, const uint32_t* groups, const uint32_t* nodes, const uint64_t* first_id,
                             const uint32_t* count, size_t n, jr_block* out, uint8_t* present) {
  if (!e || !groups || !nodes || !first_id || !count) return JR_E_INVAL;
  if (n == 0) return JR_OK;
  if (n > 0x7fffffffu) return JR_E_INVAL;
  std::vector<uint4> reqs(n);
  size_t total = 0;
  for (size_t i = 0; i < n; ++i) {
    if (groups[i] >= e->d.G || nodes[i] < 1 || nodes[i] > e->d.R) return JR_E_INVAL;
    if (first_id[i] + count[i] > 0xffffffffull) return JR_E_INVAL;
    reqs[i] = make_uint4(groups[i], nodes[i] - 1, (uint32_t)first_id[i], (uint32_t)total);
    total += count[i];
    if (total > 0xffffffffull) return JR_E_INVAL;
  }
  if (total == 0) return JR_OK;
  CK(cudaSetDevice(e->cfg.device));
  const size_t o_cnt = n * sizeof(uint4), o_blk = (o_cnt + n * sizeof(uint32_t) + 15) / 16 * 16;
  const size_t o_pre = o_blk + total * sizeof(jr_block);
  jr_status st = many_reserve(e, o_pre + total);
  if (st != JR_OK) return st;
  char* base = (char*)e->many_buf;
  CK(cudaMemcpyAsync(base, reqs.data(), n * sizeof(uint4), cudaMemcpyHostToDevice, e->stream));
  CK(cudaMemcpyAsync(base + o_cnt, count, n * sizeof(uint32_t), cudaMemcpyHostToDevice, e->stream));
  JR_LAUNCH(chain_read_kernel, (unsigned)n, 128, e->stream, e->d, (const uint4*)base, (const uint32_t*)(base + o_cnt),
            (jr_block*)(base + o_blk), (uint8_t*)(base + o_pre));
  CK(cudaGetLastError());
  if (out) CK(cudaMemcpyAsync(out, base + o_blk, total * sizeof(jr_block), cudaMemcpyDeviceToHost, e->stream));
  if (present) CK(cudaMemcpyAsync(present, base + o_pre, total, cudaMemcpyDeviceToHost, e->stream));
  CK(cudaStreamSynchronize(e->stream));   // also covers `reqs`, which lives on this stack
  return JR_OK;
}

jr_status jr_chain_read(jr_engine* e, uint32_t group, uint32_t node, uint64_t first, uint32_t n, jr_block* out,
                        uint8_t* present) {
  if (n == 0) return (!e || group >= e->d.G || node < 1 || node > e->d.R) ? JR_E_INVAL : JR_OK;
  return jr_chain_read_many(e, &group, &node, &first, &n, 1, out, present);
}

jr_status jr_state_digest(jr_engine* e, uint64_t* out) {
  if (!e || !out) return JR_E_INVAL;
  CK(cudaSetDevice(e->cfg.device));
  const size_t plane = (size_t)e->d.R * e->d.Gp;
  CK(cudaMemsetAsync(e->scratch, 0, 8 * sizeof(unsigned long long), e->stream));
  JR_LAUNCH(state_digest_kernel, (unsigned)((plane + 255) / 256), 256, e->stream, e->d, e->scratch);
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(out, e->scratch, sizeof(uint64_t), cudaMemcpyDeviceToHost, e->stream));
  CK(cudaStreamSynchronize(e->stream));
  return JR_OK;
}

static jr_status stream_sums(jr_engine* e, uint64_t v[5]) {
  CK(cudaSetDevice(e->cfg.device));
  const size_t plane = (size_t)e->d.R * e->d.Gp;
  CK(cudaMemsetAsync(e->scratch, 0, 8 * sizeof(unsigned long long), e->stream));
  JR_LAUNCH(stream_digest_kernel, (unsigned)((plane + 255) / 256), 256, e->stream, e->d, e->scratch);
  CK(cudaGetLastError());
  CK(cudaMemcpyAsync(v, e->scratch, 5 * sizeof(uint64_t), cudaMemcpyDeviceToHost, e->stream));
  CK(cudaStreamSynchronize(e->stream));
  return JR_OK;
}

jr_status jr_stream_digest(jr_engine* e, uint64_t* md, uint64_t* fd, uint64_t* nm, uint64_t* nf) {
  if (!e) return JR_E_INVAL;
  if (!(e->d.flags & JR_F_STREAM_DIGEST)) { set_err("engine created without JR_F_STREAM_DIGEST"); return JR_E_INVAL; }
  uint64_t v[5];
  jr_status st = stream_sums(e, v);
  if (st != JR_OK) return st;
  if (md) *md = v[0];
  if (fd) *fd = v[1];
  if (nm) *nm = v[2];
  if (nf) *nf = v[3];
  return JR_OK;
}

jr_status jr_fold_count(jr_engine* e, uint64_t* n) {
  if (!e || !n) return JR_E_INVAL;
  *n = 0;
  if (!e->last_launch_folded) return JR_OK;
  CK(cudaSetDevice(e->cfg.device));
  std::vector<uint8_t> h(e->d.Gp);
  CK(cudaMemcpyAsync(h.data(), e->symdone, h.size(), cudaMemcpyDeviceToHost, e->stream));
  CK(cudaStreamSynchronize(e->stream));
  for (uint32_t g = 0; g < e->d.G; ++g) *n += h[g];
  return JR_OK;
}

jr_status jr_fault_count(jr_engine* e, uint64_t* n) {
  if (!e || !n) return JR_E_INVAL;
  uint64_t v[5];
  jr_status st = stream_sums(e, v);
  if (st != JR_OK) return st;
  *n = v[4];
  return JR_OK;
}

// ---- maintenance ------------------------------------------------------------------------------

jr_status jr_compact(jr_engine* e) {
  if (!e) return JR_E_INVAL;
  CK(cudaSetDevice(e->cfg.device));
  const size_t plane = (size_t)e->d.R * e->d.Gp;
  JR_LAUNCH(compact_kernel, (unsigned)((plane + 127) / 128), 128, e->stream, e->d);
  CK(cudaGetLastError());
  return JR_OK;
}

jr_status jr_truncate(jr_engine* e, uint32_t margin) {
  if (!e) return JR_E_INVAL;
  CK(cudaSetDevice(e->cfg.device));
  JR_LAUNCH(truncate_kernel, (e->d.Gp + 127) / 128, 128, e->stream, e->d, margin, (const uint8_t*)nullptr);
  CK(cudaGetLastError());
  return JR_OK;
}

jr_status jr_host_alloc(size_t bytes, void** out) {
  if (!out || !bytes) return JR_E_INVAL;
  *out = nullptr;
  cudaError_t err = cudaHostAlloc(out, bytes, 0);
  if (err != cudaSuccess) {
    set_err("cudaHostAlloc(%zu bytes): %s", bytes, cudaGetErrorString(err));
    return err == cudaErrorMemoryAllocation ? JR_E_NOMEM : JR_E_CUDA;
  }
  return JR_OK;
}

void jr_host_free(void* p) {
  if (p) cudaFreeHost(p);
}

jr_status jr_set_auto_truncate(jr_engine* e, int enabled, uint32_t margin) {
  if (!e) return JR_E_INVAL;
  e->auto_trunc = enabled != 0;
  e->auto_trunc_margin = margin;
  return JR_OK;
}

jr_status jr_node_restart(jr_engine* e, uint32_t group, uint32_t node, uint64_t now_ms, const jr_block* blocks,
                          size_t n_blocks, uint64_t commit, int commit_key) {
  if (!e || group >= e->d.G || node < 1 || node > e->d.R || (n_blocks && !blocks)) return JR_E_INVAL;
  if (n_blocks > e->d.cap || commit >= 0xffffffffull) return JR_E_INVAL;
  CK(cudaSetDevice(e->cfg.device));
  jr_replica_state st0;
  jr_status st = jr_query(e, group, node, &st0);   // (synchronises; also tells the group's floor)
  if (st != JR_OK) return st;
  for (size_t k = 0; k < n_blocks; ++k)
    if (blocks[k].id < st0.chain_floor || blocks[k].id - st0.chain_floor >= e->d.cap || blocks[k].next >= 0xffffffffull) {
      set_err("blocks[%zu]: id outside [floor, floor + chain_capacity) or next >= 2^32-1 (D4, D7)", k);
      return JR_E_INVAL;
    }
  if ((st = many_reserve(e, std::max<size_t>(n_blocks, 1) * sizeof(jr_block))) != JR_OK) return st;
  if (n_blocks) CK(cudaMemcpyAsync(e->many_buf, blocks, n_blocks * sizeof(jr_block), cudaMemcpyHostToDevice, e->stream));
  JR_LAUNCH(node_restart_kernel, 1, 1, e->stream, e->d, group, node - 1, now_ms, (const jr_block*)e->many_buf,
            (uint32_t)n_blocks, (uint32_t)commit, commit_key ? 1u : 0u);
  CK(cudaGetLastError());
  CK(cudaStreamSynchronize(e->stream));
  return JR_OK;
}

// ---- checkpoint -----------------------------------------------------------------------------------
namespace {
struct SaveHeader {
  uint64_t magic, bytes;
  jr_config cfg;
  uint32_t cur, route_valid;
  uint64_t step_index;
};
constexpr uint64_t SAVE_MAGIC = 0x4a52454e47494e32ull;  // "JRENGIN2"
struct Segment { void* p; size_t n; };
std::vector<Segment> save_segments(jr_engine* e) {
  const Dev& d = e->d;
  const size_t plane = (size_t)d.R * d.Gp;
  const size_t rows = (size_t)d.capm + 1;
  std::vector<Segment> v = {
      {d.p0, plane * sizeof(uint4)}, {d.p1, plane * sizeof(uint4)}, {d.p2, plane * sizeof(uint4)}, {d.p3, plane * sizeof(uint4)},
      {d.pr, plane * ((d.R + 3) / 4) * sizeof(uint4)}, {d.mk, plane * sizeof(uint32_t)},
      {d.qt, plane * JR_CLIENT_QUEUE_CAP * sizeof(uint4)}, {d.dg, plane * sizeof(uint4)}, {d.cn, plane * sizeof(uint2)},
      {d.cnext, plane * rows * sizeof(uint32_t)}, {d.ctok, plane * rows * sizeof(unsigned long long)},
      {d.ob[0], plane * (size_t)d.U * sizeof(uint4)}, {d.ob[1], plane * (size_t)d.U * sizeof(uint4)},
      {d.oc[0], plane * sizeof(uint32_t)}, {d.oc[1], plane * sizeof(uint32_t)},
      {d.fs, plane * ((d.flags & JR_F_CAPTURE_FSM) ? 2 * (size_t)d.F : 1) * sizeof(uint4)}, {d.fc, plane * sizeof(uint2)},
      {d.tb, (size_t)d.Gp * sizeof(uint32_t)}, {e->route, (size_t)d.G * sizeof(uint32_t)}};
  return v;
}
}  // namespace

jr_status jr_engine_save_size(jr_engine* e, size_t* bytes) {
  if (!e || !bytes) return JR_E_INVAL;
  size_t n = sizeof(SaveHeader);
  for (const Segment& sg : save_segments(e)) n += sg.n;
  *bytes = n;
  return JR_OK;
}

jr_status jr_engine_save(jr_engine* e, void* buf, size_t cap) {
  if (!e || !buf) return JR_E_INVAL;
  size_t need = 0;
  jr_engine_save_size(e, &need);
  if (cap < need) return JR_E_CAPACITY;
  CK(cudaSetDevice(e->cfg.device));
  jr_status st = jr_engine_sync(e);
  if (st != JR_OK) return st;
  SaveHeader h;
  memset(&h, 0, sizeof h);
  h.magic = SAVE_MAGIC;
  h.bytes = need;
  h.cfg = e->cfg;
  h.cur = (uint32_t)e->cur;
  h.step_index = e->step_index;
  memcpy(buf, &h, sizeof h);
  char* at = (char*)buf + sizeof h;
  for (const Segment& sg : save_segments(e)) {
    CK(cudaMemcpyAsync(at, sg.p, sg.n, cudaMemcpyDeviceToHost, e->stream));
    at += sg.n;
  }
  CK(cudaStreamSynchronize(e->stream));
  return JR_OK;
}

jr_status jr_engine_restore(jr_engine* e, const void* buf, size_t bytes) {
  if (!e || !buf || bytes < sizeof(SaveHeader)) return JR_E_INVAL;
  SaveHeader h;
  memcpy(&h, buf, sizeof h);
  size_t need = 0;
  jr_engine_save_size(e, &need);
  jr_config a = h.cfg, b = e->cfg;
  a.device = b.device = 0;   // a checkpoint may move to another GPU
  if (h.magic != SAVE_MAGIC || h.bytes != need || bytes < need || memcmp(&a, &b, sizeof a) != 0) {
    set_err("checkpoint does not match this engine's configuration");
    return JR_E_INVAL;
  }
  CK(cudaSetDevice(e->cfg.device));
  jr_status st = jr_engine_sync(e);
  if (st != JR_OK) return st;
  const char* at = (const char*)buf + sizeof h;
  for (const Segment& sg : save_segments(e)) {
    CK(cudaMemcpyAsync(sg.p, at, sg.n, cudaMemcpyHostToDevice, e->stream));
    at += sg.n;
  }
  CK(cudaStreamSynchronize(e->stream));
  e->cur = (int)h.cur;
  e->step_index = h.step_index;
  e->fsm_npending = 0;
  return JR_OK;
}

jr_status jr_set_alive(jr_engine* e, uint32_t group, uint32_t node, int alive) {
  if (!e || group >= e->d.G || node < 1 || node > e->d.R) return JR_E_INVAL;
  CK(cudaSetDevice(e->cfg.device));
  JR_LAUNCH(set_alive_kernel, 1, 1, e->stream, e->d, group, node - 1, alive);
  CK(cudaGetLastError());
  return JR_OK;
}

jr_status jr_kill_leaders(jr_engine* e, uint64_t salt, uint32_t permille, uint64_t* n_killed) {
  if (!e) return JR_E_INVAL;
  CK(cudaSetDevice(e->cfg.device));
  CK(cudaMemsetAsync(e->scratch, 0, sizeof(unsigned long long), e->stream));
  JR_LAUNCH(kill_leaders_kernel, (e->d.G + 127) / 128, 128, e->stream, e->d, mix64(e->d.seed ^ salt), permille, e->scratch);
  CK(cudaGetLastError());
  uint64_t k = 0;
  CK(cudaMemcpyAsync(&k, e->scratch, sizeof k, cudaMemcpyDeviceToHost, e->stream));
  CK(cudaStreamSynchronize(e->stream));
  if (n_killed) *n_killed = k;
  return JR_OK;
}

jr_status jr_leader_table_device(jr_engine* e, void* dev_out) {
  if (!e || !dev_out) return JR_E_INVAL;
  CK(cudaSetDevice(e->cfg.device));
  JR_LAUNCH(leader_table_kernel, (e->d.G + 127) / 128, 128, e->stream, e->d, (jr_leader_entry*)dev_out, e->route);
  CK(cudaGetLastError());
  return JR_OK;
}

jr_status jr_leader_table_async(jr_engine* e, jr_leader_entry* host_out) {
  if (!e || !host_out) return JR_E_INVAL;
  const int b = e->tab_i;
  e->tab_i = (b + 1) % jr_engine::NBUF;
  if (e->tab_used[b]) CK(cudaStreamWaitEvent(e->stream, e->tab_free[b], 0));  // its last copy-out is done
  jr_status st = jr_leader_table_device(e, e->leaders[b]);
  if (st != JR_OK) return st;
  CK(cudaEventRecord(e->tab_ready[b], e->stream));
  CK(cudaStreamWaitEvent(e->d2h, e->tab_ready[b], 0));
  CK(cudaMemcpyAsync(host_out, e->leaders[b], (size_t)e->d.G * sizeof(jr_leader_entry), cudaMemcpyDeviceToHost, e->d2h));
  CK(cudaEventRecord(e->tab_free[b], e->d2h));
  e->tab_used[b] = true;
  std::lock_guard<std::mutex> l(e->qmu);
  if (e->tab_npending == jr_engine::NBUF) {  // the oldest one is about to be overwritten anyway
    for (int k = 0; k + 1 < jr_engine::NBUF; ++k) e->tab_pending[k] = e->tab_pending[k + 1];
    --e->tab_npending;
  }
  e->tab_pending[e->tab_npending++] = b;
  return JR_OK;
}

jr_status jr_leader_table_wait(jr_engine* e) {
  if (!e) return JR_E_INVAL;
  CK(cudaSetDevice(e->cfg.device));
  int b;
  {
    std::lock_guard<std::mutex> l(e->qmu);
    if (e->tab_npending == 0) return JR_OK;
    b = e->tab_pending[0];
    for (int k = 0; k + 1 < jr_engine::NBUF; ++k) e->tab_pending[k] = e->tab_pending[k + 1];
    --e->tab_npending;
  }
  CK(cudaEventSynchronize(e->tab_free[b]));
  return JR_OK;
}

jr_status jr_leader_table(jr_engine* e, jr_leader_entry* host_out) {
  jr_status st = jr_leader_table_async(e, host_out);
  if (st != JR_OK) return st;
  CK(cudaStreamSynchronize(e->d2h));
  e->tab_npending = 0;
  return JR_OK;
}

}  // extern "C"
