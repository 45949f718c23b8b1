/*
 * josefine_raft_abi.h -- C ABI of the B200 batched Chained-Raft engine.
 *
 * This is the drop-in boundary for josefine's Raft step path.  Every entry
 * point names the reference interface it stands in for (paths are relative to
 * the reference checkout, tychedelia/josefine @ 28b42c9):
 *
 *   jr_engine_create   <- RaftHandle::new                 src/raft/mod.rs:428-435
 *                         (Raft::<Follower>::new          src/raft/follower.rs:68-91,
 *                          Chain::new                     src/raft/chain.rs:117-137)
 *   jr_step            <- Apply::apply(self, Command)     src/raft/mod.rs:483-489,471-479
 *                         as called by event_loop         src/raft/server.rs:125,133,135,143,159
 *   jr_step outputs    <- rpc_tx.send(Message)            src/raft/mod.rs:390-400
 *                         fsm_tx.send(Instruction)        src/raft/leader.rs:94,184; follower.rs:205
 *   jr_run             <- N consecutive event_loop turns with no host traffic (Tick + peer mail)
 *   jr_run_proposals   <- N consecutive event_loop turns incl. the client arm (server.rs:156-160)
 *   jr_run_tokens      <- the same, with proposals addressed to the last announced leader
 *   jr_run_token_runs  <- the same, one arithmetic token run per group instead of one token per group-tick
 *   jr_query           <- pub fields id/state/role/chain  src/raft/mod.rs:326-341,437-447;
 *                         Chain::get_head/get_commit      src/raft/chain.rs:230-236
 *   jr_chain_read      <- Chain::range / Chain::has       src/raft/chain.rs:155-157,208-228
 *   jr_compact         <- Chain::compact                  src/raft/chain.rs:239-253
 *   jr_leader_table*   <- Leader::write_state             src/raft/leader.rs:101-121
 *   jr_set_alive       <- process death (no reference API; a node that stops calling apply)
 *   jr_fsm_records_*   <- the receiving end of fsm_tx         src/raft/fsm.rs:52-56 (Driver::run's rx.recv loop),
 *                         fed by leader.rs:87-99,177-197 and follower.rs:198-207; compact form, see jr_fsm_record
 *   jr_fsm_expand      <- Instruction::{Apply,Notify}         src/raft/fsm.rs:19-29, one per record element
 *   jr_node_restart    <- RaftHandle::new over an existing data directory: Chain::new reopening a
 *                         persisted chain                     src/raft/chain.rs:117-137
 *   jr_query_many / jr_chain_read_many <- the same pub fields, for many replicas in one call
 *   jr_engine_save / jr_engine_restore <- checkpoint of the whole engine (no reference API: sled persistence of
 *                         every node at once, chain.rs:119-123,198, plus the volatile State the reference loses)
 *   jr_truncate        <- no reference API (deviation D7)
 *
 * One engine = G independent Raft groups x R replicas, all resident in one GPU's
 * HBM.  The reference is one group, one node per process; the group dimension is
 * new.  Role is a field here, not a type (reference: RaftHandle enum,
 * mod.rs:417-424).
 *
 * Declared deviations from the reference (see DESIGN.md, "Deviations"):
 *   D1  time: `now` is an explicit u64 input in milliseconds instead of
 *       Instant::now() (mod.rs:354; follower.rs:112,141; leader.rs:79,83).
 *   D2  randomness: election timeouts come from a counter-based generator keyed
 *       (seed, group, node, draw#) (jr_election_timeout below) instead of
 *       rand::thread_rng (follower.rs:103-108).
 *   D3  panics / Err returns of the reference become a sticky per-replica
 *       fault code (JR_FAULT_*); a faulted replica stops like a dead process.
 *   D4  node ids are 1..65534 (reference: any non-zero u32, config.rs:64);
 *       block ids must be < chain_capacity (reference: any u64).
 *   D5  Block.data (Vec<u8>) is represented on the device by a 64-bit token the
 *       host maps to the payload bytes; ClientRequest.id (Uuid) likewise.
 *   D6  the sled "commit" key shares the block keyspace in the reference
 *       (chain.rs:198), so an unbounded Chain::range that runs past the last
 *       block hits it and panics in bincode (chain.rs:222-226).  That is
 *       reproduced only when JR_F_SLED_COMMIT_KEY_STRICT is set; by default the
 *       block map holds blocks only (SURVEY.md section 8 row a15).
 *   D7  log truncation (opt-in, only through jr_truncate): the reference never removes a block
 *       except in Chain::compact (chain.rs:239-253, never called outside its test), so its sled
 *       tree grows forever.  jr_truncate drops, per group, every block below
 *       floor = min(commit of the live replicas) - margin from ALL replicas of the group; block ids
 *       must then lie in [floor, floor + chain_capacity).  Removed keys read as absent, exactly as
 *       if sled had lost them (has() false, range() skips them).  An engine that never calls
 *       jr_truncate behaves as before (floor 0).
 *
 * All structs are plain data, little endian, naturally aligned.  No callbacks.
 * Buffers passed to jr_step are HOST memory owned by the caller.
 */
#ifndef JOSEFINE_RAFT_ABI_H
#define JOSEFINE_RAFT_ABI_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define JR_ABI_VERSION 2u

/* ---- limits ------------------------------------------------------------ */
#define JR_MAX_REPLICAS 8u        /* R <= 8 (reference configs use 3, 5, 7)         */
#define JR_STAGING_DEPTH 3u       /* steps a host may keep in flight on the async paths */
#define JR_MAX_AE_BLOCKS 5u       /* MAX_INFLIGHT, src/raft/progress.rs:117          */
#define JR_MAX_NODE_ID 65534u     /* deviation D4                                    */
#define JR_CLIENT_QUEUE_CAP 4u    /* queued_reqs bound per replica (reference: Vec)  */

/* ---- status codes (API misuse / resources; never consensus outcomes) ---- */
typedef enum jr_status {
  JR_OK = 0,
  JR_E_INVAL = 1,        /* bad argument / config (RaftConfig::validate, config.rs:60-84) */
  JR_E_NOMEM = 2,
  JR_E_CUDA = 3,         /* CUDA runtime error; jr_last_error() has the text            */
  JR_E_CAPACITY = 4,     /* caller output buffer too small; n_* hold the needed counts  */
  JR_E_UNKNOWN_NODE = 5, /* message addressed to / naming a node outside the group     */
  JR_E_NO_DEVICE = 6     /* no CUDA device: there is NO CPU fallback in this library   */
} jr_status;

/* ---- roles (RaftRole, src/raft/mod.rs:403-407) --------------------------- */
enum { JR_ROLE_FOLLOWER = 0, JR_ROLE_CANDIDATE = 1, JR_ROLE_LEADER = 2 };

/* ---- Command discriminants, in the order of `enum Command` (mod.rs:160-227) */
enum {
  JR_CMD_TICK = 0,
  JR_CMD_PROPOSE = 1,            /* unused by the reference state machine */
  JR_CMD_VOTE_REQUEST = 2,
  JR_CMD_VOTE_RESPONSE = 3,
  JR_CMD_APPEND_ENTRIES = 4,
  JR_CMD_APPEND_RESPONSE = 5,
  JR_CMD_HEARTBEAT = 6,
  JR_CMD_HEARTBEAT_RESPONSE = 7,
  JR_CMD_TIMEOUT = 8,
  JR_CMD_NOOP = 9,
  JR_CMD_CLIENT_REQUEST = 10,
  JR_CMD_CLIENT_RESPONSE = 11
};

/* ---- Address (src/raft/rpc.rs:5-14) ------------------------------------- */
enum { JR_ADDR_PEERS = 0, JR_ADDR_PEER = 1, JR_ADDR_LOCAL = 2, JR_ADDR_CLIENT = 3 };

/* ---- sticky per-replica fault codes (deviation D3) ------------------------
 * 1..31: one per reference panic!/assert!/unimplemented!/Err site on the path. */
enum {
  JR_FAULT_NONE = 0,
  JR_FAULT_AE_STALE_LEADER = 1,       /* assert!, follower.rs:149-153                        */
  JR_FAULT_EXTEND_PARENT_MISSING = 2, /* Err from Chain::extend chain.rs:180-185 via follower.rs:159 `?` */
  JR_FAULT_APPEND_ID_NOT_GT_HEAD = 3, /* assert!(id > self.head), chain.rs:163               */
  JR_FAULT_COMMIT_BLOCK_MISSING = 4,  /* panic!(""), chain.rs:200-202                        */
  JR_FAULT_PROGRESS_UNKNOWN_NODE = 5, /* expect("the node does not exist"), progress.rs:43   */
  JR_FAULT_LEADER_TERM_UNIMPLEMENTED = 6, /* unimplemented!(), leader.rs:33-35 via leader.rs:203 */
  JR_FAULT_CANDIDATE_TICK_ELECTED = 7,/* panic!("this should never happen"), candidate.rs:63 */
  JR_FAULT_RANGE_COMMIT_KEY = 8,      /* bincode panic on the "commit" key, chain.rs:222-226 (D6) */
  /* 64..: engine limits, not reference behaviour */
  JR_FAULT_ENGINE_CHAIN_CAPACITY = 64,   /* block id outside [floor, floor + chain_capacity) (D4, D7) */
  JR_FAULT_ENGINE_MAILBOX_OVERFLOW = 65, /* a replica emitted more than mailbox_units units  */
  JR_FAULT_ENGINE_FSM_OVERFLOW = 66,     /* retired in ABI 2: a full Instruction FIFO drops records and the drain
                                          * returns JR_E_CAPACITY; observing a node never changes consensus     */
  JR_FAULT_ENGINE_QUEUE_OVERFLOW = 67    /* more than JR_CLIENT_QUEUE_CAP queued requests: the reference's
                                          * queued_reqs is an unbounded Vec (follower.rs:23); this engine bounds it,
                                          * so the (JR_CLIENT_QUEUE_CAP+1)-th ClientRequest a leaderless follower or
                                          * a candidate receives stops that replica                              */
};

/* ---- engine flags ---------------------------------------------------------- */
enum {
  JR_F_SLED_COMMIT_KEY_STRICT = 1u << 0, /* deviation D6 off: reproduce the commit-key panic */
  JR_F_CAPTURE_MESSAGES = 1u << 1,       /* jr_step may return every emitted Message (rpc_rx) */
  JR_F_CAPTURE_FSM = 1u << 2,            /* Instructions are stored (jr_step / jr_drain_fsm)  */
  JR_F_STREAM_DIGEST = 1u << 3,          /* keep the running digests jr_stream_digest returns  */
  JR_F_NO_SYMMETRIC_FOLD = 1u << 4       /* jr_run* never take the symmetric-group fast path (DESIGN.md section 3b); results are
                                          * identical either way -- the flag exists for A/B measurements and tests      */
};

/* ---- configuration (RaftConfig, src/raft/config.rs:14-41, batched) --------- */
typedef struct jr_config {
  uint32_t abi_version;        /* JR_ABI_VERSION                                         */
  uint32_t n_groups;           /* G, groups resident in this engine                      */
  uint32_t n_replicas;         /* R; node ids of every group are 1..R (config.rs:64: !=0) */
  int32_t  device;             /* CUDA device ordinal                                    */
  uint64_t seed;               /* D2                                                     */
  uint64_t group_offset;       /* global id of local group 0 (sharding keeps D2 stable)  */
  uint32_t election_min_ms;    /* State::min_election_timeout, mod.rs:318 (500)          */
  uint32_t election_max_ms;    /* State::max_election_timeout, mod.rs:319 (1000)         */
  uint32_t heartbeat_ms;       /* RaftConfig::heartbeat_timeout, config.rs:104 (100)     */
  uint32_t chain_capacity;     /* block ids one replica's table may span above the floor (D4, D7) */
  uint32_t mailbox_units;      /* 16-byte units one replica may emit per step            */
  uint32_t fsm_units;          /* jr_fsm_record slots per replica between two drains      */
  uint32_t flags;              /* JR_F_*                                                 */
  uint32_t resident_mask;      /* bit (id-1): node id is hosted by this engine; 0 = all R.
                                * A josefine process hosts ONE node per group (RaftConfig::id,
                                * config.rs:23) and reaches the others over TCP: non-resident
                                * nodes are never stepped, and mail addressed to them is only
                                * returned through out_msgs for the host to forward.           */
  uint32_t fsm_host_records;   /* records one jr_fsm_records_async batch may hold (pinned host memory,
                                * JR_STAGING_DEPTH + 1 buffers of this size); 0 = max(3 * n_groups * n_replicas + 1024,
                                * min(n_groups * n_replicas * fsm_units, 65536))                            */
  uint32_t fsm_raw_units;      /* scratch: raw Instructions one replica may emit per launch before they are encoded into
                                * records at the launch's end; 0 = 192.  jr_run* cut their work into launches of at most
                                * fsm_raw_units / 3 ticks; a replica that still emits more loses the excess (the drain
                                * then returns JR_E_CAPACITY; consensus is unaffected)                              */
} jr_config;

/* Block (src/raft/chain.rs:86-91); `data` is the payload token (D5). */
typedef struct jr_block {
  uint64_t id;
  uint64_t next;
  uint64_t data;
} jr_block;

/*
 * Message{from,to,command} (src/raft/rpc.rs:17-21) with Command flattened.
 * Field use per command (all others zero):
 *   VOTE_REQUEST       term, node_id=candidate_id, last_term, block=head
 *   VOTE_RESPONSE      term, node_id=from, flag=granted
 *   APPEND_ENTRIES     term, node_id=leader_id, n_blocks, blocks[]
 *   APPEND_RESPONSE    node_id, term, block=head, flag=success
 *   HEARTBEAT          term, block=commit, node_id=leader_id
 *   HEARTBEAT_RESPONSE block=commit, flag=has_committed
 *   CLIENT_REQUEST     token=request/payload token (D5), client_kind/client_id=address
 *   CLIENT_RESPONSE    token
 *   TICK, TIMEOUT, NOOP, PROPOSE: no fields
 */
typedef struct jr_msg {
  uint32_t group;
  uint8_t  from_kind;   /* JR_ADDR_* */
  uint8_t  to_kind;
  uint8_t  kind;        /* JR_CMD_*  */
  uint8_t  flag;
  uint32_t from_id;
  uint32_t to_id;
  uint32_t node_id;
  uint8_t  n_blocks;
  uint8_t  client_kind;
  uint16_t reserved;
  uint32_t client_id;
  uint32_t reserved2;
  uint64_t term;
  uint64_t last_term;
  uint64_t block;
  uint64_t token;
  jr_block blocks[JR_MAX_AE_BLOCKS];
} jr_msg;

/* Instruction (src/raft/fsm.rs:19-29). */
enum { JR_FSM_APPLY = 0, JR_FSM_NOTIFY = 1 };
typedef struct jr_fsm_instr {
  uint32_t group;
  uint32_t node;        /* the replica whose fsm_tx this was sent on */
  uint8_t  kind;        /* JR_FSM_*                                   */
  uint8_t  client_kind; /* Notify.client_address                      */
  uint16_t reserved;
  uint32_t client_id;
  jr_block block;       /* Apply: the Block; Notify: block.id = block_id, block.data = request token */
} jr_fsm_instr;

/*
 * Compact form of a replica's Instruction stream (fsm_tx; fsm.rs:19-29).  One record = a run:
 *   JR_FSMR_APPLY    `count` Apply instructions of blocks id0, id0+1, ...; element i carries
 *                    Block{id0+i, next_i, tok0 + i*stride} with next_i = id0+i-1.  count == 1 is the
 *                    general case: any block, next = (uint32_t)stride, data = tok0.
 *                    addr != 0: a node mask (bit id-1) -- the run belongs to the stream of EVERY node in the
 *                    mask (symmetric followers apply the same blocks), in front of that node's own records.
 *   JR_FSMR_NOTIFY   `count` Notify instructions for block ids id0, id0+1, ..., all with client address
 *                    (addr >> 16, addr & 0xffff); element i carries request token tok0 + i*stride.
 *   JR_FSMR_PATTERN  interleaving: bit b (0 <= b < count <= 160; bits 0-63 in tok0, 64-127 in stride, 128-159 in addr)
 *                    set = the (id0+b)-th Instruction this replica emitted since the last drain is a Notify.
 *                    Positions no PATTERN record marks are Apply.  Applies and Notifies each appear in record order, so the records of one replica
 *                    reproduce its stream exactly (jr_fsm_expand does).
 * A steady-state follower needs one APPLY record per launch, a leader one APPLY + one NOTIFY + one PATTERN per
 * 160 Instructions, whatever the number of fused ticks -- when tokens advance by a constant stride.
 */
enum { JR_FSMR_APPLY = 0, JR_FSMR_NOTIFY = 1, JR_FSMR_PATTERN = 2 };
typedef struct jr_fsm_record {
  uint32_t group;
  uint32_t hdr;      /* bits 0-1 JR_FSMR_*, bits 2-4 node id - 1, bits 8-31 count */
  uint32_t id0;
  uint32_t addr;
  uint64_t tok0;
  uint64_t stride;
} jr_fsm_record;
#define JR_FSMR_KIND(hdr) ((hdr) & 3u)
#define JR_FSMR_NODE(hdr) ((((hdr) >> 2) & 7u) + 1u)
#define JR_FSMR_COUNT(hdr) ((hdr) >> 8)

/* What one jr_fsm_records_async batch holds. */
typedef struct jr_fsm_batch {
  uint64_t n_records;                          /* records in the batch, sorted by (node, group), FIFO per replica */
  uint64_t n_dropped;                          /* records lost to a full per-replica FIFO or a full batch buffer  */
  uint64_t n_instructions;                     /* Instructions the records stand for                              */
  uint32_t node_offset[JR_MAX_REPLICAS + 1];   /* records of node n are [node_offset[n-1], node_offset[n])        */
  uint32_t reserved;
} jr_fsm_batch;

/* One dense client proposal per group: ClientRequest applied to `node` (0 = none).
 * Reference: event_loop client arm, src/raft/server.rs:156-160. */
typedef struct jr_proposal {
  uint64_t token;
  uint32_t node;
  uint32_t reserved;
} jr_proposal;

/* jr_step flags */
enum {
  JR_STEP_DELIVER = 1u << 0,  /* apply peer mail emitted in the previous step        */
  JR_STEP_TICK = 1u << 1,     /* then apply Command::Tick on every replica           */
  JR_STEP_SYNTH_PROPOSALS = 1u << 2, /* every current Leader receives n_synth ClientRequests */
  JR_STEP_TRUSTED_PROPOSALS = 1u << 3, /* caller guarantees proposals[g].node <= R: skip the O(G) host check */
  JR_STEP_REPORT_FAULTS = 1u << 4     /* fill n_faulted (one more small kernel; the call synchronises) */
};

/*
 * Per replica and step, commands are applied in this fixed order (our synthetic
 * schedule; the reference's is arrival order off tokio channels):
 *   1. JR_STEP_DELIVER: peer mail of the previous step, ascending sender id,
 *      FIFO per sender (only mail addressed to Peers or to this node);
 *   2. `inject[]` entries addressed to this replica, in array order;
 *   3. the dense `proposals[group]` entry if it names this node, then the
 *      synthetic proposals;
 *   4. JR_STEP_TICK: Command::Tick.
 * Mail of the previous step that is not delivered is dropped.
 */
typedef struct jr_step_args {
  uint64_t now_ms;               /* D1 */
  uint32_t flags;                /* JR_STEP_* */
  uint32_t n_synth;              /* proposals per leader per step with JR_STEP_SYNTH_PROPOSALS */
  const jr_msg* inject;          /* host; to_kind must be JR_ADDR_PEER and to_id in 1..R */
  size_t n_inject;
  const jr_proposal* proposals;  /* host; NULL or n_groups entries */
  /* outputs (host).  NULL/0 to skip.  With capture flags off these must be NULL. */
  jr_msg* out_msgs;
  size_t cap_msgs;
  size_t n_msgs;                 /* out: messages emitted this step, group-major, sender asc, FIFO */
  jr_fsm_instr* out_fsm;
  size_t cap_fsm;
  size_t n_fsm;                  /* out: instructions, group-major, node asc, FIFO */
  uint64_t n_faulted;            /* out, with JR_STEP_REPORT_FAULTS: replicas holding a sticky fault (D3) after this step --
                                  * the reference's `?` / panic leaving event_loop (server.rs:125-159), without a query per node */
} jr_step_args;

/* Introspection: Raft<T> pub fields (mod.rs:326-341) + role state. */
typedef struct jr_replica_state {
  uint64_t current_term;      /* State.current_term, mod.rs:276            */
  uint32_t voted_for;         /* State.voted_for, 0 = None                 */
  uint32_t leader_id;         /* Follower.leader_id, 0 = None              */
  uint64_t election_time_ms;  /* State.election_time (D1)                  */
  uint32_t election_timeout_ms;
  uint32_t rng_draws;
  uint64_t head;              /* Chain.head                                */
  uint64_t commit;            /* Chain.commit                              */
  uint64_t id_gen;            /* Chain.id_gen                              */
  uint64_t max_key;           /* largest block id present                  */
  uint64_t heartbeat_time_ms; /* Leader.heartbeat_time                     */
  uint32_t votes_seen;        /* Election.votes keys, bit (id-1)           */
  uint32_t votes_granted;     /* Election.votes == true, bit (id-1)        */
  uint64_t progress_head[JR_MAX_REPLICAS]; /* ReplicationProgress heads, index id-1 */
  uint32_t progress_replicate;/* bit (id-1): NodeProgress::Replicate (else Probe) */
  uint8_t  role;              /* JR_ROLE_*                                 */
  uint8_t  fault;             /* JR_FAULT_*                                */
  uint8_t  alive;
  uint8_t  n_queued;          /* queued_reqs.len()                         */
  uint64_t chain_floor;       /* D7: ids below this were truncated (0 = never) */
} jr_replica_state;

/* Leader::write_state record (leader.rs:103-107), one per group. */
typedef struct jr_leader_entry {
  uint64_t term;
  uint32_t leader_id;   /* 0 = the group has no live leader */
  uint32_t commit;
} jr_leader_entry;

typedef struct jr_engine jr_engine;

/* ---- lifecycle ------------------------------------------------------------- */
/* Page-locked host memory for the buffers the asynchronous calls read or fill (jr_run_tokens / jr_run_token_runs input,
 * jr_leader_table_async output): a host that binds this ABI over FFI has no CUDA runtime of its own to ask.  Pageable
 * memory also works everywhere -- the copies are then staged and the calls block for their duration. */
jr_status jr_host_alloc(size_t bytes, void** out);
void jr_host_free(void* p);
/* JR_E_INVAL for a configuration RaftConfig::validate (config.rs:60-84) rejects where the field exists here
 * (heartbeat_ms < 5, election_min_ms < 5), for an empty election range (follower.rs:103-108 gen_range would
 * panic) and for sizes outside the engine's limits. */
jr_status jr_engine_create(const jr_config* cfg, jr_engine** out);
void      jr_engine_destroy(jr_engine* e);
/* Back to the state right after jr_engine_create (every replica a fresh Follower with
 * an empty chain), keeping all allocations.  Reference: dropping the RaftHandle and
 * calling RaftHandle::new again on an empty data directory. */
jr_status jr_engine_reset(jr_engine* e);
/* Run all engine work on `cuda_stream` (a cudaStream_t); NULL = the engine's own. */
jr_status jr_engine_set_stream(jr_engine* e, void* cuda_stream);
jr_status jr_engine_sync(jr_engine* e);
const char* jr_last_error(void);
/* Fills the defaults the reference uses (500/1000/100 ms) and engine sizing. */
void      jr_config_default(jr_config* cfg, uint32_t n_groups, uint32_t n_replicas);

/* ---- stepping -------------------------------------------------------------- */
jr_status jr_step(jr_engine* e, jr_step_args* args);
/*
 * n_steps fused steps with no host traffic: step k uses now = now0 + k*dt_ms and
 * flags DELIVER|TICK (+SYNTH_PROPOSALS when n_synth > 0).  Asynchronous on the
 * engine stream.  Replica state, block tables, mailboxes and digests are bit for bit
 * those of n_steps jr_step calls.  Instructions are not returned here: with
 * JR_F_CAPTURE_FSM they accumulate, run-length encoded, in a per-replica FIFO of
 * fsm_units records until jr_fsm_records_async / jr_drain_fsm takes them (a jr_step
 * call starts its own FIFO and returns its Instructions itself).
 */
jr_status jr_run(jr_engine* e, uint64_t now0_ms, uint32_t dt_ms, uint32_t n_steps, uint32_t n_synth);
/*
 * jr_run with client input: `proposals` is HOST memory holding n_steps consecutive dense
 * arrays of n_groups entries (tick k uses proposals[k*n_groups ..]); equivalent to n_steps
 * jr_step calls with flags DELIVER|TICK and that tick's array, bit for bit, but one fused
 * launch and one host-to-device copy (staged on the engine's copy stream: pass pinned memory
 * and the call is asynchronous).  `flags` may carry JR_STEP_TRUSTED_PROPOSALS.
 */
jr_status jr_run_proposals(jr_engine* e, uint64_t now0_ms, uint32_t dt_ms, uint32_t n_steps,
                           const jr_proposal* proposals, uint32_t flags);
/*
 * jr_run_proposals with leader-routed input: `tokens` is HOST memory holding n_steps consecutive
 * arrays of n_groups 64-bit payload tokens (0 = no proposal; tick k uses tokens[k*n_groups ..]).
 * Each token is proposed at the node the most recent jr_leader_table / _device / _async call on this
 * engine announced as its group's leader -- the routing a josefine client does with the leader it
 * last learnt (Leader::write_state, leader.rs:101-121) before RaftClient::propose (client.rs:35-37)
 * reaches apply_client_request (leader.rs:177-194).  A group with no announced leader (also: no
 * announce since create / reset) drops its tokens, like a request sent nowhere: no Notify follows.
 * A stale route lands on a follower, which proxies it to its leader or, leaderless, queues it
 * (follower.rs:258-270) -- at most JR_CLIENT_QUEUE_CAP requests, see JR_FAULT_ENGINE_QUEUE_OVERFLOW.
 * Bit for bit equal to jr_run_proposals with proposals[k*G+g] = {tokens[k*G+g], route[g]}, at half
 * the host-to-device bytes (8 instead of 16 per group-tick).  Same asynchrony rules.
 */
jr_status jr_run_tokens(jr_engine* e, uint64_t now0_ms, uint32_t dt_ms, uint32_t n_steps,
                        const uint64_t* tokens);
/*
 * jr_run_tokens with the input in run-length form: `runs` is HOST memory holding ONE jr_token_run per group; tick k
 * proposes token runs[g].base + k * runs[g].stride for group g (base == 0: the group proposes nothing in this call).
 * Bit for bit equal to jr_run_tokens with tokens[k*G + g] = base + k*stride; 16 bytes per group and call instead of
 * 8 bytes per group-tick on the host-to-device link.  A host that numbers a partition's requests consecutively
 * (sequence numbers, log offsets) describes a whole quantum this way -- the mirror image of jr_fsm_record on the way out.
 */
typedef struct jr_token_run {
  uint64_t base;
  uint64_t stride;
} jr_token_run;
jr_status jr_run_token_runs(jr_engine* e, uint64_t now0_ms, uint32_t dt_ms, uint32_t n_steps,
                            const jr_token_run* runs);
/* Take the Instructions accumulated by jr_run* since the last drain, expanded: group-major, node ascending,
 * FIFO per node (the order jr_step returns).  *n = Instructions there were; JR_E_CAPACITY if `out` is too
 * small or records were dropped (fsm_units / fsm_host_records too small).  Synchronous; the FIFOs are empty
 * afterwards.  Small deployments and tests -- the batched path below is the fast one. */
jr_status jr_drain_fsm(jr_engine* e, jr_fsm_instr* out, size_t cap, size_t* n);
/*
 * The batched output path.  jr_fsm_records_async ENQUEUES, after everything submitted so far: pack all records
 * accumulated since the last drain into one dense array sorted by (node, group) and write it to the engine's
 * next pinned host buffer (JR_STAGING_DEPTH + 1 = 4 buffers used in turn, filled by the copy engine: the SMs stay with
 * the next step).  The FIFOs are empty afterwards.  jr_fsm_records_wait blocks until the OLDEST outstanding batch has
 * landed and returns it: `*records` points into the engine's buffer and stays valid until the JR_STAGING_DEPTH-1'th
 * jr_fsm_records_async call after this one, also when JR_STAGING_DEPTH batches were outstanding before the wait.  JR_E_CAPACITY (batch still returned) if records were dropped.  At
 * most JR_STAGING_DEPTH batches may be outstanding.  Requires JR_F_CAPTURE_FSM.
 * Threads: an engine is driven by ONE submitting thread (josefine's event_loop task); jr_fsm_records_wait and
 * jr_leader_table_wait (and the pure host functions jr_fsm_expand / jr_fsm_fold*) may be called from ONE other thread at
 * the same time -- the counterpart of josefine's fsm::Driver task (fsm.rs:52-88), which consumes fsm_tx while the Raft
 * task keeps stepping.  That thread must have returned a batch's buffer (be done reading it) before the submitting
 * thread's JR_STAGING_DEPTH-1'th jr_fsm_records_async after it.
 */
jr_status jr_fsm_records_async(jr_engine* e);
jr_status jr_fsm_records_wait(jr_engine* e, const jr_fsm_record** records, jr_fsm_batch* batch);
/*
 * Pure host function (no device, no engine): records (any order across replicas, FIFO per replica) ->
 * Instructions, group-major, node ascending, FIFO per node.  out may be NULL to size the buffer.
 * JR_E_CAPACITY if cap is too small (*n_out = needed), JR_E_INVAL for a malformed record set.
 */
jr_status jr_fsm_expand(const jr_fsm_record* records, size_t n_records, uint32_t n_groups, uint32_t n_replicas,
                        jr_fsm_instr* out, size_t cap, size_t* n_out);
/*
 * Pure host function: the bookkeeping of fsm::Driver (fsm.rs:52-88) for a batch, without expanding it.  For every
 * APPLY record, applied_hi[(node-1) * n_groups + group] becomes the highest block id that replica's driver has
 * applied (its apply watermark); totals[0] += Apply instructions, totals[1] += Notify instructions,
 * totals[2] += records.  One linear pass; `applied_hi` (n_replicas * n_groups entries) and `totals` (3 entries)
 * are caller-owned and accumulate across batches.
 */
jr_status jr_fsm_fold(const jr_fsm_record* records, size_t n_records, uint32_t n_groups, uint32_t n_replicas,
                      uint32_t* applied_hi, uint64_t* totals);
/* The same on n_threads host threads, for a batch as jr_fsm_records_wait returns it (sorted by (node, group)): thread t
 * folds the groups [G*t/T, G*(t+1)/T) of every node section, so no two threads touch the same watermark.  An unsorted
 * batch, or n_threads <= 1, is folded on the calling thread. */
jr_status jr_fsm_fold_mt(const jr_fsm_record* records, size_t n_records, uint32_t n_groups, uint32_t n_replicas,
                         uint32_t* applied_hi, uint64_t* totals, uint32_t n_threads);

/* ---- introspection --------------------------------------------------------- */
jr_status jr_query(jr_engine* e, uint32_t group, uint32_t node, jr_replica_state* out);
/* blocks with first_id <= id < first_id+n of one replica; present[i]=0 if absent. */
jr_status jr_chain_read(jr_engine* e, uint32_t group, uint32_t node, uint64_t first_id,
                        uint32_t n, jr_block* out, uint8_t* present);
/* The same for n replicas in ONE kernel + ONE copy: replica i is (groups[i], nodes[i]). */
jr_status jr_query_many(jr_engine* e, const uint32_t* groups, const uint32_t* nodes, size_t n,
                        jr_replica_state* out);
/* n block-table reads in one kernel + one copy: request i reads ids [first_id[i], first_id[i] + count[i]) of
 * replica (groups[i], nodes[i]); results are concatenated in request order. */
jr_status jr_chain_read_many(jr_engine* e, const uint32_t* groups, const uint32_t* nodes, const uint64_t* first_id,
                             const uint32_t* count, size_t n, jr_block* out, uint8_t* present);
/* order-independent digest of all replica state + block tables, computed on the device */
jr_status jr_state_digest(jr_engine* e, uint64_t* out);
/* cumulative digests of every Message / Instruction emitted so far (order sensitive per replica) */
jr_status jr_stream_digest(jr_engine* e, uint64_t* msg_digest, uint64_t* fsm_digest,
                           uint64_t* n_msgs, uint64_t* n_fsm);
jr_status jr_fault_count(jr_engine* e, uint64_t* n_faulted);
/* Diagnostic: how many groups the most recent jr_run* launch applied through the symmetric-group fast path
 * (0 if it was not offered: see JR_F_NO_SYMMETRIC_FOLD).  Synchronises. */
jr_status jr_fold_count(jr_engine* e, uint64_t* n_groups);

/* ---- maintenance ----------------------------------------------------------- */
jr_status jr_compact(jr_engine* e);                                    /* every replica */
jr_status jr_set_alive(jr_engine* e, uint32_t group, uint32_t node, int alive);
/* D7: per group, floor = max(old floor, min(commit of the live, unfaulted replicas) - margin); every block
 * below it is dropped from all replicas of the group.  Groups without a live replica keep their floor.
 * Asynchronous on the engine stream. */
jr_status jr_truncate(jr_engine* e, uint32_t margin);
/* D7, fused: while enabled, every jr_run / jr_run_proposals / jr_run_tokens / jr_run_token_runs call ends with
 * jr_truncate(margin) -- same result as calling it right after, but groups the symmetric-group fast path applied are
 * truncated by the lane that stepped them (no extra pass over their planes).  Off by default. */
jr_status jr_set_auto_truncate(jr_engine* e, int enabled, uint32_t margin);
/*
 * Node restart: replica (group, node) becomes what RaftHandle::new builds over an existing data directory
 * (mod.rs:428-435 -> follower.rs:68-95 -> Chain::new, chain.rs:117-137): a Follower with State::default
 * (term 0, voted_for None -- the reference does not persist them), election timer started at now_ms,
 * the block table = `blocks`, commit = head = id_gen = `commit` (so the first append of a restarted
 * leader-to-be asserts id > head and faults, SURVEY note N2).  commit == 0 runs Chain::init (genesis
 * block 0 -> 0 is (re)written, id_gen = 1).  `commit_key` = the sled "commit" key exists (D6).
 * The replica's mailbox and client queue are emptied; it is alive and unfaulted afterwards.
 */
jr_status jr_node_restart(jr_engine* e, uint32_t group, uint32_t node, uint64_t now_ms, const jr_block* blocks,
                          size_t n_blocks, uint64_t commit, int commit_key);
/* Checkpoint: everything the engine holds (state planes, block tables, mailboxes, FIFOs, routing, counters).
 * jr_engine_save_size -> bytes needed; restore needs an engine created with the same jr_config. */
jr_status jr_engine_save_size(jr_engine* e, size_t* bytes);
jr_status jr_engine_save(jr_engine* e, void* buf, size_t cap);
jr_status jr_engine_restore(jr_engine* e, const void* buf, size_t bytes);
/* Silence the current leader of every group g with hash(seed,g,salt) % 1000 < permille. */
jr_status jr_kill_leaders(jr_engine* e, uint64_t salt, uint32_t permille, uint64_t* n_killed);

/* ---- leader announce ------------------------------------------------------- */
/* Writes n_groups entries to DEVICE memory `dev_out` (for a collective) */
jr_status jr_leader_table_device(jr_engine* e, void* dev_out);
/* ... or to HOST memory (synchronises the engine stream). */
jr_status jr_leader_table(jr_engine* e, jr_leader_entry* host_out);
/* Same, but only ENQUEUES the kernel and the device-to-host copy: `host_out` must be
 * pinned memory and is valid after the next jr_engine_sync().  Lets a caller pipeline
 * jr_step (proposals H2D) / kernels / results D2H tick after tick. */
jr_status jr_leader_table_async(jr_engine* e, jr_leader_entry* host_out);
/* Block until the OLDEST outstanding jr_leader_table_async copy has landed (FIFO; at most JR_STAGING_DEPTH
 * are in flight).  Lets the host consume tick/step k's result while k+1 is already running. */
jr_status jr_leader_table_wait(jr_engine* e);

/* ---- deviation D2, normative ------------------------------------------------
 * draw-th election timeout of (group, node):
 *   x = mix(mix(mix(seed ^ 0x6a09e667f3bcc908) + group) + ((uint64)node << 32 | draw))
 *   timeout = min + (((x >> 32) * (max - min)) >> 32)
 * mix = splitmix64 finaliser: x += 0x9e3779b97f4a7c15; x = (x ^ x>>30) * 0xbf58476d1ce4e5b9;
 *       x = (x ^ x>>27) * 0x94d049bb133111eb; x ^= x>>31.
 */
uint32_t jr_election_timeout(uint64_t seed, uint64_t group, uint32_t node, uint32_t draw,
                             uint32_t min_ms, uint32_t max_ms);

#ifdef __cplusplus
}
#endif
#endif /* JOSEFINE_RAFT_ABI_H */
