/* tarok_b200 -- C ABI of the B200-native batched Tarok environment (libtarok_b200.so).
 *
 * The reference (anzeA/Tarok) is pure Python and has no FFI; its seam is the Python class API
 * between the engine (Tarok.py / Igra.py / Navadna_igra.py / Klop.py / Berac.py) and the players
 * (Igralec.py).  Each entry point below names the reference code it replaces ("File.py:N" is a
 * path into the reference tree).  The reference-side binding a maintainer would add is the ctypes
 * stub shown in INTEGRATION.md (and shipped as tarok_b200/_lib.py).
 *
 * Conventions
 *   - plain pointers and sizes only; no torch / C++ types.
 *   - every function returns 0 on success, <0 on error; tarok_last_error() gives the text.
 *   - "dev" pointers are CUDA device pointers on the handle's device; "host" pointers are host
 *     memory (pinned memory makes the copies asynchronous).
 *   - all device work is enqueued on the caller's stream (a cudaStream_t passed as void*;
 *     NULL = legacy default stream).  No hidden synchronisation unless stated.
 *   - a handle is not thread-safe; use one handle per GPU per thread.
 *   - state lives in the handle as structure-of-arrays of 64-bit bitboards (bit i = card id i,
 *     Karta.v_id, Karta.py:19-23) and is lent out zero-copy as DLPack tensors (tarok_export);
 *     the 64-bit words are typed int64 in DLPack (bit 63 is never set) because torch lacks uint64 ops.
 *   - an illegal action does not raise (the reference raises, Navadna_igra.py:125-126): the game's
 *     error bit is set in `meta`, the game stops, and the error counter in `stats` increments.
 */
#ifndef TAROK_B200_H
#define TAROK_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct tarok_env tarok_t;

/* ---- DLPack (v0.8 ABI subset; identical layout to dlpack.h) ------------------------------- */
#ifndef DLPACK_DLPACK_H_
typedef struct { int32_t device_type; int32_t device_id; } DLDevice;       /* kDLCUDA = 2 */
typedef struct { uint8_t code; uint8_t bits; uint16_t lanes; } DLDataType;  /* kDLInt=0 kDLUInt=1 */
typedef struct {
    void* data; DLDevice device; int32_t ndim; DLDataType dtype;
    int64_t* shape; int64_t* strides; uint64_t byte_offset;
} DLTensor;
typedef struct DLManagedTensor {
    DLTensor dl_tensor; void* manager_ctx; void (*deleter)(struct DLManagedTensor* self);
} DLManagedTensor;
#endif

/* ---- constants ----------------------------------------------------------------------------- */
/* contract code = Tip_igre value / 10 (Tip_igre.py:5-15) */
enum { TAROK_KLOP = 0, TAROK_TRI = 1, TAROK_DVE = 2, TAROK_ENA = 3, TAROK_SOLO_TRI = 4,
       TAROK_SOLO_DVE = 5, TAROK_SOLO_ENA = 6, TAROK_BERAC = 7, TAROK_SOLO_BREZ = 8,
       TAROK_ODPRTI_BERAC = 9 };
#define TAROK_NO_KING 7
#define TAROK_NO_GROUP 0xFF
/* synthetic-input modes (DESIGN.md "Synthetic inputs") */
#define TAROK_MODE_NAVADNA_MIX 16      /* Tri/Dve/Ena uniform, declarer & king uniform (config 2) */
#define TAROK_MODE_AUCTION_UNIFORM 17  /* one uniform index2igra intent per seat, random talon group */
#define TAROK_MODE_AUCTION_BOT 18      /* Bot_igralec bidding distribution, group 0 */
/* flags for tarok_create */
#define TAROK_FLAG_HISTORY 1u          /* keep the play history (seat<<6|card per play) for observations */
/* exportable fields */
enum { TAROK_F_HANDS = 0,   /* uint64 [4, n_alloc]  hand bitboards (Roka, Roka.py:4-13) in LEADER-RELATIVE slots: row j is
                               the hand of seat (leader + j) & 3, leader = bits 13-14 of the game's meta word (0 from
                               the deal until a contract or a trick moves it), so the seat to move is always row `pos`;
                               tarok_hands_by_seat copies them out indexed by seat */
       TAROK_F_PILES = 1,   /* uint64 [4, n_alloc]  won-cards pile of seat s (Igralec.kupcek): discards at once, won tricks
                               (and the Klop talon in TAROK_F_TALON) are materialised from the trick log by tarok_score */
       TAROK_F_TALON = 2,   /* uint64 [n_alloc]     cards still in the talon                                 */
       TAROK_F_TALON_ORDER = 3, /* uint64 [n_alloc] the 6 talon ids in dealt order, 6 bits each (Igra.py:68) */
       TAROK_F_META = 4,    /* uint64 [n_alloc]     packed contract / trick state (layout in DESIGN.md)      */
       TAROK_F_MASK = 5,    /* uint64 [n_alloc]     legal-move mask of the seat to move                      */
       TAROK_F_SCORES = 6,  /* int16  [n_alloc, 4]  pisejo by seat                                           */
       TAROK_F_HIST = 7,    /* uint8  [48, n_alloc] play t of game g: seat<<6|card, 0xFF = not played        */
       TAROK_F_STATS = 8,   /* int64  [32]          accumulated statistics (layout below)                    */
       TAROK_F_HANDS0 = 9,  /* uint64 [4, n_alloc]  hands as dealt (Nevronski_igralec.zacetna_roka); HISTORY flag */
       TAROK_F_DISCARD = 10,/* uint64 [n_alloc]     declarer's discards (zalozil); HISTORY flag              */
       TAROK_F_QMAX_HIST = 11 /* float [48, n_alloc] next_Q_max recorded by tarok_select_action at play t; HISTORY flag */
};
/* stats vector: [0..3] score sum by seat, [4..7] score sum by player ((seat+game_id)%4, Tarok.py:34,59-61),
   [8..17] contract histogram, [18] finished deals, [19] env-steps (card plays), [20] error games (these at scoring);
   [21] error events: counted at once by the stepwise call that makes a game an error game (tarok_set_deals,
   tarok_auction, tarok_force_contract, tarok_exchange, tarok_step, tarok_setup_synth and the *_bots entries), so at most
   once per game and deal; the fused kernel does not count them. */
#define TAROK_STATS_LEN 32

/* ---- life cycle ---------------------------------------------------------------------------- */
int tarok_create(int device, uint64_t n_games, uint64_t seed, uint32_t flags, tarok_t** out);
int tarok_destroy(tarok_t* h);                 /* error if exported tensors are still alive */
const char* tarok_last_error(const tarok_t* h);/* h may be NULL: last error of a failed tarok_create */
/* Tuning knobs.  Option id 1 (the play_step implementation) is retired and will not be reused. */
#define TAROK_OPT_PDL 2        /* 1 (default): chain play_step launches with programmatic dependent launch */
#define TAROK_OPT_MATERIALISE 4 /* 1 (default): tarok_score writes the full piles / Klop talon back; 0: scores + stats only */
#define TAROK_OPT_CHUNKS 5      /* 1..32 (default 8): chunks of the upload/compute/download pipeline of tarok_rollout_host/_records */
#define TAROK_OPT_DRAW_CACHE 7  /* trick positions whose in-kernel random draws are read from the cache the position-0 launch leaves behind
                                   instead of recomputed: 0 off, 2 positions 1-2, 3 positions 1-3, -1 default by batch size; results identical */
#define TAROK_OPT_LAZY_MASK 6   /* 1 (default): a chain of in-kernel random steps (tarok_steps_random, the stepwise rollouts) writes
                                   TAROK_F_MASK in its LAST launch only -- the interior masks cannot be observed; 0: every launch */
#define TAROK_OPT_GRAPH 8       /* 1 (default): tarok_rollout_stepwise replays a CUDA graph of its 50 launches (captured on first use per
                                   mode; first_gid is handed over through device memory): ~13 us of host time per rollout instead
                                   of ~150 and no launch gaps on the GPU -- for batches up to 3 M deals (beyond that the kernels are
                                   long and HBM-bound and the plain launches are as fast); 2: at every size; 0: plain launches.
                                   Same results either way. */
#define TAROK_OPT_LOCKSTEP 3   /* 1 (default): play_step variants specialised per trick position for lock-step batches */
int tarok_set_option(tarok_t* h, int option, int64_t value);
uint64_t tarok_n_games(const tarok_t* h);
uint64_t tarok_n_alloc(const tarok_t* h);      /* n_games rounded up to the kernel tile */

/* ---- deal: Igra.razdeli (Igra.py:65-73) ------------------------------------------------------ */
/* Philox4x32-10 deal, replayable from (seed, global game id); game g of this handle is global
   game first_global_game_id + g.  Resets piles, meta and the per-game error bits. */
int tarok_deal(tarok_t* h, uint64_t first_global_game_id, void* stream);
/* Deal injection: perm_dev is uint8 [n_games, 54]; seat i gets perm[12i:12i+12], talon = perm[48:54]
   in order -- exactly what a patched Igra.shuffle (Igra.py:10,67) would feed Igra.razdeli. */
int tarok_set_deals(tarok_t* h, const uint8_t* perm_dev, uint64_t first_global_game_id, void* stream);
/* The current deal as the permutation Igra.razdeli would have consumed (hand slices ascending by id).
   Only meaningful before the talon exchange.  out_dev: uint8 [n_games, 54]. */
int tarok_export_perm(tarok_t* h, uint8_t* out_dev, void* stream);

/* ---- auction + dispatch: Igra.licitacija (Igra.py:75-114), Igralec.licitiram filter
        (Igralec.py:58-74), Igra.start dispatch (Igra.py:38-58), Navadna_igra.__init__ teams
        (Navadna_igra.py:20-30) ------------------------------------------------------------------ */
/* intent_dev: uint8 [n_games, 4]; one bid intent per seat as an index into
   Nevronski_igralec.index2igra (Igralec.py:717-745): 0 Naprej, 1-12 (Tri|Dve|Ena, king suit),
   13-15 Solo_tri/dve/ena, 16 Berac, 17 Solo_brez; additionally 18 Odprti_berac, 19 Klop.
   Fixed-intent semantics of Nevronski_igralec.licitiram (Igralec.py:294-306): every seat is asked at least once, so a
   game with any intent in 20..255 becomes an error game (the reference's index2igra[idx] raises). */
int tarok_auction(tarok_t* h, const uint8_t* intent_dev, void* stream);
int tarok_auction_synth(tarok_t* h, uint32_t mode /* 17 | 18 */, void* stream);
/* Bypass bidding like the per-contract constructors Klop(...)/Navadna_igra(...)/Berac(...).
   contract_dev/declarer_dev/king_dev: uint8 [n_games] (king ignored unless Tri/Dve/Ena). */
int tarok_force_contract(tarok_t* h, const uint8_t* contract_dev, const uint8_t* declarer_dev,
                         const uint8_t* king_dev, void* stream);
int tarok_force_contract_synth(tarok_t* h, uint32_t mode /* 0..9 | 16 */, void* stream);

/* ---- mixed tables: Bot_igralec seats beside caller-driven (neural) seats ----------------------------------------------
   bots_dev: uint8 [n_games], a per-game seat mask: bit s set = seat s of that game is a Bot_igralec (Igralec.py:145-171)
   whose decisions are drawn in-kernel from the same stateless Philox draws as the all-bot paths -- its bids from the bid
   block (mode 18), its king from setup-block word 2, its exchange from words 1 (group 0), its cards from play_draw -- so a
   bot seat can sit anywhere and every game stays replayable from (seed, global game id).  A game whose byte has any of
   bits 4-7 set becomes an error game (counted once in stats[21]).  A NULL bots_dev, or a pointer that breaks an alignment
   rule, fails the call (< 0) and writes nothing.  With bots_dev all zero each entry computes what its plain namesake does;
   with 0x0F everywhere, deal + the three entries + score compute what deal + tarok_auction_synth(18) +
   tarok_exchange_synth(0) + 48 x tarok_step_random + score do.
   tarok_auction_bots: tarok_auction where bot seats draw a fresh bid at every licitiram call (the draw mode 18 takes at the
     same overall call number) and their intent bytes are ignored; a bot declarer of a king game calls the king mode 18
     would, a neural one the suit of its original intent.  intent_dev 4-byte aligned, as for tarok_auction.
   tarok_exchange_bots: tarok_exchange where games whose declarer's seat is a bot take the Bot exchange (group 0, uniform
     discards) and ignore their group / discard entries.  discard_dev 8-byte aligned.
   tarok_step_bots: tarok_step where a bot to move plays the uniform legal card tarok_step_random would play at that game's
     play index; its card byte is ignored, except TAROK_CARD_SKIP, which still holds the game for this launch.  card_dev and
     bots_dev 2-byte aligned.  This entry keeps the lock-step specialisation and PDL, and neither reads nor writes the
     draw cache of the random chains. */
int tarok_auction_bots(tarok_t* h, const uint8_t* intent_dev, const uint8_t* bots_dev, void* stream);
int tarok_exchange_bots(tarok_t* h, const uint8_t* group_dev, const uint64_t* discard_dev, const uint8_t* bots_dev,
                        void* stream);
int tarok_step_bots(tarok_t* h, const uint8_t* card_dev, const uint8_t* bots_dev, void* stream);

/* ---- talon exchange: Navadna_igra.odpri_talon + start (Navadna_igra.py:36-68),
        Roka.mozno_zalozit (Roka.py:23-27), player side Igralec.py:161-171 ---------------------- */
/* group_dev: uint8 [n_games] chosen group; discard_dev: uint64 [n_games] bitboard of the k cards laid
   down.  Only games waiting for an exchange are touched. */
int tarok_exchange(tarok_t* h, const uint8_t* group_dev, const uint64_t* discard_dev, void* stream);
int tarok_exchange_synth(tarok_t* h, uint32_t random_group, void* stream);

/* ---- play: mozne_karte (Navadna_igra.py:158-168, Klop.py:96-133), krog (Navadna_igra.py:115-141,
        Klop.py:47-79), pobere_stih/primerjaj_karti (Navadna_igra.py:143-156), Berac.start
        (Berac.py:13-44) --------------------------------------------------------------------------- */
int tarok_legal_mask(tarok_t* h, uint64_t* out_dev, void* stream);   /* recomputed from the state */
/* The four hands of every game indexed by SEAT (uint64 [4, n_alloc] on the device): TAROK_F_HANDS un-rotated. */
int tarok_hands_by_seat(tarok_t* h, uint64_t* out_dev, void* stream);
/* card_dev: uint8 [n_games], one card id per live game (entries of games not waiting for a card are ignored);
   TAROK_CARD_SKIP leaves a live game untouched for this launch (advance a subset, e.g. SURVEY Q17). */
#define TAROK_CARD_SKIP 0xFE
int tarok_step(tarok_t* h, const uint8_t* card_dev, void* stream);   /* one card per live game */
int tarok_step_random(tarok_t* h, void* stream);                     /* uniform-random legal card */
int tarok_steps_random(tarok_t* h, uint32_t count, void* stream);    /* `count` back-to-back random steps */

/* ---- scoring: Roka.prestej (Roka.py:55-98), epilogues Navadna_igra.py:80-113, Klop.py:36-45,
        Berac.py:33-44; Tarok.rezultati accumulation (Tarok.py:59-61) --------------------------- */
int tarok_score(tarok_t* h, int16_t* out_dev /* [n_games,4] or NULL */, void* stream);
int tarok_reset_stats(tarok_t* h, void* stream);
/* A new run seed for an existing handle (what tarok_create's `seed` sets: the key of every synthetic Philox draw) without
   releasing the device buffers; work already enqueued keeps the old seed. */
int tarok_reseed(tarok_t* h, uint64_t seed);
int tarok_read_stats(tarok_t* h, int64_t* out_host /* [32] */, void* stream); /* synchronises stream */

/* ---- multi-GPU: the only exchange on the path (SURVEY.md 8e) ------------------------------------ */
/* Sums the statistics vector over all ranks of `nccl_comm` (an ncclComm_t passed as void*) into out_dev (int64 [32]
   on this device): one ncclAllReduce(ncclSum, ncclInt64) on the caller's stream, i.e. Tarok.rezultati (Tarok.py:59-61)
   for game shards spread over several GPUs.  The handle's own vector is left untouched.  libnccl is dlopen'ed. */
int tarok_allreduce_stats(tarok_t* h, void* nccl_comm, int64_t* out_dev, void* stream);

/* ---- whole deals ----------------------------------------------------------------------------- */
/* deal + contract(mode) + talon exchange with device-side (Philox) decisions in ONE launch; the state it
   leaves is bit-identical to tarok_deal + tarok_auction_synth/tarok_force_contract_synth + tarok_exchange_synth. */
int tarok_setup_synth(tarok_t* h, uint32_t mode, uint64_t first_global_game_id, void* stream);
/* Stepwise pipeline with in-kernel uniform-random players: setup (deal, contract(mode), exchange) ->
   48 x step_random -> score = 50 launches.  Equivalent to Tarok.paralel_start with Bot-like players. */
int tarok_rollout_stepwise(tarok_t* h, uint32_t mode, uint64_t first_global_game_id, void* stream);
/* Same result, one fused kernel with the state in registers (not HBM-bound). */
int tarok_rollout_fused(tarok_t* h, uint32_t mode, uint64_t first_global_game_id, void* stream);
/* Host-buffer entry (the end-to-end path): uploads injected deals (uint8 [n,54]) and forced
   contracts (uint8 [n] each; king may be NULL for non-king games), plays them with uniform-random
   players, downloads scores (int16 [n,4]) and the stats vector (int64 [32]).  Asynchronous on
   `stream` when the host buffers are pinned; the caller synchronises.  The host-buffer entries (this one, _host_packed,
   _records) START FROM A CLEARED statistics vector: stats_host holds the statistics of this call's deals only, and whatever
   the handle had accumulated before is gone (read it with tarok_read_stats first if it matters). */
int tarok_rollout_host(tarok_t* h, const uint8_t* perm_host, const uint8_t* contract_host,
                       const uint8_t* declarer_host, const uint8_t* king_host,
                       uint64_t first_global_game_id, int fused,
                       int16_t* scores_host, int64_t* stats_host, void* stream);

/* Deal records: the same inputs as tarok_rollout_host in 20 instead of 57 bytes per deal (the host-buffer path is
   PCIe-bound, so the bytes are the cost).  One record = 20 bytes, little endian: uint64 w0, uint64 w1, uint32 w2 (records are
   packed back to back, so only every other one is 8-byte aligned):
     bits 0..53 of w0/w1     = bit planes 0/1 of the seat (0-3) whose twelve cards of Igra.razdeli (Igra.py:65-73) hold
                               card id i (bit i = card id i); the six talon cards carry 0 in both planes;
     a 45-bit word m         = bits 54..63 of w0 (m bits 0..9), bits 54..63 of w1 (m bits 10..19) and w2 (m bits 20..44):
       m bits 0..35          = the six talon ids in talon order (karte[48:54]), 6 bits each, first card lowest;
       m bits 36..39 contract code, 40..41 declarer seat, 42..44 king suit (7 = none): the arguments of tarok_force_contract;
     every other bit is 0.
   tarok_pack_records is the host-side serialiser (plain CPU code; returns the number of rows that are not permutations
   or carry an out-of-range contract/declarer -- those become records that decode to error games -- or -1 on NULL). */
#define TAROK_RECORD_BYTES 20
int64_t tarok_pack_records(const uint8_t* perm_host, const uint8_t* contract_host, const uint8_t* declarer_host,
                           const uint8_t* king_host /* or NULL */, uint64_t n, void* records_host /* n x 20 bytes */);
/* The same serialiser spread over `threads` host threads (std::thread; callers launched by torchrun run with
   OMP_NUM_THREADS=1, so the count is explicit). */
int64_t tarok_pack_records_mt(const uint8_t* perm_host, const uint8_t* contract_host, const uint8_t* declarer_host,
                              const uint8_t* king_host /* or NULL */, uint64_t n, void* records_host, int threads);
/* The serialiser picks an AVX-512 (VBMI) implementation at run time where the CPU has it (one row per 64-bit lane, sixteen
   rows = five cache lines of records per iteration), else scalar code (BMI2 clone where available); both produce identical records.  tarok_pack_uses_avx512 tells which one runs,
   tarok_pack_force_scalar(1) pins the scalar one (returns the previous setting; a testing aid). */
int tarok_pack_uses_avx512(void);
int tarok_pack_force_scalar(int on);
/* tarok_rollout_host(fused = 1) that serialises the rows itself: each chunk of the upload/compute/download pipeline is
   packed into records by `threads` host threads (a pool kept in the handle, pinned scratch owned by the handle) right
   before its upload, so the caller keeps handing over what Igra.shuffle produces (Igra.py:65-73) and PCIe carries
   20 B/deal.  Same outputs as tarok_rollout_host, bit-identical scores.  The pack runs on the calling thread + the pool:
   the call returns when the last chunk is enqueued (device work still asynchronous on `stream`). */
int tarok_rollout_host_packed(tarok_t* h, const uint8_t* perm_host, const uint8_t* contract_host,
                              const uint8_t* declarer_host, const uint8_t* king_host, uint64_t first_global_game_id,
                              int threads, int16_t* scores_host, int64_t* stats_host, void* stream);
/* tarok_rollout_host(fused = 1) fed with deal records; same outputs, bit-identical scores. */
int tarok_rollout_records(tarok_t* h, const void* records_host, uint64_t first_global_game_id,
                          int16_t* scores_host, int64_t* stats_host, void* stream);

/* ---- observations: Nevronski_igralec.stanje_v_vektor_rek_navadna (Igralec.py:453-533) --------- */
/* Needs TAROK_FLAG_HISTORY.  net_type follows Nevronski_igralec.Tipi_NN: 0 Klop, 1 Navadna_igra (Tri/Dve/Ena),
   2 Solo (Solo_*), 3 Berac.  tarok_obs_shape gives, per game, the net type of its contract (255 = not waiting
   for a card) and the reference's padded history length T (multiple of 8), i.e. the (net, T) bucket
   predict_igraj_karto (Igralec.py:316-342) batches by.  tarok_obs_expand writes, for the seat to move of the
   n_sel selected games (sel_dev: int32 game indices, NULL = 0..n_sel-1), the fp32 input arrays in the reference's
   layout: opp [n_sel,T,3,54], hand [n_sel,T,54], talon [n_sel,6,55] (types 1,2) / [n_sel,54] (type 0),
   king [n_sel,4] (type 1), decl [n_sel,4], discard [n_sel,54], mozne [n_sel,54]; optional outputs may be NULL.
   Games that do not belong to the (net_type, rows) bucket get zeros and ok = 0. */
int tarok_obs_shape(tarok_t* h, uint8_t* type_dev, uint8_t* rows_dev, void* stream);
/* The same bucketing done on the device, for the `players` (1 or 4) players of Tarok.paralel_start -- the player of
   seat s in game i is (s + i) % 4 (Tarok.py:34), every Nevronski_igralec keeps its own queues per net type
   (Igralec.py:235-236,316-342): a stable counting sort of the games waiting for a card by
   key = player * 28 + net_type * 7 + (T / 8 - 1).  sel_dev: int32 [n_games] receives the game indices grouped by key
   (ascending key, ascending game index inside a key; only the first sum(counts) entries are written); selkey_dev
   (uint8 [n_games], optional) the key of every listed position; counts_dev: uint32 [384] = 128 bucket sizes, 128 bucket
   offsets into sel_dev (entry 255 = number of listed games), 128 bucket offsets in observation ROWS (sum of size * T over
   the earlier buckets).  The caller reads counts once per step. */
int tarok_obs_buckets(tarok_t* h, int players, int32_t* sel_dev, uint32_t* counts_dev, uint8_t* selkey_dev, void* stream);
/* The same, and the 384 counts copied to counts_host (pinned host memory, may be NULL) behind them; the three kernels and the
   copy go out as one CUDA-graph launch (TAROK_OPT_GRAPH): this call runs once per self-play step on an empty stream, where
   every launch costs its full latency.  The caller synchronises the stream before reading counts_host. */
int tarok_obs_buckets_host(tarok_t* h, int players, int32_t* sel_dev, uint32_t* counts_dev, uint8_t* selkey_dev,
                           uint32_t* counts_host, void* stream);
/* All buckets of a step in ONE launch each: tarok_obs_expand_buckets writes the inputs of every listed game into arenas
   laid out so that each bucket's arrays are contiguous -- opp [rows,3,54] / hand [rows,54] at row counts[256 + key] +
   (i - counts[128 + key]) * T for position i of sel_dev, the per-game vectors (talon [.,6,55], talon_klop [.,54], king [.,4],
   decl [.,4], discard [.,54]) at index i -- i.e. bucket `key` reads opp_dev + counts[256+key]*162 as [size,T,3,54],
   talon_dev + counts[128+key]*330 as [size,6,55] and so on.  Arena capacities: n_games * 56 rows / n_games entries.
   tarok_select_action_buckets then applies tarok_select_action to every listed game with q_ptrs_dev[key] (a device table
   of 128 device pointers, NULL = bucket not evaluated) = that bucket's [size,54] network output and
   random_card4[player] = that player's epsilon (host array of 4). */
int tarok_obs_expand_buckets(tarok_t* h, const int32_t* sel_dev, const uint8_t* selkey_dev, const uint32_t* counts_dev,
                             uint64_t n_total, float* opp_dev, float* hand_dev, float* talon_dev, float* talon_klop_dev,
                             float* king_dev, float* decl_dev, float* discard_dev, void* stream);
int tarok_select_action_buckets(tarok_t* h, const float* const* q_ptrs_dev, const int32_t* sel_dev, const uint8_t* selkey_dev,
                                const uint32_t* counts_dev, uint64_t n_total, const float* random_card4, uint8_t* card_dev,
                                float* qmax_dev, void* stream);
/* tarok_select_action_buckets with the table of 128 device pointers given in HOST memory (it travels as kernel parameters:
   nothing to fill or copy on the device). */
int tarok_select_action_buckets_tab(tarok_t* h, const float* const* q_ptrs_host, const int32_t* sel_dev, const uint8_t* selkey_dev,
                                    const uint32_t* counts_dev, uint64_t n_total, const float* random_card4, uint8_t* card_dev,
                                    float* qmax_dev, void* stream);
int tarok_obs_expand(tarok_t* h, int net_type, uint32_t rows, const int32_t* sel_dev, uint64_t n_sel, float* opp_dev,
                     float* hand_dev, float* talon_dev, float* king_dev, float* decl_dev, float* discard_dev,
                     float* mozne_dev, uint8_t* ok_dev, void* stream);

/* Action selection: Nevronski_igralec.igraj_karto (Igralec.py:344-355).  q_dev: fp32 [n_sel,54] network outputs
   for the selected games; writes card_dev[game] (uint8 [n_games], indexed by GAME, ready for tarok_step; 0xFF for
   games not to move) = first argmax over the legal cards in the reference's `mozne` order, or with probability
   random_card a uniform legal card (Philox stream 8); qmax_dev[game] (fp32 [n_games], optional) = next_Q_max. */
int tarok_select_action(tarok_t* h, const float* q_dev, const int32_t* sel_dev, uint64_t n_sel, float random_card,
                        uint8_t* card_dev, float* qmax_dev, void* stream);

/* tarok_obs_expand_at: the same arrays as they were at the decision of card play `play` (0..47) of each selected game,
   for the seat that made that play -- the `stanje` half of a replay sample (mozne_dev is left zero).
   tarok_targets: Nevronski_igralec.rezultat_stiha / rezultat_igre (Igralec.py:387-446): for finished games, dy_dev fp32
   [n_sel,48,54] row t = the target vector of card play t (-70 on illegal cards, +-trick value + final_reword_factor *
   next_Q_max / final score on the played card), seat_dev uint8 [n_sel,48] = the seat that played (0xFF = no play),
   rows_dev uint8 [n_sel,48] (optional) = the T of that sample's observation.  Uses the next_Q_max values recorded by
   tarok_select_action (TAROK_F_QMAX_HIST). */
int tarok_obs_expand_at(tarok_t* h, int play, int net_type, uint32_t rows, const int32_t* sel_dev, uint64_t n_sel,
                        float* opp_dev, float* hand_dev, float* talon_dev, float* king_dev, float* decl_dev,
                        float* discard_dev, float* mozne_dev, uint8_t* ok_dev, void* stream);
int tarok_targets(tarok_t* h, const int32_t* sel_dev, uint64_t n_sel, float final_reword_factor, float* dy_dev,
                  uint8_t* seat_dev, uint8_t* rows_dev, void* stream);

/* Bidding / exchange side of the neural player.
   tarok_obs_hands: pripavi_licitiram (Igralec.py:278-281), out_dev fp32 [n_games,4,54] = every seat's hand.
   tarok_obs_exchange: menjaj_talon_v_vektor (Igralec.py:535-543) for games waiting for an exchange:
     hand [n_sel,54] (declarer), talon [n_sel,54,6] (card x group), game [n_sel,15] one-hot.
   tarok_select_exchange: menjaj_iz_talona (Igralec.py:365-385) from the 60 network outputs p_dev [n_sel,60]:
     group_dev[game] (uint8 [n_games]) and discard_dev[game] (uint64 [n_games]) ready for tarok_exchange. */
int tarok_obs_hands(tarok_t* h, float* out_dev, void* stream);
int tarok_obs_exchange(tarok_t* h, const int32_t* sel_dev, uint64_t n_sel, float* hand_dev, float* talon_dev, float* game_dev,
                       uint8_t* ok_dev, void* stream);
int tarok_select_exchange(tarok_t* h, const float* p_dev, const int32_t* sel_dev, uint64_t n_sel, float random_card,
                          uint8_t* group_dev, uint64_t* discard_dev, void* stream);

/* ---- mixed precision: the observation and selection entries above in bf16 / fp16 ----------- */
/* Element type of the observation outputs and of the network outputs the selections read.  Every observation value is
   exactly 0 or 1, so bf16 and fp16 observations equal the fp32 ones converted, bit for bit, at half the bytes.  Network
   outputs are widened to fp32 (exact) and then selected by the fp32 rules: the first NaN wins, -inf and -max are ordinary
   values, +0 == -0, ties go by the reference's `mozne` order (cards) and by the stable mozno_zalozit order (discards).
   qmax_dev, TAROK_F_QMAX_HIST and tarok_targets stay fp32. */
#define TAROK_DTYPE_F32 0
#define TAROK_DTYPE_BF16 1
#define TAROK_DTYPE_F16 2
/* Each *_ex entry is the entry of the same name with buffers of element type `dtype` (an unknown dtype is an error); the
   fp32 entries are these at TAROK_DTYPE_F32.  Alignment at every dtype: opp / hand 16 bytes; talon, talon_klop, discard,
   mozne and the exchange hand / talon two elements (8 bytes fp32, 4 bytes bf16 / fp16); king / decl 4 bytes; every other
   buffer one element.  A call that fails its checks writes nothing. */
int tarok_obs_expand_at_ex(tarok_t* h, int dtype, int play, int net_type, uint32_t rows, const int32_t* sel_dev, uint64_t n_sel,
                           void* opp_dev, void* hand_dev, void* talon_dev, void* king_dev, void* decl_dev,
                           void* discard_dev, void* mozne_dev, uint8_t* ok_dev, void* stream);
int tarok_obs_expand_buckets_ex(tarok_t* h, int dtype, const int32_t* sel_dev, const uint8_t* selkey_dev, const uint32_t* counts_dev,
                                uint64_t n_total, void* opp_dev, void* hand_dev, void* talon_dev, void* talon_klop_dev,
                                void* king_dev, void* decl_dev, void* discard_dev, void* stream);
int tarok_obs_hands_ex(tarok_t* h, int dtype, void* out_dev, void* stream);
int tarok_obs_exchange_ex(tarok_t* h, int dtype, const int32_t* sel_dev, uint64_t n_sel, void* hand_dev, void* talon_dev,
                          void* game_dev, uint8_t* ok_dev, void* stream);
int tarok_select_action_ex(tarok_t* h, int dtype, const void* q_dev, const int32_t* sel_dev, uint64_t n_sel, float random_card,
                           uint8_t* card_dev, float* qmax_dev, void* stream);
/* One dtype for every pointer of the table. */
int tarok_select_action_buckets_tab_ex(tarok_t* h, int dtype, const void* const* q_ptrs_host, const int32_t* sel_dev,
                                       const uint8_t* selkey_dev, const uint32_t* counts_dev, uint64_t n_total,
                                       const float* random_card4, uint8_t* card_dev, float* qmax_dev, void* stream);
int tarok_select_exchange_ex(tarok_t* h, int dtype, const void* p_dev, const int32_t* sel_dev, uint64_t n_sel, float random_card,
                             uint8_t* group_dev, uint64_t* discard_dev, void* stream);

/* ---- zero-copy views ------------------------------------------------------------------------- */
/* Lends a field as a DLPack tensor that aliases the handle's device memory.  The caller (e.g.
   torch.from_dlpack) must call the deleter; the handle cannot be destroyed before that. */
int tarok_export(tarok_t* h, int field, DLManagedTensor** out);
/* Raw device pointer of a field (same memory as tarok_export), for C callers. */
void* tarok_field_ptr(tarok_t* h, int field);

/* Number of kernels this library has launched on the handle since creation (bench bookkeeping). */
uint64_t tarok_launch_count(const tarok_t* h);

#ifdef __cplusplus
}
#endif
#endif /* TAROK_B200_H */
