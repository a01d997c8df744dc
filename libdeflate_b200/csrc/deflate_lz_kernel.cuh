// deflate_lz_kernel.cuh -- LZ77 match finding + parsing + Huffman block encoding, sm_100a.
// Included by deflate_kernel.cu.
//
// Reference behaviour covered (what, not how):
//   hash-chain match finder            lib/hc_matchfinder.h:182-399, lib/matchfinder_common.h:168-222
//   greedy / lazy parsing              lib/deflate_compress.c:2529-2808
//   Huffman code construction          lib/deflate_compress.c:847-1396
//   block cost comparison + emission   lib/deflate_compress.c:1483-2038
// The output is a valid DEFLATE stream with a ratio close to the reference's at the
// same level, never the reference's bytes (libdeflate.h:76-83 makes no such promise).
//
// B200 mapping: one persistent CTA (1024 threads) per chunk; everything a chunk needs
// lives in shared memory (~224 KiB):
//   * a 64 KiB ring of the input (the sliding window), filled 16 KiB at a time by the
//     TMA bulk-copy engine (cp.async.bulk + mbarrier) -- the window never touches
//     HBM again,
//   * 13-bit hash heads (u16[8192]) and a chain table with one slot per position
//     mod 65536 (u16[65536]); a pass is 16 Ki positions and the window 32 Ki, so the
//     16 Ki slots of the FOLLOWING pass are always dead and serve as scratch,
//   * per pass of 16 Ki positions:
//       - ordered chain insertion by the whole CTA: a stable multisplit of the positions
//         by hash slice, then one warp per slice links its list (lz_insert_pass_par),
//       - guided search: every thread walks dynamically assigned runs of 16 or 32
//         positions like the reference's lazy parser, but every position ends up with a
//         (length, distance), which is what lets the parse itself be parallel,
//       - exact parallel lazy parse: per-window pointer jumping gives "where does a
//         parse entering at lane e leave this 32-position window" for all e at once,
//         the windows are chained group-parallel, __reduce_or_sync marks the visited
//         positions, a prefix sum places the tokens,
//   * tokens and per-position results go to a per-CTA buffer in global memory (L2
//     resident), symbol histograms stay in shared memory,
//   * per block (32 KiB of input): Huffman codes (length-limited to 15; parallel except
//     for the two-queue merge), exact bit cost of dynamic / static / stored (the
//     reference's three-way choice, which is also what makes
//     libdeflate_*_compress_bound() hold), then a two-pass emission: per-token bit
//     lengths -> block-wide exclusive prefix sum -> every thread ORs its codewords
//     into a shared-memory staging buffer -> coalesced stores,
//   * levels 10-12: all matches per position + iterated min-cost-path DP (see below).
//
// Algorithmic HBM bytes per chunk: in_nbytes (read once) + out_nbytes (written once).
#pragma once

#ifndef LZ_THREADS
#define LZ_THREADS   1024
#endif
#define LZ_WARPS     (LZ_THREADS / 32)
#define LZ_PASS      16384			// positions matched + parsed per pass
#define LZ_BLOCK_PASSES 2			// passes per DEFLATE block (32 KiB of input)
#define LZ_NWIN      (LZ_PASS / 32)
// Levels 1-9 run two warp groups: the search group (warps [0, LZ_A_WARPS)) loads, inserts and searches
// pass after pass; the encode group (the other warps) parses each searched pass and encodes the blocks,
// one pass behind.  -DLZ_PIPELINE=0 runs both halves on the whole CTA, one after the other (the serial
// schedule, which levels 10-12 always use).  Both schedules produce the same stream.
#ifndef LZ_PIPELINE
#define LZ_PIPELINE  1
#endif
#ifndef LZ_A_WARPS
#define LZ_A_WARPS   22
#endif
#define LZ_B_WARPS   (LZ_WARPS - LZ_A_WARPS)
#define LZ_BAR_A     1			// named barriers: the search group,
#define LZ_BAR_B     2			//   the encode group,
#define LZ_BAR_FULL  3			//   "pass s searched" (3 + s % 2, search group arrives, encode group waits)
#define LZ_BAR_EMPTY 5			//   "pass s released" (5 + s % 2, encode group arrives, search group waits)
#ifndef LZ_QUANTUM
#define LZ_QUANTUM   0			// > 0: chain steps per loop trip of the resumable search (experiment)
#endif
#define LZ_SEG       16384			// largest single TMA load
#define LZ_RING      65536
#define LZ_HASH_BITS 13
#define LZ_WIN       32768
#define LZ_LOOKAHEAD 512			// bytes past the pass kept in the ring (>= 258 + 8)
#define LZ_MAX_DIST  (LZ_WIN - LZ_LOOKAHEAD)	// the oldest LOOKAHEAD bytes of the window are overwritten
#define LZ_TOKCAP    (LZ_BLOCK_PASSES * LZ_PASS + 64)
#define LZ_STAGE_WORDS 2048			// 8 KiB emission staging
#define LZ_TPT_MAX     3			// tokens per thread per emission round: LZ_THREADS / (threads encoding),
					// so a round is <= 1024 tokens of <= 48 bits (<= 1536 staging words)

// shared memory layout
#define LZ_SM_RING   0
#define LZ_SM_NEXT   (LZ_SM_RING + LZ_RING)			// u16[65536], indexed by pos mod 65536
#define LZ_SM_HEAD   (LZ_SM_NEXT + 2 * 65536)			// u16[1 << HASH_BITS]
#define LZ_SM_R      (LZ_SM_HEAD + 2 * (1 << LZ_HASH_BITS))	// 12 KiB multi-purpose region:
#define LZ_SM_VIS    (LZ_SM_R)					//   parse: u32[NWIN] visited masks
#define LZ_SM_TOKOFF (LZ_SM_R + 4096)				//   parse: u32[NWIN + 16] token offsets
#define LZ_SM_ENTRY  (LZ_SM_R + 8320)				//   parse: u8[NWIN] entry lane per window
#define LZ_SM_ESCAN  (LZ_SM_R + 9344)				//   emission: scan scratch u32[80]
#define LZ_SM_GEXIT  (LZ_SM_R + 9728)				//   parse: u16[WARPS * 32] group exits
#define LZ_SM_GENTRY (LZ_SM_R + 11776)				//   parse: u32[WARPS] group entries (WARPS <= 32)
#define LZ_SM_ITEMS  (LZ_SM_R + 12288)				// u16[512] precode items
#define LZ_SM_FREQ   (LZ_SM_ITEMS + 1024)			// u32[288 + 32]
#define LZ_SM_LENS   (LZ_SM_FREQ + 4 * 320)			// u8[320]
#define LZ_SM_CODES  (LZ_SM_LENS + 320)				// u16[320]
#define LZ_SM_VARS   (LZ_SM_CODES + 2 * 320)			// misc scalars, mbarrier
#define LZ_SM_CMAT   (LZ_SM_VARS + 256)				// u32[A_WARPS * 16 + 32] insertion counts of the search group
#define LZ_SM_BYTES  (LZ_SM_CMAT + 4 * (LZ_A_WARPS * 16 + 32))	//   (pipelined; region R is the encode group's then)
static_assert(LZ_SM_BYTES <= 227 * 1024, "shared memory of one CTA");
static_assert(LZ_A_WARPS >= 16 && LZ_B_WARPS * 32 >= 320 && LZ_THREADS / (LZ_B_WARPS * 32) <= LZ_TPT_MAX,
	      "search group: >= one warp per hash slice; encode group: one thread per litlen+offset symbol");

// per-CTA global scratch (L2 resident): per-position results of the current pass + tokens
#define LZ_BLOCK_POS (LZ_BLOCK_PASSES * LZ_PASS)		// positions per block
#define LZ_OPT_K     8					// matches kept per position (levels 10-12)
#define LZ_DP_SEG    2048				// positions per independent DP segment (one warp each)
#define LZ_GS_RES    0						// u32[BLOCK_POS]  block-relative
#define LZ_GS_TOK    (LZ_GS_RES + 4 * LZ_BLOCK_POS)		// u32[TOKCAP]
#define LZ_GS_COST   (LZ_GS_TOK + 4 * LZ_TOKCAP)		// u32[BLOCK_POS + 320]   (levels 10-12)
#define LZ_GS_MLIST  (LZ_GS_COST + 4 * (LZ_BLOCK_POS + 320))	// u32[BLOCK_POS * K]     (levels 10-12)
#define LZ_GS_BYTES  (LZ_GS_MLIST + 4 * LZ_BLOCK_POS * LZ_OPT_K)
#define LZ_GS_EXIT   LZ_GS_MLIST				// u16[PASS] parse exits (pipelined; levels 1-9 keep no match lists)
#define LZ_FAR4_DIST  1024				// text-like input: a 4-byte match further away than this is coded as literals
#define LZ_COST_INF  0x3fffffu				// fits the 23-bit cost field of the DP reduction key

struct lz_vars {
	unsigned long long mbar;
	u32 chunk;
	u32 tok_count;		// tokens in the current block
	u32 parse_entry;	// absolute position where the parser continues
	u32 cost_dyn, cost_static, extra_bits;
	u32 hlit, hdist, hclen;
	u32 n_items;
	u32 run_counter;	// next unassigned search run of the current pass
	u32 min_len;		// shortest match worth taking (depends on the alphabet size)
	u32 far4_dist;		// 4-byte matches further away than this are coded as literals
	u32 used_lits[8];	// 256-bit set of byte values seen in the first 4 KiB
	u32 carry;		// partial output word at bit position obit (persists between flushes)
	u32 nused_lit, nused_off;
	u32 huff_over;		// a Huffman code exceeded 15 bits and was capped
	u32 obs_blk[8], obs_next[8];	// byte-class observations: current block / the pass after it
	u32 end_early;		// the next pass looks different: end the block before it
	u32 failed;
	u32 obit_lo, obit_hi;	// output bit position (64-bit)
	u32 pre_lens_packed[3];
	u32 tma_phase;
	u32 slot_chunk[2], slot_b0[2], slot_min_len[2], slot_far4[2];	// pass s handed to the encode group: slot s % 2
};
static_assert(sizeof(lz_vars) <= 256, "LZ_SM_VARS");
#define LZ_NO_CHUNK  0xffffffffu		// slot_chunk of the pass after the last one

// A warp group: thread / warp index inside the group, its size, and its barrier (0: the whole CTA).
struct lz_grp {
	u32 t, w, nt, nw, bar;
};
#ifdef LDB_EMU
// bar.sync / bar.arrive for the emulator build: a barrier completes when 'nthreads' threads have arrived.
// The emulator runs all threads of a block on one host thread (and one block at a time on it), and a
// completed barrier is back at 0 arrivals, so per-host-thread state needs no reset between blocks.
inline void lz_emu_named_barrier(u32 id, u32 nthreads, bool wait)
{
	static thread_local struct { u32 arrived, gen; } bars[16];
	auto &b = bars[id & 15];
	const u32 gen = b.gen;
	if (++b.arrived == nthreads) {
		b.arrived = 0;
		b.gen++;
		emu::tl_block->spins = 0;
	} else if (wait) {
		while (b.gen == gen) emu::yield();
	}
}
#endif
__device__ __forceinline__ void lz_bar_sync(u32 id, u32 nthreads)
{
#ifdef LDB_EMU
	if (id == 0) __syncthreads();
	else lz_emu_named_barrier(id, nthreads, true);
#else
	asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
#endif
}
__device__ __forceinline__ void lz_bar_arrive(u32 id, u32 nthreads)
{
#ifdef LDB_EMU
	lz_emu_named_barrier(id, nthreads, false);
#else
	asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
#endif
}
__device__ __forceinline__ void lz_sync(const lz_grp &gp) { lz_bar_sync(gp.bar, gp.nt); }

struct lz_params {
	int depth, nice, lazy;
	int opt_iters;	// > 0: near-optimal parsing (levels 10-12): passes of min-cost-path + cost-model update
};

__device__ __forceinline__ lz_params lz_level_params(int level)
{
	// level -> (max chain depth, nice length, lazy evaluation); cf. the reference's table
	// lib/deflate_compress.c:3927-4013 (depth/nice per level; values here are ours)
	switch (level) {
	case 1: return {2, 16, 0, 0};
	case 2: return {4, 24, 0, 0};
	case 3: return {8, 32, 0, 0};
	case 4: return {12, 48, 0, 0};
	case 5: return {12, 48, 1, 0};
#ifndef LZ_L6_DEPTH
#define LZ_L6_DEPTH 24
#endif
	case 6: return {LZ_L6_DEPTH, 96, 1, 0};
	case 7: return {48, 160, 1, 0};
	case 8: return {96, 258, 2, 0};		// lazy2: one more position of lookahead (ref: deflate_compress.c:2742-2776)
	case 9: return {200, 258, 2, 0};
	// near-optimal levels (ref: lib/deflate_compress.c:3972-4012: depth 35/100/300, passes 2/4/10)
	case 10: return {48, 96, 1, 2};
	case 11: return {96, 160, 1, 3};
	default: return {200, 258, 1, 5};
	}
}

// Shortest match length worth emitting, from the number of distinct byte values at the start
// of the input (few distinct literals => literals are cheap => short matches do not pay) and
// the search depth (shallow searches find worse matches, so be less picky).  Same heuristic as
// the reference's choose_min_match_len (lib/deflate_compress.c:2296-2326), restated as
// thresholds; our match finder starts at length 4.
__device__ __forceinline__ u32 lz_choose_min_len(u32 num_used_literals, u32 depth)
{
	u32 m;
	if (num_used_literals < 6) m = 9;
	else if (num_used_literals < 8) m = 8;
	else if (num_used_literals < 10) m = 7;
	else if (num_used_literals < 16) m = 6;
	else if (num_used_literals < 45) m = 5;
	else m = 4;
	if (depth < 16) {
		u32 cap = depth < 5 ? 4 : (depth < 10 ? 5 : 7);
		if (m > cap) m = cap;
	}
	return m;
}

// ---- ring access ------------------------------------------------------------------
__device__ __forceinline__ u32 lz_ld32(const u8 *ring, u32 pos)
{
	u32 a = pos & (LZ_RING - 1);
	const u32 *w = (const u32 *)ring;
	u32 lo = w[a >> 2];
	u32 hi = w[((a + 4) & (LZ_RING - 1)) >> 2];
	return __funnelshift_r(lo, hi, (a & 3) * 8);
}
__device__ __forceinline__ u32 lz_ld8(const u8 *ring, u32 pos) { return ring[pos & (LZ_RING - 1)]; }
__device__ __forceinline__ u32 lz_hash(u32 v) { return (v * 0x1E35A7BDu) >> (32 - LZ_HASH_BITS); }	// ref: matchfinder_common.h:168-172

// ---- TMA bulk load of one segment into the ring -------------------------------------
__device__ __forceinline__ void lz_load_segment(u8 *sm, lz_vars *v, const u8 *in, u32 from, u32 to, const lz_grp &gp)
{
	u8 *ring = sm + LZ_SM_RING;
	u32 len = to - from;
	u32 bulk = (((uintptr_t)(in + from) & 15) == 0) ? (len & ~15u) : 0;
	lz_sync(gp);	// every earlier generic-proxy access to the slots being overwritten is done
#ifndef LDB_EMU
	if (bulk) {
		u32 mbar = (u32)__cvta_generic_to_shared(&v->mbar);
		if (gp.t == 0) {
			u32 dst = (u32)__cvta_generic_to_shared(ring + (from & (LZ_RING - 1)));
			asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
			asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(mbar), "r"(bulk) : "memory");
			asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
				     ::"r"(dst), "l"(in + from), "r"(bulk), "r"(mbar) : "memory");
		}
		u32 phase = v->tma_phase;
		u32 done = 0;
		while (!done) {
			asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
				     : "=r"(done) : "r"(mbar), "r"(phase) : "memory");
		}
	}
#else
	for (u32 i = gp.t; i < bulk; i += gp.nt) ring[(from + i) & (LZ_RING - 1)] = in[from + i];
#endif
	for (u32 i = bulk + gp.t; i < len; i += gp.nt) ring[(from + i) & (LZ_RING - 1)] = in[from + i];
	lz_sync(gp);
	if (bulk && gp.t == 0) v->tma_phase ^= 1;
	lz_sync(gp);
}

// ---- length / offset slot helpers (Appendix A; ref: deflate_compress.c:237-308) ------
__device__ __forceinline__ u32 lz_len_slot(u32 len)	// len 3..258 -> 0..28
{
	if (len < 11) return len - 3;
	if (len == 258) return 28;
	u32 l = len - 3;
	u32 eb = 29 - __clz(l);		// l in [8,254]: eb = floor(log2 l) - 2
	return 4 * eb + 4 + ((l >> eb) & 3);
}
__device__ __forceinline__ u32 lz_len_extra_bits(u32 slot) { return (slot < 8 || slot == 28) ? 0 : (slot - 4) >> 2; }
__device__ __forceinline__ u32 lz_len_base(u32 slot) { return slot < 8 ? 3 + slot : (slot == 28 ? 258 : 3 + ((4 + (slot & 3)) << ((slot - 4) >> 2))); }
__device__ __forceinline__ u32 lz_off_slot(u32 off)	// off 1..32768 -> 0..29
{
	if (off < 5) return off - 1;
	u32 o = off - 1;
	u32 eb = 30 - __clz(o);		// o >= 4: eb = floor(log2 o) - 1
	return 2 * eb + 2 + ((o >> eb) & 1);
}
__device__ __forceinline__ u32 lz_off_extra_bits(u32 slot) { return slot < 4 ? 0 : (slot - 2) >> 1; }
__device__ __forceinline__ u32 lz_off_base(u32 slot) { return slot < 4 ? 1 + slot : 1 + ((2 + (slot & 1)) << ((slot - 2) >> 1)); }

__device__ __forceinline__ u32 lz_static_litlen_len(u32 sym) { return sym < 144 ? 8 : (sym < 256 ? 9 : (sym < 280 ? 7 : 8)); }

// ---- output bit staging ----------------------------------------------------------------
// The stream is assembled in 32-bit words relative to the START of the chunk's output
// buffer.  stage[0] is the word containing bit position 'obit' rounded down.
struct lz_out {
	u8 *out;
	size_t avail;
	u64 obit;		// bits emitted so far (from the start of 'out', wrapper header included)
};

__device__ __forceinline__ void lz_stage_or(u32 *stage, u32 rel_bit, u64 bits, u32 nbits)
{
	if (!nbits) return;
	u32 w = rel_bit >> 5, sh = rel_bit & 31;
	atomicOr(&stage[w], (u32)(bits << sh));
	if (sh + nbits > 32) {
		u64 rest = bits >> (32 - sh);
		atomicOr(&stage[w + 1], (u32)rest);
		if (sh + nbits > 64) atomicOr(&stage[w + 2], (u32)(rest >> 32));
	}
}

// Writes staging words [0, nwords) to the output at word index 'first_word'; all threads.
__device__ __forceinline__ void lz_flush_words(const lz_out &o, const u32 *stage, u64 first_word, u32 nwords, const lz_grp &gp)
{
	if ((((uintptr_t)o.out) & 3) == 0) {
		u32 *dst = (u32 *)o.out + first_word;
		for (u32 i = gp.t; i < nwords; i += gp.nt) dst[i] = stage[i];
	} else {
		u8 *dst = o.out + first_word * 4;
		for (u32 i = gp.t; i < nwords * 4; i += gp.nt) dst[i] = (u8)(stage[i >> 2] >> (8 * (i & 3)));
	}
}

// ---- Huffman code construction ---------------------------------------------------------
// (ref for the length-limiting idea: deflate_compress.c:1023-1091; at least two codewords like
// deflate_compress.c:1369-1378; the parallel parts live in the kernel's build_codes step)
// Two-queue Huffman merge only (one thread): leaves nodefreq[0, nused) ascending, internal nodes
// appended behind them; writes parent[] for every node but the root.  The two queue heads and their
// successors are kept in registers so that a shared-memory load is never waited for directly.
__device__ __forceinline__ void lz_huffman_merge(u32 *nodefreq, u16 *parent, u32 nused)
{
	const u32 INF = 0xffffffffu;
	u32 leaf = 0, inode = nused, nn = nused;
	u32 l0 = nodefreq[0], l1 = nused > 1 ? nodefreq[1] : INF;	// leaf queue: head, next
	u32 n0 = INF, n1 = INF;						// internal queue: head, next
	while (nn < 2 * nused - 1) {
		u32 a, b, fa, fb;
		if (l0 <= n0) { a = leaf++; fa = l0; l0 = l1; l1 = leaf + 1 < nused ? nodefreq[leaf + 1] : INF; }
		else { a = inode++; fa = n0; n0 = n1; n1 = INF; }
		if (n0 == INF && inode < nn) n0 = nodefreq[inode];
		if (l0 <= n0) { b = leaf++; fb = l0; l0 = l1; l1 = leaf + 1 < nused ? nodefreq[leaf + 1] : INF; }
		else { b = inode++; fb = n0; n0 = n1; n1 = INF; }
		const u32 sum = fa + fb;
		nodefreq[nn] = sum;
		parent[a] = (u16)nn;
		parent[b] = (u16)nn;
		nn++;
		// refill the register copies of the internal queue (the new node may be its head)
		if (n0 == INF && inode < nn) n0 = inode == nn - 1 ? sum : nodefreq[inode];
		if (n1 == INF && inode + 1 < nn) n1 = inode + 1 == nn - 1 ? sum : nodefreq[inode + 1];
	}
}

// canonical, bit-reversed codewords for an alphabet (all threads participate on disjoint syms)
__device__ __forceinline__ void lz_gen_codes_serial(const u8 *lens, u32 nsyms, u16 *codes)
{
	u32 cnt[16];
	for (u32 l = 0; l < 16; l++) cnt[l] = 0;
	for (u32 s = 0; s < nsyms; s++) cnt[lens[s]]++;
	u32 next[16];
	u32 code = 0;
	cnt[0] = 0;
	for (u32 l = 1; l < 16; l++) {
		next[l] = code;
		code = (code + cnt[l]) << 1;
	}
	for (u32 s = 0; s < nsyms; s++) {
		u32 l = lens[s];
		codes[s] = l ? (u16)(__brev(next[l]++) >> (32 - l)) : 0;
	}
}

#ifdef LZ_TIMING
#include <stdio.h>
// tuning builds only: cycles per phase, summed over all CTAs (thread 0's clock between barriers;
// the compiler may read the clock before the barrier wait, so a phase in which thread 0 finishes early
// is under-counted and the wait shows up in the next one: read 'search phase' + 'parse e1' together)
__device__ unsigned long long ldb_lz_timing[16];
#define LZ_T(k) do { if (tlead) { long long t_ = clock64(); tacc[k] += t_ - tlast; tlast = t_; } } while (0)
#else
#define LZ_T(k) do { } while (0)
#endif

// Lanes holding the same NBITS-bit key, from NBITS ballots (__match_any_sync gives the same mask
// but takes several hundred cycles when most keys are distinct, which is the common case here).
template <int NBITS>
__device__ __forceinline__ u32 lz_same_key_mask(u32 key, bool valid)
{
	u32 m = __ballot_sync(LDB_FULL_MASK, valid);
#pragma unroll
	for (int b = 0; b < NBITS; b++) {
		const u32 bal = __ballot_sync(LDB_FULL_MASK, (key >> b) & 1);
		m &= ((key >> b) & 1) ? bal : ~bal;
	}
	return m;
}

// ---- ordered hash-chain insertion of one pass by the whole CTA -------------------------------
// Chains must link every position to the previous one with the same hash, so insertion is ordered
// -- but only within a hash value.  The head table is cut into NSL (16 or 32) slices by the top hash bits
// and the pass is split stably by slice (a multisplit), after which one warp per slice links it:
//  (1) warp w hashes its contiguous range of tiles, parks each hash in the position's own next[]
//      slot (dead until the link is written) and counts its positions per slice;
//  (2) a 2-D exclusive scan of the (warp, slice) counts gives every warp its write cursor in every
//      slice list; the lists are packed into the 16 Ki next[] slots of the FOLLOWING pass, which
//      belong to positions more than 48 Ki back -- outside every search window;
//  (3) warp w re-walks its tiles in order and scatters the positions (rank inside a tile from
//      the same-slice lane mask): every list ends up sorted by position;
//  (4) warp s links list s, 32 entries at a time: predecessors inside the batch come from
//      the same-hash lane mask, the others from head[].  Same links as a serial insertion.
template <u32 NW>	// warps of the group (gp.nw)
__device__ __forceinline__ void lz_insert_pass_par(const u8 *ring, u16 *head, u16 *nextt, u32 *cmat,
						   u32 b0, u32 pend, u32 n, const lz_grp &gp, u32 lane
#ifdef LZ_TIMING
						   , long long *tacc, long long &tlast
#endif
						   )
{
	constexpr u32 NSL_BITS = NW >= 32 ? 5 : 4, NSL = 1u << NSL_BITS;	// hash slices = linking warps
	static_assert(NW >= NSL && (NW * NSL + 2 * NSL) * 4 <= 8192, "one linking warp per slice");
	const u32 tid = gp.t, warp = gp.w;
#ifdef LZ_TIMING
	const bool tlead = tid == 0;
#endif
	u32 *sbase = cmat + NW * NSL, *stot = sbase + NSL;
	const u32 lt = (1u << lane) - 1;
	const u32 LB = (b0 + LZ_PASS) & 0xffff;
	const u32 ntiles = (pend - b0 + 31) >> 5, tpw = (ntiles + NW - 1) / NW;
	const u32 r0 = b0 + warp * tpw * 32;
	const u32 r1 = r0 + tpw * 32 < pend ? r0 + tpw * 32 : pend;
	for (u32 i = tid; i < NW * NSL + 2 * NSL; i += 32 * NW) cmat[i] = 0;
	lz_sync(gp);
	for (u32 p = r0 + lane; p < r1; p += 32) {
		const u32 hv = p + 4 <= n ? lz_hash(lz_ld32(ring, p)) : 0xffffu;
		nextt[p & 0xffff] = (u16)hv;
		if (hv != 0xffffu) atomicAdd(&cmat[warp * NSL + (hv >> (LZ_HASH_BITS - NSL_BITS))], 1u);
	}
	lz_sync(gp);
	LZ_T(12);	// insertion: hashing
	if (warp == 0) {
		u32 run = 0;
		if (lane < NSL)
			for (u32 w = 0; w < NW; w++) {
				const u32 c = cmat[w * NSL + lane];
				cmat[w * NSL + lane] = run;
				run += c;
			}
		u32 incl = run;
		for (int o2 = 1; o2 < NSL; o2 <<= 1) {
			const u32 t = __shfl_up_sync(LDB_FULL_MASK, incl, o2);
			if (lane >= (u32)o2) incl += t;
		}
		if (lane < NSL) { sbase[lane] = incl - run; stot[lane] = run; }
	}
	lz_sync(gp);
	for (u32 t = 0; t < tpw; t++) {
		const u32 p = r0 + 32 * t + lane;
		const u32 hv = p < r1 ? nextt[p & 0xffff] : 0xffffu;
		const bool valid = hv != 0xffffu;
		const u32 sl = hv >> (LZ_HASH_BITS - NSL_BITS);
		const u32 m = lz_same_key_mask<NSL_BITS>(sl, valid);
		const u32 cur = valid ? cmat[warp * NSL + sl] : 0;
		__syncwarp();
		if (valid) {
			nextt[LB + sbase[sl] + cur + __popc(m & lt)] = (u16)p;
			if ((m & lt) == 0) cmat[warp * NSL + sl] = cur + __popc(m);
		}
		__syncwarp();
	}
	lz_sync(gp);
	LZ_T(13);	// insertion: slice lists
	if (warp < NSL) {
		const u32 cnt = stot[warp];
		const u16 *mylist = nextt + LB + sbase[warp];
		u32 p16n = lane < cnt ? mylist[lane] : 0;
		u32 hn = lane < cnt ? nextt[p16n] : 0;
		for (u32 b = 0; b < cnt; b += 32) {
			const bool valid = b + lane < cnt;
			const u32 p16 = p16n;
			const u32 h = valid ? hn : 0;
			if (b + 32 + lane < cnt) {		// next batch: list entry and parked hash
				p16n = mylist[b + 32 + lane];
				hn = nextt[p16n];
			}
			const u32 old_head = valid ? head[h] : 0;
			const u32 m = lz_same_key_mask<LZ_HASH_BITS - NSL_BITS>(h, valid);	// (the slice bits are equal anyway)
			const u32 below = m & lt;
			const u32 prev = __shfl_sync(LDB_FULL_MASK, p16, below ? 31 - __clz(below) : 0);
			if (valid) {
				nextt[p16] = (u16)(below ? prev : old_head);
				if ((m >> lane) == 1) head[h] = (u16)p16;	// newest position of its hash in this batch
			}
			__syncwarp();
		}
	}
	lz_sync(gp);
}

// ---- one chain search (ref: hc_matchfinder.h:182-338) ------------------------------------------
// Walks the hash chain of position p (newest first, at most 'depth' candidates within
// LZ_MAX_DIST) and returns the longest match; (best_len, best_dist) may come in pre-seeded with
// a match carried over from position p-1.  Candidates are filtered by one byte just past the
// current best, then its last 4 bytes (hc_matchfinder.h:301-304), then the first 4.
__device__ __forceinline__ void lz_search(const u8 *ring, const u16 *nextt, u32 p, u32 n, int depth, u32 nice_level,
					   u32 &best_len, u32 &best_dist)
{
	const u32 max_len = n - p < 258 ? n - p : 258;
	const u32 nice = nice_level < max_len ? nice_level : max_len;
	if (best_len) {
		// a carried-over match may continue past where its predecessor was capped
		while (best_len < max_len && lz_ld8(ring, p + best_len) == lz_ld8(ring, p - best_dist + best_len)) best_len++;
	}
	if (best_len >= nice) return;
	const u32 cur = lz_ld32(ring, p);
	u32 tailo = best_len >= 4 ? best_len - 3 : 0;
	u32 tailv = tailo ? lz_ld32(ring, p + tailo) : cur;
	const u32 lim = p < LZ_MAX_DIST ? p : LZ_MAX_DIST;
	u32 cand = nextt[p & 0xffff];
	u32 prev_dist = 0;
	for (int d = 0; d < depth; d++) {
		const u32 dist = (p - cand) & 0xffff;
		if (dist - 1 >= lim || dist <= prev_dist) break;
		prev_dist = dist;
		const u32 cq = cand;			// ring index of the candidate (positions are stored mod 65536)
		cand = nextt[cq];
		if (lz_ld8(ring, cq + tailo + 3) != (tailv >> 24)) continue;
		if (lz_ld32(ring, cq + tailo) != tailv) continue;
		if (tailo && lz_ld32(ring, cq) != cur) continue;
		u32 len = 4;
		while (len + 4 <= max_len) {
			u32 x = lz_ld32(ring, p + len) ^ lz_ld32(ring, cq + len);
			if (x) { len += (__ffs(x) - 1) >> 3; goto extended; }
			len += 4;
		}
		while (len < max_len && lz_ld8(ring, p + len) == lz_ld8(ring, cq + len)) len++;
	extended:
		if (len > best_len) {
			best_len = len;
			best_dist = dist;
			if (len >= nice) break;
			tailo = len - 3;
			tailv = lz_ld32(ring, p + tailo);
		}
	}
}

// ---- the same search, resumable: a walk is set up once and advanced a few chain steps at a time, so that
// a lane with a deep chain does not hold back the lanes of its warp that are already done (LZ_QUANTUM > 0)
struct lz_walk {
	u32 cand, prev_dist, best_len, best_dist, tailo, tailv, cur;
	int left;		// chain steps this search may still take (0: finished)
};

__device__ __forceinline__ void lz_walk_setup(const u8 *ring, const u16 *nextt, u32 p, u32 n, int depth, u32 nice_level,
					       u32 L, u32 D, lz_walk &w)
{
	const u32 max_len = n - p < 258 ? n - p : 258;
	const u32 nice = nice_level < max_len ? nice_level : max_len;
	w.best_len = L;
	w.best_dist = D;
	if (w.best_len)
		while (w.best_len < max_len && lz_ld8(ring, p + w.best_len) == lz_ld8(ring, p - w.best_dist + w.best_len)) w.best_len++;
	w.left = w.best_len >= nice ? 0 : depth;
	w.cur = lz_ld32(ring, p);
	w.tailo = w.best_len >= 4 ? w.best_len - 3 : 0;
	w.tailv = w.tailo ? lz_ld32(ring, p + w.tailo) : w.cur;
	w.cand = nextt[p & 0xffff];
	w.prev_dist = 0;
}

__device__ __forceinline__ void lz_walk_steps(const u8 *ring, const u16 *nextt, u32 p, u32 n, u32 nice_level, lz_walk &w, int quantum)
{
	const u32 max_len = n - p < 258 ? n - p : 258;
	const u32 nice = nice_level < max_len ? nice_level : max_len;
	const u32 lim = p < LZ_MAX_DIST ? p : LZ_MAX_DIST;
	for (int q = 0; q < quantum && w.left > 0; q++) {
		const u32 dist = (p - w.cand) & 0xffff;
		if (dist - 1 >= lim || dist <= w.prev_dist) { w.left = 0; break; }
		w.left--;
		w.prev_dist = dist;
		const u32 cq = w.cand;
		w.cand = nextt[cq];
		if (lz_ld8(ring, cq + w.tailo + 3) != (w.tailv >> 24)) continue;
		if (lz_ld32(ring, cq + w.tailo) != w.tailv) continue;
		if (w.tailo && lz_ld32(ring, cq) != w.cur) continue;
		u32 len = 4;
		while (len + 4 <= max_len) {
			u32 x = lz_ld32(ring, p + len) ^ lz_ld32(ring, cq + len);
			if (x) { len += (__ffs(x) - 1) >> 3; goto extended; }
			len += 4;
		}
		while (len < max_len && lz_ld8(ring, p + len) == lz_ld8(ring, cq + len)) len++;
	extended:
		if (len > w.best_len) {
			w.best_len = len;
			w.best_dist = dist;
			if (len >= nice) { w.left = 0; break; }
			w.tailo = len - 3;
			w.tailv = lz_ld32(ring, p + w.tailo);
		}
	}
}

// ---- all-matches search for the near-optimal levels (stands in for bt_matchfinder_get_matches,
// lib/bt_matchfinder.h:296: "matches of strictly increasing length", here read off the hash chain:
// every improvement met while walking newest-to-oldest is a longer match at a larger distance,
// i.e. the Pareto front the min-cost-path pass needs).  Up to LZ_OPT_K are kept (the first K-1 and
// the longest).  Entry format: len << 16 | (dist - 1); 0 terminates.
__device__ __forceinline__ void lz_search_all(const u8 *ring, const u16 *nextt, u32 p, u32 n, int depth, u32 nice_level,
					       u32 *ml, u32 &best_len, u32 &best_dist)
{
	const u32 max_len = n - p < 258 ? n - p : 258;
	const u32 nice = nice_level < max_len ? nice_level : max_len;
	const u32 cur = lz_ld32(ring, p);
	u32 tailo = 0, tailv = cur, cnt = 0;
	best_len = 0;
	best_dist = 0;
	const u32 lim = p < LZ_MAX_DIST ? p : LZ_MAX_DIST;
	u32 cand = nextt[p & 0xffff];
	u32 prev_dist = 0;
	for (int d = 0; d < depth; d++) {
		const u32 dist = (p - cand) & 0xffff;
		if (dist - 1 >= lim || dist <= prev_dist) break;
		prev_dist = dist;
		const u32 cq = cand;
		cand = nextt[cq];
		if (lz_ld8(ring, cq + tailo + 3) != (tailv >> 24)) continue;
		if (lz_ld32(ring, cq + tailo) != tailv) continue;
		if (tailo && lz_ld32(ring, cq) != cur) continue;
		u32 len = 4;
		while (len + 4 <= max_len) {
			u32 x = lz_ld32(ring, p + len) ^ lz_ld32(ring, cq + len);
			if (x) { len += (__ffs(x) - 1) >> 3; goto extended; }
			len += 4;
		}
		while (len < max_len && lz_ld8(ring, p + len) == lz_ld8(ring, cq + len)) len++;
	extended:
		if (len > best_len) {
			best_len = len;
			best_dist = dist;
			ml[cnt < LZ_OPT_K ? cnt : LZ_OPT_K - 1] = (len << 16) | (dist - 1);
			cnt++;
			if (len >= nice) break;
			tailo = len - 3;
			tailv = lz_ld32(ring, p + tailo);
		}
	}
	for (u32 k = cnt; k < LZ_OPT_K; k++) ml[k] = 0;
}

// ---- min-cost path over one DP segment, executed by ONE warp (ref: deflate_find_min_cost_path,
// lib/deflate_compress.c:3328-3399).  Block-relative positions [s0, s1), processed backwards:
//   C[i] = min( lit_cost(byte_i) + C[i+1],  min over lengths L offered by the matches at i of
//               len_cost(L) + off_cost(closest match of length >= L) + C[i+L] )
// Lane k keeps C[i+1+k] in a register (the window slides by one shuffle per position), so the
// 32 shortest candidate lengths need no memory at all; longer ones read the cost array.  A path
// never crosses s1 (segments are independent; the price is one constrained token per 2048
// positions).  The decision is written as a (length | flag, distance) pair the parallel parser
// then follows: res = L | (dist-1 | 0x8000) << 16 (0 for a literal).
__device__ void lz_dp_segment(const u8 *ring, const u32 *mlist, u32 *costg, u32 *res, const u8 *costtab,
			      u32 block_begin, u32 s0, u32 s1, u32 lane)
{
	const u8 *litc = costtab, *lenc = costtab + 256, *offc = costtab + 256 + 259;
	u32 wc = lane == 0 ? 0 : LZ_COST_INF;
	u32 i = s1;
	// tile of 4 positions x 8 match entries, one coalesced 128-byte load, fetched one tile ahead
	auto load_tile = [&](u32 top) -> u32 {
		// lane -> (q = lane >> 3: position top-1-q, j = lane & 7: entry)
		u32 q = lane >> 3;
		if (top < q + 1 || top - 1 - q < s0) return 0;
		return mlist[(size_t)(top - 1 - q) * LZ_OPT_K + (lane & 7)];
	};
	u32 nxt = load_tile(i);
	while (i > s0) {
		const u32 curt = nxt;
		nxt = i >= 4 ? load_tile(i - 4) : 0;
#pragma unroll
		for (int q = 0; q < 4; q++) {
			if (i < (u32)q + 1 || i - 1 - q < s0) break;
			const u32 pos = i - 1 - q;
			u32 m[LZ_OPT_K];
#pragma unroll
			for (int j = 0; j < LZ_OPT_K; j++) m[j] = __shfl_sync(LDB_FULL_MASK, curt, q * 8 + j);
			u32 Lmax = 0;
#pragma unroll
			for (int j = 0; j < LZ_OPT_K; j++)
				if (m[j]) Lmax = m[j] >> 16;
			const u32 cap = s1 - pos;
			if (Lmax > cap) Lmax = cap;
			const u32 byte = ring[(block_begin + pos) & (LZ_RING - 1)];
			// distance of the closest match offering length L (entries have increasing length)
			auto dist_for = [&](u32 L) -> u32 {
				u32 d = 0;
#pragma unroll
				for (int j = LZ_OPT_K - 1; j >= 0; j--)
					if (m[j] && (m[j] >> 16) >= L) d = (m[j] & 0xffff) + 1;
				return d;
			};
			u32 key;
			{
				const u32 L = lane + 1;
				u32 cand = LZ_COST_INF;
				if (lane == 0) cand = wc + litc[byte];
				else if (L >= 4 && L <= Lmax) cand = wc + lenc[L] + offc[lz_off_slot(dist_for(L))];
				if (cand > LZ_COST_INF) cand = LZ_COST_INF;
				key = (cand << 9) | (L - 1);
			}
			for (u32 base = 32; base < Lmax; base += 32) {
				const u32 L = base + lane + 1;
				if (L <= Lmax) {
					u32 c = pos + L == s1 ? 0 : costg[pos + L];
					u32 cand = c + lenc[L] + offc[lz_off_slot(dist_for(L))];
					if (cand > LZ_COST_INF) cand = LZ_COST_INF;
					u32 k2 = (cand << 9) | (L - 1);
					if (k2 < key) key = k2;
				}
			}
#pragma unroll
			for (int o = 16; o > 0; o >>= 1) {
				u32 other = __shfl_xor_sync(LDB_FULL_MASK, key, o);
				if (other < key) key = other;
			}
			const u32 C = key >> 9, bestL = (key & 511) + 1;
			if (lane == 0) {
				costg[pos] = C;
				if (bestL >= 3) {
					res[pos] = bestL | (((dist_for(bestL) - 1) | 0x8000u) << 16);
				} else {
					res[pos] = 0;
				}
			}
			const u32 t = __shfl_up_sync(LDB_FULL_MASK, wc, 1);
			wc = lane == 0 ? C : t;
		}
		i = i >= 4 ? i - 4 : 0;
	}
	__syncwarp();
}

// ---- block splitting (ref: observe_literal / do_end_block_check, lib/deflate_compress.c:2105-2190) ---
// The reference watches 8 literal classes (top 2 bits + low bit of the byte) and ends a block when
// the distribution of the newest observations differs from the block so far by >= 200/512 in L1.
// Here blocks end on pass boundaries, so the test runs once per pass, on the bytes of the pass that
// would join the block: lz_observe() counts their classes (all threads), lz_should_end_block()
// applies the reference's integer arithmetic to the two histograms.
__device__ __forceinline__ void lz_observe(const u8 *ring, u32 from, u32 to, u32 *obs, const lz_grp &gp, u32 lane)
{
	// 16 bytes per thread and round; class counts in 8 packed byte fields, reduced per warp
	for (u32 wbase = from + 512 * gp.w; wbase < to; wbase += 16 * gp.nt) {	// warp-uniform trip count
		const u32 base = wbase + 16 * lane;
		const uint4 q = *(const uint4 *)(ring + (base & (LZ_RING - 1)));	// from is 16 KiB aligned
		const u32 w[4] = {q.x, q.y, q.z, q.w};
		u64 cnt = 0;
#pragma unroll
		for (int k = 0; k < 16; k++) {
			const u32 bv = (w[k >> 2] >> (8 * (k & 3))) & 0xff;
			if (base + k < to) cnt += (u64)1 << (8 * (((bv >> 5) & 6) | (bv & 1)));
		}
		u64 lo = cnt & 0x00ff00ff00ff00ffull, hi = (cnt >> 8) & 0x00ff00ff00ff00ffull;	// classes 0,2,4,6 / 1,3,5,7
		for (int o = 16; o > 0; o >>= 1) {
			lo += __shfl_xor_sync(LDB_FULL_MASK, lo, o);
			hi += __shfl_xor_sync(LDB_FULL_MASK, hi, o);
		}
		if (lane < 4) atomicAdd(&obs[2 * lane], (u32)(lo >> (16 * lane)) & 0xffff);
		else if (lane < 8) atomicAdd(&obs[2 * (lane - 4) + 1], (u32)(hi >> (16 * (lane - 4))) & 0xffff);
	}
}

__device__ __forceinline__ bool lz_should_end_block(const u32 *obs, const u32 *obs_new, u32 block_length)
{
	u32 n_old = 0, n_new = 0;
	for (int i = 0; i < 8; i++) { n_old += obs[i]; n_new += obs_new[i]; }
	if (!n_old || !n_new) return false;
	u64 total_delta = 0;
	for (int i = 0; i < 8; i++) {
		const u64 expected = (u64)obs[i] * n_new, actual = (u64)obs_new[i] * n_old;
		total_delta += actual > expected ? actual - expected : expected - actual;
	}
	const u64 cutoff = (u64)n_new * 200 / 512 * n_old;
	return total_delta + (u64)(block_length / 4096) * n_old >= cutoff;
}

// ---- the kernel ----------------------------------------------------------------------------
__global__ void __launch_bounds__(LZ_THREADS, 1)
ldb_deflate_lz_kernel(ldb_deflate_args a)
{
	LDB_DYN_SMEM(sm);
	u8 *ring = sm + LZ_SM_RING;
	u16 *head = (u16 *)(sm + LZ_SM_HEAD);
	u16 *nextt = (u16 *)(sm + LZ_SM_NEXT);
	u32 *vis = (u32 *)(sm + LZ_SM_VIS);
	u32 *tokoff = (u32 *)(sm + LZ_SM_TOKOFF);
	u8 *entryt = sm + LZ_SM_ENTRY;
	u32 *escan = (u32 *)(sm + LZ_SM_ESCAN);
	u16 *gexit = (u16 *)(sm + LZ_SM_GEXIT);
	u32 *gentry = (u32 *)(sm + LZ_SM_GENTRY);
	u32 *freq = (u32 *)(sm + LZ_SM_FREQ);
	u8 *lens = sm + LZ_SM_LENS;
	u16 *codes = (u16 *)(sm + LZ_SM_CODES);
	lz_vars *v = (lz_vars *)(sm + LZ_SM_VARS);
	// block-flush scratch aliases the parse region R (never live at the same time)
	u32 *stage = (u32 *)(sm + LZ_SM_R);				// 8 KiB
	u16 *hsorted = (u16 *)(sm + LZ_SM_R);				// 288 * 2
	u32 *hnodefreq = (u32 *)(sm + LZ_SM_R + 1024);			// 576 * 4
	u16 *hparent = (u16 *)(sm + LZ_SM_R + 1024 + 2304);		// 576 * 2
	u16 *osorted = (u16 *)(sm + LZ_SM_R + 4608);
	u32 *onodefreq = (u32 *)(sm + LZ_SM_R + 4608 + 128);
	u16 *oparent = (u16 *)(sm + LZ_SM_R + 4608 + 128 + 512);
	u16 *items = (u16 *)(sm + LZ_SM_ITEMS);				// precode items (<= 320 + slack)
	// per-position results of the current pass live in this CTA's global scratch
	u8 *gs = a.scratch + 256 + (size_t)blockIdx.x * LZ_GS_BYTES;
	u32 *res = (u32 *)(gs + LZ_GS_RES);	// per position: match length | (distance-1 | decision flag << 15) << 16
	u32 *tokbuf = (u32 *)(gs + LZ_GS_TOK);
	u32 *costg = (u32 *)(gs + LZ_GS_COST);
	u32 *mlist = (u32 *)(gs + LZ_GS_MLIST);
	u8 *costtab = sm + LZ_SM_ITEMS;	// lit[256] len[259] off[32] bit costs of the DP (the items region is free then)

	const u32 tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
	const lz_params P = lz_level_params(a.level);
	// the two warp groups (levels 1-9), or the whole CTA for both halves (serial schedule)
	const bool pipe = LZ_PIPELINE && !P.opt_iters;
	const bool in_a = !pipe || warp < LZ_A_WARPS;
	const lz_grp gA = pipe ? lz_grp{tid, warp, 32 * LZ_A_WARPS, LZ_A_WARPS, LZ_BAR_A} : lz_grp{tid, warp, LZ_THREADS, LZ_WARPS, 0};
	const lz_grp gB = pipe ? lz_grp{tid - 32 * LZ_A_WARPS, warp - LZ_A_WARPS, 32 * LZ_B_WARPS, LZ_B_WARPS, LZ_BAR_B} : gA;
#ifdef LZ_TIMING
	long long tacc[16] = {};
	long long tlast = clock64();
	const bool tlead = (in_a ? gA : gB).t == 0;	// one clock per group
#endif

	if (tid == 0) {
		v->tma_phase = 0;
#ifndef LDB_EMU
		u32 mbar = (u32)__cvta_generic_to_shared(&v->mbar);
		asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(mbar) : "memory");
		asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
#endif
	}
	__syncthreads();

	const u32 overhead = a.format == LDB_FMT_GZIP ? 18 : (a.format == LDB_FMT_ZLIB ? 6 : 0);
	const u32 trailer = a.format == LDB_FMT_GZIP ? 8 : (a.format == LDB_FMT_ZLIB ? 4 : 0);
	const u32 hdr_bytes = overhead - trailer;
	// encode-group state of the chunk being encoded
	size_t c = 0, n64 = 0;
	u32 n = 0;
	const u8 *in = nullptr;
	lz_out o;
	o.out = nullptr; o.avail = 0; o.obit = 0;
	u32 cmin_len = 4, cfar4 = LZ_WIN;	// the chunk's minimum match length and far-4 distance (from the search group)
	u32 block_begin = 0;
	u32 block_entry = 0;	// position of the first token of the current block
	u32 pass_in_block = 0;
	// res holds two passes: pass s (numbered across chunks) at (s % 2) * PASS.  Levels 10-12 index it by
	// the pass in the block instead: their min-cost path covers the whole block.
	auto res_off = [&](u32 s) -> u32 { return (P.opt_iters ? pass_in_block : (s & 1)) * LZ_PASS; };

	auto chunk_begin = [&](const lz_grp &gp, size_t cc, u32 min_len, u32 far4) {
		c = cc;
		in = (const u8 *)a.in_ptrs[c];
		n64 = a.in_nbytes[c];
		n = (u32)n64;
		o.out = (u8 *)a.out_ptrs[c];
		o.avail = a.out_avail[c];
		cmin_len = min_len;
		cfar4 = far4;
		block_begin = 0;
		block_entry = 0;
		pass_in_block = 0;
		if (gp.t == 0) {
			v->failed = 0;
			v->parse_entry = 0;
			v->tok_count = 0;
			// wrapper header: whole words go straight to the output, the partial word is carried
			u8 h[12] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
			def_write_header(h, a.format, a.level);
			u32 whole = hdr_bytes & ~3u;
			for (u32 i = 0; i < whole; i++) o.out[i] = h[i];
			u32 cw = 0;
			for (u32 i = whole; i < hdr_bytes; i++) cw |= (u32)h[i] << (8 * (i - whole));
			v->carry = cw;
		}
		if (gp.t < 8) v->obs_blk[gp.t] = 0;
		for (u32 i = gp.t; i < 320; i += gp.nt) freq[i] = 0;
		o.obit = (u64)hdr_bytes * 8;
		lz_sync(gp);
		// byte classes of the first pass (the block-split test compares the next pass against them)
		lz_observe(ring, 0, n < LZ_PASS ? n : LZ_PASS, v->obs_blk, gp, lane);
		lz_sync(gp);
	};

	// ---- exact parallel parse of one pass (positions [pb0, ppend), results at res[aoff + i]).
	// forced: the DP already decided (flag set on matches); otherwise the lazy rule decides.
	// exitt: 16 Ki u16 of scratch in shared memory -- the link slots of the first pass that is not
	// inserted yet (dead, see lz_insert_pass_par)
	auto parse_pass = [&](const lz_grp &gp, const u32 pb0, const u32 ppend, const u32 aoff, const bool forced, u16 *exitt) {
		// (e1) per-window decisions + "exit position for every entry lane" by pointer jumping
		const u32 nwin = (ppend - pb0 + 31) >> 5;
		// (the per-position results live in L2: the loads run two windows ahead of their use)
		const u32 min_len = cmin_len, far4 = cfar4;
		auto e1_load = [&](u32 w, u32 &x0, u32 &x1, u32 &x2) {
			x0 = 0; x1 = 0; x2 = 0;
			if (w < nwin) {
				const u32 i = w * 32 + lane;
				if (pb0 + i < ppend) x0 = res[aoff + i];
				if (lane == 31 && pb0 + i + 1 < ppend) x1 = res[aoff + i + 1];	// (the others get it by shuffle)
				if (lane == 31 && P.lazy == 2 && pb0 + i + 2 < ppend) x2 = res[aoff + i + 2];
			}
		};
		u32 cW0, cW1, cW2, nW0, nW1, nW2;
		e1_load(gp.w, cW0, cW1, cW2);
		e1_load(gp.w + gp.nw, nW0, nW1, nW2);
		for (u32 w = gp.w; w < nwin; w += gp.nw) {
			u32 i = w * 32 + lane;
			u32 p = pb0 + i;
			const u32 W0 = cW0, nb = __shfl_down_sync(LDB_FULL_MASK, W0, 1), W1 = lane == 31 ? cW1 : nb;
			const u32 nb2 = __shfl_down_sync(LDB_FULL_MASK, W1, 1), W2 = lane == 31 ? cW2 : nb2;	// two ahead (lazy2)
			const u32 L0 = W0 & 0xffff, O0 = ((W0 >> 16) & 0x7fff) + 1, L1 = W1 & 0xffff, O1 = ((W1 >> 16) & 0x7fff) + 1;
			cW0 = nW0; cW1 = nW1; cW2 = nW2;
			e1_load(w + 2 * gp.nw, nW0, nW1, nW2);
			// (a shortest-possible match at a long distance costs more bits than its literals: the
			// reference's rule for length 3 beyond 8 KiB, deflate_compress.c:2666-2668, restated for our
			// minimum length 4)
			bool is_match = forced ? ((L0 >= 3) && p < ppend) : (L0 >= min_len && p < ppend && !(L0 == 4 && O0 > far4));
			if (!forced && is_match && P.lazy && p + 1 < ppend) {
				// ref: deflate_compress.c:2722-2725 -- prefer the next position's match if clearly better
				if (L1 >= L0 && L0 < (u32)P.nice &&
				    4 * ((int)L1 - (int)L0) + ((int)(31 - __clz((int)O0)) - (int)(31 - __clz((int)O1))) > 2)
					is_match = false;
				if (P.lazy == 2 && is_match && p + 2 < ppend) {
					// ref: deflate_compress.c:2757-2760 -- or the one after it, by a wider margin
					const u32 L2 = W2 & 0xffff, O2 = ((W2 >> 16) & 0x7fff) + 1;
					if (L2 >= L0 && L0 < (u32)P.nice &&
					    4 * ((int)L2 - (int)L0) + ((int)(31 - __clz((int)O0)) - (int)(31 - __clz((int)O2))) > 6)
						is_match = false;
				}
			}
			u32 step = is_match ? L0 : 1;
			// decision flag in the top bit; the neighbour that reads res[aoff + i] for its lazy test
			// masks it off, and it only reads -- the flag is published after this warp's reads
			__syncwarp();
			if (is_match && !forced) res[aoff + i] = L0 | (((O0 - 1) | 0x8000u) << 16);
			u32 j = lane + step;
#pragma unroll
			for (int k = 0; k < 5; k++) {
				u32 t = __shfl_sync(LDB_FULL_MASK, j, j & 31);
				if (j < 32) j = t;
			}
			if (p < ppend) exitt[i] = (u16)j;
		}
		lz_sync(gp);
		LZ_T(8);
		// (e2) chain the windows.  A serial walk over all windows costs ~300 cycles per window on
		// one warp, so it is split: (a) every warp composes the exits of ITS group of windows for
		// all 32 possible entry lanes of the group's first window (per-lane shuffles), (b) warp 0
		// chains the groups, (c) every warp re-walks its group along the one real trajectory and
		// records the entry lane of each window.
		{
			const u32 G = (nwin + gp.nw - 1) / gp.nw;		// windows per group
			const u32 wg0 = gp.w * G;				// first window of my group
			const u32 gstart = wg0 * 32;				// pass-relative position
			// (a) exits of the group for entries gstart + lane
			{
				u32 pos = gstart + lane;
				for (u32 k0 = 0; k0 < G; k0 += 8) {
					u32 ex[8];
#pragma unroll
					for (int k = 0; k < 8; k++) {
						u32 w = wg0 + k0 + k;
						u32 i = w * 32 + lane;
						ex[k] = (k0 + k < G && w < nwin && pb0 + i < ppend) ? exitt[i] : (lane + 1);
					}
#pragma unroll
					for (int k = 0; k < 8; k++) {
						u32 w = wg0 + k0 + k;
						u32 x = __shfl_sync(LDB_FULL_MASK, ex[k], pos & 31);
						if (k0 + k < G && w < nwin && (pos >> 5) == w) pos = (w << 5) + x;
					}
				}
				gexit[gp.w * 32 + lane] = (u16)(pos > 0xffff ? 0xffff : pos);
			}
			lz_sync(gp);
			// (b) chain the groups (warp 0, all lanes redundantly; lane 0 publishes)
			if (gp.w == 0) {
				u32 e = v->parse_entry - pb0;	// pass-relative
				for (u32 g = 0; g < gp.nw; g++) {
					const u32 gs = g * G * 32, ge = (g + 1) * G * 32;
					u32 ent = 0xffffffffu;
					if (e < ge && gs < (nwin << 5) && pb0 + e < ppend) {
						ent = e;
						if (e < gs + 32) {
							e = gexit[g * 32 + (e - gs)];
						} else {
							// entered past the group's first window (a long match jumped in): walk it
							for (u32 w = e >> 5; w < (g + 1) * G && w < nwin; w++) {
								if ((e >> 5) == w) {
									u32 i = w * 32 + (e & 31);
									u32 x = pb0 + i < ppend ? exitt[i] : ((e & 31) + 1);
									e = (w << 5) + x;
								}
							}
						}
					}
					if (lane == 0) gentry[g] = ent;
				}
				u32 fin = pb0 + e;
				if (fin < ppend) fin = ppend;
				__syncwarp();	// every lane has read parse_entry (racecheck: read/write by different lanes)
				if (lane == 0) v->parse_entry = fin;
			}
			lz_sync(gp);
			// (c) entry lane of every window of my group along the real trajectory
			{
				u32 pos = gentry[gp.w];
				for (u32 k0 = 0; k0 < G; k0 += 8) {
					u32 ex[8];
#pragma unroll
					for (int k = 0; k < 8; k++) {
						u32 w = wg0 + k0 + k;
						u32 i = w * 32 + lane;
						ex[k] = (k0 + k < G && w < nwin && pb0 + i < ppend) ? exitt[i] : (lane + 1);
					}
#pragma unroll
					for (int k = 0; k < 8; k++) {
						u32 w = wg0 + k0 + k;
						if (k0 + k < G && w < nwin) {
							bool inside = pos != 0xffffffffu && (pos >> 5) == w && pb0 + pos < ppend;
							u32 x = __shfl_sync(LDB_FULL_MASK, ex[k], pos & 31);
							if (lane == 0) entryt[w] = inside ? (u8)(pos & 31) : 0xff;
							if (inside) pos = (w << 5) + x;
						}
					}
				}
			}
		}
		lz_sync(gp);
		LZ_T(9);
		// (e3) visited sets per window (the loads of the next window are issued first)
		auto e3_load = [&](u32 w, u32 &e, u32 &x) {
			e = 0xff; x = 0;
			if (w < nwin) {
				const u32 i = w * 32 + lane;
				e = entryt[w];
				if (e != 0xff && pb0 + i < ppend) x = res[aoff + i];
			}
		};
		u32 e3_e, e3_w, e3_ne, e3_nw;
		e3_load(gp.w, e3_e, e3_w);
		e3_load(gp.w + gp.nw, e3_ne, e3_nw);
		for (u32 w = gp.w; w < nwin; w += gp.nw) {
			const u32 e = e3_e, rw = e3_w;
			e3_e = e3_ne; e3_w = e3_nw;
			e3_load(w + 2 * gp.nw, e3_ne, e3_nw);
			u32 V = 0;
			if (e != 0xff) {
				u32 step = (rw & 0x80000000u) ? (rw & 0xffff) : 1;
				u32 j = lane + step;
				u32 jk[5];
#pragma unroll
				for (int k = 0; k < 5; k++) {
					jk[k] = j;
					u32 t = __shfl_sync(LDB_FULL_MASK, j, j & 31);
					if (j < 32) j = t;
				}
				V = 1u << e;
#pragma unroll
				for (int k = 4; k >= 0; k--) {
					u32 contrib = (((V >> lane) & 1) && jk[k] < 32) ? (1u << jk[k]) : 0;
					V |= __reduce_or_sync(LDB_FULL_MASK, contrib);
				}
				// positions at or beyond the end of the pass are not tokens of this block
				const u32 wbase = pb0 + w * 32;
				if (wbase + 32 > ppend) V &= ppend > wbase ? ((1u << (ppend - wbase)) - 1) : 0;
			}
			if (lane == 0) vis[w] = V;
		}
		lz_sync(gp);
		LZ_T(10);
		// (e4) token offsets (exclusive scan over windows) by warp 0
		if (gp.w == 0) {
			u32 run = 0;
			for (u32 w0 = 0; w0 < nwin; w0 += 32) {
				u32 w = w0 + lane;
				u32 c = w < nwin ? (u32)__popc(vis[w]) : 0;
				u32 incl = c;
				for (int o2 = 1; o2 < 32; o2 <<= 1) {
					u32 t = __shfl_up_sync(LDB_FULL_MASK, incl, o2);
					if (lane >= (u32)o2) incl += t;
				}
				if (w < nwin) tokoff[w] = run + incl - c;
				run += __shfl_sync(LDB_FULL_MASK, incl, 31);
			}
			if (lane == 0) tokoff[LZ_NWIN] = run;
		}
		lz_sync(gp);
		LZ_T(11);
		// (e5) emit tokens + histograms
		const u32 tbase = v->tok_count;
		auto e5_load = [&](u32 w, u32 &V, u32 &x) {
			V = 0; x = 0;
			if (w < nwin) {
				V = vis[w];
				if ((V >> lane) & 1) x = res[aoff + w * 32 + lane];
			}
		};
		u32 e5_V, e5_w, e5_nV, e5_nw;
		e5_load(gp.w, e5_V, e5_w);
		e5_load(gp.w + gp.nw, e5_nV, e5_nw);
		for (u32 w = gp.w; w < nwin; w += gp.nw) {
			const u32 V = e5_V, ro = e5_w >> 16;
			const u32 len = e5_w & 0xffff;
			e5_V = e5_nV; e5_w = e5_nw;
			e5_load(w + 2 * gp.nw, e5_nV, e5_nw);
			if (!V) continue;
			u32 i = w * 32 + lane;
			if ((V >> lane) & 1) {
				u32 idx = tbase + tokoff[w] + __popc(V & ((1u << lane) - 1));
				u32 off = (ro & 0x7fff) + 1;
				// (a match that does not fit the data would be a bug upstream; never emit one)
				if ((ro & 0x8000) && len >= 3 && len <= 258 && off <= pb0 + i && pb0 + i + len <= n) {
					tokbuf[idx] = 0x80000000u | ((len - 3) << 15) | (off - 1);
					atomicAdd(&freq[257 + lz_len_slot(len)], 1u);
					atomicAdd(&freq[288 + lz_off_slot(off)], 1u);
				} else {
					u32 bv = lz_ld8(ring, pb0 + i);
					tokbuf[idx] = bv;
					atomicAdd(&freq[bv], 1u);
				}
			}
		}
		lz_sync(gp);
		if (gp.t == 0) v->tok_count = tbase + tokoff[LZ_NWIN];
		lz_sync(gp);
	};

	// ---- Huffman codes from freq[] -> lens[], codes[] (all threads)
	// CTA-wide exclusive scan (all threads must call it); escan[0..64] is the scratch
	auto cta_excl_scan = [&](const lz_grp &gp, u32 x, u32 &total) -> u32 {
		u32 incl = x;
		for (int o2 = 1; o2 < 32; o2 <<= 1) {
			u32 t = __shfl_up_sync(LDB_FULL_MASK, incl, o2);
			if (lane >= (u32)o2) incl += t;
		}
		lz_sync(gp);		// earlier readers of escan are done
		if (lane == 31) escan[gp.w] = incl;
		lz_sync(gp);
		if (gp.w == 0) {
			u32 y = lane < gp.nw ? escan[lane] : 0;
			u32 yi = y;
			for (int o2 = 1; o2 < 32; o2 <<= 1) {
				u32 t = __shfl_up_sync(LDB_FULL_MASK, yi, o2);
				if (lane >= (u32)o2) yi += t;
			}
			if (lane < gp.nw) escan[32 + lane] = yi - y;
			if (lane == gp.nw - 1) escan[64] = yi;
		}
		lz_sync(gp);
		total = escan[64];
		return escan[32 + gp.w] + (incl - x);
	};
	auto build_codes = [&](const lz_grp &gp) {
		// (f1) Huffman codes for both alphabets.  Parallel: rank sort by (freq, sym), leaf depths
		// (every leaf walks to the root), length assignment, canonical codewords (rank among the
		// symbols of equal length).  Serial: only the two-queue merges, on thread 0 (litlen)
		// and thread 32 (offset), and the rare Kraft repair after the 15-bit cap.
		u32 *hcount = (u32 *)(sm + LZ_SM_GEXIT + 256), *ocount = hcount + 17;	// codewords per length
		const bool is_lit = gp.t < 288;
		const u32 lo = is_lit ? 0 : 288, hi = is_lit ? 288 : 320;
		if (gp.t == 0) { v->nused_lit = 0; v->nused_off = 0; v->huff_over = 0; }
		if (gp.t < 34) hcount[gp.t] = 0;
		lz_sync(gp);
		u32 myrank = 0xffffffffu;
		if (gp.t < 320) {
			const u32 f = freq[gp.t];
			lens[gp.t] = 0;
			if (f) {
				u32 rank = 0;
				for (u32 t = lo; t < hi; t++) {
					u32 ft = freq[t];
					rank += (ft != 0) && (ft < f || (ft == f && t < gp.t));
				}
				myrank = rank;
				(is_lit ? hsorted : osorted)[rank] = (u16)(gp.t - lo);
				(is_lit ? hnodefreq : onodefreq)[rank] = f;
				atomicAdd(is_lit ? &v->nused_lit : &v->nused_off, 1u);
			}
		}
		lz_sync(gp);
		const u32 nused = is_lit ? v->nused_lit : v->nused_off;
		if (gp.t == 0 && nused >= 2) lz_huffman_merge(hnodefreq, hparent, nused);
		if (gp.t == 32) { const u32 nu = v->nused_off; if (nu >= 2) lz_huffman_merge(onodefreq, oparent, nu); }
		lz_sync(gp);
		if (gp.t < 320 && myrank != 0xffffffffu && nused >= 2) {
			const u16 *par = is_lit ? hparent : oparent;
			const u32 root = 2 * nused - 2;
			u32 node = myrank, d = 0;
			while (node != root && d <= 15) { node = par[node]; d++; }
			if (d > 15) { d = 15; v->huff_over = 1; }
			atomicAdd(&(is_lit ? hcount : ocount)[d], 1u);
		}
		lz_sync(gp);
		if ((gp.t == 0 || gp.t == 288) && nused < 2) {
			// at least two codewords (ref: deflate_compress.c:1369-1378)
			u8 *ln = lens + lo;
			u32 *cn = is_lit ? hcount : ocount;
			if (nused == 0) { ln[0] = 1; ln[1] = 1; }
			else { const u32 sy = (is_lit ? hsorted : osorted)[0]; ln[sy] = 1; ln[sy ? 0 : 1] = 1; }
			cn[1] = 2;
		}
		if ((gp.t == 0 || gp.t == 32) && v->huff_over) {
			// restore the Kraft sum to exactly 1 by lengthening the cheapest leaves
			u32 *cn = gp.t == 0 ? hcount : ocount;
			u32 kraft = 0;
			for (u32 l = 1; l <= 15; l++) kraft += cn[l] << (15 - l);
			while (kraft > (1u << 15)) {
				u32 l = 14;
				while (cn[l] == 0) l--;
				cn[l]--;
				cn[l + 1] += 2;
				cn[15]--;
				kraft -= 1;
			}
		}
		lz_sync(gp);
		if (gp.t < 320 && myrank != 0xffffffffu && nused >= 2) {
			// rarest symbols get the longest codes
			const u32 *cn = is_lit ? hcount : ocount;
			u32 cum = 0, len = 1;
			for (u32 l = 15; l >= 1; l--) {
				cum += cn[l];
				if (myrank < cum) { len = l; break; }
			}
			lens[gp.t] = (u8)len;
		}
		lz_sync(gp);
		if (gp.t < 320) {
			const u32 l = lens[gp.t];
			u32 code = 0;
			if (l) {
				const u32 *cn = is_lit ? hcount : ocount;
				u32 first = 0;
				for (u32 k = 1; k < l; k++) first = (first + cn[k]) << 1;
				u32 same = 0;
				for (u32 t = lo; t < gp.t; t++) same += lens[t] == l;
				code = __brev(first + same) >> (32 - l);
			}
			codes[gp.t] = (u16)code;
		}
		lz_sync(gp);
	};

	// ---- search half of pass [b0, pend) of input 'in' (n bytes): window loads, chain insertion,
	// guided search -> res + roff.  Levels 1-9 need nothing else of the chunk.
	u32 loaded_end = 0;
	auto search_pass = [&](const lz_grp &gp, const u8 *in, const u32 n, const u32 b0, const u32 pend, const u32 roff) {
		if (gp.t == 0) v->run_counter = 0;
		lz_sync(gp);
		// (a) window staging by the TMA engine, one pass ahead: searching this pass needs
		// [b0 - MAX_DIST, pend + LOOKAHEAD), inserting the next one (concurrently) needs the
		// bytes up to pend + PASS + 3.  The ring then still holds everything back to
		// b0 - 32768 + 16, i.e. the whole MAX_DIST window.
		{
			const u32 want = pend + LZ_PASS + 16 < n ? pend + LZ_PASS + 16 : n;
			while (loaded_end < want) {
				u32 room = LZ_RING - (loaded_end & (LZ_RING - 1));	// a segment must not wrap
				u32 to = loaded_end + (room < LZ_SEG ? room : LZ_SEG);
				if (to > want) to = want;
				lz_load_segment(sm, v, in, loaded_end, to, gp);
				loaded_end = to;
			}
		}
		if (b0 == 0) {
			// alphabet size of the first 4 KiB -> minimum match length (ref:
			// calculate_min_match_len, lib/deflate_compress.c:2329-2346)
			if (gp.t < 8) v->used_lits[gp.t] = 0;
			lz_sync(gp);
			const u32 scan = n < 4096 ? n : 4096;
			for (u32 i = gp.t; i < scan; i += gp.nt) {
				u32 bv = ring[i];
				atomicOr(&v->used_lits[bv >> 5], 1u << (bv & 31));
			}
			lz_sync(gp);
			if (gp.t == 0) {
				u32 cnt = 0;
				for (int k = 0; k < 8; k++) cnt += __popc(v->used_lits[k]);
				v->min_len = n < 512 ? 4 : lz_choose_min_len(cnt, (u32)P.depth);
				// few distinct byte values = cheap literals (text): a far 4-byte match loses against them
				v->far4_dist = cnt < 80 ? LZ_FAR4_DIST : LZ_WIN;
			}
			lz_sync(gp);
		}
		// (b) the group links this pass into the hash chains (ordered within a hash)
		LZ_T(0);	// loads + first-pass extras
#ifdef LZ_TIMING
#define LZ_TARGS , tacc, tlast
#else
#define LZ_TARGS
#endif
		if (pipe) lz_insert_pass_par<LZ_A_WARPS>(ring, head, nextt, (u32 *)(sm + LZ_SM_CMAT), b0, pend, n, gp, lane LZ_TARGS);
		else lz_insert_pass_par<LZ_WARPS>(ring, head, nextt, (u32 *)(sm + LZ_SM_R), b0, pend, n, gp, lane LZ_TARGS);
#undef LZ_TARGS
		LZ_T(3);	// insertion: linking
		{
			// (c) guided search.  Every searcher owns a run of consecutive positions and walks
			// it like the reference's lazy parser (deflate_compress.c:2605-2808): search where
			// a token could start, look one position ahead, then skip the positions the
			// chosen match covers (they inherit it at the same distance).  Every position
			// still gets a (length, distance), so the exact parallel parse below can start a
			// token anywhere.  One search call site per loop trip keeps the warp converged.
			u32 *rs = res + roff;
			if (P.opt_iters) {
				// levels 10-12: every position is searched and keeps its list of matches
				for (u32 i = gp.t; b0 + i < pend; i += gp.nt) {
					const u32 p = b0 + i;
					u32 L = 0, D = 0;
					u32 *ml = mlist + (size_t)(roff + i) * LZ_OPT_K;
					if (p + 4 <= n) {
						lz_search_all(ring, nextt, p, n, P.depth, (u32)P.nice, ml, L, D);
					} else {
						for (u32 k = 0; k < LZ_OPT_K; k++) ml[k] = 0;
					}
					rs[i] = L ? L | ((D - 1) << 16) : 0;
				}
			} else {
			const u32 min_len = v->min_len, far4 = v->far4_dist;
			// A run starts its walk without knowing where the parse really enters it, so short
			// runs cost a little ratio (L6: +0.9 % at 16 vs 32) and buy parallelism; the deep
			// levels, which are chosen for ratio, keep 32.
#ifndef LZ_RUN_SHORT
#define LZ_RUN_SHORT 16
#endif
			const u32 run_len = a.level >= 7 ? 32 : LZ_RUN_SHORT;
			// runs are handed out dynamically (shared counter): lanes whose runs are cheap
			// (long matches, few searches) take more of them, which keeps the warp busy
			u32 i = 0, i_end = 0;
			u32 pL = 0, pD = 0;		// pending match at position i-pending (lazy evaluation in progress)
			u32 pending = 0;		// 0: none, 1: looking one position ahead, 2: two positions (lazy2)
#if LZ_QUANTUM
			lz_walk wk;
			wk.left = 0; wk.best_len = 0; wk.best_dist = 0; wk.cand = 0; wk.prev_dist = 0; wk.tailo = 0; wk.tailv = 0; wk.cur = 0;
			bool in_search = false;
#endif
			for (;;) {
#if LZ_QUANTUM
				if (!in_search) {
#endif
				if (i >= i_end || b0 + i >= pend) {
					const u32 r = atomicAdd(&v->run_counter, 1u);
					i = r * run_len;
					if (b0 + i >= pend || i >= LZ_PASS) break;
					i_end = i + run_len;
					pending = 0;
				}
#if LZ_QUANTUM
					const u32 p0 = b0 + i;
					wk.best_len = 0; wk.best_dist = 0; wk.left = 0;
					if (p0 + 4 <= n) {
						u32 sL = 0, sD = 0;
						if (pending) { sL = pL - pending >= 4 ? pL - pending : 0; sD = pD; }
						lz_walk_setup(ring, nextt, p0, n, P.depth >> pending, (u32)P.nice, sL, sD, wk);
					}
					in_search = true;
				}
				lz_walk_steps(ring, nextt, b0 + i, n, (u32)P.nice, wk, LZ_QUANTUM);
				if (wk.left > 0) continue;		// the others move on; this search resumes next trip
				in_search = false;
				const u32 p = b0 + i;
				u32 L = wk.best_len, D = wk.best_dist;
#else
				const u32 p = b0 + i;
				u32 L = 0, D = 0;
				if (p + 4 <= n) {
					if (pending) { L = pL - pending >= 4 ? pL - pending : 0; D = pD; }	// the pending match continues here
					lz_search(ring, nextt, p, n, P.depth >> pending, (u32)P.nice, L, D);
				}
#endif
				rs[i] = L ? L | ((D - 1) << 16) : 0;
				u32 mpos, mL, mD;	// match to accept this trip (mL == 0: none)
				if (pending) {
					// ref: deflate_compress.c:2722-2725 (margin 2, one ahead), :2757-2760 (margin 6, two ahead)
					const int margin = pending == 1 ? 2 : 6;
					if (L >= pL && 4 * ((int)L - (int)pL) + ((int)(31 - __clz((int)pD)) - (int)(31 - __clz((int)D))) > margin) {
						// the lookahead match is clearly better: literal(s) before i, keep looking
						// ahead from i unless it is long enough to take at once
						mpos = i; mL = L >= (u32)P.nice ? L : 0; mD = D;
						if (!mL) { pL = L; pD = D; }
						pending = mL == 0 ? 1 : 0;
					} else if (pending == 1 && P.lazy == 2 && i + 1 < i_end && b0 + i + 1 < pend) {
						pending = 2;
						mpos = i; mL = 0; mD = 0;
					} else {
						mpos = i - pending; mL = pL; mD = pD;
						pending = 0;
					}
				} else if (L >= min_len && !(L == 4 && D > far4)) {
					if (P.lazy && L < (u32)P.nice && i + 1 < i_end && b0 + i + 1 < pend) {
						pending = 1; pL = L; pD = D;
						mpos = i; mL = 0; mD = 0;
					} else {
						mpos = i; mL = L; mD = D;
					}
				} else {
					mpos = i; mL = 0; mD = 0;
				}
				if (mL) {
					// positions covered by the accepted match inherit it at the same distance;
					// 'mend' (end of the match at that distance) only moves forward, so extending
					// the inherited matches (needed when the match was capped at 258) is O(1) amortised
					u32 stop = mpos + mL < i_end ? mpos + mL : i_end;
					if (b0 + stop > pend) stop = pend - b0;
					u32 mend = b0 + mpos + mL;
					for (u32 k = i + 1; k < stop; k++) {
						const u32 pk = b0 + k;
						// (the match ended on a mismatch unless it was capped at 258 bytes)
						if (mL == 258)
							while (mend < n && mend - pk < 258 && lz_ld8(ring, mend) == lz_ld8(ring, mend - mD)) mend++;
						u32 lk = mend - pk;
						rs[k] = lk >= 4 ? lk | ((mD - 1) << 16) : 0;
					}
					i = mpos + mL;
				} else {
					i++;
				}
			}
			}	// guided search (levels 1-9)
		}
		lz_sync(gp);
		LZ_T(1);	// search phase (barrier to barrier)
	};

	// ---- encode half: the block flush (Huffman codes, precode, costs, emission) of the block that ends at pend
	auto flush_block = [&](const lz_grp &gp, const u32 pend, const bool last) {
		const u32 npass_block = pass_in_block;
		pass_in_block = 0;
		const u32 block_end = pend;

		// ---- levels 10-12: near-optimal parsing of the block (ref: deflate_optimize_and_flush_block,
		// lib/deflate_compress.c:3417-3530).  Cost model = bit lengths of the Huffman codes of the
		// previous parse; min-cost path by backward DP over independent 2048-position segments
		// (one warp each); the resulting choices are re-parsed by the same parallel parser.
		for (int it = 0; it < P.opt_iters; it++) {
			if (gp.t == 0) freq[256] = 1;
			lz_sync(gp);
			build_codes(gp);
			// bit costs: unused symbols get a pessimistic default (cf. deflate_compress.c:149-151)
			for (u32 k = gp.t; k < 256 + 259 + 32; k += gp.nt) {
				u32 c;
				if (k < 256) {
					c = lens[k] ? lens[k] : 13;
				} else if (k < 256 + 259) {
					u32 len = k - 256;
					if (len < 3) c = 255;
					else { u32 sl = lz_len_slot(len); c = (lens[257 + sl] ? lens[257 + sl] : 13) + lz_len_extra_bits(sl); }
				} else {
					u32 sl = k - 256 - 259;
					c = (lens[288 + sl] ? lens[288 + sl] : 10) + lz_off_extra_bits(sl);
				}
				costtab[k] = (u8)c;
			}
			lz_sync(gp);
			{
				const u32 rel_entry = block_entry - block_begin;	// first token of the block
				const u32 blen_pos = block_end - block_begin;
				for (u32 seg = gp.w; seg * LZ_DP_SEG < blen_pos; seg += gp.nw) {
					u32 s0 = seg * LZ_DP_SEG, s1 = s0 + LZ_DP_SEG < blen_pos ? s0 + LZ_DP_SEG : blen_pos;
					if (s0 < rel_entry) s0 = rel_entry;
					if (s0 >= s1) continue;
					lz_dp_segment(ring, mlist, costg, res, costtab, block_begin, s0, s1, lane);
				}
			}
			lz_sync(gp);
			// re-parse the block with the chosen path
			for (u32 k = gp.t; k < 320; k += gp.nt) freq[k] = 0;
			if (gp.t == 0) { v->tok_count = 0; v->parse_entry = block_entry; }
			lz_sync(gp);
			for (u32 pp = 0; pp < npass_block; pp++) {
				u32 pb0 = block_begin + pp * LZ_PASS;
				u32 ppend = pb0 + LZ_PASS < block_end ? pb0 + LZ_PASS : block_end;
				parse_pass(gp, pb0, ppend, pp * LZ_PASS, true, nextt + ((block_begin + npass_block * LZ_PASS) & 0xffff));
			}
		}
		const u32 ntok = v->tok_count;

		// ======================= block flush =========================================
		LZ_T(7);	// optimal-parse iterations
		if (gp.t == 0) freq[256] = 1;
		lz_sync(gp);
		build_codes(gp);
		LZ_T(4);	// Huffman codes
		// (f2) precode items + precode, ref: deflate_compress.c:1483-1631.  Run-length items in
		// parallel: thread j looks at code length j of the hlit+hdist sequence, run starts are
		// found with ballots, every start knows in closed form how many items its run becomes,
		// a CTA scan places them.  Only the 19-symbol precode itself is built by one thread.
		u32 *pfreq_sm = (u32 *)(sm + LZ_SM_GEXIT);		// u32[19] (region unused while flushing)
		u8 *plens_sm = sm + LZ_SM_GEXIT + 128;			// u8[19]
		u16 *pcodes_sm = (u16 *)(sm + LZ_SM_GEXIT + 160);	// u16[19]
		if (gp.t == 0) {
			u32 hlit = 288;
			while (hlit > 257 && lens[hlit - 1] == 0) hlit--;
			v->hlit = hlit;
		}
		if (gp.t == 32) {
			u32 hdist = 32;
			while (hdist > 1 && lens[288 + hdist - 1] == 0) hdist--;
			v->hdist = hdist;
		}
		if (gp.t >= 64 && gp.t < 64 + 19) pfreq_sm[gp.t - 64] = 0;
		lz_sync(gp);
		{
			const u32 hlit = v->hlit, total = hlit + v->hdist;
			const u32 j = gp.t;
			const bool inb = j < total;
			const u32 val = inb ? (j < hlit ? lens[j] : lens[288 + j - hlit]) : 0xff;
			const u32 prv = (inb && j > 0) ? (j - 1 < hlit ? lens[j - 1] : lens[288 + j - 1 - hlit]) : 0xfe;
			const bool isstart = inb && val != prv;
			const u32 smask = __ballot_sync(LDB_FULL_MASK, isstart);
			if (lane == 0 && gp.w < 10) escan[66 + gp.w] = smask;
			lz_sync(gp);
			u32 run = 0, cnt = 0;
			if (isstart) {
				u32 nxt = total;
				u32 m = lane == 31 ? 0 : (smask & ~((2u << lane) - 1));
				if (m) nxt = gp.w * 32 + __ffs(m) - 1;
				else {
					for (u32 w = gp.w + 1; w < 10; w++) {
						u32 mm = escan[66 + w];
						if (mm) { nxt = w * 32 + __ffs(mm) - 1; break; }
					}
				}
				run = nxt - j;
				if (val == 0) {
					u32 rem = run % 138;
					cnt = run / 138 + (rem >= 3 ? 1 : rem);
				} else if (run >= 4) {
					u32 rem = (run - 1) % 6;
					cnt = 1 + (run - 1) / 6 + (rem >= 3 ? 1 : rem);
				} else cnt = run;
			}
			u32 ntot;
			const u32 off = cta_excl_scan(gp, cnt, ntot);
			if (isstart) {
				u32 ni = off;
				if (val == 0) {
					while (run >= 11) {
						u32 r = run < 138 ? run : 138;
						items[ni++] = (u16)(18 | ((r - 11) << 5));
						atomicAdd(&pfreq_sm[18], 1u);
						run -= r;
					}
					if (run >= 3) {
						items[ni++] = (u16)(17 | ((run - 3) << 5));
						atomicAdd(&pfreq_sm[17], 1u);
						run = 0;
					}
				} else if (run >= 4) {
					items[ni++] = (u16)val;
					atomicAdd(&pfreq_sm[val], 1u);
					run--;
					while (run >= 3) {
						u32 r = run < 6 ? run : 6;
						items[ni++] = (u16)(16 | ((r - 3) << 5));
						atomicAdd(&pfreq_sm[16], 1u);
						run -= r;
					}
				}
				if (run) atomicAdd(&pfreq_sm[val], run);
				while (run) { items[ni++] = (u16)val; run--; }
			}
			if (gp.t == 0) v->n_items = ntot;
		}
		lz_sync(gp);
		if (gp.w == 0) {
			// the 19-symbol precode, limited to 7 bits, by warp 0: lane = symbol.  Same construction
			// as build_codes (rank sort, two-queue merge on lane 0, leaf depths, Kraft repair, lengths
			// by rank, canonical codewords), with the counts per length packed into one u64.
			u32 *pnodef = (u32 *)(sm + LZ_SM_GEXIT + 512);		// u32[38]
			u16 *ppar = (u16 *)(sm + LZ_SM_GEXIT + 672);		// u16[38]
			const u32 lt = (1u << lane) - 1;
			const u32 f = lane < 19 ? pfreq_sm[lane] : 0;
			const u32 usedm = __ballot_sync(LDB_FULL_MASK, f != 0);
			const u32 nused = __popc(usedm);
			u32 rank = 0;
			for (u32 t = 0; t < 19; t++) {
				const u32 ft = __shfl_sync(LDB_FULL_MASK, f, t);
				rank += (ft != 0) && (ft < f || (ft == f && t < lane));
			}
			if (f) pnodef[rank] = f;
			__syncwarp();
			if (lane == 0 && nused >= 2) lz_huffman_merge(pnodef, ppar, nused);
			__syncwarp();
			u32 d = 0;
			bool over = false;
			if (f && nused >= 2) {
				const u32 root = 2 * nused - 2;
				u32 node = rank;
				while (node != root && d <= 7) { node = ppar[node]; d++; }
				if (d > 7) { d = 7; over = true; }
			}
			u64 cn = 0;		// codewords per length, 8 bits each
			for (u32 l = 1; l <= 7; l++) cn |= (u64)__popc(__ballot_sync(LDB_FULL_MASK, d == l)) << (8 * l);
			if (__any_sync(LDB_FULL_MASK, over)) {
				u32 kraft = 0;
				for (u32 l = 1; l <= 7; l++) kraft += (u32)((cn >> (8 * l)) & 0xff) << (7 - l);
				while (kraft > (1u << 7)) {
					u32 l = 6;
					while (((cn >> (8 * l)) & 0xff) == 0) l--;
					cn -= (u64)1 << (8 * l);
					cn += (u64)2 << (8 * (l + 1));
					cn -= (u64)1 << (8 * 7);
					kraft -= 1;
				}
			}
			u32 len = 0;
			if (nused >= 2) {
				if (f) {
					u32 cum = 0;
					len = 1;
					for (u32 l = 7; l >= 1; l--) {
						cum += (u32)((cn >> (8 * l)) & 0xff);
						if (rank < cum) { len = l; break; }
					}
				}
			} else {
				// at least two codewords
				const u32 sy = nused ? (u32)__ffs(usedm) - 1 : 0;
				len = (lane == sy || lane == (sy ? 0u : 1u)) ? 1 : 0;
				cn = (u64)2 << 8;
			}
			u32 first = 0;
			for (u32 k = 1; k < len; k++) first = (first + (u32)((cn >> (8 * k)) & 0xff)) << 1;
			const u32 samem = __match_any_sync(LDB_FULL_MASK, len);
			const u32 code = len ? __brev(first + __popc(samem & lt)) >> (32 - len) : 0;
			if (lane < 19) { plens_sm[lane] = (u8)len; pcodes_sm[lane] = (u16)code; }
			__syncwarp();
			const u8 perm[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
			const u32 nzm = __ballot_sync(LDB_FULL_MASK, lane < 19 && plens_sm[perm[lane < 19 ? lane : 0]] != 0);
			u32 hclen = nzm ? 32 - __clz(nzm) : 0;
			if (hclen < 4) hclen = 4;
			u32 cost = f * len + (lane == 16 ? 2 * f : lane == 17 ? 3 * f : lane == 18 ? 7 * f : 0);
			for (int o2 = 16; o2 > 0; o2 >>= 1) cost += __shfl_xor_sync(LDB_FULL_MASK, cost, o2);
			if (lane == 0) {
				v->cost_dyn = cost + 3 + 5 + 5 + 4 + 3 * hclen;
				v->hclen = hclen;
				v->cost_static = 3;
				v->extra_bits = 0;
			}
		}
		lz_sync(gp);
		LZ_T(5);	// precode
		// (f3) symbol costs (ref: deflate_compress.c:1750-1808)
		if (gp.t < 320) {
			u32 f = freq[gp.t];
			if (f) {
				u32 dyn = f * lens[gp.t];
				u32 extra = 0, st;
				if (gp.t < 288) {
					st = f * lz_static_litlen_len(gp.t);
					if (gp.t >= 257) extra = f * lz_len_extra_bits(gp.t - 257);
				} else {
					st = f * 5;
					extra = f * lz_off_extra_bits(gp.t - 288);
				}
				atomicAdd(&v->cost_dyn, dyn + extra);
				atomicAdd(&v->cost_static, st + extra);
			}
		}
		lz_sync(gp);
		const u32 cost_dyn = v->cost_dyn, cost_static = v->cost_static;
		// The tokens of this block cover [block_entry, parse_entry): its first token starts where the
		// previous block's last match ended and its own last match may run past block_end.  A
		// stored block must cover exactly the same bytes.
		// (past the end of the input the parser's continuation point is only window-granular)
		const u32 sbeg = block_entry, blen = (v->parse_entry < n ? v->parse_entry : n) - block_entry;
		const u32 bitoff = (u32)(o.obit & 7);
		const u32 stored_pieces = blen ? (blen + 65534) / 65535 : 1;
		// first piece: 3 header bits + pad to a byte; later pieces start byte aligned
		const u64 cost_stored = (u64)(((bitoff + 3 + 7) & ~7u) - bitoff) + 32 + (u64)8 * blen + (u64)(stored_pieces - 1) * 40;
		u32 btype;	// ties: stored, then static, then dynamic (deflate_compress.c:1804-1808)
		u64 best = cost_stored;
		btype = DEFLATE_BLOCKTYPE_STORED;
		if (cost_static < best) { best = cost_static; btype = DEFLATE_BLOCKTYPE_STATIC; }
		if (cost_dyn < best) { best = cost_dyn; btype = DEFLATE_BLOCKTYPE_DYNAMIC; }
		// single bounds check for the whole block (deflate_compress.c:1811-1814)
		const u64 need_bytes = (o.obit + best + 7) / 8 + (last ? trailer : 0);
		if (need_bytes > o.avail) {
			if (gp.t == 0) v->failed = 1;
			lz_sync(gp);
			return;
		}

		// staging covers bits starting at word 'w0' of the output; word 0 is seeded with
		// the partial word carried from the previous flush
		u64 w0 = o.obit >> 5;
		for (u32 k = gp.t; k < LZ_STAGE_WORDS; k += gp.nt) stage[k] = 0;
		lz_sync(gp);
		if (gp.t == 0) stage[0] = v->carry;
		lz_sync(gp);
		if (btype == DEFLATE_BLOCKTYPE_STORED) {
			// ---- stored: header bits via staging, raw bytes straight from the input
			u32 src = sbeg;
			for (u32 piece = 0; piece < stored_pieces; piece++) {
				u32 len = blen - (src - sbeg) > 65535 ? 65535 : blen - (src - sbeg);
				bool fin = last && piece + 1 == stored_pieces;
				if (gp.t == 0) {
					lz_stage_or(stage, (u32)(o.obit - (w0 << 5)), fin ? 1 : 0, 3);
					u64 ob = (o.obit + 3 + 7) & ~(u64)7;
					lz_stage_or(stage, (u32)(ob - (w0 << 5)), (u64)len | ((u64)(~len & 0xffff) << 16), 32);
				}
				o.obit = ((o.obit + 3 + 7) & ~(u64)7) + 32;
				lz_sync(gp);
				// flush staging up to the (byte aligned) current position, byte granular
				{
					u64 bytes_end = o.obit >> 3, bytes_begin = w0 * 4;
					for (u64 k = bytes_begin + gp.t; k < bytes_end; k += gp.nt) {
						u32 rel = (u32)(k - bytes_begin);
						o.out[k] = (u8)(stage[rel >> 2] >> (8 * (rel & 3)));
					}
				}
				lz_sync(gp);
				for (u32 k = gp.t; k < LZ_STAGE_WORDS; k += gp.nt) stage[k] = 0;
				u8 *dst = o.out + (o.obit >> 3);
				for (u32 k = gp.t; k < len; k += gp.nt) dst[k] = in[src + k];
				src += len;
				o.obit += (u64)len * 8;
				lz_sync(gp);
				// re-seed staging word 0 with the bytes already written in the current word
				w0 = o.obit >> 5;
				if (gp.t == 0) {
					u32 nb = (u32)((o.obit >> 3) & 3);
					u32 wv = 0;
					for (u32 k = 0; k < nb; k++) wv |= (u32)(*(volatile u8 *)(o.out + w0 * 4 + k)) << (8 * k);
					stage[0] = wv;
				}
				lz_sync(gp);
			}
		} else {
			// ---- Huffman block --------------------------------------------------------
			if (btype == DEFLATE_BLOCKTYPE_STATIC) {
				for (u32 s = gp.t; s < 320; s += gp.nt) lens[s] = s < 288 ? (u8)lz_static_litlen_len(s) : 5;
				lz_sync(gp);
				if (gp.t == 0) lz_gen_codes_serial(lens, 288, codes);
				if (gp.t == 32) lz_gen_codes_serial(lens + 288, 32, codes + 288);
				lz_sync(gp);
			}
			// header: fixed fields by thread 0, the precode items by one thread each (bit offsets
			// from a CTA scan), directly into staging
			u32 rel;
			{
				const u32 rb0 = (u32)(o.obit - (w0 << 5));
				u32 rb = rb0 + 3;
				if (gp.t == 0) lz_stage_or(stage, rb0, (last ? 1 : 0) | (btype << 1), 3);
				if (btype == DEFLATE_BLOCKTYPE_DYNAMIC) {
					const u32 hclen = v->hclen, nit = v->n_items;
					if (gp.t == 0)
						lz_stage_or(stage, rb, (v->hlit - 257) | ((v->hdist - 1) << 5) | ((hclen - 4) << 10), 14);
					rb += 14;
					if (gp.t < hclen) {
						const u8 perm[19] = {16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1, 15};
						lz_stage_or(stage, rb + 3 * gp.t, plens_sm[perm[gp.t]], 3);
					}
					rb += 3 * hclen;
					u32 nb = 0, bits = 0;
					if (gp.t < nit) {
						const u32 it = items[gp.t], sym = it & 31, ex = it >> 5;
						const u32 pl = plens_sm[sym];
						const u32 eb = sym == 16 ? 2 : (sym == 17 ? 3 : (sym == 18 ? 7 : 0));
						bits = pcodes_sm[sym] | (ex << pl);
						nb = pl + eb;
					}
					u32 hbits;
					const u32 hoff = cta_excl_scan(gp, nb, hbits);
					lz_stage_or(stage, rb + hoff, bits, nb);
					rb += hbits;
				}
				rel = rb;	// bits used in staging so far (relative to word w0)
			}
			lz_sync(gp);
			// token rounds: bit lengths -> exclusive scan -> OR into staging -> flush whole words
			const u32 tpt = LZ_THREADS / gp.nt;	// tokens per thread and round
			for (u32 t0 = 0; t0 <= ntok; t0 += gp.nt * tpt) {
				// (the EOB symbol is token index ntok)
				u32 mybits[LZ_TPT_MAX] = {};
				u64 myval[LZ_TPT_MAX] = {};
#pragma unroll
				for (u32 r = 0; r < LZ_TPT_MAX; r++) {
					u32 ti = t0 + gp.t * tpt + r;
					if (r >= tpt) {
					} else if (ti < ntok) {
						u32 tk = tokbuf[ti];
						if (tk & 0x80000000u) {
							u32 len = ((tk >> 15) & 0x1ff) + 3, off = (tk & 0x7fff) + 1;
							u32 ls = lz_len_slot(len), os = lz_off_slot(off);
							u32 nb = lens[257 + ls];
							u64 val = codes[257 + ls];
							u32 leb = lz_len_extra_bits(ls);
							val |= (u64)(len - lz_len_base(ls)) << nb;
							nb += leb;
							val |= (u64)codes[288 + os] << nb;
							nb += lens[288 + os];
							u32 oeb = lz_off_extra_bits(os);
							val |= (u64)(off - lz_off_base(os)) << nb;
							nb += oeb;
							mybits[r] = nb;
							myval[r] = val;
						} else {
							mybits[r] = lens[tk];
							myval[r] = codes[tk];
						}
					} else if (ti == ntok) {
						mybits[r] = lens[256];
						myval[r] = codes[256];
					}
				}
				// CTA-wide exclusive scan of the threads' bit counts
				u32 mine = 0;
#pragma unroll
				for (int r = 0; r < LZ_TPT_MAX; r++) mine += mybits[r];
				u32 incl = mine;
				for (int o2 = 1; o2 < 32; o2 <<= 1) {
					u32 t = __shfl_up_sync(LDB_FULL_MASK, incl, o2);
					if (lane >= (u32)o2) incl += t;
				}
				if (lane == 31) escan[gp.w] = incl;
				lz_sync(gp);
				if (gp.w == 0) {
					u32 x = lane < gp.nw ? escan[lane] : 0;
					u32 xi = x;
					for (int o2 = 1; o2 < 32; o2 <<= 1) {
						u32 t = __shfl_up_sync(LDB_FULL_MASK, xi, o2);
						if (lane >= (u32)o2) xi += t;
					}
					if (lane < gp.nw) escan[32 + lane] = xi - x;
					if (lane == gp.nw - 1) escan[64] = xi;
				}
				lz_sync(gp);
				u32 bitpos = rel + escan[32 + gp.w] + (incl - mine);
#pragma unroll
				for (int r = 0; r < LZ_TPT_MAX; r++) {
					lz_stage_or(stage, bitpos, myval[r], mybits[r]);
					bitpos += mybits[r];
				}
				const u32 round_bits = escan[64];
				lz_sync(gp);
				rel += round_bits;
				// flush complete words, keep the partial one as the new stage[0]
				u32 full = rel >> 5;
				if (full) {
					lz_flush_words(o, stage, w0, full, gp);
					lz_sync(gp);
					u32 carry = stage[full];
					lz_sync(gp);
					for (u32 k = gp.t; k <= full && k < LZ_STAGE_WORDS; k += gp.nt) stage[k] = 0;
					lz_sync(gp);
					if (gp.t == 0) stage[0] = carry;
					w0 += full;
					rel &= 31;
					lz_sync(gp);
				}
			}
			o.obit = (w0 << 5) + rel;
		}
		lz_sync(gp);
		if (gp.t == 0) v->carry = stage[0];
		LZ_T(6);	// costs + emission
		// ---- next block ------------------------------------------------------------
		block_begin = block_end;
		block_entry = v->parse_entry;
		for (u32 i = gp.t; i < 320; i += gp.nt) freq[i] = 0;
		if (gp.t == 0) v->tok_count = 0;
		lz_sync(gp);
	};

	// ---- encode half: end of the chunk (final partial byte + trailer)
	auto chunk_end = [&](const lz_grp &gp) {
	lz_sync(gp);
	if (v->failed) {
		if (gp.t == 0) a.out_nbytes[c] = 0;
		lz_sync(gp);
		return;
	}
	// ---- final partial byte + trailer ------------------------------------------------
	{
		u64 w0 = o.obit >> 5;
		for (u32 k = gp.t; k < LZ_STAGE_WORDS; k += gp.nt) stage[k] = 0;
		lz_sync(gp);
		if (gp.t == 0) stage[0] = v->carry;
		lz_sync(gp);
		u64 ob = (o.obit + 7) & ~(u64)7;	// pad the last byte with zero bits
		if (gp.t == 0 && trailer) {
			u8 t[8];
			def_write_trailer(t, a.format, a.checksums ? a.checksums[c] : 0, n64);
			for (u32 k = 0; k < trailer; k++) lz_stage_or(stage, (u32)(ob - (w0 << 5)) + 8 * k, t[k], 8);
		}
		ob += (u64)trailer * 8;
		lz_sync(gp);
		u64 bytes_begin = w0 * 4, bytes_end = ob >> 3;
		for (u64 k = bytes_begin + gp.t; k < bytes_end; k += gp.nt) {
			u32 rel = (u32)(k - bytes_begin);
			o.out[k] = (u8)(stage[rel >> 2] >> (8 * (rel & 3)));
		}
		if (gp.t == 0) a.out_nbytes[c] = (size_t)(ob >> 3);
	}
	lz_sync(gp);
		LZ_T(7);	// chunk prologue/epilogue
	};

	// ---- encode half of pass s: exact parallel parse -> tokens + histograms, block-split test,
	// release of the pass (its res slot and ring bytes are free again), then the block flush if the
	// block ends here.  exitt: 16 Ki u16 of scratch for the parse.
	auto encode_pass = [&](const lz_grp &gp, const u32 s, const u32 b0, u16 *exitt) {
		const u32 pend = b0 + LZ_PASS < n ? b0 + LZ_PASS : n;
		const bool last = pend >= n;
		bool end_now = true;
		if (!v->failed) {
			parse_pass(gp, b0, pend, res_off(s), false, exitt);
			LZ_T(2);	// parse
			// ---- block boundary: every LZ_BLOCK_PASSES passes, or at the end of the input --------
			// A block also ends early when the bytes of the next pass look different from the block
			// so far (the reference's block-split test, on pass granularity).
			pass_in_block++;
			if (!last) {
				if (gp.t < 8) v->obs_next[gp.t] = 0;
				lz_sync(gp);
				lz_observe(ring, pend, pend + LZ_PASS < n ? pend + LZ_PASS : n, v->obs_next, gp, lane);
				lz_sync(gp);
				if (gp.t == 0) v->end_early = lz_should_end_block(v->obs_blk, v->obs_next, pend - block_begin) ? 1 : 0;
				lz_sync(gp);
				end_now = pass_in_block == LZ_BLOCK_PASSES || v->end_early;
				lz_sync(gp);
				if (gp.t < 8) v->obs_blk[gp.t] = end_now ? v->obs_next[gp.t] : v->obs_blk[gp.t] + v->obs_next[gp.t];
			}
		}
		if (pipe) lz_bar_arrive(LZ_BAR_EMPTY + (s & 1), LZ_THREADS);
		if (end_now && !v->failed) flush_block(gp, pend, last);
		if (last) chunk_end(gp);
	};

	// ---- the schedule.  The search group takes chunks from the work counter and searches their passes;
	// pass s is handed over in slot s % 2 (res, the slot_* fields).  Pipelined, the encode group follows
	// one pass behind; serially, the whole CTA encodes each pass right after searching it.
	if (in_a) {
		u32 s = 0;		// passes searched by this CTA (numbered across chunks)
		u32 released = 0;	// passes the encode group has released (pipelined)
		u32 prev_npass = 0;	// passes of the previous chunk
		// wait until passes [0, upto) are released
		auto wait_released = [&](u32 upto) {
			while (released < upto) {
				lz_bar_sync(LZ_BAR_EMPTY + (released & 1), LZ_THREADS);
				released++;
			}
			LZ_T(14);	// search group: waiting for the encode group
		};
		for (;;) {
			if (gA.t == 0) v->chunk = atomicAdd(a.work_counter, 1u);
			lz_sync(gA);
			const size_t ca = v->chunk;
			lz_sync(gA);
			if (ca >= a.n) break;

			const u8 *ain = (const u8 *)a.in_ptrs[ca];
			const size_t an64 = a.in_nbytes[ca];
			// ---- tiny inputs and oversize chunks take the stored path (ref: deflate_compress.c:4041-4043)
			{
				const lz_grp &gp = gA;
				u8 *out = (u8 *)a.out_ptrs[ca];
				const size_t avail = a.out_avail[ca];
				const bool passthrough = an64 <= (size_t)(55 - 4 * a.level) || an64 > 0x7fff0000u;
				bool fits = !(overhead && avail <= overhead);
				if (passthrough || !fits) {
					const size_t nblocks = an64 ? (an64 + 65534) / 65535 : 1;
					fits = fits && (an64 + 5 * nblocks <= avail - overhead);
					if (!fits) {
						if (gp.t == 0) a.out_nbytes[ca] = 0;
						continue;
					}
					if (gp.t == 0) def_write_header(out, a.format, a.level);
					u8 *dst = out + hdr_bytes;
					for (size_t b = 0; b < nblocks; b++) {
						size_t off = b * 65535;
						u32 len = (u32)(an64 - off > 65535 ? 65535 : an64 - off);
						if (gp.t == 0) {
							dst[0] = (b + 1 == nblocks) ? 1 : 0;
							dst[1] = (u8)len; dst[2] = (u8)(len >> 8);
							dst[3] = (u8)~len; dst[4] = (u8)(~len >> 8);
						}
						for (u32 i = gp.t; i < len; i += gp.nt) dst[5 + i] = ain[off + i];
						dst += 5 + len;
					}
					if (gp.t == 0) {
						u32 t = def_write_trailer(dst, a.format, a.checksums ? a.checksums[ca] : 0, an64);
						a.out_nbytes[ca] = (size_t)(dst - out) + t;
					}
					continue;
				}
			}
			const u32 an = (u32)an64;
			for (u32 i = gA.t; i < (1u << LZ_HASH_BITS) / 2; i += gA.nt) ((u32 *)head)[i] = 0xffffffffu;
			loaded_end = 0;
			for (u32 b0 = 0; b0 < an; b0 += LZ_PASS, s++) {
				const u32 pend = b0 + LZ_PASS < an ? b0 + LZ_PASS : an;
				if (pipe) {
					// Pass s reuses res slot s % 2 and, with the ring one pass ahead, overwrites the ring
					// bytes of pass s - 3 and the first 16 of pass s - 2: pass s - 2 must be released.  The
					// encode group then works on pass s - 1 at most, which reads the ring bytes of passes
					// s - 1 and s.  The first pass of a chunk reloads ring slots [0, 2 PASS + 16), which the
					// previous chunk's last pass reads unless it sat in the last quarter of the ring.
					wait_released(s >= 1 ? s - 1 : 0);
					if (b0 == 0 && (prev_npass & 3) != 0) wait_released(s);
				}
				search_pass(gA, ain, an, b0, pend, res_off(s));
				if (pipe) {
					if (gA.t == 0) {
						v->slot_chunk[s & 1] = (u32)ca;
						v->slot_b0[s & 1] = b0;
						v->slot_min_len[s & 1] = v->min_len;
						v->slot_far4[s & 1] = v->far4_dist;
					}
					lz_bar_arrive(LZ_BAR_FULL + (s & 1), LZ_THREADS);
				} else {
					if (b0 == 0) chunk_begin(gA, ca, v->min_len, v->far4_dist);
					encode_pass(gA, s, b0, nextt + ((b0 + LZ_PASS) & 0xffff));	// the dead link slots of the next pass
				}
			}
			prev_npass = (an + LZ_PASS - 1) / LZ_PASS;
		}
		if (pipe) {
			wait_released(s >= 1 ? s - 1 : 0);
			if (gA.t == 0) v->slot_chunk[s & 1] = LZ_NO_CHUNK;
			lz_bar_arrive(LZ_BAR_FULL + (s & 1), LZ_THREADS);
			wait_released(s);
		}
	} else {
		// encode group: the parse cannot use the link slots of the next pass (the search group is
		// inserting it), its exits go to this CTA's global scratch
		u16 *exitg = (u16 *)(gs + LZ_GS_EXIT);
		for (u32 s = 0;; s++) {
			lz_bar_sync(LZ_BAR_FULL + (s & 1), LZ_THREADS);
			LZ_T(15);	// encode group: waiting for the search group
			const u32 cc = v->slot_chunk[s & 1];
			if (cc == LZ_NO_CHUNK) break;
			const u32 b0 = v->slot_b0[s & 1];
			if (b0 == 0) chunk_begin(gB, cc, v->slot_min_len[s & 1], v->slot_far4[s & 1]);
			encode_pass(gB, s, b0, exitg);
		}
	}
#ifdef LZ_TIMING
	if (tlead)
		for (int k = 0; k < 16; k++) atomicAdd(&ldb_lz_timing[k], (unsigned long long)tacc[k]);
#endif
}

#ifdef LZ_TIMING
extern "C" __attribute__((visibility("default"))) void ldb_lz_timing_dump(void)
{
	unsigned long long h[16], z[16] = {};
	cudaDeviceSynchronize();
	cudaMemcpyFromSymbol(h, ldb_lz_timing, sizeof(h));
	cudaMemcpyToSymbol(ldb_lz_timing, z, sizeof(z));
	const char *names[16] = {"loads+first", "search phase", "parse e5", "insert: linking", "huffman", "precode", "cost+emit", "chunk pro/epilogue",
				 "parse e1", "parse e2", "parse e3", "parse e4", "insert: hashing", "insert: slice lists",
				 "search grp waits (encode)", "encode grp waits (search)"};
	unsigned long long tot = 0;
	for (int k = 0; k < 16; k++) tot += h[k];
	for (int k = 0; k < 16; k++)
		if (h[k]) printf("  timing %-26s %14llu cycles  %5.1f%%\n", names[k], h[k], 100.0 * (double)h[k] / (double)tot);
}
#endif

// work counter (first 256 bytes) + one scratch block per CTA that a batch of n chunks launches
size_t ldb_deflate_scratch_bytes(const ldb_launch_cfg &cfg, size_t n)
{
	size_t ctas = n < (size_t)ldb_deflate_grid(cfg) ? n : (size_t)ldb_deflate_grid(cfg);
	return 256 + ctas * LZ_GS_BYTES;
}

static int ldb_launch_deflate_lz(const ldb_deflate_args &a, const ldb_launch_cfg &cfg, void *stream)
{
	// per device, cheap: set on every launch (contexts may live on different GPUs and threads)
	LDB_CUDA_CHECK_RET(cudaFuncSetAttribute(ldb_deflate_lz_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, LZ_SM_BYTES));
	ldb_deflate_args b = a;
	b.work_counter = (u32 *)a.scratch;
	LDB_CUDA_CHECK_RET(cudaMemsetAsync(b.work_counter, 0, sizeof(u32), (cudaStream_t)stream));
	size_t blocks = a.n < (size_t)ldb_deflate_grid(cfg) ? a.n : (size_t)ldb_deflate_grid(cfg);
	LDB_LAUNCH(ldb_deflate_lz_kernel, dim3((unsigned)blocks), dim3(LZ_THREADS), LZ_SM_BYTES, (cudaStream_t)stream, b);
	LDB_CUDA_CHECK_RET(cudaGetLastError());
	return 0;
}
