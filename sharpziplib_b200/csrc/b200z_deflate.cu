// b200z_deflate.cu -- the sm_100a DEFLATE compressor for the reference's lazy levels (5-9).
// Kernel decomposition and the reference lines each kernel replaces: see b200z_core.cuh and DESIGN.md.
//
//   k_links   (K1)  DeflaterEngine.InsertString / head[] / prev[]         DeflaterEngine.cs:417-439
//   k_match   (K2)  DeflaterEngine.FindLongestMatch, for every position   DeflaterEngine.cs:474-612
//   k_parse   (K3)  DeflaterEngine.DeflateSlow state machine              DeflaterEngine.cs:741-855
//   k_plan    (K4)  DeflaterHuffman.FlushBlock up to the type decision    DeflaterHuffman.cs:788-857
//   k_scan    (K5)  bit position of every block; Deflater flush padding   Deflater.cs:486-517
//   k_emit    (K6)  SendAllTrees / CompressBlock / FlushStoredBlock       DeflaterHuffman.cs:676-779
#include <cuda_pipeline.h>

#include "b200z_internal.cuh"
#include "b200z_tma.cuh"

namespace b200z {

constexpr int kRun = 65536;    // positions per k_links warp
constexpr int kTile = 32768;   // positions per k_match CTA
constexpr int kTileData = 2 * kTile + 320; // bytes of window staged per tile (history + tile + max match + pad)
constexpr int kMatchThreads = 1024;
constexpr int kMatchClasses = 16; // expected-walk-length classes of k_match (0 = nothing to search)
constexpr uint32_t kNoLink = 0xFFFFu; // k_match's staged link entry for "no predecessor": exceeds kMaxDist from any distance

// ------------------------------------------------------------------------------------------------
// K1: link[p] = distance from p to the previous inserted position with the same hash (0 = none / too far).
// One warp per run of kRun positions, 32 positions per step; a 16-bit head table in shared memory, re-based
// every 32768 positions exactly like SlideWindow (DeflaterEngine.cs:441-462) so that entries stay unambiguous.
// ------------------------------------------------------------------------------------------------
// lanes holding the same 15-bit hash, from 16 ballots (MATCH.ANY showed ~360 cycles of latency per step in ncu)
__device__ __forceinline__ uint32_t same_hash_mask(uint32_t h, bool valid, int lane) {
	uint32_t eq = __ballot_sync(0xffffffffu, valid);
#pragma unroll
	for (int b = 0; b < 15; b++) {
		const bool bit = (h >> b) & 1u;
		const uint32_t bal = __ballot_sync(0xffffffffu, bit);
		eq &= bit ? bal : ~bal;
	}
	return valid ? eq : (1u << lane);
}

// The head table is a serial dependency chain (every step reads what the previous step wrote), so the CTA splits the work:
// four PRODUCER warps compute, for groups of 32 positions, everything that does not depend on the table -- hash, validity,
// the nearest lower lane with the same hash, whether the lane is the last of its hash in the group -- and leave one word
// per position in shared memory; the CONSUMER warp then only does  read word -> read head -> write head -> store link.
// ncu before the split: one warp did both, ~570 cycles per step, 4 % of the SM's warp slots occupied.
constexpr int kLinkChunk = 512;                   // positions per hand-over between producers and consumer
constexpr int kLinkProducers = 8;
constexpr int kLinkThreads = 32 * (1 + kLinkProducers); // warp 0 consumes, the others produce
constexpr int kLinkRebase = 16384;                // head entries are re-based this often (see below)
constexpr int kLinksSmem = 65536 + 2 * kLinkChunk * 4;

__global__ void __launch_bounds__(kLinkThreads) k_links(const uint8_t *__restrict__ in, uint16_t *__restrict__ link,
                                                        const int64_t *__restrict__ in_off, const int64_t *__restrict__ in_len,
                                                        const int2 *__restrict__ run_desc, const uint32_t *__restrict__ hist,
                                                        const uint8_t *__restrict__ hmask, const int64_t *__restrict__ hm_off,
                                                        uint32_t run_len) {
	extern __shared__ __align__(16) uint8_t lsm[];
	uint16_t *head = reinterpret_cast<uint16_t *>(lsm);             // 32768 entries: position - winbase + 1, 0 = empty
	uint32_t *info = reinterpret_cast<uint32_t *>(lsm + 65536);     // two buffers of kLinkChunk words
	const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
	const int2 rd = run_desc[blockIdx.x];
	const uint32_t n = (uint32_t)in_len[rd.x];
	const uint8_t *data = in + in_off[rd.x];
	uint16_t *lnk = link + in_off[rd.x];
	const uint32_t start = (uint32_t)rd.y;
	const uint32_t run_end = (n - start > run_len) ? start + run_len : n; // run_len: kRun, or what B200Z_LINK_RUN asked for
	const uint32_t warm = start >= 32768u ? start - 32768u : 0u;
	// history (preset dictionary / earlier segments of the same stream): positions the reference never inserted
	// (the last two of a dictionary, DeflaterEngine.cs:217-226, or of a flushed segment, trap T9) are masked
	const uint32_t H = hist[rd.x];
	const uint8_t *hm = hmask + hm_off[rd.x];
	for (int i = threadIdx.x; i < 16384; i += kLinkThreads) reinterpret_cast<uint32_t *>(head)[i] = 0;
	uint32_t winbase = warm;
	auto produce = [&](uint32_t cb, int which) {
		// all of the warp's loads first (they are independent), then the ballots
		constexpr int G = kLinkChunk / 32 / kLinkProducers; // groups per producer warp and chunk
		uint32_t hh[G];
		bool vv[G];
#pragma unroll
		for (int j = 0; j < G; j++) {
			const uint32_t p = cb + 32u * (uint32_t)(warp - 1 + kLinkProducers * j) + lane;
			bool valid = p + 2 < n; // InsertString only while lookahead >= MIN_MATCH (DeflaterEngine.cs:782, :819)
			uint32_t h = 0;
			if (p + 2 < n) h = hash3(__ldg(data + p), __ldg(data + p + 1), __ldg(data + p + 2));
			if (p < H && valid) valid = __ldg(hm + p) == 0;
			hh[j] = h;
			vv[j] = valid;
		}
#pragma unroll
		for (int j = 0; j < G; j++) {
			const uint32_t g = (uint32_t)(warp - 1 + kLinkProducers * j);
			if (cb + 32u * g >= run_end) break;
			const uint32_t h = hh[j];
			const bool valid = vv[j];
			const uint32_t mask = same_hash_mask(h, valid, lane);
			const uint32_t lower = mask & ((1u << lane) - 1u);
			uint32_t w = h;
			if (valid) {
				w |= 1u << 15;
				if (lower) w |= (1u << 16) | ((uint32_t)(31 - __clz(lower)) << 17);
				if ((mask >> lane) == 1u) w |= 1u << 22;
			}
			info[which * kLinkChunk + 32u * g + lane] = w;
		}
	};
	if (warp > 0) produce(warm, 0);
	__syncthreads();
	int which = 0;
	for (uint32_t cb = warm; cb < run_end; cb += kLinkChunk, which ^= 1) {
		// The 16-bit entries are kept unambiguous like SlideWindow does (DeflaterEngine.cs:441-462), but in steps of 16384:
		// before a chunk starting 49152 or more past winbase, every entry drops by 16384 and entries that cannot be
		// within MAX_DIST of any position still to come (older than cb - 32768) vanish.  Which entries survive beyond
		// MAX_DIST is irrelevant: link[] only keeps distances <= MAX_DIST.
		if (cb - winbase >= 49152u) {
			for (int i = threadIdx.x; i < 16384; i += kLinkThreads) {
				uint32_t v = reinterpret_cast<uint32_t *>(head)[i];
				uint32_t lo = v & 0xFFFFu, hi = v >> 16;
				lo = lo > (uint32_t)kLinkRebase ? lo - kLinkRebase : 0u;
				hi = hi > (uint32_t)kLinkRebase ? hi - kLinkRebase : 0u;
				reinterpret_cast<uint32_t *>(head)[i] = lo | (hi << 16);
			}
			winbase += kLinkRebase;
			__syncthreads();
		}
		if (warp == 0) {
			const uint32_t cend = (run_end - cb > (uint32_t)kLinkChunk) ? cb + kLinkChunk : run_end;
			const uint32_t *ib = info + which * kLinkChunk;
			uint32_t w = ib[lane];
			for (uint32_t base = cb; base < cend; base += 32) {
				const uint32_t p = base + lane;
				const uint32_t wn = ib[(base + 32 - cb + lane) & (kLinkChunk - 1)]; // next group's word (unused after the last)
				// branch-free: every lane reads head[h] (h = 0 for lanes without a hash), the selects sort it out
				const uint32_t h = w & 0x7FFFu;
				const uint32_t v = head[h];
				const bool valid = (w >> 15) & 1u;
				uint32_t q = v ? winbase + v - 1 : 0xFFFFFFFFu;
				if ((w >> 16) & 1u) q = base + ((w >> 17) & 31u);
				__syncwarp();
				if (valid && ((w >> 22) & 1u)) head[h] = (uint16_t)(p - winbase + 1);
				__syncwarp();
				const uint32_t d = (valid && q != 0xFFFFFFFFu) ? p - q : 0u;
				if (p >= start && p < run_end) lnk[p] = (d <= (uint32_t)kMaxDist) ? (uint16_t)d : (uint16_t)0;
				w = wn;
			}
		} else if (cb + kLinkChunk < run_end) {
			produce(cb + kLinkChunk, which ^ 1);
		}
		__syncthreads();
	}
}

// ------------------------------------------------------------------------------------------------
// K2: per-position match table.  One CTA per 32 KiB tile; the tile's 64 KiB data window and the window's link
// entries are staged in shared memory (192 KiB), then each thread walks the chains of 32 positions.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kMatchThreads, 1)
    k_match(const uint8_t *__restrict__ in, const uint16_t *__restrict__ link, uint2 *__restrict__ mt,
            const int64_t *__restrict__ in_off, const int64_t *__restrict__ in_len, const int2 *__restrict__ tile_desc,
            const uint32_t *__restrict__ hist, const int64_t *__restrict__ bias, uint32_t *__restrict__ scratch, LevelParams lp) {
	extern __shared__ __align__(16) uint8_t smem[];
	uint8_t *s_data = smem;
	uint16_t *s_link = reinterpret_cast<uint16_t *>(smem + kTileData);
	const int2 td = tile_desc[blockIdx.x];
	const uint32_t n = (uint32_t)in_len[td.x];
	const int64_t off = in_off[td.x];
	const uint8_t *data = in + off;
	const uint16_t *lnk = link + off;
	const uint32_t t0 = (uint32_t)td.y;
	const uint32_t t1 = (n - t0 > (uint32_t)kTile) ? t0 + kTile : n;
	const uint32_t w0 = t0 >= (uint32_t)kTile ? t0 - kTile : 0u;
	uint32_t dend = t1 + 272;
	if (dend > n) dend = n;
	// Stage the tile's 64 KiB data window and its link entries (w0 and the slot base are 16-byte aligned).  The bulk of both
	// goes through the TMA engine: one thread arms an mbarrier with the byte count and issues cp.async.bulk copies, the
	// CTA waits on the barrier; the tails that are not multiples of 16 bytes are covered by scalar loops meanwhile.
	__shared__ BulkBarrier s_bar;
	if (threadIdx.x == 0) bulk_barrier_init(&s_bar);
	__syncthreads();
	{
		const uint32_t nbytes = dend - w0;
		const uint32_t nvec = nbytes >> 4;
		const uint32_t nl = t1 - w0;
		const uint32_t nlv = nl >> 3;
		if (threadIdx.x == 0) {
			bulk_expect(&s_bar, 16u * (nvec + nlv));
			bulk_copy_start(&s_bar, s_data, data + w0, 16u * nvec);
			bulk_copy_start(&s_bar, s_link, lnk + w0, 16u * nlv);
		}
		for (uint32_t i = (nvec << 4) + threadIdx.x; i < nbytes; i += kMatchThreads) s_data[i] = data[w0 + i];
		for (uint32_t i = (nlv << 3) + threadIdx.x; i < nl; i += kMatchThreads) s_link[i] = lnk[w0 + i];
	}
	bulk_wait(&s_bar, 0);
	__syncthreads();
	// k_links writes 0 for "no predecessor"; here it becomes kNoLink, so that the end of a chain and the T7 limit are one test,
	// dist + l2 >= kMaxDist.  (The entry past an odd nl is never read.)
	for (uint32_t i = threadIdx.x; i < (t1 - w0 + 1) / 2; i += kMatchThreads) {
		const uint32_t v = reinterpret_cast<uint32_t *>(s_link)[i];
		reinterpret_cast<uint32_t *>(s_link)[i] = v | ((v & 0xFFFFu) ? 0u : kNoLink) | ((v >> 16) ? 0u : kNoLink << 16);
	}
	__shared__ uint32_t s_cls[2][kMatchClasses];
	if (threadIdx.x < 2 * kMatchClasses) (&s_cls[0][0])[threadIdx.x] = 0;
	__syncthreads(); // the class pass reads entries other threads rewrote
	uint2 *out = mt + off;
	// match_search() of b200z_core.cuh with the byte-wise extension loop replaced by 4-byte compares on aligned
	// shared-memory words (ncu: the byte loop ran with ~2 of 32 lanes active and took ~30 % of the kernel).
	const uint32_t chain = (uint32_t)lp.chain, budgetB = chain >> 2;
	const uint32_t H = hist[td.x];            // positions below H are history: candidates only
	const uint32_t ab = (uint32_t)bias[td.x]; // absolute stream offset of buffer position 0 (window-slide phase, trap T8)
	// ---- order the tile's positions by expected chain length ----
	// A warp runs as long as its longest chain walk (ncu: 13 of 32 lanes active in the candidate loop).  So the positions
	// are bucketed by an estimate of their walk length (the first eight hops are exact, beyond that their hop density
	// extrapolated over the window) and handed to the threads longest first: warps then hold walks of similar length.
	// The order only decides who computes what; every position's result is unchanged.
	// (Measured in round 2 and dropped: the walks as a flat state machine -- one candidate test or four bytes of extension per
	// lane and iteration, free lanes refilled from the ordered list eight at a time.  Bit-exact, 41.5 ms instead of 21.2 ms on
	// the bench workload: every iteration pays for every state's code.  profiles/README.md.)
	uint16_t *order = reinterpret_cast<uint16_t *>(scratch + off + t0); // 4 bytes per position are free here until k_parse_gather
	uint32_t cw[4] = {0u, 0u, 0u, 0u};                                   // 32 x 4 bits: this thread's classes
	const int lane = threadIdx.x & 31;
#pragma unroll
	for (int k = 0; k < kTile / kMatchThreads; k++) {
		const uint32_t p = t0 + threadIdx.x + (uint32_t)k * kMatchThreads;
		uint32_t cls = 0;
		if (p < t1 && p >= H) {
			const uint32_t la = n - p;
			const uint32_t d = la >= (uint32_t)kMinMatch ? (uint32_t)s_link[p - w0] : kNoLink;
			if (d > (uint32_t)kMaxDist - (is_slide_pos(p + ab) ? 1u : 0u)) out[p] = make_uint2(0u, 0u); // DeflaterEngine.cs:788 + trap T8
			else {
				const uint32_t is = p - w0;
				uint32_t dist = d, hops = 1;
				while (hops < 8) {
					const uint32_t l2 = s_link[is - dist];
					if (dist + l2 >= (uint32_t)kMaxDist) break;
					dist += l2;
					++hops;
				}
				if (hops < 8) cls = hops <= 1 ? 1u : hops <= 2 ? 2u : hops <= 4 ? 3u : hops <= 6 ? 4u : 5u;
				else {
					uint32_t est = (8u * (uint32_t)kMaxDist) / dist; // candidates if the chain stays this dense
					if (est > chain) est = chain;
					cls = est <= 11 ? 6u : est <= 16 ? 7u : est <= 23 ? 8u : est <= 32 ? 9u : est <= 45 ? 10u : est <= 64 ? 11u
					      : est <= 91 ? 12u : est <= 128 ? 13u : est <= 512 ? 14u : 15u;
				}
			}
		}
		const uint32_t peers = __match_any_sync(0xffffffffu, cls);
		if (cls && lane == __ffs((int)peers) - 1) atomicAdd(&s_cls[0][cls], (uint32_t)__popc(peers));
		cw[k >> 3] |= cls << ((k & 7) * 4);
	}
	__syncthreads();
	uint32_t total = 0;
	{
		// class bases, longest walks first
		uint32_t b = 0;
		uint32_t mine = 0;
		for (int c = kMatchClasses - 1; c >= 1; c--) {
			if ((int)threadIdx.x == c) mine = b;
			b += s_cls[0][c];
		}
		total = b;
		__syncthreads();
		if (threadIdx.x >= 1 && threadIdx.x < kMatchClasses) s_cls[1][threadIdx.x] = mine;
		__syncthreads();
	}
#pragma unroll
	for (int k = 0; k < kTile / kMatchThreads; k++) {
		const uint32_t cls = (cw[k >> 3] >> ((k & 7) * 4)) & 15u;
		const uint32_t peers = __match_any_sync(0xffffffffu, cls);
		uint32_t slot = 0;
		const int leader = __ffs((int)peers) - 1;
		if (cls && lane == leader) slot = atomicAdd(&s_cls[1][cls], (uint32_t)__popc(peers));
		slot = __shfl_sync(0xffffffffu, slot, leader);
		if (cls) order[slot + (uint32_t)__popc(peers & ((1u << lane) - 1u))] = (uint16_t)(threadIdx.x + (uint32_t)k * kMatchThreads);
	}
	__syncthreads();
	// The walk keeps two running byte offsets into shared memory, both moved by each hop: icm, of the candidate's byte c[m], and il,
	// of the candidate's link entry (il = 2 * ic); the next hop's link is loaded before the quick reject, so the two shared-memory
	// latencies overlap.  The end of the chain (kNoLink) and the T7 limit are the one test il <= ilmin.  The budget is a countdown:
	// `left` candidates of the B segment (chain / 4), then B's snapshot and `rest` candidates of the A segment.
	const uint8_t *lb = reinterpret_cast<const uint8_t *>(s_link);
	for (uint32_t i = threadIdx.x; i < total; i += kMatchThreads) {
		const uint32_t p = t0 + (uint32_t)__ldcg(&order[i]);
		const uint32_t la = n - p;
		const uint32_t maxlen = la < (uint32_t)kMaxMatch ? la : (uint32_t)kMaxMatch;
		const uint32_t nice = la < (uint32_t)lp.nice ? la : (uint32_t)lp.nice;
		const uint32_t is = p - w0;
		const uint8_t *sp = s_data + is;
		// every position in the order has a first candidate: the class pass gave the others class 0
		const int ic0 = (int)is - (int)s_link[is];
		int icm = ic0 + (kMinMatch - 1), il = 2 * ic0;
		const int ilmin = 2 * ((int)is - kMaxDist); // chain entries need distance < 32506 (T7)
		uint32_t m = kMinMatch - 1, bd = 0, resB = 0;
		bool haveB = false;
		uint32_t left = budgetB ? budgetB : chain, rest = chain - left;
		const uint32_t s0 = sp[0], s1 = sp[1];
		uint32_t scan_end1 = s1, scan_end = sp[2];
		// bytes 2..9 of the scan string stay in registers: most extensions end inside them
		uint32_t sw0, sw1;
		{
			const uint32_t as = is + 2;
			const uint32_t *ws = reinterpret_cast<const uint32_t *>(s_data + (as & ~3u));
			const uint32_t w1 = ws[1], sh = (as & 3u) * 8u;
			sw0 = __funnelshift_r(ws[0], w1, sh);
			sw1 = __funnelshift_r(w1, ws[2], sh);
		}
		for (;;) { // the B segment, then the A segment
			for (;;) { // one candidate
				const uint32_t l2 = *reinterpret_cast<const uint16_t *>(lb + il);
				if (s_data[icm] == scan_end && s_data[icm - 1] == scan_end1) {
					const uint32_t ic = (uint32_t)(il >> 1);
					const uint8_t *c = s_data + ic;
					if (c[0] == s0 && c[1] == s1) {
						uint32_t l = 2;
						if (maxlen >= 10) {
							const uint32_t ac = ic + 2;
							const uint32_t *wc = reinterpret_cast<const uint32_t *>(s_data + (ac & ~3u));
							const uint32_t w1 = wc[1], sh = (ac & 3u) * 8u;
							uint32_t x = __funnelshift_r(wc[0], w1, sh) ^ sw0;
							if (x) {
								l = 2 + ((uint32_t)(__ffs((int)x) - 1) >> 3);
								goto lcp_done;
							}
							x = __funnelshift_r(w1, wc[2], sh) ^ sw1;
							if (x) {
								l = 6 + ((uint32_t)(__ffs((int)x) - 1) >> 3);
								goto lcp_done;
							}
							l = 10;
						}
						while (l + 4 <= maxlen) {
							const uint32_t ac = ic + l, as = is + l;
							const uint32_t *wc = reinterpret_cast<const uint32_t *>(s_data + (ac & ~3u));
							const uint32_t *ws = reinterpret_cast<const uint32_t *>(s_data + (as & ~3u));
							const uint32_t x = __funnelshift_r(wc[0], wc[1], (ac & 3u) * 8u) ^ __funnelshift_r(ws[0], ws[1], (as & 3u) * 8u);
							if (x) {
								l += (uint32_t)(__ffs((int)x) - 1) >> 3;
								goto lcp_done;
							}
							l += 4;
						}
						while (l < maxlen && c[l] == sp[l]) ++l;
					lcp_done:
						if (l > m) {
							m = l;
							bd = is - ic;
							if (m >= nice) goto walk_done;
							scan_end1 = sp[m - 1];
							scan_end = sp[m];
							icm = (int)(ic + m);
						}
					}
				}
				icm -= (int)l2;
				il -= 2 * (int)l2;
				if ((il <= ilmin) | (--left == 0)) break;
			}
			if (il <= ilmin || rest == 0) break;
			resB = m >= (uint32_t)kMinMatch ? pack_match(m, bd) : 0u; // B: the first chain / 4 candidates
			haveB = true;
			left = rest;
			rest = 0;
		}
	walk_done:
		const uint32_t resA = m >= (uint32_t)kMinMatch ? pack_match(m, bd) : 0u;
		out[p] = make_uint2(resA, haveB ? resB : resA);
	}
}

// ------------------------------------------------------------------------------------------------
// K3: the lazy parse (DeflateSlow's state machine, DeflaterEngine.cs:741-855), parallel at three levels.
//
//  lanes   : a ROUND is 32 segments x kSeg positions.  The round's table entries and bytes are staged in shared memory
//            (cp.async), every lane parses its own segment starting from a guessed clean state, then each lane hands
//            its exit state to the next lane as that lane's entry; lanes whose entry changed parse again.  Lane 0's
//            entry is the true carried state, so after k hand-offs the first k+1 lanes are exact; because the parse
//            re-synchronises within a few symbols the hand-offs normally stop changing anything after one iteration.
//            A final pass emits the round's symbols into the round's own slot.
//  chunks  : k_parse_chunk runs one warp per CHUNK of a stream (many chunks per stream, all concurrent), every chunk
//            but the first starting from a guessed clean state; per round it records the exit state and symbol count.
//  fix-up  : k_parse_fix walks the chunks of a stream in order and re-runs rounds of a chunk from the true entry state
//            until a round's exit state equals the recorded one -- from there on the speculative result stands.
//  gather  : k_parse_scan prefix-sums the rounds' symbol counts, k_parse_gather moves the symbols to their final
//            positions and records the block cuts (every 16384 symbols, DeflaterHuffman.cs:863).
// ------------------------------------------------------------------------------------------------
constexpr int kSegShift = 5;
constexpr int kSeg = 1 << kSegShift; // 32 positions per lane: 9.6 KiB of shared memory per warp, 22 warps per SM (64: 4.5 ms, 32: 3.2 ms, 16: 3.4 ms)
constexpr int kRound = 32 * kSeg;
constexpr int kParseWarm = 128; // positions a chunk parses in front of its first one to find its entry state (k_parse_chunk)
constexpr int kSegStride = kSeg + 2; // uint2 entries; +2 keeps 16-byte alignment for cp.async and staggers the banks
constexpr int kParseDatOff = 32 * kSegStride * 8;
constexpr int kParseSmem = kParseDatOff + kRound + 48;

struct ChunkDesc {
	int32_t stream;
	uint32_t c0, c1; // positions [c0, c1) of the stream, c0 a multiple of kRound
};

__device__ __forceinline__ ParseCarry shfl_carry(const ParseCarry &c, int src) {
	ParseCarry r;
	r.st.p = __shfl_sync(0xffffffffu, c.st.p, src);
	r.st.mlen = __shfl_sync(0xffffffffu, c.st.mlen, src);
	r.st.mstart = __shfl_sync(0xffffffffu, c.st.mstart, src);
	r.st.prevAvail = __shfl_sync(0xffffffffu, c.st.prevAvail, src);
	r.last_top = __shfl_sync(0xffffffffu, c.last_top, src);
	return r;
}

__device__ __forceinline__ ParseCarry clean_carry(uint32_t p) {
	ParseCarry c;
	parse_init(c.st);
	c.st.p = p;
	c.last_top = p;
	return c;
}

struct RoundRec { // what a round leaves behind (5 + 1 words)
	uint32_t p, mlen, mstart, prevAvail, last_top, cnt;
};
__device__ __forceinline__ ParseCarry rec_carry(const RoundRec &r) {
	ParseCarry c;
	c.st.p = r.p;
	c.st.mlen = r.mlen;
	c.st.mstart = r.mstart;
	c.st.prevAvail = r.prevAvail;
	c.last_top = r.last_top;
	return c;
}

// One round [base, base + kRound) of a stream, entered with `carry` (uniform across the warp; updated to the round's
// exit state).  The round's symbols go to sround[0 .. cnt).  Returns cnt (uniform).
__device__ __forceinline__ uint32_t parse_round(uint8_t *smem, const uint8_t *data, const uint16_t *lnk, const uint2 *tab,
                                                uint32_t n, uint32_t H, uint32_t ab, uint32_t base, const LevelParams &lp,
                                                int strategy, ParseCarry &carry, uint32_t *sround) {
	uint2 *s_tab = reinterpret_cast<uint2 *>(smem);
	uint8_t *s_dat = smem + kParseDatOff; // s_dat[16 + i] = byte at position base + i (16 bytes of history in front)
	const int lane = threadIdx.x & 31;
	const uint32_t rn = (n - base > (uint32_t)kRound) ? (uint32_t)kRound : n - base;
	__syncwarp();
	// stage the round with 16-byte async copies (LDGSTS): all of them are in flight at once, no register staging
	for (uint32_t i = 2 * lane; i + 1 < rn; i += 64)
		__pipeline_memcpy_async(&s_tab[(i >> kSegShift) * kSegStride + (i & (kSeg - 1))], &tab[base + i], 16);
	{
		// bytes [base - 16, base + rn) rounded up to 16 (the input slot has 16 bytes of slack behind n)
		const uint32_t c0 = base ? 0u : 1u, c1 = (16 + rn + 15) >> 4;
		for (uint32_t c = c0 + lane; c < c1; c += 32) __pipeline_memcpy_async(s_dat + 16 * c, data + base - 16 + 16 * c, 16);
	}
	__pipeline_commit();
	if ((rn & 1) && lane == 0) s_tab[((rn - 1) >> kSegShift) * kSegStride + ((rn - 1) & (kSeg - 1))] = tab[base + rn - 1];
	__pipeline_wait_prior(0);
	__syncwarp();
	const uint32_t seg_end = base + (uint32_t)(lane + 1) * kSeg;
	auto tabf = [&](uint32_t p, uint32_t &a, uint32_t &b) {
		const uint32_t i = p - base;
		const uint2 t = s_tab[(i >> kSegShift) * kSegStride + (i & (kSeg - 1))];
		a = t.x;
		b = t.y;
	};
	auto bytef = [&](uint32_t q) { return (uint32_t)s_dat[q + 16 - base]; };
	auto slowf = [&](uint32_t p, uint32_t m0, uint32_t budget) { return match_search_above(data, lnk, p, n, m0, budget, ab); };
	ParseCarry entry, ex;
	if (lane == 0) entry = carry;
	else {
		const uint32_t ss = base + (uint32_t)lane * kSeg;
		entry = clean_carry(ss > H ? ss : H); // history positions are never parsed; the state at H is exactly "clean"
	}
	ex = entry;
	uint32_t cnt = 0;
	bool changed = true;
	const uint32_t lim = seg_end < n ? seg_end : n;
	for (int it = 0; it < 34; it++) {
		// all lanes step together and re-converge every iteration (a per-lane loop would leave them diverged)
		if (changed) {
			ex = entry;
			cnt = 0;
		}
		bool act = changed && ex.st.p < lim;
		while (__any_sync(0xffffffffu, act)) {
			if (act) {
				ex.last_top = ex.st.p;
				uint32_t s2;
				cnt += (uint32_t)parse_step(ex.st, n, lp, strategy, tabf, bytef, slowf, s2);
				act = ex.st.p < lim;
			}
			__syncwarp();
		}
		const ParseCarry ne = shfl_carry(ex, lane == 0 ? 0 : lane - 1);
		changed = false;
		if (lane > 0) {
			changed = !carry_equal(ne, entry);
			entry = ne;
		}
		if (!__any_sync(0xffffffffu, changed)) break;
	}
	// final pass: emit at prefix-summed offsets inside the round's slot
	uint32_t incl = cnt;
	for (int o = 1; o < 32; o <<= 1) {
		const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
		if (lane >= o) incl += t;
	}
	uint32_t idx = incl - cnt;
	ParseCarry c = entry;
	{
		bool act = c.st.p < lim;
		while (__any_sync(0xffffffffu, act)) {
			if (act) {
				c.last_top = c.st.p;
				uint32_t s2;
				if (parse_step(c.st, n, lp, strategy, tabf, bytef, slowf, s2)) sround[idx++] = s2;
				act = c.st.p < lim;
			}
			__syncwarp();
		}
	}
	carry = shfl_carry(c, 31);
	return __shfl_sync(0xffffffffu, incl, 31);
}

__global__ void __launch_bounds__(32)
    k_parse_chunk(const uint8_t *__restrict__ in, const uint16_t *__restrict__ link, const uint2 *__restrict__ mt,
                  uint32_t *__restrict__ sym_local, const int64_t *__restrict__ in_off, const int64_t *__restrict__ in_len,
                  const ChunkDesc *__restrict__ chunks, const uint32_t *__restrict__ rnd_off, RoundRec *__restrict__ recs,
                  RoundRec *__restrict__ ents, const uint32_t *__restrict__ hist, const int64_t *__restrict__ bias, LevelParams lp,
                  int strategy, int warm) {
	extern __shared__ __align__(16) uint8_t smem[];
	const ChunkDesc cd = chunks[blockIdx.x];
	const uint32_t n = (uint32_t)in_len[cd.stream];
	const int64_t off = in_off[cd.stream];
	RoundRec *rr = recs + rnd_off[cd.stream];
	const uint32_t H = hist[cd.stream], ab = (uint32_t)bias[cd.stream];
	// exact for the first chunk (DeflaterEngine.Reset :234-253; also the state right after a dictionary or a flush).  Every
	// other chunk parses kParseWarm positions in front of its first one from a clean state (lane 0, straight from global
	// memory): DeflateSlow's state re-synchronises within a few symbols, so the state this reaches at c0 is the true one at
	// 99.8 % of the boundaries (tools/tile_fixup.cpp).  It is recorded; k_parse_fix compares it with the exit of the chunk in
	// front and parses again only where they differ.
	ParseCarry carry = clean_carry(cd.c0 > H ? cd.c0 : H);
	if (cd.c0 > H && warm > 0) {
		if (threadIdx.x == 0) {
			const uint8_t *data = in + off;
			const uint16_t *lnk = link + off;
			const uint2 *tab = mt + off;
			const uint32_t ws = cd.c0 - H > (uint32_t)warm ? cd.c0 - (uint32_t)warm : H;
			ParseCarry w = clean_carry(ws);
			auto tabg = [&](uint32_t p, uint32_t &a, uint32_t &b) {
				const uint2 t = tab[p];
				a = t.x;
				b = t.y;
			};
			auto byteg = [&](uint32_t q) { return (uint32_t)data[q]; };
			auto slowg = [&](uint32_t p, uint32_t m0, uint32_t budget) { return match_search_above(data, lnk, p, n, m0, budget, ab); };
			while (w.st.p < cd.c0) {
				w.last_top = w.st.p;
				uint32_t s2;
				parse_step(w.st, n, lp, strategy, tabg, byteg, slowg, s2);
			}
			carry = w;
		}
		carry = shfl_carry(carry, 0);
	}
	if (threadIdx.x == 0) {
		RoundRec e;
		e.p = carry.st.p;
		e.mlen = carry.st.mlen;
		e.mstart = carry.st.mstart;
		e.prevAvail = carry.st.prevAvail;
		e.last_top = carry.last_top;
		e.cnt = 0;
		ents[rnd_off[cd.stream] + cd.c0 / kRound] = e;
	}
	for (uint32_t base = cd.c0; base < cd.c1; base += kRound) {
		const uint32_t cnt = parse_round(smem, in + off, link + off, mt + off, n, H, ab, base, lp, strategy, carry, sym_local + off + base);
		if (threadIdx.x == 0) {
			RoundRec r;
			r.p = carry.st.p;
			r.mlen = carry.st.mlen;
			r.mstart = carry.st.mstart;
			r.prevAvail = carry.st.prevAvail;
			r.last_top = carry.last_top;
			r.cnt = cnt;
			rr[base / kRound] = r;
		}
	}
}

__global__ void __launch_bounds__(32)
    k_parse_fix(const uint8_t *__restrict__ in, const uint16_t *__restrict__ link, const uint2 *__restrict__ mt,
                uint32_t *__restrict__ sym_local, const int64_t *__restrict__ in_off, const int64_t *__restrict__ in_len,
                const uint32_t *__restrict__ rnd_off, RoundRec *__restrict__ recs, const RoundRec *__restrict__ ents, uint32_t chunk,
                const uint32_t *__restrict__ hist, const int64_t *__restrict__ bias, LevelParams lp, int strategy) {
	extern __shared__ __align__(16) uint8_t smem[];
	const int stream = blockIdx.x;
	const uint32_t n = (uint32_t)in_len[stream];
	if (n <= chunk) return; // a single chunk was parsed from the true initial state
	const int64_t off = in_off[stream];
	RoundRec *rr = recs + rnd_off[stream];
	const RoundRec *en = ents + rnd_off[stream];
	const uint32_t H = hist[stream], ab = (uint32_t)bias[stream];
	const uint32_t nchunks = (n + chunk - 1) / chunk;
	const int lane = threadIdx.x;
	// Boundaries are checked 32 at a time: the entry a chunk used against the exit of the chunk in front (exact by induction
	// once every boundary before it has been checked).  The first that differs is parsed again from the true state until a
	// round's exit equals the recorded one; the scan then goes on behind it (its own exit may have changed).
	uint32_t k0 = 1;
	while (k0 < nchunks) {
		const uint32_t k = k0 + (uint32_t)lane;
		bool bad = false;
		if (k < nchunks) {
			const uint32_t c0 = k * chunk;
			const ParseCarry truth = rec_carry(rr[c0 / kRound - 1]);
			ParseCarry used = rec_carry(en[c0 / kRound]);
			used.last_top = truth.last_top; // irrelevant here: the chunk processes at least one loop top
			bad = !carry_equal(truth, used);
		}
		const uint32_t mask = __ballot_sync(0xffffffffu, bad);
		if (!mask) {
			k0 += 32;
			continue;
		}
		const uint32_t kk = k0 + (uint32_t)(__ffs((int)mask) - 1);
		const uint32_t c0 = kk * chunk;
		const uint32_t c1 = (n - c0 > chunk) ? c0 + chunk : n;
		ParseCarry truth = rec_carry(rr[c0 / kRound - 1]);
		for (uint32_t base = c0; base < c1; base += kRound) {
			const ParseCarry old_exit = rec_carry(rr[base / kRound]);
			const uint32_t cnt = parse_round(smem, in + off, link + off, mt + off, n, H, ab, base, lp, strategy, truth, sym_local + off + base);
			__syncwarp();
			if (lane == 0) {
				RoundRec r;
				r.p = truth.st.p;
				r.mlen = truth.st.mlen;
				r.mstart = truth.st.mstart;
				r.prevAvail = truth.st.prevAvail;
				r.last_top = truth.last_top;
				r.cnt = cnt;
				rr[base / kRound] = r;
			}
			__syncwarp();
			if (carry_equal(truth, old_exit)) break; // re-synchronised: the rest of the chunk stands as parsed
		}
		__syncwarp();
		k0 = kk + 1;
	}
}

// exclusive scan of the rounds' symbol counts of one stream; also the end-of-stream bookkeeping
__global__ void __launch_bounds__(256)
    k_parse_scan(const uint8_t *__restrict__ in, const int64_t *__restrict__ in_off, const int64_t *__restrict__ in_len,
                 const uint32_t *__restrict__ rnd_off, const RoundRec *__restrict__ recs, uint32_t *__restrict__ rnd_symoff,
                 uint32_t *__restrict__ sym, uint32_t *__restrict__ nsyms, uint32_t *__restrict__ nblocks,
                 const uint32_t *__restrict__ blk_off, uint32_t *__restrict__ blk_start, uint32_t *__restrict__ blk_ptop,
                 const uint32_t *__restrict__ hist, int end_mode) {
	__shared__ uint32_t s_part[8];
	__shared__ uint32_t s_carry;
	const int stream = blockIdx.x;
	const uint32_t n = (uint32_t)in_len[stream];
	const uint32_t nr = (n + kRound - 1) / kRound;
	const RoundRec *rr = recs + rnd_off[stream];
	uint32_t *so = rnd_symoff + rnd_off[stream];
	if (threadIdx.x == 0) s_carry = 0;
	__syncthreads();
	for (uint32_t b = 0; b < nr; b += 256) {
		const uint32_t i = b + threadIdx.x;
		const uint32_t v = i < nr ? rr[i].cnt : 0u;
		uint32_t incl = v;
		for (int o = 1; o < 32; o <<= 1) {
			const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
			if ((threadIdx.x & 31) >= o) incl += t;
		}
		if ((threadIdx.x & 31) == 31) s_part[threadIdx.x >> 5] = incl;
		__syncthreads();
		uint32_t woff = 0;
		for (int k = 0; k < (int)(threadIdx.x >> 5); k++) woff += s_part[k];
		const uint32_t carry = s_carry;
		if (i < nr) so[i] = carry + woff + incl - v;
		__syncthreads();
		if (threadIdx.x == 255) s_carry = carry + woff + incl;
		__syncthreads();
	}
	if (threadIdx.x == 0) {
		uint32_t total = s_carry;
		const uint32_t H = hist[stream];
		ParseCarry fin = nr ? rec_carry(rr[nr - 1]) : clean_carry(H);
		uint32_t *bstart = blk_start + blk_off[stream];
		uint32_t *bptop = blk_ptop + blk_off[stream];
		bstart[0] = H;
		uint32_t nblk = total >> 14;
		const bool ended_full = end_mode == B200Z_END_FINISH && total > 0 && (total & (uint32_t)(kBlockSyms - 1)) == 0 && !fin.st.prevAvail;
		if (!ended_full) {
			// final flush at lookahead == 0 (DeflaterEngine.cs:750-768)
			if (fin.st.prevAvail) (sym + in_off[stream])[total++] = sym_lit(in[in_off[stream] + fin.st.p - 1]);
			bptop[nblk] = fin.last_top;
			++nblk;
		}
		nsyms[stream] = total;
		nblocks[stream] = nblk;
	}
}

// moves every round's symbols to their final place and records the block cuts that fall inside the round
__global__ void __launch_bounds__(128)
    k_parse_gather(const uint32_t *__restrict__ sym_local, uint32_t *__restrict__ sym, const int64_t *__restrict__ in_off,
                   const int64_t *__restrict__ in_len, const int2 *__restrict__ rnd_desc, const uint32_t *__restrict__ rnd_off,
                   const RoundRec *__restrict__ recs, const uint32_t *__restrict__ rnd_symoff, const uint32_t *__restrict__ blk_off,
                   uint32_t *__restrict__ blk_start, uint32_t *__restrict__ blk_ptop, const uint32_t *__restrict__ hist) {
	const int2 d = rnd_desc[blockIdx.x]; // (stream, first round of this CTA's group of 4)
	const int64_t off = in_off[d.x];
	const uint32_t n = (uint32_t)in_len[d.x];
	const uint32_t nr = (n + kRound - 1) / kRound;
	const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
	const uint32_t r = (uint32_t)d.y + (uint32_t)w;
	if (r >= nr) return;
	const RoundRec *rr = recs + rnd_off[d.x];
	const uint32_t cnt = rr[r].cnt;
	const uint32_t dst0 = rnd_symoff[rnd_off[d.x] + r];
	const uint32_t *src = sym_local + off + r * (uint32_t)kRound;
	uint32_t *dst = sym + off + dst0;
	for (uint32_t i = lane; i < cnt; i += 32) dst[i] = src[i];
	// block cuts: global symbol index idx with (idx + 1) % 16384 == 0
	if (lane == 0 && cnt) {
		const uint32_t first_b = (dst0 + (uint32_t)kBlockSyms) >> 14;          // smallest b with b * 16384 - 1 >= dst0
		const uint32_t last_idx = dst0 + cnt - 1;
		if (first_b * (uint32_t)kBlockSyms - 1 <= last_idx) {
			// bytes covered before this round's first symbol: entry.p, minus the pending literal if there is one
			uint32_t bytes;
			if (r == 0) bytes = hist[d.x];
			else bytes = rr[r - 1].p - (rr[r - 1].prevAvail ? 1u : 0u);
			uint32_t *bstart = blk_start + blk_off[d.x];
			uint32_t *bptop = blk_ptop + blk_off[d.x];
			uint32_t nextb = first_b;
			for (uint32_t i = 0; i < cnt; i++) {
				const uint32_t s2 = src[i];
				const uint32_t L = sym_len(s2);
				bytes += L;
				if (dst0 + i + 1 == nextb * (uint32_t)kBlockSyms) {
					// the loop top at which the symbol was tallied: literal -> the position after it; match -> its start + 1
					bptop[nextb - 1] = sym_dist(s2) ? bytes - L + 1 : bytes;
					bstart[nextb] = bytes;
					++nextb;
				}
			}
		}
	}
}

// ------------------------------------------------------------------------------------------------
// Levels 1-4: DeflateFast.  The chains depend on the parse, so a stream is parsed serially by lane 0 with the
// reference's own head[]/prev[] tables (shared memory, 128 KiB); SlideWindow's table sweep is done by the whole warp.
// All streams of the batch run concurrently (one warp each).  Symbols and block cuts feed k_plan / k_scan / k_emit.
// ------------------------------------------------------------------------------------------------
constexpr int kFastSmem = 2 * 32768 * 2; // prev[] (+ head[] when a batch has no more streams than the GPU has SMs)

// eight window bytes starting at slot byte `a`, first byte in the low bits of lo (aligned words; the slot is 256-byte
// aligned and has 16 bytes of slack behind its data)
__device__ __forceinline__ void fast_load8(const uint8_t *__restrict__ in, uint32_t a, uint32_t &lo, uint32_t &hi) {
	const uint32_t *p = reinterpret_cast<const uint32_t *>(in + (a & ~3u));
	const uint32_t w0 = p[0], w1 = p[1], w2 = p[2];
	const uint32_t sh = (a & 3u) * 8u;
	lo = __funnelshift_r(w0, w1, sh);
	hi = __funnelshift_r(w1, w2, sh);
}

// The warp-wide group step of DeflateFast (DeflaterEngine.cs:651-739), `nl` consecutive loop tops at once.
//
// What makes DeflateFast serial is that a match longer than max_lazy leaves its inner positions out of the hash chains
// (:699-715); a literal or a match of at most max_lazy bytes inserts every position it covers.  So as long as no long match
// is taken, "every position of the group is a chain member" is the truth, and the searches of all loop tops can run at once:
// lane j takes window index s0 + j, its chain head is the nearest lower lane with the same hash (else head[]), links of
// group positions are written to prev[] up front (slots of positions further back than MAX_DIST are never read again), every
// lane runs FindLongestMatch from matchLen = 2 with the level's chain budget and remembers which group positions it
// tested (`used`).  The parse is replayed over the lanes' results in order by a cursor v that all lanes keep: a lane is
// resolved once its walk is complete; a long match at lane v takes positions v+1 .. v+len-1 out (set N) and ends their
// walks; a later lane whose walk touched N is not trusted -- the group ends in front of it and the next step starts there.
// Lanes behind a long match that never touched N saw exactly the chains the reference sees (a walk that read a link into N
// either tested that position -- then it is in `used` -- or had run out of budget).  At commit the links of the inserted
// positions are recomputed over the inserted lanes only, head[] gets the last inserted position of every hash, the visited
// lanes write their symbols in order.
//
// Latency is what this kernel pays for, so: a lane gathers up to four chain members before it loads any of them (one
// memory round trip per four candidates); a candidate that still matches after 16 bytes waits until its lane is the
// cursor and is then extended by the whole warp (8 bytes per lane) -- lanes inside a long repeat never get there, the match
// of the lane in front of them covers them first.
//
// s0 / la / nsym / total: the engine's strstart, lookahead, symbols in the block, symbols written (uniform over the warp; the
// caller keeps lane 0's FastEngine in step).  Returns 1 if the last action was a long match (UpdateHash is due, :712-714).
__device__ __forceinline__ int fast_lcp8(uint32_t alo, uint32_t ahi, uint32_t blo, uint32_t bhi) {
	uint32_t x = alo ^ blo;
	if (x) return (__ffs((int)x) - 1) >> 3;
	x = ahi ^ bhi;
	if (x) return 4 + ((__ffs((int)x) - 1) >> 3);
	return 8;
}

__device__ __forceinline__ int fast_group_step(const uint8_t *__restrict__ in, uint32_t woff, uint16_t *head, uint16_t *prev,
                                               const LevelParams &lp, int lane, int nl, int &s0, int &la, uint32_t &nsym,
                                               uint32_t *__restrict__ sout, uint32_t &total, int &last_h, int &match_start) {
	const uint32_t full = 0xffffffffu;
	const uint32_t lt = (1u << lane) - 1u;
	const int q = s0 + lane;
	const uint32_t qa = (uint32_t)q + woff;
	const bool active = lane < nl;
	uint32_t lo, hi;
	fast_load8(in, qa, lo, hi);
#if !defined(B200Z_EMU)
	// the bytes a later step starts from: one 128-byte line per lane pair, 2 KiB ahead (reads past the slot stay inside the
	// plan's input blob or its tail padding; a prefetch does not fault)
	if (la > 4096 && (lane & 1)) asm volatile("prefetch.global.L2 [%0];" ::"l"(in + ((qa + 2048u + 64u * (uint32_t)lane) & ~127u)));
#endif
	const uint32_t h = hash3(lo & 255u, (lo >> 8) & 255u, (lo >> 16) & 255u);
	const int hh = head[h];
	const uint32_t same = __match_any_sync(full, active ? h : (0x8000u | (uint32_t)lane));
	const uint32_t pm = same & lt;
	const int cand0 = pm ? s0 + (31 - __clz((int)pm)) : hh;
	if (active) prev[q & 32767] = (uint16_t)cand0;
	__syncwarp();

	// FindLongestMatch (:474-612) from matchLen = MIN_MATCH - 1: the longest common prefix with every chain member in chain
	// order, the first longest wins, stop at nice_length; the reference's scan_end tests only skip members that cannot win
	int best = kMinMatch - 1, bestc = 0, chain = lp.chain;
	uint32_t used = 0;
	const int limit = q - kMaxDist > 0 ? q - kMaxDist : 0;
	int cand = (active && cand0 != 0 && q - cand0 <= kMaxDist) ? cand0 : 0; // next chain member to gather (0: none left)
	bool go = cand != 0;    // the walk is not complete
	bool pend = false;      // the member at bi matches for >= 16 bytes and waits for the warp
	int c0 = 0, c1 = 0, c2 = 0, c3 = 0, nb = 0, bi = 0;
	uint32_t l0 = 0, h0 = 0, l1 = 0, h1 = 0, l2 = 0, h2 = 0, l3 = 0, h3 = 0;
	uint32_t visited = 0, N = 0;
	int v = 0, last_long = 0;
	bool stop = false;
	for (;;) {
		if (go && bi == nb) {
			// the next (up to) four members: `do test while ((cur = prev[cur]) > limit && --chain)`
			nb = 0;
			bi = 0;
#define B200Z_GATHER(C)                                                                                                           \
	if (cand) {                                                                                                                    \
		C = cand;                                                                                                                   \
		++nb;                                                                                                                       \
		const int nx = prev[cand & 32767];                                                                                          \
		cand = (nx > limit && --chain != 0) ? nx : 0;                                                                               \
	}
			B200Z_GATHER(c0)
			B200Z_GATHER(c1)
			B200Z_GATHER(c2)
			B200Z_GATHER(c3)
#undef B200Z_GATHER
			if (nb > 0) fast_load8(in, (uint32_t)c0 + woff, l0, h0);
			if (nb > 1) fast_load8(in, (uint32_t)c1 + woff, l1, h1);
			if (nb > 2) fast_load8(in, (uint32_t)c2 + woff, l2, h2);
			if (nb > 3) fast_load8(in, (uint32_t)c3 + woff, l3, h3);
			if (nb == 0) go = false;
		}
#define B200Z_TEST(K, C, CL, CH)                                                                                                 \
	if (go && !pend && bi == K && K < nb) {                                                                                        \
		if (C >= s0) used |= 1u << (C - s0);                                                                                        \
		int l = fast_lcp8(CL, CH, lo, hi);                                                                                          \
		if (l == 8) {                                                                                                               \
			uint32_t a0, a1, b0, b1;                                                                                                 \
			fast_load8(in, (uint32_t)C + woff + 8u, a0, a1);                                                                         \
			fast_load8(in, qa + 8u, b0, b1);                                                                                         \
			l += fast_lcp8(a0, a1, b0, b1);                                                                                          \
		}                                                                                                                           \
		if (l == 16) {                                                                                                              \
			pend = true;                                                                                                             \
		} else {                                                                                                                    \
			if (l > best) {                                                                                                          \
				best = l;                                                                                                             \
				bestc = C;                                                                                                            \
				if (best >= lp.nice) go = false;                                                                                      \
			}                                                                                                                        \
			bi = K + 1;                                                                                                              \
		}                                                                                                                           \
	}
		B200Z_TEST(0, c0, l0, h0)
		B200Z_TEST(1, c1, l1, h1)
		B200Z_TEST(2, c2, l2, h2)
		B200Z_TEST(3, c3, l3, h3)
#undef B200Z_TEST
		if (go && !pend && bi == nb && cand == 0) go = false; // every member tested
		// the cursor's lane is extended by the warp: lane k compares bytes 16 + 8k .. 16 + 8k + 7 (MAX_MATCH = 258 < 16 + 256)
		if (__shfl_sync(full, (int)pend, v)) {
			const int pc = bi == 0 ? c0 : bi == 1 ? c1 : bi == 2 ? c2 : c3;
			const uint32_t ca = (uint32_t)__shfl_sync(full, pc, v) + woff + 16u + 8u * (uint32_t)lane;
			const uint32_t sa = (uint32_t)(s0 + v) + woff + 16u + 8u * (uint32_t)lane;
			int first = 8;
			if (16 + 8 * lane < kMaxMatch) {
				uint32_t a0, a1, b0, b1;
				fast_load8(in, ca, a0, a1);
				fast_load8(in, sa, b0, b1);
				first = fast_lcp8(a0, a1, b0, b1);
			}
			const uint32_t mm = __ballot_sync(full, first < 8);
			const int fl = mm ? __ffs((int)mm) - 1 : 0;
			const int ff = __shfl_sync(full, first, fl);
			int ll = mm ? 16 + 8 * fl + ff : kMaxMatch;
			if (ll > kMaxMatch) ll = kMaxMatch;
			if (lane == v) {
				pend = false;
				if (ll > best) {
					best = ll;
					bestc = pc;
					if (best >= lp.nice) go = false;
				}
				++bi;
				if (go && bi == nb && cand == 0) go = false;
			}
		}
		// replay: the cursor passes every lane whose walk is complete
		const uint32_t fin = __ballot_sync(full, !go);
		if ((fin >> v) & 1u) {
			const uint32_t litm = __ballot_sync(full, active && best < kMinMatch);
			const uint32_t shortm = __ballot_sync(full, best >= kMinMatch && best <= lp.lazy);
			const uint32_t e0 = __ballot_sync(full, best & 1), e1 = __ballot_sync(full, best & 2), e2 = __ballot_sync(full, best & 4);
			uint32_t bad = N ? __ballot_sync(full, (used & N) != 0) : 0u;
			while (v < nl && ((fin >> v) & 1u)) {
				if ((bad >> v) & 1u) {
					stop = true;
					break;
				}
				if ((litm >> v) & 1u) {
					const uint32_t r = ~((litm & fin & ~bad) >> v); // a run of literals
					const int run = r ? __ffs((int)r) - 1 : 32 - v;
					visited |= (run >= 32 ? full : ((1u << run) - 1u)) << v;
					v += run;
					last_long = 0;
				} else if ((shortm >> v) & 1u) {
					const int L = (int)(((e0 >> v) & 1u) | (((e1 >> v) & 1u) << 1) | (((e2 >> v) & 1u) << 2));
					if (v + L > nl) { // its inner positions would need inserting behind the group: the next step takes it
						stop = true;
						break;
					}
					visited |= 1u << v;
					v += L;
					last_long = 0;
				} else {
					const int L = __shfl_sync(full, best, v);
					visited |= 1u << v;
					const int lo_b = v + 1, hi_b = v + L < 32 ? v + L : 32; // positions v+1 .. v+L-1 are not inserted
					if (hi_b > lo_b) N |= (hi_b >= 32 ? full : ((1u << hi_b) - 1u)) & ~((1u << lo_b) - 1u);
					if ((N >> lane) & 1u) { // covered: nobody will ask for this lane's result
						go = false;
						pend = false;
					}
					bad = __ballot_sync(full, (used & N) != 0);
					v += L;
					last_long = 1;
				}
			}
			if (stop || v >= nl) break;
		}
	}
	const int len = best >= kMinMatch ? best : 0;
	// commit
	const uint32_t below = v >= 32 ? full : ((1u << v) - 1u);
	const uint32_t ins = below & ~N & (nl >= 32 ? full : ((1u << nl) - 1u));
	const bool inserted = (ins >> lane) & 1u;
	if (inserted) {
		if (N) {
			const uint32_t pi = same & ins & lt;
			prev[q & 32767] = (uint16_t)(pi ? s0 + (31 - __clz((int)pi)) : hh);
		}
		if (((same & ins) >> lane) == 1u) head[h] = (uint16_t)q;
	}
	if ((visited >> lane) & 1u)
		sout[total + (uint32_t)__popc(visited & lt)] = len ? sym_match((uint32_t)len, (uint32_t)(q - bestc)) : sym_lit(lo & 255u);
	const uint32_t vm = __ballot_sync(full, ((visited >> lane) & 1u) && len != 0);
	if (vm) match_start = __shfl_sync(full, bestc, 31 - __clz((int)vm));
	if (!last_long) last_h = (int)__shfl_sync(full, h, (v - 1) & 31);
	const int nv = __popc(visited);
	total += (uint32_t)nv;
	nsym += (uint32_t)nv;
	s0 += v;
	la -= v;
	__syncwarp();
	return last_long;
}

// B200Z_PARSE_WARM=<positions> (0 .. 4096): how far in front of its first position a parse chunk starts (0: every chunk enters
// with the clean guess and k_parse_fix parses again at most boundaries, as in round 1; for tests and timing)
static int parse_warm() {
	const char *e = getenv("B200Z_PARSE_WARM");
	if (!e) return kParseWarm;
	const long v = atol(e);
	return v < 0 ? 0 : v > 4096 ? 4096 : (int)v;
}

// B200Z_FAST_GROUP=0 keeps every loop top on lane 0 (the serial statement; for measurements and for the tests that compare)
static int fast_group_enabled() {
	const char *e = getenv("B200Z_FAST_GROUP");
	return !(e && e[0] == '0');
}

// One stream's DeflateFast run by one warp.  head[] (32768 entries, read once per loop top) lives in the CTA's slot of a
// global pool and stays in L2; prev[] (read for every chain member) is the CTA's shared memory.
__device__ __forceinline__ void fast_stream(const int stream, const int lane, uint16_t *head, uint16_t *prev, const uint8_t *__restrict__ in,
                                            uint32_t *__restrict__ sym, const int64_t *__restrict__ in_off,
                                            const int64_t *__restrict__ in_len, uint32_t *__restrict__ nsyms,
                                            uint32_t *__restrict__ nblocks, const uint32_t *__restrict__ blk_off,
                                            uint32_t *__restrict__ blk_start, uint32_t *__restrict__ blk_ptop,
                                            const uint32_t *__restrict__ hist, const LevelParams &lp, int strategy, int end_mode,
                                            int prev_entries, const uint32_t *__restrict__ sched, const uint32_t *__restrict__ sched_off,
                                            const int32_t *__restrict__ undrained, uint8_t *const *__restrict__ fstate, int cont,
                                            int group) {
	// prev[] is indexed by window position & 32767; when no stream of the batch is longer than prev_entries - 2 bytes the
	// positions never reach prev_entries, so the table (and the CTA's shared-memory footprint) can be that much smaller
	// and more CTAs share an SM.  (Plans that carry engine state between segments use whole tables.)
	const uint32_t n = (uint32_t)in_len[stream];
	const int64_t off = in_off[stream];
	uint32_t *sout = sym + off;
	uint32_t *bstart = blk_start + blk_off[stream];
	uint32_t *bptop = blk_ptop + blk_off[stream];
	uint8_t *st = fstate[stream]; // engine state carried between the segments of this stream (b200z_history.engine_state)
	const bool resume = cont != 0 && st != nullptr;
	FastEngine e;
	if (resume) {
		// the stream goes on behind a Flush(): tables and scalars as the previous segment's run left them
		const uint4 *src = reinterpret_cast<const uint4 *>(st);
		for (int i = lane; i < 65536 / 16; i += 32) reinterpret_cast<uint4 *>(head)[i] = src[i];
		for (int i = lane; i < 65536 / 16; i += 32) reinterpret_cast<uint4 *>(prev)[i] = src[65536 / 16 + i];
		__syncwarp();
		FastCarry c = *reinterpret_cast<const FastCarry *>(st + 131072);
		fe_load(e, c, in + off, n, hist[stream], head, prev);
	} else {
		for (int i = lane; i < 65536 / 16; i += 32) reinterpret_cast<uint4 *>(head)[i] = make_uint4(0u, 0u, 0u, 0u);
		for (int i = lane; i < prev_entries / 2; i += 32) reinterpret_cast<uint32_t *>(prev)[i] = 0;
		__syncwarp();
		fe_init(e, in + off, n, head, prev);
		if (lane == 0) fe_set_dictionary(e, hist[stream]); // preset dictionary in front of the data (0 = none)
	}
	e.coop = group ? 2 : 1;
	// the SetInput schedule of the segment (fe_run in b200z_core.cuh is the serial statement of this loop)
	const uint32_t *cum = sched + sched_off[stream];
	const int nsched = (int)(sched_off[stream + 1] - sched_off[stream]);
	const int nc = nsched > 0 ? nsched : 1;
	const bool busy_last = undrained[stream] == 0;
	uint32_t seg_base = 0, seg_len = 0;
	if (lane == 0) {
		seg_base = e.inputOff;
		seg_len = 32768u * e.slides - 1u - e.woff + e.slot_len - e.inputOff;
		e.n = seg_base + (nsched > 0 ? cum[0] : seg_len);
	}
	uint32_t total = 0, nblk = 0;
#ifdef B200Z_FAST_STATS
	uint32_t st_steps = 0, st_pos = 0, st_lanes = 0;
#endif
	int ci = 0;
	int phase = (nc == 1 && !busy_last) ? 1 : 0; // 0: BUSY_STATE drain of chunk ci, 1: Flush()/Finish()
	bool in_deflate = false; // re-entering DeflateFast after a cooperative slide must not run FillWindow again
	const bool finish = end_mode == B200Z_END_FINISH;
	for (;;) {
		int r = kFeTrue;
		if (lane == 0) {
			bool filled = true;
			if (!in_deflate) filled = fe_fill_window(e);
			if (!filled) {
				r = kFeNeedSlide;
			} else {
				in_deflate = true;
				// engine.Deflate(flush, finish): canFlush = flush && inputOff == inputEnd (DeflaterEngine.cs:104-137)
				r = fe_deflate_fast(
				    e, phase == 1 && e.inputOff == e.n, phase == 1 && finish, lp, strategy, [&](uint32_t s2) { sout[total++] = s2; },
				    [&](uint32_t start, bool ok, bool) {
					    bstart[nblk] = start;
					    bptop[nblk] = ok ? 0xFFFFFFFEu : 0xFFFFFFFFu; // storedOffset sign decided by the engine (trap T4)
					    ++nblk;
				    });
				if (r != kFeNeedSlide && r != kFeGroup) in_deflate = false;
			}
		}
		r = __shfl_sync(0xffffffffu, r, 0);
		if (r == kFeGroup) {
			// steady-state loop tops ahead: the warp takes them in groups (fast_group_step) until a slide, a full block or the
			// end of the lookahead comes near; lane 0's engine is brought in step afterwards
			int s0 = __shfl_sync(0xffffffffu, e.strstart, 0), la = __shfl_sync(0xffffffffu, e.lookahead, 0);
			uint32_t nsym = __shfl_sync(0xffffffffu, e.nsym, 0);
			const uint32_t woff = __shfl_sync(0xffffffffu, e.woff, 0);
			total = __shfl_sync(0xffffffffu, total, 0);
			int last_h = 0, match_start = __shfl_sync(0xffffffffu, e.matchStart, 0), last_long = 0, nl;
			while ((nl = fe_group_lanes(s0, la, nsym)) >= kFeGroupMin) {
#ifdef B200Z_FAST_STATS
				const int s_before = s0;
#endif
				last_long = fast_group_step(in + off, woff, head, prev, lp, lane, nl, s0, la, nsym, sout, total, last_h, match_start);
#ifdef B200Z_FAST_STATS
				++st_steps;
				st_pos += (uint32_t)(s0 - s_before);
				st_lanes += (uint32_t)(s0 - s_before < 32 ? s0 - s_before : 32);
#endif
			}
			if (lane == 0) {
				e.strstart = s0;
				e.lookahead = la;
				e.nsym = nsym;
				e.matchStart = match_start;
				e.matchLen = kMinMatch - 1;
				if (last_long)
					fe_update_hash(e); // :712-714 (lookahead >= MIN_MATCH - 1 holds: it was >= 262 before a match of <= 258)
				else
					e.ins_h = last_h;
				// back at the top of DeflateFast's loop: `while (lookahead >= MIN_LOOKAHEAD || flush)` (:658)
				const bool flush = phase == 1 && e.inputOff == e.n;
				if (e.lookahead < kMaxMatch + kMinMatch + 1 && !flush) {
					in_deflate = false; // the loop ends, DeflateFast returns true (:738)
					r = kFeTrue;
				}
			}
			r = __shfl_sync(0xffffffffu, r, 0);
			if (r == kFeGroup) continue; // lane 0 goes on inside DeflateFast (in_deflate is still set)
		}
		r = __shfl_sync(0xffffffffu, r, 0);
		if (r == kFeNeedSlide) {
			// SlideWindow (DeflaterEngine.cs:441-462): scalars by lane 0, both tables by the warp
			if (lane == 0) fe_slide_scalars(e);
			for (int t = 0; t < 2; t++) { // 2 entries per 32-bit word (a slide means a stream beyond 64 KiB: whole tables)
				uint32_t *tab = reinterpret_cast<uint32_t *>(t ? prev : head);
				for (int i = lane; i < 16384; i += 32) {
					const uint32_t v = tab[i];
					uint32_t lo = v & 0xFFFFu, hi = v >> 16;
					lo = lo >= 32768u ? lo - 32768u : 0u;
					hi = hi >= 32768u ? hi - 32768u : 0u;
					tab[i] = lo | (hi << 16);
				}
			}
			__syncwarp();
			continue;
		}
		if (r == kFeFalse) {
			if (phase == 1) break;
			// chunk ci is drained ("needs input"): the next SetInput, or Flush()/Finish()
			++ci;
			if (ci < nc) {
				if (lane == 0) e.n = seg_base + cum[ci];
				if (ci == nc - 1 && !busy_last) phase = 1;
			} else {
				phase = 1;
			}
		}
	}
	if (lane == 0) {
		nsyms[stream] = total;
		nblocks[stream] = nblk;
#ifdef B200Z_FAST_STATS
		printf("k_fast stream %d: n %u, group steps %u, positions by groups %u (%.1f per step, %.1f lanes used), symbols %u\n", stream, n,
		       st_steps, st_pos, st_steps ? (double)st_pos / st_steps : 0.0, st_steps ? (double)st_lanes / st_steps : 0.0, total);
#endif
	}
	if (st) {
		// what the next segment of this stream starts from
		__syncwarp();
		uint4 *dst = reinterpret_cast<uint4 *>(st);
		for (int i = lane; i < 65536 / 16; i += 32) dst[i] = reinterpret_cast<const uint4 *>(head)[i];
		const int words = prev_entries * 2 / 16;
		for (int i = lane; i < words; i += 32) dst[65536 / 16 + i] = reinterpret_cast<const uint4 *>(prev)[i];
		for (int i = words + lane; i < 65536 / 16; i += 32) dst[65536 / 16 + i] = make_uint4(0u, 0u, 0u, 0u);
		if (lane == 0) {
			FastCarry c;
			fe_save(e, c);
			*reinterpret_cast<FastCarry *>(st + 131072) = c;
		}
	}
}

// persistent CTAs of one warp: streams are taken off a counter, so a batch of uneven streams keeps every CTA busy
__global__ void __launch_bounds__(32)
    k_fast(const uint8_t *__restrict__ in, uint32_t *__restrict__ sym, const int64_t *__restrict__ in_off,
           const int64_t *__restrict__ in_len, uint32_t *__restrict__ nsyms, uint32_t *__restrict__ nblocks,
           const uint32_t *__restrict__ blk_off, uint32_t *__restrict__ blk_start, uint32_t *__restrict__ blk_ptop,
           const uint32_t *__restrict__ hist, LevelParams lp, int strategy, int end_mode, int prev_entries,
           const uint32_t *__restrict__ sched, const uint32_t *__restrict__ sched_off, const int32_t *__restrict__ undrained,
           uint8_t *const *__restrict__ fstate, int cont, int group, int nstreams, uint16_t *__restrict__ head_pool,
           uint32_t *__restrict__ counter) {
	extern __shared__ __align__(16) uint8_t fsm[];
	uint16_t *prev = reinterpret_cast<uint16_t *>(fsm);
	// head_pool == nullptr: a batch of at most one stream per SM -- head[] sits behind prev[] in shared memory (one CTA per
	// SM then, whose L1 holds the stream's window: 1.7x faster per stream than with three CTAs sharing the SM)
	uint16_t *head = head_pool ? head_pool + 32768ll * blockIdx.x : prev + prev_entries;
	const int lane = threadIdx.x;
	for (;;) {
		int stream = 0;
		if (lane == 0) stream = (int)atomicAdd(counter, 1u);
		stream = __shfl_sync(0xffffffffu, stream, 0);
		if (stream >= nstreams) break;
		fast_stream(stream, lane, head, prev, in, sym, in_off, in_len, nsyms, nblocks, blk_off, blk_start, blk_ptop, hist, lp, strategy,
		            end_mode, prev_entries, sched, sched_off, undrained, fstate, cont, group);
		__syncwarp();
	}
}

// ------------------------------------------------------------------------------------------------
// Level 0: DeflateStored.  Block boundaries are pure bookkeeping (stored_run, computed when the plan is built);
// the kernel writes 1 header byte, LEN, ~LEN and copies the bytes (FlushStoredBlock, DeflaterHuffman.cs:766-779).
// ------------------------------------------------------------------------------------------------
struct StoredBlock {
	int32_t stream;
	uint32_t src;     // first input byte inside the stream
	uint32_t len;
	uint32_t last;
	uint64_t dst;     // byte offset of the block inside the stream's output slot
};

__global__ void __launch_bounds__(256)
    k_stored(const uint8_t *__restrict__ in, uint8_t *__restrict__ out, const int64_t *__restrict__ in_off,
             const int64_t *__restrict__ out_off, const StoredBlock *__restrict__ blocks) {
	const StoredBlock b = blocks[blockIdx.x];
	const uint8_t *src = in + in_off[b.stream] + b.src;
	uint8_t *dst = out + out_off[b.stream] + b.dst;
	if (threadIdx.x == 0) {
		dst[0] = (uint8_t)(b.last ? 1 : 0); // 3 header bits (STORED_BLOCK << 1 | last) then AlignToByte
		dst[1] = (uint8_t)b.len;
		dst[2] = (uint8_t)(b.len >> 8);
		dst[3] = (uint8_t)~b.len;
		dst[4] = (uint8_t)(~b.len >> 8);
	}
	for (uint32_t i = threadIdx.x; i < b.len; i += blockDim.x) dst[5 + i] = src[i];
}

__global__ void k_set_results(int n, const int64_t *__restrict__ lens, int64_t *__restrict__ out_len, int32_t *__restrict__ status,
                              int64_t *__restrict__ out_bits) {
	const int i = blockIdx.x * blockDim.x + threadIdx.x;
	if (i >= n) return;
	out_len[i] = lens[i];
	status[i] = B200Z_OK;
	if (out_bits) out_bits[i] = 8 * lens[i];
}

// ------------------------------------------------------------------------------------------------
// K4: per-block histograms, the reference's Huffman construction and the block type decision.
// ------------------------------------------------------------------------------------------------
constexpr int kPlanThreads = 64;
__global__ void __launch_bounds__(kPlanThreads)
    k_plan(const uint32_t *__restrict__ sym, const int64_t *__restrict__ in_off, const int64_t *__restrict__ in_len,
           const uint32_t *__restrict__ nsyms, const uint32_t *__restrict__ nblocks, const uint32_t *__restrict__ blk_off,
           const int32_t *__restrict__ blk_desc, const uint32_t *__restrict__ blk_start, const uint32_t *__restrict__ blk_ptop,
           BlockMeta *__restrict__ meta, BlockTables *__restrict__ tables, const int64_t *__restrict__ bias, int end_mode) {
	__shared__ int s_lit[kLiteralNum];
	__shared__ int s_dist[kDistNum];
	__shared__ int s_extra;
	__shared__ int s_scratch[kTreeScratchInts];
	__shared__ int s_scratch2[10 * kDistNum];
	__shared__ int s_lit_blc[15], s_dist_blc[15], s_nc[2];
	__shared__ BlockTables s_tab;
	const int g = blockIdx.x;
	const int stream = blk_desc[g];
	const uint32_t b = (uint32_t)g - blk_off[stream];
	const uint32_t nb = nblocks[stream];
	if (b >= nb) return;
	const uint32_t ns = nsyms[stream];
	const uint32_t s0 = b * (uint32_t)kBlockSyms;
	const uint32_t s1 = (ns - s0 > (uint32_t)kBlockSyms) ? s0 + kBlockSyms : ns;
	const uint32_t *sp = sym + in_off[stream];
	for (int i = threadIdx.x; i < kLiteralNum; i += blockDim.x) s_lit[i] = 0;
	for (int i = threadIdx.x; i < kDistNum; i += blockDim.x) s_dist[i] = 0;
	for (int i = threadIdx.x; i < kHdrWords; i += blockDim.x) s_tab.hdr[i] = 0;
	if (threadIdx.x == 0) s_extra = 0;
	__syncthreads();
	int extra = 0;
	for (uint32_t i0 = s0 + threadIdx.x; i0 < s1; i0 += 8 * blockDim.x) {
		// eight independent loads in flight per thread (ncu: the one-load-per-trip loop sat on long_scoreboard)
		uint32_t sv[8];
#pragma unroll
		for (int k = 0; k < 8; k++) {
			const uint32_t i = i0 + (uint32_t)k * blockDim.x;
			sv[k] = i < s1 ? __ldg(sp + i) : 0xFFFFFFFFu;
		}
#pragma unroll
		for (int k = 0; k < 8; k++) {
			const uint32_t s = sv[k];
			if (s == 0xFFFFFFFFu) continue; // (not a symbol: distances stop at 32506)
			if (sym_dist(s) == 0) {
				atomicAdd(&s_lit[s & 0xFF], 1);
			} else {
				const int lc = lcode((int)(s & 0xFF)), dc = dcode((int)sym_dist(s) - 1);
				atomicAdd(&s_lit[lc], 1);
				atomicAdd(&s_dist[dc], 1);
				extra += tally_extra_bits(lc, dc);
			}
		}
	}
	for (int o = 16; o > 0; o >>= 1) extra += __shfl_down_sync(0xffffffffu, extra, o);
	if ((threadIdx.x & 31) == 0 && extra) atomicAdd(&s_extra, extra);
	__syncthreads();
	if (threadIdx.x == 0) s_lit[256] += 1; // FlushBlock: literalTree.freqs[EOF_SYMBOL]++ (:790)
	__syncthreads();
	// the two big trees are independent: build them on two warps at once
	if (threadIdx.x == 0) s_nc[0] = build_tree(s_lit, kLiteralNum, 257, 15, s_tab.lit_len, s_lit_blc, s_scratch);
	if (threadIdx.x == 32) s_nc[1] = build_tree(s_dist, kDistNum, 1, 15, s_tab.dist_len, s_dist_blc, s_scratch2);
	__syncthreads();
	if (threadIdx.x == 0) {
		const uint32_t *bstart = blk_start + blk_off[stream];
		const uint32_t *bptop = blk_ptop + blk_off[stream];
		const uint32_t byte_start = bstart[b];
		const uint32_t n = (uint32_t)in_len[stream];
		const uint32_t byte_len = (b + 1 < nb ? bstart[b + 1] : n) - byte_start;
		// storedOffset is window relative and goes negative once the block start has been slid out (trap T4)
		const long long ab = bias[stream]; // absolute stream offset of buffer position 0
		long long storedOffset = (long long)byte_start + ab + 1 - 32768ll * (long long)slides_done((uint32_t)(bptop[b] + ab));
		if (bptop[b] >= 0xFFFFFFFEu) storedOffset = bptop[b] == 0xFFFFFFFEu ? 0 : -1; // levels 1-4: decided by k_fast
		const int last = (b + 1 == nb) && end_mode == B200Z_END_FINISH;
		BlockPlan plan;
		plan_block_finish(s_lit, s_dist, s_extra, storedOffset >= 0, (int)byte_len, last, s_nc[0], s_lit_blc, s_nc[1], s_dist_blc,
		                  s_tab.lit_len, s_tab.lit_codes, s_tab.dist_len, s_tab.dist_codes, s_tab.hdr, s_scratch, plan);
		BlockMeta m;
		m.byte_start = byte_start;
		m.byte_len = byte_len;
		m.nsyms = s1 - s0;
		m.hdr_bits = plan.hdr_bits;
		m.body_bits = plan.body_bits;
		m.type = (uint32_t)plan.type;
		m.bit_off = 0;
		meta[g] = m;
	}
	__syncthreads();
	// copy the tables out (16-byte vectors)
	const uint4 *src = reinterpret_cast<const uint4 *>(&s_tab);
	uint4 *dst = reinterpret_cast<uint4 *>(&tables[g]);
	for (int i = threadIdx.x; i < (int)(sizeof(BlockTables) / 16); i += blockDim.x) dst[i] = src[i];
}

__device__ __forceinline__ void or_bits(uint32_t *out_words, uint64_t bitpos, uint64_t bits, int nbits) {
	// nbits <= 57; spreads over at most three 32-bit words
	if (nbits == 0) return;
	const uint64_t idx = bitpos >> 5;
	const uint32_t sh = (uint32_t)(bitpos & 31);
	const uint64_t lo = bits << sh;
	atomicOr(out_words + idx, (uint32_t)lo);
	if (sh + nbits > 32) {
		atomicOr(out_words + idx + 1, (uint32_t)(lo >> 32));
		if (sh + nbits > 64) atomicOr(out_words + idx + 2, (uint32_t)(bits >> (64 - sh)));
	}
}

// ------------------------------------------------------------------------------------------------
// K5: bit offset of every block inside its stream (stored blocks byte-align), end-of-stream bits, sizes.
// ------------------------------------------------------------------------------------------------
__global__ void k_scan(int nstreams, const uint32_t *__restrict__ nblocks, const uint32_t *__restrict__ blk_off,
                       BlockMeta *__restrict__ meta, uint8_t *__restrict__ out, const int64_t *__restrict__ out_off,
                       const int64_t *__restrict__ out_cap, int64_t *__restrict__ out_len, int32_t *__restrict__ status,
                       int64_t *__restrict__ out_bits, const uint32_t *__restrict__ bit_base, int end_mode) {
	const int stream = blockIdx.x * blockDim.x + threadIdx.x;
	if (stream >= nstreams) return;
	const uint32_t nb = nblocks[stream];
	BlockMeta *m = meta + blk_off[stream];
	uint64_t cur = bit_base[stream]; // 0..7: a continued stream starts inside the byte the previous segment ended in
	for (uint32_t b = 0; b < nb; b++) {
		m[b].bit_off = cur;
		if (m[b].type == 0) cur = ((cur + 3 + 7) & ~7ull) + 32 + 8ull * m[b].byte_len;
		else cur += (uint64_t)m[b].hdr_bits + m[b].body_bits;
	}
	uint64_t tail0 = cur;
	int ntail10 = 0; // number of 10-bit empty static blocks: "WriteBits(2, 10)" (Deflater.cs:486-504)
	if (end_mode != B200Z_END_FINISH) {
		int neededbits = 8 + (int)((0 - cur) & 7);
		while (neededbits > 0) {
			++ntail10;
			cur += 10;
			neededbits -= 10;
		}
	}
	if (end_mode == B200Z_END_FLUSH_FINISH) cur += 10; // the final empty static block (3, 10 bits)
	const uint64_t nbytes = (cur + 7) >> 3; // FINISHING_STATE: pending.AlignToByte() (Deflater.cs:507)
	if ((int64_t)(((nbytes + 3) >> 2) << 2) > out_cap[stream]) {
		status[stream] = B200Z_E_NOMEM;
		out_len[stream] = 0;
		if (out_bits) out_bits[stream] = 0;
		for (uint32_t b = 0; b < nb; b++) m[b].type = 0xFFu; // tells k_emit to skip
		return;
	}
	uint32_t *ow = reinterpret_cast<uint32_t *>(out + out_off[stream]);
	uint64_t t = tail0;
	for (int i = 0; i < ntail10; i++, t += 10) or_bits(ow, t, 2, 10);
	if (end_mode == B200Z_END_FLUSH_FINISH) or_bits(ow, t, 3, 10);
	status[stream] = B200Z_OK;
	out_len[stream] = (int64_t)nbytes;
	if (out_bits) out_bits[stream] = (int64_t)cur; // exact length; a flushed stream may end inside its last byte
}

// ------------------------------------------------------------------------------------------------
// K6: bit emission.  One CTA per block; symbols are encoded 256 at a time, a block-wide exclusive scan of the code
// lengths gives every symbol its bit position, and the code words are OR-ed into the (zeroed) output words.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
    k_emit(const uint8_t *__restrict__ in, const uint32_t *__restrict__ sym, uint8_t *__restrict__ out,
           const int64_t *__restrict__ in_off, const int64_t *__restrict__ out_off, const uint32_t *__restrict__ nblocks,
           const uint32_t *__restrict__ blk_off, const int32_t *__restrict__ blk_desc, const BlockMeta *__restrict__ meta,
           const BlockTables *__restrict__ tables) {
	__shared__ BlockTables s_tab;
	__shared__ uint32_t s_warp[8];
	__shared__ uint64_t s_base;
	const int g = blockIdx.x;
	const int stream = blk_desc[g];
	const uint32_t b = (uint32_t)g - blk_off[stream];
	if (b >= nblocks[stream]) return;
	const BlockMeta m = meta[g];
	if (m.type == 0xFFu) return;
	uint32_t *ow = reinterpret_cast<uint32_t *>(out + out_off[stream]);
	if (m.type == 0) {
		// FlushStoredBlock (:766-779): 3 header bits, pad to byte, LEN, ~LEN, raw bytes
		const uint8_t *src = in + in_off[stream] + m.byte_start;
		const uint64_t hb = ((m.bit_off + 3 + 7) & ~7ull);
		if (threadIdx.x == 0) {
			or_bits(ow, m.bit_off, tables[g].hdr[0] & 7u, 3);
			or_bits(ow, hb, m.byte_len & 0xFFFFu, 16);
			or_bits(ow, hb + 16, (~m.byte_len) & 0xFFFFu, 16);
		}
		const uint64_t d0 = (hb + 32) >> 3; // byte offset of the payload in the stream's output
		uint8_t *ob = out + out_off[stream];
		// head bytes up to a word boundary and tail bytes go through atomicOr; whole words are plain stores
		const uint32_t len = m.byte_len;
		uint32_t headn = (uint32_t)((4 - (d0 & 3)) & 3);
		if (headn > len) headn = len;
		const uint32_t nwords = (len - headn) >> 2;
		const uint32_t tailn = len - headn - (nwords << 2);
		for (uint32_t i = threadIdx.x; i < headn; i += blockDim.x) or_bits(ow, (d0 + i) << 3, src[i], 8);
		uint32_t *wdst = reinterpret_cast<uint32_t *>(ob + d0 + headn);
		for (uint32_t i = threadIdx.x; i < nwords; i += blockDim.x) {
			const uint8_t *s4 = src + headn + (i << 2);
			wdst[i] = (uint32_t)s4[0] | ((uint32_t)s4[1] << 8) | ((uint32_t)s4[2] << 16) | ((uint32_t)s4[3] << 24);
		}
		for (uint32_t i = threadIdx.x; i < tailn; i += blockDim.x)
			or_bits(ow, (d0 + headn + (nwords << 2) + i) << 3, src[headn + (nwords << 2) + i], 8);
		return;
	}
	{
		const uint4 *src = reinterpret_cast<const uint4 *>(&tables[g]);
		uint4 *dst = reinterpret_cast<uint4 *>(&s_tab);
		for (int i = threadIdx.x; i < (int)(sizeof(BlockTables) / 16); i += blockDim.x) dst[i] = src[i];
	}
	if (threadIdx.x == 0) s_base = m.bit_off + m.hdr_bits;
	__syncthreads();
	// header words
	for (uint32_t i = threadIdx.x; i * 32 < m.hdr_bits; i += blockDim.x) {
		const uint32_t rem = m.hdr_bits - i * 32;
		const int nbw = rem < 32 ? (int)rem : 32;
		uint32_t v = s_tab.hdr[i];
		if (nbw < 32) v &= (1u << nbw) - 1u;
		or_bits(ow, m.bit_off + i * 32ull, v, nbw);
	}
	const uint32_t *sp = sym + in_off[stream] + b * (uint32_t)kBlockSyms;
	const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
	for (uint32_t i0 = 0; i0 < m.nsyms; i0 += blockDim.x) {
		const uint32_t i = i0 + threadIdx.x;
		uint64_t bits = 0;
		int nb = 0;
		if (i < m.nsyms) encode_symbol(sp[i], s_tab.lit_codes, s_tab.lit_len, s_tab.dist_codes, s_tab.dist_len, bits, nb);
		// block-wide exclusive scan of nb
		uint32_t incl = (uint32_t)nb;
		for (int o = 1; o < 32; o <<= 1) {
			uint32_t t = __shfl_up_sync(0xffffffffu, incl, o);
			if (lane >= o) incl += t;
		}
		if (lane == 31) s_warp[wid] = incl;
		__syncthreads();
		uint32_t woff = 0, tot = 0;
		for (int k = 0; k < 8; k++) {
			const uint32_t v = s_warp[k];
			if (k < wid) woff += v;
			tot += v;
		}
		const uint64_t base = s_base;
		or_bits(ow, base + woff + incl - (uint32_t)nb, bits, nb);
		__syncthreads();
		if (threadIdx.x == 0) s_base = base + tot;
		__syncthreads();
	}
	if (threadIdx.x == 0) or_bits(ow, s_base, s_tab.lit_codes[256], s_tab.lit_len[256]); // EOF_SYMBOL (:750)
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
int deflate_plan_build(b200z_plan *p) {
	const LevelParams lp = level_params(p->level);
	const int n = p->n;
	std::vector<StoredBlock> sblocks; // level 0 only
	std::vector<int64_t> slens;
	p->in_off.resize(n);
	p->out_off.resize(n);
	p->out_cap.resize(n);
	int64_t io = 0, oo = 0;
	std::vector<int2> runs, tiles, rgroups;
	std::vector<ChunkDesc> chunks;
	std::vector<uint32_t> rnd_off(n + 1);
	uint32_t nrounds = 0;
	int64_t maxlen = 0;
	for (int i = 0; i < n; i++) maxlen = p->in_len[i] > maxlen ? p->in_len[i] : maxlen;
	// chunk of the parse: 32 Ki positions (one warp each); k_parse_fix only compares states at their boundaries, so a long
	// stream may have tens of thousands of them (grown beyond 65536 chunks per stream)
	uint32_t chunk = 32768;
	{
		const int64_t need = (maxlen / 65536 + kRound - 1) / kRound * kRound;
		if (need > (int64_t)chunk) chunk = (uint32_t)need;
	}
	// Run length of k_links (a multiple of 32768, 65536 .. 1048576).  Every run but a stream's first re-walks 32768 positions
	// to warm its head table up (37 % more steps than positions with 64 Ki runs on 256 KiB buffers, 12 % with 128 Ki runs,
	// none with 256 Ki runs), while fewer, longer CTAs fill the last wave worse (three CTAs fit an SM).  The plan takes the
	// length with the smallest estimate of waves x steps per run; B200Z_LINK_RUN=<positions> overrides it for timing.
	p->link_run = kRun;
	{
		int sms = 148;
		int dev = 0;
		if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
		const int64_t slots = 3ll * sms;
		double best = 0;
		for (int64_t run = 65536; run <= 1048576; run *= 2) {
			int64_t ctas = 0, longest = 0;
			for (int i = 0; i < n; i++) {
				const int64_t len = p->in_len[i];
				ctas += (len + run - 1) / run;
				const int64_t first = len < run ? len : run;
				const int64_t steps = len > run ? run + 32768 : first; // a run behind the first also walks its warm-up
				longest = steps > longest ? steps : longest;
			}
			const double est = (double)((ctas + slots - 1) / slots) * (double)longest;
			if (best == 0 || est < best * 0.97) { // (a longer run has to win clearly: its CTAs are the less balanced ones)
				best = est;
				p->link_run = (int)run;
			}
			if (run >= maxlen) break;
		}
	}
	if (const char *e = getenv("B200Z_LINK_RUN")) {
		const long v = atol(e);
		if (v >= 65536 && v <= 1048576 && v % 32768 == 0) p->link_run = (int)v;
	}
	p->parse_chunk = chunk;
	{
		// levels 1-4: size of k_fast's prev[] table (see there)
		int64_t need = maxlen + 2;
		int pe = 32768;
		if (need <= 32768 && p->engine_state.empty()) pe = (int)((need + 255) / 256 * 256); // (a carried state holds whole tables)
		p->fast_prev_entries = pe;
		// persistent one-warp CTAs: as many per SM as their prev[] tables fit (head[] is in the pool), 16 at most
		int sms = 148, dev = 0;
		if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
		int per_sm = (int)((227 * 1024) / (2 * pe + 1024));
		if (per_sm > 16) per_sm = 16;
		if (per_sm < 1) per_sm = 1;
		const int64_t slots = (int64_t)sms * per_sm;
		p->fast_ctas = (int)(n < slots ? n : slots);
		p->fast_head_smem = n <= sms; // nothing to gain from sharing SMs: keep head[] next to prev[] (k_fast)
		if (const char *e = getenv("B200Z_FAST_HEAD")) p->fast_head_smem = e[0] == 's'; // "smem" / "pool": for tests and timing
	}
	std::vector<uint32_t> blk_off(n + 1);
	std::vector<int32_t> blk_desc;
	uint32_t nblk = 0;
	const bool has_hist = !p->hist.empty();
	std::vector<uint32_t> hist32(n, 0u), bitbase32(n, 0u);
	std::vector<int64_t> bias64(n, 0), hm_off(n, 0), ck_off(n), ck_len(n);
	std::vector<uint8_t> hmask;
	std::vector<int64_t> stored_taken(n, -1);
	for (int i = 0; i < n; i++) {
		const int64_t len = p->in_len[i];
		if (len < 0 || len > 0xFFFF0000ll) {
			set_error("stream %d: length %lld out of range", i, (long long)len);
			return B200Z_E_ARG;
		}
		const int64_t H = has_hist ? p->hist[i] : 0;
		if (has_hist) {
			hist32[i] = (uint32_t)H;
			bias64[i] = p->pos_base[i] - H;
			bitbase32[i] = (uint32_t)p->bit_base[i];
			hm_off[i] = (int64_t)hmask.size();
			hmask.resize(hmask.size() + (size_t)H + 1, 0);
			uint8_t *m = hmask.data() + hm_off[i];
			if (i < (int)p->hist_mask.size() && !p->hist_mask[i].empty()) memcpy(m, p->hist_mask[i].data(), (size_t)H);
			else if (H) m[H - 1] = 1, m[H > 1 ? H - 2 : 0] = 1; // the last two positions of a dictionary/segment are never inserted
		}
		p->in_off[i] = io;
		io += align_up(len + 16, kAlign);
		p->out_off[i] = oo;
		p->out_cap[i] = align_up(b200z_deflate_bound(len), kAlign);
		oo += p->out_cap[i];
		for (int64_t s = 0; s < len; s += p->link_run) runs.push_back(make_int2(i, (int)s));
		for (int64_t s = 0; s < len; s += kTile) tiles.push_back(make_int2(i, (int)s));
		for (int64_t s = 0; s < len; s += chunk)
			chunks.push_back(ChunkDesc{i, (uint32_t)s, (uint32_t)(len - s > (int64_t)chunk ? s + chunk : len)});
		rnd_off[i] = nrounds;
		const uint32_t nr = (uint32_t)((len + kRound - 1) / kRound);
		for (uint32_t r = 0; r < nr; r += 4) rgroups.push_back(make_int2(i, (int)r));
		nrounds += nr;
		blk_off[i] = nblk;
		const uint32_t maxb = (uint32_t)(len / kBlockSyms) + 2;
		for (uint32_t b = 0; b < maxb; b++) blk_desc.push_back(i);
		nblk += maxb;
		if (lp.func == 0) {
			uint64_t dst = 0;
			const bool cont = p->hist_kind == B200Z_HIST_CONTINUE;
			const uint32_t *cum = (i < (int)p->sched_cum.size() && !p->sched_cum[i].empty()) ? p->sched_cum[i].data() : nullptr;
			const int nch = cum ? (int)p->sched_cum[i].size() : 0;
			const bool busy_last = !(i < (int)p->undrained.size() && p->undrained[i]);
			StoredCarry cin{0, 0, 0, 0}, cout{0, 0, 0, 0};
			if (cont) { // checked when the plan was created: stored_state is there
				cin.strstart = p->stored_state[i].strstart;
				cin.blockStart = p->stored_state[i].block_start;
				cin.slides = p->stored_state[i].slides;
				cin.inputOff = p->stored_state[i].input_off;
			}
			stored_run((uint32_t)(len - H), cont ? 0u : (uint32_t)H, p->end_mode, [&](uint32_t start, uint32_t blen, bool last) {
				sblocks.push_back(StoredBlock{i, start, blen, last ? 1u : 0u, dst});
				dst += 5 + (uint64_t)blen;
			}, cum, nch, cont ? &cin : nullptr, &cout, cont ? (uint32_t)(p->pos_base[i] - H) : 0u, busy_last);
			// what the window took in: everything, except when Finish() right behind an undrained SetInput makes
			// DeflateStored end the stream early (lastBlock = finish although input is left, DeflaterEngine.cs:629-641);
			// TotalIn and the Adler-32 of the reference then cover the consumed bytes only, and so do ours
			stored_taken[i] = (int64_t)(uint32_t)(cout.inputOff - (cont ? cin.inputOff : 0u));
			if (p->stored_state) {
				p->stored_state[i].strstart = cout.strstart;
				p->stored_state[i].block_start = cout.blockStart;
				p->stored_state[i].slides = cout.slides;
				p->stored_state[i].input_off = cout.inputOff;
			}
			slens.push_back((int64_t)dst);
		}
	}
	rnd_off[n] = nrounds;
	if (lp.func != 2) {
		runs.clear();
		tiles.clear();
		chunks.clear();
		rgroups.clear();
	}
	p->n_chunks = (int)chunks.size();
	p->n_rgroups = (int)rgroups.size();
	blk_off[n] = nblk;
	p->in_bytes = io;
	p->out_bytes = oo;
	p->n_runs = (int)runs.size();
	p->n_tiles = (int)tiles.size();
	p->n_blkmax = (int)nblk;
	Arena &ws = p->ws;
	p->o_in_off = ws.reserve(8ll * n);
	p->o_in_len = ws.reserve(8ll * n);
	p->o_out_off = ws.reserve(8ll * n);
	p->o_out_cap = ws.reserve(8ll * n);
	p->o_run_desc = ws.reserve(8ll * (runs.size() + 1));
	p->o_tile_desc = ws.reserve(8ll * (tiles.size() + 1));
	p->o_blk_desc = ws.reserve(4ll * (nblk + 1));
	p->o_blk_off = ws.reserve(4ll * (n + 1));
	p->o_nsyms = ws.reserve(4ll * n);
	p->o_nblocks = ws.reserve(4ll * n);
	p->o_blk_start = ws.reserve(4ll * (nblk + 1));
	p->o_blk_ptop = ws.reserve(4ll * (nblk + 1));
	p->o_meta = ws.reserve((int64_t)sizeof(BlockMeta) * (nblk + 1));
	p->o_tables = ws.reserve((int64_t)sizeof(BlockTables) * (nblk + 1));
	if (lp.func == 2) {
		p->o_link = ws.reserve(2ll * io + 64);
		p->o_mt = ws.reserve(8ll * io + 64);
		p->o_sym_local = ws.reserve(4ll * io + 64);
		p->o_chunks = ws.reserve((int64_t)sizeof(ChunkDesc) * (chunks.size() + 1));
		p->o_rgroups = ws.reserve(8ll * (rgroups.size() + 1));
		p->o_rnd_off = ws.reserve(4ll * (n + 1));
		p->o_recs = ws.reserve((int64_t)sizeof(RoundRec) * (nrounds + 1));
		p->o_ents = ws.reserve((int64_t)sizeof(RoundRec) * (nrounds + 1));
		p->o_rnd_symoff = ws.reserve(4ll * (nrounds + 1));
	}
	if (lp.func != 0) p->o_sym = ws.reserve(4ll * io + 64);
	if (lp.func == 0) {
		p->n_stored = (int)sblocks.size();
		p->o_stored = ws.reserve((int64_t)sizeof(StoredBlock) * (sblocks.size() + 1));
		p->o_slens = ws.reserve(8ll * (n + 1));
	}
	std::vector<uint32_t> sched_flat, sched_off(n + 1, 0u);
	std::vector<int32_t> undrained32(n, 0);
	std::vector<void *> fstate(n, nullptr);
	if (lp.func == 1) {
		for (int i = 0; i < n; i++) {
			sched_off[i] = (uint32_t)sched_flat.size();
			if (i < (int)p->sched_cum.size()) sched_flat.insert(sched_flat.end(), p->sched_cum[i].begin(), p->sched_cum[i].end());
			if (i < (int)p->undrained.size()) undrained32[i] = p->undrained[i] ? 1 : 0;
			if (i < (int)p->engine_state.size()) fstate[i] = p->engine_state[i];
		}
		sched_off[n] = (uint32_t)sched_flat.size();
		p->o_sched = ws.reserve(4ll * (sched_flat.size() + 1));
		p->o_sched_off = ws.reserve(4ll * (n + 1));
		p->o_undrained = ws.reserve(4ll * (n + 1));
		p->o_fstate = ws.reserve(8ll * (n + 1));
		p->o_fhead = ws.reserve(p->fast_head_smem ? 256 : 65536ll * p->fast_ctas);
		p->o_fcounter = ws.reserve(256);
	}
	p->o_hist = ws.reserve(4ll * (n + 1));
	p->o_bias = ws.reserve(8ll * (n + 1));
	p->o_bitbase = ws.reserve(4ll * (n + 1));
	p->o_hm_off = ws.reserve(8ll * (n + 1));
	p->o_hmask = ws.reserve((int64_t)hmask.size() + 16);
	std::vector<CkTile> ck_tiles;
	if (p->wrap != B200Z_WRAP_RAW) {
		for (int i = 0; i < n; i++) { // the checksum covers the data, never the history
			ck_off[i] = p->in_off[i] + hist32[i];
			ck_len[i] = p->in_len[i] - hist32[i];
			if (stored_taken[i] >= 0 && stored_taken[i] < ck_len[i]) ck_len[i] = stored_taken[i]; // level 0, see above
		}
		p->o_ck_off = ws.reserve(8ll * (n + 1));
		p->o_ck_len = ws.reserve(8ll * (n + 1));
		checksum_tiles(ck_len.data(), n, ck_tiles, p->wrap == B200Z_WRAP_ZLIB ? 1 : 0);
		p->n_ck_tiles = (int)ck_tiles.size();
		p->o_ck_desc = ws.reserve((int64_t)sizeof(CkTile) * (ck_tiles.size() + 1));
		p->o_ck_acc = ws.reserve(16ll * (n + 1));
	}
	int rc = ws.alloc();
	if (rc) return rc;
	B200Z_CUDA(cudaMemcpy(ws.at<int64_t>(p->o_in_off), p->in_off.data(), 8ll * n, cudaMemcpyHostToDevice));
	B200Z_CUDA(cudaMemcpy(ws.at<int64_t>(p->o_in_len), p->in_len.data(), 8ll * n, cudaMemcpyHostToDevice));
	B200Z_CUDA(cudaMemcpy(ws.at<int64_t>(p->o_out_off), p->out_off.data(), 8ll * n, cudaMemcpyHostToDevice));
	B200Z_CUDA(cudaMemcpy(ws.at<int64_t>(p->o_out_cap), p->out_cap.data(), 8ll * n, cudaMemcpyHostToDevice));
	if (n) {
		B200Z_CUDA(cudaMemcpy(ws.at<uint32_t>(p->o_hist), hist32.data(), 4ll * n, cudaMemcpyHostToDevice));
		B200Z_CUDA(cudaMemcpy(ws.at<int64_t>(p->o_bias), bias64.data(), 8ll * n, cudaMemcpyHostToDevice));
		B200Z_CUDA(cudaMemcpy(ws.at<uint32_t>(p->o_bitbase), bitbase32.data(), 4ll * n, cudaMemcpyHostToDevice));
		B200Z_CUDA(cudaMemcpy(ws.at<int64_t>(p->o_hm_off), hm_off.data(), 8ll * n, cudaMemcpyHostToDevice));
		if (!hmask.empty()) B200Z_CUDA(cudaMemcpy(ws.at<uint8_t>(p->o_hmask), hmask.data(), hmask.size(), cudaMemcpyHostToDevice));
		if (p->wrap != B200Z_WRAP_RAW) {
			B200Z_CUDA(cudaMemcpy(ws.at<int64_t>(p->o_ck_off), ck_off.data(), 8ll * n, cudaMemcpyHostToDevice));
			B200Z_CUDA(cudaMemcpy(ws.at<int64_t>(p->o_ck_len), ck_len.data(), 8ll * n, cudaMemcpyHostToDevice));
		}
	}
	if (!runs.empty()) B200Z_CUDA(cudaMemcpy(ws.at<int2>(p->o_run_desc), runs.data(), 8ll * runs.size(), cudaMemcpyHostToDevice));
	if (!tiles.empty()) B200Z_CUDA(cudaMemcpy(ws.at<int2>(p->o_tile_desc), tiles.data(), 8ll * tiles.size(), cudaMemcpyHostToDevice));
	B200Z_CUDA(cudaMemcpy(ws.at<int32_t>(p->o_blk_desc), blk_desc.data(), 4ll * nblk, cudaMemcpyHostToDevice));
	B200Z_CUDA(cudaMemcpy(ws.at<uint32_t>(p->o_blk_off), blk_off.data(), 4ll * (n + 1), cudaMemcpyHostToDevice));
	if (!ck_tiles.empty())
		B200Z_CUDA(cudaMemcpy(ws.at<CkTile>(p->o_ck_desc), ck_tiles.data(), sizeof(CkTile) * ck_tiles.size(),
		                      cudaMemcpyHostToDevice));
	if (lp.func == 2) {
		if (!chunks.empty())
			B200Z_CUDA(cudaMemcpy(ws.at<ChunkDesc>(p->o_chunks), chunks.data(), sizeof(ChunkDesc) * chunks.size(), cudaMemcpyHostToDevice));
		if (!rgroups.empty())
			B200Z_CUDA(cudaMemcpy(ws.at<int2>(p->o_rgroups), rgroups.data(), 8ll * rgroups.size(), cudaMemcpyHostToDevice));
		B200Z_CUDA(cudaMemcpy(ws.at<uint32_t>(p->o_rnd_off), rnd_off.data(), 4ll * (n + 1), cudaMemcpyHostToDevice));
	}
	if (lp.func == 1 && n) {
		if (!sched_flat.empty())
			B200Z_CUDA(cudaMemcpy(ws.at<uint32_t>(p->o_sched), sched_flat.data(), 4ll * sched_flat.size(), cudaMemcpyHostToDevice));
		B200Z_CUDA(cudaMemcpy(ws.at<uint32_t>(p->o_sched_off), sched_off.data(), 4ll * (n + 1), cudaMemcpyHostToDevice));
		B200Z_CUDA(cudaMemcpy(ws.at<int32_t>(p->o_undrained), undrained32.data(), 4ll * n, cudaMemcpyHostToDevice));
		B200Z_CUDA(cudaMemcpy(ws.at<void *>(p->o_fstate), fstate.data(), 8ll * n, cudaMemcpyHostToDevice));
	}
	if (!sblocks.empty())
		B200Z_CUDA(cudaMemcpy(ws.at<StoredBlock>(p->o_stored), sblocks.data(), sizeof(StoredBlock) * sblocks.size(), cudaMemcpyHostToDevice));
	if (!slens.empty()) B200Z_CUDA(cudaMemcpy(ws.at<int64_t>(p->o_slens), slens.data(), 8ll * slens.size(), cudaMemcpyHostToDevice));
	B200Z_CUDA(cudaFuncSetAttribute(k_fast, cudaFuncAttributeMaxDynamicSharedMemorySize, kFastSmem));
	B200Z_CUDA(cudaFuncSetAttribute(k_links, cudaFuncAttributeMaxDynamicSharedMemorySize, kLinksSmem));
	B200Z_CUDA(cudaFuncSetAttribute(k_match, cudaFuncAttributeMaxDynamicSharedMemorySize, kTileData + 2 * 2 * kTile));
	p->launches = (lp.func == 2 ? 9 : (lp.func == 1 ? 4 : 2)) + (p->wrap != B200Z_WRAP_RAW ? 3 : 0); // + one memset node
	return B200Z_OK;
}

int deflate_plan_run(b200z_plan *p, const uint8_t *d_in, uint8_t *d_out, int64_t *d_out_len, int32_t *d_status,
                     uint32_t *d_check, int64_t *d_out_bits, cudaStream_t s, int stages) {
	const Arena &ws = p->ws;
	const int n = p->n;
	if (n == 0) return B200Z_OK;
	const LevelParams lp = level_params(p->level);
	const int64_t *in_off = ws.at<int64_t>(p->o_in_off), *in_len = ws.at<int64_t>(p->o_in_len);
	const int64_t *out_off = ws.at<int64_t>(p->o_out_off), *out_cap = ws.at<int64_t>(p->o_out_cap);
	uint16_t *link = lp.func == 2 ? ws.at<uint16_t>(p->o_link) : nullptr;
	uint2 *mt = lp.func == 2 ? ws.at<uint2>(p->o_mt) : nullptr;
	uint32_t *sym = lp.func != 0 ? ws.at<uint32_t>(p->o_sym) : nullptr;
	uint32_t *nsyms = ws.at<uint32_t>(p->o_nsyms), *nblocks = ws.at<uint32_t>(p->o_nblocks);
	uint32_t *blk_off = ws.at<uint32_t>(p->o_blk_off);
	int32_t *blk_desc = ws.at<int32_t>(p->o_blk_desc);
	uint32_t *blk_start = ws.at<uint32_t>(p->o_blk_start), *blk_ptop = ws.at<uint32_t>(p->o_blk_ptop);
	BlockMeta *meta = ws.at<BlockMeta>(p->o_meta);
	BlockTables *tables = ws.at<BlockTables>(p->o_tables);
	const uint32_t *hist = ws.at<uint32_t>(p->o_hist), *bit_base = ws.at<uint32_t>(p->o_bitbase);
	const int64_t *bias = ws.at<int64_t>(p->o_bias);
	const int ck_fresh = p->check_seeded ? 0 : 1;

	// stages: B200Z_STAGE_SEARCH = match finding (levels 5-9: k_links, k_match), B200Z_STAGE_ENCODE = everything else.
	// Splitting lets a caller put other work (e.g. an inflate plan on a second stream) next to the ENCODE kernels, which
	// leave most of an SM's shared memory free, instead of next to k_match, which takes all of it.
	const bool do_search = (stages & B200Z_STAGE_SEARCH) != 0, do_encode = (stages & B200Z_STAGE_ENCODE) != 0;
	const bool was_timing = p->timing;
	if (stages != (B200Z_STAGE_SEARCH | B200Z_STAGE_ENCODE)) p->timing = false; // per-kernel times are for whole runs
	struct TimingRestore {
		b200z_plan *p;
		bool v;
		~TimingRestore() { p->timing = v; }
	} timing_restore{p, was_timing};
	if (lp.func != 2 && !do_encode) return B200Z_OK; // levels 0-4 have no separate search stage
	p->ev_used = 0;
	if (lp.func == 0) {
		// level 0: stored blocks laid out when the plan was built
		p->mark(s, "k_stored");
		if (p->n_stored) k_stored<<<p->n_stored, 256, 0, s>>>(d_in, d_out, in_off, out_off, ws.at<StoredBlock>(p->o_stored));
		k_set_results<<<(n + 127) / 128, 128, 0, s>>>(n, ws.at<int64_t>(p->o_slens), d_out_len, d_status, d_out_bits);
		p->mark(s, "checksum");
		if (p->wrap != B200Z_WRAP_RAW && d_check) {
			int rc = checksum_launch(p->wrap == B200Z_WRAP_ZLIB ? 1 : 0, d_in, ws.at<int64_t>(p->o_ck_off), ws.at<int64_t>(p->o_ck_len), n,
			                         ws.at<CkTile>(p->o_ck_desc), p->n_ck_tiles, ws.at<unsigned long long>(p->o_ck_acc), d_check,
			                         ck_fresh, s);
			if (rc) return rc;
		}
		p->mark(s, "end");
		B200Z_CUDA(cudaGetLastError());
		return B200Z_OK;
	}
	if (do_encode) {
		p->mark(s, "memset");
		B200Z_CUDA(cudaMemsetAsync(d_out, 0, (size_t)p->out_bytes, s));
	}
	if (lp.func == 1) {
		p->mark(s, "k_fast");
		B200Z_CUDA(cudaMemsetAsync(ws.at<uint32_t>(p->o_fcounter), 0, 4, s));
		k_fast<<<p->fast_ctas, 32, 2 * p->fast_prev_entries + (p->fast_head_smem ? 65536 : 0), s>>>(
		    d_in, sym, in_off, in_len, nsyms, nblocks, blk_off, blk_start, blk_ptop, hist, lp, p->strategy, p->end_mode,
		    p->fast_prev_entries, ws.at<uint32_t>(p->o_sched), ws.at<uint32_t>(p->o_sched_off), ws.at<int32_t>(p->o_undrained),
		    ws.at<uint8_t *>(p->o_fstate), p->hist_kind == B200Z_HIST_CONTINUE ? 1 : 0, fast_group_enabled(), n,
		    p->fast_head_smem ? nullptr : ws.at<uint16_t>(p->o_fhead), ws.at<uint32_t>(p->o_fcounter));
	} else {
		if (do_search) {
		p->mark(s, "k_links");
		if (p->n_runs) k_links<<<p->n_runs, kLinkThreads, kLinksSmem, s>>>(d_in, link, in_off, in_len, ws.at<int2>(p->o_run_desc), hist,
			                                                         ws.at<uint8_t>(p->o_hmask), ws.at<int64_t>(p->o_hm_off), (uint32_t)p->link_run);
		p->mark(s, "k_match");
		if (p->n_tiles)
			k_match<<<p->n_tiles, kMatchThreads, kTileData + 2 * 2 * kTile, s>>>(d_in, link, mt, in_off, in_len,
			                                                                   ws.at<int2>(p->o_tile_desc), hist, bias, sym, lp);
		}
		if (!do_encode) {
			B200Z_CUDA(cudaGetLastError());
			return B200Z_OK;
		}
		p->mark(s, "k_parse");
		{
			uint32_t *sym_local = ws.at<uint32_t>(p->o_sym_local);
			const uint32_t *rnd_off = ws.at<uint32_t>(p->o_rnd_off);
			RoundRec *recs = ws.at<RoundRec>(p->o_recs);
			uint32_t *rnd_symoff = ws.at<uint32_t>(p->o_rnd_symoff);
			if (p->n_chunks)
				k_parse_chunk<<<p->n_chunks, 32, kParseSmem, s>>>(d_in, link, mt, sym_local, in_off, in_len, ws.at<ChunkDesc>(p->o_chunks),
				                                                 rnd_off, recs, ws.at<RoundRec>(p->o_ents), hist, bias, lp, p->strategy, parse_warm());
			k_parse_fix<<<n, 32, kParseSmem, s>>>(d_in, link, mt, sym_local, in_off, in_len, rnd_off, recs, ws.at<RoundRec>(p->o_ents),
			                                      p->parse_chunk, hist, bias, lp, p->strategy);
			k_parse_scan<<<n, 256, 0, s>>>(d_in, in_off, in_len, rnd_off, recs, rnd_symoff, sym, nsyms, nblocks, blk_off, blk_start,
			                               blk_ptop, hist, p->end_mode);
			if (p->n_rgroups)
				k_parse_gather<<<p->n_rgroups, 128, 0, s>>>(sym_local, sym, in_off, in_len, ws.at<int2>(p->o_rgroups), rnd_off, recs,
				                                           rnd_symoff, blk_off, blk_start, blk_ptop, hist);
		}
	}
	p->mark(s, "k_plan");
	k_plan<<<p->n_blkmax, kPlanThreads, 0, s>>>(sym, in_off, in_len, nsyms, nblocks, blk_off, blk_desc, blk_start, blk_ptop, meta,
	                                   tables, bias, p->end_mode);
	p->mark(s, "k_scan");
	k_scan<<<(n + 127) / 128, 128, 0, s>>>(n, nblocks, blk_off, meta, d_out, out_off, out_cap, d_out_len, d_status,
	                                       d_out_bits, bit_base, p->end_mode);
	p->mark(s, "k_emit");
	k_emit<<<p->n_blkmax, 256, 0, s>>>(d_in, sym, d_out, in_off, out_off, nblocks, blk_off, blk_desc, meta, tables);
	p->mark(s, "checksum");
	if (p->wrap != B200Z_WRAP_RAW && d_check) {
		int rc = checksum_launch(p->wrap == B200Z_WRAP_ZLIB ? 1 : 0, d_in, ws.at<int64_t>(p->o_ck_off), ws.at<int64_t>(p->o_ck_len), n,
		                         ws.at<CkTile>(p->o_ck_desc), p->n_ck_tiles, ws.at<unsigned long long>(p->o_ck_acc), d_check,
		                         ck_fresh, s);
		if (rc) return rc;
	}
	p->mark(s, "end");
	B200Z_CUDA(cudaGetLastError());
	return B200Z_OK;
}

int deflate_plan_match_table(b200z_plan *p, int32_t i, uint16_t *link, uint32_t *ab, cudaStream_t s) {
	const int64_t off = p->in_off[i], n = p->in_len[i], H = p->hist.empty() ? 0 : p->hist[i];
	if (link) B200Z_CUDA(cudaMemcpyAsync(link, p->ws.at<uint16_t>(p->o_link) + off, 2 * n, cudaMemcpyDeviceToHost, s));
	B200Z_CUDA(cudaMemcpyAsync(ab, p->ws.at<uint2>(p->o_mt) + off + H, 8 * (n - H), cudaMemcpyDeviceToHost, s));
	B200Z_CUDA(cudaStreamSynchronize(s));
	return B200Z_OK;
}

} // namespace b200z
