// match_stats.cpp -- DEVELOPMENT AID (not product, not test): work counts of the level 5-9 search on the bench workload,
// taken on the CPU with the same functions the kernels call (b200z_core.cuh).  It answers, without a GPU, how much of
// k_match's work the parser ever looks at and where the candidate loop spends its steps:
//   * candidates walked per position when EVERY position is searched from threshold 2 (what k_match does)
//   * candidates the reference walks (only at the positions DeflateSlow visits, with the carried threshold and budget)
//   * how often a candidate passes the first quick-reject byte / the whole quick reject / improves the match
// build: g++ -O2 -std=c++17 -I sharpziplib_b200/csrc -o /tmp/match_stats tools/match_stats.cpp
// run:   /tmp/match_stats <file of concatenated buffers> <buffer size> <level> [reuse]
//        (with "reuse": only the count of extension work that position p+1's result could replace)
#include "b200z_core.cuh"
#include <cstdio>
#include <cstdlib>
#include <vector>

using namespace b200z;

static void links(const uint8_t *data, uint32_t n, std::vector<uint16_t> &link) {
	link.assign(n, 0);
	std::vector<int64_t> head(32768, -1);
	for (uint32_t p = 0; p + 2 < n; p++) {
		const uint32_t h = hash3(data[p], data[p + 1], data[p + 2]);
		if (head[h] >= 0 && p - head[h] <= (uint32_t)kMaxDist) link[p] = (uint16_t)(p - head[h]);
		head[h] = p;
	}
}

struct Cnt {
	uint64_t pos = 0, searched = 0, cands = 0, fb = 0, qr = 0, impr = 0, ext = 0, nice_stop = 0;
	uint64_t hist[9] = {0}; // candidates per searched position: 1, 2, <=4, <=8, ... <=128, more
	void add_hist(uint32_t c) {
		int b = 0;
		while ((1u << b) < c && b < 8) b++;
		hist[b]++;
	}
};

// the walk of match_search (threshold m0, budget), counting
static uint32_t walk(const uint8_t *data, const uint16_t *link, uint32_t p, uint32_t n, uint32_t m0, uint32_t budget, uint32_t nice_lp,
                     Cnt &c) {
	const uint32_t la = n - p;
	if (la < 3) return 0;
	uint32_t d = link[p];
	if (d == 0) return 0;
	const uint32_t maxlen = la < 258 ? la : 258, nice = la < nice_lp ? la : nice_lp;
	if (m0 >= maxlen) return 0;
	const uint8_t *s = data + p;
	uint32_t m = m0, dist = d, cnt = 0, bd = 0;
	c.searched++;
	for (;;) {
		const uint8_t *cc = s - dist;
		++cnt;
		if (cc[m] == s[m]) {
			c.fb++;
			if (cc[m - 1] == s[m - 1] && cc[0] == s[0] && cc[1] == s[1]) {
				c.qr++;
				uint32_t l = 2;
				while (l < maxlen && cc[l] == s[l]) ++l;
				c.ext += l - 2;
				if (l > m) {
					c.impr++;
					m = l;
					bd = dist;
					if (m >= nice) {
						c.nice_stop++;
						break;
					}
				}
			}
		}
		if (cnt == budget) break;
		const uint32_t l2 = link[p - dist];
		if (l2 == 0) break;
		dist += l2;
		if (dist >= (uint32_t)kMaxDist) break;
	}
	c.cands += cnt;
	c.add_hist(cnt);
	return m > m0 ? pack_match(m, bd) : 0;
}

// k_match's extension after a passed quick reject: the two register compares of bytes 2..9, then the loop of 4-byte compares
// and the byte tail.  Returns the lcp; `words` gets the iterations of the 4-byte loop plus the tail's byte steps.
static uint32_t kernel_extension(const uint8_t *s, const uint8_t *c, uint32_t maxlen, uint64_t &words) {
	uint32_t l = 2;
	if (maxlen >= 10) {
		while (l < 10 && c[l] == s[l]) ++l;
		if (l < 10) return l;
	}
	while (l + 4 <= maxlen) {
		++words;
		uint32_t k = 0;
		while (k < 4 && c[l + k] == s[l + k]) ++k;
		l += k;
		if (k < 4) return l;
	}
	while (l < maxlen && c[l] == s[l]) {
		++words;
		++l;
	}
	return l;
}

// How much of k_match's extension loop the lcp of position p+1 could replace: for a candidate at p+1's best distance d
// that passes the quick reject, lcp(p, d) = min(lcp(p + 1, d) + 1, maxlen(p)) without extending.  Counted as if every
// position's predecessor p+1 ran on the same thread just before it (an upper bound: the class order splits some pairs).
static void reuse_stats(const uint8_t *data, const uint16_t *link, uint32_t n, const LevelParams &lp, uint64_t &words,
                        uint64_t &reusable, uint64_t &hits) {
	uint32_t prev_d = 0, prev_l = 0; // p+1's best distance and its full capped lcp (0: none)
	for (uint32_t p = n; p-- > 0;) {
		const uint32_t la = n - p;
		uint32_t d = la >= (uint32_t)kMinMatch ? link[p] : 0u;
		uint32_t best_d = 0, m = kMinMatch - 1;
		if (d != 0 && d <= (uint32_t)kMaxDist) {
			const uint32_t maxlen = la < (uint32_t)kMaxMatch ? la : (uint32_t)kMaxMatch;
			const uint32_t nice = la < (uint32_t)lp.nice ? la : (uint32_t)lp.nice;
			const uint8_t *s = data + p;
			uint32_t dist = d, cnt = 0;
			for (;;) {
				const uint8_t *c = s - dist;
				++cnt;
				if (c[m] == s[m] && c[m - 1] == s[m - 1] && c[0] == s[0] && c[1] == s[1]) {
					uint64_t w = 0;
					const uint32_t l = kernel_extension(s, c, maxlen, w);
					words += w;
					if (dist == prev_d && prev_l) {
						reusable += w;
						hits++;
					}
					if (l > m) {
						m = l;
						best_d = dist;
						if (m >= nice) break;
					}
				}
				if (cnt == (uint32_t)lp.chain) break;
				const uint32_t l2 = link[p - dist];
				if (l2 == 0) break;
				dist += l2;
				if (dist >= (uint32_t)kMaxDist) break;
			}
		}
		prev_d = best_d;
		prev_l = best_d ? m : 0;
	}
}

int main(int argc, char **argv) {
	if (argc < 4) return 1;
	FILE *f = fopen(argv[1], "rb");
	const uint32_t bs = (uint32_t)atoi(argv[2]);
	const int level = atoi(argv[3]);
	const LevelParams lp = level_params(level);
	std::vector<uint8_t> buf(bs + 16);
	if (argc > 4) { // "reuse": only this count
		uint64_t words = 0, reusable = 0, hits = 0;
		while (fread(buf.data(), 1, bs, f) == bs) {
			std::vector<uint16_t> link;
			links(buf.data(), bs, link);
			reuse_stats(buf.data(), link.data(), bs, lp, words, reusable, hits);
		}
		printf("extension reuse from p+1: %llu of %llu word steps of the extension loop (%.1f%%) fall on p+1's best distance "
		       "(%llu candidates)\n", (unsigned long long)reusable, (unsigned long long)words, 100.0 * reusable / (words ? words : 1),
		       (unsigned long long)hits);
		return 0;
	}
	Cnt all, ref;
	uint64_t visited = 0, used_a = 0, used_b = 0, useful = 0, nsym = 0;
	int nb = 0;
	while (fread(buf.data(), 1, bs, f) == bs) {
		nb++;
		const uint32_t n = bs;
		std::vector<uint16_t> link;
		links(buf.data(), n, link);
		std::vector<uint32_t> A(n, 0), B(n, 0);
		for (uint32_t p = 0; p < n; p++) {
			all.pos++;
			match_search(buf.data(), link.data(), 0u, p, n, lp, A[p], B[p]);
			walk(buf.data(), link.data(), p, n, 2, (uint32_t)lp.chain, (uint32_t)lp.nice, all); // the same walk, counted
		}
		// the parse: which positions are looked at, with which threshold
		ParseState st;
		parse_init(st);
		st.p = 0;
		auto tabf = [&](uint32_t p, uint32_t &a, uint32_t &b) {
			a = A[p];
			b = B[p];
			visited++;
			const uint32_t m0 = st.mlen < 2 ? 2 : st.mlen;
			const bool quarter = m0 >= (uint32_t)lp.good;
			(quarter ? used_b : used_a)++;
			const uint32_t r = walk(buf.data(), link.data(), p, n, m0, quarter ? (uint32_t)lp.chain >> 2 : (uint32_t)lp.chain,
			                        (uint32_t)lp.nice, ref);
			if (r) useful++;
			ref.pos++;
		};
		auto bytef = [&](uint32_t q) { return (uint32_t)buf[q]; };
		auto slowf = [&](uint32_t p, uint32_t m0, uint32_t budget) { return match_search_above(buf.data(), link.data(), p, n, m0, budget, 0u); };
		while (st.p < n) {
			uint32_t s2;
			nsym += (uint64_t)parse_step(st, n, lp, 0, tabf, bytef, slowf, s2);
		}
	}
	// how well does a cheap proxy parse (tables from the first `hops` candidates only) predict the positions the real parse visits?
	for (int hops : {1, 2, 4, 8}) {
		rewind(f);
		uint64_t vt = 0, vp = 0, both = 0, cands_pred = 0, cands_miss = 0, misses = 0;
		while (fread(buf.data(), 1, bs, f) == bs) {
			const uint32_t n = bs;
			std::vector<uint16_t> link;
			links(buf.data(), n, link);
			std::vector<uint32_t> A(n, 0), B(n, 0), A1(n, 0), B1(n, 0);
			LevelParams lq = lp;
			lq.chain = hops;
			for (uint32_t p = 0; p < n; p++) {
				match_search(buf.data(), link.data(), 0u, p, n, lp, A[p], B[p]);
				match_search(buf.data(), link.data(), 0u, p, n, lq, A1[p], B1[p]);
			}
			std::vector<uint8_t> vis(n, 0);
			for (int pass = 0; pass < 2; pass++) {
				ParseState st;
				parse_init(st);
				st.p = 0;
				auto tabf = [&](uint32_t p, uint32_t &a, uint32_t &b) {
					a = pass ? A1[p] : A[p];
					b = pass ? B1[p] : B[p];
					vis[p] |= (uint8_t)(1 << pass);
				};
				auto bytef = [&](uint32_t q) { return (uint32_t)buf[q]; };
				auto slowf = [&](uint32_t p, uint32_t m0, uint32_t budget) { return match_search_above(buf.data(), link.data(), p, n, m0, budget, 0u); };
				while (st.p < n) {
					uint32_t s2;
					parse_step(st, n, lp, 0, tabf, bytef, slowf, s2);
				}
			}
			for (uint32_t p = 0; p < n; p++) {
				vt += vis[p] & 1;
				vp += (vis[p] >> 1) & 1;
				both += vis[p] == 3;
				if (vis[p] & 2) { // predicted: searched in full, balanced like k_match
					Cnt c;
					walk(buf.data(), link.data(), p, n, 2, (uint32_t)lp.chain, (uint32_t)lp.nice, c);
					cands_pred += c.cands;
				} else if (vis[p] & 1) { // visited by the real parse but not predicted: searched on demand inside the parse
					Cnt c;
					walk(buf.data(), link.data(), p, n, 2, (uint32_t)lp.chain, (uint32_t)lp.nice, c);
					cands_miss += c.cands;
					misses++;
				}
			}
		}
		printf("proxy parse with %d-hop tables: visits %.1f%% of positions, covers %.1f%% of the real parse's visits; searching the "
		       "predicted set walks %.1f candidates per position (all positions: %.1f), the %.2f%% of positions it misses walk %.2f\n",
		       hops, 100.0 * vp / all.pos, 100.0 * both / (vt ? vt : 1), (double)cands_pred / all.pos, (double)all.cands / all.pos,
		       100.0 * misses / all.pos, (double)cands_miss / all.pos);
	}
	// ---- lock-step cost of the tile kernel (experimental/k_tile_parse.cuh): a warp's loop iteration costs what its slowest
	// lane walks in that iteration; passes as the kernel runs them (speculative pass, hand-off passes with memo, emit pass)
	{
		rewind(f);
		const uint32_t kSeg = 32, kFTile = 16384, kFThreads = 512;
		uint64_t warp_steps = 0, lane_cands = 0, iters = 0, parse_steps = 0;
		while (fread(buf.data(), 1, bs, f) == bs) {
			const uint32_t n = bs;
			std::vector<uint16_t> link;
			links(buf.data(), n, link);
			auto bytef = [&](uint32_t q) { return (uint32_t)buf[q]; };
			auto slowf = [&](uint32_t p, uint32_t m0, uint32_t budget) { return match_search_above(buf.data(), link.data(), p, n, m0, budget, 0u); };
			for (uint32_t t0 = 0; t0 < n; t0 += kFTile) {
				std::vector<uint32_t> memoA(kFTile, 0xFFFFFFFFu), memoB(kFTile, 0);
				std::vector<ParseCarry> entry(kFThreads), ex(kFThreads);
				std::vector<uint32_t> lim(kFThreads);
				std::vector<char> changed(kFThreads, 1);
				auto clean = [&](uint32_t p) { ParseCarry c; parse_init(c.st); c.st.p = p; c.last_top = p; return c; };
				for (uint32_t t = 0; t < kFThreads; t++) {
					const uint32_t seg0 = t0 + t * kSeg;
					lim[t] = seg0 + kSeg < n ? seg0 + kSeg : n;
					entry[t] = clean(seg0);
				}
				uint32_t last_cost = 0;
				auto tabf = [&](uint32_t p, uint32_t &a, uint32_t &b) {
					last_cost = 1; // a memo hit still costs a step
					if (memoA[p - t0] == 0xFFFFFFFFu) {
						Cnt c;
						match_search(buf.data(), link.data(), 0u, p, n, lp, memoA[p - t0], memoB[p - t0]);
						walk(buf.data(), link.data(), p, n, 2, (uint32_t)lp.chain, (uint32_t)lp.nice, c);
						last_cost = (uint32_t)c.cands + 1;
						lane_cands += c.cands;
					}
					a = memoA[p - t0];
					b = memoB[p - t0];
				};
				for (int pass = 0; pass < 64; pass++) {
					// warps in lock step: iteration i runs the i-th parse step of every lane that (re-)parses
					for (uint32_t w = 0; w < kFThreads / 32; w++) {
						bool any = true;
						for (uint32_t l = 0; l < 32; l++)
							if (changed[w * 32 + l]) ex[w * 32 + l] = entry[w * 32 + l];
						while (any) {
							any = false;
							uint32_t worst = 0;
							for (uint32_t l = 0; l < 32; l++) {
								const uint32_t t = w * 32 + l;
								if (!changed[t] || ex[t].st.p >= lim[t]) continue;
								any = true;
								ex[t].last_top = ex[t].st.p;
								uint32_t s2;
								last_cost = 1;
								parse_step(ex[t].st, n, lp, 0, tabf, bytef, slowf, s2);
								parse_steps++;
								if (last_cost > worst) worst = last_cost;
							}
							if (any) {
								warp_steps += worst;
								iters++;
							}
						}
					}
					bool again = false;
					changed[0] = 0;
					std::vector<ParseCarry> prev(ex);
					for (uint32_t t = 1; t < kFThreads; t++) {
						changed[t] = !carry_equal(prev[t - 1], entry[t]);
						entry[t] = prev[t - 1];
						again |= changed[t] != 0;
					}
					if (!again) break;
				}
				// emit pass: every lane parses its segment once more, all from the memo
				for (uint32_t w = 0; w < kFThreads / 32; w++) {
					uint32_t longest = 0;
					for (uint32_t l = 0; l < 32; l++) {
						ParseCarry c = entry[w * 32 + l];
						uint32_t k = 0;
						while (c.st.p < lim[w * 32 + l]) {
							uint32_t s2;
							parse_step(c.st, n, lp, 0, tabf, bytef, slowf, s2);
							k++;
						}
						if (k > longest) longest = k;
					}
					warp_steps += longest;
					iters += longest;
				}
			}
		}
		const double km_steps = (double)all.cands / 32.0 / (14.8 / 32.0); // k_match: measured 14.8 of 32 lanes per instruction
		printf("tile kernel, lock-step model: %llu warp candidate-steps (%.2f per position), %llu loop iterations, lanes busy %.1f%%;\n"
		       "   k_match at its measured lane occupancy: %.0f warp candidate-steps (%.2f per position) -> ratio %.2fx fewer\n",
		       (unsigned long long)warp_steps, (double)warp_steps / all.pos, (unsigned long long)iters,
		       100.0 * (double)(lane_cands + parse_steps) / (32.0 * (double)warp_steps), km_steps, km_steps / all.pos,
		       km_steps / (double)warp_steps);
	}
	// ---- variant: tile-local "guess, batch, re-parse".  Every 32-position segment parses with the exact entry where one is
	// known and a 1-hop proxy entry otherwise, noting the positions it consulted without an exact entry; those are searched as
	// one balanced batch (k_match's ordering), then the segments whose inputs changed parse again; until a pass consults
	// nothing unknown and the hand-off is stable.
	{
		rewind(f);
		const uint32_t kSeg = 32, kFTile = 16384, kFThreads = 512;
		uint64_t batch_cands[16] = {0}, batch_req[16] = {0}, pass_iters[16] = {0}, tiles = 0, passes_total = 0;
		int max_pass = 0;
		LevelParams l1 = lp;
		l1.chain = 1;
		while (fread(buf.data(), 1, bs, f) == bs) {
			const uint32_t n = bs;
			std::vector<uint16_t> link;
			links(buf.data(), n, link);
			auto bytef = [&](uint32_t q) { return (uint32_t)buf[q]; };
			auto slowf = [&](uint32_t p, uint32_t m0, uint32_t budget) { return match_search_above(buf.data(), link.data(), p, n, m0, budget, 0u); };
			for (uint32_t t0 = 0; t0 < n; t0 += kFTile) {
				tiles++;
				std::vector<uint32_t> exA(kFTile, 0xFFFFFFFFu), exB(kFTile, 0), prA(kFTile, 0), prB(kFTile, 0);
				std::vector<char> asked(kFTile, 0);
				for (uint32_t i = 0; i < kFTile && t0 + i < n; i++) match_search(buf.data(), link.data(), 0u, t0 + i, n, l1, prA[i], prB[i]);
				std::vector<ParseCarry> entry(kFThreads), ex(kFThreads);
				std::vector<uint32_t> lim(kFThreads);
				std::vector<char> dirty(kFThreads, 1); // segment must parse again (entry changed or an entry it used became exact)
				std::vector<std::vector<uint32_t>> used(kFThreads); // inexact positions a segment consulted in its last parse
				auto clean = [&](uint32_t p) { ParseCarry c; parse_init(c.st); c.st.p = p; c.last_top = p; return c; };
				for (uint32_t t = 0; t < kFThreads; t++) {
					const uint32_t seg0 = t0 + t * kSeg;
					lim[t] = seg0 + kSeg < n ? seg0 + kSeg : n;
					entry[t] = clean(seg0);
					ex[t] = entry[t];
				}
				int pass = 0;
				for (;; pass++) {
					std::vector<uint32_t> req;
					for (uint32_t w = 0; w < kFThreads / 32; w++) {
						uint32_t longest = 0;
						for (uint32_t l = 0; l < 32; l++) {
							const uint32_t t = w * 32 + l;
							if (!dirty[t]) continue;
							used[t].clear();
							ex[t] = entry[t];
							uint32_t k = 0;
							auto tabf = [&](uint32_t p, uint32_t &a, uint32_t &b) {
								const uint32_t i = p - t0;
								if (exA[i] != 0xFFFFFFFFu) { a = exA[i]; b = exB[i]; return; }
								a = prA[i]; b = prB[i];
								used[t].push_back(p);
								if (!asked[i] && link[p]) { asked[i] = 1; req.push_back(p); }
								else if (!link[p]) { exA[i] = 0; exB[i] = 0; }
							};
							while (ex[t].st.p < lim[t]) {
								ex[t].last_top = ex[t].st.p;
								uint32_t s2;
								parse_step(ex[t].st, n, lp, 0, tabf, bytef, slowf, s2);
								k++;
							}
							if (k > longest) longest = k;
						}
						if (pass < 16) pass_iters[pass] += longest;
					}
					// the batch
					for (uint32_t p : req) {
						Cnt c;
						match_search(buf.data(), link.data(), 0u, p, n, lp, exA[p - t0], exB[p - t0]);
						walk(buf.data(), link.data(), p, n, 2, (uint32_t)lp.chain, (uint32_t)lp.nice, c);
						if (pass < 16) batch_cands[pass] += c.cands;
					}
					if (pass < 16) batch_req[pass] += req.size();
					// who parses again: entry changed, or it used an entry that is exact now (and differs from the proxy)
					bool again = false;
					std::vector<ParseCarry> prev(ex);
					for (uint32_t t = 0; t < kFThreads; t++) {
						bool d = false;
						if (t > 0 && !carry_equal(prev[t - 1], entry[t])) { entry[t] = prev[t - 1]; d = true; }
						for (uint32_t p : used[t]) {
							const uint32_t i = p - t0;
							if (exA[i] != 0xFFFFFFFFu && (exA[i] != prA[i] || exB[i] != prB[i])) d = true;
						}
						// (an entry that is exact now and equals the proxy changes nothing)
						dirty[t] = d;
						again |= d;
					}
					if (!again) break;
				}
				passes_total += (uint64_t)pass + 1;
				if (pass + 1 > max_pass) max_pass = pass + 1;
			}
		}
		printf("guess / batch / re-parse per tile: %.2f passes per tile on average, %d at most\n", (double)passes_total / tiles, max_pass);
		double tot_c = 0, tot_i = 0;
		for (int k = 0; k < 8; k++) {
			if (!batch_req[k] && !pass_iters[k]) continue;
			printf("   pass %d: parse %.3f lock-step iterations per position; batch: %.2f%% of positions, %.2f candidates per position\n", k,
			       (double)pass_iters[k] / all.pos, 100.0 * batch_req[k] / all.pos, (double)batch_cands[k] / all.pos);
			tot_c += (double)batch_cands[k];
			tot_i += (double)pass_iters[k];
		}
		printf("   total: %.2f candidates per position in balanced batches (k_match: %.2f), %.3f parse iterations per position + 1 proxy hop per position\n",
		       tot_c / all.pos, (double)all.cands / all.pos, tot_i / all.pos);
	}
	auto pr = [&](const char *name, const Cnt &c) {
		printf("%s: positions %llu, searched %llu (%.1f%%), candidates %llu (%.1f per searched, %.1f per position)\n", name,
		       (unsigned long long)c.pos, (unsigned long long)c.searched, 100.0 * c.searched / c.pos, (unsigned long long)c.cands,
		       (double)c.cands / (c.searched ? c.searched : 1), (double)c.cands / c.pos);
		printf("   first-byte pass %.1f%% of candidates, quick-reject pass %.2f%%, improvements %.2f%% (%.2f per searched), "
		       "extension bytes %.1f per quick-reject pass, nice stops %.2f%% of searched\n",
		       100.0 * c.fb / c.cands, 100.0 * c.qr / c.cands, 100.0 * c.impr / c.cands, (double)c.impr / c.searched,
		       (double)c.ext / (c.qr ? c.qr : 1), 100.0 * c.nice_stop / c.searched);
		printf("   candidates per searched position, share of positions: ");
		const char *lab[9] = {"1", "2", "<=4", "<=8", "<=16", "<=32", "<=64", "<=128", ">128"};
		for (int i = 0; i < 9; i++) printf("%s %.1f%%  ", lab[i], 100.0 * c.hist[i] / (c.searched ? c.searched : 1));
		printf("\n");
	};
	printf("level %d, %d buffers of %u bytes\n", level, nb, bs);
	pr("every position from threshold 2 (k_match)", all);
	pr("the reference's own searches (DeflateSlow)", ref);
	printf("parser: %llu of %llu positions visited (%.1f%%), table A used %llu, table B (quarter budget) %llu, searches that "
	       "improved the carried match %.1f%%, symbols %llu\n",
	       (unsigned long long)visited, (unsigned long long)all.pos, 100.0 * visited / all.pos, (unsigned long long)used_a,
	       (unsigned long long)used_b, 100.0 * useful / (visited ? visited : 1), (unsigned long long)nsym);
	printf("work ratio: k_match walks %.2fx the candidates the reference walks\n", (double)all.cands / (ref.cands ? ref.cands : 1));
	return 0;
}
