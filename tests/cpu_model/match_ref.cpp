// match_ref.cpp -- the match table as match_search() of b200z_core.cuh states it, over the data and the hash-chain links
// a plan's SEARCH stage used (tests/test_match_table.py compares k_match's table against it entry for entry).
#include "b200z_core.cuh"

using namespace b200z;

// ab[2 * (p - H)], ab[2 * (p - H) + 1] = (A, B) of data position p (H <= p < n); abs_bias = stream offset of position 0
extern "C" void ref_match_table(const uint8_t *data, const uint16_t *link, uint32_t n, uint32_t H, uint32_t abs_bias, int level,
                                uint32_t *ab) {
	const LevelParams lp = level_params(level);
	for (uint32_t p = H; p < n; p++) match_search(data, link, 0u, p, n, lp, ab[2 * (p - H)], ab[2 * (p - H) + 1], abs_bias);
}
