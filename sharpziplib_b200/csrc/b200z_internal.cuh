// b200z_internal.cuh -- shared host-side plumbing of libb200z.so (context, error reporting, plan object).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <string>
#include <vector>

#include "../../include/b200z.h"
#include "b200z_core.cuh"
#include "b200z_crc.cuh"

namespace b200z {

void set_error(const char *fmt, ...);
int cuda_fail(cudaError_t e, const char *what, const char *file, int line);

#define B200Z_CUDA(call)                                                                   \
	do {                                                                                   \
		cudaError_t e__ = (call);                                                          \
		if (e__ != cudaSuccess) return ::b200z::cuda_fail(e__, #call, __FILE__, __LINE__); \
	} while (0)

int ensure_init(); // picks up the current device if b200z_init() was not called explicitly
int current_device(); // the device b200z_init() chose for the calling thread (the CUDA current device otherwise)

// Every object (plan, pipeline, handle) remembers the device it was created on; its entry points run there and leave the
// calling thread's current device as they found it, so that one host thread can drive several GPUs.
struct DeviceGuard {
	int prev = -1;
	explicit DeviceGuard(int dev) {
		if (dev < 0) return;
		int cur = -1;
		if (cudaGetDevice(&cur) == cudaSuccess && cur != dev) {
			prev = cur;
			cudaSetDevice(dev);
		}
	}
	~DeviceGuard() {
		if (prev >= 0) cudaSetDevice(prev);
	}
};

constexpr int64_t kAlign = 256; // stream slots in the blobs start on 256-byte boundaries (vector loads / bulk copies)
inline int64_t align_up(int64_t v, int64_t a) { return (v + a - 1) / a * a; }

// One device allocation carved into typed arrays.
struct Arena {
	uint8_t *base = nullptr;
	int64_t size = 0, used = 0;
	int64_t reserve(int64_t bytes) { // planning pass: returns offset
		int64_t off = align_up(used, 256);
		used = off + bytes;
		return off;
	}
	int alloc();
	void release();
	template <class T> T *at(int64_t off) const { return reinterpret_cast<T *>(base + off); }
};

// per-block tables produced by k_plan and consumed by k_emit
struct __align__(16) BlockTables {
	uint16_t lit_codes[kLiteralNum];
	uint16_t dist_codes[kDistNum];
	uint8_t lit_len[kLiteralNum];
	uint8_t dist_len[kDistNum];
	uint32_t hdr[kHdrWords];
};

struct __align__(16) BlockMeta {
	uint32_t byte_start; // first input byte covered by the block
	uint32_t byte_len;   // storedLength
	uint32_t nsyms;
	uint32_t hdr_bits;
	uint32_t body_bits;
	uint32_t type; // 0 stored, 1 static, 2 dynamic
	uint64_t bit_off; // absolute bit offset inside the stream's output slot (k_scan)
};

// Inflate: one LZ77 back-reference to resolve (phase 2)
struct __align__(8) MatchTok {
	uint32_t out_pos;
	uint16_t len;
	uint16_t dist;
};

} // namespace b200z

struct b200z_plan {
	int kind = 0; // 0 deflate, 1 inflate
	int device = -1; // the device the plan's workspace lives on
	int n = 0;
	int level = 6, strategy = 0, wrap = 0, end_mode = 0;
	int host_wrap = 0; // the framing the host-buffer pipeline writes around this plan's streams (b200z_pipeline_*)
	std::vector<int64_t> in_len, in_off, out_off, out_cap;
	int64_t in_bytes = 0, out_bytes = 0;
	// deflate with history (b200z_deflate_plan_create_ex): in_len[] is history + data; an inflate plan keeps the
	// preset-dictionary lengths in hist[]
	int hist_kind = 0; // B200Z_HIST_*
	bool check_seeded = false;
	std::vector<int64_t> hist, pos_base;
	std::vector<int32_t> bit_base;
	std::vector<std::vector<uint8_t>> hist_mask;
	int64_t o_hist = 0, o_bias = 0, o_bitbase = 0, o_hm_off = 0, o_hmask = 0, o_ck_off = 0, o_ck_len = 0;
	b200z::Arena ws;
	int launches = 0;
	// deflate workspace offsets
	int64_t o_in_off = 0, o_in_len = 0, o_out_off = 0, o_out_cap = 0;
	int64_t o_run_desc = 0, o_tile_desc = 0, o_blk_desc = 0, o_blk_off = 0;
	int64_t o_link = 0, o_mt = 0, o_sym = 0, o_nsyms = 0, o_nblocks = 0;
	int64_t o_blk_start = 0, o_blk_ptop = 0, o_meta = 0, o_tables = 0;
	int n_runs = 0, n_tiles = 0, n_blkmax = 0;
	int64_t o_sym_local = 0, o_chunks = 0, o_rgroups = 0, o_rnd_off = 0, o_recs = 0, o_ents = 0, o_rnd_symoff = 0; // chunked parse
	int n_chunks = 0, n_rgroups = 0;
	uint32_t parse_chunk = 32768;
	int link_run = 65536; // positions per k_links CTA (B200Z_LINK_RUN)
	int fast_prev_entries = 32768; // k_fast's prev[] size for this batch
	int fast_ctas = 1;             // k_fast's persistent CTAs (each owns a head[] slot of the pool)
	bool fast_head_smem = false;   // ... or keeps head[] in shared memory (few streams)
	int64_t o_stored = 0, o_slens = 0; // level 0: stored-block list and per-stream output lengths
	// levels 0-4: the SetInput schedule of every stream (cumulative sizes), "Flush()/Finish() behind an undrained SetInput",
	// and the engine state carried between the segments of a stream (b200z_history)
	std::vector<std::vector<uint32_t>> sched_cum;
	std::vector<int32_t> undrained;
	std::vector<void *> engine_state;             // device pointers (levels 1-4)
	struct b200z_stored_state *stored_state = nullptr; // caller's host array (level 0), used while the plan is built
	int64_t o_sched = 0, o_sched_off = 0, o_undrained = 0, o_fstate = 0, o_fhead = 0, o_fcounter = 0;
	int n_stored = 0;
	// inflate workspace offsets
	int64_t o_tok = 0, o_ntok = 0, o_tok_off = 0;
	int64_t o_start_bit = 0, o_pre = 0; // inflate framing: first deflate bit and header verdict per stream
	int64_t o_restart = 0;              // inflate: per stream (bit, output position) of the last block header reached
	bool has_start_bits = false;        // raw inflate plans: caller-supplied first bit (b200z_inflate_plan_set_start_bits)
	std::vector<int64_t> comp_off, comp_cap, dict_cap; // inflate: where the compressed bytes start in the blob; capacities (b200z_inflate_plan_set_lengths)
	// inflate, block-parallel pipeline (b200z_inflate_par.cuh)
	bool inf_parallel = true;           // false: the serial kernel only (B200Z_INFLATE=serial)
	int64_t o_win_base = 0, o_win_stream = 0, o_cand = 0, o_ftiles = 0, o_fs_list = 0, o_ctr = 0, o_segs = 0, o_seg_list = 0;
	int64_t o_rounds = 0, o_hdrs = 0, o_mlist = 0, o_mt_off = 0, o_match_cap = 0, o_str_nm = 0, o_fallback = 0;
	uint32_t nwin_total = 0, n_ftiles = 0, fs_cap = 0, round_cap = 0, hdr_cap = 0;
	int dec1_grid = 0, dec2_grid = 0, find3_grid = 0;
	// checksum scratch
	int64_t o_ck_desc = 0, o_ck_acc = 0;
	int n_ck_tiles = 0;
	// optional per-kernel timing (b200z_plan_set_timing): events recorded on the run's stream between kernels
	bool timing = false;
	std::vector<cudaEvent_t> ev;
	std::vector<const char *> ev_name; // ev_name[i] labels the interval ev[i] -> ev[i+1]
	int ev_used = 0;
	void mark(cudaStream_t s, const char *next_name) {
		if (!timing) return;
		if ((int)ev.size() <= ev_used) {
			cudaEvent_t e;
			cudaEventCreate(&e);
			ev.push_back(e);
			ev_name.push_back("");
		}
		cudaEventRecord(ev[ev_used], s);
		ev_name[ev_used] = next_name;
		++ev_used;
	}
};

namespace b200z {
// implemented in b200z_deflate.cu / b200z_inflate.cu / b200z_checksum.cu
int deflate_plan_build(b200z_plan *p);
int deflate_plan_run(b200z_plan *p, const uint8_t *d_in, uint8_t *d_out, int64_t *d_out_len, int32_t *d_status,
                     uint32_t *d_check, int64_t *d_out_bits, cudaStream_t s, int stages);
int deflate_plan_match_table(b200z_plan *p, int32_t i, uint16_t *link, uint32_t *ab, cudaStream_t s);
int inflate_plan_build(b200z_plan *p);
int inflate_plan_stats(b200z_plan *p, uint32_t *v, int32_t cap, cudaStream_t s);
int inflate_plan_run(b200z_plan *p, const uint8_t *d_in, uint8_t *d_out, int64_t *d_out_len, int32_t *d_status,
                     uint32_t *d_check, int64_t *d_in_used, cudaStream_t s);
// checksum over n device buffers (kind 0 = CRC32, 1 = Adler32); d_acc = 2 x uint64 scratch per stream;
// value in/out (device uint32), `fresh` != 0 starts from the Reset() value instead of reading d_value.
int checksum_launch(int kind, const uint8_t *d_data, const int64_t *d_off, const int64_t *d_len, int32_t n,
                    const CkTile *d_tiles, int32_t n_tiles, unsigned long long *d_acc, uint32_t *d_value, int fresh,
                    cudaStream_t s);
int checksum_tiles(const int64_t *len, int32_t n, std::vector<CkTile> &tiles, int kind, bool dynamic = false);
int checksum_init_tables();
} // namespace b200z
