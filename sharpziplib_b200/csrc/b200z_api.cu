// b200z_api.cu -- the C-ABI of libb200z.so (include/b200z.h): context, plans, host-buffer batch calls and the
// streaming handles that mirror Deflater.cs / Inflater.cs member for member.  No CPU codec lives here: every byte of
// compressed or decompressed data is produced by the kernels in b200z_deflate.cu / b200z_inflate.cu.
#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <functional>
#include <mutex>
#include <thread>
#include <utility>

#include "b200z_internal.cuh"
#include <dlfcn.h>

namespace b200z {

static thread_local std::string g_err;
static std::mutex g_mu;
static thread_local int t_device = -1; // what b200z_init() chose for this thread

void set_error(const char *fmt, ...) {
	char buf[512];
	va_list ap;
	va_start(ap, fmt);
	vsnprintf(buf, sizeof(buf), fmt, ap);
	va_end(ap);
	g_err = buf;
}

int cuda_fail(cudaError_t e, const char *what, const char *file, int line) {
	set_error("CUDA error %d (%s) at %s:%d in %s", (int)e, cudaGetErrorString(e), file, line, what);
	return B200Z_E_CUDA;
}

int ensure_init() {
	std::lock_guard<std::mutex> lk(g_mu);
	if (t_device >= 0) return B200Z_OK;
	int cnt = 0;
	cudaError_t e = cudaGetDeviceCount(&cnt);
	if (e != cudaSuccess || cnt == 0) {
		set_error("no CUDA device: libb200z has no CPU fallback (%s)", e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
		return B200Z_E_CUDA;
	}
	int dev = 0;
	B200Z_CUDA(cudaGetDevice(&dev));
	t_device = dev;
	return B200Z_OK;
}

int current_device() {
	if (t_device >= 0) return t_device;
	int dev = 0;
	if (cudaGetDevice(&dev) != cudaSuccess) return -1;
	return dev;
}

int Arena::alloc() {
	size = align_up(used + 256, 256);
	cudaError_t e = cudaMalloc(&base, (size_t)size);
	if (e != cudaSuccess) {
		base = nullptr;
		set_error("cudaMalloc of %lld workspace bytes failed: %s", (long long)size, cudaGetErrorString(e));
		return B200Z_E_NOMEM;
	}
	return B200Z_OK;
}
void Arena::release() {
	if (base) cudaFree(base);
	base = nullptr;
}

// ---- static tables blob ---------------------------------------------------------------------------
static void fill_static_blob(uint8_t *b) {
	// encoder side: DeflaterHuffman static ctor (:602-642); decoder side: InflaterHuffmanTree static ctor (:34-70)
	size_t o = 0;
	for (int i = 0; i < kLiteralNum; i++) {
		uint16_t c = (uint16_t)static_lcode(i);
		memcpy(b + o, &c, 2);
		o += 2;
	}
	for (int i = 0; i < kLiteralNum; i++) b[o++] = (uint8_t)static_llen(i);
	for (int i = 0; i < kDistNum; i++) {
		uint16_t c = (uint16_t)static_dcode(i);
		memcpy(b + o, &c, 2);
		o += 2;
	}
	for (int i = 0; i < kDistNum; i++) b[o++] = 5;
	for (int i = 0; i < 288; i++) b[o++] = (uint8_t)(i < 144 ? 8 : (i < 256 ? 9 : (i < 280 ? 7 : 8)));
	for (int i = 0; i < 32; i++) b[o++] = 5;
}
constexpr int kStaticBlob = kLiteralNum * 3 + kDistNum * 3 + 288 + 32;

// ---- small host helpers ----------------------------------------------------------------------------
struct HostBits { // carries the sub-byte tail of a flushed stream on the host (PendingBuffer's `bits`, :23-24)
	uint32_t bits = 0;
	int count = 0;
	void put(std::vector<uint8_t> &out, uint32_t v, int n) {
		bits |= v << count;
		count += n;
		while (count >= 8) {
			out.push_back((uint8_t)bits);
			bits >>= 8;
			count -= 8;
		}
	}
	void align(std::vector<uint8_t> &out) {
		if (count > 0) out.push_back((uint8_t)bits);
		bits = 0;
		count = 0;
	}
};

struct PinnedBuf {
	uint8_t *p = nullptr;
	size_t cap = 0;
	int ensure(size_t n) {
		if (n <= cap) return B200Z_OK;
		if (p) cudaFreeHost(p);
		p = nullptr;
		cap = 0;
		cudaError_t e = cudaHostAlloc((void **)&p, n, cudaHostAllocDefault);
		if (e != cudaSuccess) {
			set_error("cudaHostAlloc of %zu bytes failed: %s", n, cudaGetErrorString(e));
			return B200Z_E_NOMEM;
		}
		cap = n;
		return B200Z_OK;
	}
	~PinnedBuf() {
		if (p) cudaFreeHost(p);
	}
};

struct DevBuf {
	uint8_t *p = nullptr;
	size_t cap = 0;
	int ensure(size_t n) {
		if (n <= cap) return B200Z_OK;
		if (p) cudaFree(p);
		p = nullptr;
		cap = 0;
		cudaError_t e = cudaMalloc((void **)&p, n);
		if (e != cudaSuccess) {
			set_error("cudaMalloc of %zu bytes failed: %s", n, cudaGetErrorString(e));
			return B200Z_E_NOMEM;
		}
		cap = n;
		return B200Z_OK;
	}
	~DevBuf() {
		if (p) cudaFree(p);
	}
};

// Runs one plan end to end from host buffers: pinned staging, H2D, kernels, D2H.
struct HostRunResult {
	std::vector<int64_t> out_len, in_used;
	std::vector<int32_t> status;
	std::vector<uint32_t> check;
};

static int run_plan_host(b200z_plan *plan, const uint8_t *const *in, PinnedBuf &hin, PinnedBuf &hout, DevBuf &din,
                         DevBuf &dout, DevBuf &dmeta, HostRunResult &r, bool fetch_all_out, const uint32_t *check_seed = nullptr) {
	const int n = plan->n;
	int rc;
	if ((rc = hin.ensure((size_t)plan->in_bytes + 256))) return rc;
	if ((rc = din.ensure((size_t)plan->in_bytes + 256))) return rc;
	if ((rc = dout.ensure((size_t)plan->out_bytes + 256))) return rc;
	const size_t meta_bytes = (size_t)n * (8 + 8 + 4 + 4) + 256;
	if ((rc = dmeta.ensure(meta_bytes))) return rc;
	for (int i = 0; i < n; i++)
		if (plan->in_len[i]) memcpy(hin.p + plan->in_off[i], in[i], (size_t)plan->in_len[i]);
	cudaStream_t s = 0;
	int64_t used = 0; // (a plan run below its capacity: b200z_inflate_plan_set_lengths)
	for (int i = 0; i < n; i++) used = std::max(used, plan->in_off[i] + plan->in_len[i]);
	used = std::min<int64_t>(plan->in_bytes, (used + 255) / 256 * 256);
	B200Z_CUDA(cudaMemcpyAsync(din.p, hin.p, (size_t)used, cudaMemcpyHostToDevice, s));
	int64_t *d_out_len = reinterpret_cast<int64_t *>(dmeta.p);
	int64_t *d_in_used = d_out_len + n;
	int32_t *d_status = reinterpret_cast<int32_t *>(d_in_used + n);
	uint32_t *d_check = reinterpret_cast<uint32_t *>(d_status + n);
	if (check_seed) B200Z_CUDA(cudaMemcpyAsync(d_check, check_seed, 4ull * n, cudaMemcpyHostToDevice, s)); // running values
	rc = b200z_plan_run(plan, din.p, dout.p, d_out_len, d_status, d_check, d_in_used, (void *)s);
	if (rc) return rc;
	r.out_len.assign(n, 0);
	r.in_used.assign(n, 0);
	r.status.assign(n, 0);
	r.check.assign(n, 0);
	B200Z_CUDA(cudaMemcpyAsync(r.out_len.data(), d_out_len, 8ull * n, cudaMemcpyDeviceToHost, s));
	B200Z_CUDA(cudaMemcpyAsync(r.in_used.data(), d_in_used, 8ull * n, cudaMemcpyDeviceToHost, s));
	B200Z_CUDA(cudaMemcpyAsync(r.status.data(), d_status, 4ull * n, cudaMemcpyDeviceToHost, s));
	B200Z_CUDA(cudaMemcpyAsync(r.check.data(), d_check, 4ull * n, cudaMemcpyDeviceToHost, s));
	if ((rc = hout.ensure((size_t)plan->out_bytes + 256))) return rc;
	if (fetch_all_out) {
		B200Z_CUDA(cudaMemcpyAsync(hout.p, dout.p, (size_t)plan->out_bytes, cudaMemcpyDeviceToHost, s));
		B200Z_CUDA(cudaStreamSynchronize(s));
	} else {
		B200Z_CUDA(cudaStreamSynchronize(s));
		for (int i = 0; i < n; i++) {
			if (r.out_len[i] > 0)
				B200Z_CUDA(cudaMemcpyAsync(hout.p + plan->out_off[i], dout.p + plan->out_off[i], (size_t)r.out_len[i],
				                           cudaMemcpyDeviceToHost, s));
		}
		B200Z_CUDA(cudaStreamSynchronize(s));
	}
	return B200Z_OK;
}

} // namespace b200z

using namespace b200z;

extern "C" {

const char *b200z_last_error(void) { return g_err.c_str(); }
int b200z_version(void) { return 100; }

int b200z_init(int device) {
	{
		std::lock_guard<std::mutex> lk(g_mu);
		int cnt = 0;
		cudaError_t e = cudaGetDeviceCount(&cnt);
		if (e != cudaSuccess || cnt == 0) {
			set_error("no CUDA device: libb200z has no CPU fallback (%s)", e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
			return B200Z_E_CUDA;
		}
		if (device < 0 || device >= cnt) {
			set_error("device %d out of range (%d devices)", device, cnt);
			return B200Z_E_ARG;
		}
		B200Z_CUDA(cudaSetDevice(device));
		t_device = device;
	}
	return checksum_init_tables();
}

int b200z_static_tables_size(void) { return kStaticBlob; }
int b200z_static_tables_export(uint8_t *blob, int32_t cap) {
	if (!blob || cap < kStaticBlob) {
		set_error("static table blob needs %d bytes", kStaticBlob);
		return B200Z_E_ARG;
	}
	fill_static_blob(blob);
	return B200Z_OK;
}
int b200z_static_tables_import(const uint8_t *blob, int32_t len) {
	// The kernels derive the static codes arithmetically (b200z_core.cuh static_lcode/static_llen), so installing a
	// broadcast copy reduces to verifying that the sender's tables are the ones this rank would use.
	if (!blob || len != kStaticBlob) {
		set_error("static table blob has %d bytes, expected %d", len, kStaticBlob);
		return B200Z_E_ARG;
	}
	uint8_t mine[kStaticBlob];
	fill_static_blob(mine);
	if (memcmp(mine, blob, kStaticBlob) != 0) {
		set_error("static Huffman tables received from the root differ from the local ones");
		return B200Z_E_DATA;
	}
	return B200Z_OK;
}

// ncclBroadcast inside the library, for a host that owns a communicator (one process per GPU).  NCCL is not linked: the
// two entry points are taken from the libnccl the process has loaded (or can load) at run time.
typedef int (*nccl_bcast_fn)(const void *, void *, size_t, int, int, void *, cudaStream_t);
typedef const char *(*nccl_errstr_fn)(int);
int b200z_static_tables_broadcast(void *nccl_comm, int32_t root, int32_t rank, void *cuda_stream) {
	if (!nccl_comm || root < 0 || rank < 0) {
		set_error("b200z_static_tables_broadcast: communicator, root and rank are required");
		return B200Z_E_ARG;
	}
	int rc = ensure_init();
	if (rc) return rc;
	static nccl_bcast_fn bcast = nullptr;
	static nccl_errstr_fn errstr = nullptr;
	if (!bcast) {
		void *h = nullptr;
		const char *names[] = {"libnccl.so.2", "libnccl.so"};
		for (int k = 0; k < 2 && !h; k++) h = dlopen(names[k], RTLD_NOW | RTLD_NOLOAD);
		for (int k = 0; k < 2 && !h; k++) h = dlopen(names[k], RTLD_NOW | RTLD_GLOBAL);
		if (h) {
			bcast = (nccl_bcast_fn)dlsym(h, "ncclBroadcast");
			errstr = (nccl_errstr_fn)dlsym(h, "ncclGetErrorString");
		}
		if (!bcast) {
			set_error("b200z_static_tables_broadcast: no libnccl in this process (dlopen libnccl.so.2 failed)");
			return B200Z_E_UNSUPPORTED;
		}
	}
	cudaStream_t s = (cudaStream_t)cuda_stream;
	uint8_t *d = nullptr;
	B200Z_CUDA(cudaMalloc(&d, kStaticBlob));
	uint8_t blob[kStaticBlob];
	cudaError_t e = cudaSuccess;
	if (rank == root) {
		fill_static_blob(blob);
		e = cudaMemcpyAsync(d, blob, kStaticBlob, cudaMemcpyHostToDevice, s);
	}
	int nr = 0;
	if (e == cudaSuccess) nr = bcast(d, d, (size_t)kStaticBlob, /* ncclUint8 */ 1, root, nccl_comm, s);
	if (e == cudaSuccess && nr == 0) e = cudaMemcpyAsync(blob, d, kStaticBlob, cudaMemcpyDeviceToHost, s);
	if (e == cudaSuccess && nr == 0) e = cudaStreamSynchronize(s);
	cudaFree(d);
	if (nr != 0) {
		set_error("ncclBroadcast failed: %s", errstr ? errstr(nr) : "?");
		return B200Z_E_CUDA;
	}
	if (e != cudaSuccess) return cuda_fail(e, "b200z_static_tables_broadcast", __FILE__, __LINE__);
	return b200z_static_tables_import(blob, kStaticBlob);
}

int64_t b200z_deflate_bound(int64_t len) { return len + (len >> 3) + 1024; }
int64_t b200z_engine_state_bytes(void) { return kFastStateBytes; }

// ---- plans -------------------------------------------------------------------------------------------
int b200z_deflate_plan_create(int32_t n, const int64_t *in_len, int level, int strategy, int wrap, int end_mode,
                              b200z_plan **plan) {
	return b200z_deflate_plan_create_ex(n, in_len, level, strategy, wrap, end_mode, nullptr, plan);
}

int b200z_deflate_plan_create_ex(int32_t n, const int64_t *in_len, int level, int strategy, int wrap, int end_mode,
                                 const b200z_history *hist, b200z_plan **plan) {
	if (!plan || n < 0 || (n > 0 && !in_len)) {
		set_error("bad arguments");
		return B200Z_E_ARG;
	}
	if (level == -1) level = 6;
	if (level < 0 || level > 9) {
		set_error("level");
		return B200Z_E_ARG;
	}
	if (strategy < 0 || strategy > 2 || wrap < 0 || wrap > B200Z_WRAP_RAW_CRC32 || end_mode < 0 || end_mode > 2) {
		set_error("strategy/wrap/end_mode");
		return B200Z_E_ARG;
	}
	int rc = ensure_init();
	if (rc) return rc;
	DeviceGuard guard(current_device());
	b200z_plan *p = new b200z_plan();
	p->device = current_device();
	p->kind = 0;
	p->n = n;
	p->level = level;
	p->strategy = strategy;
	p->wrap = wrap;
	p->end_mode = end_mode;
	p->in_len.assign(in_len, in_len + n);
	if (hist && n > 0 && level <= 4) {
		// levels 0-4: the call pattern and the engine state between segments (header: "streams with history")
		if (hist->chunk_count) {
			if (!hist->chunk_len) {
				set_error("history: chunk_count without chunk_len");
				delete p;
				return B200Z_E_ARG;
			}
			p->sched_cum.resize(n);
			for (int i = 0; i < n; i++) {
				int64_t sum = 0;
				for (int k = 0; k < hist->chunk_count[i]; k++) {
					const int64_t c = hist->chunk_len[i] ? hist->chunk_len[i][k] : -1;
					if (c < 0) {
						set_error("stream %d: SetInput size %d", i, k);
						delete p;
						return B200Z_E_ARG;
					}
					sum += c;
					p->sched_cum[i].push_back((uint32_t)sum);
				}
				if (hist->chunk_count[i] < 0 || (hist->chunk_count[i] > 0 && sum != in_len[i])) {
					set_error("stream %d: the SetInput sizes add up to %lld, the stream has %lld bytes", i, (long long)sum,
					          (long long)in_len[i]);
					delete p;
					return B200Z_E_ARG;
				}
			}
		}
		if (hist->undrained_last) p->undrained.assign(hist->undrained_last, hist->undrained_last + n);
		if (hist->engine_state && level >= 1) p->engine_state.assign(hist->engine_state, hist->engine_state + n);
		if (hist->stored_state && level == 0) p->stored_state = hist->stored_state;
	}
	if (hist && hist->kind != B200Z_HIST_NONE && n > 0) {
		if ((hist->kind != B200Z_HIST_DICTIONARY && hist->kind != B200Z_HIST_CONTINUE) || !hist->hist_len) {
			set_error("history: kind/hist_len");
			delete p;
			return B200Z_E_ARG;
		}
		if (hist->kind == B200Z_HIST_CONTINUE && level < 5) {
			// DeflateStored / DeflateFast keep window-relative state across Deflate() calls that is not a function of the
			// stream position: it has to come from the run of the previous segment
			bool have = level == 0 ? p->stored_state != nullptr : !p->engine_state.empty();
			for (void *q : p->engine_state) have = have && q != nullptr;
			if (!have) {
				set_error("continuing a stream after Flush() at levels 0-4 needs the engine state of the previous segment "
				          "(b200z_history.engine_state / stored_state)");
				delete p;
				return B200Z_E_UNSUPPORTED;
			}
		}
		p->hist_kind = hist->kind;
		p->check_seeded = hist->check_seeded != 0;
		p->hist.assign(hist->hist_len, hist->hist_len + n);
		p->pos_base.resize(n);
		p->bit_base.resize(n);
		p->hist_mask.resize(n);
		for (int i = 0; i < n; i++) {
			const int64_t H = p->hist[i];
			if (H < 0 || H > 32768 || (hist->kind == B200Z_HIST_DICTIONARY && H > kMaxDist)) {
				set_error("stream %d: history of %lld bytes (at most %d)", i, (long long)H,
				          hist->kind == B200Z_HIST_DICTIONARY ? kMaxDist : 32768);
				delete p;
				return B200Z_E_ARG;
			}
			p->pos_base[i] = (hist->pos_base && hist->kind == B200Z_HIST_CONTINUE) ? hist->pos_base[i] : H;
			p->bit_base[i] = hist->bit_base ? hist->bit_base[i] : 0;
			if (p->pos_base[i] < H || p->pos_base[i] > 0xFFFF0000ll || p->bit_base[i] < 0 || p->bit_base[i] > 7) {
				set_error("stream %d: pos_base/bit_base", i);
				delete p;
				return B200Z_E_ARG;
			}
			if (hist->hist_mask && hist->hist_mask[i]) p->hist_mask[i].assign(hist->hist_mask[i], hist->hist_mask[i] + H);
			p->in_len[i] += H; // the input slot holds history + data
		}
	}
	rc = deflate_plan_build(p);
	if (rc) {
		p->ws.release();
		delete p;
		return rc;
	}
	*plan = p;
	return B200Z_OK;
}

int b200z_inflate_plan_create(int32_t n, const int64_t *comp_len, const int64_t *out_cap, int wrap, b200z_plan **plan) {
	return b200z_inflate_plan_create_ex(n, comp_len, out_cap, wrap, nullptr, plan);
}

int b200z_inflate_plan_create_ex(int32_t n, const int64_t *comp_len, const int64_t *out_cap, int wrap, const int64_t *dict_len,
                                 b200z_plan **plan) {
	if (!plan || n < 0 || (n > 0 && (!comp_len || !out_cap)) || wrap < 0 || wrap > B200Z_WRAP_RAW_CRC32) {
		set_error("bad arguments");
		return B200Z_E_ARG;
	}
	int rc = ensure_init();
	if (rc) return rc;
	DeviceGuard guard(current_device());
	b200z_plan *p = new b200z_plan();
	p->device = current_device();
	p->kind = 1;
	p->n = n;
	p->wrap = wrap;
	p->in_len.assign(comp_len, comp_len + n);
	p->out_cap.assign(out_cap, out_cap + n);
	if (dict_len && n > 0) {
		p->hist_kind = B200Z_HIST_DICTIONARY;
		p->hist.assign(dict_len, dict_len + n);
		for (int i = 0; i < n; i++) {
			if (p->hist[i] < 0 || p->hist[i] > 32768) { // OutputWindow.CopyDict keeps the last WindowSize bytes (:160-166)
				set_error("stream %d: dictionary of %lld bytes (at most 32768)", i, (long long)p->hist[i]);
				delete p;
				return B200Z_E_ARG;
			}
			p->in_len[i] += p->hist[i];
		}
	}
	rc = inflate_plan_build(p);
	if (rc) {
		p->ws.release();
		delete p;
		return rc;
	}
	*plan = p;
	return B200Z_OK;
}

int b200z_inflate_plan_set_start_bits(b200z_plan *plan, const int32_t *start_bit) {
	DeviceGuard guard(plan ? plan->device : -1);
	if (!plan || plan->kind != 1 || (plan->n > 0 && !start_bit)) {
		set_error("bad arguments");
		return B200Z_E_ARG;
	}
	if (plan->wrap != B200Z_WRAP_RAW && plan->wrap != B200Z_WRAP_RAW_CRC32) {
		set_error("start bits are for raw streams (a framed stream starts behind its header)");
		return B200Z_E_ARG;
	}
	std::vector<uint32_t> sb((size_t)plan->n);
	for (int i = 0; i < plan->n; i++) {
		if (start_bit[i] < 0 || start_bit[i] > 7) {
			set_error("stream %d: start bit %d (0..7)", i, start_bit[i]);
			return B200Z_E_ARG;
		}
		sb[(size_t)i] = (uint32_t)start_bit[i];
	}
	if (plan->n) B200Z_CUDA(cudaMemcpy(plan->ws.at<uint32_t>(plan->o_start_bit), sb.data(), 4ull * plan->n, cudaMemcpyHostToDevice));
	plan->has_start_bits = true;
	return B200Z_OK;
}

int b200z_inflate_plan_set_lengths(b200z_plan *plan, const int64_t *comp_len, const int64_t *dict_len) {
	DeviceGuard guard(plan ? plan->device : -1);
	if (!plan || plan->kind != 1 || (plan->n > 0 && !comp_len)) {
		set_error("bad arguments");
		return B200Z_E_ARG;
	}
	const int n = plan->n;
	std::vector<int64_t> dl((size_t)n);
	std::vector<uint32_t> d32((size_t)n);
	for (int i = 0; i < n; i++) {
		const int64_t D = dict_len ? dict_len[i] : 0;
		if (comp_len[i] < 0 || comp_len[i] > plan->comp_cap[(size_t)i] || D < 0 || D > plan->dict_cap[(size_t)i]) {
			set_error("stream %d: %lld compressed / %lld dictionary bytes exceed what the plan was created for (%lld / %lld)", i,
			          (long long)comp_len[i], (long long)D, (long long)plan->comp_cap[(size_t)i], (long long)plan->dict_cap[(size_t)i]);
			return B200Z_E_ARG;
		}
		dl[(size_t)i] = comp_len[i];
		d32[(size_t)i] = (uint32_t)D;
	}
	for (int i = 0; i < n; i++) { // the dictionary ends where the compressed bytes start
		if (!plan->hist.empty()) plan->hist[(size_t)i] = d32[(size_t)i];
		plan->in_off[(size_t)i] = plan->comp_off[(size_t)i] - d32[(size_t)i];
		plan->in_len[(size_t)i] = comp_len[i] + d32[(size_t)i];
	}
	if (n) {
		B200Z_CUDA(cudaMemcpy(plan->ws.at<int64_t>(plan->o_in_len), dl.data(), 8ull * n, cudaMemcpyHostToDevice));
		B200Z_CUDA(cudaMemcpy(plan->ws.at<uint32_t>(plan->o_hist), d32.data(), 4ull * n, cudaMemcpyHostToDevice));
	}
	return B200Z_OK;
}

int b200z_plan_get_restart_points(b200z_plan *plan, int64_t *bit, int64_t *out_pos, void *cuda_stream) {
	DeviceGuard guard(plan ? plan->device : -1);
	if (!plan || plan->kind != 1 || (plan->n > 0 && (!bit || !out_pos))) {
		set_error("bad arguments");
		return B200Z_E_ARG;
	}
	if (plan->n == 0) return B200Z_OK;
	std::vector<int64_t> rp(2 * (size_t)plan->n);
	cudaStream_t s = (cudaStream_t)cuda_stream;
	B200Z_CUDA(cudaMemcpyAsync(rp.data(), plan->ws.at<int64_t>(plan->o_restart), 16ull * plan->n, cudaMemcpyDeviceToHost, s));
	B200Z_CUDA(cudaStreamSynchronize(s));
	for (int i = 0; i < plan->n; i++) {
		bit[i] = rp[2 * (size_t)i];
		out_pos[i] = rp[2 * (size_t)i + 1];
	}
	return B200Z_OK;
}

int b200z_plan_get_stats(b200z_plan *plan, uint32_t *v, int32_t cap, void *cuda_stream) {
	DeviceGuard guard(plan ? plan->device : -1);
	if (!plan || plan->kind != 1 || !v || cap < 0) {
		set_error("bad arguments");
		return B200Z_E_ARG;
	}
	return inflate_plan_stats(plan, v, cap, (cudaStream_t)cuda_stream);
}

int b200z_plan_get_match_table(b200z_plan *plan, int32_t i, uint16_t *link, uint32_t *ab, void *cuda_stream) {
	DeviceGuard guard(plan ? plan->device : -1);
	if (!plan || plan->kind != 0 || plan->level < 5 || i < 0 || i >= plan->n || !ab) {
		set_error("bad arguments");
		return B200Z_E_ARG;
	}
	return deflate_plan_match_table(plan, i, link, ab, (cudaStream_t)cuda_stream);
}

int b200z_plan_set_timing(b200z_plan *plan, int enable) {
	if (!plan) return B200Z_E_ARG;
	plan->timing = enable != 0;
	plan->ev_used = 0;
	return B200Z_OK;
}

int b200z_plan_get_timings(b200z_plan *plan, char *names, int32_t names_cap, float *ms, int32_t cap, int32_t *count) {
	DeviceGuard guard(plan ? plan->device : -1);
	if (!plan || !ms || !count) return B200Z_E_ARG;
	*count = 0;
	std::string nm;
	for (int i = 0; i + 1 < plan->ev_used && *count < cap; i++) {
		float t = 0;
		cudaError_t e = cudaEventElapsedTime(&t, plan->ev[i], plan->ev[i + 1]);
		if (e != cudaSuccess) return cuda_fail(e, "cudaEventElapsedTime", __FILE__, __LINE__);
		ms[*count] = t;
		nm += plan->ev_name[i];
		nm += ";";
		++*count;
	}
	if (names && names_cap > 0) {
		strncpy(names, nm.c_str(), (size_t)names_cap - 1);
		names[names_cap - 1] = 0;
	}
	return B200Z_OK;
}

int b200z_plan_destroy(b200z_plan *plan) {
	DeviceGuard guard(plan ? plan->device : -1);
	if (!plan) return B200Z_OK;
	for (cudaEvent_t e : plan->ev) cudaEventDestroy(e);
	plan->ws.release();
	delete plan;
	return B200Z_OK;
}
int64_t b200z_plan_in_bytes(const b200z_plan *p) { return p->in_bytes; }
int64_t b200z_plan_out_bytes(const b200z_plan *p) { return p->out_bytes; }
int64_t b200z_plan_in_offset(const b200z_plan *p, int32_t i) { return p->in_off[i]; }
int64_t b200z_plan_data_offset(const b200z_plan *p, int32_t i) {
	return p->in_off[i] + (p->hist.empty() ? 0 : p->hist[i]); // behind the history / dictionary
}
int64_t b200z_plan_out_offset(const b200z_plan *p, int32_t i) { return p->out_off[i]; }
int64_t b200z_plan_out_capacity(const b200z_plan *p, int32_t i) { return p->out_cap[i]; }
int64_t b200z_plan_workspace_bytes(const b200z_plan *p) { return p->ws.size; }
int32_t b200z_plan_launches(const b200z_plan *p) { return p->launches; }

int b200z_plan_run(b200z_plan *plan, const uint8_t *d_in, uint8_t *d_out, int64_t *d_out_len, int32_t *d_status,
                   uint32_t *d_check, int64_t *d_in_used, void *cuda_stream) {
	return b200z_plan_run_stages(plan, d_in, d_out, d_out_len, d_status, d_check, d_in_used, B200Z_STAGE_SEARCH | B200Z_STAGE_ENCODE,
	                             cuda_stream);
}

int b200z_plan_run_stages(b200z_plan *plan, const uint8_t *d_in, uint8_t *d_out, int64_t *d_out_len, int32_t *d_status,
                          uint32_t *d_check, int64_t *d_in_used, int stages, void *cuda_stream) {
	DeviceGuard guard(plan ? plan->device : -1);
	if (!plan || !d_in || !d_out || !d_out_len || !d_status || (stages & ~3) || stages == 0) {
		set_error("bad arguments");
		return B200Z_E_ARG;
	}
	cudaStream_t s = (cudaStream_t)cuda_stream;
	if (plan->kind == 0) return deflate_plan_run(plan, d_in, d_out, d_out_len, d_status, d_check, d_in_used, s, stages);
	if (!(stages & B200Z_STAGE_ENCODE)) return B200Z_OK; // an inflate plan is a single stage
	return inflate_plan_run(plan, d_in, d_out, d_out_len, d_status, d_check, d_in_used, s);
}

} // extern "C" (reopened below)

// ---- packing the produced streams back to back (so a caller copies only what was produced) -----------------
namespace b200z {
__global__ void k_pack_offsets(int n, const int64_t *__restrict__ len, int64_t *__restrict__ off) {
	// n is a batch size (thousands at most): one thread block, serial carry between 1024-element chunks
	__shared__ int64_t s_part[32];
	__shared__ int64_t s_carry;
	if (threadIdx.x == 0) s_carry = 0;
	__syncthreads();
	for (int base = 0; base < n; base += 1024) {
		const int i = base + threadIdx.x;
		const int64_t v = i < n ? ((len[i] + 15) & ~15ll) : 0; // 16-byte aligned starts: vector copies on both sides
		int64_t incl = v;
		for (int o = 1; o < 32; o <<= 1) {
			const int64_t t = __shfl_up_sync(0xffffffffu, incl, o);
			if ((threadIdx.x & 31) >= o) incl += t;
		}
		if ((threadIdx.x & 31) == 31) s_part[threadIdx.x >> 5] = incl;
		__syncthreads();
		int64_t woff = 0;
		for (int k = 0; k < (int)(threadIdx.x >> 5); k++) woff += s_part[k];
		const int64_t carry = s_carry;
		if (i < n) off[i] = carry + woff + incl - v;
		__syncthreads();
		if (threadIdx.x == 1023) s_carry = carry + woff + incl;
		__syncthreads();
	}
	if (threadIdx.x == 0) off[n] = s_carry;
}

__global__ void __launch_bounds__(256)
    k_pack(const uint8_t *__restrict__ out, const int64_t *__restrict__ out_off, const int64_t *__restrict__ len,
           const int64_t *__restrict__ off, uint8_t *__restrict__ packed) {
	const int i = blockIdx.x;
	const uint8_t *src = out + out_off[i];
	uint8_t *dst = packed + off[i];
	const int64_t nb = len[i];
	const int64_t nv = (nb + 15) >> 4; // the slot is 256-byte aligned and at least 16 bytes longer than the data
	const uint4 *sv = reinterpret_cast<const uint4 *>(src);
	uint4 *dv = reinterpret_cast<uint4 *>(dst);
	for (int64_t k = threadIdx.x; k < nv; k += blockDim.x) dv[k] = sv[k];
}
} // namespace b200z

extern "C" int b200z_plan_pack(b200z_plan *plan, const uint8_t *d_out, const int64_t *d_out_len, uint8_t *d_packed,
                               int64_t *d_packed_off, void *cuda_stream) {
	DeviceGuard guard(plan ? plan->device : -1);
	if (!plan || !d_out || !d_out_len || !d_packed || !d_packed_off) {
		set_error("bad arguments");
		return B200Z_E_ARG;
	}
	if (plan->n == 0) return B200Z_OK;
	cudaStream_t s = (cudaStream_t)cuda_stream;
	k_pack_offsets<<<1, 1024, 0, s>>>(plan->n, d_out_len, d_packed_off);
	k_pack<<<plan->n, 256, 0, s>>>(d_out, plan->ws.at<int64_t>(plan->o_out_off), d_out_len, d_packed_off, d_packed);
	B200Z_CUDA(cudaGetLastError());
	return B200Z_OK;
}

extern "C" {

// ---- checksums ---------------------------------------------------------------------------------------
static int checksum_host(int kind, const uint8_t *buf, int64_t len, uint32_t *value) {
	if (!value || len < 0 || (len > 0 && !buf)) {
		set_error("bad arguments");
		return B200Z_E_ARG;
	}
	int rc = ensure_init();
	if (rc) return rc;
	if (len == 0) return B200Z_OK;
	DevBuf d, meta;
	if ((rc = d.ensure((size_t)len + 256))) return rc;
	B200Z_CUDA(cudaMemcpy(d.p, buf, (size_t)len, cudaMemcpyHostToDevice));
	std::vector<CkTile> tiles;
	checksum_tiles(&len, 1, tiles, kind);
	const size_t tb = sizeof(CkTile) * tiles.size();
	if ((rc = meta.ensure(tb + 256))) return rc;
	int64_t *d_off = reinterpret_cast<int64_t *>(meta.p);
	int64_t *d_len = d_off + 1;
	unsigned long long *d_acc = reinterpret_cast<unsigned long long *>(d_len + 1);
	uint32_t *d_val = reinterpret_cast<uint32_t *>(d_acc + 2);
	CkTile *d_tiles = reinterpret_cast<CkTile *>(meta.p + 64);
	int64_t zero = 0;
	B200Z_CUDA(cudaMemcpy(d_off, &zero, 8, cudaMemcpyHostToDevice));
	B200Z_CUDA(cudaMemcpy(d_len, &len, 8, cudaMemcpyHostToDevice));
	B200Z_CUDA(cudaMemcpy(d_val, value, 4, cudaMemcpyHostToDevice));
	B200Z_CUDA(cudaMemcpy(d_tiles, tiles.data(), tb, cudaMemcpyHostToDevice));
	rc = checksum_launch(kind, d.p, d_off, d_len, 1, d_tiles, (int32_t)tiles.size(), d_acc, d_val, 0, 0);
	if (rc) return rc;
	B200Z_CUDA(cudaMemcpy(value, d_val, 4, cudaMemcpyDeviceToHost));
	return B200Z_OK;
}
int b200z_crc32(const uint8_t *buf, int64_t len, uint32_t *value) { return checksum_host(0, buf, len, value); }
int b200z_adler32(const uint8_t *buf, int64_t len, uint32_t *value) { return checksum_host(1, buf, len, value); }

int b200z_checksum_batch_device(int kind, const uint8_t *d_data, const int64_t *off, const int64_t *len, int32_t n,
                                uint32_t *d_value, void *cuda_stream) {
	if (kind < 0 || kind > 1 || n < 0 || (n > 0 && (!d_data || !off || !len || !d_value))) {
		set_error("bad arguments");
		return B200Z_E_ARG;
	}
	int rc = ensure_init();
	if (rc) return rc;
	if (n == 0) return B200Z_OK;
	cudaStream_t s = (cudaStream_t)cuda_stream;
	std::vector<CkTile> tiles;
	checksum_tiles(len, n, tiles, kind);
	const size_t tb = sizeof(CkTile) * tiles.size();
	uint8_t *meta = nullptr;
	const size_t bytes = 16ull * n + 16ull * n + tb + 256;
	B200Z_CUDA(cudaMallocAsync((void **)&meta, bytes, s));
	int64_t *d_off = reinterpret_cast<int64_t *>(meta);
	int64_t *d_len = d_off + n;
	unsigned long long *d_acc = reinterpret_cast<unsigned long long *>(d_len + n);
	CkTile *d_tiles = reinterpret_cast<CkTile *>(d_acc + 2 * n);
	B200Z_CUDA(cudaMemcpyAsync(d_off, off, 8ull * n, cudaMemcpyHostToDevice, s));
	B200Z_CUDA(cudaMemcpyAsync(d_len, len, 8ull * n, cudaMemcpyHostToDevice, s));
	if (tb) B200Z_CUDA(cudaMemcpyAsync(d_tiles, tiles.data(), tb, cudaMemcpyHostToDevice, s));
	rc = checksum_launch(kind, d_data, d_off, d_len, n, d_tiles, (int32_t)tiles.size(), d_acc, d_value, 0, s);
	B200Z_CUDA(cudaStreamSynchronize(s)); // the pageable descriptor copies above must finish before `tiles` dies
	B200Z_CUDA(cudaFreeAsync(meta, s));
	return rc;
}

static const char *inflate_detail_msg(int detail);

// ---- host-buffer batch calls ----------------------------------------------------------------------------
static void zlib_header(int level, uint8_t h[2], bool preset_dict = false) { // Deflater.cs:436-464 (trap T11)
	int header = (8 + (7 << 4)) << 8;
	int level_flags = (level - 1) >> 1;
	if (level_flags < 0 || level_flags > 3) level_flags = 3;
	header |= level_flags << 6;
	if (preset_dict) header |= 0x20; // DeflaterConstants.PRESET_DICT
	header += 31 - (header % 31);
	h[0] = (uint8_t)(header >> 8);
	h[1] = (uint8_t)header;
}

// ---- host-buffer pipelines ---------------------------------------------------------------------------------
// What a host that keeps a GPU busy does, inside the library: a pipeline owns the plan of one batch shape, `depth` slots of
// pinned staging + device buffers and three streams.  submit() stages a batch from host pointers and enqueues upload and
// kernels without waiting; collect() waits for the oldest batch, fetches exactly the bytes produced and hands them to the
// caller's buffers.  With depth >= 2 the upload of batch i+1 and the download of batch i-1 overlap the kernels of batch i.
// Host pointers that CUDA knows as pinned (cudaHostAlloc / cudaHostRegister) are the DMA source / target directly; plain
// pageable memory goes through the slot's pinned staging, copied by a few host threads.
} // extern "C"

namespace b200z {

static void host_parallel_for(int n_items, int64_t total_bytes, const std::function<void(int, int)> &fn) {
	// fn(first, last) over [0, n_items), on up to 8 threads when there is enough to copy
	int nt = total_bytes >= (8ll << 20) ? 8 : 1;
	const int hw = (int)std::thread::hardware_concurrency();
	if (hw > 0 && nt > hw) nt = hw;
	if (nt > n_items) nt = n_items > 0 ? n_items : 1;
	if (nt <= 1) {
		fn(0, n_items);
		return;
	}
	std::vector<std::thread> th;
	for (int t = 0; t < nt; t++) th.emplace_back([=, &fn] { fn((int)((int64_t)n_items * t / nt), (int)((int64_t)n_items * (t + 1) / nt)); });
	for (auto &t : th) t.join();
}

static bool host_ptr_is_pinned(const void *p) {
	cudaPointerAttributes a;
	if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
		cudaGetLastError();
		return false;
	}
	return a.type == cudaMemoryTypeHost;
}

struct PipeMeta { // per slot, pinned: what a run reports
	int64_t *out_len, *in_used, *poff;
	int32_t *status;
	uint32_t *check;
};

struct PipeSlot {
	PinnedBuf hin, hout, hmeta;
	DevBuf din, dout, dpack, dmeta;
	PipeMeta h, d;
	cudaEvent_t ev_up = nullptr, ev_run = nullptr;
	bool busy = false;
};

} // namespace b200z

struct b200z_pipeline {
	b200z_plan *plan = nullptr;
	int depth = 1;
	std::vector<b200z::PipeSlot> slots;
	cudaStream_t s_up = nullptr, s_run = nullptr, s_down = nullptr;
	int64_t head = 0, tail = 0; // batches submitted / collected
	int64_t in_total = 0;
	std::vector<int64_t> data_off; // where stream i's data goes in the input blob
};

namespace b200z {

static void pipe_meta_layout(uint8_t *base, int n, PipeMeta &m) {
	m.out_len = reinterpret_cast<int64_t *>(base);
	m.in_used = m.out_len + n;
	m.poff = m.in_used + n;
	m.status = reinterpret_cast<int32_t *>(m.poff + n + 1);
	m.check = reinterpret_cast<uint32_t *>(m.status + n);
}
static size_t pipe_meta_bytes(int n) { return (size_t)n * (8 + 8 + 8 + 4 + 4) + 8 + 256; }

static int pipeline_finish_create(b200z_plan *plan, int depth, b200z_pipeline **out) {
	DeviceGuard guard(plan->device);
	if (depth < 1 || depth > 8) {
		b200z_plan_destroy(plan);
		set_error("depth");
		return B200Z_E_ARG;
	}
	b200z_pipeline *p = new b200z_pipeline();
	p->plan = plan;
	p->depth = depth;
	p->slots.resize((size_t)depth);
	const int n = plan->n;
	int rc = B200Z_OK;
	auto fail = [&](int code) {
		b200z_pipeline_destroy(p);
		return code;
	};
	if (cudaStreamCreateWithFlags(&p->s_up, cudaStreamNonBlocking) != cudaSuccess || cudaStreamCreateWithFlags(&p->s_run, cudaStreamNonBlocking) != cudaSuccess ||
	    cudaStreamCreateWithFlags(&p->s_down, cudaStreamNonBlocking) != cudaSuccess) {
		set_error("cudaStreamCreate failed");
		return fail(B200Z_E_CUDA);
	}
	for (auto &sl : p->slots) {
		if ((rc = sl.hin.ensure((size_t)plan->in_bytes + 256))) return fail(rc);
		if ((rc = sl.hout.ensure((size_t)plan->out_bytes + 256))) return fail(rc);
		if ((rc = sl.hmeta.ensure(pipe_meta_bytes(n)))) return fail(rc);
		if ((rc = sl.din.ensure((size_t)plan->in_bytes + 256))) return fail(rc);
		if ((rc = sl.dout.ensure((size_t)plan->out_bytes + 256))) return fail(rc);
		if (plan->kind == 0 && (rc = sl.dpack.ensure((size_t)plan->out_bytes + 256))) return fail(rc);
		if ((rc = sl.dmeta.ensure(pipe_meta_bytes(n)))) return fail(rc);
		pipe_meta_layout(sl.hmeta.p, n, sl.h);
		pipe_meta_layout(sl.dmeta.p, n, sl.d);
		memset(sl.hin.p, 0, (size_t)plan->in_bytes + 256);
		if (cudaEventCreateWithFlags(&sl.ev_up, cudaEventDisableTiming) != cudaSuccess || cudaEventCreateWithFlags(&sl.ev_run, cudaEventDisableTiming) != cudaSuccess) {
			set_error("cudaEventCreate failed");
			return fail(B200Z_E_CUDA);
		}
		// the bytes between the slots of the input blob are never written again: clear them once
		if (cudaMemset(sl.din.p, 0, (size_t)plan->in_bytes + 256) != cudaSuccess) return fail(B200Z_E_CUDA);
	}
	p->data_off.resize((size_t)n);
	for (int i = 0; i < n; i++) {
		p->data_off[(size_t)i] = b200z_plan_data_offset(plan, i);
		p->in_total += plan->in_len[(size_t)i] - (plan->hist.empty() ? 0 : plan->hist[(size_t)i]);
	}
	*out = p;
	return B200Z_OK;
}

} // namespace b200z

extern "C" {

int b200z_deflate_pipeline_create(int32_t n, const int64_t *in_len, int level, int strategy, int wrap, int end_mode, int depth,
                                  b200z_pipeline **pipe) {
	if (!pipe) {
		set_error("bad arguments");
		return B200Z_E_ARG;
	}
	if (level == -1) level = 6;
	b200z_plan *plan = nullptr;
	// gzip: the plan delivers the raw stream and the CRC-32; collect() writes header and trailer (GzipOutputStream.cs:315-375)
	int rc = b200z_deflate_plan_create(n, in_len, level, strategy, wrap == B200Z_WRAP_GZIP ? B200Z_WRAP_RAW_CRC32 : wrap, end_mode, &plan);
	if (rc) return rc;
	plan->host_wrap = wrap;
	return pipeline_finish_create(plan, depth, pipe);
}

int b200z_inflate_pipeline_create(int32_t n, const int64_t *comp_len, const int64_t *out_cap, int wrap, int depth, b200z_pipeline **pipe) {
	if (!pipe) {
		set_error("bad arguments");
		return B200Z_E_ARG;
	}
	b200z_plan *plan = nullptr;
	int rc = b200z_inflate_plan_create(n, comp_len, out_cap, wrap, &plan);
	if (rc) return rc;
	plan->host_wrap = wrap;
	return pipeline_finish_create(plan, depth, pipe);
}

int b200z_pipeline_destroy(b200z_pipeline *p) {
	DeviceGuard guard((p && p->plan) ? p->plan->device : -1);
	if (!p) return B200Z_OK;
	if (p->s_up) cudaStreamSynchronize(p->s_up);
	if (p->s_run) cudaStreamSynchronize(p->s_run);
	if (p->s_down) cudaStreamSynchronize(p->s_down);
	for (auto &sl : p->slots) {
		if (sl.ev_up) cudaEventDestroy(sl.ev_up);
		if (sl.ev_run) cudaEventDestroy(sl.ev_run);
	}
	if (p->s_up) cudaStreamDestroy(p->s_up);
	if (p->s_run) cudaStreamDestroy(p->s_run);
	if (p->s_down) cudaStreamDestroy(p->s_down);
	b200z_plan_destroy(p->plan);
	delete p;
	return B200Z_OK;
}

int32_t b200z_pipeline_in_flight(const b200z_pipeline *p) { return p ? (int32_t)(p->head - p->tail) : 0; }

int b200z_pipeline_submit(b200z_pipeline *p, const uint8_t *const *in) {
	DeviceGuard guard((p && p->plan) ? p->plan->device : -1);
	if (!p || (p->plan->n > 0 && !in)) {
		set_error("bad arguments");
		return B200Z_E_ARG;
	}
	if (p->head - p->tail >= p->depth) {
		set_error("pipeline: %d batches in flight, collect one first", p->depth);
		return B200Z_E_STATE;
	}
	b200z_plan *plan = p->plan;
	const int n = plan->n;
	PipeSlot &sl = p->slots[(size_t)(p->head % p->depth)];
	bool all_pinned = n > 0;
	for (int i = 0; i < n && all_pinned; i++) {
		const int64_t len = plan->in_len[(size_t)i];
		if (len > 0 && !in[i]) {
			set_error("stream %d: null input", i);
			return B200Z_E_ARG;
		}
		if (len > 0 && (i < 4 || (i & 63) == 0)) all_pinned = host_ptr_is_pinned(in[i]); // (sampled: the check is not free)
	}
	if (all_pinned) {
		for (int i = 0; i < n; i++)
			if (plan->in_len[(size_t)i] > 0)
				B200Z_CUDA(cudaMemcpyAsync(sl.din.p + plan->in_off[(size_t)i], in[i], (size_t)plan->in_len[(size_t)i], cudaMemcpyHostToDevice, p->s_up));
	} else {
		host_parallel_for(n, p->in_total, [&](int a, int b) {
			for (int i = a; i < b; i++)
				if (plan->in_len[(size_t)i] > 0) memcpy(sl.hin.p + plan->in_off[(size_t)i], in[i], (size_t)plan->in_len[(size_t)i]);
		});
		B200Z_CUDA(cudaMemcpyAsync(sl.din.p, sl.hin.p, (size_t)plan->in_bytes, cudaMemcpyHostToDevice, p->s_up));
	}
	B200Z_CUDA(cudaEventRecord(sl.ev_up, p->s_up));
	B200Z_CUDA(cudaStreamWaitEvent(p->s_run, sl.ev_up, 0));
	int rc = b200z_plan_run(plan, sl.din.p, sl.dout.p, sl.d.out_len, sl.d.status, sl.d.check, sl.d.in_used, (void *)p->s_run);
	if (rc) return rc;
	if (plan->kind == 0) {
		rc = b200z_plan_pack(plan, sl.dout.p, sl.d.out_len, sl.dpack.p, sl.d.poff, (void *)p->s_run);
		if (rc) return rc;
	}
	B200Z_CUDA(cudaMemcpyAsync(sl.hmeta.p, sl.dmeta.p, pipe_meta_bytes(n) - 256, cudaMemcpyDeviceToHost, p->s_run));
	B200Z_CUDA(cudaEventRecord(sl.ev_run, p->s_run));
	sl.busy = true;
	++p->head;
	return B200Z_OK;
}

int b200z_pipeline_collect(b200z_pipeline *p, uint8_t *const *out, const int64_t *out_cap, int64_t *out_len, int64_t *in_used,
                           uint32_t *check, int32_t *status) {
	DeviceGuard guard((p && p->plan) ? p->plan->device : -1);
	if (!p || (p->plan->n > 0 && (!out || !out_cap || !out_len))) {
		set_error("bad arguments");
		return B200Z_E_ARG;
	}
	if (p->head == p->tail) {
		set_error("pipeline: nothing submitted");
		return B200Z_E_STATE;
	}
	b200z_plan *plan = p->plan;
	const int n = plan->n;
	PipeSlot &sl = p->slots[(size_t)(p->tail % p->depth)];
	B200Z_CUDA(cudaEventSynchronize(sl.ev_run)); // the run's sizes, statuses and checksums are on the host
	const int wrap = plan->host_wrap;
	int first = B200Z_OK, first_detail = 0;
	int64_t moved = 0;
	if (plan->kind == 0) {
		// ---- deflate: exactly the produced bytes cross PCIe (packed back to back on the device) ----
		const int64_t total = n ? sl.h.poff[n] : 0;
		if (total > 0) B200Z_CUDA(cudaMemcpyAsync(sl.hout.p, sl.dpack.p, (size_t)total, cudaMemcpyDeviceToHost, p->s_down));
		B200Z_CUDA(cudaStreamSynchronize(p->s_down));
		const int hdr = wrap == B200Z_WRAP_ZLIB ? 2 : (wrap == B200Z_WRAP_GZIP ? 10 : 0);
		const int trl = wrap == B200Z_WRAP_ZLIB ? 4 : (wrap == B200Z_WRAP_GZIP ? 8 : 0);
		for (int i = 0; i < n; i++) {
			int st = sl.h.status[i] & 0xFF;
			const int64_t need = sl.h.out_len[i] + hdr + trl;
			if (st == B200Z_OK && need > out_cap[i]) st = B200Z_E_NOMEM;
			out_len[i] = st == B200Z_OK ? need : 0;
			if (status) status[i] = st;
			if (check) check[i] = sl.h.check[i];
			if (in_used) in_used[i] = 0;
			if (st != B200Z_OK && first == B200Z_OK) first = st;
			if (st == B200Z_OK) moved += need;
		}
		host_parallel_for(n, moved, [&](int a, int b) {
			for (int i = a; i < b; i++) {
				if (out_len[i] == 0) continue;
				uint8_t *o = out[i];
				if (wrap == B200Z_WRAP_ZLIB) {
					zlib_header(plan->level, o);
					o += 2;
				} else if (wrap == B200Z_WRAP_GZIP) {
					// GzipOutputStream.GetHeader (:339-375) with MTIME 0 and no FNAME: 1F 8B 08 00 <mtime> 00 FF (trap T15)
					const uint8_t h[10] = {0x1F, 0x8B, 8, 0, 0, 0, 0, 0, 0, 0xFF};
					memcpy(o, h, 10);
					o += 10;
				}
				memcpy(o, sl.hout.p + sl.h.poff[i], (size_t)sl.h.out_len[i]);
				o += sl.h.out_len[i];
				const uint32_t a32 = sl.h.check[i];
				if (wrap == B200Z_WRAP_ZLIB) { // Adler32 trailer, big endian (Deflater.cs:509-514)
					o[0] = (uint8_t)(a32 >> 24);
					o[1] = (uint8_t)(a32 >> 16);
					o[2] = (uint8_t)(a32 >> 8);
					o[3] = (uint8_t)a32;
				} else if (wrap == B200Z_WRAP_GZIP) { // GetFooter (:315-337): CRC32, ISIZE = TotalIn & 0xFFFFFFFF, little endian
					const uint32_t isz = (uint32_t)((uint64_t)plan->in_len[(size_t)i] & 0xFFFFFFFFull);
					for (int k = 0; k < 4; k++) o[k] = (uint8_t)(a32 >> (8 * k));
					for (int k = 0; k < 4; k++) o[4 + k] = (uint8_t)(isz >> (8 * k));
				}
			}
		});
	} else {
		// ---- inflate: every stream's produced bytes; straight into the caller's buffers when CUDA knows them as pinned ----
		bool all_pinned = n > 0;
		for (int i = 0; i < n && all_pinned; i++)
			if (sl.h.out_len[i] > 0 && (i < 4 || (i & 63) == 0)) all_pinned = host_ptr_is_pinned(out[i]);
		for (int i = 0; i < n; i++) {
			const int64_t L = sl.h.out_len[i];
			if (L > 0)
				B200Z_CUDA(cudaMemcpyAsync(all_pinned ? out[i] : sl.hout.p + plan->out_off[(size_t)i], sl.dout.p + plan->out_off[(size_t)i], (size_t)L,
				                           cudaMemcpyDeviceToHost, p->s_down));
			moved += L;
		}
		B200Z_CUDA(cudaStreamSynchronize(p->s_down));
		if (!all_pinned)
			host_parallel_for(n, moved, [&](int a, int b) {
				for (int i = a; i < b; i++)
					if (sl.h.out_len[i] > 0) memcpy(out[i], sl.hout.p + plan->out_off[(size_t)i], (size_t)sl.h.out_len[i]);
			});
		for (int i = 0; i < n; i++) {
			const int st = sl.h.status[i];
			out_len[i] = sl.h.out_len[i];
			if (in_used) in_used[i] = sl.h.in_used[i];
			if (status) status[i] = st;
			if (check) check[i] = wrap != B200Z_WRAP_RAW ? sl.h.check[i] : 0u;
			if ((st & 0xFF) != B200Z_OK && first == B200Z_OK) {
				first = st & 0xFF;
				first_detail = (st >> 8) & 0xFF;
			}
		}
	}
	sl.busy = false;
	++p->tail;
	if (first == B200Z_E_DATA && plan->kind == 1) set_error("%s", inflate_detail_msg(first_detail)); // the reference's exception message
	else if (first != B200Z_OK) set_error("stream failed with status %d", first);
	return first;
}

} // extern "C"

// ---- host-buffer batch calls: one submit + collect on a cached pipeline of the batch's shape --------------------------
namespace b200z {
struct PipeKey {
	int kind, n, level, strategy, wrap, end_mode;
	std::vector<int64_t> a, b;
	bool operator==(const PipeKey &o) const {
		return kind == o.kind && n == o.n && level == o.level && strategy == o.strategy && wrap == o.wrap && end_mode == o.end_mode && a == o.a && b == o.b;
	}
};
struct PipeCache { // per host thread: the last few shapes keep their plan, staging and device buffers
	std::vector<std::pair<PipeKey, b200z_pipeline *>> items;
	~PipeCache() {
		for (auto &it : items) b200z_pipeline_destroy(it.second);
	}
	b200z_pipeline *find(const PipeKey &k) {
		for (size_t i = 0; i < items.size(); i++)
			if (items[i].first == k) {
				auto it = items[i];
				items.erase(items.begin() + (ptrdiff_t)i);
				items.insert(items.begin(), it);
				return it.second;
			}
		return nullptr;
	}
	void put(PipeKey k, b200z_pipeline *p) {
		items.insert(items.begin(), std::make_pair(std::move(k), p));
		while (items.size() > 4) {
			b200z_pipeline_destroy(items.back().second);
			items.pop_back();
		}
	}
	void clear() {
		for (auto &it : items) b200z_pipeline_destroy(it.second);
		items.clear();
	}
};
static thread_local PipeCache g_pipes;
struct MultiKey {
	int device;
	PipeKey key;
};
static thread_local std::vector<std::pair<MultiKey, b200z_pipeline *>> g_multi_pipes; // b200z_*_batch_multi: a few per device
} // namespace b200z

extern "C" {

int b200z_release_cached(void) { // frees what the host-buffer batch calls of this thread keep between calls
	for (auto &it : g_multi_pipes) b200z_pipeline_destroy(it.second);
	g_multi_pipes.clear();
	g_pipes.clear();
	return B200Z_OK;
}

int b200z_deflate_batch(const uint8_t *const *in, const int64_t *in_len, int32_t n, int level, int strategy, int wrap,
                        int end_mode, uint8_t *const *out, const int64_t *out_cap, int64_t *out_len, uint32_t *check,
                        int32_t *status) {
	if (n < 0 || (n > 0 && (!in || !in_len || !out || !out_cap || !out_len))) {
		set_error("bad arguments");
		return B200Z_E_ARG;
	}
	if (level == -1) level = 6;
	PipeKey key{0, n, level, strategy, wrap, end_mode, std::vector<int64_t>(in_len, in_len + n), {}};
	b200z_pipeline *p = g_pipes.find(key);
	if (!p) {
		int rc = b200z_deflate_pipeline_create(n, in_len, level, strategy, wrap, end_mode, 1, &p);
		if (rc) return rc;
		g_pipes.put(std::move(key), p);
	}
	int rc = b200z_pipeline_submit(p, in);
	if (rc) return rc;
	return b200z_pipeline_collect(p, out, out_cap, out_len, nullptr, check, status);
}

int b200z_inflate_batch(const uint8_t *const *in, const int64_t *in_len, int32_t n, int wrap, uint8_t *const *out,
                        const int64_t *out_cap, int64_t *out_len, int64_t *in_used, uint32_t *check, int32_t *status) {
	if (n < 0 || (n > 0 && (!in || !in_len || !out || !out_cap || !out_len))) {
		set_error("bad arguments");
		return B200Z_E_ARG;
	}
	PipeKey key{1, n, 0, 0, wrap, 0, std::vector<int64_t>(in_len, in_len + n), std::vector<int64_t>(out_cap, out_cap + n)};
	b200z_pipeline *p = g_pipes.find(key);
	if (!p) {
		int rc = b200z_inflate_pipeline_create(n, in_len, out_cap, wrap, 1, &p);
		if (rc) return rc;
		g_pipes.put(std::move(key), p);
	}
	int rc = b200z_pipeline_submit(p, in);
	if (rc) return rc;
	return b200z_pipeline_collect(p, out, out_cap, out_len, in_used, check, status);
}

// ---- one host thread, several GPUs ----------------------------------------------------------------------------------
// The streams of a batch are independent (a fresh Deflater / Inflater each): they are cut into contiguous ranges of
// about equal bytes (SURVEY.md 8e), every range goes to one device's pipeline, all submits are issued before the first
// collect -- the devices work at the same time, the calling thread only stages and waits.
int b200z_device_count(void) {
	int cnt = 0;
	if (cudaGetDeviceCount(&cnt) != cudaSuccess) {
		cudaGetLastError();
		return 0;
	}
	return cnt;
}

int b200z_partition_by_bytes(const int64_t *len, int32_t n, int32_t parts, int32_t *first) {
	if (n < 0 || parts < 1 || !first || (n > 0 && !len)) {
		set_error("bad arguments");
		return B200Z_E_ARG;
	}
	int64_t total = 0;
	for (int i = 0; i < n; i++) total += len[i] > 0 ? len[i] : 0;
	// part r starts at the first stream whose cumulative start offset is >= floor(r T / R)
	int32_t i = 0;
	int64_t start = 0; // cumulative start of stream i
	first[0] = 0;
	for (int r = 1; r < parts; r++) {
		const int64_t cut = (int64_t)(((__int128)total * r) / parts);
		while (i < n && start < cut) {
			start += len[i] > 0 ? len[i] : 0;
			++i;
		}
		first[r] = i;
	}
	first[parts] = n;
	return B200Z_OK;
}

} // extern "C"

namespace b200z {
static b200z_pipeline *multi_find(int device, const PipeKey &k) {
	for (auto &it : g_multi_pipes)
		if (it.first.device == device && it.first.key == k) return it.second;
	return nullptr;
}
static void multi_put(int device, PipeKey k, b200z_pipeline *p) {
	int same = 0;
	for (size_t i = g_multi_pipes.size(); i-- > 0;) { // the newest four shapes per device stay; never one with a batch in flight
		if (g_multi_pipes[i].first.device != device) continue;
		if (++same >= 4 && b200z_pipeline_in_flight(g_multi_pipes[i].second) == 0) {
			b200z_pipeline_destroy(g_multi_pipes[i].second);
			g_multi_pipes.erase(g_multi_pipes.begin() + (ptrdiff_t)i);
		}
	}
	g_multi_pipes.push_back(std::make_pair(MultiKey{device, std::move(k)}, p));
}

static int multi_batch(int kind, const int32_t *devices, int32_t n_devices, const uint8_t *const *in, const int64_t *in_len, int32_t n, int level,
                       int strategy, int wrap, int end_mode, uint8_t *const *out, const int64_t *out_cap, int64_t *out_len, int64_t *in_used,
                       uint32_t *check, int32_t *status) {
	if (n < 0 || n_devices < 1 || !devices || (n > 0 && (!in || !in_len || !out || !out_cap || !out_len))) {
		set_error("bad arguments");
		return B200Z_E_ARG;
	}
	const int ndev_all = b200z_device_count();
	for (int d = 0; d < n_devices; d++)
		if (devices[d] < 0 || devices[d] >= ndev_all) {
			set_error("device %d out of range (%d devices)", devices[d], ndev_all);
			return B200Z_E_ARG;
		}
	std::vector<int32_t> first((size_t)n_devices + 1);
	int rc = b200z_partition_by_bytes(in_len, n, n_devices, first.data());
	if (rc) return rc;
	const int saved = t_device;
	std::vector<b200z_pipeline *> pipes((size_t)n_devices, nullptr);
	int result = B200Z_OK;
	for (int d = 0; d < n_devices && result == B200Z_OK; d++) {
		const int a = first[(size_t)d], cnt = first[(size_t)d + 1] - a;
		if (cnt == 0) continue;
		PipeKey key{kind, cnt, level, strategy, wrap, end_mode, std::vector<int64_t>(in_len + a, in_len + a + cnt),
		            kind == 1 ? std::vector<int64_t>(out_cap + a, out_cap + a + cnt) : std::vector<int64_t>()};
		b200z_pipeline *p = multi_find(devices[d], key);
		if (!p) {
			if ((rc = b200z_init(devices[d]))) { result = rc; break; } // (makes the device this thread's current one for the creation)
			rc = kind == 0 ? b200z_deflate_pipeline_create(cnt, in_len + a, level, strategy, wrap, end_mode, 1, &p)
			               : b200z_inflate_pipeline_create(cnt, in_len + a, out_cap + a, wrap, 1, &p);
			if (rc) { result = rc; break; }
			multi_put(devices[d], std::move(key), p);
		}
		pipes[(size_t)d] = p;
		if ((rc = b200z_pipeline_submit(p, in + a))) result = rc;
	}
	for (int d = 0; d < n_devices; d++) { // everything that was submitted is collected, whatever happened to the others
		b200z_pipeline *p = pipes[(size_t)d];
		if (!p || b200z_pipeline_in_flight(p) == 0) continue;
		const int a = first[(size_t)d];
		rc = b200z_pipeline_collect(p, out + a, out_cap + a, out_len + a, in_used ? in_used + a : nullptr, check ? check + a : nullptr,
		                            status ? status + a : nullptr);
		if (rc && result == B200Z_OK) result = rc;
	}
	t_device = saved;
	if (saved >= 0) cudaSetDevice(saved);
	return result;
}
} // namespace b200z

extern "C" {

int b200z_deflate_batch_multi(const int32_t *devices, int32_t n_devices, const uint8_t *const *in, const int64_t *in_len, int32_t n, int level,
                              int strategy, int wrap, int end_mode, uint8_t *const *out, const int64_t *out_cap, int64_t *out_len,
                              uint32_t *check, int32_t *status) {
	if (level == -1) level = 6;
	return multi_batch(0, devices, n_devices, in, in_len, n, level, strategy, wrap, end_mode, out, out_cap, out_len, nullptr, check, status);
}

int b200z_inflate_batch_multi(const int32_t *devices, int32_t n_devices, const uint8_t *const *in, const int64_t *in_len, int32_t n, int wrap,
                              uint8_t *const *out, const int64_t *out_cap, int64_t *out_len, int64_t *in_used, uint32_t *check,
                              int32_t *status) {
	return multi_batch(1, devices, n_devices, in, in_len, n, 0, 0, wrap, 0, out, out_cap, out_len, in_used, check, status);
}

// =====================================================================================================
// Streaming handles
// =====================================================================================================
struct DeflaterH {
	int level = 6, strategy = 0;
	bool raw = false;
	// Deflater.cs state bits (:96-110)
	bool flushing = false, finishing = false, finished = false;
	bool header_done = false;
	bool flushed_once = false; // a sync flush has been emitted and nothing was compressed since
	// what the engine's window has seen so far, cut to its last 32768 bytes (preset dictionary, then every compressed
	// segment); hist_mask flags the positions InsertString never saw (the last two of the dictionary / of each segment)
	std::vector<uint8_t> history, hist_mask;
	int64_t window_seen = 0;  // dictionary bytes kept + TotalIn: the SlideWindow phase of the next segment
	bool dict_set = false, deflate_called = false, started = false;
	uint32_t dict_adler = 0;
	std::vector<uint8_t> input;    // everything SetInput handed over and not yet compressed
	std::vector<uint8_t> pending;  // produced bytes not yet drained by Deflate()
	size_t pending_pos = 0;
	HostBits tail;                 // sub-byte tail carried between device runs
	int64_t total_in = 0, total_out = 0;
	uint32_t adler = 1;
	// levels 0-4 depend on the call pattern (trap T9) and keep engine state across Flush(): the sizes of the SetInput calls
	// since the last run, whether Deflate() was called behind the last of them, and what the engines carry
	std::vector<int64_t> chunks;
	bool undrained = false;
	b200z_stored_state sstate = {0, 0, 0, 0}; // level 0 (DeflateStored)
	DevBuf fstate;                            // levels 1-4 (DeflateFast: head[], prev[], scalars), on the device
	PinnedBuf hin, hout;
	DevBuf din, dout, dmeta;
};

static void deflater_remember(DeflaterH *d, const uint8_t *seg, size_t len, size_t uninserted) {
	// append a dictionary/segment to the carried window image
	d->history.insert(d->history.end(), seg, seg + len);
	d->hist_mask.insert(d->hist_mask.end(), len, 0);
	for (size_t k = 0; k < uninserted && k < len; k++) d->hist_mask[d->hist_mask.size() - 1 - k] = 1;
	if (d->history.size() > 32768) {
		const size_t cut = d->history.size() - 32768;
		d->history.erase(d->history.begin(), d->history.begin() + (ptrdiff_t)cut);
		d->hist_mask.erase(d->hist_mask.begin(), d->hist_mask.begin() + (ptrdiff_t)cut);
	}
	d->window_seen += (int64_t)len;
}

static int deflater_run_device(DeflaterH *d, int end_mode) {
	// compresses d->input as the next segment of the stream; END_FLUSH keeps the stream open and may end inside a byte
	const int64_t len = (int64_t)d->input.size();
	const int64_t H = (int64_t)d->history.size();
	const bool continuing = d->started; // an earlier segment (possibly empty) has been emitted
	b200z_history hs;
	memset(&hs, 0, sizeof hs);
	const int32_t n_chunks = (int32_t)d->chunks.size();
	const int64_t *chunk_ptr = d->chunks.data();
	const int32_t undrained = (d->undrained && n_chunks > 0) ? 1 : 0;
	void *fstate_ptr = nullptr;
	if (d->level <= 4) {
		hs.chunk_count = &n_chunks;
		hs.chunk_len = &chunk_ptr;
		hs.undrained_last = &undrained;
		if (d->level == 0) hs.stored_state = &d->sstate;
		else {
			int rc0 = d->fstate.ensure((size_t)b200z_engine_state_bytes());
			if (rc0) return rc0;
			fstate_ptr = d->fstate.p;
			hs.engine_state = &fstate_ptr;
		}
	}
	const int64_t pos_base = d->window_seen;
	const int32_t bit_base = d->tail.count;
	const uint8_t *mask = d->hist_mask.data();
	hs.kind = continuing ? B200Z_HIST_CONTINUE : (H ? B200Z_HIST_DICTIONARY : B200Z_HIST_NONE);
	hs.check_seeded = 1;
	hs.hist_len = &H;
	hs.pos_base = &pos_base;
	hs.bit_base = &bit_base;
	hs.hist_mask = &mask;
	const uint32_t stored_before = d->sstate.input_off;
	b200z_plan *plan = nullptr;
	int rc = b200z_deflate_plan_create_ex(1, &len, d->level, d->strategy, d->raw ? B200Z_WRAP_RAW : B200Z_WRAP_ZLIB, end_mode,
	                                      (hs.kind != B200Z_HIST_NONE || d->level <= 4) ? &hs : nullptr, &plan);
	if (rc) return rc;
	std::vector<uint8_t> slot;
	const uint8_t *inp = d->input.data();
	if (H) {
		slot.reserve((size_t)(H + len));
		slot.insert(slot.end(), d->history.begin(), d->history.end());
		slot.insert(slot.end(), d->input.begin(), d->input.end());
		inp = slot.data();
	}
	HostRunResult r;
	const uint32_t seed = d->adler;
	rc = run_plan_host(plan, &inp, d->hin, d->hout, d->din, d->dout, d->dmeta, r, false,
	                   (plan->check_seeded && !d->raw) ? &seed : nullptr);
	if (!rc && (r.status[0] & 0xFF) != B200Z_OK) {
		rc = r.status[0] & 0xFF;
		set_error("device deflate failed with status %d", rc);
	}
	if (!rc) {
		const uint8_t *o = d->hout.p + plan->out_off[0];
		const int64_t bits = r.in_used[0]; // deflate plans report the exact bit length here (bit_base included)
		const int64_t whole = bits >> 3;
		std::vector<uint8_t> seg(o, o + ((bits + 7) >> 3));
		if (!seg.empty()) seg[0] |= (uint8_t)d->tail.bits; // the carried sub-byte tail completes the first byte
		d->pending.insert(d->pending.end(), seg.begin(), seg.begin() + (ptrdiff_t)whole);
		// PendingBuffer keeps the sub-byte tail in `bits` until later writes complete the byte (:168-189)
		d->tail.count = (int)(bits & 7);
		d->tail.bits = d->tail.count ? (seg[(size_t)whole] & ((1u << d->tail.count) - 1u)) : 0u;
		if (end_mode == B200Z_END_FINISH) d->tail.align(d->pending); // FINISHING_STATE: AlignToByte (:507)
		if (!d->raw) d->adler = r.check[0];
		// (level 0: Finish() behind an undrained SetInput can end the stream before all input is taken, see stored_run)
		d->total_in += d->level == 0 ? (int64_t)(uint32_t)(d->sstate.input_off - stored_before) : len;
		d->started = true;
		deflater_remember(d, d->input.data(), (size_t)len, 2);
		d->input.clear();
		d->chunks.clear();
		d->undrained = false;
	}
	b200z_plan_destroy(plan);
	return rc;
}

int b200z_deflater_create(int level, int raw, void **h) {
	if (!h) {
		set_error("h");
		return B200Z_E_ARG;
	}
	if (level == -1) level = 6;
	else if (level < 0 || level > 9) {
		set_error("level"); // ArgumentOutOfRangeException(nameof(level)), Deflater.cs:184-187
		return B200Z_E_ARG;
	}
	DeflaterH *d = new DeflaterH();
	d->level = level;
	d->raw = raw != 0;
	*h = d;
	return B200Z_OK;
}
int b200z_deflater_destroy(void *h) {
	delete (DeflaterH *)h;
	return B200Z_OK;
}
int b200z_deflater_reset(void *h) { // Deflater.Reset :204-210 keeps level and strategy
	DeflaterH *d = (DeflaterH *)h;
	d->flushing = d->finishing = d->finished = false;
	d->header_done = false;
	d->flushed_once = false;
	d->input.clear();
	d->pending.clear();
	d->pending_pos = 0;
	d->tail = HostBits();
	d->total_in = d->total_out = 0;
	d->adler = 1;
	d->history.clear();
	d->hist_mask.clear();
	d->window_seen = 0;
	d->dict_set = d->deflate_called = d->started = false;
	d->dict_adler = 0;
	d->chunks.clear();
	d->undrained = false;
	d->sstate = b200z_stored_state{0, 0, 0, 0};
	return B200Z_OK;
}
int b200z_deflater_set_level(void *h, int level) {
	DeflaterH *d = (DeflaterH *)h;
	if (level == -1) level = 6;
	else if (level < 0 || level > 9) {
		set_error("level");
		return B200Z_E_ARG;
	}
	if (level != d->level && (!d->input.empty() || d->total_in > 0)) {
		set_error("SetLevel in mid-stream (DeflaterEngine.SetLevel flushes a block, trap T17) is not accelerated");
		return B200Z_E_UNSUPPORTED;
	}
	d->level = level;
	return B200Z_OK;
}
int b200z_deflater_get_level(void *h, int *level) {
	*level = ((DeflaterH *)h)->level;
	return B200Z_OK;
}
int b200z_deflater_set_strategy(void *h, int strategy) {
	if (strategy < 0 || strategy > 2) {
		set_error("strategy");
		return B200Z_E_ARG;
	}
	DeflaterH *d = (DeflaterH *)h;
	if (strategy != d->strategy && !d->input.empty()) {
		// the reference switches at the engine's current strstart (DeflaterEngine.cs:283-298), somewhere inside the input it
		// holds -- like SetLevel in mid-stream; behind a completed Flush() the switch is exact and allowed
		set_error("SetStrategy between SetInput and Flush()/Finish() is not accelerated");
		return B200Z_E_UNSUPPORTED;
	}
	d->strategy = strategy;
	return B200Z_OK;
}
int b200z_deflater_set_dictionary(void *h, const uint8_t *dict, int32_t len) {
	DeflaterH *d = (DeflaterH *)h;
	// Deflater.SetDictionary :372-381: only in INIT_STATE (before the header went out); the header's FDICT bit and
	// DICTID come from the engine's Adler-32 over the dictionary, which is then reset (:386-401)
	if (d->raw || d->deflate_called || d->header_done || d->total_in > 0 || d->dict_set) {
		// state != INIT_STATE (:561): a raw deflater starts in BUSY_STATE (:206), Deflate() leaves INIT_STATE (:436-464)
		set_error("SetDictionary: not in the initial state"); // InvalidOperationException
		return B200Z_E_STATE;
	}
	if (len < 0 || (len > 0 && !dict)) {
		set_error("dictionary/count");
		return B200Z_E_ARG;
	}
	uint32_t a = 1;
	if (len > 0) {
		int rc = b200z_adler32(dict, len, &a);
		if (rc) return rc;
	}
	d->dict_adler = a;
	d->dict_set = true;
	if (len < kMinMatch) return B200Z_OK; // DeflaterEngine.cs:207-210: too short to matter, not even copied
	const int32_t keep = len > kMaxDist ? kMaxDist : len; // :212-216
	deflater_remember(d, dict + (len - keep), (size_t)keep, 2);
	return B200Z_OK;
}
int b200z_deflater_set_input(void *h, const uint8_t *buf, int32_t len) {
	DeflaterH *d = (DeflaterH *)h;
	if (d->finishing) {
		set_error("Finish() already called"); // Deflater.cs:335
		return B200Z_E_STATE;
	}
	if (len < 0 || (len > 0 && !buf)) {
		set_error("buffer/count");
		return B200Z_E_ARG;
	}
	// one plan slot addresses 4 GiB - 64 KiB (32-bit positions, the window phase included): refuse what could not be
	// compressed instead of accepting it and failing at Flush() / Finish()
	if ((int64_t)d->input.size() + len + 32768 > 0xFFFF0000ll || d->window_seen + (int64_t)d->input.size() + len > 0xFFFF0000ll) {
		set_error("Deflater handle: more than 4 GiB - 64 KiB in one stream (TotalIn %lld, %lld buffered, %d more): use several "
		          "streams or the batch API",
		          (long long)d->total_in, (long long)d->input.size(), len);
		return B200Z_E_UNSUPPORTED;
	}
	if (len > 0) d->flushed_once = false;
	d->input.insert(d->input.end(), buf, buf + len);
	if (len > 0) {
		// engine.NeedsInput (DeflaterEngine.cs:187-190) is false until Deflate() has taken the bytes; a zero-length SetInput
		// leaves it true, so the stream classes do not even call Deflate() for it
		d->undrained = true;
		if (d->level <= 4) d->chunks.push_back(len); // the schedule matters for DeflateStored / DeflateFast only (trap T9)
	}
	return B200Z_OK;
}
int b200z_deflater_flush(void *h) {
	((DeflaterH *)h)->flushing = true;
	return B200Z_OK;
}
int b200z_deflater_finish(void *h) {
	DeflaterH *d = (DeflaterH *)h;
	d->flushing = d->finishing = true;
	return B200Z_OK;
}

int b200z_deflater_deflate(void *h, uint8_t *out, int32_t cap, int32_t *produced) {
	DeflaterH *d = (DeflaterH *)h;
	if (!produced || cap < 0 || (cap > 0 && !out)) {
		set_error("bad arguments");
		return B200Z_E_ARG;
	}
	*produced = 0;
	d->deflate_called = true;
	if (!d->flushing && !d->finishing) d->undrained = false; // BUSY_STATE: the engine takes everything SetInput handed over
	// make output due (Deflater.Deflate :427-522)
	if (!d->finished && d->pending_pos == d->pending.size() && (d->flushing || d->finishing)) {
		d->pending.clear();
		d->pending_pos = 0;
		if (!d->header_done && !d->raw) {
			uint8_t hd[2];
			zlib_header(d->level, hd, d->dict_set);
			d->pending.push_back(hd[0]);
			d->pending.push_back(hd[1]);
			if (d->dict_set) { // DICTID = Adler-32 of the whole dictionary, MSB first (:455-461)
				for (int sh = 24; sh >= 0; sh -= 8) d->pending.push_back((uint8_t)(d->dict_adler >> sh));
			}
		}
		d->header_done = true;
		if (d->finishing) {
			if (d->flushed_once) {
				// Flush() already emitted every block + the sync padding; Finish adds the final empty block:
				// levels 1-9 FlushBlock on an empty buffer = static header 011 + EOB 0000000 = value 3 in 10 bits
				// (DeflaterEngine.cs:750-768); level 0 an empty stored block 01 00 00 FF FF (:614-649)
				if (d->level == 0) {
					const uint8_t e5[5] = {1, 0, 0, 0xFF, 0xFF};
					d->pending.insert(d->pending.end(), e5, e5 + 5);
				} else {
					d->tail.put(d->pending, 3, 10);
					d->tail.align(d->pending);
				}
			} else {
				int rc = deflater_run_device(d, B200Z_END_FINISH);
				if (rc) return rc;
			}
			if (!d->raw) {
				d->pending.push_back((uint8_t)(d->adler >> 24));
				d->pending.push_back((uint8_t)(d->adler >> 16));
				d->pending.push_back((uint8_t)(d->adler >> 8));
				d->pending.push_back((uint8_t)d->adler);
			}
			d->finished = true;
		} else {
			// sync flush (level 0 skips the padding, :488)
			int rc = deflater_run_device(d, B200Z_END_FLUSH);
			if (rc) return rc;
			d->flushed_once = true;
			d->flushing = false;
		}
	}
	size_t avail = d->pending.size() - d->pending_pos;
	size_t take = avail < (size_t)cap ? avail : (size_t)cap;
	if (take) memcpy(out, d->pending.data() + d->pending_pos, take);
	d->pending_pos += take;
	d->total_out += (int64_t)take;
	*produced = (int32_t)take;
	return B200Z_OK;
}
int b200z_deflater_needs_input(void *h, int *flag) {
	// DeflaterEngine.NeedsInput (:187-190): false between SetInput and the Deflate() call that takes the bytes.  The
	// handle copies on SetInput, but it reports what the reference reports: DeflaterOutputStream.Write calls Deflate()
	// exactly while this is false (Streams/DeflaterOutputStream.cs:245-275), and whether that call happened before
	// Flush() / Finish() changes the bytes at levels 0-4 (b200z_history.undrained_last)
	*flag = ((DeflaterH *)h)->undrained ? 0 : 1;
	return B200Z_OK;
}
int b200z_deflater_is_finished(void *h, int *flag) {
	DeflaterH *d = (DeflaterH *)h;
	*flag = (d->finished && d->pending_pos == d->pending.size()) ? 1 : 0; // Deflater.cs:271-277
	return B200Z_OK;
}
int b200z_deflater_total_in(void *h, int64_t *v) {
	DeflaterH *d = (DeflaterH *)h;
	*v = d->total_in;
	return B200Z_OK;
}
int b200z_deflater_total_out(void *h, int64_t *v) {
	*v = ((DeflaterH *)h)->total_out;
	return B200Z_OK;
}
int b200z_deflater_adler(void *h, uint32_t *v) {
	DeflaterH *d = (DeflaterH *)h;
	*v = d->raw ? 0u : d->adler;
	return B200Z_OK;
}

// ---- Inflater handle ----------------------------------------------------------------------------------
// The reference's Inflater is a mode machine that stops at any bit and resumes (Inflater.cs:73-86, :429-552).  The kernel
// decodes whole plans, so the handle resumes at BLOCK granularity: k_inflate reports the last block header it reached
// (bit position, output position -- the "restart point"); when more input arrives decoding continues from that header
// with the last 32 KiB of output in front of it as the window image.  Bytes of a block that was only partly available
// are decoded again by the next run (they were already delivered; the new run's output replaces them byte for byte).
// Work is linear in the stream for any SetInput granularity as long as blocks are bounded (the reference's own Deflater
// cuts a block every 16384 symbols), and the handle holds one block of input / output plus the window, not the stream.
struct InflaterH {
	bool raw = false;
	std::vector<uint8_t> input; // compressed bytes from absolute offset in_base on (what lies in front of the restart point is dropped)
	int64_t in_base = 0, in_total = 0; // in_total = bytes handed over since Reset = in_base + input.size()
	bool new_input = false;
	bool finished = false;
	bool need_dict = false;
	bool header_done = false;
	uint32_t read_adler = 0;   // DICTID from the header (Inflater.readAdler)
	int64_t raw_off = 0;       // where the raw deflate data starts (behind the zlib header)
	int64_t rs_bit = 0;        // restart point: bit offset from raw_off of the block header decoding continues at
	int64_t rs_out = 0;        //                output position of that header
	std::vector<uint8_t> window; // last <= 32768 bytes of (dictionary ++ output[0, rs_out)): OutputWindow's contents there
	uint32_t run_adler = 1;    // Adler-32 of output[0, rs_out)
	std::vector<uint8_t> output; // decoded bytes from output position out_base on (delivered bytes in front of rs_out are dropped)
	int64_t out_base = 0;
	int64_t delivered = 0;
	int64_t consumed = 0; // bytes of input the decoder has used (header + raw + trailer), absolute
	uint32_t adler = 1;
	int error = 0;
	std::string error_msg;
	PinnedBuf hin, hout;
	DevBuf din, dout, dmeta;
	// one plan per handle, created for capacities and run below them (b200z_inflate_plan_set_lengths): a SetInput + Inflate
	// pair costs the copies and the kernels, no allocation
	b200z_plan *plan = nullptr;
	int64_t plan_comp_cap = 0, plan_out_cap = 0;
	~InflaterH() { b200z_plan_destroy(plan); }
	int64_t out_total() const { return out_base + (int64_t)output.size(); }
};

static const char *inflate_detail_msg(int detail) {
	switch (detail) {
	case 1: return "Unknown block type";
	case 2: return "broken uncompressed block";
	case 3: return "Illegal rep length code";
	case 4: return "Illegal rep dist code";
	case 5: return "Encountered invalid codelength 0";
	case 6: return "ValueOutOfRangeException: dynamic header code count";
	case 7: return "Cannot repeat previous code length when no other code length has been read";
	case 8: return "Cannot repeat code lengths past total number of data code lengths";
	case 9: return "Inflater dynamic header end-of-block code missing";
	case 10: return "Code lengths oversubscribed";
	case 11: return "Adler chksum doesn't match";
	case 12: return "GZIP crc sum mismatch";
	case 13: return "Number of bytes mismatch in footer";
	case 14: return "Error GZIP header, first magic byte doesn't match";
	case 15: return "Error GZIP header,  second magic byte doesn't match";
	case 16: return "Error GZIP header, data not in deflate format";
	case 17: return "Reserved flag bits in GZIP header != 0";
	case 18: return "Header CRC value mismatch";
	case 19: return "Header checksum illegal";
	case 20: return "Compression Method unknown";
	case 22: return "Needs a preset dictionary";
	default: return "corrupt deflate data";
	}
}

// decodes from the restart point to the end of what is available; fills output / consumed / finished and moves the
// restart point forward
static int inflater_run_device(InflaterH *d) {
	const int64_t slice_abs = d->raw_off + (d->rs_bit >> 3); // absolute offset of the first compressed byte of this run
	const int32_t sbit = (int32_t)(d->rs_bit & 7);
	const int64_t avail = d->in_total - slice_abs;
	if (avail < 0 || slice_abs < d->in_base) {
		set_error("inflater restart point outside the kept input");
		return B200Z_E_INTERNAL;
	}
	int64_t cap = avail * 8 + 65536;
	for (int attempt = 0; attempt < 8; attempt++) {
		const int64_t D = (int64_t)d->window.size();
		int rc;
		if (!d->plan || avail > d->plan_comp_cap || cap > d->plan_out_cap) {
			b200z_plan_destroy(d->plan);
			d->plan = nullptr;
			int64_t cc = 65536;
			while (cc < avail) cc *= 2;
			const int64_t oc = std::max(cap, cc * 8 + 65536), dc = 32768;
			if ((rc = b200z_inflate_plan_create_ex(1, &cc, &oc, B200Z_WRAP_RAW, &dc, &d->plan))) return rc;
			d->plan_comp_cap = cc;
			d->plan_out_cap = oc;
		}
		b200z_plan *plan = d->plan;
		if ((rc = b200z_inflate_plan_set_lengths(plan, &avail, &D))) return rc;
		if ((rc = b200z_inflate_plan_set_start_bits(plan, &sbit))) return rc;
		const uint8_t *inp = d->input.data() + (slice_abs - d->in_base);
		std::vector<uint8_t> slot;
		if (D) { // window image (dictionary, earlier output) directly in front of the compressed bytes
			slot.reserve((size_t)(D + avail));
			slot.insert(slot.end(), d->window.begin(), d->window.end());
			slot.insert(slot.end(), inp, inp + avail);
			inp = slot.data();
		}
		HostRunResult r;
		rc = run_plan_host(plan, &inp, d->hin, d->hout, d->din, d->dout, d->dmeta, r, false);
		int64_t rbit = 0, rout = 0;
		if (!rc) rc = b200z_plan_get_restart_points(plan, &rbit, &rout, nullptr);
		if (rc) return rc;
		const int st = r.status[0] & 0xFF, detail = (r.status[0] >> 8) & 0xFF;
		if (st == B200Z_E_NOMEM) {
			cap = d->plan_out_cap * 8; // (the next attempt makes a larger plan)
			continue;
		}
		// this run's output is output[rs_out, rs_out + out_len): it replaces what an earlier run decoded behind the
		// restart point (the same bytes, and at least as many)
		const uint8_t *o = d->hout.p + plan->out_off[0];
		d->output.resize((size_t)(d->rs_out - d->out_base));
		d->output.insert(d->output.end(), o, o + r.out_len[0]);
		if (st == B200Z_OK) {
			d->finished = true;
			d->consumed = slice_abs + r.in_used[0];
		} else if (st == B200Z_E_NEED_INPUT) {
			d->consumed = d->in_total;
		} else {
			d->error = st;
			d->error_msg = inflate_detail_msg(detail);
			return B200Z_OK;
		}
		if (rout < 0 || rout > r.out_len[0] || rbit < sbit || rbit > 8 * avail) {
			set_error("inflater restart point out of range");
			return B200Z_E_INTERNAL;
		}
		if (rout > 0 || rbit != sbit) {
			// move the restart point: checksum and window advance over output[rs_out, rs_out + rout)
			const uint8_t *seg = d->output.data() + (d->rs_out - d->out_base);
			if (!d->raw && rout > 0 && (rc = b200z_adler32(seg, rout, &d->run_adler))) return rc;
			if (rout >= 32768) d->window.assign(seg + rout - 32768, seg + rout);
			else {
				d->window.insert(d->window.end(), seg, seg + rout);
				if (d->window.size() > 32768) d->window.erase(d->window.begin(), d->window.end() - 32768);
			}
			d->rs_out += rout;
			d->rs_bit = (d->rs_bit & ~7ll) + rbit;
		}
		if (st == B200Z_E_NEED_INPUT) {
			// compressed bytes in front of the restart point are never looked at again
			const int64_t keep_from = d->raw_off + (d->rs_bit >> 3);
			if (keep_from > d->in_base) {
				d->input.erase(d->input.begin(), d->input.begin() + (keep_from - d->in_base));
				d->in_base = keep_from;
			}
		}
		return B200Z_OK;
	}
	set_error("output larger than any capacity tried");
	return B200Z_E_NOMEM;
}

// output in front of both the restart point and the delivery position is not needed any more
static void inflater_trim_output(InflaterH *d) {
	const int64_t keep_from = d->delivered < d->rs_out ? d->delivered : d->rs_out;
	if (keep_from - d->out_base >= 65536) {
		d->output.erase(d->output.begin(), d->output.begin() + (keep_from - d->out_base));
		d->out_base = keep_from;
	}
}

int b200z_inflater_create(int raw, void **h) {
	if (!h) {
		set_error("h");
		return B200Z_E_ARG;
	}
	InflaterH *d = new InflaterH();
	d->raw = raw != 0;
	*h = d;
	return B200Z_OK;
}
int b200z_inflater_destroy(void *h) {
	delete (InflaterH *)h;
	return B200Z_OK;
}
int b200z_inflater_reset(void *h) {
	InflaterH *d = (InflaterH *)h;
	d->input.clear();
	d->output.clear();
	d->window.clear();
	d->new_input = d->finished = d->need_dict = d->header_done = false;
	d->in_base = d->in_total = 0;
	d->raw_off = 0;
	d->rs_bit = d->rs_out = 0;
	d->run_adler = 1;
	d->out_base = 0;
	d->delivered = 0;
	d->consumed = 0;
	d->adler = 1;
	d->error = 0;
	d->read_adler = 0;
	return B200Z_OK;
}
int b200z_inflater_set_dictionary(void *h, const uint8_t *dict, int32_t len) {
	InflaterH *d = (InflaterH *)h;
	// Inflater.SetDictionary :589-620
	if (len < 0 || (len > 0 && !dict)) {
		set_error("buffer/count");
		return B200Z_E_ARG;
	}
	if (!d->need_dict) {
		set_error("Dictionary is not needed"); // InvalidOperationException
		return B200Z_E_STATE;
	}
	uint32_t a = 1;
	if (len > 0) {
		int rc = b200z_adler32(dict, len, &a);
		if (rc) return rc;
	}
	if (a != d->read_adler) {
		set_error("Wrong adler checksum"); // SharpZipBaseException
		return B200Z_E_DATA;
	}
	const int32_t keep = len > 32768 ? 32768 : len; // OutputWindow.CopyDict :160-166
	d->window.assign(dict + (len - keep), dict + len);
	d->need_dict = false;
	d->adler = 1;
	d->new_input = true; // what was handed over behind the header can be decoded now
	return B200Z_OK;
}
int b200z_inflater_set_input(void *h, const uint8_t *buf, int32_t len) {
	InflaterH *d = (InflaterH *)h;
	if (len < 0 || (len > 0 && !buf)) {
		set_error("buffer/count");
		return B200Z_E_ARG;
	}
	if (d->in_total > d->consumed && !d->finished) {
		set_error("Old input was not completely processed"); // StreamManipulator.cs:263
		return B200Z_E_STATE;
	}
	if (d->finished) {
		// after the end of the stream the reference keeps unread bytes as RemainingInput; replace them
		d->input.resize((size_t)(d->consumed - d->in_base));
		d->in_total = d->consumed;
	}
	d->input.insert(d->input.end(), buf, buf + len);
	d->in_total += len;
	d->new_input = true;
	return B200Z_OK;
}

int b200z_inflater_inflate(void *h, uint8_t *out, int32_t cap, int32_t *produced) {
	InflaterH *d = (InflaterH *)h;
	if (!produced || cap < 0 || (cap > 0 && !out)) {
		set_error("bad arguments");
		return B200Z_E_ARG;
	}
	*produced = 0;
	if (d->error) {
		set_error("%s", d->error_msg.c_str());
		return d->error;
	}
	if (!d->finished && d->new_input) {
		d->new_input = false;
		if (!d->raw && !d->header_done) {
			// (nothing is dropped from `input` before the header is done: in_base == 0 here)
			if (d->input.size() < 2) {
				d->consumed = (int64_t)d->input.size();
				return B200Z_OK; // DecodeHeader needs 16 bits (Inflater.cs:209-215)
			}
			const int header = (d->input[0] << 8) | d->input[1];
			if (header % 31 != 0) {
				d->error = B200Z_E_DATA;
				d->error_msg = "Header checksum illegal";
			} else if ((header & 0x0f00) != (8 << 8)) {
				d->error = B200Z_E_DATA;
				d->error_msg = "Compression Method unknown";
			}
			if (d->error) {
				set_error("%s", d->error_msg.c_str());
				return d->error;
			}
			if (header & 0x0020) {
				// PRESET_DICT: DecodeDict reads the 4-byte DICTID MSB first (:185-203); Inflate() then returns 0 until
				// SetDictionary supplies a dictionary with that Adler-32
				if (d->input.size() < 6) {
					d->consumed = (int64_t)d->input.size();
					return B200Z_OK;
				}
				d->read_adler = ((uint32_t)d->input[2] << 24) | ((uint32_t)d->input[3] << 16) | ((uint32_t)d->input[4] << 8) | d->input[5];
				d->need_dict = true;
				d->adler = d->read_adler; // Inflater.Adler reports readAdler while the dictionary is awaited (:823-836)
				d->header_done = true;
				d->raw_off = 6;
				d->consumed = 6;
				d->new_input = true; // the bytes behind the DICTID wait for SetDictionary
				return B200Z_OK;
			}
			d->header_done = true;
			d->raw_off = 2;
		}
		if (d->need_dict) {
			d->new_input = true;
			return B200Z_OK;
		}
		int rc = inflater_run_device(d);
		if (rc) return rc;
		if (d->finished && !d->raw) {
			// Adler32 trailer, read MSB first (DecodeChksum :397-418); until it is complete the reference withholds
			// nothing that was already decoded but is not "finished"
			if (d->in_total - d->consumed < 4) {
				d->finished = false;
				d->consumed = d->in_total;
				// keep output; the last block is decoded again when the trailer arrives
			} else {
				const uint8_t *t = d->input.data() + (d->consumed - d->in_base);
				const uint32_t want = ((uint32_t)t[0] << 24) | ((uint32_t)t[1] << 16) | ((uint32_t)t[2] << 8) | t[3];
				uint32_t got = d->run_adler; // output[0, rs_out) is in it already
				const int64_t rest = d->out_total() - d->rs_out;
				int rc2 = rest > 0 ? b200z_adler32(d->output.data() + (d->rs_out - d->out_base), rest, &got) : B200Z_OK;
				if (rc2) return rc2;
				d->adler = got;
				if (got != want) {
					d->error = B200Z_E_DATA;
					d->error_msg = "Adler chksum doesn't match";
				}
				d->consumed += 4;
			}
		}
	}
	size_t avail = (size_t)(d->out_total() - d->delivered);
	size_t take = avail < (size_t)cap ? avail : (size_t)cap;
	if (take) memcpy(out, d->output.data() + (d->delivered - d->out_base), take);
	d->delivered += (int64_t)take;
	*produced = (int32_t)take;
	inflater_trim_output(d);
	if (take == 0 && d->error) {
		set_error("%s", d->error_msg.c_str());
		return d->error;
	}
	return B200Z_OK;
}
int b200z_inflater_needs_input(void *h, int *flag) {
	InflaterH *d = (InflaterH *)h;
	*flag = (d->in_total <= d->consumed) ? 1 : 0; // StreamManipulator.IsNeedingInput
	return B200Z_OK;
}
int b200z_inflater_needs_dictionary(void *h, int *flag) {
	*flag = ((InflaterH *)h)->need_dict ? 1 : 0; // mode == DECODE_DICT && neededBits == 0 (Inflater.cs:792-798)
	return B200Z_OK;
}
int b200z_inflater_is_finished(void *h, int *flag) {
	InflaterH *d = (InflaterH *)h;
	// Inflater.cs:806-812; a trailer that did not verify is an exception from Inflate() in the reference (DecodeChksum
	// :397-418), so the stream is not "finished" as long as that error has not been delivered
	*flag = (d->finished && !d->error && d->delivered == d->out_total()) ? 1 : 0;
	return B200Z_OK;
}
int b200z_inflater_remaining_input(void *h, int32_t *v) {
	InflaterH *d = (InflaterH *)h;
	*v = (int32_t)(d->in_total - d->consumed);
	return B200Z_OK;
}
int b200z_inflater_total_in(void *h, int64_t *v) {
	*v = ((InflaterH *)h)->consumed; // totalIn - RemainingInput (Inflater.cs:862-868)
	return B200Z_OK;
}
int b200z_inflater_total_out(void *h, int64_t *v) {
	*v = ((InflaterH *)h)->delivered;
	return B200Z_OK;
}
int b200z_inflater_adler(void *h, uint32_t *v) {
	InflaterH *d = (InflaterH *)h;
	*v = d->raw ? 0u : d->adler;
	return B200Z_OK;
}

} // extern "C"
