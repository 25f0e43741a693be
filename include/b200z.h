/* b200z.h -- C-ABI of libb200z.so, the B200 (sm_100a) DEFLATE engine that replaces the managed inner loops of
 * ICSharpCode.SharpZipLib.Zip.Compression.{Deflater,Inflater} and ICSharpCode.SharpZipLib.Checksum.{Crc32,Adler32}.
 *
 * Plain pointers and sizes only: this is what a P/Invoke (C#), ctypes (Python) or cgo binding declares.
 * Paths cited below are relative to /root/reference/src/ICSharpCode.SharpZipLib/ .
 *
 * Every function returns a b200z_status (0 = OK) unless noted; b200z_last_error() gives the message of the last
 * failure on the calling thread.  The status -> .NET exception mapping the C# shim applies is in INTEGRATION.md.
 * There is NO CPU fallback: without a CUDA device every compute entry point fails with B200Z_E_CUDA.
 */
#ifndef B200Z_H
#define B200Z_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

typedef enum b200z_status {
	B200Z_OK = 0,
	B200Z_E_ARG = 1,         /* ArgumentNullException / ArgumentOutOfRangeException / ArgumentException */
	B200Z_E_STATE = 2,       /* InvalidOperationException ("Finish() already called", "Old input was not completely processed") */
	B200Z_E_DATA = 3,        /* SharpZipBaseException family (corrupt deflate data, checksum mismatch) */
	B200Z_E_INTERNAL = 4,    /* the reference would fail with a non-SharpZip exception (e.g. PendingBuffer overflow, trap T12) */
	B200Z_E_CUDA = 5,        /* CUDA runtime failure / no device */
	B200Z_E_UNSUPPORTED = 6, /* a call sequence this build does not accelerate; never silently emulated on the CPU */
	B200Z_E_NOMEM = 7,       /* device or host allocation failed, or an output capacity was too small */
	B200Z_E_NEED_INPUT = 8   /* inflate: the compressed stream ended before the final block (stream layer: "Unexpected EOF") */
} b200z_status;

/* wrapper around the raw deflate stream */
enum { B200Z_WRAP_RAW = 0, B200Z_WRAP_ZLIB = 1, B200Z_WRAP_GZIP = 2, B200Z_WRAP_RAW_CRC32 = 3 /* raw stream plus the CRC-32 of the uncompressed bytes in `check`: zip entries */ };
/* DeflateStrategy, Zip/Compression/DeflaterEngine.cs:9-28 */
enum { B200Z_STRATEGY_DEFAULT = 0, B200Z_STRATEGY_FILTERED = 1, B200Z_STRATEGY_HUFFMAN_ONLY = 2 };
/* how a deflate plan ends each stream (which Deflater calls the bytes correspond to) */
enum {
	B200Z_END_FINISH = 0,       /* SetInput* -> Finish()                       (Deflater.cs:262; DeflaterOutputStream.Finish :100) */
	B200Z_END_FLUSH_FINISH = 1, /* SetInput* -> Flush() -> Finish()            (test pattern InflaterDeflaterTests.cs:49-62)      */
	B200Z_END_FLUSH = 2         /* SetInput* -> Flush(), stream continues      (Deflater.cs:252, sync padding :486-504)           */
};

const char *b200z_last_error(void);
int b200z_version(void);
/* Selects the CUDA device the calling thread creates plans, pipelines and handles on (one process per GPU: call it once;
 * one process for several GPUs: see "one host process, several GPUs" below) and loads the device's constant tables.
 * Idempotent.  Mirrors nothing in the reference: the reference has no device. */
int b200z_init(int device);
/* Static Huffman tables (DeflaterHuffman static ctor :602-642 and InflaterHuffmanTree static ctor :34-70) as one
 * byte blob, so that rank 0 can broadcast them (NCCL) and the others install them: north_star's only collective. */
int b200z_static_tables_size(void);
int b200z_static_tables_export(uint8_t *blob, int32_t cap);
int b200z_static_tables_import(const uint8_t *blob, int32_t len);
/* The same collective inside the library, for a host process that owns an NCCL communicator (one process per GPU; SURVEY.md
 * 8b): rank `root` exports, ncclBroadcast over `nccl_comm` (an ncclComm_t) on `cuda_stream`, every rank installs / verifies.
 * NCCL is resolved from the process at run time (libnccl.so.2); B200Z_E_UNSUPPORTED when there is none. */
int b200z_static_tables_broadcast(void *nccl_comm, int32_t root, int32_t rank, void *cuda_stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Checksums -- IChecksum (Checksum/IChecksum.cs), Crc32 (Checksum/Crc32.cs:47-171), Adler32 (Checksum/Adler32.cs:56-161).
 * `value` in/out is the checksum's Value over everything fed so far (Crc32.Reset -> 0, Adler32.Reset -> 1).
 * Host-buffer forms copy to the device and reduce there; _device forms take device pointers.
 * ------------------------------------------------------------------------------------------------------------- */
int b200z_crc32(const uint8_t *buf, int64_t len, uint32_t *value);
int b200z_adler32(const uint8_t *buf, int64_t len, uint32_t *value);
/* n independent buffers resident on the device: buffer i is d_data[off[i] .. off[i]+len[i]); seeds/results in
 * d_value[i] (device).  kind: 0 = CRC32, 1 = Adler32.  off/len are host arrays.  Asynchronous on `stream`. */
int b200z_checksum_batch_device(int kind, const uint8_t *d_data, const int64_t *off, const int64_t *len, int32_t n,
                                uint32_t *d_value, void *cuda_stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Batch plans -- what the benchmark drives.  A plan fixes the shape of a batch (number of streams, their sizes,
 * level/strategy), owns the device workspace, and lays the streams out in one input blob and one output blob at
 * aligned offsets it reports.  run() only launches kernels on `stream` (no host synchronisation), so it can be
 * timed with CUDA events or captured in a CUDA graph.  Stream i of the batch is one self-contained DEFLATE stream:
 * a fresh `new Deflater(level, true)` / `new Inflater(true)` per buffer in the reference.
 * ------------------------------------------------------------------------------------------------------------- */
typedef struct b200z_plan b200z_plan;

/* ---- streams with history ---------------------------------------------------------------------------------
 * A deflate stream whose window is not empty when the data starts:
 *   B200Z_HIST_DICTIONARY  Deflater.SetDictionary (Deflater.cs:372-381 -> DeflaterEngine.SetDictionary :198-229): the
 *                          history is the dictionary cut to its last MAX_DIST (32506) bytes; dictionaries shorter than
 *                          MIN_MATCH are ignored by the reference, pass hist_len 0 for them.  All levels.
 *   B200Z_HIST_CONTINUE    more input after Deflater.Flush() (Deflater.cs:488-506 leaves the engine re-entrant): the
 *                          history is the last min(32768, bytes so far) bytes of everything the window has seen
 *                          (dictionary included).  Levels 5-9 (DeflateSlow) need nothing else; DeflateFast (1-4) and
 *                          DeflateStored (0) keep window-relative state across Deflate() calls that is not a function of
 *                          the stream position (DeflaterEngine.cs:80-94: head/prev, strstart, blockStart), so every
 *                          segment of such a stream must be run with engine_state / stored_state (below), which the
 *                          run of one segment fills and the run of the next one reads; B200Z_E_UNSUPPORTED without.
 * Levels 0-4 also depend on HOW the data arrives (SURVEY.md trap T9: FillWindow slides at strstart >= 65274 whenever it is
 * called, DeflateFast at > 65274; DeflateStored cuts blocks by what it has seen so far): chunk_count / chunk_len give the
 * SetInput calls that delivered a stream's data, each followed by Deflate() until IsNeedingInput as DeflaterOutputStream
 * .Write does (Streams/DeflaterOutputStream.cs:506-510); without them one SetInput with everything is assumed.  Levels 5-9
 * ignore the schedule (their output does not depend on it).
 * Input slot i of such a plan holds hist_len[i] history bytes directly followed by the in_len[i] data bytes;
 * b200z_plan_in_offset(i) is the start of the history.  The checksum covers the data only; with check_seeded the
 * d_check array handed to b200z_plan_run carries the running values in and the updated values out (Adler32.Update /
 * Crc32.Update on an existing value).  The produced bits start at bit `bit_base` of output byte 0 (the bits below are
 * left zero: OR in the tail of the previous segment, PendingBuffer.cs:168-189 keeps it in its bit register). */
#define B200Z_HIST_NONE 0
#define B200Z_HIST_DICTIONARY 1
#define B200Z_HIST_CONTINUE 2
typedef struct b200z_history {
	int32_t kind;                   /* B200Z_HIST_* for every stream of the plan */
	int32_t check_seeded;           /* != 0: d_check is in/out (running checksum) instead of out */
	const int64_t *hist_len;        /* [n] history bytes in front of the data */
	const int64_t *pos_base;        /* [n] CONTINUE: bytes the window has seen before the data (dictionary + TotalIn);
	                                   decides the SlideWindow phase (DeflaterEngine.cs:441-462); NULL/DICTIONARY: hist_len */
	const int32_t *bit_base;        /* [n] 0..7 bits already taken in the first output byte; NULL = 0 */
	const uint8_t *const *hist_mask; /* [n] hist_len[i] flags, 1 = position was never entered into the hash chains
	                                   (InsertString needs MIN_MATCH bytes of lookahead, :782/:819: the last two positions
	                                   of every earlier segment); NULL entry = the last two history positions */
	/* ---- levels 0-4 (all optional; kind may be B200Z_HIST_NONE, hist_len then may be NULL) ---- */
	const int32_t *chunk_count;     /* [n] number of SetInput calls that delivered stream i's data; NULL or 0 = one */
	const int64_t *const *chunk_len; /* [n] chunk_count[i] sizes (>= 0) summing to in_len[i] */
	const int32_t *undrained_last;  /* [n] != 0: Flush() / Finish() came right behind the last SetInput, no Deflate() call in
	                                   between (a raw Deflater user; the stream classes always drain); NULL = 0 */
	void *const *engine_state;      /* [n] levels 1-4: DEVICE buffers of b200z_engine_state_bytes() bytes, one per stream:
	                                   head[], prev[] and DeflateFast's scalars, written at the end of every run, read at
	                                   the start of a B200Z_HIST_CONTINUE run */
	struct b200z_stored_state *stored_state; /* [n] level 0: HOST array, read by a B200Z_HIST_CONTINUE plan when it is
	                                   created and overwritten with the state behind this segment */
} b200z_history;
typedef struct b200z_stored_state { /* DeflateStored's fields between Deflate() calls (DeflaterEngine.cs:614-649) */
	int32_t strstart, block_start;
	uint32_t slides, input_off;
} b200z_stored_state;
int64_t b200z_engine_state_bytes(void);
int b200z_deflate_plan_create_ex(int32_t n, const int64_t *in_len, int level, int strategy, int wrap, int end_mode,
                                 const b200z_history *hist, b200z_plan **plan);

int b200z_deflate_plan_create(int32_t n, const int64_t *in_len, int level, int strategy, int wrap, int end_mode,
                              b200z_plan **plan);
int b200z_inflate_plan_create(int32_t n, const int64_t *comp_len, const int64_t *out_cap, int wrap, b200z_plan **plan);
/* Inflater.SetDictionary (Inflater.cs:589-620 -> OutputWindow.CopyDict, OutputWindow.cs:151-171): dict_len[i] <= 32768
 * bytes (the dictionary's tail) stored directly in front of stream i's compressed bytes; b200z_plan_in_offset(i) is
 * where the dictionary starts, b200z_plan_data_offset(i) where the compressed bytes start (16-byte aligned). */
int b200z_inflate_plan_create_ex(int32_t n, const int64_t *comp_len, const int64_t *out_cap, int wrap,
                                 const int64_t *dict_len, b200z_plan **plan);
/* Decoding a stream in pieces (what Inflater does between SetInput calls, Inflater.cs:73-86 / :429-552: its mode machine
 * stops anywhere and resumes).  Across a block boundary the decoder carries only the window (= the last 32 KiB of
 * output) and the bit position, so a raw inflate plan can start in the middle of a stream: at bit start_bit[i] (0..7) of
 * the first compressed byte handed over, a block header, with the window image passed as the "dictionary".  After a run,
 * restart points tell where the last block header the decoder reached lies: bit[i] (counted from the first compressed
 * byte of the slot) and out_pos[i] (bytes of output in front of it).  A stream that ended with B200Z_E_NEED_INPUT is
 * continued from there once more input has arrived.  Host arrays of n entries; get_restart_points synchronises the stream. */
int b200z_inflate_plan_set_start_bits(b200z_plan *plan, const int32_t *start_bit);
/* Runs an inflate plan below the sizes it was created for: stream i's next run has comp_len[i] compressed bytes behind a
 * dictionary / window image of dict_len[i] bytes (NULL = none), each at most what b200z_inflate_plan_create_ex was given.
 * The dictionary still ends where the compressed bytes start: b200z_plan_in_offset(i) moves accordingly,
 * b200z_plan_data_offset(i) stays.  This is how the Inflater handle keeps ONE plan between SetInput calls. */
int b200z_inflate_plan_set_lengths(b200z_plan *plan, const int64_t *comp_len, const int64_t *dict_len);
int b200z_plan_get_restart_points(b200z_plan *plan, int64_t *bit, int64_t *out_pos, void *cuda_stream);
/* Diagnostics of the last run of an inflate plan (synchronises `stream`): v[0] positions that passed the finder's first
 * two stages, v[1] segments decoded (stream starts + block-header candidates), v[2] round slots taken, v[3] Huffman blocks
 * decoded, v[4] rounds, v[5] speculative passes over them, v[6] streams handed back to the serial kernel, v[7] 1 if the
 * plan runs the block-parallel pipeline.  Mirrors nothing in the reference. */
int b200z_plan_get_stats(b200z_plan *plan, uint32_t *v, int32_t cap, void *cuda_stream);
/* What the last SEARCH stage of a level 5-9 deflate plan left for stream i (synchronises `stream`), for tests that check
 * the match search entry for entry: link[hist_len[i] + in_len[i]] (uint16, may be NULL) the hash-chain links of every
 * position of the slot, history first (0 = no predecessor), and ab[2 * in_len[i]] (uint32) the (A, B) table entries of the
 * data positions (A: best match with the full chain budget, B: with a quarter of it; len << 16 | dist, 0 = none). */
int b200z_plan_get_match_table(b200z_plan *plan, int32_t i, uint16_t *link, uint32_t *ab, void *cuda_stream);
int b200z_plan_destroy(b200z_plan *plan);
int64_t b200z_plan_in_bytes(const b200z_plan *plan);          /* size of the input blob  */
int64_t b200z_plan_out_bytes(const b200z_plan *plan);         /* size of the output blob */
int64_t b200z_plan_in_offset(const b200z_plan *plan, int32_t i);   /* start of slot i (history/dictionary first) */
int64_t b200z_plan_data_offset(const b200z_plan *plan, int32_t i); /* start of slot i's data behind the history */
int64_t b200z_plan_out_offset(const b200z_plan *plan, int32_t i);
int64_t b200z_plan_out_capacity(const b200z_plan *plan, int32_t i);
int64_t b200z_plan_workspace_bytes(const b200z_plan *plan);
/* kernels launched by one run() (for the benchmark's gpu_launches accounting) */
int32_t b200z_plan_launches(const b200z_plan *plan);
/* Per-kernel device times: when enabled, run() records CUDA events on its stream between kernels; after the stream
 * has been synchronised get_timings() returns the milliseconds of each interval of the last run and a ';'-separated
 * list of kernel names.  Measurement aid for bench.py's roofline line; off by default. */
int b200z_plan_set_timing(b200z_plan *plan, int enable);
int b200z_plan_get_timings(b200z_plan *plan, char *names, int32_t names_cap, float *ms, int32_t cap, int32_t *count);
/* d_in / d_out: device blobs laid out as the plan reports.  d_out_len[n] (int64), d_status[n] (int32, b200z_status)
 * and d_check[n] (uint32: Adler32 for zlib, CRC32 for gzip, untouched for raw; may be NULL for raw) are device
 * arrays.  For inflate plans d_in_used[n] (int64, may be NULL) receives the compressed bytes consumed, i.e.
 * comp_len - Inflater.RemainingInput (Inflater.cs:878, trap T14). */
int b200z_plan_run(b200z_plan *plan, const uint8_t *d_in, uint8_t *d_out, int64_t *d_out_len, int32_t *d_status,
                   uint32_t *d_check, int64_t *d_in_used, void *cuda_stream);
/* The same in two halves, for callers that overlap independent work on other streams: SEARCH is the match finding of a
 * level 5-9 deflate plan (its kernels take a whole SM's shared memory), ENCODE everything else (parse, Huffman planning,
 * bit packing, checksums; all of a level 0-4 or inflate plan).  Run SEARCH then ENCODE with the same arguments on the
 * same stream; b200z_plan_run is both.  Per-kernel timing is only recorded by whole runs. */
#define B200Z_STAGE_SEARCH 1
#define B200Z_STAGE_ENCODE 2
int b200z_plan_run_stages(b200z_plan *plan, const uint8_t *d_in, uint8_t *d_out, int64_t *d_out_len, int32_t *d_status,
                          uint32_t *d_check, int64_t *d_in_used, int stages, void *cuda_stream);

/* Packs the streams a run produced back to back (16-byte aligned starts) into d_packed, so a caller copies only the
 * produced bytes to the host: d_packed_off[n + 1] (device) receives the start of every stream and, last, the total.
 * d_packed needs b200z_plan_out_bytes() of room.  Asynchronous on `stream`. */
int b200z_plan_pack(b200z_plan *plan, const uint8_t *d_out, const int64_t *d_out_len, uint8_t *d_packed,
                    int64_t *d_packed_off, void *cuda_stream);

/* ---------------------------------------------------------------------------------------------------------------
 * Host-buffer pipelines -- the end-to-end path a host process drives (what DeflaterOutputStream / InflaterInputStream
 * callers with many independent buffers amount to: ZipOutputStream entries, Streams/DeflaterOutputStream.cs:245-275).
 * A pipeline owns the plan of one batch shape, `depth` (1..8) slots of pinned staging + device buffers and its own CUDA
 * streams.  submit() takes HOST pointers (in[i]: stream i's bytes, the sizes given at creation), stages them and enqueues
 * upload and kernels without waiting; collect() waits for the oldest submitted batch, moves exactly the produced bytes
 * across PCIe and into out[i] (HOST pointers), and reports per stream what the batch calls below report.  With
 * depth >= 2, submit(i+1) before collect(i) overlaps the upload of batch i+1 and the download of batch i-1 with the
 * kernels of batch i.  Host memory CUDA knows as pinned (cudaHostAlloc / cudaHostRegister) is the DMA source / target
 * directly; pageable memory goes through the slot's pinned staging.  wrap = B200Z_WRAP_GZIP on the deflate side writes
 * GZipOutputStream's bytes with MTIME = 0 and no FNAME (GZip/GzipOutputStream.cs:315-375: 1F 8B 08 00 00000000 00 FF,
 * raw stream, CRC32, ISIZE); a caller with its own MTIME / FNAME patches bytes 4..7 or uses B200Z_WRAP_RAW_CRC32.
 * One pipeline = one host thread at a time.  E_STATE: submit with `depth` batches in flight, collect with none.
 * ------------------------------------------------------------------------------------------------------------- */
typedef struct b200z_pipeline b200z_pipeline;
int b200z_deflate_pipeline_create(int32_t n, const int64_t *in_len, int level, int strategy, int wrap, int end_mode, int depth,
                                  b200z_pipeline **pipe);
int b200z_inflate_pipeline_create(int32_t n, const int64_t *comp_len, const int64_t *out_cap, int wrap, int depth,
                                  b200z_pipeline **pipe);
int b200z_pipeline_submit(b200z_pipeline *pipe, const uint8_t *const *in);
int b200z_pipeline_collect(b200z_pipeline *pipe, uint8_t *const *out, const int64_t *out_cap, int64_t *out_len, int64_t *in_used,
                           uint32_t *check, int32_t *status);
int32_t b200z_pipeline_in_flight(const b200z_pipeline *pipe); /* batches submitted and not yet collected */
int b200z_pipeline_destroy(b200z_pipeline *pipe);

/* Host-buffer batch calls: one submit + collect on a pipeline of depth 1 that the calling thread keeps for the batch's
 * shape (the last four shapes stay cached: plan, pinned staging and device buffers are not allocated again; 
 * b200z_release_cached() frees them).  in[i]/out[i] are HOST pointers; status[i] is per stream.  The return value is the
 * first non-OK status, if any. */
int b200z_deflate_batch(const uint8_t *const *in, const int64_t *in_len, int32_t n, int level, int strategy, int wrap,
                        int end_mode, uint8_t *const *out, const int64_t *out_cap, int64_t *out_len, uint32_t *check,
                        int32_t *status);
int b200z_inflate_batch(const uint8_t *const *in, const int64_t *in_len, int32_t n, int wrap, uint8_t *const *out,
                        const int64_t *out_cap, int64_t *out_len, int64_t *in_used, uint32_t *check, int32_t *status);
int b200z_release_cached(void);

/* ---- one host process, several GPUs ------------------------------------------------------------------------------
 * b200z_init(device) may be called for several devices: it makes `device` the one the CALLING THREAD creates plans,
 * pipelines and handles on.  Every such object stays on its device; its entry points run there whatever the thread's
 * current device is and leave that as they found it.  The _multi batch calls cut a batch into contiguous ranges of about
 * equal bytes (b200z_partition_by_bytes: part r starts at first[r], first[parts] = n), run range r on devices[r] -- all
 * devices at the same time, every submit before the first collect -- and fill the caller's arrays as the single-device
 * calls do.  The streams of a batch are independent, so there is no device-to-device traffic (SURVEY.md 8e). */
int b200z_device_count(void);
int b200z_partition_by_bytes(const int64_t *len, int32_t n, int32_t parts, int32_t *first);
int b200z_deflate_batch_multi(const int32_t *devices, int32_t n_devices, const uint8_t *const *in, const int64_t *in_len, int32_t n,
                              int level, int strategy, int wrap, int end_mode, uint8_t *const *out, const int64_t *out_cap,
                              int64_t *out_len, uint32_t *check, int32_t *status);
int b200z_inflate_batch_multi(const int32_t *devices, int32_t n_devices, const uint8_t *const *in, const int64_t *in_len, int32_t n,
                              int wrap, uint8_t *const *out, const int64_t *out_cap, int64_t *out_len, int64_t *in_used,
                              uint32_t *check, int32_t *status);
/* worst-case compressed size for `len` input bytes at any level (capacity a caller should provide) */
int64_t b200z_deflate_bound(int64_t len);

/* ---------------------------------------------------------------------------------------------------------------
 * Streaming handles -- 1:1 with the members of Deflater (Zip/Compression/Deflater.cs) and Inflater
 * (Zip/Compression/Inflater.cs) that DeflaterOutputStream / InflaterInputStream / GZip / Zip call
 * (Streams/DeflaterOutputStream.cs:100-139, 245-275, 388-393, 506-510; Streams/InflaterInputStream.cs:658-690).
 * A handle buffers input on the host and runs the device pipeline when Flush()/Finish() makes output due; the
 * concatenated output equals the reference's for the same sequence of calls (SURVEY.md 8b).  One handle = one
 * logical thread at a time; different handles may be used from different threads.
 * ------------------------------------------------------------------------------------------------------------- */
int b200z_deflater_create(int level, int raw /* noZlibHeaderOrFooter */, void **h); /* Deflater.cs:178 */
int b200z_deflater_destroy(void *h);
int b200z_deflater_reset(void *h);                                                  /* :204 */
int b200z_deflater_set_level(void *h, int level);                                   /* :349 */
int b200z_deflater_get_level(void *h, int *level);                                  /* :371 */
int b200z_deflater_set_strategy(void *h, int strategy);                             /* :385 */
int b200z_deflater_set_dictionary(void *h, const uint8_t *dict, int32_t len);       /* :559 */
int b200z_deflater_set_input(void *h, const uint8_t *buf, int32_t len);             /* :331 (copies) */
int b200z_deflater_flush(void *h);                                                  /* :252 */
int b200z_deflater_finish(void *h);                                                 /* :262 */
int b200z_deflater_deflate(void *h, uint8_t *out, int32_t cap, int32_t *produced);  /* :427 */
int b200z_deflater_needs_input(void *h, int *flag);                                 /* :285 */
int b200z_deflater_is_finished(void *h, int *flag);                                 /* :271 */
int b200z_deflater_total_in(void *h, int64_t *v);                                   /* :226 */
int b200z_deflater_total_out(void *h, int64_t *v);                                  /* :237 */
int b200z_deflater_adler(void *h, uint32_t *v);                                     /* :215 */

int b200z_inflater_create(int raw /* noHeader */, void **h);                        /* Inflater.cs:172 */
int b200z_inflater_destroy(void *h);
int b200z_inflater_reset(void *h);                                                  /* :188 */
int b200z_inflater_set_dictionary(void *h, const uint8_t *dict, int32_t len);       /* :589 */
int b200z_inflater_set_input(void *h, const uint8_t *buf, int32_t len);             /* :653 (copies) */
int b200z_inflater_inflate(void *h, uint8_t *out, int32_t cap, int32_t *produced);  /* :715 */
int b200z_inflater_needs_input(void *h, int *flag);                                 /* :783 */
int b200z_inflater_needs_dictionary(void *h, int *flag);                            /* :794 */
int b200z_inflater_is_finished(void *h, int *flag);                                 /* :806 */
int b200z_inflater_remaining_input(void *h, int32_t *v);                            /* :878 */
int b200z_inflater_total_in(void *h, int64_t *v);                                   /* :862 */
int b200z_inflater_total_out(void *h, int64_t *v);                                  /* :848 */
int b200z_inflater_adler(void *h, uint32_t *v);                                     /* :823 */

/* ---- Entry ciphers applied to compressed bytes (SURVEY.md row f4) ---------------------------------------------------
 * Encryption/ZipAESTransform.cs (WinZip AES: AES-CTR + HMAC-SHA1, keys by PBKDF2) and Encryption/PkzipClassic.cs, the
 * ICryptoTransform objects Streams/DeflaterOutputStream.cs:227-231 (EncryptBlock) and Zip/ZipFile.cs feed with the codec's
 * output.  AES-CTR is one thread per 16-byte block; SHA-1 and the classic cipher are serial per stream and run one thread
 * per stream (they scale with the number of entries).  `keys` of the AES calls: per stream 2 * key_bytes + 2 bytes, key1 |
 * key2 | password verifier, exactly the three GetBytes() results of ZipAESTransform.cs:62-68. */
typedef struct b200z_aes_transform b200z_aes_transform;
/* ZipAESTransform constructor :41-72 for n entries: pw_off[n + 1] offsets into the password blob, salts n x key_bytes / 2
 * bytes, key_bytes 16 or 32 (:43-46), keys_out n x (2 * key_bytes + 2).  Host pointers; PBKDF2 runs on the device. */
int b200z_aes_derive_keys(const uint8_t *passwords, const int64_t *pw_off, const uint8_t *salts, int32_t key_bytes, int32_t n,
                          uint8_t *keys_out);
/* bytes of per-stream state the device call carries between TransformBlock calls (zero-filled = a fresh transform) */
int64_t b200z_aes_state_bytes(void);
/* TransformBlock :75-112 on device memory for n streams at once: stream i is d_len[i] bytes at d_in + d_off[i] (d_out may be
 * d_in), max_len >= every length.  d_state: n x b200z_aes_state_bytes().  finish != 0 also writes GetAuthCode() (:122, 20
 * bytes per stream, the archive keeps the first 10) to d_auth.  No host synchronisation. */
int b200z_aes_device(const uint8_t *d_in, uint8_t *d_out, const int64_t *d_off, const int64_t *d_len, int64_t max_len, int32_t n,
                     int32_t key_bytes, const uint8_t *d_keys, int32_t write_mode, uint8_t *d_state, int32_t finish, uint8_t *d_auth,
                     void *cuda_stream);
/* the same for whole entries in host memory: out[i] = TransformBlock(in[i]), auth + 20 * i = GetAuthCode() */
int b200z_aes_batch(const uint8_t *const *in, const int64_t *len, int32_t n, int32_t key_bytes, const uint8_t *keys, int32_t write_mode,
                    uint8_t *const *out, uint8_t *auth);
/* one ZipAESTransform as a handle: constructor :41, TransformBlock :75, PwdVerifier :117, GetAuthCode :122, Dispose :172 */
int b200z_aes_transform_create(const uint8_t *password, int32_t password_len, const uint8_t *salt, int32_t key_bytes, int32_t write_mode,
                               b200z_aes_transform **out);
int b200z_aes_transform_block(b200z_aes_transform *t, const uint8_t *in, int64_t count, uint8_t *out);
int b200z_aes_transform_pwd_verifier(const b200z_aes_transform *t, uint8_t *out2);
int b200z_aes_transform_auth_code(b200z_aes_transform *t, uint8_t *out20);
int b200z_aes_transform_destroy(b200z_aes_transform *t);
/* PkzipClassic.GenerateKeys :19-50 (12 bytes: keys[0..2] little-endian, what SetKeys :84-100 takes) */
int b200z_pkzip_generate_keys(const uint8_t *seed, int64_t n, uint8_t *keys12);
/* PkzipClassicEncryptCryptoTransform.TransformBlock :170-178 / PkzipClassicDecryptCryptoTransform.TransformBlock :279-288 for
 * n streams: d_keys n x 3 words, updated in place (a stream goes on where its last call ended) */
int b200z_pkzip_device(const uint8_t *d_in, uint8_t *d_out, const int64_t *d_off, const int64_t *d_len, int32_t n, uint32_t *d_keys,
                       int32_t encrypt, void *cuda_stream);
int b200z_pkzip_batch(const uint8_t *const *in, const int64_t *len, int32_t n, uint8_t *keys12, int32_t encrypt, uint8_t *const *out);

#ifdef __cplusplus
}
#endif
#endif /* B200Z_H */
