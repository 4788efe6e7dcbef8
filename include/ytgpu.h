/* ytgpu.h — C ABI of the B200-native sort/shuffle + scan→filter→group-by hot path.
 *
 * This is the drop-in boundary a YTsaurus job proxy / CHYT instance binds to
 * (INTEGRATION.md shows the C++ adapters).  Plain pointers and sizes only; no
 * torch / CUDA types in signatures (a CUDA stream travels as void*).
 *
 * Every entry point cites the reference interface it replaces (paths relative
 * to the YTsaurus tree).  All calls are asynchronous with respect to the
 * context's stream unless they return data to HOST memory, in which case they
 * synchronise that stream before returning.  Calls never fall back to a CPU
 * implementation: if the device cannot run the request the call fails with
 * YTGPU_ERR_UNSUPPORTED / YTGPU_ERR_CUDA.
 */
#ifndef YTGPU_H_
#define YTGPU_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define YTGPU_ABI_VERSION 2

/* ---- status / errors (replaces TErrorException, THROW_ERROR_EXCEPTION) ---- */
typedef enum ytgpu_status {
    YTGPU_OK = 0,
    YTGPU_ERR_INVALID_ARGUMENT = 1,
    YTGPU_ERR_UNSUPPORTED = 2,      /* e.g. Any/Composite key columns (need the YSON comparer) */
    YTGPU_ERR_CUDA = 3,
    YTGPU_ERR_OUT_OF_MEMORY = 4,
    YTGPU_ERR_SCHEMA_VIOLATION = 5, /* value type differs from the declared key column type */
    YTGPU_ERR_PARTITION_BAD_TYPE = 10,     /* partitioner.cpp:143-149 */
    YTGPU_ERR_PARTITION_NEGATIVE = 11,     /* partitioner.cpp:151-156 */
    YTGPU_ERR_PARTITION_OUT_OF_BOUNDS = 12,/* partitioner.cpp:158-163 */
    YTGPU_ERR_PARTITION_NO_COLUMN = 13     /* partitioner.cpp:167 */
} ytgpu_status;

typedef struct ytgpu_error {
    int32_t code;       /* ytgpu_status */
    int32_t cuda_error; /* cudaError_t when code == YTGPU_ERR_CUDA */
    char message[248];
} ytgpu_error;

/* ---- memory spaces ---- */
typedef enum ytgpu_mem { YTGPU_MEM_DEVICE = 0, YTGPU_MEM_HOST = 1 } ytgpu_mem;

/* ---- per-device context (explicit; no thread-local CUDA state is assumed, YT fibers migrate) ----
 * Calls made on ONE context are serialised by the library (each entry point locks the context), so readers,
 * partitioners and writers living on different threads may share it; use one context per job slot / stream for
 * concurrency.  A process may own contexts on several devices. */
typedef struct ytgpu_context ytgpu_context;

/* cuda_stream: a cudaStream_t to run on (e.g. torch's current stream; pass cudaStreamLegacy == (void*)1
 * for the legacy default stream), or NULL for a private non-blocking stream. */
int ytgpu_context_create(int device, void* cuda_stream, ytgpu_context** out, ytgpu_error* err);
void ytgpu_context_destroy(ytgpu_context* ctx);
int ytgpu_context_synchronize(ytgpu_context* ctx, ytgpu_error* err);
/* Number of kernel launches issued through this context since creation (bench.py's gpu_launches). */
uint64_t ytgpu_context_launch_count(const ytgpu_context* ctx);
/* Device time (ms) of the dominant kernel class measured with CUDA events on the context stream,
 * accumulated since the last reset: which = 0 radix passes that moved data (timed launch by launch), 1 row
 * gather / peer scatter, 2 key extraction, 3 histogram / tie fix-up, 4 partition, 5 group-by, 6 decode / block
 * codec, 7 radix pass launches that were skipped on the device (inactive digit), 8 the in-box
 * shuffle's row scatter over NVLink, 9 its sampling / pivot selection / count exchange / peer barriers (includes the
 * time spent WAITING for the other ranks), 10 sorted-input segmented reduce.
 * launches (nullable) receives the number of launches behind the returned time. */
double ytgpu_context_kernel_ms(ytgpu_context* ctx, int which, uint64_t* launches);
void ytgpu_context_reset_timers(ytgpu_context* ctx);
/* Radix passes that actually moved data in the most recent sort on this context (digits whose
 * histogram has a single bin are skipped); synchronises the stream. */
uint64_t ytgpu_context_last_sort_passes(ytgpu_context* ctx);
void ytgpu_context_enable_timers(ytgpu_context* ctx, int enabled);
/* Options of one context.  Each chooses between two algorithms that produce the same result; the defaults are the
 * faster ones.  A new context starts with the defaults:
 *   "sort_hybrid"  1 (default): single-chunk keys are sorted by their most significant active digits first and short
 *                  runs of equal prefixes are fixed up; 0: always the full LSD schedule.
 *   "merge_path"   1 (default): ytgpu_merge_sorted_runs merges up to 16 sorted runs pairwise (merge path); 0: always the
 *                  stable sort of the concatenated runs.
 * Returns INVALID_ARGUMENT for an unknown name. */
int ytgpu_context_set_option(ytgpu_context* ctx, const char* name, int64_t value, ytgpu_error* err);
/* Reads an option back, or one of the read-only counters:
 *   "last_merge_used_merge_path"  1 when the most recent ytgpu_merge_sorted_runs took the merge-path rounds, 0 when it
 *                                 sorted (many runs, an unsorted run, or the option switched off). */
int ytgpu_context_get_option(ytgpu_context* ctx, const char* name, int64_t* value, ytgpu_error* err);

/* Completion notification without blocking a thread: `fn(user)` runs on a driver thread once everything enqueued on the
 * context's stream so far has finished (cudaLaunchHostFunc).  The adapters set the TFuture<void> behind GetReadyEvent()
 * from it, so a YT fiber never sits in cudaStreamSynchronize (SURVEY §8b "Threading"; sorting_reader.cpp:53-55 runs
 * DoOpen via AsyncVia for the same reason).  DEVICE-flavour calls are asynchronous; enqueue the call(s), then the
 * notification.  The callback must not call back into the library. */
typedef void (*ytgpu_callback)(void* user);
int ytgpu_context_notify(ytgpu_context* ctx, ytgpu_callback fn, void* user, ytgpu_error* err);

/* Pinned host buffers for the HOST-memory flavour of the calls (cudaHostAlloc). */
void* ytgpu_host_alloc(size_t bytes);
void ytgpu_host_free(void* p);

int ytgpu_abi_version(void);

/* ---- row model ---- */
/* EValueType, yt/yt/client/table_client/row_base.h:11-28 */
enum {
    YTGPU_TYPE_MIN = 0x00, YTGPU_TYPE_BOTTOM = 0x01, YTGPU_TYPE_NULL = 0x02, YTGPU_TYPE_INT64 = 0x03,
    YTGPU_TYPE_UINT64 = 0x04, YTGPU_TYPE_DOUBLE = 0x05, YTGPU_TYPE_BOOLEAN = 0x06, YTGPU_TYPE_STRING = 0x10,
    YTGPU_TYPE_ANY = 0x11, YTGPU_TYPE_COMPOSITE = 0x12, YTGPU_TYPE_MAX = 0xef
};

/* TUnversionedValue, yt/yt/client/table_client/unversioned_value.h:37-62 (same 16-byte layout).
 * For string-like types `data` is a byte OFFSET into the rowset's string heap. */
typedef struct ytgpu_value {
    uint16_t id;
    uint8_t type;
    uint8_t flags;
    uint32_t length;
    uint64_t data;
} ytgpu_value;

/* A drained TRange<TUnversionedRow> (unversioned_row.h:272-352): row_count rows of value_count values. */
typedef struct ytgpu_rowset_view {
    const ytgpu_value* values;
    uint64_t row_count;
    uint32_t value_count;
    uint32_t reserved;
    const uint8_t* string_heap;
    uint64_t string_heap_bytes;
    int32_t mem; /* ytgpu_mem of values and string_heap */
} ytgpu_rowset_view;

/* Fixed-width packed rows: schemaful rows whose columns are all required fixed-size scalars or
 * fixed-length strings (the benchmark's "64-byte row": uint64 key + string[56]). */
typedef struct ytgpu_fixed_rows_view {
    const uint8_t* rows;
    uint64_t row_count;
    uint32_t row_bytes; /* multiple of 16 */
    int32_t mem;
} ytgpu_fixed_rows_view;

/* One key column: TColumnSortSchema{Name, SortOrder} + the type information of TColumnSchema.
 *  rowset:     `index` = position of the value in the row; `type` = declared EValueType or 0 for "any
 *              scalar" (schemaless keys); `required` drops the type byte (TColumnSchema::Required());
 *              `width` = maximum string length (0 = measure it on the device).
 *  fixed rows: `index` = byte offset in the row; `type` one of INT64/UINT64/DOUBLE/BOOLEAN/STRING;
 *              `width` = exact string length. */
typedef struct ytgpu_key_column {
    uint32_t index;
    uint32_t width;
    uint8_t type;
    uint8_t descending; /* ESortOrder::Descending, comparator.cpp:56-58 */
    uint8_t required;
    uint8_t reserved;
} ytgpu_key_column;

typedef struct ytgpu_sort_spec {
    const ytgpu_key_column* columns; /* host memory */
    uint32_t column_count;           /* == TComparator::GetLength() */
} ytgpu_sort_spec;

/* ---- sort ----
 * Replaces TSortingReader::DoOpen's std::sort (yt/yt/ytlib/table_client/sorting_reader.cpp:163-188,
 * factory sorting_reader.h:15-20) and TPartitionSortReader's bucket sort + merge
 * (partition_sort_reader.cpp:384-529).  The sort is STABLE (rows with equal keys keep input order),
 * which is one of the orders the reference's unstable std::sort may produce.
 * out_perm[i] = input index of the i-th output row. */
int ytgpu_sort_rowset(ytgpu_context* ctx, const ytgpu_rowset_view* in, const ytgpu_sort_spec* spec,
                      uint32_t* out_perm, ytgpu_value* out_values /* nullable: rows gathered in sorted order */,
                      int out_mem, ytgpu_error* err);

int ytgpu_sort_fixed_rows(ytgpu_context* ctx, const ytgpu_fixed_rows_view* in, const ytgpu_sort_spec* spec,
                          uint8_t* out_rows /* nullable */, uint32_t* out_perm /* nullable */, int out_mem,
                          ytgpu_error* err);

/* Replaces CreateSortedMergingReader (sorted_merging_reader.cpp:771-788; order = CompareStreams :395-409):
 * `in` is the concatenation of run_count sorted runs, run r = rows [run_offsets[r], run_offsets[r+1]).
 * Ties are broken by run index, then by position in the run. */
int ytgpu_merge_sorted_runs(ytgpu_context* ctx, const ytgpu_rowset_view* in, const ytgpu_sort_spec* spec,
                            const uint64_t* run_offsets /* host */, uint32_t run_count, uint32_t* out_perm,
                            int out_mem, ytgpu_error* err);

/* Replaces CreateSortedJoiningReader / TSortedJoiningReader::Read (sorted_merging_reader.cpp:566-760, factory :790-815):
 * run 0 of `in` is the PRIMARY stream (the already merged primary readers), runs 1.. are the FOREIGN streams; every run
 * is sorted by the join key = the first join_key_column_count columns of `spec`.  The remaining spec columns only break
 * ties between streams: the reference's heap orders streams with equal keys by their table index (CompareStreams
 * :395-409; one index per stream, taken from its first row :101-104), so the adapters append that index as the last
 * key column.  The result is the stable order by all spec columns in which a foreign row survives iff its join key
 * occurs in the primary stream (:722-738: it equals the last primary key consumed or the next one).
 * out_perm (capacity row_count) receives the input indices of the emitted rows, *out_row_count (host) their number. */
int ytgpu_join_sorted_runs(ytgpu_context* ctx, const ytgpu_rowset_view* in, const ytgpu_sort_spec* spec,
                           uint32_t join_key_column_count, const uint64_t* run_offsets /* host */, uint32_t run_count,
                           uint32_t* out_perm, uint64_t* out_row_count, int out_mem, ytgpu_error* err);

/* ---- partition ----
 * Replaces the per-row IPartitioner::GetPartitionIndex loop of TPartitionMultiChunkWriter::WriteRow
 * (yt/yt/ytlib/table_client/partitioner.h:14-19, partitioner.cpp:41-57,99-107,122-173,
 * schemaless_chunk_writer.cpp:1604-1623) and CreatePartitioner (ytlib/job_proxy/helpers.cpp:113-147). */
typedef enum ytgpu_partitioner_kind {
    YTGPU_PARTITION_ORDERED = 0, YTGPU_PARTITION_HASH = 1, YTGPU_PARTITION_COLUMN = 2
} ytgpu_partitioner_kind;

typedef struct ytgpu_partition_spec {
    int32_t kind;
    int32_t partition_count;          /* ordered: number of lower bounds incl. the universal bound 0 */
    /* ordered: */
    ytgpu_sort_spec key;              /* comparator */
    const ytgpu_value* bounds;        /* host; partition_count rows of bound_value_count values */
    const uint8_t* bounds_heap;       /* host */
    uint64_t bounds_heap_bytes;
    uint32_t bound_value_count;
    const uint32_t* bound_prefix_length; /* host; values of the prefix used by bound b (0 = universal) */
    const uint8_t* bound_inclusive;      /* host */
    /* hash: */
    int32_t key_column_count;         /* reduce_key_column_count */
    uint64_t salt;                    /* partition_task_level; Salt_ = FarmHash(salt), partitioner.cpp:88-91 */
    /* column: */
    uint16_t partition_column_id;
} ytgpu_partition_spec;

/* out_index (nullable) gets the partition of every row; out_histogram (nullable, partition_count
 * entries) the rows per partition.  Both live in out_mem. */
int ytgpu_partition_rowset(ytgpu_context* ctx, const ytgpu_rowset_view* in, const ytgpu_partition_spec* spec,
                           int32_t* out_index, uint64_t* out_histogram, int out_mem, ytgpu_error* err);

/* The same with the rows scattered into partition-contiguous slabs (stable inside a partition) for VARIABLE-length rows:
 * out_slab_values (nullable, row_count * value_count values) receives the rows' values grouped by partition — string
 * values keep their offsets into the INPUT heap, which therefore serves all slabs — and out_slab_perm (nullable,
 * row_count entries) the input row index of every slab row.  Partition p's rows are [sum(hist[0..p)), +hist[p]).
 * This is what the P per-partition block writers of TPartitionMultiChunkWriter accumulate
 * (schemaless_chunk_writer.cpp:1604-1623) before FlushBlock encodes a partition's rows. */
int ytgpu_partition_rowset_slabs(ytgpu_context* ctx, const ytgpu_rowset_view* in, const ytgpu_partition_spec* spec,
                                 int32_t* out_index, uint64_t* out_histogram, ytgpu_value* out_slab_values,
                                 uint32_t* out_slab_perm, int out_mem, ytgpu_error* err);

/* Fixed-row flavour used by the in-box shuffle: additionally scatters the rows into
 * partition-contiguous slabs (stable inside a partition) — the GPU equivalent of the P per-partition
 * block writers (schemaless_chunk_writer.cpp:1609-1616).  out_slab_rows nullable. */
int ytgpu_partition_fixed_rows(ytgpu_context* ctx, const ytgpu_fixed_rows_view* in,
                               const ytgpu_partition_spec* spec, int32_t* out_index, uint64_t* out_histogram,
                               uint8_t* out_slab_rows, int out_mem, ytgpu_error* err);

/* ---- in-box shuffle over NVLink peer memory ----
 * Inside one 8-GPU box the reference's materialised shuffle (partition jobs tag blocks with partition_index,
 * schemaless_chunk_writer.cpp:1650-1667; sort jobs fetch them by tag, partition_chunk_reader.cpp:82-86) becomes one
 * kernel that writes each destination's slab straight into that GPU's receive buffer.  One process per GPU:
 * receive buffers are shared through CUDA IPC handles (64 opaque bytes, exchanged by the host plumbing). */
#define YTGPU_IPC_HANDLE_BYTES 64
int ytgpu_peer_buffer_create(ytgpu_context* ctx, uint64_t bytes, void** out_dev_ptr, uint8_t* out_handle /*[64]*/,
                             ytgpu_error* err);
int ytgpu_peer_buffer_destroy(ytgpu_context* ctx, void* dev_ptr, ytgpu_error* err);
int ytgpu_peer_buffer_open(ytgpu_context* ctx, const uint8_t* handle /*[64]*/, void** out_dev_ptr, ytgpu_error* err);
int ytgpu_peer_buffer_close(ytgpu_context* ctx, void* dev_ptr, ytgpu_error* err);
/* Fused slab scatter + exchange.  `in` (DEVICE) holds the rows, partition_index (DEVICE) their partitions as returned
 * by ytgpu_partition_fixed_rows, partition_rows (host) the rows per partition.  Partition p's rows are written in
 * stable order to dest_base[p] (host array of device pointers: local memory or peer-mapped receive buffers).
 * Returns after the kernel completed on this GPU; a cross-rank barrier makes the data visible to its readers. */
int ytgpu_scatter_rows_to_peers(ytgpu_context* ctx, const ytgpu_fixed_rows_view* in, const int32_t* partition_index,
                                int32_t partition_count, const uint64_t* partition_rows, void* const* dest_base,
                                ytgpu_error* err);

/* ---- in-box distributed sort: the whole Partition -> Sort hand-off of the sort controller for the GPUs of one box ----
 * Reference shape: samples -> BuildPartitionKeysFromSamples (yt/yt/server/controller_agent/helpers.cpp:263-425) ->
 * partition jobs with the ordered partitioner (partitioner.cpp:41-57) -> sort jobs per partition
 * (sort_controller.cpp:3444-3456).  One process (or thread) per GPU makes the same calls; rank r ends up with key range
 * r sorted (stable: ties keep (source rank, input position) order), so the concatenation over ranks is the sorted
 * table.  Ranks communicate only through peer-mapped device memory over NVLink: sample keys, the g x g row-count
 * matrix, device-side barriers and the rows themselves (fused slab scatter) — no NCCL, no host barrier; the host reads
 * the count matrix once per sort.  Pivot selection handles skew like the reference (weighted samples, maniac
 * partitions for heavily duplicated keys).
 * Setup: every rank creates its shuffle (receive buffer of capacity_rows rows) and obtains a 64-byte CUDA IPC handle;
 * the caller's own plumbing (job proxy RPC / torch.distributed in bench.py) gathers the handles of all ranks, in rank
 * order, and every rank passes the array to ytgpu_shuffle_connect. */
#define YTGPU_MAX_SHUFFLE_RANKS 32
typedef struct ytgpu_shuffle ytgpu_shuffle;
typedef struct ytgpu_shuffle_stats {
    uint64_t rows_in;                             /* rows this rank contributed */
    uint64_t rows_out;                            /* rows of this rank's key range */
    uint64_t sent[YTGPU_MAX_SHUFFLE_RANKS];       /* rows sent to every rank */
    uint64_t received[YTGPU_MAX_SHUFFLE_RANKS];   /* rows received from every rank */
    uint32_t world;
    uint32_t maniac;                              /* this rank's partition holds a single key (no sort was needed) */
} ytgpu_shuffle_stats;
int ytgpu_shuffle_create(ytgpu_context* ctx, int world, int rank, uint64_t capacity_rows, uint32_t row_bytes,
                         ytgpu_shuffle** out, uint8_t* out_handle /*[64]*/, ytgpu_error* err);
int ytgpu_shuffle_connect(ytgpu_shuffle* shuffle, const uint8_t* handles /*[world][64], rank order*/, ytgpu_error* err);
/* Collective: every rank calls it with its shard (`in`, DEVICE memory) and the same spec.  out_rows (DEVICE, nullable)
 * receives the rank's sorted key range, *out_row_count its size; INVALID_ARGUMENT when it exceeds out_capacity_rows or
 * when any rank's range exceeds its receive buffer (all ranks fail together).  Synchronises the stream once. */
int ytgpu_shuffle_sort(ytgpu_shuffle* shuffle, const ytgpu_fixed_rows_view* in, const ytgpu_sort_spec* spec,
                       uint8_t* out_rows, uint64_t out_capacity_rows, uint64_t* out_row_count, ytgpu_shuffle_stats* stats,
                       ytgpu_error* err);
int ytgpu_shuffle_destroy(ytgpu_shuffle* shuffle, ytgpu_error* err);

/* GetFarmFingerprint(row.FirstNElements(k)), unversioned_row.cpp:586-594, farm_hash.h:51-59. */
int ytgpu_farm_fingerprint_rowset(ytgpu_context* ctx, const ytgpu_rowset_view* in, uint32_t key_column_count,
                                  uint64_t* out, int out_mem, ytgpu_error* err);

/* ---- horizontal (schemaless) block codec: the intermediate-chunk wire format of partition / sort jobs ----
 * block = ui32 offsets[row_count] ++ rows; row = varuint32 value_count, then per value varuint32 id, varuint32 type,
 * payload (Int64 zig-zag varint, Uint64 varint, Double 8 raw bytes, Boolean 1 byte, String/Any varuint32 length +
 * bytes; Composite is written as Any).
 * Decode replaces THorizontalBlockReader::JumpToRowIndex/GetRow + ReadRowValue
 * (yt/yt/ytlib/table_client/schemaless_block_reader.cpp:187-246,323-349; unversioned_row.cpp:208-280): the first
 * value_count values of every row (short rows padded with Null, id 0xffff); a string value's `data` is the byte
 * offset of its payload INSIDE THE BLOCK (pass the block as the string heap of the resulting rowset).
 * out_row_value_counts (nullable) receives each row's real value count.  Malformed input -> INVALID_ARGUMENT. */
int ytgpu_decode_horizontal_block(ytgpu_context* ctx, const uint8_t* block, uint64_t block_bytes, uint32_t row_count,
                                  uint32_t value_count, ytgpu_value* out_values, uint32_t* out_row_value_counts,
                                  int mem, ytgpu_error* err);
/* Encode replaces THorizontalBlockWriter::WriteRow/FlushBlock + WriteRowValue
 * (schemaless_block_writer.cpp:40-86; unversioned_row.cpp:159-206).  row_value_counts (nullable, same memory space
 * as `rows`) gives the values actually present in each row.  *out_block_bytes is always set to the size the block
 * needs; the call fails with INVALID_ARGUMENT when out_capacity is smaller. */
int ytgpu_encode_horizontal_block(ytgpu_context* ctx, const ytgpu_rowset_view* rows, const uint32_t* row_value_counts,
                                  uint8_t* out_block, uint64_t out_capacity, uint64_t* out_block_bytes, int out_mem,
                                  ytgpu_error* err);

/* ---- columnar batches ----
 * Mirrors IUnversionedColumnarRowBatch::TColumn (yt/yt/client/table_client/row_batch.h:49-191) so a
 * MaterializeColumns() result can be described without copying semantics.  All pointers of one
 * view share `mem`.  Integer/double/boolean columns only (strings: offsets helper below). */
#define YTGPU_COLUMN_ARROW_VALIDITY 1u
typedef struct ytgpu_column_view {
    int64_t start_index;            /* TColumn::StartIndex */
    int64_t value_count;            /* TColumn::ValueCount */
    uint8_t value_type;             /* YTGPU_TYPE_INT64 / UINT64 / DOUBLE / BOOLEAN */
    uint8_t has_values;             /* TColumn::Values present (else: all null) */
    uint8_t zigzag;                 /* TValueBuffer::ZigZagEncoded */
    uint8_t bit_width;              /* 8/16/32/64, 0 when `values` is a TBitPackedUnsignedVector, 1 when it is a plain
                                       TBitmap (boolean columns: boolean_column_reader.cpp:134-172) */
    uint32_t reserved;              /* flags; bit 0 (YTGPU_COLUMN_ARROW_VALIDITY): null_bitmap is an Arrow validity
                                       bitmap (bit set = VALID), so an Arrow block — the input of YQL's
                                       BlockCombineHashed — is described without rewriting its bitmap */
    uint64_t base_value;            /* TValueBuffer::BaseValue */
    const void* values;             /* value vector of the (leaf) value column: dictionary values when
                                       dictionary-encoded, RLE values when RLE-encoded, else direct */
    uint64_t values_count;
    const uint8_t* null_bitmap;     /* nullable; bit i set = value i of the value vector is null */
    const uint32_t* dictionary_indexes; /* nullable; 1-based, 0 = null (ZeroMeansNull) */
    uint64_t dictionary_index_count;
    const uint64_t* rle_indexes;    /* nullable; start index of each run; rle_indexes[0] == 0 */
    uint64_t rle_count;
    int32_t mem;
} ytgpu_column_view;

/* DecodeIntegerVector + BuildNullBytemapForCHColumn (columnar-inl.h:355-376,
 * yt/chyt/server/columnar_conversion.cpp:204-234,948-999; bit unpack
 * yt/yt/core/misc/bit_packed_unsigned_vector-inl.h:115-173).  out_values gets value_count 64-bit
 * values (nulls decode to 0), out_null_bytemap (nullable) value_count bytes (1 = null). */
int ytgpu_decode_column(ytgpu_context* ctx, const ytgpu_column_view* column, uint64_t* out_values,
                        uint8_t* out_null_bytemap, int out_mem, ytgpu_error* err);

/* The same decode into a ClickHouse ColumnVector<T>: ConvertIntegerYTColumnToCHColumn (yt/chyt/server/
 * columnar_conversion.cpp:204-234,1001-1050) assigns the decoded 64-bit value to the column's element type (Int8 .. UInt64,
 * Date = UInt16, Date32 = Int32, Datetime = UInt32, DateTime64 = Int64: element_bytes 1 / 2 / 4 / 8, narrowed by truncation);
 * ConvertFloatingPointYTColumnToCHColumn (:341-369): a value vector of 32-bit floats (value_type Double, bit_width 32)
 * read with element_bytes 8 is widened to doubles, with element_bytes 4 copied; doubles are copied with element_bytes 8. */
int ytgpu_decode_column_typed(ytgpu_context* ctx, const ytgpu_column_view* column, uint32_t element_bytes, void* out_values,
                              uint8_t* out_null_bytemap, int out_mem, ytgpu_error* err);

/* DecodeStringOffsets, columnar.cpp:654-684: out[k-start] = offset(k) - offset(start), k in [start,end]. */
int ytgpu_decode_string_offsets(ytgpu_context* ctx, const uint32_t* encoded, uint32_t avg_length,
                                int64_t start_index, int64_t end_index, uint32_t* out, int mem,
                                ytgpu_error* err);

/* DecodeStringPointersAndLengths, columnar.cpp:686-707 (the string column reader's dense / dictionary value decode,
 * string_column_reader.cpp:266-520): value i of a string segment starts at out_start[i] inside the segment's string data
 * and is out_length[i] bytes long; end(i) = avg_length * (i + 1) + ZigZagDecode(encoded[i]).  `count` values. */
int ytgpu_decode_string_pointers_and_lengths(ytgpu_context* ctx, const uint32_t* encoded, uint32_t avg_length, uint64_t count,
                                             uint32_t* out_start, int32_t* out_length, int mem, ytgpu_error* err);

/* ---- null / dictionary-index helpers of the column readers (client/table_client/columnar.h:13-200) ----
 * The reference builds Arrow validity bitmaps, ClickHouse null bytemaps and Arrow dictionary indexes out of two kinds of
 * per-value flags: "the 1-based dictionary index is 0" (ZeroMeansNull) and "the bit of a TBitmap is set", either
 * addressed directly by the row or through RLE run starts.  One flag source + three consumers cover the family:
 *
 *   reference function (columnar.cpp)                                  entry point                      source     rle  negate
 *   BuildValidityBitmapFromDictionaryIndexesWithZeroNull    :286-331   ytgpu_build_bitmap_from_flags    DICT_ZERO  no   1
 *   BuildValidityBitmapFromRleDictionaryIndexesWithZeroNull :333-348   ytgpu_build_bitmap_from_flags    DICT_ZERO  yes  1
 *   BuildValidityBitmapFromRleNullBitmap                    :623-636   ytgpu_build_bitmap_from_flags    BITMAP     yes  1
 *   CopyBitmapRangeToBitmap / ...Negated                    :577-601   ytgpu_build_bitmap_from_flags    BITMAP     no   0 / 1
 *   BuildNullBytemapFromDictionaryIndexesWithZeroNull       :350-364   ytgpu_build_bytemap_from_flags   DICT_ZERO  no   0
 *   BuildNullBytemapFromRleDictionaryIndexesWithZeroNull    :366-382   ytgpu_build_bytemap_from_flags   DICT_ZERO  yes  0
 *   BuildNullBytemapFromRleNullBitmap                       :638-652   ytgpu_build_bytemap_from_flags   BITMAP     yes  0
 *   DecodeBytemapFromBitmap                                 :603-621   ytgpu_build_bytemap_from_flags   BITMAP     no   0
 *   CountNullsInDictionaryIndexesWithZeroNull               :454-466   ytgpu_count_flags                DICT_ZERO  no
 *   CountNullsInRleDictionaryIndexesWithZeroNull            :468-493   ytgpu_count_flags                DICT_ZERO  yes
 *   CountOnesInBitmap                                       :495-548   ytgpu_count_flags                BITMAP     no
 *   CountOnesInRleBitmap                                    :550-575   ytgpu_count_flags                BITMAP     yes
 *   BuildDictionaryIndexesFromDictionaryIndexesWithZeroNull :384-398   ytgpu_build_dictionary_indexes   (rle_indexes NULL)
 *   BuildDictionaryIndexesFromRleDictionaryIndexesWithZeroNull :400-420 ytgpu_build_dictionary_indexes
 *   BuildIotaDictionaryIndexesFromRleIndexes                :422-452   ytgpu_build_dictionary_indexes   (dictionary_indexes NULL)
 *   CountTotalStringLengthInRleDictionaryIndexesWithZeroNull :709-735  ytgpu_count_total_string_length
 *   TranslateRleIndex / ...StartIndex / ...EndIndex         :737-768   ytgpu_translate_rle_indexes
 *
 * Rows [start_index, end_index) are produced.  Bitmaps are written as GetBitmapByteSize(end - start) bytes, the unused
 * bits of the last byte zero; bytes behind them are not touched.  Bytemap bytes are 0 / 1.  YT_VERIFY conditions of the
 * reference (negative or reversed ranges, rle_indexes[0] != 0, ranges past the data) come back as
 * YTGPU_ERR_INVALID_ARGUMENT. */
typedef enum ytgpu_flag_kind {
    YTGPU_FLAGS_DICTIONARY_ZERO = 0, /* flag(i) = (dictionary_indexes[k(i)] == 0); data = uint32 indexes */
    YTGPU_FLAGS_BITMAP = 1           /* flag(i) = bit k(i) of a TBitmap; data = bitmap bytes */
} ytgpu_flag_kind;

typedef struct ytgpu_flag_source {
    int32_t kind;                /* ytgpu_flag_kind */
    int32_t reserved;
    const void* data;
    uint64_t data_count;         /* number of dictionary indexes | number of BITS in the bitmap */
    const uint64_t* rle_indexes; /* nullable: k(i) = i; else k(i) = TranslateRleIndex(rle_indexes, i), rle_indexes[0] == 0 */
    uint64_t rle_count;
} ytgpu_flag_source;

/* `mem` names the space of every buffer of the call (source data, rle indexes, dst); counts are returned to the host. */
int ytgpu_build_bitmap_from_flags(ytgpu_context* ctx, const ytgpu_flag_source* source, int64_t start_index, int64_t end_index,
                                  int negate, uint8_t* dst, int mem, ytgpu_error* err);
int ytgpu_build_bytemap_from_flags(ytgpu_context* ctx, const ytgpu_flag_source* source, int64_t start_index, int64_t end_index,
                                   int negate, uint8_t* dst, int mem, ytgpu_error* err);
int ytgpu_count_flags(ytgpu_context* ctx, const ytgpu_flag_source* source, int64_t start_index, int64_t end_index,
                      int64_t* out_count, int mem, ytgpu_error* err);
/* dst[i - start] = dictionary_indexes[k(i)] - 1 (a null becomes 0xFFFFFFFF); dictionary_indexes == NULL: the number of
 * the run holding row i, counted from the run holding start_index (rle_indexes required). */
int ytgpu_build_dictionary_indexes(ytgpu_context* ctx, const uint32_t* dictionary_indexes, uint64_t dictionary_index_count,
                                   const uint64_t* rle_indexes, uint64_t rle_count, int64_t start_index, int64_t end_index,
                                   uint32_t* dst, int mem, ytgpu_error* err);
/* sum over rows [start, end) of string_lengths[dictionary_indexes[k(i)] - 1], nulls counting 0. */
int ytgpu_count_total_string_length(ytgpu_context* ctx, const uint32_t* dictionary_indexes, const uint64_t* rle_indexes,
                                    uint64_t rle_count, const int32_t* string_lengths, uint64_t string_count,
                                    int64_t start_index, int64_t end_index, int64_t* out_total, int mem, ytgpu_error* err);
/* out[j] = TranslateRleIndex(rle_indexes, indexes[j]) (end_flavour 0; also TranslateRleStartIndex) or
 * TranslateRleEndIndex(rle_indexes, indexes[j]) (end_flavour 1). */
int ytgpu_translate_rle_indexes(ytgpu_context* ctx, const uint64_t* rle_indexes, uint64_t rle_count, const int64_t* indexes,
                                uint64_t count, int end_flavour, int64_t* out, int mem, ytgpu_error* err);

/* ---- scan -> filter -> GROUP BY key: SUM(val), COUNT(*) ----
 * Replaces the scan loop + hash aggregation of
 *   CHYT: TSecondaryQuerySourceBase::generate (yt/chyt/server/secondary_query_source.cpp:293-400) feeding
 *         DB::Aggregator::executeOnBlock (key64, AggregateFunctionSum/Count), and
 *   YT QL: ScanOpHelper/GroupOpHelper/InsertGroupRow (library/query/engine/cg_routines/registry.cpp:315-438,
 *         1783-1920) with the `sum` aggregate (engine/udf/sum.c:12-36).
 * Semantics: NULL key is its own group; SUM skips nulls and is NULL when no non-null value was seen;
 * integer SUM wraps mod 2^64; COUNT(*) counts every row that passes the filter. */
typedef enum ytgpu_cmp_op {
    YTGPU_CMP_NONE = 0, YTGPU_CMP_LT = 1, YTGPU_CMP_LE = 2, YTGPU_CMP_GT = 3, YTGPU_CMP_GE = 4,
    YTGPU_CMP_EQ = 5, YTGPU_CMP_NE = 6
} ytgpu_cmp_op;

typedef struct ytgpu_predicate {
    int32_t op;        /* compares the VALUE column with `constant`; a null value never passes */
    int32_t reserved;
    uint64_t constant; /* bit pattern in the column's value type */
} ytgpu_predicate;

typedef struct ytgpu_groupby_result {
    uint64_t group_count;
    uint64_t* keys;          /* [capacity] */
    uint8_t* key_null;       /* [capacity] */
    uint64_t* sums;          /* [capacity] bit patterns in the value type */
    uint8_t* sum_null;       /* [capacity] */
    uint64_t* counts;        /* [capacity] */
    uint64_t capacity;       /* in: allocated groups; YTGPU_ERR_INVALID_ARGUMENT if exceeded */
    uint64_t* first_rows;    /* [capacity], nullable: index (inside the batch) of the first row of every group.
                                YT QL emits groups in first-seen order (InsertGroupRow, cg_routines/registry.cpp:
                                1571-1655): sort the result by first_rows to reproduce it */
    uint64_t* mins;          /* [capacity], nullable: MIN(value) / MAX(value) of every group over its non-NULL values that */
    uint64_t* maxs;          /* passed the predicate, bit patterns in the value type; 0 where sum_null is set (the
                                aggregate is NULL: udf/min.c:21-56, max.c).  Integers: exact.  Doubles are ordered like
                                AggLess (mkql_block_agg_minmax.cpp:20-31): NaN is the biggest value (returned as the
                                canonical quiet NaN); -0.0 orders below +0.0 (the reference keeps whichever zero its row
                                order met last).  Either pointer may be given alone. */
} ytgpu_groupby_result;

/* Groups are emitted ordered by (key_null, key) — ClickHouse's order is hash-table order (unspecified), QL's is
 * first-seen: pass out->first_rows to get every group's first row index and order by it.
 * group_count_hint is a HINT (expected number of groups, 0 = unknown): it sizes the hash table; when the table turns
 * out too small the pass is repeated with a doubled table, it never fails because of the hint.  Hints up to 2048 use a
 * shared-memory front table per CTA. */
int ytgpu_scan_filter_groupby(ytgpu_context* ctx, const ytgpu_column_view* key_column,
                              const ytgpu_column_view* value_column, const ytgpu_predicate* predicate,
                              uint64_t group_count_hint, ytgpu_groupby_result* out, int out_mem,
                              ytgpu_error* err);

/* ---- GROUP BY over a key TUPLE with a LIST of aggregates (the general form of the call above) ----
 * Replaces GroupOpHelper / InsertGroupRow with several group items and aggregate items (registry.cpp:1571-1655,1783-1920;
 * aggregates of library/query/base/builtin_function_types.cpp:201-254: sum, min, max — engine/udf/sum.c, min.c, max.c —,
 * avg, argmin, argmax — engine/builtin_function_profiler.cpp:1300-1620 —, first — registry.cpp:3633-3693 — and count),
 * ClickHouse's Aggregator over a multi-column key and YQL's BlockCombineHashed over tuple keys
 * (mkql_block_agg.cpp:1234-1400).  Semantics, per aggregate, over the rows of a group that passed the predicate:
 *   SUM    skips NULLs, NULL when no value was seen; integers wrap mod 2^64; doubles are added in arbitrary order
 *   MIN / MAX  skip NULLs, NULL without values; doubles ordered like AggLess (NaN is the biggest, -0.0 < +0.0)
 *   COUNT  number of non-NULL values of the column (COUNT(*) is out->counts)
 *   AVG    double(sum) / double(count of non-NULL values), NULL without values; result bits are a double
 *   ARGMIN / ARGMAX  value of `column` in the FIRST row (smallest index) that attains MIN / MAX of `by_column` among the
 *          rows where both are non-NULL (the reference replaces its state only on a strict comparison)
 *   FIRST  the first non-NULL value of the column
 * Key columns are compared as (is-null, 64-bit payload) tuples — doubles by bit pattern.  Groups are emitted in
 * FIRST-SEEN order (QL's order; ClickHouse's is unspecified).  At most 8 key columns, 32 aggregates, 2^30 rows per call. */
typedef enum ytgpu_agg_op {
    YTGPU_AGG_SUM = 0, YTGPU_AGG_MIN = 1, YTGPU_AGG_MAX = 2, YTGPU_AGG_COUNT = 3, YTGPU_AGG_AVG = 4,
    YTGPU_AGG_ARGMIN = 5, YTGPU_AGG_ARGMAX = 6, YTGPU_AGG_FIRST = 7
} ytgpu_agg_op;

typedef struct ytgpu_aggregate {
    int32_t op;         /* ytgpu_agg_op */
    int32_t column;     /* index into value_columns: the aggregated (argmin / argmax: the returned) column */
    int32_t by_column;  /* argmin / argmax: the column that is minimised / maximised */
    int32_t reserved;
} ytgpu_aggregate;

typedef struct ytgpu_groupby_multi_result {
    uint64_t group_count;        /* out */
    uint64_t capacity;           /* in: entries of every output array; INVALID_ARGUMENT if exceeded */
    uint64_t* const* keys;       /* host array of key_count arrays [capacity] */
    uint8_t* const* key_null;    /* host array of key_count arrays [capacity] */
    uint64_t* const* values;     /* host array of aggregate_count arrays [capacity]: bit patterns in the result type */
    uint8_t* const* value_null;  /* host array of aggregate_count arrays [capacity] */
    uint64_t* counts;            /* [capacity], nullable: COUNT(*) */
    uint64_t* first_rows;        /* [capacity], nullable: index of the group's first row (ascending in the output) */
} ytgpu_groupby_multi_result;

/* predicate (nullable) compares value_columns[predicate_column]; a NULL there never passes.  All columns hold the
 * same number of rows.  group_count_hint as above (0 = unknown). */
int ytgpu_scan_filter_groupby_multi(ytgpu_context* ctx, const ytgpu_column_view* key_columns, uint32_t key_count,
                                    const ytgpu_column_view* value_columns, uint32_t value_count,
                                    const ytgpu_aggregate* aggregates, uint32_t aggregate_count,
                                    const ytgpu_predicate* predicate, int32_t predicate_column, uint64_t group_count_hint,
                                    ytgpu_groupby_multi_result* out, int out_mem, ytgpu_error* err);

/* ---- segmented SUM / COUNT over rows ALREADY SORTED by the group key (the aggregate stage after a sort) ----
 * Consecutive rows with equal keys form a group; no hash table.  Replaces the per-group accumulation of a GROUP BY
 * over a sorted stream / a sorted reduce (yt/yt/library/query/engine/cg_routines/registry.cpp:1838-1920 for the
 * aggregation itself; sort_controller.cpp:3444-3456 produces the sorted partitions).  `in` (DEVICE) holds fixed-width
 * rows whose 8-byte key column at key_offset is non-decreasing (only equality of neighbours is used); the value column
 * at value_offset is INT64 / UINT64 (sums wrap mod 2^64) or DOUBLE.  out_* (DEVICE, `capacity` entries) receive one
 * entry per group in input order, *out_group_count (host) the number of groups; INVALID_ARGUMENT when it exceeds
 * capacity.  Same sums / counts as ytgpu_scan_filter_groupby over the same rows. */
int ytgpu_reduce_sorted_fixed_rows(ytgpu_context* ctx, const ytgpu_fixed_rows_view* in, uint32_t key_offset,
                                   uint32_t value_offset, uint8_t value_type, uint64_t* out_keys, uint64_t* out_sums,
                                   uint64_t* out_counts, uint64_t capacity, uint64_t* out_group_count, ytgpu_error* err);

/* ---- YQL block aggregators over Arrow blocks, "combine all" form ----
 * A fixed-width arrow::ArrayData as TArrowBlock hands it to an aggregator: buffers[0] = validity (LSB bit order,
 * 1 = valid, NULL = no nulls), buffers[1] = 64-bit values; element i is values[offset + i], its validity bit is
 * bit (offset + i).  `nullable` = the YQL item type is Optional<T> (the aggregators' IsNullable template argument). */
typedef struct ytgpu_arrow_array {
    const void* values;
    const uint8_t* validity;
    int64_t offset;
    int64_t length;
    uint8_t value_type;   /* YTGPU_TYPE_INT64 / UINT64 / DOUBLE */
    uint8_t nullable;
    uint16_t reserved;
    int32_t mem;          /* ytgpu_mem of values / validity / the filter */
} ytgpu_arrow_array;

/* The states of the fixed-width aggregators side by side (TSumState, TAvgState, TState<IsNullable,TIn,IsMin>, count):
 * values are bit patterns in the column's type; *_valid mirror IsValid (always 1 for a non-optional column). */
typedef struct ytgpu_block_agg_state {
    uint64_t sum;         /* integers wrap mod 2^64 */
    uint64_t min_value;
    uint64_t max_value;
    uint64_t count;       /* Count(column) == Avg's Count: non-null rows that passed the filter */
    uint64_t count_all;   /* CountAll: rows that passed the filter */
    uint8_t sum_valid, min_valid, max_valid, value_type;
    uint32_t reserved;
} ytgpu_block_agg_state;

/* InitState: zero sums/counts, InitialStateValue for min/max (mkql_block_agg_minmax.cpp:76-101). */
void ytgpu_block_agg_state_init(ytgpu_block_agg_state* state, uint8_t value_type, uint8_t nullable);

/* IBlockAggregatorCombineAll::AddMany (yql/essentials/minikql/comp_nodes/mkql_block_agg_factory.h:34-45) of the sum /
 * avg / min / max / count / count_all aggregators (mkql_block_agg_sum.cpp:160-232,421-485, mkql_block_agg_minmax.cpp:
 * 697-770, mkql_block_agg_count.cpp) in ONE pass over the block: folds the batch into *state (host).  `filter`
 * (nullable) is the non-nullable bool filter column, one byte per row.  Same IsValid rules as the reference,
 * including its quirks (a filtered batch without nulls raises sum's IsValid even if no row passed).  Floating point:
 * the sum is a tree reduction (reproducible for a given length), min/max follow AggLess (NaN is the biggest). */
int ytgpu_block_combine_all(ytgpu_context* ctx, const ytgpu_arrow_array* column, const uint8_t* filter,
                            ytgpu_block_agg_state* state, ytgpu_error* err);

/* ---- columnar write side: rows -> columns -> scan-optimised integer segments ----
 * ytgpu_convert_integer_column replaces TIntegerColumnConverter<T>::Convert
 * (yt/yt/library/column_converters/integer_column_converter.cpp:69-161): value `column_index` of every row becomes
 * one 64-bit word (Int64 zig-zag encoded, Null -> 0) minus *out_base_value, plus a null bitmap (bit i of byte i/8,
 * 1 = null, 8*ceil(n/64) bytes).  The reference never lowers MinValue_ below its initial 2^64-1, so the base is
 * always 2^64-1 and the words are value+1 (mod 2^64); that is kept, the column decodes to the same values.
 * A value that is neither Null nor `value_type` (YTGPU_TYPE_INT64 / UINT64) -> YTGPU_ERR_SCHEMA_VIOLATION. */
int ytgpu_convert_integer_column(ytgpu_context* ctx, const ytgpu_rowset_view* rows, uint32_t column_index,
                                 uint8_t value_type, uint64_t* out_values, uint8_t* out_null_bitmap,
                                 uint64_t* out_base_value /* host */, int out_mem, ytgpu_error* err);

/* One segment of an unversioned integer column as TUnversionedIntegerColumnWriter<T>::DumpSegment emits it
 * (yt/yt/ytlib/table_chunk_format/integer_column_writer.cpp:353-538).  Data parts, in writer order:
 *   DirectDense     : bit-packed (value - min)            | null bitmap (1 bit per row)
 *   DictionaryDense : bit-packed dictionary (value - min) | bit-packed ids (0 = null, else 1-based first-seen id)
 *   DirectRle       : bit-packed run values               | null bitmap (1 bit per run) | bit-packed run starts
 *   DictionaryRle   : bit-packed dictionary               | bit-packed run ids          | bit-packed run starts
 * Bit-packed vectors are TBitPackedUnsignedVector: header word size | width << 56, then ceil(width*size/64) words
 * (yt/yt/core/misc/bit_packed_unsigned_vector-inl.h:31-90); bitmaps are 8*ceil(bits/64) bytes (bitmap.h:131-200). */
typedef struct ytgpu_integer_segment {
    uint32_t type;              /* EUnversionedIntegerSegmentType (table_chunk_format/private.h:25-30):
                                   0 DictionaryRle, 1 DictionaryDense, 2 DirectRle, 3 DirectDense */
    uint32_t row_count;         /* TSegmentMeta::row_count */
    uint64_t chunk_row_count;   /* rows of the chunk up to and including this segment */
    uint64_t min_value;         /* TIntegerSegmentMeta::min_value == TIntegerMeta::BaseValue (encoded domain) */
    uint64_t data_offset;       /* first byte of the segment's data in out_data */
    uint64_t data_bytes;
    uint64_t part_bytes[3];     /* sizes of the data parts in writer order (0 = absent) */
    uint32_t values_size;       /* TIntegerMeta::ValuesSize */
    uint32_t ids_size;          /* TIntegerMeta::IdsSize (dictionary types) */
    uint32_t row_indexes_size;  /* TKeyIndexMeta::RowIndexesSize (RLE types) */
    uint8_t values_width, ids_width, row_indexes_width;
    uint8_t direct;             /* TIntegerMeta::Direct */
} ytgpu_integer_segment;

/* Replaces AddValues + DumpSegment of the unversioned Int64/Uint64 column writer: `values` are the raw 64-bit
 * payloads (is_signed: zig-zag encoded first, integer_column_writer.cpp:24-33), null_bytemap (nullable) marks nulls.
 * A segment is cut every max_segment_value_count rows (config.cpp:130, default 131072) and encoded with whichever of
 * the four layouts the reference's size estimate makes smallest (first minimum in enum order).  chunk_row_offset =
 * rows already written to the chunk (it enters the RLE size estimate).  Segment descriptors go to HOST memory;
 * *out_data_bytes is always set, INVALID_ARGUMENT when out_capacity or segment_capacity is too small. */
int ytgpu_encode_integer_column(ytgpu_context* ctx, const uint64_t* values, const uint8_t* null_bytemap,
                                uint64_t row_count, int is_signed, uint32_t max_segment_value_count,
                                uint64_t chunk_row_offset, int mem, uint8_t* out_data, uint64_t out_capacity,
                                uint64_t* out_data_bytes, ytgpu_integer_segment* out_segments,
                                uint32_t segment_capacity, uint32_t* out_segment_count, ytgpu_error* err);

/* ---- floating-point and boolean column writers ----
 * One segment of an unversioned double / boolean column as the reference's writers dump it:
 *   TUnversionedFloatingPointColumnWriter<double>::DumpSegment (yt/yt/ytlib/table_chunk_format/
 *     floating_point_column_writer.cpp:213-240): ui64 value count | raw doubles (:21-31)  ||  null bitmap
 *   TUnversionedBooleanColumnWriter::DumpSegment (boolean_column_writer.cpp:196-216, DumpBooleanValues :18-28):
 *     ui64 value count  ||  value bitmap  ||  null bitmap
 * Bitmaps: bit i of byte i/8, 8*ceil(rows/64) bytes.  A NULL row stores a zero payload / a false bit (the payload of a
 * Null TUnversionedValue, AddValues :247-256 / :228-238).  Both segment metas are type 0, version 0. */
typedef struct ytgpu_plain_segment {
    uint32_t row_count;         /* TSegmentMeta::row_count */
    uint32_t reserved;
    uint64_t chunk_row_count;   /* rows of the chunk up to and including this segment */
    uint64_t data_offset;       /* first byte of the segment's data in out_data */
    uint64_t data_bytes;
    uint64_t part_bytes[3];     /* sizes of the data parts in writer order (0 = absent) */
} ytgpu_plain_segment;

/* `values`: raw 64-bit patterns of the doubles, null_bytemap (nullable) marks NULL rows.  A segment is cut every
 * max_segment_value_count rows (the reference finishes a segment once it holds at least that many values,
 * floating_point_column_writer.cpp:242-251).  Same capacity protocol as ytgpu_encode_integer_column. */
int ytgpu_encode_double_column(ytgpu_context* ctx, const uint64_t* values, const uint8_t* null_bytemap, uint64_t row_count,
                               uint32_t max_segment_value_count, uint64_t chunk_row_offset, int mem, uint8_t* out_data,
                               uint64_t out_capacity, uint64_t* out_data_bytes, ytgpu_plain_segment* out_segments,
                               uint32_t segment_capacity, uint32_t* out_segment_count, ytgpu_error* err);
/* `values`: one byte per row (non-zero = true).  The reference cuts boolean segments only at block boundaries; the
 * caller chooses max_segment_value_count (pass row_count for one segment). */
int ytgpu_encode_boolean_column(ytgpu_context* ctx, const uint8_t* values, const uint8_t* null_bytemap, uint64_t row_count,
                                uint32_t max_segment_value_count, uint64_t chunk_row_offset, int mem, uint8_t* out_data,
                                uint64_t out_capacity, uint64_t* out_data_bytes, ytgpu_plain_segment* out_segments,
                                uint32_t segment_capacity, uint32_t* out_segment_count, ytgpu_error* err);

/* Rows -> one flat column: the AddValues loops of the column converters / writers for Double, Boolean and String columns
 * (yt/yt/library/column_converters/floating_point_column_converter.cpp:117-127, boolean_column_converter.cpp,
 * string_column_converter.cpp:288-296; floating_point_column_writer.cpp:247-256, boolean_column_writer.cpp:228-238,
 * string_column_writer.cpp:689-705).  out_payload[i] = bit pattern of the double / 0 or 1 / the integer / the string's
 * offset in the rowset's heap; out_lengths (strings; nullable otherwise) its length; out_null_bytemap (nullable) 1 for a
 * Null value, whose payload and length are 0.  The outputs are the inputs of ytgpu_encode_double_column /
 * _boolean_column (one byte per row: narrow the 0 / 1 payloads) / _string_column (starts = payload, heap = the rowset's heap) and of
 * ytgpu_string_value_ids.  A value of another type -> YTGPU_ERR_SCHEMA_VIOLATION. */
int ytgpu_extract_column(ytgpu_context* ctx, const ytgpu_rowset_view* rows, uint32_t column_index, uint8_t value_type,
                         uint64_t* out_payload, uint32_t* out_lengths, uint8_t* out_null_bytemap, int out_mem, ytgpu_error* err);

/* ---- YT string column -> ClickHouse ColumnString (the string path of the CHYT scan) ----
 * ConvertStringLikeYTColumnToCHColumn (yt/chyt/server/columnar_conversion.cpp:429-648,907-912): rows
 * [start_index, start_index + value_count) of a string column in any of its encodings — direct, dictionary (1-based
 * indexes, 0 = null), RLE, dictionary + RLE — become ColumnString's `chars` (every value followed by a zero byte) and
 * `offsets` (offsets[i] = end of value i including that zero byte).  A null row and, with a filter hint
 * (:506-541, CountTotalStringLengthWithFilterHint :397-427), a row whose hint byte is 0 become empty strings; nulls
 * themselves travel in the separate null bytemap (ytgpu_build_bytemap_from_flags).  String i of the value column spans
 * [offset(i), offset(i + 1)) of `chars` with offset(0) = 0, offset(k) = avg_length * k + ZigZagDecode32(offsets[k - 1])
 * (DecodeStringRange, client/table_client/columnar-inl.h:20-50).
 * Two calls per batch: out_chars == NULL returns the exact size in *out_chars_bytes (the reference pre-computes it the
 * same way for the RLE and filter-hint shapes, :506-518,:566-575, and grows its buffer otherwise); then the call with a
 * buffer of at least that many bytes fills out_chars and out_offsets (value_count entries).  A too small capacity is
 * YTGPU_ERR_INVALID_ARGUMENT with the needed size in *out_chars_bytes. */
typedef struct ytgpu_string_column_view {
    const uint32_t* offsets;            /* TStrings: zig-zag encoded differences from avg_length * k (BitWidth 32) */
    uint64_t string_count;              /* strings in the value column (dictionary size when dictionary-encoded) */
    uint32_t avg_length;
    int32_t mem;                        /* ytgpu_mem of every input buffer (and of filter_hint) */
    const uint8_t* chars;
    uint64_t chars_bytes;
    const uint32_t* dictionary_indexes; /* nullable */
    uint64_t dictionary_index_count;
    const uint64_t* rle_indexes;        /* nullable; rle_indexes[0] == 0 */
    uint64_t rle_count;
    int64_t start_index;                /* TColumn::StartIndex */
    int64_t value_count;                /* TColumn::ValueCount */
} ytgpu_string_column_view;

int ytgpu_convert_string_column_to_ch(ytgpu_context* ctx, const ytgpu_string_column_view* column, const uint8_t* filter_hint,
                                      uint8_t* out_chars, uint64_t out_chars_capacity, uint64_t* out_offsets,
                                      uint64_t* out_chars_bytes /* host */, int out_mem, ytgpu_error* err);

/* ---- ClickHouse column -> unversioned values (the write-back side of CHYT) ----
 * TCHToYTConverter::ConvertColumnToUnversionedValues (yt/chyt/server/ch_to_yt_converter.cpp:970-1040) for the types whose
 * logical type is a "V1" simple type, i.e. TSimpleValueConverter::FillValueRange (:131-215) under an optional
 * TNullableConverter (:374-386): every row becomes one 16-byte value with id 0.
 *   INT8..INT64 -> Int64 (sign extended); UINT8..UINT64 -> Uint64; FLOAT32 (widened) / FLOAT64 -> Double;
 *   BOOL: a UInt8 that must be 0 or 1 -> Boolean, anything else fails the call ("Cannot convert value ... to YT boolean",
 *         :183-186; checked for every row, as the reference fills the nested column before it applies the null map);
 *   STRING: ColumnString (chars + offsets, offsets[i] = END of value i INCLUDING its terminating zero byte,
 *         contrib/clickhouse/src/Columns/ColumnString.h:46-53,122-126) -> String values that point into `chars`
 *         (data = offset of the first byte, length = size without the zero byte) — zero copy, as in the reference;
 *   DATE (UInt16) / DATETIME (UInt32) -> Uint64, DATE32 (Int32) / DATETIME64 (Int64) -> Int64, each after adding
 *         time_adjustment and casting back to the ClickHouse type (:150-155, :203-206); TIMESTAMP (DateTime64 mapped to
 *         the YT timestamp type) -> Uint64, a negative adjusted value fails the call (:189-195).
 * null_map (nullable): ColumnNullable's byte map; a non-zero byte turns the row into Null (MakeUnversionedNullValue).
 * Composite / decimal / enum / low-cardinality columns are YSON- or string-building paths and stay on the CPU. */
typedef enum ytgpu_ch_type {
    YTGPU_CH_INT8 = 1, YTGPU_CH_INT16 = 2, YTGPU_CH_INT32 = 3, YTGPU_CH_INT64 = 4,
    YTGPU_CH_UINT8 = 5, YTGPU_CH_UINT16 = 6, YTGPU_CH_UINT32 = 7, YTGPU_CH_UINT64 = 8,
    YTGPU_CH_FLOAT32 = 9, YTGPU_CH_FLOAT64 = 10, YTGPU_CH_BOOL = 11, YTGPU_CH_STRING = 12,
    YTGPU_CH_DATE = 13, YTGPU_CH_DATE32 = 14, YTGPU_CH_DATETIME = 15, YTGPU_CH_DATETIME64 = 16, YTGPU_CH_TIMESTAMP = 17
} ytgpu_ch_type;

typedef struct ytgpu_ch_column {
    int32_t type;              /* ytgpu_ch_type */
    int32_t mem;               /* ytgpu_mem of data, offsets, null_map */
    const void* data;          /* row_count fixed-width elements; STRING: the chars */
    const uint64_t* offsets;   /* STRING only: row_count end offsets */
    uint64_t chars_bytes;      /* STRING only */
    const uint8_t* null_map;   /* nullable */
    int64_t time_adjustment;   /* TimezoneAdjustmentSeconds_ (date / time types), normally 0 */
    uint64_t row_count;
} ytgpu_ch_column;

int ytgpu_convert_ch_column_to_values(ytgpu_context* ctx, const ytgpu_ch_column* column, ytgpu_value* out_values, int out_mem,
                                      ytgpu_error* err);

/* ---- string column writer ----
 * One segment of an unversioned string column as TUnversionedStringColumnWriter<String>::DumpSegment emits it
 * (yt/yt/ytlib/table_chunk_format/string_column_writer.cpp:589-636).  Data parts, in writer order:
 *   DirectDense     : bit-packed offsets | null bitmap (1 bit per row) | string bytes of all rows        (:201-229)
 *   DictionaryDense : bit-packed ids (0 = null, else 1-based first-seen id) | bit-packed dictionary offsets | dictionary bytes (:152-199)
 *   DirectRle       : bit-packed run starts | bit-packed offsets | null bitmap (1 bit per run) | string bytes of the runs (:496-537)
 *   DictionaryRle   : bit-packed run starts | bit-packed run ids | bit-packed dictionary offsets | dictionary bytes      (:539-586)
 * Offsets are END offsets stored as zig-zag differences from (i + 1) * expected_length (PrepareDiffFromExpected,
 * yt/yt/core/misc/bit_packed_unsigned_vector.cpp:11-33); DecodeStringPointersAndLengths reads them back. */
typedef struct ytgpu_string_segment {
    uint32_t type;              /* EUnversionedStringSegmentType (table_chunk_format/private.h:32-37):
                                   0 DictionaryRle, 1 DictionaryDense, 2 DirectRle, 3 DirectDense */
    uint32_t row_count;         /* TSegmentMeta::row_count */
    uint64_t chunk_row_count;   /* rows of the chunk up to and including this segment */
    uint64_t data_offset;       /* first byte of the segment's data in out_data (8-byte aligned) */
    uint64_t data_bytes;
    uint64_t part_bytes[4];     /* sizes of the data parts in writer order (0 = absent) */
    uint32_t expected_length;   /* TStringSegmentMeta::expected_length */
    uint32_t offsets_size;      /* TBlobMeta::OffsetsSize */
    uint32_t ids_size;          /* TBlobMeta::IdsSize (dictionary types) */
    uint32_t row_indexes_size;  /* TKeyIndexMeta::RowIndexesSize (RLE types) */
    uint8_t offsets_width, ids_width, row_indexes_width;
    uint8_t direct;             /* TBlobMeta::Direct */
    uint32_t reserved;
} ytgpu_string_segment;

/* Replaces AddValues + DumpSegment of the unversioned String column writer: value i is the lengths[i] bytes at
 * string_heap + starts[i]; null_bytemap (nullable) marks NULL rows (their starts / lengths are ignored).  A segment ends
 * once it holds max_segment_value_count values or more than max_buffer_bytes string bytes (0 = the reference's 32 MB,
 * string_column_writer.cpp:25,:701-703) and is encoded with whichever of the four layouts the reference's size estimate
 * makes smallest (first minimum in enum order, :589-593,:646-676).  Same capacity protocol as
 * ytgpu_encode_integer_column; out_data needs 8-byte alignment in DEVICE memory. */
int ytgpu_encode_string_column(ytgpu_context* ctx, const uint8_t* string_heap, uint64_t string_heap_bytes, const uint64_t* starts,
                               const uint32_t* lengths, const uint8_t* null_bytemap, uint64_t row_count,
                               uint32_t max_segment_value_count, uint64_t max_buffer_bytes, uint64_t chunk_row_offset, int mem,
                               uint8_t* out_data, uint64_t out_capacity, uint64_t* out_data_bytes,
                               ytgpu_string_segment* out_segments, uint32_t segment_capacity, uint32_t* out_segment_count,
                               ytgpu_error* err);

/* String GROUP BY keys: out_ids[i] = index of the FIRST row whose string equals row i's (so equal strings get equal ids and
 * the id of a group names a row that holds its key); NULL rows get id 0 and out_null_bytemap[i] = 1 (nullable output).
 * Feed out_ids (+ the bytemap as a null bitmap) to ytgpu_scan_filter_groupby[_multi] as a UINT64 key column: that is the
 * hashed aggregation over string keys of YT QL (GroupOpHelper with a string group item, cg_routines/registry.cpp:1571-1655:
 * the reference hashes and compares the string bytes per row) and of YQL's BlockCombineHashed over string keys
 * (mkql_block_agg.cpp:1234-1400).  Inputs as for ytgpu_encode_string_column; at most 2^30 rows per call. */
int ytgpu_string_value_ids(ytgpu_context* ctx, const uint8_t* string_heap, uint64_t string_heap_bytes, const uint64_t* starts,
                           const uint32_t* lengths, const uint8_t* null_bytemap, uint64_t row_count, uint64_t* out_ids,
                           uint8_t* out_null_bytemap, int mem, ytgpu_error* err);

/* Replaces the value extraction of the four unversioned string segment readers (string_column_reader.cpp: extractors
 * :39-71,:84-97,:130-143, readers :266-520): for every row of the segment the position of its string — out_start[i] bytes
 * from the segment's first byte, out_length[i] bytes long, so `segment_data` serves as the heap of the resulting values —
 * and out_null_bytemap[i] (nullable; a NULL row gets start 0, length 0).  `segment` (host) carries type, row_count,
 * expected_length, data_bytes and part_bytes; `segment_data` points at the segment's data_bytes bytes (8-byte aligned in
 * DEVICE memory).  Inconsistent sizes -> INVALID_ARGUMENT. */
int ytgpu_decode_string_segment(ytgpu_context* ctx, const ytgpu_string_segment* segment, const uint8_t* segment_data,
                                uint32_t* out_start, uint32_t* out_length, uint8_t* out_null_bytemap, int mem, ytgpu_error* err);

#ifdef __cplusplus
}
#endif
#endif /* YTGPU_H_ */
