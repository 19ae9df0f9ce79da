/*
 * dj_b200.h -- C ABI of libdj_b200.so, the B200-native (sm_100a) replacement for the device
 * side of rapidsai/distributed-join's hot path:
 *
 *     hash-partition  ->  all-to-all  ->  local hash join
 *
 * Every entry point is `extern "C"`, takes plain pointers and sizes (no torch / cuDF / RMM
 * types), is stream-ordered on the cudaStream_t passed as `void* stream`, and returns 0 on
 * success or a non-zero code (dj_last_error() gives the message).  Device pointers are
 * prefixed d_, host pointers h_.  Row counts are int64_t (the reference's cudf::size_type
 * is int32; config 5 exceeds it).
 *
 * For each function the comment names the reference interface it replaces (file:line in
 * rapidsai/distributed-join @ 26e84fee).  The C++ mirror of the reference API that calls
 * this ABI lives in distributed-join_b200/host/; INTEGRATION.md shows the binding a
 * reference maintainer would add.
 */
#ifndef DJ_B200_H
#define DJ_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif
#if defined(DJ_BUILDING) && defined(__GNUC__)
#pragma GCC visibility push(default) /* the library hides everything but this ABI */
#endif

#define DJ_VERSION 100

/* mirrors cudf::hash_id as used by the reference (src/shuffle_on.hpp:49-50,
 * test/test_shuffle_on.cpp:66) */
enum { DJ_HASH_IDENTITY = 0, DJ_HASH_MURMUR3 = 1 };

/* error codes */
enum {
  DJ_OK            = 0,
  DJ_ERR_CUDA      = 1, /* a CUDA runtime call or kernel launch failed              */
  DJ_ERR_ARG       = 2, /* invalid argument (the reference throws std::runtime_error) */
  DJ_ERR_WORKSPACE = 3, /* workspace too small                                        */
  DJ_ERR_NCCL      = 4, /* an NCCL call failed                                        */
  DJ_ERR_OVERFLOW  = 5  /* output capacity too small (count is still exact)           */
};

int dj_version(void);
const char* dj_last_error(void);
/* number of kernels this library has launched in this process (bench.py's gpu_launches) */
int64_t dj_kernel_launch_count(void);

/* Per-kernel device timing for bench.py's roofline: when enabled, every launch of the four
 * kernel categories is bracketed by CUDA events on its own stream.  dj_profile_read
 * synchronises those events, returns the summed milliseconds and launch counts per category
 * (hist, scatter, join, other) and clears the record. */
enum { DJ_PROF_HIST = 0, DJ_PROF_SCATTER = 1, DJ_PROF_JOIN = 2, DJ_PROF_OTHER = 3, DJ_PROF_NCAT = 4 };
int dj_profile_enable(int on);
int dj_profile_read(double* h_ms4, int64_t* h_launches4);

/* ------------------------------------------------------------------------------------
 * Hashing.  partition id = (murmur3_x86_32(key bytes, seed) + 0x9e3779b9) % nparts,
 * restating cudf::hash_partition's row hash for one int64 key column
 * (call sites src/distributed_join.cpp:213-225, src/shuffle_on.cpp:59-60).
 */
int dj_partition_ids_i64(const int64_t* d_keys, int64_t nrows, uint32_t seed, int hash_id,
                         int nparts, int32_t* d_out_ids, void* stream);

/* ------------------------------------------------------------------------------------
 * dj_hash_partition_i64 -- replaces cudf::hash_partition(table, {0}, nparts, hash, seed)
 * (src/distributed_join.cpp:213-225, src/shuffle_on.cpp:59-60): reorders the key column
 * and `npayload` (1..3) int64 payload columns so that partition p is the contiguous row
 * range [d_offsets[p], d_offsets[p+1]) of the outputs.  Order inside a partition is
 * unspecified (as in cuDF).  d_offsets has nparts+1 entries (the reference appends
 * num_rows itself, src/distributed_join.cpp:232-233).  2 <= nparts <= 1024.
 * h_payload_cols / h_out_payload_cols are HOST arrays of device pointers.
 */
size_t dj_hash_partition_workspace_bytes(int64_t nrows, int nparts);
int dj_hash_partition_i64(const int64_t* d_key, const int64_t* const* h_payload_cols, int npayload,
                          int64_t nrows, int nparts, uint32_t seed, int hash_id,
                          int64_t* d_out_key, int64_t* const* h_out_payload_cols,
                          int64_t* d_offsets, void* d_workspace, size_t workspace_bytes,
                          void* stream);

/* ------------------------------------------------------------------------------------
 * dj_inner_join_i64 -- replaces cudf::inner_join(left, right, {0}, {0}) as called by
 * local_join_helper (src/distributed_join.cpp:71-83) for int64 key + int64 payload tables.
 * Multimap semantics (duplicate build keys produce all pairs).  Output columns are
 * (build key, build payload, probe key, probe payload); the C++ layer maps them to
 * left ++ right.  Writes at most out_capacity rows; *d_out_count always receives the exact
 * cardinality, so a caller that under-allocated can retry.  Either side empty -> 0 rows
 * (src/distributed_join.cpp:76-82).  No host synchronisation.
 */
size_t dj_inner_join_workspace_bytes(int64_t nbuild, int64_t nprobe);
int dj_inner_join_i64(const int64_t* d_build_key, const int64_t* d_build_payload, int64_t nbuild,
                      const int64_t* d_probe_key, const int64_t* d_probe_payload, int64_t nprobe,
                      int64_t* d_out_build_key, int64_t* d_out_build_payload,
                      int64_t* d_out_probe_key, int64_t* d_out_probe_payload,
                      int64_t out_capacity, int64_t* d_out_count,
                      void* d_workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------
 * Wide tables: an int64 key plus 0..DJ_MAX_PAYLOAD_COLUMNS fixed-width payload columns per
 * side, each 4 or 8 bytes wide (h_elem_bytes[c]).  Columns are moved bitwise, so any 4- or
 * 8-byte type works (int32, float, timestamps, double ...).  Both calls run the pipelines
 * above on (key, row index) and then gather every payload column through the resulting row
 * indices at its own width (late materialization), so the partition and join kernels move
 * 16 bytes per row whatever the table's width.  h_cols / h_out_cols are HOST arrays of
 * device pointers.  Arguments are checked before any CUDA call: a column count out of range,
 * a width other than 4 or 8, or a null column / key pointer where rows are read or written
 * returns DJ_ERR_ARG; a workspace below the matching *_workspace_bytes query returns
 * DJ_ERR_WORKSPACE.  The workspace queries need no GPU.
 */
#define DJ_MAX_PAYLOAD_COLUMNS 15

/* dj_hash_partition_cols -- cudf::hash_partition(table, {key}, nparts, hash, seed) for a wide
 * table, with the contract of dj_hash_partition_i64: d_offsets (nparts+1 entries) is
 * bit-identical to dj_hash_partition_i64's for the same keys, seed and nparts, so wide and
 * 2-column tables partitioned with the same seed co-locate; order inside a partition is
 * unspecified; every output row is one intact input row.  1 <= nparts <= 1024. */
size_t dj_hash_partition_cols_workspace_bytes(int64_t nrows, int nparts);
int dj_hash_partition_cols(const int64_t* d_key, const void* const* h_cols, const int* h_elem_bytes,
                           int ncols, int64_t nrows, int nparts, uint32_t seed, int hash_id,
                           int64_t* d_out_key, void* const* h_out_cols, int64_t* d_offsets,
                           void* d_workspace, size_t workspace_bytes, void* stream);

/* dj_inner_join_cols -- cudf::inner_join(left, right, {key}, {key}) for wide tables, with the
 * contract of dj_inner_join_i64: multimap semantics; outputs are (build key, build columns,
 * probe key, probe columns), each column at its input's width; at most out_capacity rows are
 * written and *d_out_count always receives the exact cardinality, so a caller that
 * under-allocated can retry with a larger output (and workspace: it grows with out_capacity);
 * either side empty -> 0 rows.  No host synchronisation: the payload gathers read the count
 * on the device. */
size_t dj_inner_join_cols_workspace_bytes(int64_t nbuild, int64_t nprobe, int64_t out_capacity);
int dj_inner_join_cols(const int64_t* d_build_key, const void* const* h_build_cols,
                       const int* h_build_elem_bytes, int nbuild_cols, int64_t nbuild,
                       const int64_t* d_probe_key, const void* const* h_probe_cols,
                       const int* h_probe_elem_bytes, int nprobe_cols, int64_t nprobe,
                       int64_t* d_out_build_key, void* const* h_out_build_cols,
                       int64_t* d_out_probe_key, void* const* h_out_probe_cols,
                       int64_t out_capacity, int64_t* d_out_count,
                       void* d_workspace, size_t workspace_bytes, void* stream);

/* ------------------------------------------------------------------------------------
 * Input generator -- replaces generate_input_tables / generate_tables_distributed
 * (generate_dataset/generate_dataset.cuh:163-260, src/generate_table.cuh:155-272) with a
 * counter-based restatement (Philox4x32-10 + Feistel permutation) shared bit-for-bit with
 * oracle/dj_oracle.c.  Generates rows [row_begin, row_begin+count) of source rank `src`'s
 * local build (which=0) / probe (which=1) table including the rank offsets
 * (src/generate_table.cuh:192-202).  d_bitmap ((rand_max+1+31)/32 words) is only used when
 * unique_build_keys == 0: fill it with dj_generate_build_bitmap first.
 */
typedef struct {
  int64_t nb;       /* build rows per source rank                                            */
  int64_t np;       /* probe rows per source rank                                            */
  int64_t rand_max; /* per-rank key range [0, rand_max] (benchmark/distributed_join.cu:187)  */
  double selectivity;
  uint64_t seed;    /* reference: 1234 (generate_dataset.cuh:44)                             */
  int32_t unique_build_keys;
  int32_t pad;
} dj_gen_params;

int dj_generate_build_bitmap(const dj_gen_params* h_params, int src_rank, uint32_t* d_bitmap,
                             void* stream);
int dj_generate_rows_i64(const dj_gen_params* h_params, int which, int src_rank, int64_t row_begin,
                         int64_t count, const uint32_t* d_bitmap, int64_t* d_keys,
                         int64_t* d_payload, void* stream);

/* Order-independent 128-bit checksum of a 4-column int64 row multiset (verification helper,
 * the role of the reference tests' verify_correctness kernels,
 * test/compare_against_analytical.cu:44-54).  d_out2[0..1] must be zeroed by the caller;
 * results accumulate so that per-rank tables can be summed. */
int dj_multiset_checksum4(const int64_t* d_c0, const int64_t* d_c1, const int64_t* d_c2,
                          const int64_t* d_c3, int64_t nrows, uint64_t* d_out2, void* stream);

/* ------------------------------------------------------------------------------------
 * Communication -- replaces NCCLCommunicator (src/communicator.cpp:799-875) and the table
 * all-to-all (src/all_to_all_comm.cpp:126-189,307-356).  No MPI: the 128-byte ncclUniqueId
 * is produced by dj_comm_unique_id on rank 0 and handed to the other ranks by the launcher
 * (torch.distributed / file / env).
 */
typedef struct dj_comm dj_comm_t;

int dj_comm_unique_id(void* h_id128);
int dj_comm_create(int rank, int size, const void* h_id128, dj_comm_t** out);
int dj_comm_destroy(dj_comm_t* comm);
/* Collective.  Closes every rank's CUDA IPC mappings of the peers' join workspaces; call it on all
 * ranks before freeing or reallocating a workspace that a distributed join has used. */
int dj_comm_release_workspace(dj_comm_t* comm);
/* The underlying ncclComm_t (as void*; NULL for a single-rank communicator): what
 * NCCLCommunicator::nccl_comm exposes in the reference (src/communicator.hpp:346-347). */
void* dj_comm_nccl_handle(dj_comm_t* comm);
int dj_comm_rank(const dj_comm_t* comm);
int dj_comm_size(const dj_comm_t* comm);

/* communicate_sizes (src/all_to_all_comm.cpp:54-111) without MPI: all-gathers each rank's
 * `n` int64 values over NCCL; h_all receives size*n values (blocking, tiny). */
int dj_comm_allgather_i64(dj_comm_t* comm, const int64_t* h_mine, int n, int64_t* h_all,
                          void* stream);
int dj_comm_barrier(dj_comm_t* comm, void* stream);

/* One grouped ncclSend/ncclRecv exchange for `ncols` columns: column c sends elements
 * [h_send_offsets[i], h_send_offsets[i+1]) to group member i and receives into
 * [h_recv_offsets[i], h_recv_offsets[i+1]) (element size h_elem_sizes[c]).  group_ranks
 * maps group index -> communicator rank (CommunicationGroup::get_global_rank,
 * src/all_to_all_comm.hpp:102).  With include_self == 0 the self partition is skipped
 * (all_to_all_comm(..., include_current_rank=false)); with 1 it is copied device-to-device.
 * Asynchronous on `stream`; no staging copies (the reference's 2 extra D2D copies,
 * src/communicator.cpp:831-832,855-859, are gone). */
int dj_all_to_all(dj_comm_t* comm, int group_size, const int* h_group_ranks, int self_idx,
                  const void* const* h_send_cols, void* const* h_recv_cols,
                  const int64_t* h_send_offsets, const int64_t* h_recv_offsets,
                  const int* h_elem_sizes, int ncols, int include_self, void* stream);

/* raw point-to-point pieces for the Communicator mirror (start/send/recv/stop) */
int dj_comm_group_start(dj_comm_t* comm);
int dj_comm_group_end(dj_comm_t* comm);
int dj_comm_send(dj_comm_t* comm, const void* d_buf, int64_t nbytes, int dest, void* stream);
int dj_comm_recv(dj_comm_t* comm, void* d_buf, int64_t nbytes, int source, void* stream);

/* ------------------------------------------------------------------------------------
 * dj_distributed_inner_join_i64 -- the whole hot path of distributed_inner_join
 * (src/distributed_join.cpp:134-340) for int64 key + int64 payload tables on one NVSwitch
 * box: hash-partition both tables into size*odf buckets (seed 12345678, :211), exchange
 * batch by batch, join each batch locally, results appended into one output (no
 * cudf::concatenate).  Collective over `comm` (NULL or size 1: local join only, :186-199).
 * Output columns are left ++ right: (left key, left payload, right key, right payload).
 * *h_out_count receives this rank's cardinality (the call synchronises the stream once at
 * the end to return it).  If it exceeds out_capacity on ANY rank, every rank returns
 * DJ_ERR_OVERFLOW (the verdict is all-gathered) and the outputs hold the first out_capacity
 * rows; *h_out_count is still exact, so callers can retry together with a larger output.
 */
typedef struct {
  int over_decom_factor; /* >= 1 (src/distributed_join.hpp:72)              */
  int report_timing;     /* print the reference's per-stage lines to stdout */
  double t_partition_ms, t_comm_ms, t_join_ms; /* filled when report_timing */
  int64_t bytes_sent;    /* bytes this rank sent over NVLink                 */
  int64_t workspace_needed; /* out: with DJ_ERR_WORKSPACE, the bytes THIS rank needs (every rank
                               returns the error together, so callers can grow and retry)      */
  int measure_exchange;  /* in: time this rank's NVLink pushes with CUDA events                */
  int pad_;
  double t_exchange_ms[2]; /* out (measure_exchange): per table, from its first push starting to
                              its last push complete (over all peer streams)                   */
  double t_exchange_total_ms; /* out: first push of the left table -> last push of the right     */
} dj_join_options;

size_t dj_distributed_inner_join_workspace_bytes(int64_t nleft, int64_t nright, int world,
                                                 int over_decom_factor);
int dj_distributed_inner_join_i64(dj_comm_t* comm,
                                  const int64_t* d_left_key, const int64_t* d_left_payload,
                                  int64_t nleft,
                                  const int64_t* d_right_key, const int64_t* d_right_payload,
                                  int64_t nright,
                                  int64_t* d_out_lk, int64_t* d_out_lp, int64_t* d_out_rk,
                                  int64_t* d_out_rp, int64_t out_capacity, int64_t* h_out_count,
                                  dj_join_options* opts, void* d_workspace,
                                  size_t workspace_bytes, void* stream);

/* Same join with HOST input/output buffers (pinned recommended): the end-to-end entry
 * bench.py times.  Copies inputs host->device, runs the device path above, copies the
 * result columns device->host.  Device memory is taken from d_workspace. */
size_t dj_distributed_inner_join_host_workspace_bytes(int64_t nleft, int64_t nright,
                                                      int64_t out_capacity, int world,
                                                      int over_decom_factor);
int dj_distributed_inner_join_i64_host(dj_comm_t* comm,
                                       const int64_t* h_left_key, const int64_t* h_left_payload,
                                       int64_t nleft,
                                       const int64_t* h_right_key, const int64_t* h_right_payload,
                                       int64_t nright,
                                       int64_t* h_out_lk, int64_t* h_out_lp, int64_t* h_out_rk,
                                       int64_t* h_out_rp, int64_t out_capacity,
                                       int64_t* h_out_count, dj_join_options* opts,
                                       void* d_workspace, size_t workspace_bytes, void* stream);

#if defined(DJ_BUILDING) && defined(__GNUC__)
#pragma GCC visibility pop
#endif
#ifdef __cplusplus
}
#endif
#endif /* DJ_B200_H */
