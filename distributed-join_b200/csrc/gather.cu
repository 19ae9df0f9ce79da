// gather.cu -- wide tables by late materialization: dj_hash_partition_cols and dj_inner_join_cols.
//
// The partition and join pipelines move 16-byte (key, payload) rows (dj_internal.h: Row).  A wide
// table runs them unchanged on (key, row index): an iota takes the payload slot, so what comes out
// is a permutation (partition) or a pair of index columns (join).  One gather per side then pulls
// every payload column through those indices at its own width (4 or 8 bytes).
#include <algorithm>

#include "dj_device.cuh"
#include "dj_internal.h"

namespace dj {
namespace {

constexpr int kGatherThreads = 256;
constexpr int kGatherRows    = 2;  // rows per thread and step: 2 * 15 loads in flight per thread

// Kernel argument of one gather (one side, all its columns).
struct GatherArgs {
  const void* in[DJ_MAX_PAYLOAD_COLUMNS];
  void* out[DJ_MAX_PAYLOAD_COLUMNS];
  int bytes[DJ_MAX_PAYLOAD_COLUMNS];  // 4 or 8
  int ncols;
  const int64_t* idx;      // [capacity] source row of every output row
  const int64_t* d_count;  // rows to gather, read on the device (nullptr: capacity)
  int64_t capacity;        // the output columns' length: the count is clamped to it
};

__global__ void __launch_bounds__(kGatherThreads) iota_kernel(int64_t* out, int64_t n)
{
  for (int64_t i = blockIdx.x * (int64_t)kGatherThreads + threadIdx.x; i < n;
       i += (int64_t)gridDim.x * kGatherThreads)
    out[i] = i;
}

// out_c[i] = in_c[idx[i]] for every column c and i < min(*d_count, capacity).  Each thread reads
// its indices once (coalesced), then issues every column's random loads before the first store, so
// up to kGatherRows * ncols reads are in flight per thread; stores are coalesced per column.
__global__ void __launch_bounds__(kGatherThreads) gather_kernel(const __grid_constant__ GatherArgs a)
{
  int64_t n = a.capacity;
  if (a.d_count) n = min(n, *a.d_count);
  const int64_t step = (int64_t)gridDim.x * kGatherThreads * kGatherRows;
  for (int64_t base = blockIdx.x * (int64_t)kGatherThreads * kGatherRows + threadIdx.x; base < n; base += step) {
    int64_t src[kGatherRows];
#pragma unroll
    for (int r = 0; r < kGatherRows; r++) {
      const int64_t row = base + (int64_t)r * kGatherThreads;
      src[r]            = row < n ? __ldg(a.idx + row) : -1;
    }
    uint64_t v[DJ_MAX_PAYLOAD_COLUMNS][kGatherRows];
#pragma unroll
    for (int c = 0; c < DJ_MAX_PAYLOAD_COLUMNS; c++) {
      if (c >= a.ncols) break;
#pragma unroll
      for (int r = 0; r < kGatherRows; r++) {
        if (src[r] < 0) continue;
        v[c][r] = a.bytes[c] == 8 ? __ldg(static_cast<const unsigned long long*>(a.in[c]) + src[r])
                                  : __ldg(static_cast<const unsigned int*>(a.in[c]) + src[r]);
      }
    }
#pragma unroll
    for (int c = 0; c < DJ_MAX_PAYLOAD_COLUMNS; c++) {
      if (c >= a.ncols) break;
#pragma unroll
      for (int r = 0; r < kGatherRows; r++) {
        if (src[r] < 0) continue;
        const int64_t row = base + (int64_t)r * kGatherThreads;
        if (a.bytes[c] == 8)
          static_cast<unsigned long long*>(a.out[c])[row] = v[c][r];
        else
          static_cast<unsigned int*>(a.out[c])[row] = (unsigned int)v[c][r];
      }
    }
  }
}

int grid_for_rows(int64_t n, int64_t rows_per_block)
{
  const int64_t blocks = (n + rows_per_block - 1) / rows_per_block;
  return (int)std::max<int64_t>(1, std::min<int64_t>(blocks, (int64_t)sm_count() * 16));
}

int launch_iota(int64_t* out, int64_t n, cudaStream_t stream)
{
  if (n <= 0) return DJ_OK;
  ProfScope prof(DJ_PROF_OTHER, stream);
  iota_kernel<<<grid_for_rows(n, kGatherThreads), kGatherThreads, 0, stream>>>(out, n);
  DJ_LAUNCH_CHECK();
  return DJ_OK;
}

int launch_gather(const void* const* in, void* const* out, const int* bytes, int ncols, const int64_t* idx,
                  const int64_t* d_count, int64_t capacity, cudaStream_t stream)
{
  if (ncols == 0 || capacity <= 0) return DJ_OK;
  GatherArgs a{};
  for (int c = 0; c < ncols; c++) {
    a.in[c]    = in[c];
    a.out[c]   = out[c];
    a.bytes[c] = bytes[c];
  }
  a.ncols    = ncols;
  a.idx      = idx;
  a.d_count  = d_count;
  a.capacity = capacity;
  ProfScope prof(DJ_PROF_OTHER, stream);
  gather_kernel<<<grid_for_rows(capacity, (int64_t)kGatherThreads * kGatherRows), kGatherThreads, 0, stream>>>(a);
  DJ_LAUNCH_CHECK();
  return DJ_OK;
}

// Host-side checks of one side's column list: 0..DJ_MAX_PAYLOAD_COLUMNS columns, each 4 or 8 bytes,
// and no null column where `rows` > 0 rows are read or written.
int check_cols(const char* what, const char* side, const void* const* cols, const int* bytes, int ncols,
               int64_t rows)
{
  DJ_REQUIRE(ncols >= 0 && ncols <= DJ_MAX_PAYLOAD_COLUMNS, "%s: %d %s columns (supported: 0..%d)", what, ncols,
             side, DJ_MAX_PAYLOAD_COLUMNS);
  if (ncols == 0) return DJ_OK;
  DJ_REQUIRE(cols && bytes, "%s: %s column or width array missing", what, side);
  for (int c = 0; c < ncols; c++) {
    DJ_REQUIRE(bytes[c] == 4 || bytes[c] == 8, "%s: %s column %d is %d bytes wide (supported: 4 or 8)", what, side, c,
               bytes[c]);
    DJ_REQUIRE(rows == 0 || cols[c], "%s: %s column %d is null", what, side, c);
  }
  return DJ_OK;
}

size_t rows_bytes(int64_t n) { return align_up((size_t)std::max<int64_t>(n, 0) * sizeof(int64_t), 256) + 256; }

}  // namespace
}  // namespace dj

using namespace dj;

#define DJ_TRY(expr)           \
  do {                         \
    const int _rc = (expr);    \
    if (_rc) return _rc;       \
  } while (0)

extern "C" size_t dj_hash_partition_cols_workspace_bytes(int64_t nrows, int nparts)
{
  if (nparts < 1) nparts = 1;
  // iota + permutation, then the partition pass's own scratch
  return 2 * rows_bytes(nrows) + pass_workspace_bytes(1, nparts) + 4096;
}

extern "C" int dj_hash_partition_cols(const int64_t* d_key, const void* const* h_cols, const int* h_elem_bytes,
                                      int ncols, int64_t nrows, int nparts, uint32_t seed, int hash_id,
                                      int64_t* d_out_key, void* const* h_out_cols, int64_t* d_offsets,
                                      void* d_workspace, size_t workspace_bytes, void* stream)
{
  DJ_REQUIRE(nparts >= 1 && nparts <= kMaxFanout, "hash_partition_cols: nparts %d not in [1, %d]", nparts,
             kMaxFanout);
  DJ_REQUIRE(hash_id == DJ_HASH_MURMUR3 || hash_id == DJ_HASH_IDENTITY, "hash_partition_cols: bad hash id");
  DJ_REQUIRE(nrows >= 0 && d_offsets && d_workspace, "hash_partition_cols: bad argument");
  DJ_REQUIRE(nrows == 0 || (d_key && d_out_key), "hash_partition_cols: key column is null");
  DJ_TRY(check_cols("hash_partition_cols", "input", h_cols, h_elem_bytes, ncols, nrows));
  DJ_TRY(check_cols("hash_partition_cols", "output", (const void* const*)h_out_cols, h_elem_bytes, ncols, nrows));
  const size_t need = dj_hash_partition_cols_workspace_bytes(nrows, nparts);
  if (workspace_bytes < need) {
    set_error("hash_partition_cols: workspace of %zu bytes, %zu needed", workspace_bytes, need);
    return DJ_ERR_WORKSPACE;
  }
  cudaStream_t st = (cudaStream_t)stream;
  Arena arena(d_workspace, workspace_bytes);
  int64_t* iota = arena.take<int64_t>((size_t)nrows);
  int64_t* perm = arena.take<int64_t>((size_t)nrows);
  char* pass_ws = arena.take<char>(pass_workspace_bytes(1, nparts));
  if (!iota || !perm || !pass_ws) {
    set_error("hash_partition_cols: workspace too small");
    return DJ_ERR_WORKSPACE;
  }
  DJ_TRY(launch_iota(iota, nrows, st));
  // the same pass dj_hash_partition_i64 runs with one payload column: identical offsets
  PassDesc desc{0, seed, hash_id, 0, nparts, 1, 1};
  PassBuffers buf{};
  buf.in_key       = d_key;
  buf.in_pay[0]    = iota;
  buf.out_key      = d_out_key;
  buf.out_pay[0]   = perm;
  buf.nrows        = nrows;
  buf.d_parent_off = nullptr;
  buf.d_child_off  = d_offsets;
  DJ_TRY(run_partition_pass(desc, buf, pass_ws, workspace_bytes - (size_t)(pass_ws - (char*)d_workspace), st));
  // d_offsets[nparts] == nrows: the gather reads its count from there like the join's
  return launch_gather(h_cols, h_out_cols, h_elem_bytes, ncols, perm, d_offsets + nparts, nrows, st);
}

extern "C" size_t dj_inner_join_cols_workspace_bytes(int64_t nbuild, int64_t nprobe, int64_t out_capacity)
{
  // the key-only join's scratch, one iota shared by both sides, two index columns of out_capacity rows
  return dj_inner_join_workspace_bytes(nbuild, nprobe) + rows_bytes(std::max(nbuild, nprobe)) +
         2 * rows_bytes(out_capacity) + 4096;
}

extern "C" int dj_inner_join_cols(const int64_t* d_build_key, const void* const* h_build_cols,
                                  const int* h_build_elem_bytes, int nbuild_cols, int64_t nbuild,
                                  const int64_t* d_probe_key, const void* const* h_probe_cols,
                                  const int* h_probe_elem_bytes, int nprobe_cols, int64_t nprobe,
                                  int64_t* d_out_build_key, void* const* h_out_build_cols,
                                  int64_t* d_out_probe_key, void* const* h_out_probe_cols,
                                  int64_t out_capacity, int64_t* d_out_count, void* d_workspace,
                                  size_t workspace_bytes, void* stream)
{
  const char* what = "inner_join_cols";
  DJ_REQUIRE(nbuild >= 0 && nprobe >= 0 && out_capacity >= 0 && d_out_count, "%s: bad argument", what);
  DJ_REQUIRE(nbuild == 0 || d_build_key, "%s: build key column is null", what);
  DJ_REQUIRE(nprobe == 0 || d_probe_key, "%s: probe key column is null", what);
  DJ_REQUIRE(out_capacity == 0 || (d_out_build_key && d_out_probe_key), "%s: output key column is null", what);
  DJ_TRY(check_cols(what, "build", h_build_cols, h_build_elem_bytes, nbuild_cols, nbuild));
  DJ_TRY(check_cols(what, "probe", h_probe_cols, h_probe_elem_bytes, nprobe_cols, nprobe));
  DJ_TRY(check_cols(what, "build output", (const void* const*)h_out_build_cols, h_build_elem_bytes, nbuild_cols,
                    out_capacity));
  DJ_TRY(check_cols(what, "probe output", (const void* const*)h_out_probe_cols, h_probe_elem_bytes, nprobe_cols,
                    out_capacity));
  const size_t need = dj_inner_join_cols_workspace_bytes(nbuild, nprobe, out_capacity);
  if (workspace_bytes < need) {
    set_error("%s: workspace of %zu bytes, %zu needed", what, workspace_bytes, need);
    return DJ_ERR_WORKSPACE;
  }
  DJ_REQUIRE(d_workspace, "%s: workspace missing", what);
  cudaStream_t st = (cudaStream_t)stream;
  DJ_CUDA_TRY(cudaMemsetAsync(d_out_count, 0, sizeof(int64_t), st));
  if (nbuild == 0 || nprobe == 0) return DJ_OK;
  Arena arena(d_workspace, workspace_bytes);
  int64_t* build_idx = arena.take<int64_t>((size_t)out_capacity);
  int64_t* probe_idx = arena.take<int64_t>((size_t)out_capacity);
  int64_t* iota      = arena.take<int64_t>((size_t)std::max(nbuild, nprobe));
  if (!build_idx || !probe_idx || !iota) {
    set_error("%s: workspace too small", what);
    return DJ_ERR_WORKSPACE;
  }
  DJ_TRY(launch_iota(iota, std::max(nbuild, nprobe), st));
  int64_t* out[4] = {d_out_build_key, build_idx, d_out_probe_key, probe_idx};
  DJ_TRY(local_join(d_build_key, iota, nbuild, d_probe_key, iota, nprobe, out, out_capacity, d_out_count, false,
                    arena, st));
  // the count stays on the device: the gathers read it and clamp it to out_capacity
  DJ_TRY(launch_gather(h_build_cols, h_out_build_cols, h_build_elem_bytes, nbuild_cols, build_idx, d_out_count,
                       out_capacity, st));
  return launch_gather(h_probe_cols, h_out_probe_cols, h_probe_elem_bytes, nprobe_cols, probe_idx, d_out_count,
                       out_capacity, st);
}
