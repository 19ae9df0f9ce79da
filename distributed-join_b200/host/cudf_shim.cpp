#include "cudf_shim.hpp"

#include <algorithm>
#include <string>

namespace cudf {

namespace {
void require_fixed_width(table_view const& t, const char* what)
{
  for (auto const& c : t)
    if (!is_fixed_width(c.type()))
      throw std::runtime_error(std::string(what) + ": the B200 build handles fixed-width columns only");
}

__global__ void widen_kernel(const int32_t* in, int64_t* out, int64_t n)
{
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    out[i] = in[i];
}
__global__ void narrow_kernel(const int64_t* in, int32_t* out, int64_t n)
{
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    out[i] = (int32_t)in[i];
}
int grid_for(int64_t n) { return (int)std::max<int64_t>(1, std::min<int64_t>((n + 255) / 256, 148 * 16)); }

// The key column of a wide table as int64, which is what the library hashes and compares: an
// 8-byte key is used in place, a 4-byte key is sign-extended into `scratch` (as widen_to_i64 does).
const int64_t* key_as_i64(column_view const& c, rmm::device_buffer& scratch)
{
  if (size_of(c.type()) == 8) return c.head<int64_t>();
  const int64_t n = c.size();
  scratch         = rmm::device_buffer((size_t)n * 8);
  if (n > 0) widen_kernel<<<grid_for(n), 256>>>(c.head<int32_t>(), (int64_t*)scratch.data(), n);
  CUDA_RT_CALL(cudaGetLastError());
  return (const int64_t*)scratch.data();
}

// Where the library writes an output key column: the column itself when it is 8 bytes wide,
// otherwise `scratch`, narrowed into the column by finish_key once the rows are known.
int64_t* key_out_i64(column& c, int64_t capacity, rmm::device_buffer& scratch)
{
  if (size_of(c.type()) == 8) return c.mutable_view().head<int64_t>();
  scratch = rmm::device_buffer((size_t)capacity * 8);
  return (int64_t*)scratch.data();
}

void finish_key(column& c, int64_t n, rmm::device_buffer const& scratch)
{
  if (size_of(c.type()) == 8 || n == 0) return;
  narrow_kernel<<<grid_for(n), 256>>>((const int64_t*)scratch.data(), c.mutable_view().head<int32_t>(), n);
  CUDA_RT_CALL(cudaGetLastError());
}

// The columns of `t` other than `key`, in table order: input pointers and widths for the _cols ABI.
struct PayloadCols {
  std::vector<const void*> in;
  std::vector<int> bytes;
  std::vector<size_type> index;  // table position of each payload column
};
PayloadCols payload_cols(table_view const& t, size_type key)
{
  PayloadCols p;
  for (size_type c = 0; c < t.num_columns(); c++) {
    if (c == key) continue;
    p.in.push_back(t.column(c).head());
    p.bytes.push_back((int)size_of(t.column(c).type()));
    p.index.push_back(c);
  }
  return p;
}

void require_wide_table(table_view const& t, size_type key, const char* what)
{
  if (key < 0 || key >= t.num_columns())
    throw std::runtime_error(std::string(what) + ": key column index out of range");
  if (t.num_columns() > DJ_MAX_PAYLOAD_COLUMNS + 1)
    throw std::runtime_error(std::string(what) + ": at most " + std::to_string(DJ_MAX_PAYLOAD_COLUMNS + 1) +
                             " columns (key + " + std::to_string(DJ_MAX_PAYLOAD_COLUMNS) + ") are supported");
  require_fixed_width(t, what);
}

// Any other fixed-width table: dj_hash_partition_cols partitions (key, row index) and gathers the
// other columns at their own widths.  Rows land in the same partitions as on the 2..4-column path.
std::pair<std::unique_ptr<table>, std::vector<size_type>> hash_partition_wide(table_view const& input, size_type key,
                                                                              int num_partitions,
                                                                              hash_id hash_function, uint32_t seed)
{
  require_wide_table(input, key, "hash_partition");
  const int64_t n = input.num_rows();
  std::vector<std::unique_ptr<column>> out_cols;
  for (auto const& c : input) out_cols.push_back(make_fixed_width_column(c.type(), (size_type)n));
  PayloadCols pay = payload_cols(input, key);
  std::vector<void*> out_pay;
  for (size_type c : pay.index) out_pay.push_back(out_cols[c]->mutable_view().head());
  rmm::device_buffer key_in, key_out;
  const int64_t* d_key = key_as_i64(input.column(key), key_in);
  int64_t* d_out_key   = key_out_i64(*out_cols[key], n, key_out);
  rmm::device_buffer d_offsets(((size_t)num_partitions + 1) * 8);
  const size_t ws_bytes = dj_hash_partition_cols_workspace_bytes(n, num_partitions);
  rmm::device_buffer ws(ws_bytes);
  DJ_CALL(dj_hash_partition_cols(d_key, pay.in.data(), pay.bytes.data(), (int)pay.in.size(), n, num_partitions, seed,
                                 (int)hash_function, d_out_key, out_pay.data(), (int64_t*)d_offsets.data(), ws.data(),
                                 ws_bytes, nullptr));
  finish_key(*out_cols[key], n, key_out);
  std::vector<int64_t> off64((size_t)num_partitions + 1);
  CUDA_RT_CALL(cudaMemcpyAsync(off64.data(), d_offsets.data(), off64.size() * 8, cudaMemcpyDeviceToHost, nullptr));
  CUDA_RT_CALL(cudaStreamSynchronize(nullptr));
  std::vector<size_type> offsets(off64.begin(), off64.end() - 1);
  return {std::make_unique<table>(std::move(out_cols)), std::move(offsets)};
}

// Tables other than key + payload: dj_inner_join_cols joins (key, row index) and gathers every other
// column.  Output is all left columns ++ all right columns in their positions and types.
std::unique_ptr<table> inner_join_wide(table_view const& left, table_view const& right, size_type lk, size_type rk)
{
  require_wide_table(left, lk, "inner_join");
  require_wide_table(right, rk, "inner_join");
  const int64_t nl = left.num_rows(), nr = right.num_rows();
  const bool build_left = nl <= nr;  // build on the smaller side, as on the 2-column path
  table_view const& B = build_left ? left : right;
  table_view const& P = build_left ? right : left;
  const size_type bk = build_left ? lk : rk, pk = build_left ? rk : lk;
  const size_type b0 = build_left ? 0 : left.num_columns(), p0 = build_left ? left.num_columns() : 0;
  PayloadCols bpay = payload_cols(B, bk), ppay = payload_cols(P, pk);
  rmm::device_buffer bkey_in, pkey_in, d_count(8);
  const int64_t* d_bk = key_as_i64(B.column(bk), bkey_in);
  const int64_t* d_pk = key_as_i64(P.column(pk), pkey_in);
  int64_t capacity = std::max<int64_t>(std::max(nl, nr), 1);
  for (;;) {
    std::vector<std::unique_ptr<column>> cols;
    for (auto const& c : left) cols.push_back(make_fixed_width_column(c.type(), (size_type)capacity));
    for (auto const& c : right) cols.push_back(make_fixed_width_column(c.type(), (size_type)capacity));
    std::vector<void*> bout, pout;
    for (size_type c : bpay.index) bout.push_back(cols[b0 + c]->mutable_view().head());
    for (size_type c : ppay.index) pout.push_back(cols[p0 + c]->mutable_view().head());
    rmm::device_buffer bkey_out, pkey_out;
    int64_t* d_bko = key_out_i64(*cols[b0 + bk], capacity, bkey_out);
    int64_t* d_pko = key_out_i64(*cols[p0 + pk], capacity, pkey_out);
    const size_t ws_bytes = dj_inner_join_cols_workspace_bytes(B.num_rows(), P.num_rows(), capacity);
    rmm::device_buffer ws(ws_bytes);
    DJ_CALL(dj_inner_join_cols(d_bk, bpay.in.data(), bpay.bytes.data(), (int)bpay.in.size(), B.num_rows(), d_pk,
                               ppay.in.data(), ppay.bytes.data(), (int)ppay.in.size(), P.num_rows(), d_bko,
                               bout.data(), d_pko, pout.data(), capacity, (int64_t*)d_count.data(), ws.data(),
                               ws_bytes, nullptr));
    int64_t n_out = 0;
    CUDA_RT_CALL(cudaMemcpyAsync(&n_out, d_count.data(), 8, cudaMemcpyDeviceToHost, nullptr));
    CUDA_RT_CALL(cudaStreamSynchronize(nullptr));
    if (n_out <= capacity) {
      finish_key(*cols[b0 + bk], n_out, bkey_out);
      finish_key(*cols[p0 + pk], n_out, pkey_out);
      for (auto& c : cols) c->set_size((size_type)n_out);
      return std::make_unique<table>(std::move(cols));
    }
    if (n_out > INT32_MAX) throw std::runtime_error("inner_join: result exceeds cudf::size_type rows");
    capacity = n_out;  // exact retry
  }
}
}  // namespace

bool all_i64(table_view const& t)
{
  for (auto const& c : t)
    if (size_of(c.type()) != 8) return false;
  return true;
}

std::unique_ptr<table> widen_to_i64(table_view const& t)
{
  require_fixed_width(t, "widen");
  std::vector<std::unique_ptr<column>> cols;
  const int64_t n = t.num_rows();
  for (auto const& c : t) {
    cols.push_back(make_fixed_width_column(data_type(type_id::INT64), (size_type)n));
    if (n == 0) continue;
    if (size_of(c.type()) == 8)
      CUDA_RT_CALL(cudaMemcpyAsync(cols.back()->mutable_view().head(), c.head(), (size_t)n * 8,
                                   cudaMemcpyDeviceToDevice, nullptr));
    else
      widen_kernel<<<grid_for(n), 256>>>(c.head<int32_t>(), cols.back()->mutable_view().head<int64_t>(), n);
  }
  CUDA_RT_CALL(cudaGetLastError());
  return std::make_unique<table>(std::move(cols));
}

std::unique_ptr<table> narrow_like(table_view const& t, std::vector<data_type> const& types)
{
  if ((size_t)t.num_columns() != types.size()) throw std::runtime_error("narrow_like: column count mismatch");
  std::vector<std::unique_ptr<column>> cols;
  const int64_t n = t.num_rows();
  for (size_type c = 0; c < t.num_columns(); c++) {
    cols.push_back(make_fixed_width_column(types[c], (size_type)n));
    if (n == 0) continue;
    if (size_of(types[c]) == 8)
      CUDA_RT_CALL(cudaMemcpyAsync(cols.back()->mutable_view().head(), t.column(c).head(), (size_t)n * 8,
                                   cudaMemcpyDeviceToDevice, nullptr));
    else
      narrow_kernel<<<grid_for(n), 256>>>(t.column(c).head<int64_t>(), cols.back()->mutable_view().head<int32_t>(), n);
  }
  CUDA_RT_CALL(cudaGetLastError());
  return std::make_unique<table>(std::move(cols));
}

std::pair<std::unique_ptr<table>, std::vector<size_type>> hash_partition(
  table_view const& input, std::vector<size_type> const& columns_to_hash, int num_partitions, hash_id hash_function,
  uint32_t seed)
{
  if (columns_to_hash.size() != 1) throw std::runtime_error("hash_partition: exactly one key column is supported");
  if (input.num_columns() < 2 || input.num_columns() > 4)
    return hash_partition_wide(input, columns_to_hash[0], num_partitions, hash_function, seed);
  require_fixed_width(input, "hash_partition");
  if (!all_i64(input)) {
    std::vector<data_type> types;
    for (auto const& c : input) types.push_back(c.type());
    auto wide   = widen_to_i64(input);
    auto result = hash_partition(wide->view(), columns_to_hash, num_partitions, hash_function, seed);
    return {narrow_like(result.first->view(), types), std::move(result.second)};
  }
  const size_type n   = input.num_rows();
  const size_type key = columns_to_hash[0];

  std::vector<std::unique_ptr<column>> out_cols;
  for (size_type c = 0; c < input.num_columns(); c++)
    out_cols.push_back(make_fixed_width_column(data_type(type_id::INT64), n));
  std::vector<const int64_t*> in_pay;
  std::vector<int64_t*> out_pay;
  for (size_type c = 0; c < input.num_columns(); c++) {
    if (c == key) continue;
    in_pay.push_back(input.column(c).head<int64_t>());
    out_pay.push_back(out_cols[c]->mutable_view().head<int64_t>());
  }
  rmm::device_buffer d_offsets(((size_t)num_partitions + 1) * 8);
  const size_t ws_bytes = dj_hash_partition_workspace_bytes(n, num_partitions);
  rmm::device_buffer ws(ws_bytes);
  DJ_CALL(dj_hash_partition_i64(input.column(key).head<int64_t>(), in_pay.data(), (int)in_pay.size(), n,
                                num_partitions, seed, (int)hash_function,
                                out_cols[key]->mutable_view().head<int64_t>(), out_pay.data(),
                                (int64_t*)d_offsets.data(), ws.data(), ws_bytes, nullptr));
  std::vector<int64_t> off64((size_t)num_partitions + 1);
  CUDA_RT_CALL(cudaMemcpyAsync(off64.data(), d_offsets.data(), off64.size() * 8, cudaMemcpyDeviceToHost, nullptr));
  CUDA_RT_CALL(cudaStreamSynchronize(nullptr));
  // cuDF returns the num_partitions start offsets; callers append num_rows themselves
  std::vector<size_type> offsets(off64.begin(), off64.end() - 1);
  return {std::make_unique<table>(std::move(out_cols)), std::move(offsets)};
}

std::unique_ptr<table> inner_join(table_view const& left, table_view const& right,
                                  std::vector<size_type> const& left_on, std::vector<size_type> const& right_on)
{
  if (left_on.size() != 1 || right_on.size() != 1)
    throw std::runtime_error("inner_join: exactly one key column per side is supported");
  if (left.num_columns() != 2 || right.num_columns() != 2) return inner_join_wide(left, right, left_on[0], right_on[0]);
  require_fixed_width(left, "inner_join");
  require_fixed_width(right, "inner_join");
  if (!all_i64(left) || !all_i64(right)) {
    std::vector<data_type> types;
    for (auto const& c : left) types.push_back(c.type());
    for (auto const& c : right) types.push_back(c.type());
    auto wl = widen_to_i64(left), wr = widen_to_i64(right);
    auto joined = inner_join(wl->view(), wr->view(), left_on, right_on);
    return narrow_like(joined->view(), types);
  }
  const size_type lk = left_on[0], rk = right_on[0];
  const int64_t nl = left.num_rows(), nr = right.num_rows();
  // build on the smaller side; the output stays left columns ++ right columns
  const bool build_left = nl <= nr;
  table_view const& B = build_left ? left : right;
  table_view const& P = build_left ? right : left;
  const size_type bk = build_left ? lk : rk, pk = build_left ? rk : lk;
  const size_t ws_bytes = dj_inner_join_workspace_bytes(B.num_rows(), P.num_rows());
  rmm::device_buffer ws(ws_bytes), d_count(8);
  int64_t capacity = std::max<int64_t>(std::max(nl, nr), 1);
  for (;;) {
    std::vector<std::unique_ptr<column>> cols;
    for (int c = 0; c < 4; c++) cols.push_back(make_fixed_width_column(data_type(type_id::INT64), (size_type)capacity));
    // output column order of the join kernel is (build key, build payload, probe key, probe payload)
    int64_t* o[4];
    for (int c = 0; c < 4; c++) o[c] = cols[c]->mutable_view().head<int64_t>();
    int64_t* bo_k = build_left ? o[lk] : o[2 + rk];
    int64_t* bo_p = build_left ? o[1 - lk] : o[2 + 1 - rk];
    int64_t* po_k = build_left ? o[2 + rk] : o[lk];
    int64_t* po_p = build_left ? o[2 + 1 - rk] : o[1 - lk];
    DJ_CALL(dj_inner_join_i64(B.column(bk).head<int64_t>(), B.column(1 - bk).head<int64_t>(), B.num_rows(),
                              P.column(pk).head<int64_t>(), P.column(1 - pk).head<int64_t>(), P.num_rows(), bo_k,
                              bo_p, po_k, po_p, capacity, (int64_t*)d_count.data(), ws.data(), ws_bytes, nullptr));
    int64_t n_out = 0;
    CUDA_RT_CALL(cudaMemcpyAsync(&n_out, d_count.data(), 8, cudaMemcpyDeviceToHost, nullptr));
    CUDA_RT_CALL(cudaStreamSynchronize(nullptr));
    if (n_out <= capacity) {
      for (auto& c : cols) c->set_size((size_type)n_out);
      return std::make_unique<table>(std::move(cols));
    }
    if (n_out > INT32_MAX) throw std::runtime_error("inner_join: result exceeds cudf::size_type rows");
    capacity = n_out;  // exact retry
  }
}

std::unique_ptr<table> concatenate(std::vector<table_view> const& views)
{
  if (views.empty()) return std::make_unique<table>();
  size_type ncols = 0;
  int64_t rows    = 0;
  for (auto const& v : views) {
    if (v.num_columns() > ncols) ncols = v.num_columns();
    rows += v.num_rows();
  }
  if (rows > INT32_MAX) throw std::runtime_error("concatenate: result exceeds cudf::size_type rows");
  std::vector<std::unique_ptr<column>> cols;
  for (size_type c = 0; c < ncols; c++) {
    data_type t(type_id::INT64);
    for (auto const& v : views)
      if (v.num_columns() == ncols) t = v.column(c).type();
    cols.push_back(make_fixed_width_column(t, (size_type)rows));
    int64_t at      = 0;
    const size_t es = size_of(t);
    for (auto const& v : views) {
      if (v.num_columns() != ncols || v.num_rows() == 0) continue;  // empty batch results have no columns
      CUDA_RT_CALL(cudaMemcpyAsync(cols.back()->mutable_view().head<char>() + at * es, v.column(c).head<char>(),
                                   (size_t)v.num_rows() * es, cudaMemcpyDeviceToDevice, nullptr));
      at += v.num_rows();
    }
  }
  CUDA_RT_CALL(cudaStreamSynchronize(nullptr));
  return std::make_unique<table>(std::move(cols));
}

}  // namespace cudf
