// cudf_shim.hpp -- the small slice of the cuDF / RMM vocabulary that the reference's public
// API and drivers are written against (SURVEY.md App. C), implemented over plain CUDA memory and
// the dj_b200 C ABI.  Only what the hot path touches exists: fixed-width columns, non-owning
// views, tables, hash_partition / inner_join / concatenate for 4- and 8-byte columns.
//
// This is what lets benchmark/distributed_join.cu keep its source shape
//   (cudf::table_view, std::unique_ptr<cudf::table>, cudf::hash_id::HASH_MURMUR3, rmm pool ...)
// while every device byte is moved by libdj_b200.so.
#pragma once

#include <cuda_runtime.h>

#include <cstddef>
#include <cstdint>
#include <memory>
#include <stdexcept>
#include <utility>
#include <vector>

#include "../../include/dj_b200.h"
#include "error.hpp"

// ------------------------------------------------------------------------------------ rmm
namespace rmm {
namespace mr {

// Stream-ordered device memory (cudaMallocAsync).  The reference creates one RMM pool of
// free/284*256 bytes up front (src/setup.cpp:64-74); the CUDA async pool with an unlimited
// release threshold gives the same "allocate once, reuse" behaviour without carving it by hand.
class device_memory_resource {
 public:
  virtual ~device_memory_resource() = default;
  virtual void* allocate(std::size_t bytes, cudaStream_t stream = nullptr)
  {
    void* p = nullptr;
    if (bytes == 0) return p;
    CUDA_RT_CALL(cudaMallocAsync(&p, bytes, stream));
    return p;
  }
  virtual void deallocate(void* p, std::size_t, cudaStream_t stream = nullptr)
  {
    if (p) CUDA_RT_CALL(cudaFreeAsync(p, stream));
  }
};

template <typename Upstream>
class pool_memory_resource : public device_memory_resource {
 public:
  pool_memory_resource(Upstream* upstream, std::size_t initial_size, std::size_t /*max_size*/)
    : upstream_(upstream)
  {
    int dev = 0;
    CUDA_RT_CALL(cudaGetDevice(&dev));
    cudaMemPool_t pool;
    CUDA_RT_CALL(cudaDeviceGetDefaultMemPool(&pool, dev));
    unsigned long long keep = ~0ull;  // never trim: behaves like a grown-once pool
    CUDA_RT_CALL(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep));
    initial_ = initial_size;
  }
  Upstream* get_upstream() const { return upstream_; }
  std::size_t initial_size() const { return initial_; }

 private:
  Upstream* upstream_;
  std::size_t initial_ = 0;
};

inline device_memory_resource*& current_resource_slot()
{
  static device_memory_resource default_mr;
  static thread_local device_memory_resource* cur = &default_mr;
  return cur;
}
inline device_memory_resource* get_current_device_resource() { return current_resource_slot(); }
inline device_memory_resource* set_current_device_resource(device_memory_resource* mr)
{
  auto* old               = current_resource_slot();
  current_resource_slot() = mr;
  return old;
}

}  // namespace mr

class device_buffer {
 public:
  device_buffer() = default;
  explicit device_buffer(std::size_t bytes, cudaStream_t stream = nullptr)
    : size_(bytes), stream_(stream)
  {
    data_ = mr::get_current_device_resource()->allocate(bytes, stream);
  }
  device_buffer(device_buffer&& o) noexcept { *this = std::move(o); }
  device_buffer& operator=(device_buffer&& o) noexcept
  {
    release();
    data_   = o.data_;
    size_   = o.size_;
    stream_ = o.stream_;
    o.data_ = nullptr;
    o.size_ = 0;
    return *this;
  }
  device_buffer(const device_buffer&) = delete;
  device_buffer& operator=(const device_buffer&) = delete;
  ~device_buffer() { release(); }
  void* data() { return data_; }
  const void* data() const { return data_; }
  std::size_t size() const { return size_; }

 private:
  void release()
  {
    if (data_) mr::get_current_device_resource()->deallocate(data_, size_, stream_);
    data_ = nullptr;
  }
  void* data_          = nullptr;
  std::size_t size_    = 0;
  cudaStream_t stream_ = nullptr;
};

}  // namespace rmm

// ------------------------------------------------------------------------------------ cudf
namespace cudf {

using size_type = int32_t;  // as in cuDF 0.19; the C ABI underneath counts rows in int64

// fixed-width types of the reference's test matrix (test/compare_against_single_gpu.cu:237-268):
// 4-byte and 8-byte integers plus the timestamp / duration types that are integers underneath
enum class type_id : int32_t {
  EMPTY = 0,
  INT32,
  INT64,
  TIMESTAMP_DAYS,          // int32
  TIMESTAMP_MILLISECONDS,  // int64
  TIMESTAMP_NANOSECONDS,   // int64
  DURATION_DAYS,           // int32
  DURATION_SECONDS,        // int64
  DURATION_MICROSECONDS,   // int64
  STRING
};
enum class hash_id : int32_t { HASH_IDENTITY = DJ_HASH_IDENTITY, HASH_MURMUR3 = DJ_HASH_MURMUR3 };
constexpr uint32_t DEFAULT_HASH_SEED = 0;

class data_type {
 public:
  data_type() = default;
  explicit data_type(type_id id) : id_(id) {}
  type_id id() const { return id_; }
  bool operator==(data_type o) const { return id_ == o.id_; }

 private:
  type_id id_ = type_id::EMPTY;
};

template <typename T>
constexpr type_id type_to_id();
template <>
constexpr type_id type_to_id<int32_t>() { return type_id::INT32; }
template <>
constexpr type_id type_to_id<int64_t>() { return type_id::INT64; }

inline std::size_t size_of(data_type t)
{
  switch (t.id()) {
    case type_id::INT32:
    case type_id::TIMESTAMP_DAYS:
    case type_id::DURATION_DAYS: return 4;
    case type_id::INT64:
    case type_id::TIMESTAMP_MILLISECONDS:
    case type_id::TIMESTAMP_NANOSECONDS:
    case type_id::DURATION_SECONDS:
    case type_id::DURATION_MICROSECONDS: return 8;
    default: throw std::runtime_error("cudf shim: size_of is defined for fixed-width types only");
  }
}
inline bool is_fixed_width(data_type t) { return t.id() != type_id::EMPTY && t.id() != type_id::STRING; }

class column_view {
 public:
  column_view() = default;
  column_view(data_type t, size_type n, const void* p) : type_(t), size_(n), data_(p) {}
  data_type type() const { return type_; }
  size_type size() const { return size_; }
  template <typename T = void>
  const T* head() const { return static_cast<const T*>(data_); }
  template <typename T>
  const T* begin() const { return head<T>(); }
  template <typename T>
  const T* end() const { return head<T>() + size_; }

 protected:
  data_type type_;
  size_type size_   = 0;
  const void* data_ = nullptr;
};

class mutable_column_view : public column_view {
 public:
  mutable_column_view() = default;
  mutable_column_view(data_type t, size_type n, void* p) : column_view(t, n, p) {}
  template <typename T = void>
  T* head() const { return static_cast<T*>(const_cast<void*>(data_)); }
  template <typename T>
  T* begin() const { return head<T>(); }
};

class column {
 public:
  column() = default;
  column(data_type t, size_type n, rmm::device_buffer&& buf) : type_(t), size_(n), data_(std::move(buf)) {}
  data_type type() const { return type_; }
  size_type size() const { return size_; }
  column_view view() const { return column_view(type_, size_, data_.data()); }
  mutable_column_view mutable_view() { return mutable_column_view(type_, size_, data_.data()); }
  // shrink the logical row count without reallocating (join outputs are over-allocated)
  void set_size(size_type n) { size_ = n; }

 private:
  data_type type_;
  size_type size_ = 0;
  rmm::device_buffer data_;
};

template <typename ColumnView>
class table_view_base {
 public:
  table_view_base() = default;
  explicit table_view_base(std::vector<ColumnView> cols) : cols_(std::move(cols)) {}
  size_type num_columns() const { return (size_type)cols_.size(); }
  size_type num_rows() const { return cols_.empty() ? 0 : cols_[0].size(); }
  const ColumnView& column(size_type i) const { return cols_.at(i); }
  auto begin() const { return cols_.begin(); }
  auto end() const { return cols_.end(); }

 private:
  std::vector<ColumnView> cols_;
};
using table_view         = table_view_base<column_view>;
using mutable_table_view = table_view_base<mutable_column_view>;

class table {
 public:
  table() = default;
  explicit table(std::vector<std::unique_ptr<column>>&& cols) : cols_(std::move(cols)) {}
  size_type num_columns() const { return (size_type)cols_.size(); }
  size_type num_rows() const { return cols_.empty() ? 0 : cols_[0]->size(); }
  column& get_column(size_type i) { return *cols_.at(i); }
  table_view view() const
  {
    std::vector<column_view> v;
    for (auto& c : cols_) v.push_back(c->view());
    return table_view(std::move(v));
  }
  mutable_table_view mutable_view()
  {
    std::vector<mutable_column_view> v;
    for (auto& c : cols_) v.push_back(c->mutable_view());
    return mutable_table_view(std::move(v));
  }

 private:
  std::vector<std::unique_ptr<column>> cols_;
};

inline std::unique_ptr<column> make_fixed_width_column(data_type t, size_type n, cudaStream_t stream = nullptr)
{
  return std::make_unique<column>(t, n, rmm::device_buffer((std::size_t)n * size_of(t), stream));
}
inline std::unique_ptr<column> make_numeric_column(data_type t, size_type n, cudaStream_t stream = nullptr)
{
  return make_fixed_width_column(t, n, stream);
}

// The kernels underneath move 8-byte values.  4-byte columns are widened (sign-extended) into
// temporary INT64 columns on the way in and narrowed back on the way out; results are identical,
// only the partition a key lands in differs from cuDF's 4-byte murmur (results never depend on it).
std::unique_ptr<table> widen_to_i64(table_view const& t);                     // every column -> INT64
std::unique_ptr<table> narrow_like(table_view const& t, std::vector<data_type> const& types);
bool all_i64(table_view const& t);

// cudf::hash_partition(table, {key column}, nparts, hash, seed) -> (partitioned table, offsets[nparts])
// (call sites src/distributed_join.cpp:213-225, src/shuffle_on.cpp:59-60).  Fixed-width columns, one
// key column at any position.  A key plus 1..3 further columns runs dj_hash_partition_i64 (4-byte
// columns widened as above); any other table -- a key alone or with up to DJ_MAX_PAYLOAD_COLUMNS
// further columns -- runs dj_hash_partition_cols, which moves every non-key column at its own width
// (only a 4-byte key is widened).  Both hash the same int64 key, so a row lands in the same partition
// whichever path its table takes.  Stream 0.
std::pair<std::unique_ptr<table>, std::vector<size_type>> hash_partition(
  table_view const& input, std::vector<size_type> const& columns_to_hash, int num_partitions,
  hash_id hash_function = hash_id::HASH_MURMUR3, uint32_t seed = DEFAULT_HASH_SEED);

// cudf::inner_join(left, right, {0}, {0}) -> left columns ++ right columns
// (src/distributed_join.cpp:79).  One key column per side at any position.  Two fixed-width columns
// per side run dj_inner_join_i64; any other fixed-width tables (key + 0..DJ_MAX_PAYLOAD_COLUMNS
// columns per side) run dj_inner_join_cols, which joins (key, row index) and gathers the other
// columns at their own widths.  Builds on the smaller side; the output is all left columns ++ all
// right columns in their original positions and types.
std::unique_ptr<table> inner_join(table_view const& left, table_view const& right,
                                  std::vector<size_type> const& left_on,
                                  std::vector<size_type> const& right_on);

// cudf::concatenate of tables with identical schemas (src/distributed_join.cpp:339).
std::unique_ptr<table> concatenate(std::vector<table_view> const& views);

}  // namespace cudf
