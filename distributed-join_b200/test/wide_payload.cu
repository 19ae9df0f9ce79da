// wide_payload.cu -- distributed_inner_join on tables with several fixed-width payload columns, in
// the shape of the reference's string-payload test (test/string_payload.cu) with fixed-width columns
// in place of the string column.  Left keys are 3i and right keys 5j (offset per rank), so the join
// has n*world/5 rows, each with equal keys divisible by 15.  Every payload column holds a fixed
// function of its row's key, so each joined row can be checked column by column.
//
// Table shapes: both sides wide (key + INT32, INT64, TIMESTAMP_DAYS, TIMESTAMP_NANOSECONDS,
// DURATION_SECONDS), the left key at position 2 instead of 0, and a 2-column left table against a
// wide right one (the two take different partition paths and must still co-locate).  Each runs with
// INT32 and INT64 keys, 12 000 and 120 000 rows per rank, odf 1 and 2, and nvlink_domain_size 1
// (the IB-stage shuffle) and world.
#include <cstdint>
#include <cstring>
#include <iostream>
#include <memory>
#include <sstream>
#include <string>
#include <vector>

#include "../host/bootstrap.hpp"
#include "../host/compression.hpp"
#include "../host/distributed_join.hpp"
#include "../host/error.hpp"
#include "../host/setup.hpp"

using cudf::data_type;
using cudf::type_id;

static const std::vector<type_id> kWidePayload = {type_id::INT32, type_id::INT64, type_id::TIMESTAMP_DAYS,
                                                  type_id::TIMESTAMP_NANOSECONDS, type_id::DURATION_SECONDS};

// Value of payload column c of a row with key k on side s (0 left, 1 right); 4-byte columns keep the
// low 32 bits.  Distinct per side and column, and 8-byte columns use their high bits.
static int64_t payload_value(int side, int c, int64_t key, size_t width)
{
  const int64_t v = key * (c + 2) + 17 * c + side;
  return width == 8 ? v * 1000003 - side : (int64_t)(int32_t)v;
}

struct Shape {
  std::vector<type_id> payload;  // payload column types, in table order around the key
  cudf::size_type key_pos;
};

// Rows with keys start, start+multiple, ...: the key column at shape.key_pos, payloads around it.
static std::unique_ptr<cudf::table> make_table(int side, Shape const& shape, type_id key_t, int64_t n, int64_t start,
                                               int64_t multiple)
{
  std::vector<type_id> types = shape.payload;
  types.insert(types.begin() + shape.key_pos, key_t);
  std::vector<std::unique_ptr<cudf::column>> cols;
  for (size_t t = 0, c = 0; t < types.size(); t++) {
    const size_t es = cudf::size_of(data_type(types[t]));
    std::vector<char> h((size_t)n * es);
    for (int64_t i = 0; i < n; i++) {
      const int64_t key = start + i * multiple;
      const int64_t v   = (int)t == shape.key_pos ? key : payload_value(side, (int)c, key, es);
      if (es == 8)
        std::memcpy(h.data() + i * es, &v, 8);
      else {
        const int32_t v32 = (int32_t)v;
        std::memcpy(h.data() + i * es, &v32, 4);
      }
    }
    if ((int)t != shape.key_pos) c++;
    cols.push_back(cudf::make_fixed_width_column(data_type(types[t]), (cudf::size_type)n));
    CUDA_RT_CALL(cudaMemcpy(cols.back()->mutable_view().head(), h.data(), h.size(), cudaMemcpyHostToDevice));
  }
  return std::make_unique<cudf::table>(std::move(cols));
}

// Host copy of column `c` of `t`, every value sign-extended to int64.
static std::vector<int64_t> column_values(cudf::table_view const& t, cudf::size_type c)
{
  const int64_t n  = t.num_rows();
  const size_t es  = cudf::size_of(t.column(c).type());
  std::vector<char> h((size_t)n * es);
  CUDA_RT_CALL(cudaMemcpy(h.data(), t.column(c).head(), h.size(), cudaMemcpyDeviceToHost));
  std::vector<int64_t> v((size_t)n);
  for (int64_t i = 0; i < n; i++)
    v[i] = es == 8 ? reinterpret_cast<const int64_t*>(h.data())[i] : reinterpret_cast<const int32_t*>(h.data())[i];
  return v;
}

// Violations in this rank's result: column count / types other than left ++ right, unequal keys,
// keys not divisible by 15, payloads that are not their key's function.
static int64_t check_result(cudf::table_view const& result, Shape const& ls, Shape const& rs, type_id key_t)
{
  const int64_t n = result.num_rows();
  if (n == 0) return 0;  // an empty local result carries no columns (src/distributed_join.cpp:76-82)
  std::vector<type_id> want;
  for (const Shape* s : {&ls, &rs}) {
    std::vector<type_id> t = s->payload;
    t.insert(t.begin() + s->key_pos, key_t);
    want.insert(want.end(), t.begin(), t.end());
  }
  if (result.num_columns() != (cudf::size_type)want.size()) return n;
  for (size_t c = 0; c < want.size(); c++)
    if (!(result.column((cudf::size_type)c).type() == data_type(want[c]))) return n;
  const cudf::size_type right0 = (cudf::size_type)ls.payload.size() + 1;
  const std::vector<int64_t> lkey = column_values(result, ls.key_pos);
  const std::vector<int64_t> rkey = column_values(result, right0 + rs.key_pos);
  std::vector<char> bad((size_t)n, 0);
  for (int64_t i = 0; i < n; i++) bad[i] = lkey[i] != rkey[i] || lkey[i] % 15 != 0;
  for (int side = 0; side < 2; side++) {
    Shape const& s = side ? rs : ls;
    const cudf::size_type base = side ? right0 : 0;
    for (size_t c = 0; c < s.payload.size(); c++) {
      const cudf::size_type pos = base + (cudf::size_type)c + ((cudf::size_type)c >= s.key_pos ? 1 : 0);
      const size_t es           = cudf::size_of(data_type(s.payload[c]));
      const std::vector<int64_t> v = column_values(result, pos);
      for (int64_t i = 0; i < n; i++) bad[i] |= v[i] != payload_value(side, (int)c, lkey[i], es);
    }
  }
  int64_t total = 0;
  for (char b : bad) total += b;
  return total;
}

static bool run_test(const char* name, Shape const& ls, Shape const& rs, type_id key_t, int64_t n, int odf, int nvl,
                     Communicator* communicator)
{
  const int rank = communicator->mpi_rank, world = communicator->mpi_size;
  auto left  = make_table(0, ls, key_t, n, n * rank * 3, 3);
  auto right = make_table(1, rs, key_t, n, n * rank * 5, 5);
  auto result = distributed_inner_join(left->view(), right->view(), {ls.key_pos}, {rs.key_pos}, communicator,
                                       generate_none_compression_options(left->view()),
                                       generate_none_compression_options(right->view()), odf, false, nullptr, nvl);
  const int64_t rows = dj_bootstrap::allreduce_sum(result->num_rows());
  const int64_t bad  = dj_bootstrap::allreduce_sum(check_result(result->view(), ls, rs, key_t));
  const bool ok      = rows == n * world / 5 && bad == 0;
  if (rank == 0) {
    std::ostringstream desc;
    desc << "(" << name << ", " << (key_t == type_id::INT32 ? "int32_t" : "int64_t") << " key, " << n
         << " rows per rank, odf " << odf << ", nvlink_domain_size " << nvl << ")";
    if (ok)
      std::cerr << "Test case \"wide_payload\" passes successfully. " << desc.str() << "\n";
    else
      std::cerr << "Test case \"wide_payload\" FAILED " << desc.str() << ": " << rows << " rows (want "
                << n * world / 5 << "), " << bad << " bad rows\n";
  }
  return ok;
}

int main(int argc, char* argv[])
{
  dj_bootstrap::init(&argc, &argv);
  set_cuda_device();
  Communicator* communicator{nullptr};
  registered_memory_resource* registered_mr{nullptr};
  rmm::mr::pool_memory_resource<rmm::mr::device_memory_resource>* pool_mr{nullptr};
  setup_memory_pool_and_communicator(communicator, registered_mr, pool_mr, "NCCL", "none", 0);
  const int world = communicator->mpi_size;
  const Shape wide{kWidePayload, 0}, wide_key2{kWidePayload, 2}, narrow{{type_id::INT64}, 0};
  bool ok = true;
  for (type_id key_t : {type_id::INT32, type_id::INT64})
    for (int64_t n : {12'000, 120'000})
      for (int odf : {1, 2})
        for (int nvl : {1, world}) {
          ok &= run_test("wide x wide", wide, wide, key_t, n, odf, nvl, communicator);
          ok &= run_test("left key at 2", wide_key2, wide, key_t, n, odf, nvl, communicator);
          ok &= run_test("2 columns x wide", narrow, wide, key_t, n, odf, nvl, communicator);
        }
  destroy_memory_pool_and_communicator(communicator, registered_mr, pool_mr, "NCCL", "none");
  dj_bootstrap::finalize();
  return ok ? 0 : 1;
}
