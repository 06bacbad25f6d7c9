// Handle registry and C-ABI guard shared by the translation units of libzkp_b200.
#pragma once
#include <cstring>
#include <memory>
#include <unordered_map>
#include <vector>
#include "../../include/zkp_b200.h"
#include "common.cuh"

namespace zkp {

enum class HandleKind : int { G1Table = 1, G2Table = 2, Scalars = 3, Sparse = 4, WitnessProgram = 5 };

struct Resource {
  HandleKind kind;
  uint64_t n = 0;  // elements (points or scalars)
  int pre_c = 0;   // point tables: window width of the precomputed layout [w][i] (0 = plain)
  DevBuf buf;
  // sparse matrices (CSR): n rows; buf = values (Montgomery), aux[0] = row_ptr, aux[1] = column indices
  uint64_t cols = 0, nnz = 0;
  DevBuf aux[3];
  // witness programs (csrc/witness.cuh): the four forms of every step as one CSR of 4 * steps rows over `cols`
  // variables in buf / aux[0] / aux[1]; aux[2] = out_var[steps] | level_ptr[levels + 1] | in_var[inputs]
  uint64_t steps = 0, levels = 0, inputs = 0;
  Resource() = default;
  Resource(const Resource&) = delete;
  Resource& operator=(const Resource&) = delete;
  // a half-built resource dropped by an exception, or a handle erased from the registry, gives its
  // buffers back to the pool (recycle() is a no-op on an empty buffer)
  ~Resource() {
    buf.recycle();
    for (DevBuf& b : aux) b.recycle();
  }
};

struct Registry {
  std::unordered_map<uint64_t, std::unique_ptr<Resource>> items;
  uint64_t next = 1;
  uint64_t put(std::unique_ptr<Resource> r) {
    uint64_t h = next++;
    items[h] = std::move(r);
    return h;
  }
  Resource* get(uint64_t h, HandleKind k) {
    auto it = items.find(h);
    if (it == items.end() || it->second->kind != k) return nullptr;
    return it->second.get();
  }
};

Registry& registry();
void set_last_error(const std::string& s);

struct BadHandle : std::runtime_error {
  using std::runtime_error::runtime_error;
};
struct InvalidArgument : std::runtime_error {
  using std::runtime_error::runtime_error;
};
struct NotDivisible : std::runtime_error {
  using std::runtime_error::runtime_error;
};

inline Resource* need(uint64_t h, HandleKind k, const char* what) {
  Resource* r = registry().get(h, k);
  if (!r) throw BadHandle(std::string("bad handle for ") + what);
  return r;
}

// Runs `fn` under the context mutex and maps exceptions to ABI error codes.
template <class Fn>
int guarded(Fn&& fn) {
  try {
    if (!ctx_ready()) {
      set_last_error("zkp_init has not been called successfully (no CPU fallback exists)");
      return ZKP_ERR_NOT_INITIALISED;
    }
    Context& c = ctx();
    std::lock_guard<std::mutex> lk(c.mu);
    CUDA_CHECK(cudaSetDevice(c.device));
    fn(c);
    return ZKP_OK;
  } catch (const BadHandle& e) {
    set_last_error(e.what());
    return ZKP_ERR_BAD_HANDLE;
  } catch (const InvalidArgument& e) {
    set_last_error(e.what());
    return ZKP_ERR_INVALID_ARGUMENT;
  } catch (const NotDivisible& e) {
    set_last_error(e.what());
    return ZKP_ERR_NOT_DIVISIBLE;
  } catch (const std::exception& e) {
    set_last_error(e.what());
    return ZKP_ERR_CUDA;
  }
}

}  // namespace zkp
