// Witness solving on the device: `count` witnesses of one circuit per call (zkp_witness_program_load,
// zkp_witness_solve_many_dev).  Included once, by poly.cu, after qap.cuh (shares sparse_upload, hptr, the arena).
//
// The reference computes witnesses on the host, one at a time: zkp/groth16/code_to_r1cs.py assigns the variables of
// the flattened program gate by gate (code_to_r1cs_with_inputs / assign_variables), and zkp/plonk/circuit.py fills the
// wire vectors a, b, c while the circuit is built.  Both compile (zkp/witness.py) into one format, a STEP PROGRAM:
//   variables v_0 .. v_{V-1} per witness, v_0 = 1, inputs from the caller;
//   step s has four sparse linear forms alpha, beta, gamma, delta over the variables:
//     N = (alpha . v)(beta . v) + gamma . v,   D = delta . v
//   a solve step writes v_out = N / D (D = 0 fails that witness); delta = 1 v_0 marks a constant denominator the
//   compiler has folded into alpha and gamma, and costs no inversion; a check step (out_var = WIT_CHECK) requires N = 0.
//   Steps are sorted by level (1 + the highest level of the variables they read; v_0 and the inputs are level 0):
//   the steps of one level are independent.
// One launch walks every level.  Each block owns `wpb` witnesses; its threads take the (witness, step) items of the
// current level, with a block barrier between levels.  Witnesses are independent, so blocks never wait for each
// other.  Variables live in the output vector itself, in Montgomery form during the walk, canonical at the end.
// A deep, narrow program (a chain) costs about one dependent memory round trip per level: latency, not throughput.
#pragma once
#include <algorithm>

namespace zkp {

static constexpr uint32_t WIT_CHECK = 0xFFFFFFFFu;  // out_var of a check step
static constexpr int WIT_THREADS = 256;

__device__ __forceinline__ Fr wit_form(const uint32_t* __restrict__ rp, const uint32_t* __restrict__ col,
                                       const Fr* __restrict__ val, uint64_t row, const Fr* v) {
  Fr acc = Fr::zero();
  for (uint32_t e = rp[row]; e < rp[row + 1]; e++) acc = acc + val[e] * v[col[e]];
  return acc;
}

// rp / col / val: the 4 * S form rows (row 4s + f, f = alpha, beta, gamma, delta; values Montgomery).
// in: count * n_in canonical inputs; out: count * V canonical values.  *first_bad = min over failing (j * S + s).
__global__ void __launch_bounds__(WIT_THREADS) witness_solve_kernel(
    const uint32_t* __restrict__ rp, const uint32_t* __restrict__ col, const Fr* __restrict__ val,
    const uint32_t* __restrict__ out_var, const uint32_t* __restrict__ level_ptr, uint32_t levels,
    const uint32_t* __restrict__ in_var, uint32_t n_in, uint64_t V, uint64_t S, const Fr* __restrict__ in, uint32_t count,
    uint32_t wpb, Fr* out, unsigned long long* first_bad) {
  const uint64_t j0 = (uint64_t)blockIdx.x * wpb;
  const uint64_t nw = min((uint64_t)wpb, count - j0);
  Fr* base = out + j0 * V;
  const uint64_t row0 = (uint64_t)n_in + 1;
  for (uint64_t t = threadIdx.x; t < nw * row0; t += blockDim.x) {
    const uint64_t w = t / row0, i = t - w * row0;
    if (i == 0) base[w * V] = Fr::one();
    else base[w * V + in_var[i - 1]] = in[(j0 + w) * n_in + i - 1].to_mont();
  }
  __syncthreads();
  for (uint32_t l = 0; l < levels; l++) {
    const uint32_t s0 = level_ptr[l], width = level_ptr[l + 1] - s0;
    for (uint64_t t = threadIdx.x; t < nw * width; t += blockDim.x) {
      const uint64_t w = t / width;
      const uint32_t s = s0 + (uint32_t)(t - w * width);
      Fr* v = base + w * V;
      const uint64_t r = 4 * (uint64_t)s;
      const Fr n = wit_form(rp, col, val, r, v) * wit_form(rp, col, val, r + 1, v) + wit_form(rp, col, val, r + 2, v);
      const uint32_t o = out_var[s];
      bool bad;
      if (o == WIT_CHECK) {
        bad = !n.is_zero();
      } else {
        const uint32_t e = rp[r + 3];
        if (rp[r + 4] == e + 1 && col[e] == 0 && val[e] == Fr::one()) {
          v[o] = n;
          bad = false;
        } else {
          const Fr d = wit_form(rp, col, val, r + 3, v);
          bad = d.is_zero();
          v[o] = n * d.inv();  // inv(0) = 0: a failed witness stays deterministic
        }
      }
      if (bad) atomicMin(first_bad, (unsigned long long)((j0 + w) * S + s));
    }
    __syncthreads();
  }
  for (uint64_t t = threadIdx.x; t < nw * V; t += blockDim.x) base[t] = base[t].from_mont();
}

}  // namespace zkp

using namespace zkp;

extern "C" {

int zkp_witness_program_load(const uint32_t* row_ptr, const uint32_t* col_idx, const uint8_t* values, uint64_t nnz,
                             const uint32_t* out_var, uint64_t steps, const uint32_t* level_ptr, uint64_t levels,
                             const uint32_t* in_var, uint64_t n_in, uint64_t vars, uint64_t* handle) {
  return guarded([&](Context& c) {
    const char* what = "zkp_witness_program_load";
    if (!handle || !level_ptr || (steps && !out_var) || (n_in && !in_var)) throw InvalidArgument(std::string(what) + ": null argument");
    if (!vars || vars >= WIT_CHECK || steps >= (uint64_t(1) << 29) || levels > steps || n_in >= vars)
      throw InvalidArgument(std::string(what) + ": sizes out of range");
    if (level_ptr[0] != 0 || level_ptr[levels] != steps) throw InvalidArgument(std::string(what) + ": level_ptr must run from 0 to steps");
    // level of every variable: 0 for v_0 and the inputs, the level of its step otherwise; each written once
    std::vector<uint32_t> var_level(vars, WIT_CHECK);
    var_level[0] = 0;
    for (uint64_t i = 0; i < n_in; i++) {
      if (in_var[i] == 0 || in_var[i] >= vars || var_level[in_var[i]] != WIT_CHECK)
        throw InvalidArgument(std::string(what) + ": input variables must be distinct and in [1, vars)");
      var_level[in_var[i]] = 0;
    }
    uint64_t written = 0;
    for (uint64_t l = 0; l < levels; l++) {
      if (level_ptr[l] > level_ptr[l + 1]) throw InvalidArgument(std::string(what) + ": level_ptr is not monotone");
      for (uint64_t s = level_ptr[l]; s < level_ptr[l + 1]; s++) {
        const uint32_t o = out_var[s];
        if (o == WIT_CHECK) continue;
        if (o == 0 || o >= vars || var_level[o] != WIT_CHECK)
          throw InvalidArgument(std::string(what) + ": a step writes v_0, an input, a variable out of range or one already written");
        var_level[o] = (uint32_t)(l + 1);
        written++;
      }
    }
    if (written + n_in + 1 != vars) throw InvalidArgument(std::string(what) + ": some variable is never written");
    auto r = std::make_unique<Resource>();
    r->kind = HandleKind::WitnessProgram;
    sparse_upload(c, *r, row_ptr, col_idx, values, 4 * steps, vars, nnz, what);
    // a step reads only variables of lower levels: the steps of one level never race
    for (uint64_t l = 0; l < levels; l++)
      for (uint64_t s = level_ptr[l]; s < level_ptr[l + 1]; s++)
        for (uint32_t e = row_ptr[4 * s]; e < row_ptr[4 * s + 4]; e++)
          if (var_level[col_idx[e]] > l) throw InvalidArgument(std::string(what) + ": a step reads a variable of its own or a later level");
    r->steps = steps;
    r->levels = levels;
    r->inputs = n_in;
    const uint64_t n32 = steps + levels + 1 + n_in;
    r->aux[2].reserve_pooled(n32 * 4);
    if (steps) CUDA_CHECK(cudaMemcpyAsync(r->aux[2].p, out_var, steps * 4, cudaMemcpyHostToDevice, c.stream));
    CUDA_CHECK(cudaMemcpyAsync(r->aux[2].as<uint32_t>() + steps, level_ptr, (levels + 1) * 4, cudaMemcpyHostToDevice, c.stream));
    if (n_in) CUDA_CHECK(cudaMemcpyAsync(r->aux[2].as<uint32_t>() + steps + levels + 1, in_var, n_in * 4, cudaMemcpyHostToDevice, c.stream));
    CUDA_CHECK(cudaStreamSynchronize(c.stream));
    *handle = registry().put(std::move(r));
  });
}

int zkp_witness_solve_many_dev(uint64_t program, uint64_t inputs, uint64_t in_off, uint32_t count, uint64_t out,
                               uint64_t out_off, uint64_t* first_bad) {
  return guarded([&](Context& c) {
    const char* what = "zkp_witness_solve_many_dev";
    Resource* p = need(program, HandleKind::WitnessProgram, what);
    if (!first_bad) throw InvalidArgument(std::string(what) + ": null argument");
    const uint64_t V = p->cols, S = p->steps, n_in = p->inputs;
    const Fr* x = hptr(inputs, in_off, count * n_in, what);
    Fr* o = hptr(out, out_off, count * V, what);
    if (inputs == out && x < o + count * V && o < x + count * n_in)
      throw InvalidArgument(std::string(what) + ": inputs and outputs overlap");
    *first_bad = ~uint64_t(0);
    if (!count) return;
    // witnesses per block: enough to give every thread an item on an average level, while count still spreads over
    // about two blocks per SM; a narrow program (a chain) then runs in small blocks of many witnesses
    const uint64_t avg = std::max<uint64_t>(1, S / std::max<uint64_t>(1, p->levels));
    uint64_t wpb = std::min<uint64_t>((WIT_THREADS + avg - 1) / avg, (count + 2 * c.sm_count - 1) / (2 * c.sm_count));
    wpb = std::max<uint64_t>(1, std::min<uint64_t>(wpb, count));
    int threads = 32;
    while (threads < WIT_THREADS && (uint64_t)threads < wpb * avg) threads *= 2;
    const uint64_t blocks = (count + wpb - 1) / wpb;
    if (blocks >= (uint64_t(1) << 31)) throw InvalidArgument(std::string(what) + ": count too large for one grid");
    ArenaScope scope;
    Fr* bad = g_arena.alloc(1);
    CUDA_CHECK(cudaMemsetAsync(bad, 0xFF, sizeof(uint64_t), c.stream));
    const uint32_t* aux = p->aux[2].as<uint32_t>();
    witness_solve_kernel<<<(unsigned)blocks, threads, 0, c.stream>>>(
        p->aux[0].as<uint32_t>(), p->aux[1].as<uint32_t>(), p->buf.as<Fr>(), aux, aux + S, (uint32_t)p->levels,
        aux + S + p->levels + 1, (uint32_t)n_in, V, S, x, count, (uint32_t)wpb, o, reinterpret_cast<unsigned long long*>(bad));
    CUDA_CHECK_LAUNCH();
    c.launches++;
    uint64_t fb = 0;
    CUDA_CHECK(cudaMemcpyAsync(&fb, bad, sizeof(uint64_t), cudaMemcpyDeviceToHost, c.stream));
    CUDA_CHECK(cudaStreamSynchronize(c.stream));
    *first_bad = fb;
  });
}

}  // extern "C"
