// Generic fused vertex-program kernel: interprets a lowered execution unit.
//
// The reference turns every fused unit into CUDA text (Jinja templates
// stgraph/compiler/code_gen/templates/fa/tpl_fa_csr*.jinja:1-57, per-op C snippets in
// stgraph/compiler/registry.py:195-406) and compiles it with nvcc at run time
// (code_gen/compiler.py:14-44).  Here the unit is lowered once (compiler/lowering.py) to a small
// register program and ONE pre-compiled sm_100a kernel evaluates it with the same loop
// structure as the reference template:
//     per (row, feature lane):  PRE instrs;  for e in row: LOOP instrs;  POST instrs
// Differences that matter: lanes of a row sit in one warp (a GROUP of 2^k lanes per row when the
// unit is narrower than a warp, several rows per warp), cross-lane reductions ([H,D] -> [H,1]
// outputs, the reference's per-lane atomicAdd, kernel_context.py:126-149) use segmented warp
// shuffles when the segment is a power of two, and aggregations onto the *other* side are never
// written with atomics from inside the loop: lowering runs a second launch on the transposed CSR.
// Virtual registers live in shared memory ([reg][thread], conflict-free); a register holds four consecutive
// elements (float4) when the unit's inner dimension allows it.
// This is the generality path; hot shapes are matched to agg.cu / gat.cu first.
//
// The mixed form (MIXED = true, stg_vm_run_mixed) also reads bf16 / fp16 tensors: LOAD widens each element to fp32 as
// it is loaded, and registers, accumulators, arithmetic and every stored tensor stay fp32.  Its lanes are those of the
// fp32 form on the widened tensors, so it computes the fp32 program's operations in the same order.
#include "common.cuh"
#include "h16.cuh"

#include <type_traits>

namespace stg {
namespace {

constexpr int kVmThreads = 128;
// One block per long row.  Scalar lanes: 32 warps share its edges; float4 lanes (a register is 16 bytes per
// thread in shared memory): 8 warps, so that several blocks still fit an SM.
template <int VEC> struct HubThreads { static constexpr int value = VEC == 4 ? 256 : 1024; };

// Rows longer than this are split over a whole block (interpreting an instruction costs a few hundred
// cycles, so long rows dominate otherwise).  The hub launch finds them by scanning the row lengths itself.
constexpr int kVmHubThreshold = 96;

struct VmArgs {
  StgCsrView g;
  void* tensors[STG_VM_MAX_TENSORS];
};

__device__ __forceinline__ int tensor_elem(const StgVmTensor& t, int i0, int i1, int dim1) {
  return (t.bc0 ? i0 : 0) * (t.bc1 ? dim1 : 1) + (t.bc1 ? i1 : 0);
}
__device__ __forceinline__ int tensor_size(const StgVmTensor& t, int dim0, int dim1) {
  return (t.bc0 ? dim0 : 1) * (t.bc1 ? dim1 : 1);
}

// A virtual register holds VEC consecutive elements of the unit's flattened [dim0, dim1] lane space: VEC = 4 when
// dim1 % 4 == 0 (the four elements then share their dim0 index), so a [8,16] unit is ONE pass of 32 lanes with
// 128-bit loads instead of four passes of scalar lanes -- the interpreter's per-instruction cost is paid once per
// four elements.  VEC = 1 is the general form.
template <int VEC> struct Vec;
template <> struct Vec<1> {
  using T = float;
  static __device__ __forceinline__ T splat(float v) { return v; }
  static __device__ __forceinline__ float first(T v) { return v; }
  static __device__ __forceinline__ float hsum(T v) { return v; }
  static __device__ __forceinline__ T load(const float* p) { return __ldg(p); }
  static __device__ __forceinline__ void store(float* p, T v) { *p = v; }
  static __device__ __forceinline__ void atomic_add(float* p, T v) { atomicAdd(p, v); }
  template <class F> static __device__ __forceinline__ T map(T a, F f) { return f(a); }
  template <class F> static __device__ __forceinline__ T map2(T a, T b, F f) { return f(a, b); }
};
template <> struct Vec<4> {
  using T = float4;
  static __device__ __forceinline__ T splat(float v) { return make_float4(v, v, v, v); }
  static __device__ __forceinline__ float first(T v) { return v.x; }
  static __device__ __forceinline__ float hsum(T v) { return (v.x + v.y) + (v.z + v.w); }
  static __device__ __forceinline__ T load(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
  static __device__ __forceinline__ void store(float* p, T v) { *reinterpret_cast<float4*>(p) = v; }
  static __device__ __forceinline__ void atomic_add(float* p, T v) {
    atomicAdd(p, v.x); atomicAdd(p + 1, v.y); atomicAdd(p + 2, v.z); atomicAdd(p + 3, v.w);
  }
  template <class F> static __device__ __forceinline__ T map(T a, F f) { return make_float4(f(a.x), f(a.y), f(a.z), f(a.w)); }
  template <class F> static __device__ __forceinline__ T map2(T a, T b, F f) {
    return make_float4(f(a.x, b.x), f(a.y, b.y), f(a.z, b.z), f(a.w, b.w));
  }
};

// A 16-bit LOAD of the mixed form: one 8-byte load of 4 elements for a float4 register read along dim1 (wide), else one
// 2-byte load, splatted when the tensor is broadcast along dim1.
template <int VEC>
__device__ __forceinline__ typename Vec<VEC>::T load_h16(const unsigned short* p, bool wide, bool bf16) {
  if constexpr (VEC == 4) {
    if (wide) {
      const uint2 r = __ldg(reinterpret_cast<const uint2*>(p));
      float f[4];
      if (bf16) unpack<__nv_bfloat16, 4>(r, f);
      else unpack<__half, 4>(r, f);
      return make_float4(f[0], f[1], f[2], f[3]);
    }
  }
  const unsigned short r = __ldg(p);
  float f[1];
  if (bf16) unpack<__nv_bfloat16, 1>(r, f);
  else unpack<__half, 1>(r, f);
  return Vec<VEC>::splat(f[0]);
}

// HUB = false: one lane group per row (rows longer than the VM's hub threshold are skipped).
// HUB = true : one BLOCK per hub row; every (warp, group) slot takes a strided share of the row's edges,
//              the accumulators are merged through shared memory by kind (sum / max / min) in a fixed
//              order, and slot 0 alone runs the POST phase.
// U = edges interpreted together: every LOOP instruction is executed for U edges of the row before the next one
// is decoded, so U neighbour loads are in flight per instruction (a register lives in shared memory, hence a LOAD
// cannot overlap the instruction after it) and the decode cost is paid once per U edges.  Slot u of a register is
// private to edge u of the batch; PRE runs for every slot (row-level values), POST for slot 0 after the
// accumulators of the U slots have been merged in a fixed order.
// MIXED = true: a LOAD reads its tensor in the type its StgVmTensor::dtype names (the same code for every lane, so the
// branch is uniform); MIXED = false is the fp32 kernel.
template <int GROUP, bool HUB, int VEC, int U, bool MIXED>
__global__ void __launch_bounds__(HUB ? HubThreads<VEC>::value : kVmThreads)
    vm_kernel(const __grid_constant__ VmArgs a, const __grid_constant__ StgVmProgram prog) {
  using V = Vec<VEC>;
  using T = typename V::T;
  constexpr int NT = HUB ? HubThreads<VEC>::value : kVmThreads;     // threads per block
  extern __shared__ __align__(16) float smem[];
  T* regs = reinterpret_cast<T*>(smem);                    // [n_regs][U][NT]
  T* accs = regs + prog.n_regs * U * NT;                   // [n_acc][U][NT]
  float* scratch = reinterpret_cast<float*>(accs + prog.n_acc * U * NT);   // [NT] lane-reduction staging
  constexpr int GROUPS_PER_WARP = 32 / GROUP;
  const int tid = threadIdx.x;
  const int lane = tid & 31;
  const int gl = lane & (GROUP - 1);
  const unsigned gmask = (GROUP == 32) ? 0xffffffffu : (((1u << GROUP) - 1u) << (lane & ~(GROUP - 1)));
  constexpr int NSLOT = HUB ? (NT / 32) * GROUPS_PER_WARP : 1;
  const int slot = HUB ? (tid >> 5) * GROUPS_PER_WARP + lane / GROUP : 0;
  const int dim1 = prog.dim1;
  const int dim1v = dim1 / VEC;                            // lanes per dim0 slice
  const int lanes = prog.dim0 * dim1v;                     // lanes of VEC elements each
  const int n_iter = HUB ? a.g.num_nodes : 1;
  for (int it = HUB ? blockIdx.x : 0; it < n_iter; it += HUB ? gridDim.x : 1) {
  int row;
  if (HUB) {
    row = it;
  } else {
    const int warp = blockIdx.x * (kVmThreads / 32) + (tid >> 5);
    row = warp * GROUPS_PER_WARP + lane / GROUP;
    if (row >= a.g.num_nodes) return;
  }
  const int beg = __ldg(a.g.row_offset + row);
  const int end = __ldg(a.g.row_offset + row + 1);
  if (HUB && (end - beg) <= kVmHubThreshold) continue;    // block-uniform: every thread sees the same row
  if (!HUB && (end - beg) > kVmHubThreshold) return;      // the hub launch owns this row
  const bool seg_pow2 = (dim1v & (dim1v - 1)) == 0 && dim1v <= GROUP;
  // lanes per chunk: whole dim0 slices only, so a slice never straddles two chunks
  const int chunk = (dim1v <= GROUP) ? (GROUP / dim1v) * dim1v : GROUP;
  // sum over the dim1v consecutive lanes of this lane's slice, result in every lane of the slice
  auto segment_sum = [&](float v, int i1v) -> float {
    if (seg_pow2) {
      for (int o = 1; o < dim1v; o <<= 1) v += __shfl_xor_sync(gmask, v, o, GROUP);
      return v;
    }
    scratch[tid] = v;
    __syncwarp(gmask);
    float s = 0.f;
    for (int k = 0; k < dim1v; ++k) s += scratch[tid - i1v + k];
    __syncwarp(gmask);
    return s;
  };

#define R(i) regs[((i) * U + u) * NT + tid]
#define ACC(i) accs[((i) * U + u) * NT + tid]

  for (int tx0 = 0; tx0 < lanes; tx0 += chunk) {
    const int tx = tx0 + gl;
    const bool active = gl < chunk && tx < lanes;
    const int txc = active ? tx : lanes - 1;
    const int i0 = txc / dim1v, i1v = txc - i0 * dim1v;
    const int i1 = i1v * VEC;                               // first of this lane's VEC elements along dim1
    for (int k = 0; k < prog.n_acc; ++k) {
#pragma unroll
      for (int u = 0; u < U; ++u) ACC(k) = V::splat(prog.acc_init[k]);
    }

    int nbr[U], eid[U];
    bool valid[U];                      // slot u holds an edge of this row (always true outside the LOOP phase)
#pragma unroll
    for (int u = 0; u < U; ++u) nbr[u] = 0, eid[u] = 0, valid[u] = true;
    // NU = slots the instruction runs for: U in PRE / LOOP, 1 in POST
    auto exec = [&](const StgVmInstr& in, auto nu) {
      constexpr int NU = decltype(nu)::value;
      switch (in.op) {
        case STG_OP_LOAD: {
          const StgVmTensor& t = prog.tensors[in.a];
          if constexpr (MIXED) {
            if (t.dtype != STG_DTYPE_F32) {
              const bool bf16 = t.dtype == STG_DTYPE_BF16;
              const unsigned short* base = static_cast<const unsigned short*>(a.tensors[in.a]);
              const int tsz = tensor_size(t, prog.dim0, dim1), tel = tensor_elem(t, i0, i1, dim1);
              T v[NU];
#pragma unroll
              for (int u = 0; u < NU; ++u) {
                long long id = 0;
                if (t.side == STG_VM_CENTER) id = row;
                else if (t.side == STG_VM_NBR) id = nbr[u];
                else if (t.side == STG_VM_EDGE) id = eid[u];
                const unsigned short* src = base + id * tsz + tel;     // in elements of 2 bytes
                v[u] = V::splat(0.f);
                if (valid[u]) v[u] = load_h16<VEC>(src, t.bc1, bf16);
              }
#pragma unroll
              for (int u = 0; u < NU; ++u) R(in.dst) = v[u];
              break;
            }
          }
          const float* base = static_cast<const float*>(a.tensors[in.a]);
          const int tsz = tensor_size(t, prog.dim0, dim1), tel = tensor_elem(t, i0, i1, dim1);
          T v[NU];
#pragma unroll
          for (int u = 0; u < NU; ++u) {
            long long id = 0;
            if (t.side == STG_VM_CENTER) id = row;
            else if (t.side == STG_VM_NBR) id = nbr[u];
            else if (t.side == STG_VM_EDGE) id = eid[u];
            const float* src = base + id * tsz + tel;
            v[u] = V::splat(0.f);
            if (valid[u]) v[u] = t.bc1 ? V::load(src) : V::splat(__ldg(src));
          }
#pragma unroll
          for (int u = 0; u < NU; ++u) R(in.dst) = v[u];
          break;
        }
#define STG_VM_EACH(expr)                     \
  _Pragma("unroll") for (int u = 0; u < NU; ++u) { expr; } \
  break;
        case STG_OP_CONST: STG_VM_EACH(R(in.dst) = V::splat(in.imm))
        case STG_OP_ADD: STG_VM_EACH(R(in.dst) = V::map2(R(in.a), R(in.b), [](float x, float y) { return x + y; }))
        case STG_OP_SUB: STG_VM_EACH(R(in.dst) = V::map2(R(in.a), R(in.b), [](float x, float y) { return x - y; }))
        case STG_OP_MUL: STG_VM_EACH(R(in.dst) = V::map2(R(in.a), R(in.b), [](float x, float y) { return x * y; }))
        case STG_OP_DIV: STG_VM_EACH(R(in.dst) = V::map2(R(in.a), R(in.b), [](float x, float y) { return x / y; }))
        case STG_OP_EXP: STG_VM_EACH(R(in.dst) = V::map(R(in.a), [](float x) { return expf(x); }))
        case STG_OP_LRELU: { const float m = in.imm; STG_VM_EACH(R(in.dst) = V::map(R(in.a), [m](float x) { return x > 0.f ? x : m * x; })) }
        case STG_OP_LRELU_BWD: { const float m = in.imm; STG_VM_EACH(R(in.dst) = V::map(R(in.a), [m](float x) { return x > 0.f ? 1.f : m; })) }
        case STG_OP_RELU: STG_VM_EACH(R(in.dst) = V::map(R(in.a), [](float x) { return x > 0.f ? x : 0.f; }))
        case STG_OP_RELU_BWD: STG_VM_EACH(R(in.dst) = V::map2(R(in.a), R(in.b), [](float x, float y) { return x > 0.f ? y : 0.f; }))
        case STG_OP_AMAX_BWD: STG_VM_EACH(R(in.dst) = V::map2(R(in.a), R(in.b), [](float x, float y) { return x == y ? 1.f : 0.f; }))
        case STG_OP_ACC_SUM: STG_VM_EACH(if (valid[u]) ACC(in.dst) = V::map2(ACC(in.dst), R(in.a), [](float x, float y) { return x + y; }))
        case STG_OP_ACC_MAX: STG_VM_EACH(if (valid[u]) ACC(in.dst) = V::map2(ACC(in.dst), R(in.a), [](float x, float y) { return fmaxf(x, y); }))
        case STG_OP_ACC_MIN: STG_VM_EACH(if (valid[u]) ACC(in.dst) = V::map2(ACC(in.dst), R(in.a), [](float x, float y) { return fminf(x, y); }))
        case STG_OP_ACC_READ: {
          const float len = static_cast<float>(end - beg);
          const bool nonempty = end > beg;
          const bool mean = in.b == 1;
          STG_VM_EACH(R(in.dst) = mean ? V::map(ACC(in.a), [len, nonempty](float x) { return nonempty ? x / len : 0.f; }) : ACC(in.a))
        }
        // sum over dim1 inside each dim0 slice, broadcast back to every element of the slice (every lane of the
        // group takes part in the shuffles, also for slots without an edge)
        case STG_OP_GSUM: STG_VM_EACH(R(in.dst) = V::splat(segment_sum(active ? V::hsum(R(in.a)) : 0.f, i1v)))
#undef STG_VM_EACH
        case STG_OP_STORE: {
          const StgVmTensor& t = prog.tensors[in.a];
          float* base = static_cast<float*>(a.tensors[in.a]);
          const int tsz = tensor_size(t, prog.dim0, dim1), tel = tensor_elem(t, i0, i1, dim1);
          const bool full = t.bc0 && t.bc1;
#pragma unroll
          for (int u = 0; u < NU; ++u) {
            long long id = 0;
            if (t.side == STG_VM_CENTER) id = row;
            else if (t.side == STG_VM_NBR) id = nbr[u];
            else if (t.side == STG_VM_EDGE) id = eid[u];
            float* dst = base + id * tsz + tel;
            const T v = R(in.b);
            const bool on = active && valid[u];
            if (in.imm == 0.f) {
              // value already has the tensor's shape: one lane per distinct element writes
              const bool leader = (t.bc0 || i0 == 0) && (t.bc1 || i1 == 0);
              if (on && leader) {
                if (t.bc1) V::store(dst, v);
                else *dst = V::first(v);
              }
            } else if (full) {
              if (on) V::store(dst, v);
            } else if (t.bc0 && !t.bc1 && dim1v <= GROUP) {
              // [dim0,dim1] -> [dim0,1]: segmented reduction over the lanes of one dim0 slice
              const float sum = segment_sum(active ? V::hsum(v) : 0.f, i1v);
              if (on && i1 == 0) *dst = sum;
            } else if (on) {
              // caller zero-fills; generic cross-lane reduction
              if (t.bc1) V::atomic_add(dst, v);
              else atomicAdd(dst, V::hsum(v));
            }
          }
          break;
        }
        default: break;
      }
    };
    using AllSlots = std::integral_constant<int, U>;
    using OneSlot = std::integral_constant<int, 1>;

    int pc = 0;
    for (; pc < prog.n_pre; ++pc) {             // row-level values are computed for every edge slot; a store happens once
      if (prog.instr[pc].op == STG_OP_STORE) exec(prog.instr[pc], OneSlot{});
      else exec(prog.instr[pc], AllSlots{});
    }
    const int loop_end = prog.n_pre + prog.n_loop;
    if (prog.n_loop > 0) {
      for (int e0 = beg + slot * U; e0 < end; e0 += NSLOT * U) {
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int e = e0 + u;
          valid[u] = e < end;
          nbr[u] = valid[u] ? __ldg(a.g.column_indices + e) : 0;
          eid[u] = a.g.eids_identity ? e : (valid[u] ? __ldg(a.g.eids + e) - a.g.eid_base : 0);
        }
        for (int q = prog.n_pre; q < loop_end; ++q) exec(prog.instr[q], AllSlots{});
      }
#pragma unroll
      for (int u = 0; u < U; ++u) valid[u] = true;
    }
    // merge the U edge slots of this thread into slot 0 (fixed order)
    for (int k = 0; k < prog.n_acc; ++k) {
      const int kind = prog.acc_kind[k];
      T v = accs[(k * U) * NT + tid];
#pragma unroll
      for (int u = 1; u < U; ++u) {
        const T o = accs[(k * U + u) * NT + tid];
        v = V::map2(v, o, [kind](float x, float y) { return kind == 1 ? fmaxf(x, y) : kind == 2 ? fminf(x, y) : x + y; });
      }
      accs[(k * U) * NT + tid] = v;
    }
    if (HUB) {
      __syncthreads();
      if (slot == 0) {
        for (int k = 0; k < prog.n_acc; ++k) {
          T v = accs[(k * U) * NT + tid];
          const int kind = prog.acc_kind[k];
          for (int s2 = 1; s2 < NSLOT; ++s2) {
            const int other = (s2 / GROUPS_PER_WARP) * 32 + (s2 % GROUPS_PER_WARP) * GROUP + gl;
            const T o = accs[(k * U) * NT + other];
            v = V::map2(v, o, [kind](float x, float y) { return kind == 1 ? fmaxf(x, y) : kind == 2 ? fminf(x, y) : x + y; });
          }
          accs[(k * U) * NT + tid] = v;
        }
        for (int q = loop_end; q < prog.n_instr; ++q) exec(prog.instr[q], OneSlot{});
      }
      __syncthreads();
    } else {
      for (int q = loop_end; q < prog.n_instr; ++q) exec(prog.instr[q], OneSlot{});
    }
  }
  }
#undef R
#undef ACC
}

template <int GROUP, int VEC, int U, bool MIXED>
int launch_vm_rows(const VmArgs& a, const StgVmProgram& prog, cudaStream_t stream) {
  const int rows_per_block = (kVmThreads / 32) * (32 / GROUP);
  const int blocks = (a.g.num_nodes + rows_per_block - 1) / rows_per_block;
  const size_t per_thread = static_cast<size_t>(prog.n_regs + prog.n_acc) * U * VEC * sizeof(float) + sizeof(float);
  const size_t smem = per_thread * kVmThreads;
  static size_t configured = 48 * 1024;
  if (smem > configured) {
    STG_CUDA(cudaFuncSetAttribute(vm_kernel<GROUP, false, VEC, U, MIXED>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  static_cast<int>(smem)));
    configured = smem;
  }
  vm_kernel<GROUP, false, VEC, U, MIXED><<<blocks, kVmThreads, smem, stream>>>(a, prog);
  STG_LAUNCH_CHECK("vm_kernel");
  return STG_OK;
}

template <int GROUP, int VEC, int U, bool MIXED>
int launch_vm_hub(const VmArgs& a, const StgVmProgram& prog, cudaStream_t stream) {
  constexpr int ht = HubThreads<VEC>::value;
  const size_t per_thread = static_cast<size_t>(prog.n_regs + prog.n_acc) * U * VEC * sizeof(float) + sizeof(float);
  const size_t hub_smem = per_thread * ht;
  static size_t configured = 48 * 1024;
  if (hub_smem > configured) {
    STG_CUDA(cudaFuncSetAttribute(vm_kernel<GROUP, true, VEC, U, MIXED>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  static_cast<int>(hub_smem)));
    configured = hub_smem;
  }
  vm_kernel<GROUP, true, VEC, U, MIXED><<<(VEC == 4 ? 4 : 2) * sm_count(), ht, hub_smem, stream>>>(a, prog);
  STG_LAUNCH_CHECK("vm_kernel(hub)");
  return STG_OK;
}

// Edges per batch, measured on the stock GAT program of config 3 (profiles/r01_results.md): the one-row-per-group
// kernel gains from U = 4 only with scalar lanes (a float4 register file is already 16 bytes per access and most rows
// are shorter than a batch), the block-per-row kernel only with float4 lanes (long rows, latency-bound).  The
// float4 hub kernel falls back to 2 / 1 when its register file would not fit shared memory.
template <int GROUP, int VEC, bool MIXED>
int launch_vm(const VmArgs& a, const StgVmProgram& prog, cudaStream_t stream) {
  int rc;
  if constexpr (VEC == 4) rc = launch_vm_rows<GROUP, 4, 1, MIXED>(a, prog, stream);
  else rc = launch_vm_rows<GROUP, 1, 4, MIXED>(a, prog, stream);
  if (rc != STG_OK) return rc;
  if (a.g.num_edges <= kVmHubThreshold) return STG_OK;     // a row longer than the threshold cannot exist
  if constexpr (VEC == 4) {
    const size_t slot_bytes = static_cast<size_t>(prog.n_regs + prog.n_acc) * 16 * HubThreads<4>::value;
    if (4 * slot_bytes <= 160 * 1024) return launch_vm_hub<GROUP, 4, 4, MIXED>(a, prog, stream);
    if (2 * slot_bytes <= 160 * 1024) return launch_vm_hub<GROUP, 4, 2, MIXED>(a, prog, stream);
    return launch_vm_hub<GROUP, 4, 1, MIXED>(a, prog, stream);
  } else {
    return launch_vm_hub<GROUP, 1, 1, MIXED>(a, prog, stream);
  }
}

template <int VEC, bool MIXED>
int dispatch_vm(const VmArgs& a, const StgVmProgram& prog, cudaStream_t s) {
  const int lanes = prog.dim0 * prog.dim1 / VEC;
  if (lanes <= 1) return launch_vm<1, VEC, MIXED>(a, prog, s);
  if (lanes <= 2) return launch_vm<2, VEC, MIXED>(a, prog, s);
  if (lanes <= 4) return launch_vm<4, VEC, MIXED>(a, prog, s);
  if (lanes <= 8) return launch_vm<8, VEC, MIXED>(a, prog, s);
  if (lanes <= 16) return launch_vm<16, VEC, MIXED>(a, prog, s);
  return launch_vm<32, VEC, MIXED>(a, prog, s);
}

// The argument checks of both entry points, then the launch.  mixed = false: every tensor must be fp32.
int vm_run(const StgCsrView* g, const StgVmProgram* prog, void* const* tensors, void* stream, bool mixed) {
  STG_CHECK_ARG(g && prog && tensors, "NULL argument");
  STG_CHECK_ARG(g->row_offset != nullptr, "row_offset is NULL");
  STG_CHECK_ARG(prog->dim0 > 0 && prog->dim1 > 0, "program dims must be positive");
  STG_CHECK_ARG(prog->n_tensors >= 0 && prog->n_tensors <= STG_VM_MAX_TENSORS, "too many tensors (%d)", prog->n_tensors);
  STG_CHECK_ARG(prog->n_instr >= 0 && prog->n_instr <= STG_VM_MAX_INSTR, "too many instructions (%d)", prog->n_instr);
  STG_CHECK_ARG(prog->n_regs >= 0 && prog->n_regs <= STG_VM_MAX_REGS, "too many registers (%d)", prog->n_regs);
  STG_CHECK_ARG(prog->n_acc >= 0 && prog->n_acc <= STG_VM_MAX_ACC, "too many accumulators (%d)", prog->n_acc);
  STG_CHECK_ARG(prog->n_pre >= 0 && prog->n_loop >= 0 && prog->n_pre + prog->n_loop <= prog->n_instr,
                "inconsistent phase counts");
  bool needs_eids = false;
  for (int i = 0; i < prog->n_instr; ++i) {
    const StgVmInstr& in = prog->instr[i];
    STG_CHECK_ARG(in.op >= 0 && in.op < STG_OP_COUNT_, "bad opcode %d at %d", in.op, i);
    if (in.op == STG_OP_LOAD || in.op == STG_OP_STORE) {
      STG_CHECK_ARG(in.a >= 0 && in.a < prog->n_tensors, "tensor index out of range at instr %d", i);
      STG_CHECK_ARG(tensors[in.a] != nullptr, "tensor %d is NULL", in.a);
      if (prog->tensors[in.a].side == STG_VM_EDGE) needs_eids = true;
    }
    if (in.op == STG_OP_GSUM) {
      const int d1 = prog->dim1;
      STG_CHECK_ARG(d1 <= 32, "GSUM needs dim1 <= 32 (got %d)", d1);
    }
  }
  for (int i = 0; i < prog->n_tensors; ++i) {
    const int code = prog->tensors[i].dtype;
    if (mixed) {
      STG_CHECK_ARG(code == STG_DTYPE_F32 || code == STG_DTYPE_BF16 || code == STG_DTYPE_F16,
                    "unknown dtype code %d of tensor %d (STG_DTYPE_F32 = 0, STG_DTYPE_BF16 = 1, STG_DTYPE_F16 = 2)", code, i);
    } else {
      STG_CHECK_ARG(code == STG_DTYPE_F32, "tensor %d has dtype code %d: stg_vm_run_f32 takes fp32 tensors only "
                    "(16-bit tensors go to stg_vm_run_mixed)", i, code);
    }
  }
  for (int i = 0; i < prog->n_instr; ++i) {
    const StgVmInstr& in = prog->instr[i];
    STG_CHECK_ARG(in.op != STG_OP_STORE || prog->tensors[in.a].dtype == STG_DTYPE_F32,
                  "STORE at instr %d writes tensor %d with dtype code %d: the VM writes fp32 tensors only", i, in.a,
                  prog->tensors[in.a].dtype);
  }
  STG_CHECK_ARG(!needs_eids || g->eids_identity || g->eids || g->num_edges == 0, "eids is NULL");
  if (g->num_nodes == 0) return STG_OK;
  STG_CHECK_ARG(g->num_edges == 0 || g->column_indices, "column_indices is NULL");
  VmArgs a;
  a.g = *g;
  for (int i = 0; i < STG_VM_MAX_TENSORS; ++i) a.tensors[i] = i < prog->n_tensors ? tensors[i] : nullptr;
  cudaStream_t s = as_stream(stream);
  // float4 lanes when the four elements of a lane share their dim0 index and every tensor that is indexed along
  // dim1 is aligned to four of its elements (16 bytes for fp32, 8 for 16-bit; its per-row size is then a multiple of 4
  // elements).  A 16-bit view and an fp32 view at the same element offset therefore choose the same lanes.
  bool vec4 = prog->dim1 % 4 == 0;
  for (int i = 0; vec4 && i < prog->n_tensors; ++i) {
    const bool f32 = prog->tensors[i].dtype == STG_DTYPE_F32;
    if (prog->tensors[i].bc1 && tensors[i] != nullptr && !(f32 ? aligned16(tensors[i]) : aligned8(tensors[i]))) vec4 = false;
  }
  // the largest float4 register file the hub block may need must fit one SM's shared memory
  const size_t hub_bytes = (static_cast<size_t>(prog->n_regs + prog->n_acc) * 16 + 4) * HubThreads<4>::value;
  if (vec4 && hub_bytes <= 200 * 1024) return mixed ? dispatch_vm<4, true>(a, *prog, s) : dispatch_vm<4, false>(a, *prog, s);
  return mixed ? dispatch_vm<1, true>(a, *prog, s) : dispatch_vm<1, false>(a, *prog, s);
}

}  // namespace
}  // namespace stg

using namespace stg;

STG_API int stg_vm_run_f32(const StgCsrView* g, const StgVmProgram* prog, void* const* tensors, void* stream) {
  return vm_run(g, prog, tensors, stream, false);
}

STG_API int stg_vm_run_mixed(const StgCsrView* g, const StgVmProgram* prog, void* const* tensors, void* stream) {
  return vm_run(g, prog, tensors, stream, true);
}
