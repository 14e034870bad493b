/*
 * stgraph_b200 -- C ABI of the B200-native backend for STGraph's vertex-centric
 * aggregation hot path.
 *
 * Every entry point:
 *   - takes plain device (or, where the name ends in _host, host) pointers and sizes,
 *   - takes an explicit cudaStream_t (as void*) and enqueues work on it: no
 *     synchronisation, no allocation behind the caller's back (workspaces are
 *     passed in; sizes are queried with the *_workspace_bytes functions), so all
 *     device-pointer entry points are CUDA-graph capturable,
 *   - returns 0 on success or a negative StgStatus; it never throws and never
 *     prints.  stg_last_error() returns a thread-local description.
 *
 * "Replaces" comments cite the reference interface each entry point stands in
 * for (paths relative to the STGraph source tree, v1.1.0).
 */
#ifndef STGRAPH_B200_H_
#define STGRAPH_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define STG_ABI_VERSION 7

typedef enum StgStatus {
  STG_OK = 0,
  STG_ERR_INVALID_ARGUMENT = -1,
  STG_ERR_CUDA = -2,
  STG_ERR_UNSUPPORTED = -3,
  STG_ERR_WORKSPACE_TOO_SMALL = -4,
  STG_ERR_CAPACITY = -5
} StgStatus;

/* One direction of a graph snapshot in CSR form -- the same four device arrays
 * the reference hands to every generated kernel
 * (stgraph/graph/stgraph_base.py:51-59; kernel signature
 * stgraph/compiler/code_gen/templates/fa/tpl_fa_csr.jinja:1-11).
 * Rows are destinations for the forward (in-edge) view and sources for the
 * backward (out-edge) view. */
typedef struct StgCsrView {
  const int32_t* row_offset;     /* [num_nodes+1] */
  const int32_t* column_indices; /* [num_edges]   */
  const int32_t* eids;           /* [num_edges] edge id (or 1-based label) of each slot; may be NULL when eids_identity */
  const int32_t* node_ids;       /* [num_nodes] degree-descending row order; may be NULL (natural order) */
  int32_t num_nodes;
  int32_t num_edges;
  int32_t eid_base;      /* 0 for CSR (StaticGraph/NaiveGraph), 1 for PCSR/GPMA labels
                            (tpl_fa_pcsr.jinja:32-34, tpl_fa_gpma.jinja:32-34) */
  int32_t eids_identity; /* 1 if eids[i] == i + eid_base for all i (forward StaticGraph) */
  /* Optional hub-row schedule (rows longer than hub_threshold are processed by a
   * block-per-row kernel).  hub_rows/hub_count are device arrays produced by
   * stg_csr_hub_rows(); NULL disables the split. */
  const int32_t* hub_rows;
  const int32_t* hub_count;
  int32_t hub_threshold;
  int32_t hub_capacity;
  /* Optional global row queue of the aggregation kernels: two zero-initialised int32 counters in device
   * memory owned by the graph object ({next chunk, finished blocks}).  The row kernel draws chunks of
   * consecutive rows from it (so that all resident warps work inside one narrow window of rows and the
   * source rows of a graph with locality stay in L2) and rearms it before it exits.  One queue per view
   * and per stream: two launches that use the SAME queue must be ordered.  NULL = static block ranges. */
  int32_t* work_queue;
} StgCsrView;

/* ------------------------------------------------------------------ misc */
int stg_abi_version(void);
const char* stg_last_error(void);
/* Device properties the Python side sizes grids/benchmarks with. */
int stg_device_info(int device, int32_t* sm_count, int64_t* l2_bytes, int32_t* cc_major, int32_t* cc_minor);

/* ----------------------------------------------------- aggregation (hot) */
/* out[r,:] = row_scale[r] * sum_{e in row r} nbr_scale[col[e]] * edge_scale[eid(e)] * x[col[e],:]
 *
 * Replaces the generated Seastar kernels K0/K1 for GCNConv
 * (stgraph/nn/pytorch/static/gcn_conv.py:162-182; emitted from
 * templates/fa/tpl_fa_csr*.jinja:1-57 and launched by
 * stgraph/compiler/execution_unit.py:359-372).  With the in-edge view it is the
 * forward aggregation, with the out-edge view and x = grad_out the backward one.
 * Any of nbr_scale [N], edge_scale [E], row_scale [N] may be NULL (= 1).
 * x and out are row-major fp32 [num_nodes, feat]; they must not alias. */
int stg_agg_scaled_sum_f32(const StgCsrView* g, const float* x, int32_t feat,
                           const float* nbr_scale, const float* edge_scale,
                           const float* row_scale, float* out, void* stream);

/* Packed edge metadata: one {column, scale} pair per CSR slot, in CSR order, with
 * scale = nbr_scale[column] * edge_scale[eid].  The aggregation then issues ONE coalesced 8-byte load per
 * edge instead of a column load followed by dependent scattered 4-byte gathers (one 32-byte L2 sector
 * request per edge).  For a static graph with a fixed norm (GCNConv: stgraph/nn/pytorch/static/
 * gcn_conv.py:162-182 reads the same g.ndata["norm"] every call) the packing is paid once per graph. */
typedef struct StgEdgeMeta {
  int32_t col;
  float scale;
} StgEdgeMeta;

/* meta[e] = {column_indices[e], nbr_scale[column_indices[e]] * edge_scale[eid(e)]} for every slot e of the
 * view's CSR arrays (either scale may be NULL = 1).  meta: [num_edges] device array, 8-byte aligned. */
int stg_csr_pack_edge_meta_f32(const StgCsrView* g, const float* nbr_scale, const float* edge_scale,
                               StgEdgeMeta* meta, void* stream);

/* out[r,:] (=, +=, red.add= for accumulate 0, 1, 2) row_scale[r] * sum_{e in row r} meta[e].scale * x[meta[e].col,:]
 * -- the same sums, bit for bit, as stg_agg_scaled_sum_f32 with the scales meta was packed from. */
int stg_agg_packed_sum_f32(const StgCsrView* g, const StgEdgeMeta* meta, const float* x, int32_t feat,
                           const float* row_scale, float* out, int32_t accumulate, void* stream);

/* The same with explicit row strides (in floats, >= feat) for x and out, so that column blocks of a wider
 * buffer (e.g. one gate of the fused TGCN cell's [N, 3H] tensor) or row-padded buffers are aggregated in place.
 * (Padding F=100 rows to 512-byte lines was measured: no faster -- the gather is not bound by line alignment.) */
int stg_agg_packed_sum_strided_f32(const StgCsrView* g, const StgEdgeMeta* meta, const float* x, int32_t feat,
                                   int32_t x_ld, const float* row_scale, float* out, int32_t out_ld,
                                   int32_t accumulate, void* stream);

/* 16-bit feature rows (torch.autocast): x and out are [num_nodes, feat] row-major bf16, or both fp16, as `dtype` says.
 * The scales and the packed records stay fp32; every product and the running sum are fp32, and each output element is
 * rounded to the 16-bit type once.  Assign mode only.  A graph's packed array (stg_csr_pack_edge_meta_f32) serves the
 * fp32 and the 16-bit entry points alike, and the packed sums equal the plain ones bit for bit.  feat == 0 is a no-op. */
typedef enum StgDtype { STG_DTYPE_F32 = 0, STG_DTYPE_BF16 = 1, STG_DTYPE_F16 = 2 } StgDtype;
int stg_agg_scaled_sum_h16(const StgCsrView* g, const void* x, int32_t feat, int32_t dtype,
                           const float* nbr_scale, const float* edge_scale, const float* row_scale,
                           void* out, void* stream);
int stg_agg_packed_sum_h16(const StgCsrView* g, const StgEdgeMeta* meta, const void* x, int32_t feat,
                           int32_t dtype, const float* row_scale, void* out, void* stream);

/* Accumulating form: out[r,:] += row_scale[r] * sum(...).  Used when a row's edge set is split in two CSRs
 * (edges to locally owned sources / edges to halo sources) so that the first pass overlaps the halo
 * exchange; the passes run in a fixed order, so the result stays deterministic. */
int stg_agg_scaled_sum_accum_f32(const StgCsrView* g, const float* x, int32_t feat, const float* nbr_scale,
                                 const float* edge_scale, const float* row_scale, float* out, void* stream);

/* Reducing form: out[r,:] += ... issued as red.global.add (vector atomics, no read round trip); rows without
 * edges are not touched.  Lets the two passes over a split edge set run CONCURRENTLY on two streams into a
 * zero-filled buffer: every element then receives at most two addends, and 0 + a + b == 0 + b + a exactly,
 * so the result is independent of the interleaving (deterministic). */
int stg_agg_scaled_sum_red_f32(const StgCsrView* g, const float* x, int32_t feat, const float* nbr_scale,
                               const float* edge_scale, const float* row_scale, float* out, void* stream);

/* Row-subset form: the view holds only a SUBSET of the output rows (view row i is output row out_rows[i];
 * out_rows strictly increasing).  out[out_rows[i],:] (=, +=, red.add= for accumulate 0, 1, 2)
 * row_scale[out_rows[i]] * sum over view row i.  The multi-GPU halo-source pass uses it with
 * accumulate = 1: only the rows that have at least one remote neighbour are walked, after the
 * own-source pass has written every row. */
int stg_agg_scaled_sum_rows_f32(const StgCsrView* g, const int32_t* out_rows, const float* x, int32_t feat,
                                const float* nbr_scale, const float* edge_scale, const float* row_scale, float* out,
                                int32_t accumulate, void* stream);

/* Row-subset form of the packed kernel: view row i is output row out_rows[i] (see stg_agg_scaled_sum_rows_f32);
 * out_rows == NULL: identity.  The multi-GPU passes use it for both sub-CSRs of a rank (own-source edges over all
 * rows, halo-source edges over the rows that have any). */
int stg_agg_packed_sum_rows_f32(const StgCsrView* g, const StgEdgeMeta* meta, const int32_t* out_rows, const float* x,
                                int32_t feat, const float* row_scale, float* out, int32_t accumulate, void* stream);

/* Same operation with the source matrix ROW-PARTITIONED into num_parts blocks (multi-GPU): block q holds
 * rows [part_bounds[q], part_bounds[q+1]) of x and may live in a peer GPU's memory mapped into this
 * process (CUDA IPC / symmetric memory): the kernel then fetches remote neighbour rows with NVLink
 * loads while it aggregates -- the halo exchange is fused into the gather, tile by tile, and no
 * all-gather is materialised.  g is this rank's row slice of the CSR (global column ids).
 * x_parts / part_bounds are HOST arrays (num_parts <= STG_MAX_PARTS).  nbr_scale is indexed by global id.
 * New: the reference is single-GPU (SURVEY.md section 2 #23). */
#define STG_MAX_PARTS 16
int stg_agg_scaled_sum_parts_f32(const StgCsrView* g, const float* const* x_parts, const int32_t* part_bounds,
                                 int32_t num_parts, int32_t feat, const float* nbr_scale, const float* edge_scale,
                                 const float* row_scale, float* out, void* stream);

/* Halo pull: out[i,:] = row ids[i] of the row-partitioned matrix (blocks may be peer-GPU memory), i < n_ids.
 * max_blocks bounds the grid (<= 0: 32) so the copy overlaps a concurrently running aggregation kernel. */
int stg_halo_pull_f32(const float* const* x_parts, const int32_t* part_bounds, int32_t num_parts, const int64_t* ids,
                      int64_t n_ids, int32_t feat, float* out, int32_t max_blocks, void* stream);

/* Halo push: the owner writes local row send_rows[j] to row send_slot[j] of peer send_peer[j]'s halo buffer
 * (peer_halo[q] = base address of rank q's buffer mapped into this process).  NVLink stores are posted,
 * so a small grid reaches link rate while the aggregation kernel runs on the other SMs. */
int stg_halo_push_f32(const float* own, int32_t feat, const int64_t* send_rows, const int32_t* send_peer,
                      const int64_t* send_slot, int64_t n_items, float* const* peer_halo, int32_t num_parts,
                      int32_t max_blocks, void* stream);

/* Copy-engine halo exchange (multi-GPU; new -- the reference is single-GPU, SURVEY.md section 2 #23).
 *   stg_rows_gather_f32 : buf[j,:] = own[rows[j],:], j < n  -- packs the rows the peers need, grouped by peer;
 *   stg_halo_send_f32   : one cudaMemcpyAsync per peer q != my_rank of rows [send_off[q], send_off[q+1]) of
 *                         send_buf to peer_dst[q] (an address inside peer q's halo buffer, mapped into this
 *                         process: CUDA IPC / symmetric memory).  send_off / peer_dst are HOST arrays;
 *   stg_peer_signal     : after everything enqueued so far on `stream`, write `value` to *peer_flags[q] for every
 *                         q != my_rank (release, system scope);
 *   stg_peer_wait       : block `stream` (a one-warp spinning kernel) until flags[q] has reached value (compared
 *                         modulo 2^16: ((flags[q] - value) & 0xFFFF) < 0x8000) for every q != my_rank
 *                         (acquire, system scope); gives up after timeout_cycles SM clocks
 *                         (<= 0: 2^32) and then sets *status = 1 + q (status may be NULL).
 * No SM takes part in the transfer itself, so it overlaps the own-source aggregation pass for free. */
int stg_rows_gather_f32(const float* own, int32_t feat, const int64_t* rows, int64_t n, float* buf, int32_t max_blocks,
                        void* stream);
int stg_halo_send_f32(const float* send_buf, int32_t feat, int32_t num_parts, int32_t my_rank, const int64_t* send_off,
                      float* const* peer_dst, void* stream);
/* The three steps above in one call, with the flags written by the copy engines as well: gather, P-1 data copies,
 * then for every peer q one 4-byte copy seq_values[value] -> *peer_flags[q] (seq_values: device table with
 * seq_values[j] == j for j < 65536; value: this step's sequence number modulo 2^16, which is how stg_peer_wait
 * compares).  Nothing after the gather needs an SM. */
int stg_halo_exchange_f32(const float* own, int32_t feat, const int64_t* send_rows, const int64_t* send_off,
                          float* send_buf, float* const* peer_dst, int32_t* const* peer_flags, const int32_t* seq_values,
                          int32_t value, int32_t num_parts, int32_t my_rank, int32_t gather_blocks, void* stream);
int stg_peer_signal(int32_t* const* peer_flags, int32_t num_parts, int32_t my_rank, int32_t value, void* stream);
int stg_peer_wait(const int32_t* flags, int32_t num_parts, int32_t my_rank, int32_t value, int64_t timeout_cycles,
                  int32_t* status, void* stream);

/* Same operation with HOST buffers: copies x (and the scale vectors) to the
 * device scratch the caller provides, runs the kernel, copies out back.
 * dev_scratch must hold 2*N*feat + 2*N + E floats.  Used for the end-to-end
 * (host-to-host) figure in bench.py; synchronises the stream before returning. */
int stg_agg_scaled_sum_f32_host(const StgCsrView* g, const float* x_host, int32_t feat,
                                const float* nbr_scale_host, const float* edge_scale_host,
                                const float* row_scale_host, float* out_host,
                                void* dev_scratch, size_t dev_scratch_bytes, void* stream);

/* The same without the final stream synchronisation: the H2D copies, the kernels and the D2H copy are only
 * ENQUEUED on `stream`; out_host is valid once the caller has synchronised that stream.  Two calls on two
 * streams with two scratch buffers overlap one call's H2D with the other's D2H (PCIe is full duplex), which
 * halves the host-to-host time of a forward + backward step (bench.py `e2e`).  Host buffers must be pinned. */
int stg_agg_scaled_sum_f32_host_async(const StgCsrView* g, const float* x_host, int32_t feat,
                                const float* nbr_scale_host, const float* edge_scale_host,
                                const float* row_scale_host, float* out_host,
                                void* dev_scratch, size_t dev_scratch_bytes, void* stream);

/* Fused edge-softmax attention aggregation (one pass, online softmax per head):
 *   score_e = leaky_relu(el[col[e],h] + er[r,h]);  alpha = softmax over the row
 *   out[r,h,:] = sum_e alpha_e * feat[col[e],h,:]
 * row_max / row_sum ([N,H]) are saved for the backward pass.
 * Replaces the two-kernel K0+K1 sequence of GATConv with a materialised [E,H]
 * tensor (stgraph/nn/pytorch/static/gat_conv.py:48-56; SURVEY.md A.3). */
int stg_gat_softmax_fwd_f32(const StgCsrView* g_in, const float* el, const float* er,
                            const float* feat, int32_t heads, int32_t dim, float slope,
                            float* out, float* row_max, float* row_sum, void* stream);
/* Backward of the above, atomic-free: a destination-parallel pass over the
 * in-edge view produces d_er and the per-destination dot products, a
 * source-parallel pass over the out-edge view produces d_feat and d_el.
 * dot_scratch: [N,H] floats.  Replaces K2 (SURVEY.md A.3) and its E*H*D atomics. */
int stg_gat_softmax_bwd_f32(const StgCsrView* g_in, const StgCsrView* g_out,
                            const float* el, const float* er, const float* feat,
                            const float* out, const float* grad_out,
                            const float* row_max, const float* row_sum,
                            int32_t heads, int32_t dim, float slope,
                            float* d_feat, float* d_el, float* d_er,
                            float* dot_scratch, void* stream);
/* 16-bit form of the two above (torch.autocast): feat and d_feat are [N,H,D] bf16, or both fp16, as `dtype`
 * (StgDtype) says; el, er, out, grad_out, row_max, row_sum, d_el, d_er and dot_scratch stay fp32.  An element of feat is
 * widened to fp32 when it is loaded and d_feat is rounded to nearest even once, when it is stored.  The lanes are laid
 * out as in the fp32 entry points (4 elements per lane when dim % 4 == 0, feat / d_feat are 8-byte and out / grad_out
 * 16-byte aligned; otherwise 1), so the results equal those of the fp32 entry points on the widened feat bit for bit,
 * and d_feat equals their d_feat rounded to the 16-bit type. */
int stg_gat_softmax_fwd_h16(const StgCsrView* g_in, const float* el, const float* er, const void* feat,
                            int32_t heads, int32_t dim, int32_t dtype, float slope,
                            float* out, float* row_max, float* row_sum, void* stream);
int stg_gat_softmax_bwd_h16(const StgCsrView* g_in, const StgCsrView* g_out, const float* el, const float* er,
                            const void* feat, const float* out, const float* grad_out, const float* row_max,
                            const float* row_sum, int32_t heads, int32_t dim, int32_t dtype, float slope,
                            void* d_feat, float* d_el, float* d_er, float* dot_scratch, void* stream);

/* ------------------------------------------- generic fused vertex program */
/* A lowered execution unit: straight-line register code evaluated per
 * (row, feature lane) with one pass over the row's edges.  Replaces the Jinja
 * code generator + run-time nvcc (stgraph/compiler/code_gen/code_gen.py:39-116,
 * compiler.py:14-44): the traced IR is interpreted by one pre-compiled kernel. */
enum { STG_VM_MAX_TENSORS = 24, STG_VM_MAX_INSTR = 96, STG_VM_MAX_REGS = 48, STG_VM_MAX_ACC = 8 };

typedef enum StgVmSide { STG_VM_CENTER = 0, STG_VM_NBR = 1, STG_VM_EDGE = 2, STG_VM_PARAM = 3 } StgVmSide;
typedef enum StgVmPhase { STG_VM_PRE = 0, STG_VM_LOOP = 1, STG_VM_POST = 2 } StgVmPhase;
typedef enum StgVmOp {
  STG_OP_LOAD = 0,   /* r[dst] = tensor[a] (indexed by its side, broadcast per its bc flags) */
  STG_OP_CONST,      /* r[dst] = imm */
  STG_OP_ADD, STG_OP_SUB, STG_OP_MUL, STG_OP_DIV,   /* r[dst] = r[a] op r[b] */
  STG_OP_EXP,        /* r[dst] = expf(r[a]) */
  STG_OP_LRELU,      /* r[dst] = r[a] > 0 ? r[a] : imm * r[a] */
  STG_OP_LRELU_BWD,  /* r[dst] = r[a] > 0 ? 1 : imm */
  STG_OP_RELU,       /* r[dst] = r[a] > 0 ? r[a] : 0 */
  STG_OP_RELU_BWD,   /* r[dst] = r[a] > 0 ? r[b] : 0 */
  STG_OP_AMAX_BWD,   /* r[dst] = r[a] == r[b] ? 1 : 0 */
  STG_OP_ACC_SUM,    /* acc[dst] += r[a]             (LOOP only) */
  STG_OP_ACC_MAX,    /* acc[dst] = max(acc[dst], r[a]) */
  STG_OP_ACC_MIN,
  STG_OP_ACC_READ,   /* r[dst] = acc[a]; b=1: divide by the row length (AggMean) (POST only) */
  STG_OP_STORE,      /* tensor[a] = r[b]; imm != 0: sum r[b] over the lanes the tensor is broadcast across */
  STG_OP_GSUM,       /* r[dst] = sum of r[a] over dim1 (b=1) within each dim0 slice, broadcast back */
  STG_OP_COUNT_
} StgVmOp;

/* A tensor of the unit.  Its per-element shape is (bc0 ? dim0 : 1) x (bc1 ? dim1 : 1); feature lane
 * tx = i0*dim1 + i1 reads element (bc0 ? i0 : 0, bc1 ? i1 : 0)
 * (the reference's broadcast index, kernel_context.py:179-204). */
typedef struct StgVmTensor {
  int32_t side; /* StgVmSide */
  int32_t bc0;
  int32_t bc1;
  int32_t dtype; /* StgDtype of the bound tensor: STG_DTYPE_F32 (0) for stg_vm_run_f32 */
} StgVmTensor;

typedef struct StgVmInstr {
  int16_t op;    /* StgVmOp */
  int16_t phase; /* StgVmPhase; instructions are ordered PRE..., LOOP..., POST... */
  int16_t dst, a, b;
  int16_t pad;
  float imm;
} StgVmInstr;

typedef struct StgVmProgram {
  int32_t dim0, dim1;  /* the unit's widest per-element shape; lanes = dim0*dim1 */
  int32_t n_tensors, n_instr, n_regs, n_acc;
  int32_t n_pre, n_loop;   /* instr[0,n_pre) PRE, [n_pre,n_pre+n_loop) LOOP, rest POST */
  float acc_init[STG_VM_MAX_ACC];
  int32_t acc_kind[STG_VM_MAX_ACC];  /* 0 sum, 1 max, 2 min: how partial accumulators of a split hub row merge */
  StgVmTensor tensors[STG_VM_MAX_TENSORS];
  StgVmInstr instr[STG_VM_MAX_INSTR];
} StgVmProgram;

/* Runs the program once per (row, lane) of the given view (rows = "center" side). Tensors written
 * with a reducing STORE must be zero-filled by the caller (atomic accumulation may be used). */
int stg_vm_run_f32(const StgCsrView* g, const StgVmProgram* prog, void* const* tensors, void* stream);
/* The same program with bf16 / fp16 tensors among its inputs (torch.autocast): tensors[i] is stored as
 * prog->tensors[i].dtype says.  A LOAD widens each element to fp32; registers, accumulators, arithmetic and every STORE
 * target stay fp32 (a STORE to a 16-bit tensor is rejected).  The lanes are those of stg_vm_run_f32 with the alignment
 * taken in elements (4 elements per lane when dim1 % 4 == 0 and every tensor read along dim1 is aligned to 4 of its
 * elements: 16 bytes for fp32, 8 for 16-bit), so the results equal those of stg_vm_run_f32 on the widened tensors bit
 * for bit.  It makes stg_vm_run_f32's checks with the same messages and rejects unknown dtype codes before any launch;
 * stg_vm_run_f32 rejects any code but STG_DTYPE_F32. */
int stg_vm_run_mixed(const StgCsrView* g, const StgVmProgram* prog, void* const* tensors, void* stream);

/* ------------------------------------------------ link-prediction decode */
/* out[p] = sum_f z[a[p], f] * z[b[p], f] for p < n_pairs (a, b: int64 vertex ids, z: [N, feat] fp32).
 * Replaces STGraphTGCN.decode of the dynamic-temporal benchmark
 * (benchmarking/dynamic-temporal-tgcn/seastar/model.py:18-21: two [P, F] gathers, a multiply, a row sum). */
int stg_edge_dot_f32(const float* z, int32_t feat, const int64_t* a, const int64_t* b, int64_t n_pairs, float* out,
                     void* stream);
/* Its backward: d_z[a[p], :] += grad_out[p] * z[b[p], :] and d_z[b[p], :] += grad_out[p] * z[a[p], :]
 * (vector red.global.add; d_z must be zero-filled or hold the gradient to add to). */
int stg_edge_dot_bwd_f32(const float* z, int32_t feat, const int64_t* a, const int64_t* b, int64_t n_pairs,
                         const float* grad_out, float* d_z, void* stream);

/* --------------------------------------------------- graph structure ops */
/* ------------------------------------------------- TGCN (GRU) cell, element-wise */
/* The element-wise pieces of the TGCN cell (stgraph/nn/pytorch/temporal/tgcn.py:21-47) as three fused passes
 * forward and three backward; the GEMMs between them stay cuBLAS.  All tensors are contiguous fp32 with n elements
 * ([N, H] flattened) unless stated.
 *   bias_clamp : a[r, c] = clamp(a[r, c] + bias[c], lo, hi) in place (bias may be NULL) -- GCNConv's bias add
 *                (gcn_conv.py:184-186) and the cell's clamp(+-1e6) (tgcn.py:23) on the [N, 3H] aggregation output;
 *   clamp_bwd  : d_a = d_y where lo < y < hi, else 0 (y = the clamped value);
 *   reset      : hr = h * sigmoid(pr)                         (tgcn.py:33-41: R, then H * R for the candidate state)
 *   update     : out = z * h + (1 - z) * tanh(ph), z = sigmoid(pz)                                  (tgcn.py:43-47)
 * The backward entry points recompute the activations from the pre-activations. */
int stg_bias_clamp_f32(float* a, const float* bias, int64_t rows, int32_t cols, float lo, float hi, void* stream);
int stg_clamp_bwd_f32(const float* y, const float* d_y, float* d_a, int64_t n, float lo, float hi, void* stream);
int stg_gru_reset_fwd_f32(const float* pr, const float* h, float* hr, int64_t n, void* stream);
int stg_gru_reset_bwd_f32(const float* pr, const float* h, const float* d_hr, float* d_pr, float* d_h, int64_t n,
                          void* stream);
int stg_gru_update_fwd_f32(const float* pz, const float* ph, const float* h, float* out, int64_t n, void* stream);
int stg_gru_update_bwd_f32(const float* pz, const float* ph, const float* h, const float* d_out, float* d_pz,
                           float* d_ph, float* d_h, int64_t n, void* stream);
/* The same gate arithmetic on the block layout of the one-Function cell (stgraph_b200/ops_tgcn.py): p and d_p are
 * [rows, 3*hid] row-major holding the gate pre-activations as column blocks (z | r | h); h, hr, out, d_out, d_hr, d_h are
 * [rows, hid].  update_bwd writes the z and h blocks of d_p and d_h = d_out * z; reset_bwd writes the r block of d_p and
 * ADDS d_hr * r to d_h (call it after update_bwd). */
int stg_tgcn_reset_fwd_f32(const float* p, const float* h, float* hr, int64_t rows, int32_t hid, void* stream);
int stg_tgcn_reset_bwd_f32(const float* p, const float* h, const float* d_hr, float* d_p, float* d_h, int64_t rows,
                           int32_t hid, void* stream);
int stg_tgcn_update_fwd_f32(const float* p, const float* h, float* out, int64_t rows, int32_t hid, void* stream);
int stg_tgcn_update_bwd_f32(const float* p, const float* h, const float* d_out, float* d_p, float* d_h, int64_t rows,
                            int32_t hid, void* stream);
/* The 16-bit cell (torch.autocast): the tensors that only feed GEMMs are stored as bf16 / fp16 (dtype, StgDtype), the
 * rest stays fp32; the arithmetic is the fp32 entry points', in fp32, and a value is rounded once, when it is stored.
 *   bias_clamp_h16 : y = clamp(a + bias[c], lo, hi) with a and y [rows, cols] 16-bit, bias fp32 (may be NULL); y may be a;
 *   clamp_bwd_h16  : d_a = d_y where lo < a + bias[c] < hi in fp32, else 0 (a, d_y, d_a 16-bit; d_a may be d_y) -- the
 *                    fp32 cell's mask on the unrounded clamp input, which the rounded y cannot give (bf16: 1e6 -> 999424);
 *   reset_fwd_h16  : stg_tgcn_reset_fwd_f32 with a 16-bit hr;
 *   reset_bwd_h16, update_bwd_h16 : the fp32 entry points, and the blocks of d_p they write once more, rounded, into the
 *                    16-bit [rows, 3*hid] d_p16. */
int stg_tgcn_bias_clamp_h16(const void* a, const float* bias, void* y, int64_t rows, int32_t cols, int32_t dtype, float lo,
                            float hi, void* stream);
int stg_tgcn_clamp_bwd_h16(const void* a, const float* bias, const void* d_y, void* d_a, int64_t rows, int32_t cols,
                           int32_t dtype, float lo, float hi, void* stream);
int stg_tgcn_reset_fwd_h16(const float* p, const float* h, void* hr, int64_t rows, int32_t hid, int32_t dtype, void* stream);
int stg_tgcn_reset_bwd_h16(const float* p, const float* h, const float* d_hr, float* d_p, void* d_p16, float* d_h,
                           int64_t rows, int32_t hid, int32_t dtype, void* stream);
int stg_tgcn_update_bwd_h16(const float* p, const float* h, const float* d_out, float* d_p, void* d_p16, float* d_h,
                            int64_t rows, int32_t hid, int32_t dtype, void* stream);

/* Weight-gradient GEMM of the cell: C[K, Nc] = A[M, K]^T * B[M, Nc] in exact fp32 for M >> K, Nc (what torch autograd
 * computes with cuBLAS for the gradients of conv_*.weight and linear_*.weight, tgcn.py:16-47), and, if colsum_b is not
 * NULL, colsum_b[Nc] = column sums of B (the bias gradient).  A and B are row-major with leading dimensions lda >= K,
 * ldb >= Nc (column blocks of wider matrices are fine); C is contiguous.  The M rows are split into slabs whose partial
 * results are summed in slab order (deterministic); workspace: stg_gemm_tn_workspace_bytes(M, K, Nc) bytes (0 for small
 * M: pass NULL). */
size_t stg_gemm_tn_workspace_bytes(int64_t M, int32_t K, int32_t Nc);
int stg_gemm_tn_f32(const float* A, int64_t lda, const float* B, int64_t ldb, int64_t M, int32_t K, int32_t Nc, float* C,
                    float* colsum_b, void* workspace, size_t workspace_bytes, void* stream);

/* Workspace needed by stg_csr_build for E edges / N nodes. */
size_t stg_csr_build_workspace_bytes(int64_t num_edges, int32_t num_nodes);

/* Builds both directions of a static graph on the GPU from an (unsorted) edge list.
 *   forward : rows = dst, sorted by (dst,src); fwd_eids[i] = i
 *   backward: rows = src, sorted by (src,dst); bwd_eids = forward eid of each edge
 *   in_degree / out_degree [N]; fwd/bwd node_ids [N] = rows by non-increasing length
 *   (stable, ascending id within a tie).
 * edge_perm [E] (optional): edge_perm[i] = position in the caller's list of the
 * edge that received forward eid i (lets callers permute their edge weights).
 * num_unique (optional, device int32): number of distinct (src,dst) pairs
 * (static_graph.py:49 sizes edge tensors by len(set(edge_list))).
 * Replaces the host loop + 4 cudaMemcpy of CSR::CSR
 * (stgraph/graph/static/csr.cu:68-170) and the Python tuple sorts of
 * stgraph/graph/static/static_graph.py:65-78. */
int stg_csr_build(const int32_t* src, const int32_t* dst, int64_t num_edges, int32_t num_nodes,
                  int32_t* fwd_row_offset, int32_t* fwd_col, int32_t* fwd_eids, int32_t* fwd_node_ids,
                  int32_t* bwd_row_offset, int32_t* bwd_col, int32_t* bwd_eids, int32_t* bwd_node_ids,
                  int32_t* in_degree, int32_t* out_degree, int32_t* edge_perm, int32_t* num_unique,
                  void* workspace, size_t workspace_bytes, void* stream);

/* norm[v] = deg[v] > 0 ? deg[v]^-0.5 : 0   (benchmarking/gcn/seastar/train.py:53-57) */
int stg_degree_norm_f32(const int32_t* degree, int32_t num_nodes, float* norm, void* stream);

/* weighted_degree[r] = sum over row r of w[eid]  (csr.cu:126, fp32, row order) */
int stg_weighted_row_degree_f32(const StgCsrView* g, const float* edge_weight, float* out, void* stream);

/* hub_rows = { r : row length > threshold }, *hub_count = how many (clamped to capacity). */
int stg_csr_hub_rows(const int32_t* row_offset, int32_t num_nodes, int32_t threshold,
                     int32_t* hub_rows, int32_t capacity, int32_t* hub_count, void* stream);

/* ------------------------------------------------ dynamic-graph snapshots */
/* A snapshot is the sorted array of its live edge keys (dst<<32 | src), i.e. a packed memory array
 * without gaps; see csrc/snapshot.cu for why that is the B200 design.  All counts are written to
 * DEVICE memory (int64) so that nothing synchronises; callers that know the sizes from
 * preprocessing never read them back. */
size_t stg_snapshot_workspace_bytes(int64_t max_items);

/* keys_out = sorted, de-duplicated keys of an edge list (dynamic_graph.py:58-63 set()). */
int stg_snapshot_keys_from_edges(const int32_t* src, const int32_t* dst, int64_t n, int32_t num_nodes,
                                 uint64_t* keys_out, int64_t* count_out, void* ws, size_t ws_bytes, void* stream);

/* out = a \ b for sorted unique key arrays: the per-timestamp "add" / "delete" lists
 * (dynamic_graph.py:66-79). */
int stg_snapshot_diff(const uint64_t* a, int64_t na, const uint64_t* b, int64_t nb, uint64_t* out,
                      int64_t* count_out, void* ws, size_t ws_bytes, void* stream);

/* out = (keys \ del) U add -- one batched insert/delete step (gpma.cu:1064-1119 edge_update_t /
 * pcsr.cu:658-717 edge_update_list); swap add/del to revert a timestamp. out needs n + na slots. */
int stg_snapshot_apply(const uint64_t* keys, int64_t n, const uint64_t* add, int64_t na, const uint64_t* del,
                       int64_t nd, uint64_t* out, int64_t* count_out, void* ws, size_t ws_bytes, void* stream);

/* Labelled CSR views of a snapshot: forward (rows = dst) and, if bwd_row_offset != NULL, backward
 * (rows = src, dense transpose carrying the forward labels; gpma.cu:1165-1231, pcsr.cu:794-809).
 * label = label_base + rank among live keys (1 for PCSR/GPMA, 0 for NaiveGraph).
 * descending_rows != 0 emits every row back to front (PCSR, pcsr.cu:842-855).
 * node_ids / degree outputs may be NULL. ws must hold max(n, num_nodes) items. */
int stg_snapshot_views(const uint64_t* keys, int64_t n, int32_t num_nodes, int32_t descending_rows, int32_t label_base,
                       int32_t* fwd_row_offset, int32_t* fwd_col, int32_t* fwd_labels, int32_t* fwd_node_ids,
                       int32_t* bwd_row_offset, int32_t* bwd_col, int32_t* bwd_labels, int32_t* bwd_node_ids,
                       int32_t* in_degree, int32_t* out_degree, void* ws, size_t ws_bytes, void* stream);

/* D2H copy of an int32 device array -- test hook (csr.cu:172-179 get_array). */
int stg_get_array_i32(const int32_t* dev_ptr, int64_t count, int32_t* host_out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* STGRAPH_B200_H_ */
