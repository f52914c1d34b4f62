/*
 * liblkg -- C ABI of the B200-native LiteralKG message-passing + scoring path.
 *
 * The reference (NSLab-CUK/LiteralKG) is pure Python/PyTorch and has no FFI of its own
 * (SURVEY.md 8(b)); the drop-in surface is the Python class API of model.py / gate.py /
 * dataloader.py.  This header is the boundary underneath that surface: every entry point below
 * replaces the body of one reference function (cited as file:line next to it) and is what a
 * maintainer binds with ctypes (see INTEGRATION.md).
 *
 * Conventions
 *   - plain C: pointers + sizes only, no C++ / torch types;
 *   - every function returns an lkg_status (0 = ok, < 0 = error); lkg_last_error() gives the
 *     thread-local message of the last failure;
 *   - all pointers are DEVICE pointers unless a parameter is documented as "host";
 *   - buffers are borrowed for the duration of the call: the library never allocates, frees or
 *     retains device memory (callers size scratch with the *_workspace_bytes queries);
 *   - `stream` is a cudaStream_t passed as void*; calls are asynchronous w.r.t. the host unless
 *     documented otherwise.  A graph plan (lkg_graph) carries device scratch its kernels mutate during a
 *     launch (row counter, seg_tickets, seg_scratch): ONE plan may be used by ONE stream at a time.  The only
 *     process-wide state is the error string (thread local) and the lkg_gemm_set_cta_group tuning knob;
 *   - row-major matrices; `ld*` arguments are leading dimensions in ELEMENTS;
 *   - sm_100 only: there is no CPU or other-architecture fallback by design.
 */
#ifndef LKG_H_
#define LKG_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LKG_ABI_VERSION 8

typedef enum {
    LKG_OK = 0,
    LKG_ERR_INVALID = -1,      /* bad argument / shape / alignment */
    LKG_ERR_UNSUPPORTED = -2,  /* shape outside the compiled kernel envelope */
    LKG_ERR_CUDA = -3,         /* CUDA runtime / launch failure (message has the cudaError) */
    LKG_ERR_ARCH = -4,         /* device is not sm_100 */
    LKG_ERR_WORKSPACE = -5     /* workspace too small */
} lkg_status;

/* CSR plan of the knowledge graph, all arrays int32, built once per edge list by lkg_plan_build.
 *   "att" order: the E kept triples sorted by (head, relation, tail); used by the attention update,
 *                where tanh(e_h + e_r) is shared by a whole (head, relation) run;
 *   "agg" order: the nnz UNIQUE (head, tail) pairs sorted by (head, tail) == the coalesced A_in of
 *                the reference (model.py:466-471); att_seg maps every triple to its pair. */
typedef struct {
    int64_t n_entities;
    int64_t n_edges;            /* E   : triples kept (relation filter applied)            */
    int64_t nnz;                /* E'  : unique (h,t) pairs                                  */
    int32_t n_relations;
    int64_t row_begin;          /* kernels process head rows [row_begin, row_end): the row partition */
    int64_t row_end;            /* owned by this rank (0, N on a single GPU)                          */
    const int32_t* att_rowptr;  /* [N+1] */
    const int32_t* att_tail;    /* [E]   */
    const int32_t* att_rel;     /* [E]   */
    const int32_t* att_seg;     /* [E]   bits 0-30: index into the agg arrays; bit 31: the pair has several triples */
    const int32_t* rowptr;      /* [N+1] */
    const int32_t* col;         /* [nnz] */
    const int32_t* row_order;   /* [row_end - row_begin] the rows of the partition, most triples first: the
                                   kernels take rows in this order so that the heaviest rows of a power-law
                                   graph start first (nullable: natural order) */
    const int32_t* row_sched;   /* [row_end - row_begin][8] the same order as 32-byte records {row, att_rowptr[row],
                                   att_rowptr[row+1], rowptr[row], rowptr[row+1], 0, 0, 0} (required by
                                   lkg_attn_update; 16-byte aligned) */
    int64_t n_solo_rows;        /* leading rows of row_order with more than LKG_SOLO_DEGREE triples (0 = unknown): the
                                   narrow-row aggregation kernel gives each of them a warp of its own */
    /* Segmented heavy rows.  A row with more than LKG_SEG_DEGREE triples may appear in row_sched as nseg <= LKG_MAX_SEGS
     * records {row, att sub-range, agg sub-range, nseg, ticket, segment index}: different warps process the pieces, a
     * per-row ticket counter elects the last one to finish the row (softmax / combine).  Records of ordinary rows have
     * nseg == 0.  The host side builds the expanded schedule (graph.py); n_sched == 0 means "one record per row". */
    int64_t n_sched;            /* records in row_sched */
    int32_t* seg_tickets;       /* [number of segmented rows] zero between launches (the electing warp resets it) */
    float* seg_scratch;         /* [segmented rows * LKG_MAX_SEGS][seg_stride] partial sums of the aggregation kernel */
    int64_t seg_stride;         /* floats per scratch slot (>= d_in + d_out) */
} lkg_graph;
#define LKG_SOLO_DEGREE 256
#define LKG_SEG_DEGREE 512
#define LKG_MAX_SEGS 8

/* fp16 "planes" operand of the tensor-core GEMMs.  A value x is stored as hi = fp16(s*x) and
 * lo = fp16(s*x - hi): two fp16 matrices [rows, ld] that are `plane_stride` elements apart (hi first), 22
 * significand bits in the footprint of the fp32 value.  s is a power of two kept in a device "scale
 * record" (below) that parks max|s*x| in [2^11, 2^12), far from fp16's overflow and subnormal ranges.
 * An operand is a K-concatenation of up to LKG_MAX_SEGMENTS such matrices (the virtual torch.cat of
 * gate.py:23 / model.py:309): logical A[m, :] = [ seg0[m, 0:k0] | seg1[m, 0:k1] | ... ].
 * Base pointers, row strides and plane strides must be 16-byte aligned (ld % 8 == 0). */
#define LKG_MAX_SEGMENTS 4
/* Scale record: device float[LKG_SCALE_FLOATS] = { absmax, scale, 1/scale, (scratch) ... }; written by
 * lkg_scale_from_data / lkg_scale_from_bound / lkg_pack_weight, read by every kernel that writes or
 * multiplies planes.  Never read by the host: no call of this library synchronises. */
#define LKG_SCALE_FLOATS 8
typedef struct {
    int32_t n_segments;
    const uint16_t* ptr[LKG_MAX_SEGMENTS];
    int64_t ld[LKG_MAX_SEGMENTS];
    int64_t plane_stride[LKG_MAX_SEGMENTS];
    int32_t k[LKG_MAX_SEGMENTS];
    const float* scale[LKG_MAX_SEGMENTS];   /* scale record of each segment (device) */
} lkg_planes;

typedef enum {
    LKG_ACT_NONE = 0,
    LKG_ACT_LEAKY_RELU = 1,
    LKG_ACT_TANH = 2,
    LKG_ACT_ACCUMULATE = 256 /* flag, OR-ed in: out += act(result) (gradient accumulation of the backward pass) */
} lkg_activation;
typedef enum { LKG_AGG_GCN = 0, LKG_AGG_GRAPHSAGE = 1, LKG_AGG_BI_INTERACTION = 2 } lkg_aggregator;

/* ---- library ------------------------------------------------------------------------------ */
int lkg_abi_version(void);
const char* lkg_last_error(void);
/* LKG_OK iff `device` is an sm_100 GPU (B200).  Host call. */
int lkg_device_check(int device);

/* Stores `nbytes` (multiple of 16) of local device memory into n_dst <= 8 destinations that are PEER-mapped device
 * pointers (the same block of every peer's copy of a symmetric-memory exchange table) with one kernel on n_ctas CTAs:
 * every 16-byte vector is loaded once and stored over NVLink to all destinations.  dst: HOST array of device pointers.
 * Completion is stream ordered; visibility at the peers needs the caller's cross-rank barrier afterwards. */
int lkg_peer_push(const void* src, int64_t nbytes, void* const* dst /*host array*/, int32_t n_dst, int32_t n_ctas,
                  void* stream);

/* ---- graph plan: replaces DataLoader.construct_data's tensor products + the coalesce/sort that
 *      torch.sparse.softmax performs inside update_attention (dataloader.py:369-424,
 *      model.py:462-470) ------------------------------------------------------------------------ */
int lkg_plan_workspace_bytes(int64_t n_edges, int64_t n_entities, size_t* bytes /*host out*/);
/* h,t,r: int64 [n_edges] in file order.  row_order (nullable) int32 [n_entities]: all rows by decreasing
 * triple count (stable); row_sched (nullable) int32 [n_entities][8]: the schedule records of lkg_graph.  rel_keep: optional uint8 [n_relations]; triples whose
 * relation has rel_keep == 0 are dropped (a `relations` list that omits ids, model.py:451).
 * Outputs are caller-allocated: att_* and col sized for n_edges, rowptrs for n_entities+1,
 * coo_rows/coo_cols (nullable) int64 [n_edges] receive the coalesced COO indices, file_seg
 * (nullable) int32 [n_edges] receives for every INPUT triple the index of its (h,t) pair (-1 if
 * dropped), counts_dev int64[3] receives {E kept, nnz, number of out-of-range ids (must be 0)}. */
int lkg_plan_build(const int64_t* h, const int64_t* t, const int64_t* r, int64_t n_edges,
                   int64_t n_entities, int32_t n_relations, const uint8_t* rel_keep,
                   int32_t* att_rowptr, int32_t* att_tail, int32_t* att_rel, int32_t* att_seg,
                   int32_t* rowptr, int32_t* col, int32_t* row_order, int32_t* row_sched, int64_t* coo_rows,
                   int64_t* coo_cols,
                   int32_t* file_seg, int64_t* counts_dev, void* workspace, size_t workspace_bytes,
                   void* stream);
/* values_out[file_seg[i]] += values_in[i]: imports an un-coalesced COO value list (e.g. an A_in taken
 * from a checkpoint, model.py:257-261) into plan order, summing duplicates like coalesce(). */
int lkg_segment_scatter_add(const float* values_in, const int32_t* file_seg, int64_t n_edges,
                            float* values_out, int64_t nnz, void* stream);

/* Order-independent 128-bit fingerprint of an edge list (fp_dev: uint64[2], zeroed by the call); used by
 * the host side to recognise an unchanged (h, t, r) list and reuse its plan across update_att calls. */
int lkg_edge_fingerprint(const int64_t* h, const int64_t* t, const int64_t* r, int64_t n_edges,
                         uint64_t* fp_dev, void* stream);

/* Initial A_in = sum_r D_r^-1 A_r (random-walk) or D_r^-1/2 A_r D_r^-1/2 (symmetric, row sums on
 * both sides), float64 accumulation then fp32 cast (dataloader.py:449-495).  values: [nnz];
 * scratch: float64 [nnz] accumulator. */
int lkg_laplacian_init(const lkg_graph* g, int symmetric, float* values, double* scratch, void* stream);

/* ---- attention update (model.py:430-471): per triple v = sum_d e_t[d]*tanh(e_h[d]+e_r[d]) on the
 *      raw tables, duplicate (h,t) logits summed, max-subtracted softmax per head row.
 *      values: [nnz] in agg order. ------------------------------------------------------------ */
int lkg_attn_workspace_bytes(int32_t n_relations, int32_t dim, size_t* bytes /*host out*/);
int lkg_attn_update(const lkg_graph* g, const float* entity, int64_t ld_entity,
                    const float* relation, int64_t ld_relation, int32_t dim,
                    float* values, void* workspace, void* stream);

/* ---- relation-projected attention (north star (b); the formula the reference keeps commented out, model.py:436-439):
 *      v(h,r,t) = (e_t W_r) . tanh(e_h W_r + e_r).  Because the tanh factor only depends on (h, r), v = e_t . u_{h,r}
 *      with u_{h,r} = W_r tanh(W_r^T e_h + e_r): the two projections run once per (head, relation) RUN of the att
 *      order, bucketed by relation, as two chained tensor-core GEMMs (lkg_split_planes with the run heads as row
 *      gather -> lkg_linear_fwd with LKG_ACT_TANH writing planes -> lkg_linear_fwd), and the per-triple work is the
 *      same 1 200-byte tail-row gather as lkg_attn_update:
 *   lkg_attn_run_logits  logits[e] = entity[att_tail[e]] . run_w[run_slot[run]] for every triple e of every run
 *                        (run_ptr [n_runs + 1]: the runs' triple ranges in att order; run_w [n_runs, dim] fp32);
 *   lkg_row_softmax      in-place max-subtracted softmax of values[rowptr[i] : rowptr[i + 1]] for every row (after the
 *                        duplicate (h,t) logits were summed with lkg_segment_scatter_add). */
int lkg_attn_run_logits(const int32_t* run_ptr, const int32_t* run_slot, int64_t n_runs, const int32_t* att_tail,
                        const float* entity, int64_t ld_entity, int32_t dim, const float* run_w, int64_t ld_w,
                        float* logits, void* stream);
int lkg_row_softmax(const int32_t* rowptr, int64_t n_rows, float* values, void* stream);

/* ---- dense: C[M,N] = epilogue(A[M,K] @ B[N,K]^T) on tcgen05 tensor cores, three fp16 products per
 *      k-step (hi*hi + lo*hi + hi*lo) accumulated in fp32 TMEM (torch Linear layout: B is [out, in]) ---- */
/* rec <- record of max(|src[rows or all, 0:k]|, floor).  src fp32 [*, ld], optional int64 row gather. */
int lkg_scale_from_data(const float* src, int64_t ld, const int64_t* rows /*nullable*/, int64_t m, int32_t k,
                        float floor, float* rec, void* stream);
/* Records built by the kernels that PRODUCE a matrix (no pass re-reads it): zero a float[LKG_SCALE_FLOATS], hand it to
 * the producers' `amax` arguments (lkg_leaky_bwd, lkg_layer_bwd_rows, lkg_bi_bwd_rows, lkg_gate_bwd) and / or raise it
 * with lkg_absmax_accumulate for the parts other kernels wrote, then lkg_scale_finish(floor, rec) turns element 0 into
 * the record of max(element 0, floor).  A record only has to BOUND its data: every factor of two of slack costs one of
 * the 36 bits the hi/lo pair resolves below the bound. */
int lkg_absmax_accumulate(const float* src, int64_t ld, const int64_t* rows /*nullable*/, int64_t m, int32_t k,
                          float* rec, void* stream);
int lkg_scale_finish(float floor, float* rec, void* stream);
/* rec <- record of max(bound, other[0]) where `other` is an optional existing record (e.g. the gate output
 * is bounded by max(1, max|entity|): a convex mix of the entity row and a tanh). */
int lkg_scale_from_bound(float bound, const float* other /*nullable*/, float* rec, void* stream);
/* fp32 [m, k] (row stride ld, optional row gather) -> planes [2][m][ld_planes] scaled by rec, columns >= k
 * zero filled. */
int lkg_split_planes(const float* src, int64_t ld, const int64_t* rows /*nullable*/, int64_t m, int32_t k,
                     const float* rec, uint16_t* planes, int64_t ld_planes, int64_t plane_stride, void* stream);
/* Number of columns of a packed weight: every K segment is padded to a multiple of 64. Host call. */
int lkg_packed_weight_cols(const int32_t* seg_k /*host*/, int32_t n_segments, int32_t* cols /*host out*/);
/* fp32 weight [n, sum(seg_k)] -> fp16 hi/lo planes [2][n][packed cols] with per-segment zero padding.
 * a_recs (host array of n_segments device pointers): the scale records of the A segments this weight will
 * meet; segment i of the weight is scaled by S / a_scale_i with one power of two S chosen so that the
 * largest scaled weight lands in [2^11, 2^12): every product of the GEMM then carries the same factor S,
 * and w_rec receives {., S, 1/S} for the epilogue. */
int lkg_pack_weight(const float* w, int64_t ldw, int32_t n, const int32_t* seg_k /*host*/, int32_t n_segments,
                    const float* const* a_recs /*host array of device ptrs*/, uint16_t* planes,
                    int64_t plane_stride, float* w_rec, void* stream);
/* out = act(A @ B^T + bias)  (linear_gat model.py:309-310; the h0 @ Q residual terms).  b: packed weight
 * planes (one segment descriptor whose k is the packed column count and whose scale is w_rec).
 * out_planes (nullable) receives the split of the result scaled by out_rec for a following GEMM. */
int lkg_linear_fwd(const lkg_planes* a, int64_t m, const lkg_planes* b, int32_t n,
                   const float* bias /*nullable [n]*/, int32_t activation, float* out, int64_t ldo,
                   uint16_t* out_planes, int64_t ld_planes, int64_t plane_stride, const float* out_rec,
                   void* stream);
/* The same GEMM with two destinations: columns [0, split_col) go to out, columns [split_col, n) to
 * out2[row * ld2 + col - split_col] (split_col a multiple of 4).  The stacked h0 @ Q GEMM writes layer 1's pre-projected
 * sum term z straight into the [h0 | z] table the aggregation gathers from (no copy between the two layouts). */
int lkg_linear_fwd_split(const lkg_planes* a, int64_t m, const lkg_planes* b, int32_t n,
                         const float* bias /*nullable [n]*/, int32_t activation, float* out, int64_t ldo,
                         float* out2 /*nullable*/, int64_t ld2, int32_t split_col,
                         uint16_t* out_planes, int64_t ld_planes, int64_t plane_stride, const float* out_rec,
                         void* stream);
/* Tuning / test knob of the GEMM engine (host call, process wide): 0 = automatic (a CTA pair issuing
 * tcgen05.mma.cta_group::2 over 256-row tiles whenever there is a tile for every SM pair, else one CTA per 128-row
 * tile), 1 / 2 = force the CTA-group size.  Results are bit-identical either way (same products, same order). */
int lkg_gemm_set_cta_group(int32_t cta_group);
/* Literal gate (gate.py:22-28 / :45-51).  x = (entity | literals...) planes; w_pair = packed planes of
 * the [2*dim, K] matrix with row 2j = g.weight[j,:] and row 2j+1 = the stacked gate_* weights of output
 * j; bias_pair [2*dim] likewise (g.bias[j], gate_bias[j]); x_ent = fp32 entity table for the mix
 * out = (1 - z) * x_ent + z * tanh(g).  gz_out (nullable, training): the activated pairs
 * (tanh g_j, sigmoid z_j) interleaved like w_pair's rows, [m, 2*dim], saved for lkg_gate_bwd. */
int lkg_gate_fwd(const lkg_planes* x, int64_t m, const lkg_planes* w_pair, const float* bias_pair,
                 int32_t dim, const float* x_ent, int64_t ld_ent, float* out, int64_t ldo,
                 uint16_t* out_planes, int64_t ld_planes, int64_t plane_stride, const float* out_rec,
                 float* gz_out, int64_t ld_gz, void* stream);

/* ---- one aggregator layer, forward (model.py:101-164 + F.normalize of model.py:305) ----------
 * side = A_in @ ego fused with the combine, LeakyReLU, LayerNorm, optional dropout mask and the
 * L2-normalised copy for the concat buffer.  The residual connection (model.py:90-99) and the
 * Linear layers are passed FOLDED (see DESIGN.md section 4):
 *     o1 = ego @ Pa + side @ Pb + r1[row]          (Pa may be NULL: term folded into r1)
 *     o2 = (ego * side) @ P2 + r2[row]             (bi-interaction only, P2 non-NULL)
 *     emb = leaky(o1) (+ leaky(o2));  x = LayerNorm(emb) * mask;  xn = x / max(|x|_2, 1e-12)
 * Pa, Pb, P2: [d_in, d_out] row-major.  r1/r2: per-row terms with leading dimension ld_r
 * (ld_r == 0 broadcasts one [d_out] vector, i.e. a plain bias).
 * Envelope: d_in % 4 == 0, d_in <= 512, d_out <= 64, and the chosen kernel's shared memory within 227 KB.  The
 * two-matrix modes (Pa != Pb, or P2) keep both [d_in, d_out] tiles in shared memory: at d_in >= 404 they need
 * d_out <= 60.  The pre-projected z mode runs on the wide-row stream kernel only, which exists for
 * ceil(d_in / 128) in {1, 2, 3, 4} with d_out <= 32 and for ceil(d_in / 128) == 3 with d_out <= 64, within the same
 * shared-memory limit (e.g. not at d_in = 256 with d_out > 32, nor at d_in = 300 with d_out >= 56).  lkg_aggregate_supported tells
 * which shapes run. */
typedef enum {
    LKG_AGG_MODE_ONE_TERM = 0,   /* P2 NULL, Pa NULL or Pa == Pb */
    LKG_AGG_MODE_TWO_TERMS = 1,  /* P2 NULL, Pa != Pb */
    LKG_AGG_MODE_BI = 2,         /* P2 given, z NULL */
    LKG_AGG_MODE_BI_Z = 3        /* P2 and z given */
} lkg_agg_mode;
/* *ok = 1 iff lkg_aggregate_fwd runs (d_in, d_out) in `mode` with 16-byte aligned operands and a plan that has a row
 * schedule (every plan of lkg_plan_build), 0 if it refuses the shape.  Host call, no device needed. */
int lkg_aggregate_supported(int32_t d_in, int32_t d_out, int32_t mode, int32_t* ok /*host out*/);
int lkg_aggregate_workspace_bytes(size_t* bytes /*host out*/);
int lkg_aggregate_fwd(const lkg_graph* g, const float* a_values, const float* ego, int64_t ld_ego,
                      int32_t d_in, int32_t d_out, const float* pa, const float* pb, const float* p2,
                      const float* r1, const float* r2, int64_t ld_r,
                      const float* ln_weight, const float* ln_bias,
                      const float* drop_mask /*nullable [N,d_out] multiplicative*/,
                      float* x_out, int64_t ld_x, float* xn_out /*nullable*/, int64_t ld_xn,
                      uint16_t* xn_planes /*nullable: hi/lo copy of xn*/, int64_t ld_planes, int64_t plane_stride,
                      const float* xn_rec /*scale record of xn_planes (bound 1)*/,
                      int64_t local_row_base /*r1, r2, drop_mask, xn_out, xn_planes hold rows [local_row_base, ...):
                                               the row partition's local buffers (0 on one GPU); ego and x_out
                                               are indexed by the global row*/,
                      const float* z /*nullable*/, int64_t ld_z /*pre-projected sum term of the bi-interaction
                                               layer: z = ego @ Pb [N, d_out], e.g. extra columns of the h0 @ Q GEMM;
                                               then o1 = r1[row] + sum_j A[row,j] z[col_j], pa = pb = NULL, and
                                               only P2 is combined in the kernel (wide rows only)*/,
                      float* o_out /*nullable, training: pre-activations [o1 | o2] of every local row*/, int64_t ld_o,
                      float* side_out /*nullable, training: side = A @ ego of every local row*/, int64_t ld_side,
                      void* workspace, void* stream);

/* ---- backward of the embedding pass (what loss.backward() replays through model.py:298-314) -------------
 * Transposed plan: the nnz (head, tail) pairs sorted by (tail, head) as a COO list; t_perm[i] = position of the
 * pair in agg order (index of its A_in value).  Stable radix sort: bit-exact, deterministic. */
int lkg_plan_transpose_workspace_bytes(int64_t nnz, size_t* bytes /*host out*/);
int lkg_plan_transpose(const lkg_graph* g, int32_t* t_tail, int32_t* t_head, int32_t* t_perm,
                       void* workspace, size_t workspace_bytes, void* stream);
/* out[seg[i], :] += vals[perm ? perm[i] : i] * x[src[i], :] over a COO list sorted by seg (segmented reduction,
 * equal nnz per worker).  With (t_tail, t_head, t_perm) this is out += A_in^T @ x: the backward of torch.sparse.mm
 * (model.py:106).  d % 4 == 0, d <= 512. */
int lkg_spmm_coo(const int32_t* seg, const int32_t* src, const int32_t* perm /*nullable*/, const float* vals,
                 int64_t nnz, const float* x, int64_t ldx, int32_t d, float* out, int64_t ldo, void* stream);
/* Row-local backward of one aggregator layer (model.py:108-130, 161-164 and F.normalize of :305):
 *   dy = dy_in + d normalize(y)^T dyn;  dropout mask;  LayerNorm backward;  LeakyReLU backward of both paths.
 * y: the layer output, o: the pre-activations saved by lkg_aggregate_fwd ([o1 | o2], has_o2 for
 * bi-interaction).  Writes d_o = [do1 | do2] and ACCUMULATES dgamma_dbeta[2*c] (LayerNorm weight / bias).
 * amax / amax2 (nullable): scale records under construction (zeroed float[LKG_SCALE_FLOATS]) whose element 0 is raised
 * to max|d_o| -- see lkg_scale_finish. */
int lkg_layer_bwd_rows(int64_t n, int32_t c, int32_t has_o2, const float* y, int64_t ld_y, const float* o,
                       int64_t ld_o, const float* mask /*nullable [n, c]*/, const float* dy_in /*nullable*/,
                       int64_t ld_dy, const float* dyn /*nullable*/, int64_t ld_dyn, const float* ln_weight,
                       float* d_o, int64_t ld_do, float* dgamma_dbeta, float* amax, float* amax2, void* stream);
/* Product path of bi-interaction (model.py:127-128): V = do2 @ P2^T;  w_out = V * x (the operand of the
 * A^T gather);  dx (+)= V * side;  xs_out (nullable) = x * side, the row operand of d P2 = (x * side)^T do2;
 * xs_amax (nullable): record under construction raised to max|xs_out|. */
int lkg_bi_bwd_rows(int64_t n, int32_t d, int32_t c, const float* d_o2, int64_t ld_do, const float* p2 /*[d, c]*/,
                    const float* x, int64_t ld_x, const float* side, int64_t ld_side, float* w_out, int64_t ld_w,
                    float* dx, int64_t ld_dx, int32_t accumulate, float* xs_out, int64_t ld_xs, float* xs_amax,
                    void* stream);
/* Parameter gradients: out[i, j] += sum_rows x[row, i] * (x2 ? x2[row, i] : 1) * y[row, j]; x == NULL with dx == 1
 * gives the column sums of y (bias gradients).  out [dx, cy] is accumulated into (zero it first). */
int lkg_xt_y(const float* x /*nullable*/, int64_t ld_x, const float* x2 /*nullable*/, int64_t ld_x2, int32_t dx,
             const float* y, int64_t ld_y, int32_t cy, int64_t n, float* out, int64_t ld_out, void* stream);
/* The same reduction on the tensor cores: out[dx, cy] += x^T y with both operands given as fp16 hi/lo planes
 * ([n_rows, k] row-major, single segment; the planes the forward GEMMs already use).  MN-major tcgen05 operands,
 * split over row ranges, fp32 atomics into out. */
int lkg_xt_y_planes(const lkg_planes* x, const lkg_planes* y, int64_t n_rows, float* out, int64_t ld_out, void* stream);
/* out[j] += sum_rows y[row, j]  (bias gradients). */
int lkg_colsum(const float* y, int64_t ld_y, int64_t n, int32_t c, float* out, void* stream);
/* Literal gate backward, elementwise part (gate.py:22-28): from dh = d loss / d out and the saved (g, z) pairs:
 * d_pre (interleaved like w_pair's rows) and the direct entity term d_ent = dh * (1 - z); pre_amax (nullable):
 * record under construction raised to max|d_pre|. */
int lkg_gate_bwd(const float* dh, int64_t ld_dh, const float* gz, int64_t ld_gz, const float* ent, int64_t ld_ent,
                 int64_t n, int32_t dim, float* d_pre, int64_t ld_pre, float* d_ent, int64_t ld_de, float* pre_amax,
                 void* stream);
/* d_pre = grad * LeakyReLU'(out) from the activated output (model.py:311); amax (nullable): record under
 * construction raised to max|d_pre|. */
int lkg_leaky_bwd(const float* grad, int64_t ld_g, const float* out, int64_t ld_out, int64_t n, int32_t c,
                  float* d_pre, int64_t ld_d, float* amax, void* stream);

/* ---- loss heads of the training modes: value and gradients over one minibatch ---------------------------------
 * Both losses are batch means (+ l2_lambda * the reference's _L2_loss_mean terms).  `loss` (nullable) is a device
 * scalar ACCUMULATED into (zero it first); the gradient buffers (nullable: forward only) are accumulated into as
 * well; grad_scale (nullable = 1) is the upstream d / d loss as a device scalar, so no call synchronises. */
/* calculate_prediction_loss (model.py:316-348): BPR, -log sigmoid(h.t+ - h.t-) on rows of the final embeddings. */
int lkg_bpr_loss(const float* emb, int64_t ld_emb, int32_t g_dim, const int64_t* h, const int64_t* pos,
                 const int64_t* neg, int64_t batch, float l2_lambda, float* loss, const float* grad_scale,
                 float* d_emb, int64_t ld_d, void* stream);
/* calc_triplet_loss (model.py:364-428): TransR, rows projected by gat_trans_M[r] ([R, g_dim, r_dim]),
 * -log sigmoid(|h_r + e_r - t-_r|^2 - |h_r + e_r - t+_r|^2).  d_relation [R, r_dim], d_trans_m like trans_m. */
int lkg_transr_loss(const float* emb, int64_t ld_emb, int32_t g_dim, const float* relation, int64_t ld_rel,
                    int32_t r_dim, const float* trans_m, const int64_t* h, const int64_t* r, const int64_t* pos,
                    const int64_t* neg, int64_t batch, float l2_lambda, float* loss, const float* grad_scale,
                    float* d_emb, int64_t ld_d, float* d_relation, float* d_trans_m, void* stream);

/* ---- variant heads (SURVEY.md 8(f) rank 3) ------------------------------------------------------------------------
 * TransE triplet loss of the BCE variant (model_bce.py:329-368): -log sigmoid(|h + e_r - t-|^2 - |h + e_r - t+|^2) on
 * rows of the final embeddings (relation_dim must equal their width) + l2_lambda * the four _L2_loss_mean terms.  Same
 * conventions as the two losses above; d_relation [R, dim] contiguous. */
int lkg_transe_loss(const float* emb, int64_t ld_emb, int32_t dim, const float* relation, int64_t ld_rel,
                    const int64_t* h, const int64_t* r, const int64_t* pos, const int64_t* neg, int64_t batch,
                    float l2_lambda, float* loss, const float* grad_scale, float* d_emb, int64_t ld_d,
                    float* d_relation, void* stream);
/* The `mlp` mode head (model.py:499-519 initialize_MLP / train_MLP, model_bce.py:423-436):
 *   x = [emb[h] | emb[t]] -> norm1(relu(fc1 x)) -> norm2(relu(fc2 .)) -> sigmoid(fc3 .)
 * as a chain of fused fully-connected steps over one minibatch.  The input of a step is
 *   pair mode   (rows_a / rows_b != NULL): in = embedding matrix, element (b, c) = in[rows_a[b], c] for c < half,
 *               in[rows_b[b], c - half] otherwise (the torch.cat of the two gathered row blocks, never written);
 *   affine mode (in_scale / in_shift != NULL): in[b, c] * in_scale[c] + in_shift[c] (the previous BatchNorm, folded);
 *   plain       otherwise.
 * out[b, j] = act(sum_c input(b, c) w[j, c] + bias[j]), act: 0 none, 1 ReLU, 2 sigmoid.  stats (nullable, device
 * double[2 n], zero it first): column sums of out and out^2 for the BatchNorm that follows. */
int lkg_mlp_fc_fwd(const float* in, int64_t ld_in, const int64_t* rows_a, const int64_t* rows_b, int32_t half,
                   const float* in_scale, const float* in_shift, int64_t m, int32_t k, const float* w, int64_t ldw,
                   const float* bias /*nullable*/, int32_t n, int32_t act, float* out, int64_t ld_out, double* stats,
                   void* stream);
/* nn.BatchNorm1d bookkeeping: training != 0: batch mean / biased variance from stats (m rows), running buffers updated
 * with `momentum` and the unbiased variance; training == 0: the running buffers.  Writes scale = gamma * rstd,
 * shift = beta - mean * scale (the folded affine of the next step) and mean / rstd (nullable) for the backward. */
int lkg_bn_finalize(const double* stats, int64_t m, int32_t n, const float* gamma, const float* beta, float eps,
                    float momentum, float* running_mean, float* running_var, int32_t training, float* scale,
                    float* shift, float* mean_out, float* rstd_out, void* stream);
/* dw[j, c] += sum_b dz[b, j] input(b, c), db[j] (nullable) += sum_b dz[b, j]; input as in lkg_mlp_fc_fwd. */
int lkg_mlp_fc_bwd_weight(const float* dz, int64_t ld_dz, const float* in, int64_t ld_in, const int64_t* rows_a,
                          const int64_t* rows_b, int32_t half, const float* in_scale, const float* in_shift, int64_t m,
                          int32_t k, int32_t n, float* dw, int64_t ld_dw, float* db, void* stream);
/* dx[b, c] = sum_j dz[b, j] w[j, c].  Pair mode: ACCUMULATED into dx[rows_a[b], c] / dx[rows_b[b], c - half] (dx = the
 * gradient of the embedding matrix).  Otherwise written to dx [m, k]; with bn_stats (device double[2 k], zero it first)
 * the sums of the BatchNorm backward are accumulated: sum_b dx and sum_b dx * xhat, xhat = (a - mean) * rstd. */
int lkg_mlp_fc_bwd_input(const float* dz, int64_t ld_dz, int64_t m, int32_t n, const float* w, int64_t ldw, int32_t k,
                         float* dx, int64_t ld_dx, const int64_t* rows_a, const int64_t* rows_b, int32_t half,
                         const float* a, int64_t ld_a, const float* mean, const float* rstd, double* bn_stats,
                         void* stream);
/* BatchNorm + ReLU backward: dz = [a > 0] gamma rstd (dy - s1 / m - xhat s2 / m) with the sums of bn_stats
 * (training == 0: dz = [a > 0] gamma rstd dy); dgamma += s2, dbeta += s1. */
int lkg_bn_relu_bwd(const float* dy, int64_t ld_dy, const float* a, int64_t ld_a, const float* mean, const float* rstd,
                    const float* gamma, const double* bn_stats, int64_t m, int32_t k, int32_t training, float* dz,
                    int64_t ld_dz, float* dgamma, float* dbeta, void* stream);
/* dz = dy * y * (1 - y). */
int lkg_sigmoid_bwd(const float* dy, const float* y, int64_t m, float* dz, void* stream);

/* ---- minibatch assembly (dataloader.py:192-318): per head one positive (tail, relation) drawn uniformly from the
 *      head's triples and neg_rate negative tails drawn from `candidates` by rejection (not a positive of the head
 *      under the drawn relation -- any relation when use_relation == 0 -- and not drawn before).  rowptr / tails / rels:
 *      a CSR over heads whose rows are sorted by (relation, tail) (lkg_graph att_rowptr / att_tail / att_rel).
 *      Outputs are [n_heads * neg_rate], head / relation / positive repeated neg_rate times like
 *      generate_batch_by_neg_rate (dataloader.py:320-333).  Counter-based generator: the same seed gives the same
 *      batch.  n_failed (device int32, accumulated): draws that found no admissible tail in max_tries (the last candidate
 *      drawn is emitted, so ids always stay valid) or heads without triples; callers must treat n_failed > 0 as an error. */
int lkg_sample_batch(const int32_t* rowptr, const int32_t* tails, const int32_t* rels, const int64_t* heads,
                     int64_t n_heads, const int64_t* candidates, int64_t n_candidates, int32_t neg_rate,
                     int32_t use_relation, uint64_t seed, int32_t max_tries, int64_t* out_h,
                     int64_t* out_r /*nullable*/, int64_t* out_pos, int64_t* out_neg, int32_t* n_failed, void* stream);

/* ---- scoring (model.py:473-491) and the top-k / rank extension of BASELINE.json ------------- */
/* scores[B,Nt] = heads @ tails^T with both operands given as planes (heads: gathered rows of the final
 * embeddings, tails: the candidate rows); minmax_dev (nullable) is an opaque uint32[2] running
 * {min, max} state (order-preserving encoding) that must be reset with lkg_minmax_reset first. */
int lkg_score(const lkg_planes* heads, int64_t n_heads, const lkg_planes* tails, int64_t n_tails,
              float* scores, int64_t ld_scores, uint32_t* minmax_dev, void* stream);
int lkg_minmax_reset(uint32_t* minmax_dev, void* stream);
/* pred = ((s - min) / (max - min) > milestone) as int32 (model.py:490-491); NaN compares false. */
int lkg_predict_threshold(const float* scores, int64_t ld_scores, int64_t n_heads, int64_t n_tails,
                          const uint32_t* minmax_dev, float milestone, int32_t* pred, int64_t ld_pred,
                          void* stream);
/* Per-row top-k of a score matrix: larger score first, ties -> lower column.  k <= 1024.
 * target_cols (nullable) int64 [n_rows]: ranks_out[i] = number of columns that beat target_cols[i]. */
int lkg_topk_rows(const float* scores, int64_t ld_scores, int64_t n_rows, int64_t n_cols, int32_t k,
                  float* top_values, int64_t* top_cols, const int64_t* target_cols,
                  int64_t* ranks_out, void* stream);


/* k-way merge of `parts` per-rank survivor lists (sharded scoring): vals / ids [parts][n_rows][k], ids = global tail
 * positions (-1 = padding), every list ordered (score desc, position asc); parts * k <= 1024.  Output: the k best per
 * row under the same order. */
int lkg_topk_merge(const float* vals, const int64_t* ids, int32_t parts, int64_t n_rows, int32_t k, float* top_values,
                   int64_t* top_ids, void* stream);

/* ---- fused all-entity scoring + top-k: the B x Nt score matrix is never materialised --------------
 * Index of a set of embedding rows (heads of a batch, or the candidate tails): the scaled fp16 "hi" plane
 * [m, ld_hi] the filter GEMM reads, the rows' norms (scaled units) and their maximum (device scalar, reset by
 * the call).  rec: scale record that bounds emb (lkg_scale_from_data); rows: optional int64 gather. */
int lkg_score_index(const float* emb, int64_t ld, const int64_t* rows /*nullable*/, int64_t m, int32_t dim,
                    const float* rec, uint16_t* hi, int64_t ld_hi, float* norms /*[m]*/, float* max_norm,
                    void* stream);
/* ---- rank of a given tail per head without the score matrix (north star (d): top-k AND rank epilogue) -------------
 * rank_i = #{ j : s_ij > s_it or (s_ij == s_it and j < t_i) }, s = the exact scores the fused top-k returns, t_i =
 * target_pos[i] (a position in the tail list).  Three calls on one stream:
 *   lkg_rank_prepare  tau [n_heads] = exact target scores, thr [n_heads][2] = tau -/+ a rigorous bound of the
 *                     3-product GEMM's error (tail_max_norm / rec: the score index of the tails the GEMM multiplies).
 *                     center (nullable): the GEMM's tails are t_j - center -- a common shift leaves every head's
 *                     ranking unchanged and shrinks the bound from |h| max|t| to |h| max|t - center|; the thresholds
 *                     are then taken around tau - h . center;
 *   lkg_score_rank    the scoring GEMM (heads / tails as hi/lo planes sharing one scale record) with a counting
 *                     epilogue: above[i] += columns certainly better, band_cnt[i] += columns inside the band, the first
 *                     band_cap of them listed in band [n_heads][band_cap] (zero above / band_cnt first);
 *   lkg_rank_finalize the listed columns re-scored exactly; a head whose band overflowed is re-scanned exactly. */
/* out[r, :] = src[rows ? rows[r] : r, :] - center: the shifted tails of the rank GEMM (center = their mean). */
int lkg_shift_rows(const float* src, int64_t ld, const int64_t* rows /*nullable*/, int64_t m, int32_t k,
                   const float* center, float* out, int64_t ld_out, void* stream);
int lkg_rank_prepare(const float* emb, int64_t ld_emb, const int64_t* tail_rows /*nullable*/, const float* head_emb,
                     int64_t ld_head_emb, const int64_t* head_rows /*nullable*/, const int64_t* target_pos,
                     int64_t n_heads, int32_t dim, const float* tail_max_norm, const float* rec,
                     const float* center /*nullable [dim]*/, float* tau, float* thr, void* stream);
int lkg_score_rank(const lkg_planes* heads, int64_t n_heads, const lkg_planes* tails, int64_t n_tails, const float* thr,
                   int32_t* above, int32_t* band_cnt, int32_t* band, int32_t band_cap, void* stream);
int lkg_rank_finalize(const float* emb, int64_t ld_emb, const int64_t* tail_rows, const float* head_emb,
                      int64_t ld_head_emb, const int64_t* head_rows, const int64_t* target_pos, const float* tau,
                      const int32_t* above, const int32_t* band_cnt, const int32_t* band, int32_t band_cap,
                      int64_t n_heads, int64_t n_tails, int32_t dim, int64_t* ranks, void* stream);
/* ---- filtered rank (link-prediction evaluation): ranks[i] -= #{ f in F(i) that beat the target } --------------------
 * Query i = (heads[i], rels[i], target at candidate position target_pos[i]).  F(i) = the distinct tails t' of the known
 * triples (heads[i], rels[i], t') taken from the att order of `known` (rels NULL or rels[i] < 0: of any relation, from
 * its agg order); the target itself and entities without a candidate position are skipped.  cand_map (nullable) int32
 * [known->n_entities]: candidate position of an entity, -1 = not a candidate; NULL = the identity.  heads in
 * [0, known->n_entities).  Applied in place to the raw ranks, on the scores those ranks were counted on:
 *   lkg_rank_filter         after lkg_rank_finalize: tau = its target scores; emb [*, ld_emb] the matrix holding both the
 *                           head rows (heads[i]) and the candidate rows (entity f = row f); f is re-scored with the
 *                           finalize kernel's exact dot product, so a tail is subtracted exactly when finalize counted it;
 *   lkg_rank_filter_scores  after lkg_topk_rows: scores [n_queries, n_cols] the matrix whose row i was ranked. */
int lkg_rank_filter(const lkg_graph* known, const int64_t* heads, const int64_t* rels /*nullable*/,
                    const int32_t* cand_map /*nullable*/, const int64_t* target_pos, int64_t n_queries, const float* emb,
                    int64_t ld_emb, int32_t dim, const float* tau, int64_t* ranks, void* stream);
int lkg_rank_filter_scores(const lkg_graph* known, const int64_t* heads, const int64_t* rels /*nullable*/,
                           const int32_t* cand_map /*nullable*/, const int64_t* target_pos, int64_t n_queries,
                           const float* scores, int64_t ld_scores, int64_t n_cols, int64_t* ranks, void* stream);
/* ---- distance rank: the triple score s(h, r, t) = -|q - p_t|^2 of TransR / TransE (link-prediction evaluation) -------
 * q = the query rows (emb[h] M_r + e_r for (h, r, ?); emb[t] M_r - e_r for (?, r, t)), p_j = the candidates' projected
 * rows (emb[j] M_r; TransE: M_r = I), both fp32 [*, dim] with dim % 4 == 0, dim <= 508, 16-byte aligned rows.
 * d_j = |q - p_j|^2 EXACTLY (differences and squares in fp64, summed in fp64, rounded once to fp32); rank_i =
 * #{ j : d_j < d_t or (d_j == d_t and j < t_i) } with t_i = target_pos[i] (a row of the candidate table).  With
 * c = the candidates' mean row, d_j = |q - c|^2 - 2 ((q - c) . (p_j - c) - |p_j - c|^2 / 2): the counting GEMM of
 * lkg_score_rank, unchanged, on augmented operands of width K = dim + 4.  Calls on one stream:
 *   lkg_l2_rank_rows     out [m, ld_out >= dim + 4] = the augmented rows of src[rows ? rows[r] : r] - center:
 *                        LKG_L2_CANDIDATE: [p - c, -|p - c|^2 / (2 alpha), 0..] and stats (float[2]) = {max |p - c|,
 *                        max row norm}, rounded up (two passes: the first finds max |p - c|, which fixes the power of
 *                        two alpha); LKG_L2_QUERY: [q - c, alpha, 0..] with alpha read from the candidates' stats;
 *   (lkg_split_planes of both, each with its own scale record)
 *   lkg_rank_prepare_l2  tau = d_t (exact), thr = the band around the target's GEMM value, a rigorous bound of the GEMM's
 *                        error at K (rec_query / rec_cand: the planes' scale records) and of the fp32 roundings of
 *                        q - c, p - c and the norm column;
 *   lkg_score_rank       the query planes against the candidate planes;
 *   lkg_rank_finalize_l2 the band columns (every column on overflow) re-scored exactly;
 *   lkg_rank_filter_l2   as lkg_rank_filter; f is re-scored with the same exact distance against its row of the
 *                        candidate table, cand_map[f] (NULL: row f), and the same tau. */
enum lkg_l2_mode { LKG_L2_QUERY = 0, LKG_L2_CANDIDATE = 1 };
int lkg_l2_rank_rows(const float* src, int64_t ld, const int64_t* rows /*nullable*/, int64_t m, int32_t dim,
                     const float* center, int32_t mode, float* stats, float* out, int64_t ld_out, void* stream);
int lkg_rank_prepare_l2(const float* cand, int64_t ld_cand, const float* query, int64_t ld_query, const float* query_aug,
                        int64_t ld_aug, const int64_t* target_pos, int64_t n_queries, int32_t dim, const float* stats,
                        const float* rec_query, const float* rec_cand, float* tau, float* thr, void* stream);
int lkg_rank_finalize_l2(const float* cand, int64_t ld_cand, const float* query, int64_t ld_query,
                         const int64_t* target_pos, const float* tau, const int32_t* above, const int32_t* band_cnt,
                         const int32_t* band, int32_t band_cap, int64_t n_queries, int64_t n_cand, int32_t dim,
                         int64_t* ranks, void* stream);
int lkg_rank_filter_l2(const lkg_graph* known, const int64_t* anchors, const int64_t* rels /*nullable*/,
                       const int32_t* cand_map /*nullable*/, const int64_t* target_pos, int64_t n_queries,
                       const float* cand, int64_t ld_cand, const float* query, int64_t ld_query, int32_t dim,
                       const float* tau, int64_t* ranks, void* stream);
/* ---- relation-aware top-k under the triple score: the k best candidates of (h, r, ?) / (?, r, t) ----------------------
 * Rows and d_j as for the distance rank above.  Per query i the k candidates j not excluded with the smallest d_j, ties
 * -> lower position: dist [n_queries, k] fp32 ascending, pos [n_queries, k] int64 candidate positions (rows of the
 * candidate table), padded with +inf / -1 when fewer than k remain.  Excluded (known NULL: nothing): the candidates
 * whose entity id (cand_ids[j], NULL: j) is in the run of (anchors[i], rels[i]) of `known` (rels NULL: of any
 * relation); duplicate triples count once.  Calls on one stream, after lkg_l2_rank_rows / lkg_split_planes of the
 * query operand as for the rank:
 *   lkg_topk_threshold_l2  theta_i = the exact k-th smallest distance among the n_sample (1 <= n_sample <= n_cand)
 *                          strided positions floor(s n_cand / n_sample) that are not excluded (+inf if fewer than k);
 *                          thr [n_queries][2] = {sigma - M, +inf}, sigma = (|u|^2 - theta) / 2 and M the band margin of
 *                          lkg_rank_prepare_l2 with d_t = theta (-inf when theta is +inf); theta (nullable) [n_queries];
 *   lkg_score_rank         the query planes against the candidate planes with thr: every column with a GEMM value
 *                          >= sigma - M is listed in band (band_cnt / above zeroed first; above stays 0).  A column not
 *                          listed is farther than theta, so every member of the top-k is listed;
 *   lkg_topk_finalize_l2   the listed columns re-scored exactly, excluded ones dropped, sorted, first k written; a query
 *                          whose list overflowed (band_cnt > cap) is re-scanned exactly over every candidate.
 *                          1 <= k <= 1024, 2k <= cap <= 16384; shared memory next_pow2(cap) * 8 bytes per CTA. */
int lkg_topk_threshold_l2(const float* cand, int64_t ld_cand, int64_t n_cand, const float* query, int64_t ld_query,
                          const float* query_aug, int64_t ld_aug, int64_t n_queries, int32_t dim, const float* stats,
                          const float* rec_query, const float* rec_cand, int32_t k, int32_t n_sample,
                          const lkg_graph* known /*nullable*/, const int64_t* anchors, const int64_t* rels /*nullable*/,
                          const int64_t* cand_ids /*nullable*/, float* thr, float* theta /*nullable*/, void* stream);
int lkg_topk_finalize_l2(const float* cand, int64_t ld_cand, int64_t n_cand, const float* query, int64_t ld_query,
                         int64_t n_queries, int32_t dim, const int32_t* band_cnt, const int32_t* band, int32_t cap,
                         int32_t k, const lkg_graph* known /*nullable*/, const int64_t* anchors,
                         const int64_t* rels /*nullable*/, const int64_t* cand_ids /*nullable*/, float* dist,
                         int64_t* pos, void* stream);
/* ---- filtered top-k under the dot score: the k best new links of an anchor ----------------------------------------
 * s_j = emb[a] . emb[j], the exact dot product of lkg_score_topk (fp32 products summed in fp64, rounded once), on rows
 * of width dim (dim % 4 == 0, 4 <= dim <= 512, 16-byte aligned).  Query i's row is query[query_rows[i]] (query_rows
 * NULL: row i), candidate position p's row is cand[cand_rows[p]] (cand_rows NULL: row p).  Per query the k candidates
 * not excluded with the largest s_j, ties -> lower position: score [n_queries, k] fp32 descending, pos [n_queries, k]
 * int64 candidate positions, padded with -inf / -1 when fewer than k remain.  Excluded: as for the distance top-k
 * above (the run of (anchors[i], rels[i]) of `known`, rels NULL: of any relation; by entity id cand_ids[p], NULL: p).
 * Calls on one stream, with the candidate operand of ScoreIndex.centered (the rows w_p = fl(t_p - center) as hi/lo
 * planes, their max norm cand_max_norm as lkg_score_index records it) and lkg_split_planes of the query rows:
 *   lkg_topk_threshold_dot  theta_i = the exact k-th largest score among the n_sample (1 <= n_sample <= n_cand)
 *                           strided positions floor(s n_cand / n_sample) that are not excluded (-inf if fewer than k);
 *                           thr [n_queries][2] = {theta - h . center - M, +inf} rounded down, M the band margin of the
 *                           3-product GEMM at K = dim (-inf when theta is -inf); theta (nullable) [n_queries];
 *   lkg_score_rank          the query planes against the centred candidate planes with thr: every column whose GEMM
 *                           value reaches thr is listed in band (band_cnt / above zeroed first; above stays 0).  A
 *                           column not listed scores below theta, so every member of the top-k is listed;
 *   lkg_topk_finalize_dot   the listed columns re-scored exactly on the uncentred rows, excluded ones dropped, sorted,
 *                           first k written; a query whose list overflowed (band_cnt > cap) is re-scanned exactly.
 *                           1 <= k <= 1024, 2k <= cap <= 16384; shared memory next_pow2(cap) * 8 bytes per CTA. */
int lkg_topk_threshold_dot(const float* cand, int64_t ld_cand, const int64_t* cand_rows /*nullable*/, int64_t n_cand,
                           const float* query, int64_t ld_query, const int64_t* query_rows /*nullable*/,
                           int64_t n_queries, int32_t dim, const float* center, const float* cand_max_norm,
                           const float* rec_query, const float* rec_cand, int32_t k, int32_t n_sample,
                           const lkg_graph* known /*nullable*/, const int64_t* anchors,
                           const int64_t* rels /*nullable*/, const int64_t* cand_ids /*nullable*/, float* thr,
                           float* theta /*nullable*/, void* stream);
int lkg_topk_finalize_dot(const float* cand, int64_t ld_cand, const int64_t* cand_rows /*nullable*/, int64_t n_cand,
                          const float* query, int64_t ld_query, const int64_t* query_rows /*nullable*/,
                          int64_t n_queries, int32_t dim, const int32_t* band_cnt, const int32_t* band, int32_t cap,
                          int32_t k, const lkg_graph* known /*nullable*/, const int64_t* anchors,
                          const int64_t* rels /*nullable*/, const int64_t* cand_ids /*nullable*/, float* score,
                          int64_t* pos, void* stream);
int lkg_score_topk_workspace_bytes(int64_t n_heads, int32_t cap, int32_t sample_tiles, size_t* bytes /*host out*/);
/* Per head the k best tails by emb[head] . emb[tail]: larger score first, ties -> lower position in the tail
 * list; values are the exact dot products (fp32 products summed in fp64, rounded once).
 *   theta [n_heads] (element stride theta_stride, nullable): a caller-supplied lower bound of each head's k-th
 *     best EXACT score; the filter keeps every tail whose single-product fp16 score reaches theta minus a
 *     rigorous error bound, so a loose theta only costs time;
 *   sample_tiles (used when theta is NULL): the library derives the bound itself from the k-th largest tile
 *     maximum over this many evenly strided 128-tail tiles (a first, short pass of the same GEMM kernel);
 *     needs sample_tiles >= k to give a bound; 0 = no bound, every tail is a candidate;
 *   cap: candidate slots per head (power of two, >= 2k); a head that overflows is re-scanned exactly;
 *   emb: the fp32 matrix behind the tails index; head_emb (nullable = emb): the one behind the heads index
 *     (a separate matrix when the heads' rows were gathered from other ranks);
 *   head_rows / tail_rows (nullable): the rows of those matrices behind the two indexes (NULL = identity);
 *   dim <= 256, dim % 4 == 0.  top_values [n_heads, k] fp32, top_cols [n_heads, k] int64 (-inf / -1 past n_tails). */
int lkg_score_topk(const uint16_t* heads_hi, int64_t ld_heads_hi, const float* head_norms, int64_t n_heads,
                   const uint16_t* tails_hi, int64_t ld_tails_hi, const float* tail_max_norm, int64_t n_tails,
                   int32_t dim, const float* rec, const float* theta, int64_t theta_stride, int32_t sample_tiles,
                   const float* emb, int64_t ld_emb, const float* head_emb, int64_t ld_head_emb,
                   const int64_t* head_rows, const int64_t* tail_rows, int32_t k, int32_t cap, float* top_values,
                   int64_t* top_cols, void* workspace, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* LKG_H_ */
