/* hg_b200.h — C ABI of the B200-native hyper-greco GKR/Lasso proving path.
 *
 * This is the boundary a Rust `extern "C"` FFI crate binds (INTEGRATION.md shows the binding). Plain pointers and
 * sizes only; no C++ / torch types. Every entry point cites the reference interface it replaces, paths relative to
 * /root/reference.
 *
 * Conventions
 *   field ids        HG_FIELD_GOLDILOCKS: F = Goldilocks, E = GoldilocksExt2 (bfv-gkr/src/sk_encryption_circuit.rs:554-612)
 *                    HG_FIELD_BN254     : F = E = bn256::Fr                  (bfv-gkr/src/sk_encryption_circuit.rs:616-626)
 *   element encoding canonical integer in little-endian u64 limbs: base element = HG limbs(field) u64,
 *                    extension element = degree(field) base elements in `as_bases()` order.
 *   return value     0 = ok, non-zero = error; hg_last_error() returns the message (thread-local). No C++ exception
 *                    and no sticky CUDA error crosses this boundary.
 *   threading        one hg_ctx = one device + one stream, driven by one host thread at a time. Distinct contexts may be
 *                    driven concurrently from different threads, objects of any shapes may be alive together, and one
 *                    process may hold contexts on several devices. The per-kernel dynamic shared-memory limits are
 *                    shared by the whole process; hg_ctx_create sets them for its device to the device's maximum, the
 *                    same value on every call, so no object can lower a limit another one needs.
 *   ownership        handles are created/destroyed only through this API; the library never frees caller memory and
 *                    never keeps a host pointer after a call returns.
 */
#ifndef HG_B200_H
#define HG_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HG_FIELD_GOLDILOCKS 0
#define HG_FIELD_BN254 1

#define HG_MODE_PREFETCH 0    /* challenges squeezed up front; legal for Keccak256Transcript (transcript.rs:156,183-203) */
#define HG_MODE_INTERACTIVE 1 /* one host round trip per squeeze; legal for any transcript */

/* Upstream-format switches (SURVEY.md Appendix B): ids for hg_ctx_set_option */
#define HG_OPT_A3_WIRE 3       /* 0 coefficients c0,c2..cd (default) / 1 evaluations h(0),h(2)..h(d) */
#define HG_OPT_A3_H1 31        /* 0 h(1) := claim - h(0) (default) / 1 h(1) from the tables */
#define HG_OPT_A5_ASCENDING 5  /* distribute_powers: 1 ascending (default) / 0 first expression highest power */
#define HG_OPT_TWO_STREAMS 100 /* scheduling only, no effect on results: 1 (default) hg_gkr_prove runs the layer sumchecks on a second
                                * stream next to the Lasso node in prefetch mode / 0 everything on the context's stream */

typedef struct hg_ctx hg_ctx;
typedef struct hg_transcript hg_transcript;
typedef struct hg_lasso_pp hg_lasso_pp;
typedef struct hg_lasso_node hg_lasso_node;
typedef struct hg_buf hg_buf;
typedef struct hg_circuit hg_circuit;
typedef struct hg_verifier hg_verifier;

const char* hg_last_error(void);
int hg_version(void);

/* ---- context ------------------------------------------------------------------------------------------------ */
int hg_ctx_create(int device, int field_id, hg_ctx** out);
void hg_ctx_destroy(hg_ctx* ctx);
int hg_ctx_set_option(hg_ctx* ctx, int option, int value);
int hg_ctx_synchronize(hg_ctx* ctx);
/* kernels enqueued by this context so far */
uint64_t hg_ctx_launch_count(hg_ctx* ctx);
/* per-kernel-class CUDA-event timing on the launching stream (bench.py's roofline leg). hg_ctx_profile(ctx,1) resets and
 * starts recording, hg_ctx_profile(ctx,0) stops; hg_ctx_profile_read returns the launches, summed device milliseconds and
 * summed ALGORITHMIC bytes (DESIGN.md, per-kernel table) of one class. */
int hg_ctx_profile(hg_ctx* ctx, int enable);
int hg_ctx_profile_read(hg_ctx* ctx, int kernel_class, uint64_t* launches, double* ms, uint64_t* algorithmic_bytes);
int hg_kernel_class_count(void);
const char* hg_kernel_class_name(int kernel_class);
/* the CUDA stream kernels are launched on (cudaStream_t), for event timing by the caller */
void* hg_ctx_stream(hg_ctx* ctx);

/* ---- device buffers (owned by the caller through the handle; Rust frees them in Drop) --------------------------- */
int hg_buf_alloc(hg_ctx* ctx, size_t bytes, hg_buf** out);
int hg_buf_upload(hg_ctx* ctx, hg_buf* buf, size_t offset, const void* host, size_t bytes);
/* the same without waiting: `host` must stay valid (and should be page-locked) until a later call synchronises the context */
int hg_buf_upload_async(hg_ctx* ctx, hg_buf* buf, size_t offset, const void* host, size_t bytes);
int hg_buf_download(hg_ctx* ctx, const hg_buf* buf, size_t offset, void* host, size_t bytes);
/* read `bytes` from any device pointer the library handed out (hg_circuit_node_value), in stream order behind the context's work */
int hg_device_download(hg_ctx* ctx, const void* d_ptr, void* host, size_t bytes);
void* hg_buf_device_ptr(hg_buf* buf);
size_t hg_buf_size(const hg_buf* buf);
void hg_buf_free(hg_buf* buf);

/* Device tables hold the library's internal representation: canonical u64 for Goldilocks, 4x64-bit Montgomery form for BN254
 * (32 bytes per element). hg_field_encode converts n base elements that were uploaded as canonical little-endian limbs, in
 * place; hg_field_decode converts back. Both are no-ops for Goldilocks. Host-pointer inputs of hg_lasso_node_prove are encoded
 * by the library. */
size_t hg_field_base_bytes(int field_id);
int hg_field_encode(hg_ctx* ctx, void* d_data, size_t n);
int hg_field_decode(hg_ctx* ctx, void* d_data, size_t n);

/* ---- transcript: replaces Keccak256Transcript (bfv-gkr/src/transcript.rs:117-203) ----------------------------- */
int hg_transcript_new(int field_id, hg_transcript** out);                                      /* ::default()      :431 of sk_encryption_circuit.rs */
int hg_transcript_from_proof(int field_id, const uint8_t* proof, size_t len, hg_transcript** out); /* ::from_proof  transcript.rs:131-135 */
/* A transcript OWNED BY THE CALLER, i.e. the `&mut dyn TranscriptWrite<F, E>` / `&mut dyn TranscriptRead<F, E>` that
 * gkr::prove_gkr hands to Node::prove_claim_reduction / verify_claim_reduction (lasso/src/lasso.rs:58-63, :117-121). The three
 * primitives the path uses are forwarded to C callbacks over canonical little-endian limbs (same encoding as everywhere
 * in this header): squeeze_challenge (transcript.rs:146-157), write_felt_ext (:191-195), read_felt_ext (:172-177). A
 * callback returns 0 on success; anything else aborts the call with an error. `write` may be NULL for a verifier
 * transcript, `read` for a prover one. Such a transcript may absorb what is written to it, so every prove call that
 * receives it runs in HG_MODE_INTERACTIVE (one round trip per squeeze, messages delivered strictly in protocol order)
 * unless message_independent != 0, by which the caller promises that challenges do not depend on written messages (true
 * for the reference's Keccak256Transcript, transcript.rs:156,183-203) and thereby allows HG_MODE_PREFETCH: all challenges
 * of the call are squeezed first, all messages are written afterwards, still in protocol order.
 * hg_transcript_proof_len/_copy return nothing for it (the bytes live with the caller). */
typedef int (*hg_squeeze_fn)(void* user, uint64_t* out_ext);
typedef int (*hg_write_fn)(void* user, const uint64_t* ext);
typedef int (*hg_read_fn)(void* user, uint64_t* out_ext);
int hg_transcript_from_callbacks(int field_id, void* user, hg_squeeze_fn squeeze, hg_write_fn write, hg_read_fn read, int message_independent,
                                 hg_transcript** out);
void hg_transcript_free(hg_transcript* t);
int hg_transcript_squeeze_challenge(hg_transcript* t, uint64_t* out_ext);   /* transcript.rs:149-154 */
int hg_transcript_squeeze_challenges(hg_transcript* t, size_t n, uint64_t* out_ext); /* n consecutive squeezes (TranscriptWrite::squeeze_challenges) */
int hg_transcript_write_felt_ext(hg_transcript* t, const uint64_t* ext);    /* transcript.rs:191-195 */
int hg_transcript_read_felt_ext(hg_transcript* t, uint64_t* out_ext);       /* transcript.rs:172-177 */
size_t hg_transcript_proof_len(const hg_transcript* t);                     /* into_proof, transcript.rs:126-128 */
int hg_transcript_proof_copy(const hg_transcript* t, uint8_t* out, size_t cap);
/* append bytes that were serialised elsewhere (the per-rank parts of a sharded proof, hg_gkr_emit_shard_part_dev); not for callback transcripts */
int hg_transcript_append_bytes(hg_transcript* t, const uint8_t* bytes, size_t n);
size_t hg_transcript_num_squeezed(const hg_transcript* t);                  /* base-field squeezes so far */

/* ---- Lasso preprocessing: LassoPreprocessing::preprocess::<C, M> over RangeLookup types (lasso/src/lasso.rs:527-627,
 *      lasso/src/table/range.rs:177-274). `bounds[i]` is the argument of RangeLookup::new_boxed. ---------------- */
int hg_lasso_preprocess(const uint64_t* bounds, size_t n_bounds, size_t C, size_t M, hg_lasso_pp** out);
/* Plug-in lookup types: LookupType / LassoSubtable (lasso/src/table.rs:16-67) described by DATA, for tables other than the range checks.
 * What the prove / verify path takes from the traits: the subtable's M entries (materialize; evaluate_mle is computed from them, the
 * MLE being unique), the dimensions it serves (SubtableIndices as a bit mask over chunk indices), chunk_bits (low chunk first; the
 * index is truncated to their sum, lasso.rs:388-389, and split into log2(M)-bit chunks, range.rs:254-256) and the combination
 * g(operands) = sum_t combine_weight^t * operand_t over the lookup's memories (combine_lookups, range.rs:184-204: weight M).
 * A subtable id must always denote the same table. Lookups are ordered by their id STRING and de-duplicated, as the reference's
 * BTreeMap does (lasso.rs:530-541). hg_lasso_preprocess(bounds) is the special case lookup_id "range_<bound>". */
typedef struct hg_lookup_desc {
    const char* lookup_id;
    size_t n_subtables;
    const char* const* subtable_ids;     /* n_subtables NUL-terminated ids */
    const uint64_t* const* tables;       /* n_subtables tables of M entries (lifted with F::from(u64)) */
    const uint64_t* dimension_masks;     /* n_subtables masks: bit d = the subtable serves chunk (dimension) d */
    size_t n_chunk_bits;                 /* number of chunks this lookup type uses (<= C) */
    const uint32_t* chunk_bits;
    uint64_t combine_weight;
} hg_lookup_desc;
int hg_lasso_preprocess_lookups(const hg_lookup_desc* lookups, size_t n_lookups, size_t C, size_t M, hg_lasso_pp** out);
int hg_lasso_pp_lookup_index_by_id(const hg_lasso_pp* pp, const char* lookup_id);  /* index in preprocessing (BTreeMap) order, or -1 */
void hg_lasso_pp_free(hg_lasso_pp* pp);
size_t hg_lasso_pp_num_lookups(const hg_lasso_pp* pp);
size_t hg_lasso_pp_num_subtables(const hg_lasso_pp* pp);
size_t hg_lasso_pp_num_memories(const hg_lasso_pp* pp);
/* index of RangeLookup::id_for(bound) in preprocessing (BTreeMap) order, or -1 */
int hg_lasso_pp_lookup_index(const hg_lasso_pp* pp, uint64_t bound);
/* memory_to_subtable_index / memory_to_dimension_index (lasso.rs:575-585); arrays of num_memories */
int hg_lasso_pp_memory_maps(const hg_lasso_pp* pp, uint32_t* mem_to_subtable, uint32_t* mem_to_dimension);
/* subtable id string ("full", "bound_<b>") of subtable `idx`, NUL-terminated into out[cap] */
int hg_lasso_pp_subtable_id(const hg_lasso_pp* pp, size_t idx, char* out, size_t cap);

/* ---- Lasso node: LassoNode::<F, E, C, M>::new + Node::prove_claim_reduction (lasso/src/lasso.rs:143-154, :57-114) -- */
/* lookups: Vec<LookupId> given as run-length segments (bound of the RangeLookup, run length), in row order. */
int hg_lasso_node_new(hg_ctx* ctx, const hg_lasso_pp* pp, size_t num_vars, const uint64_t* seg_bounds, const uint64_t* seg_lens, size_t n_segs,
                      hg_lasso_node** out);
/* the same with the lookups given by their ids (any LookupType, e.g. one made by hg_lasso_preprocess_lookups) */
int hg_lasso_node_new_ids(hg_ctx* ctx, const hg_lasso_pp* pp, size_t num_vars, const char* const* seg_lookup_ids, const uint64_t* seg_lens, size_t n_segs,
                          hg_lasso_node** out);
void hg_lasso_node_free(hg_lasso_node* node);
size_t hg_lasso_node_log2_input_size(const hg_lasso_node* node);  /* Node::log2_input_size, lasso.rs:45-47 */
size_t hg_lasso_node_device_bytes(const hg_lasso_node* node);
/* prove_claim_reduction. `inputs` is inputs[0] of the node (n_inputs base elements): a HOST pointer when
 * inputs_on_device == 0 (copied to the device inside the call), else a device pointer (e.g. hg_buf_device_ptr).
 * Messages are appended to `t` exactly as the reference writes them (SURVEY.md Appendix D). On return
 * out_point[num_vars] / out_value hold the single EvalClaim the node returns for its input (lasso.rs:97,113). */
int hg_lasso_node_prove(hg_lasso_node* node, const void* inputs, size_t n_inputs, int inputs_on_device, hg_transcript* t, int mode,
                        uint64_t* out_point, uint64_t* out_value);
/* Node::verify_claim_reduction (lasso/src/lasso.rs:116-139; memory_checking/verifier.rs:61-95,130-235) on the HOST: reads the node's
 * part of the proof from `t` (a transcript made by hg_transcript_from_proof, positioned where the node starts and having
 * squeezed what the prover had squeezed before it), checks the grand-product base relation and the memory hashes, and returns
 * the node's claim (point of num_vars challenges, claimed sum). options3 = {HG_OPT_A3_WIRE, HG_OPT_A3_H1, HG_OPT_A5_ASCENDING}
 * values or NULL for the defaults. Needs no GPU and no context. Error (non-zero) = the reference's Err / panic. */
int hg_lasso_node_verify(const hg_lasso_pp* pp, size_t num_vars, hg_transcript* t, const int* options3, uint64_t* out_point, uint64_t* out_value);
/* ---- one proof over several GPUs (SURVEY.md §8e). Every message of the node is either a sum over the 2m grand-product
 * vectors (round polynomials) or belongs to a single vector / memory (roots, evaluations, openings), and the verifier's
 * challenges do not depend on the messages (SURVEY.md F3). Rank r of `world` computes the part owned by r from its own
 * copy of the inputs and returns the node's message buffer with every other slot zero. The caller adds the buffers of all
 * ranks element-wise (hg_shard_merge, or any exchange that sums field elements) and rank 0 serialises the result into its
 * transcript with hg_lasso_node_emit_shard; the bytes equal those of hg_lasso_node_prove on one GPU. Words are the
 * library's device representation (not canonical limbs): only add them with hg_shard_merge. All ranks must pass
 * transcripts in the same state. */
size_t hg_lasso_node_shard_words(const hg_lasso_node* node); /* capacity (64-bit words) that always fits the message buffer */
int hg_lasso_node_prove_shard(hg_lasso_node* node, const void* inputs, size_t n_inputs, int inputs_on_device, hg_transcript* t, int rank, int world,
                              uint64_t* out_words, size_t cap_words, size_t* n_words);
int hg_shard_merge(int field_id, uint64_t* acc_words, const uint64_t* part_words, size_t n_words); /* acc += part, element-wise in the field */
int hg_lasso_node_emit_shard(hg_lasso_node* node, const uint64_t* merged_words, size_t n_words, uint64_t* out_point, uint64_t* out_value);
/* The same exchange without leaving the devices (what bench.py and the multi-GPU tests use): every rank's partial buffer is
 * copied into device memory of the caller (d_out_words, stream-ordered on the context's stream, no host synchronisation),
 * the caller all-gathers the buffers of all ranks over NVLink (NCCL all_gather enqueued behind hg_ctx_stream(); world *
 * n_words * 8 bytes, ~80 KB per rank at n = 32768), hg_shard_merge_device sums the `world` gathered buffers ([world][n_words],
 * rank-major) in the field with one kernel, and rank 0 serialises the sum with the *_emit_shard_dev call (one device-to-host
 * copy of n_words * 8 bytes). The collective carries messages only: tables never cross the link. */
int hg_lasso_node_prove_shard_dev(hg_lasso_node* node, const void* inputs, size_t n_inputs, int inputs_on_device, hg_transcript* t, int rank, int world,
                                  void* d_out_words, size_t cap_words, size_t* n_words);
int hg_shard_merge_device(hg_ctx* ctx, const void* d_parts_words, int world, size_t n_words, void* d_acc_words);
int hg_lasso_node_emit_shard_dev(hg_lasso_node* node, const void* d_merged_words, size_t n_words, uint64_t* out_point, uint64_t* out_value);
/* test hook: polynomialised witness of the last prove (lasso.rs:157-250). dims: C x R u16, read_cts: chunks x R u32,
 * final_cts: chunks x M u32, e_polys: num_memories x R base elements. Any pointer may be NULL. */
int hg_lasso_node_download_polys(hg_lasso_node* node, uint16_t* dims, uint32_t* read_cts, uint32_t* final_cts, uint64_t* e_polys);
size_t hg_lasso_node_num_chunks(const hg_lasso_node* node);
/* host-side phases of the last prove, microseconds: [squeeze+upload challenges, enqueue kernels, wait for the GPU, serialise proof] */
void hg_lasso_node_timing(const hg_lasso_node* node, double* out_us4);

/* ---- generic sumcheck: gkr::sum_check::prove_sum_check with a Generic function of the shape the lasso crate builds
 *      (lasso/src/lasso.rs:457-475, lasso/src/memory_checking/prover.rs:268-279):
 *          g = poly(0) * sum_{i<n_terms} coeffs[i] * prod_{k<arity} poly(arity*i + k)
 *      tables: device pointer to n_terms*arity base tables of 2^num_vars elements, back to back.
 *      Writes the round messages to `t`, squeezes one challenge per round; out_point[num_vars], out_evals[n_terms*arity]. */
int hg_sumcheck_prove(hg_ctx* ctx, int arity, size_t n_terms, size_t num_vars, const uint64_t* coeffs_ext, const void* d_tables,
                      const uint64_t* claim_ext, hg_transcript* t, int mode, uint64_t* out_point, uint64_t* out_evals);

/* ---- batched multilinear evaluation: MultilinearPoly::evaluate (lasso/src/memory_checking/mod.rs:80-93) ---------
 *      d_tables: n_tables base tables of 2^num_vars elements (stride elements apart); point: num_vars ext elements (host).
 *      For num_vars >= 2 every table must start 16-byte aligned (Goldilocks: an even stride); otherwise this is an error. */
int hg_mle_eval_batch(hg_ctx* ctx, const void* d_tables, size_t n_tables, size_t stride, size_t num_vars, const uint64_t* point_ext,
                      uint64_t* out_ext);

/* ---- FFT layers: FftNode::forward / ::inverse evaluation (call sites bfv-gkr/src/sk_encryption_circuit.rs:224,249,251; the
 *      transform lives in the un-vendored gkr crate: radix-2 over ROOT_OF_UNITY^(2^(S-log_n)), natural order, inverse scaled
 *      by 1/n). In place on `batch` consecutive transforms of 2^log_n base elements at the DEVICE pointer d_data. */
int hg_ntt(hg_ctx* ctx, void* d_data, size_t log_n, int inverse, size_t batch);


/* ---- GKR circuit: gkr::circuit::Circuit::{insert, connect, evaluate} and gkr::prove_gkr for the node shapes bfv-gkr builds
 *      (bfv-gkr/src/sk_encryption_circuit.rs:86-293, :442, :455-457). The engine is the un-vendored `gkr` crate; the per-node
 *      protocol restated here is in DESIGN.md section 3 (parity with the crate's bytes is unpinned). Node ids are returned in
 *      insertion order, as `circuit.insert` does. ------------------------------------------------------------------------- */
int hg_circuit_new(hg_ctx* ctx, hg_circuit** out);
void hg_circuit_free(hg_circuit* c);
int hg_circuit_insert_input(hg_circuit* c, size_t log2_size, size_t num_reps, int* out_id);   /* InputNode::new */
int hg_circuit_insert_fft(hg_circuit* c, size_t log2_size, int inverse, int* out_id);          /* FftNode::forward / ::inverse */
int hg_circuit_insert_lasso(hg_circuit* c, hg_lasso_node* node, int* out_id);                  /* LassoNode (ownership stays with the caller) */
/* VanillaNode::new(input_arity, log2_sub_input_size, gates, num_reps); gates in CSR form:
 *   gate g = consts[g] (if has_const[g]) + sum_{e in [add_ptr[g], add_ptr[g+1])} add_coef[e] * input[add_input[e]][rep*2^sub + add_wire[e]]
 *                                        + sum_{e in [mul_ptr[g], mul_ptr[g+1])} mul_coef[e] * input[mul_in0[e]][.. + mul_w0[e]] * input[mul_in1[e]][.. + mul_w1[e]]
 * Every gate shape is supported, on the device and by the host verifier: layers with additive gates only and the element-wise
 * product layer (VanillaGate::mul((0,i),(1,i)), num_reps = 1) keep their own layer sumcheck; any other layer with a product term
 * (squares, products of any two wires, with coefficients, mixed with constants and sums, num_reps > 1) is proved by the two-phase
 * layer sumcheck of DESIGN.md section 3. The CSR arrays are validated before they are used; a NULL array is an error. */
int hg_circuit_insert_vanilla(hg_circuit* c, size_t input_arity, size_t log2_sub_input_size, size_t num_reps, size_t n_gates, const uint8_t* has_const,
                              const uint64_t* consts, const uint64_t* add_ptr, const uint64_t* add_coef, const uint32_t* add_input,
                              const uint64_t* add_wire, const uint64_t* mul_ptr, const uint64_t* mul_coef, const uint32_t* mul_in0, const uint64_t* mul_w0,
                              const uint32_t* mul_in1, const uint64_t* mul_w1, int* out_id);
int hg_circuit_connect(hg_circuit* c, int from, int to);                                       /* circuit.connect(from, to) */
/* circuit.evaluate(inputs): device pointers for the input nodes in insertion order; node values stay on the device */
int hg_circuit_evaluate(hg_circuit* c, const void* const* d_inputs, size_t n_inputs);
/* The same from HOST vectors, as the reference passes them (sk_encryption_circuit.rs:438-442): input i has n_elems[i] base
 * elements in canonical little-endian limbs. They are copied into device buffers owned by the circuit (asynchronously when the
 * host memory is page-locked) and the circuit is evaluated; the host vectors must stay valid until the next call that
 * synchronises the context (hg_gkr_prove, hg_mle_eval_batch, hg_ctx_synchronize). */
int hg_circuit_evaluate_host(hg_circuit* c, const void* const* host_inputs, const size_t* n_elems, size_t n_inputs);
int hg_circuit_node_value(hg_circuit* c, int id, const void** d_ptr, size_t* len);
/* gkr::prove_gkr(&circuit, &values, &output_claims, &mut transcript): one claim per output node (insertion order); point i has
 * point_lens[i] extension elements (concatenated in points_ext), values_ext one extension element per claim. The claims that
 * reach the input nodes are read back with the hg_gkr_input_claim* getters (what verify() checks, :512-516). */
int hg_gkr_prove(hg_circuit* c, size_t n_output_claims, const size_t* point_lens, const uint64_t* points_ext, const uint64_t* values_ext,
                 hg_transcript* t, int mode);
/* ONE gkr::prove_gkr over `world` GPUs (BASELINE.json config 4). With prefetched challenges every node's claim reduction is an
 * independent job; rank r runs the generic node sumchecks q with q % world == r and its share of the Lasso node (grand-product
 * vectors, openings and access counters split as in hg_lasso_node_prove_shard), every other message slot stays zero. Same
 * exchange as above: all-gather of hg_gkr_shard_words() words per rank, hg_shard_merge_device, then rank 0 calls
 * hg_gkr_emit_shard_dev, which writes the proof into the transcript given to ITS prove call and fills the input claims.
 * Every rank must have evaluated the circuit on the same inputs and pass transcripts in the same state. */
size_t hg_gkr_shard_words(hg_circuit* c);
int hg_gkr_prove_shard_dev(hg_circuit* c, size_t n_output_claims, const size_t* point_lens, const uint64_t* points_ext, const uint64_t* values_ext, hg_transcript* t,
                           int rank, int world, void* d_out_words, size_t cap_words, size_t* n_words);
int hg_gkr_emit_shard_dev(hg_circuit* c, const void* d_merged_words, size_t n_words);
/* The serialisation split over the ranks as well (rank 0's host work is what bounds a sharded proof): after the merge EVERY rank calls
 * this with part = its rank, nparts = world, and gets the bytes of one contiguous range of the proof; the ranges, concatenated in rank
 * order (any exchange of < 256 KB), are appended to rank 0's transcript with hg_transcript_append_bytes. The input claims are valid
 * on every rank afterwards. Bytes equal those of hg_gkr_emit_shard_dev. */
int hg_gkr_emit_shard_part_dev(hg_circuit* c, const void* d_merged_words, size_t n_words, int part, int nparts, uint8_t* out_bytes, size_t cap, size_t* out_len);
/* ---- BfvEncryptBlock::configure (bfv-gkr/src/sk_encryption_circuit.rs:86-293) in the library: builds the whole circuit of the BFV secret-key
 *      encryption proof into `c` with the calls above, node for node and connection for connection (a Rust caller that keeps its own
 *      `configure` binds hg_circuit_insert_* / hg_circuit_connect instead; the result is the same circuit). qis / k0is / r1_bounds /
 *      r2_bounds: arrays of K (BfvSkEncryptConstans, constants/mod.rs:16-35), K a power of two. The Lasso node: for a device circuit the
 *      node made by hg_lasso_node_new (lasso_pp may be NULL); for a host-only description (hg_circuit_new_host) its preprocessing and
 *      num_vars (lasso_node NULL). out_ids6 (may be NULL): node ids of s, e, k1, lasso_inputs_batched, the Lasso node, sum. */
int hg_bfv_configure(hg_circuit* c, size_t log2_size, size_t K, const uint64_t* qis, const uint64_t* k0is, const uint64_t* r1_bounds, const uint64_t* r2_bounds,
                     uint64_t s_bound, uint64_t e_bound, uint64_t k1_bound, hg_lasso_node* lasso_node, const hg_lasso_pp* lasso_pp, size_t lasso_num_vars,
                     int* out_ids6);
/* ---- synthetic witness on the device: the arithmetic of scripts/circuit_sk.py:72-140 (ct0i_hat = a_i s + e + k0_i k1 over Z, exact;
 *      centred reduction mod (x^n + 1, q_i); r2i, r1i; the bound assertions), written straight into the BfvEncrypt::get_inputs layout
 *      (sk_encryption_circuit.rs:365-415). The random draws stay with the caller (HOST arrays, lowest degree first): s in {-1,0,1} and e as
 *      int8, k1 as int32, a as [K][n] int64 with |a_i| <= (q_i - 1) / 2. Outputs are DEVICE pointers in the library's representation,
 *      ready for hg_circuit_evaluate (input-node order s, e, k1, ais.., r1is.., r2is) and hg_mle_eval_batch (ct0is):
 *        d_s, d_e, d_k1: 2n elements;  d_ais, d_r1is, d_ct0is: K x 2n;  d_r2is: K x n.
 *      A failed assertion of the reference script (not a multiple of x^n + 1, not divisible by q_i, r1 / r2 out of range) is an error. */
int hg_bfv_witness_generate(hg_ctx* ctx, size_t n, size_t K, const uint64_t* qis, const uint64_t* k0is, const uint64_t* r1_bounds, const uint64_t* r2_bounds,
                            const int8_t* s, const int8_t* e, const int32_t* k1, const int64_t* a, void* d_s, void* d_e, void* d_k1, void* d_ais, void* d_r1is,
                            void* d_r2is, void* d_ct0is);
/* ---- BFV PUBLIC-key encryption, Greco's second relation: for every modulus i < K over Z[x],
 *        ct0_i = pk0_i u + e0 + k0_i k1 + r1_i q_i + r2_i (x^n + 1)      ct1_i = pk1_i u + e1 + p1_i q_i + p2_i (x^n + 1)
 *      hg_bfv_pk_configure builds its circuit as hg_bfv_configure builds the SK one (same Lasso-node arguments), with the bounds of
 *      the quotients p1 / p2 and of u added. The public pk coefficients are not range-checked. Node order (DESIGN.md section 3, A12):
 *      inputs u, e0, e1, k1; pk0is.., pk1is.., r1is.., p1is..; r2is, p2is (n x K each). The Lasso node range-checks r1is | p1is |
 *      r2 chunks | p2 chunks | u | e0 | e1 | k1, every element shifted by the bound of its own vector and modulus. Outputs in order:
 *      the Lasso node, sum0 (= ct0is, K x 2n), sum1 (= ct1is). out_ids8 (may be NULL): node ids of u, e0, e1, k1, the Lasso node's
 *      input layer, the Lasso node, sum0, sum1. */
int hg_bfv_pk_configure(hg_circuit* c, size_t log2_size, size_t K, const uint64_t* qis, const uint64_t* k0is, const uint64_t* r1_bounds, const uint64_t* r2_bounds,
                        const uint64_t* p1_bounds, const uint64_t* p2_bounds, uint64_t u_bound, uint64_t e_bound, uint64_t k1_bound, hg_lasso_node* lasso_node,
                        const hg_lasso_pp* lasso_pp, size_t lasso_num_vars, int* out_ids8);
/* ---- synthetic witness of the public-key relation on the device, as hg_bfv_witness_generate for the SK one: exact products pk0_i u
 *      and pk1_i u over Z, centred reductions, the quotients r1 / r2 (ct0) and p1 / p2 (ct1) with their bound checks, in the input
 *      layout of hg_bfv_pk_configure. Host draws, lowest degree first: u in {-1,0,1}, e0, e1 as int8, k1 as int32, pk0 and pk1 as
 *      [K][n] int64 with |pk| < 2^59. Device outputs in the library's representation:
 *        d_u, d_e0, d_e1, d_k1: 2n elements;  d_pk0is, d_pk1is, d_r1is, d_p1is, d_ct0is, d_ct1is: K x 2n;  d_r2is, d_p2is: K x n.
 *      A witness that does not satisfy the relation is an error naming the component (ct0 / ct1) and the quotient. */
int hg_bfv_pk_witness_generate(hg_ctx* ctx, size_t n, size_t K, const uint64_t* qis, const uint64_t* k0is, const uint64_t* r1_bounds, const uint64_t* r2_bounds,
                               const uint64_t* p1_bounds, const uint64_t* p2_bounds, const int8_t* u, const int8_t* e0, const int8_t* e1, const int32_t* k1,
                               const int64_t* pk0, const int64_t* pk1, void* d_u, void* d_e0, void* d_e1, void* d_k1, void* d_pk0is, void* d_pk1is, void* d_r1is,
                               void* d_p1is, void* d_r2is, void* d_p2is, void* d_ct0is, void* d_ct1is);
/* ---- verifier: BfvEncrypt::verify (bfv-gkr/src/sk_encryption_circuit.rs:462-517) on the HOST, no GPU and no context.
 *      hg_circuit_new_host makes a circuit DESCRIPTION: the hg_circuit_insert_input / _fft / _vanilla / _connect calls above build it
 *      exactly as for a device circuit, the Lasso node is described by its preprocessing and num_vars (hg_circuit_insert_lasso_host);
 *      evaluate / prove calls on it fail. hg_gkr_verify is gkr::verify_gkr (:509-510): it reads the proof from `t` (made by
 *      hg_transcript_from_proof, or a caller-owned one with a read callback), checks every node's sumcheck and final evaluation and the
 *      Lasso node (as hg_lasso_node_verify), and leaves the claims on the input nodes in the hg_gkr_input_claim* getters. The
 *      caller finishes :512-516 by comparing each claim with the MLE of the corresponding input (hg_mle_eval_host).
 *      options3 as in hg_lasso_node_verify. Non-zero return = the reference's Err / panic. */
int hg_circuit_new_host(int field_id, hg_circuit** out);
int hg_circuit_insert_lasso_host(hg_circuit* c, const hg_lasso_pp* pp, size_t num_vars, int* out_id);
int hg_gkr_verify(hg_circuit* c, size_t n_output_claims, const size_t* point_lens, const uint64_t* points_ext, const uint64_t* values_ext, hg_transcript* t,
                  const int* options3);
/* MultilinearPoly::evaluate on the host: table of 2^num_vars base elements (canonical limbs), point of num_vars extension elements */
int hg_mle_eval_host(int field_id, const uint64_t* table_limbs, size_t n, size_t num_vars, const uint64_t* point_ext, uint64_t* out_ext);
/* ---- batched verifier on the device: B proofs of one circuit per call.
 *      hg_verifier_new takes a host-only description (hg_circuit_new_host + hg_bfv_configure or the insert / connect calls) of the
 *      context's field, uploads its wiring (edges and constants of the linear and general layers, the product edges of the general
 *      layers) and its Lasso subtables once, and serves batches of up to max_batch proofs. At most one Lasso node per circuit.
 *      hg_gkr_verify_batch verifies n_proofs proofs: each is replayed on the host exactly as hg_gkr_verify does (every transcript
 *      operation and scalar check), the checks whose cost is linear in the circuit size (FFT and linear layers at the sumcheck
 *      point, general layers at their two points, Lasso subtables, every input claim) are evaluated on the device for the whole
 *      batch, and quantities that several proofs share (the same points, as with hg_transcript_new / hg_transcript_from_proof)
 *      are computed once. It is hg_gkr_verify followed by the input-claim comparison of :512-516, with the same verdict.
 *        transcripts[p]      proof p's transcript (hg_transcript_from_proof, or a caller-owned one with a read callback), read as
 *                            hg_gkr_verify reads it; the caller can check for trailing bytes afterwards
 *        output claims       n_output_claims per proof with the same point_lens for every proof; proof p's points start at
 *                            points_ext + p * sum(point_lens) * X limbs, its values at values_ext + p * n_output_claims * X limbs
 *        inputs[p * I + i]   input node i of proof p (I input nodes, insertion order): device tables in the library's representation
 *                            (inputs_on_device = 1, as hg_bfv_witness_generate writes them) or host vectors of canonical limbs
 *        out_status[p]       1 accepted, 0 rejected; hg_verifier_reason(v, p) names the failed check of a rejected proof until
 *                            the next batch (only the reason may differ from hg_gkr_verify's, never the verdict)
 *      A malformed, truncated or tampered proof is a rejection, not an error. Invalid arguments, n_proofs > max_batch and CUDA
 *      failures return non-zero. */
int hg_verifier_new(hg_ctx* ctx, const hg_circuit* desc, size_t max_batch, hg_verifier** out);
void hg_verifier_free(hg_verifier* v);
int hg_gkr_verify_batch(hg_verifier* v, size_t n_proofs, hg_transcript* const* transcripts, size_t n_output_claims, const size_t* point_lens,
                        const uint64_t* points_ext, const uint64_t* values_ext, const void* const* inputs, int inputs_on_device, const int* options3,
                        int* out_status);
const char* hg_verifier_reason(const hg_verifier* v, size_t proof);
/* input nodes of the verifier's circuit and the elements of input i (insertion order; 0 out of range) */
size_t hg_verifier_num_inputs(const hg_verifier* v);
size_t hg_verifier_input_len(const hg_verifier* v, size_t input);
/* host microseconds of the last hg_gkr_verify_batch: [replays of every proof, device stages (enqueue and wait), closing the records] */
void hg_verifier_timing(const hg_verifier* v, double* out_us3);
/* MLEs of n_items base tables, each at its own point, on the device: table i has 2^num_vars[i] elements (device tables in the
 * library's representation when tables_on_device, else host vectors of canonical limbs); the points lie back to back in
 * points_ext (num_vars[i] extension elements each); out_ext receives one extension element per item */
int hg_mle_eval_multi(hg_ctx* ctx, size_t n_items, const void* const* tables, const size_t* num_vars, const uint64_t* points_ext, int tables_on_device,
                      uint64_t* out_ext);
/* host phases of the last hg_gkr_prove in microseconds: [witness kernels enqueue, squeeze+upload challenges, protocol walk,
 * batched layer enqueue, wait for the GPU, serialise]; number of extension challenges one proof squeezes */
void hg_gkr_timing(const hg_circuit* c, double* out_us6);
size_t hg_gkr_num_challenges(const hg_circuit* c);
size_t hg_gkr_num_inputs(const hg_circuit* c);
size_t hg_gkr_num_input_claims(const hg_circuit* c, size_t input);
size_t hg_gkr_input_claim_num_vars(const hg_circuit* c, size_t input, size_t k);
int hg_gkr_input_claim(const hg_circuit* c, size_t input, size_t k, uint64_t* point_ext, uint64_t* value_ext);

/* field self-test kernel: out[i] = a[i] (op) b[i] on extension elements, op 0 add 1 sub 2 mul (device arithmetic check) */
int hg_field_selftest(hg_ctx* ctx, int op, const uint64_t* a_ext, const uint64_t* b_ext, size_t n, uint64_t* out_ext);

#ifdef __cplusplus
}
#endif
#endif /* HG_B200_H */
