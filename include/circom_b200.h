/*
 * circom_b200 — C ABI of the Blackwell (sm_100a) witness-generation and R1CS
 * evaluation back end for circom circuits.
 *
 * This is the drop-in boundary a `code_producers/src/cuda_elements` producer
 * (sibling of c_elements / wasm_elements, code_producers/src/lib.rs:1-7) and its
 * Rust host would bind through FFI.  Every entry point names the piece of the
 * reference runtime it replaces.  Plain pointers and sizes only; all field
 * elements crossing the ABI are CANONICAL integers in [0,q) as 4 little-endian
 * uint64 limbs (the same 32 bytes the reference writes to .wtns,
 * c_elements/common/main.cpp:328-332).  Montgomery form is internal.
 *
 * Error convention: functions return CW_OK (0) or a negative CW_E* code;
 * cw_last_error() gives a thread-local message.  The reference instead
 * assert()s / throws (calcwit.cpp:60-66,80-92, main.cpp:168,265-274).
 *
 * Threading: handles are not shared between threads; one CUDA stream per batch.
 */
#ifndef CIRCOM_B200_H
#define CIRCOM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CW_OK 0
#define CW_EINVAL (-1)   /* bad argument */
#define CW_EIO (-2)      /* file problem */
#define CW_EFORMAT (-3)  /* malformed .cb2c / .r1cs / .wtns */
#define CW_ECUDA (-4)    /* CUDA runtime error (message in cw_last_error) */
#define CW_ENOTFOUND (-5)/* "Signal not found" (calcwit.cpp:60-66) */
#define CW_ESTATE (-6)   /* e.g. "Signal assigned twice" (calcwit.cpp:88-91), inputs missing */
#define CW_ENODEV (-7)   /* no CUDA device: the product has NO CPU fallback */

/* primes (program_structure/src/utils/constants.rs:3-6) */
#define CW_PRIME_BN128 0
#define CW_PRIME_BLS12381 1
/* the other primes of constants.rs:7-13 (one shared kernel build).  goldilocks (c_elements/goldilocks/fr.hpp:10-60) runs
 * in the same 32-byte elements with its upper 24 bytes zero; its .wtns / .r1cs files carry 8-byte elements
 * (c_elements/common64/main.cpp:327, constraint_list/src/r1cs_porting.rs:6-10) */
#define CW_PRIME_GRUMPKIN 2
#define CW_PRIME_PALLAS 3
#define CW_PRIME_VESTA 4
#define CW_PRIME_SECQ256R1 5
#define CW_PRIME_BLS12377 6
#define CW_PRIME_GOLDILOCKS 7

/* cw_circuit_load flags */
#define CW_FLAG_NO_ASSERTS 1u /* --sanity_check 0: drop `===` asserts (assert_bucket.rs:73) */
#define CW_FLAG_HOST_ONLY 2u  /* lower the tape but do not touch a GPU (CPU-side tests of the lowering) */
#define CW_FLAG_NO_PEEPHOLE 8u /* lower IR ops one to one (no bit-field / boolean-assert / shift fusions) */
#define CW_FLAG_BITPLANE 16u   /* bits written by bit runs live in a packed per-instance bit plane */
#define CW_FLAG_REUSE 32u      /* values that are not witness entries share slots (allocated like registers) */
#define CW_FLAG_FUSE 64u       /* single-use values are evaluated inside their reader's work item (two accumulators) instead
                                  of travelling through the value store: half the levels, 30 % fewer stores; pays only for large
                                  batches (measured: DESIGN.md section 7) */
#define CW_FLAG_NO_TYPED 128u /* keep the generic operators where the range analysis proves a narrower one exact (width-typed
                                  additions, multiplications and constant shifts; for A/B measurements and parity tests) */
#define CW_FLAG_COMPACT (CW_FLAG_BITPLANE | CW_FLAG_REUSE) /* the compact value store: what cw_batch_* runs best on */
#define CW_FLAG_O0 4u         /* --O0: keep every signal in the witness and every `signal = signal` constraint */

/* IR opcodes = OperatorType, compiler/src/intermediate_representation/compute_bucket.rs:7-34 */
enum cw_op {
    CW_OP_NOP = 0, CW_OP_MUL = 1, CW_OP_DIV = 2, CW_OP_ADD = 3, CW_OP_SUB = 4, CW_OP_POW = 5,
    CW_OP_IDIV = 6, CW_OP_MOD = 7, CW_OP_SHL = 8, CW_OP_SHR = 9, CW_OP_LEQ = 10, CW_OP_GEQ = 11,
    CW_OP_LT = 12, CW_OP_GT = 13, CW_OP_EQ = 14, CW_OP_NEQ = 15, CW_OP_LOR = 16, CW_OP_LAND = 17,
    CW_OP_LNOT = 18, CW_OP_BOR = 19, CW_OP_BAND = 20, CW_OP_BXOR = 21, CW_OP_BNOT = 22,
    CW_OP_NEG = 23, CW_OP_COPY = 24, CW_OP_SELECT = 25, CW_OP_ASSERT = 26, CW_OP_ASSERT_EQ = 27,
    /* device-only opcodes produced by the lowering */
    CW_OP_INV = 28
};

typedef struct cw_circuit cw_circuit; /* replaces Circom_Circuit (circom.hpp:36-43) + generated <name>.cpp */
typedef struct cw_batch cw_batch;     /* replaces Circom_CalcWit (calcwit.hpp:17-66), for `batch` inputs at once */
typedef struct cw_r1cs cw_r1cs;       /* CSR form of a .r1cs (constraint_writers/src/r1cs_writer.rs) */

typedef struct cw_stats {
    uint64_t n_signals;      /* get_total_signal_no() */
    uint64_t n_witness;      /* get_size_of_witness() */
    uint64_t n_inputs;       /* get_main_input_signal_no() */
    uint64_t n_outputs;      /* get_main_input_signal_start() - 1 */
    uint64_t n_components;   /* get_number_of_components() */
    uint64_t n_constants;    /* device constant-table entries */
    uint64_t n_ir_ops;       /* field operations before lowering (incl. moves) */
    uint64_t n_tape_ops;     /* device tape instructions after aliasing / form inference / DCE */
    uint64_t n_slots;        /* value slots per instance (32 B each) */
    uint64_t n_levels;       /* dependency levels */
    uint64_t n_constraints;  /* R1CS rows */
    uint64_t n_nnz;          /* nnz(A)+nnz(B)+nnz(C) */
    uint64_t n_mul_ops;      /* Montgomery multiplications in the tape (incl. conversions) */
    uint64_t n_conv_ops;     /* of which representation changes inserted by the lowering */
    uint64_t max_level_width;
    uint64_t n_slot_operands; /* operand reads of value slots in the tape */
    uint64_t n_bitwords;      /* 32-bit words of the per-instance bit plane (CW_FLAG_BITPLANE), else 0 */
    uint64_t n_resident_slots;/* slots holding witness entries; slots beyond are reused temporaries (CW_FLAG_REUSE) */
    uint64_t n_items;         /* work items of the tape: a work item is 1..24 tape words evaluated by one thread (single-use values
                                 fused into their reader); n_levels are levels of work items */
    uint64_t n_stored;        /* values that reach the value store per instance (n_values minus the fused ones) */
    uint64_t n_values;        /* values the tape computes per instance: every destination, each bit of a bit run (the S_w of SURVEY.md 8(d),
                                 independent of how the values are stored) */
} cw_stats;

/* ---- library ---------------------------------------------------------------------------- */
int cw_version(void);
const char *cw_last_error(void);
int cw_device_count(void); /* number of CUDA devices, 0 if none */

/* ---- circuit: load + lower (replaces loadCircuit main.cpp:22-124 and the g++ build of <name>.cpp) */
int cw_circuit_load(const char *cb2c_path, uint32_t flags, cw_circuit **out);
int cw_circuit_load_mem(const void *data, size_t len, uint32_t flags, cw_circuit **out);
void cw_circuit_destroy(cw_circuit *c);
int cw_circuit_stats(const cw_circuit *c, cw_stats *out);
int cw_circuit_prime(const cw_circuit *c, int *prime_id, uint64_t q[4]);
/* size getters, same meaning as circom.hpp:79-87 */
uint32_t cw_get_main_input_signal_start(const cw_circuit *c);
uint32_t cw_get_main_input_signal_no(const cw_circuit *c);
uint32_t cw_get_total_signal_no(const cw_circuit *c);
uint32_t cw_get_number_of_components(const cw_circuit *c);
uint32_t cw_get_size_of_input_hashmap(const cw_circuit *c);
uint32_t cw_get_size_of_witness(const cw_circuit *c);
uint32_t cw_get_size_of_constants(const cw_circuit *c);
/* FNV-1a 64 of a qualified input name (calcwit.cpp:17-24) */
uint64_t cw_fnv1a(const char *name);
/* Circom_CalcWit::getInputSignalSize (calcwit.cpp:99-102); CW_ENOTFOUND if absent */
int cw_get_input_signal_size(const cw_circuit *c, uint64_t name_hash, uint64_t *size);
/* global signal id of element 0 of that input (InputHashMap[pos].signalid, calcwit.cpp:86) */
int cw_get_input_signal_id(const cw_circuit *c, uint64_t name_hash, uint64_t *signal_id);
/* copies of the lowered tape for inspection / tests (sizes from cw_circuit_stats):
 * ops: n_tape_ops x 4 uint32 {opcode | flags<<8, a, b, c}; operand bit31 = constant-table index;
 * level_start: n_levels+1 uint32 (indexes WORK ITEMS, see cw_circuit_tape_items); witness_slot: n_witness uint32 (bit31 = value held in Montgomery form) */
int cw_circuit_tape(const cw_circuit *c, uint32_t *ops, uint32_t *level_start, uint32_t *witness_slot);
/* items: n_items+1 uint32 - work item k is the tape words [items[k], items[k+1]); level_start indexes work items.
 * Inner words of an item write an accumulator (destination field 0xFFFFFE / 0xFFFFFF), operands with bit 28 read one. */
int cw_circuit_tape_items(const cw_circuit *c, uint32_t *items);
/* value slots of one instance by the width the lowering's range analysis proves: out[0] one bit, out[1] <= 32 bits,
 * out[2] <= 64 bits, out[3] wider (today every slot is a 32-byte element; the census sizes a narrow-slot layout) */
int cw_circuit_slot_census(const cw_circuit *c, uint64_t out[4]);
/* the circuit's functions (FunctionCodeInfo, function.rs:9-20) as lowered: *n = their number; info (may be NULL) receives 4
 * words per function: {code offset, instructions, registers of a call frame after register allocation, parameters} */
int cw_circuit_functions(const cw_circuit *c, uint32_t *n, uint32_t *info);
/* witness2SignalList (calcwit.hpp:54-56, c_code_generator.rs:605-614): n_witness entries */
int cw_circuit_witness2signal(const cw_circuit *c, uint64_t *out);
/* the reference's .dat (generate_dat_file, c_code_generator.rs:818-865): input hash map (:575-603), witness2signal list
 * (:605-614), circuit constants in the 40-byte tagged Montgomery form (:616-679); the io-map section is empty */
int cw_circuit_write_dat(const cw_circuit *c, const char *path);
/* the compiler's .sym (constraint_writers/src/sym_writer.rs:4-38, dag/src/sym_porting.rs:16-33): one line per signal,
 * `signal id,witness index or -1,node id,main.<path>.<name>`.  Needs a description with a symbols section (docs/CB2C.md);
 * CW_ESTATE otherwise (also for circuits restored with cw_circuit_deserialize: the blob carries no names). */
int cw_circuit_write_sym(const cw_circuit *c, const char *path);

/* ---- batch: Circom_CalcWit for `batch` independent inputs on one GPU ------------------------ */
int cw_batch_create(const cw_circuit *c, uint32_t batch, int device, cw_batch **out);
void cw_batch_destroy(cw_batch *b);
/* how the batch lays its values out on the device: log2 of the instances per tile (0: one instance per CTA, lanes
 * along the ops of a level; 5: a warp per op over 32 instances), threads per CTA, bytes of value store per instance
 * (32 * n_slots + 4 * n_bitwords).  Environment overrides: CW_BT_LOG2, CW_THREADS. */
int cw_batch_layout(const cw_batch *b, uint32_t *bt_log2, uint32_t *threads, uint64_t *bytes_per_instance);
/* Circom_CalcWit::setInputSignal(h, i, val) for one instance (calcwit.cpp:77-97); host staging */
int cw_batch_set_input(cw_batch *b, uint32_t instance, uint64_t name_hash, uint32_t idx, const uint64_t limbs[4]);
/* getRemaingInputsToBeSet (calcwit.hpp:50-52) for one instance */
int cw_batch_remaining_inputs(const cw_batch *b, uint32_t instance, uint32_t *remaining);
/* bulk: inputs[batch][n_inputs][4] canonical, in main-input signal order; host or device pointer */
int cw_batch_set_inputs(cw_batch *b, const uint64_t *inputs, int is_device_ptr);
/* run(ctx) (calcwit.cpp:6, generated Main_run) for the whole batch; asynchronous on the batch stream */
int cw_batch_run(cw_batch *b);
int cw_batch_sync(cw_batch *b);
/* The text the reference prints for failed assert number `assert_no` (the k - 1 of cw_batch_status below):
 * "Failed assert in template/function <template>. Followed trace of components: main.<component path>"
 * (build_failed_assert_message, c_code_generator.rs:461-468; the description carries no line numbers, the trace needs
 * its symbols section - without it the message ends after the template name).  Writes at most cap bytes incl. the
 * terminator; *len = length of the whole message.  Not available on a circuit received through cw_circuit_broadcast. */
int cw_circuit_assert_info(const cw_circuit *c, uint32_t assert_no, char *buf, size_t cap, size_t *len);
/* What the log() calls of the circuit print for one witness (LogBucket, log_bucket.rs:104-162: the arguments of a call
 * separated by blanks, values as canonical decimals, a newline per call; calls in the reference's execution order).
 * witness = n_witness x 4 u64 in host memory.  Writes at most cap bytes incl. the terminator; *len = length of the whole text.
 * Arguments are strings, constants and signals (a producer logs an expression through the signal that holds it). */
int cw_circuit_format_log(const cw_circuit *c, const uint64_t *witness, char *buf, size_t cap, size_t *len);
/* the same for instance `inst` of a batch that has run (its witness row is fetched from the device) */
int cw_batch_log(cw_batch *b, uint32_t inst, char *buf, size_t cap, size_t *len);
/* per instance: 0 = ok, k>0 = first failed assert is IR assert number k-1, <0 = runtime error */
int cw_batch_status(cw_batch *b, int32_t *status);
/* getWitness(i) for all i and all instances, after Fr_toLongNormal (main.cpp:328-332):
 * out[batch][n_witness][4]; host pointer */
int cw_batch_get_witness(cw_batch *b, uint64_t *out);
/* the same on a helper thread, chunk by chunk (pack kernel + copy of chunk k+1 overlap the host-side expansion of
 * chunk k); meanwhile the caller may stage and run OTHER batches, whose tapes then execute under the transfer.
 * cw_batch_get_witness_wait returns the transfer's status; the batch must not be run again before it. */
int cw_batch_get_witness_async(cw_batch *b, uint64_t *out);
int cw_batch_get_witness_wait(cw_batch *b);
/* the packed records themselves (out[batch][info[0]] uint32; layout: cw_circuit_pack_info) for consumers that do
 * not need the reference's 32-byte rows */
int cw_batch_get_witness_packed(cw_batch *b, uint32_t *out_words);
/* packed-record layout: info = {words per instance, plane words, extra-bit words, u64 entries, full entries};
 * entry[n_witness] = (class << 30) | index - class 0: bit `index` of the plane section, 1: bit `index` of the
 * extra-bit section, 2: u64 entry `index`, 3: 32-byte entry `index`; the sections follow each other in that order */
int cw_circuit_pack_info(const cw_circuit *c, uint64_t info[5], uint32_t *entry);
/* host side of that layout: one packed record -> the n_witness canonical 32-byte rows of the instance (what
 * cw_batch_get_witness does per instance; zero-extension only).  store_bits: 0 = the widest vector stores the CPU
 * has, or at most 128 / 256 / 512.  cw_host_expand_isa names what 0 selects ("avx512" / "avx2" / "sse2"). */
int cw_circuit_expand_record(const cw_circuit *c, const uint32_t *record, uint64_t *rows, int store_bits);
const char *cw_host_expand_isa(void);
/* the worker threads of the expansion: count, NUMA pinning, store width (environment: CW_UNPACK_THREADS,
 * CW_UNPACK_PIN=0, CW_EXPAND_ISA=128|256|512) */
const char *cw_host_pool_info(void);
/* host-only probe of that expansion (no GPU): `reps` passes over n_inst instances of a fresh buffer; mode 0 = the
 * expansion itself (all-zero records), 1 = a plain streaming fill of the same bytes, 2 = memset; gbps[reps] */
int cw_host_expand_bench(const cw_circuit *c, uint32_t n_inst, uint32_t reps, int mode, double *gbps);
/* bytes that crossed PCIe in the last cw_batch_get_witness (entries proven to be bits / 64-bit values travel
 * packed and are zero-extended on the host; CW_PACKED_D2H=0 disables) */
uint64_t cw_batch_last_d2h_bytes(const cw_batch *b);
/* device pointer of the same array (valid until the next run / destroy) */
int cw_batch_witness_device(cw_batch *b, const uint64_t **dptr);
/* dense rows of instances [first, first + count) into caller-provided device memory (32-byte aligned,
 * count * n_witness * 32 bytes), asynchronously on the batch stream: the compact value store keeps the witness as
 * resident slots + a bit plane and materialises the reference's layout only on request */
int cw_batch_expand_witness(cw_batch *b, uint32_t first, uint32_t count, uint64_t *dst_device);
/* zero-copy view: witness row i starts at dptr + i*stride_elems*4 uint64 (the tape writes witness entries into
 * the first n_witness slots of each instance's slot store; stride_elems = slots per instance) */
int cw_batch_witness_strided(cw_batch *b, const uint64_t **dptr, uint64_t *stride_elems);
/* CUDA stream of the batch (cudaStream_t as void*) and last device time of run+gather in ms */
void *cw_batch_stream(cw_batch *b);
int cw_batch_last_ms(cw_batch *b, float *exec_ms, float *gather_ms);
/* writeBinWitness (main.cpp:288-334): byte-identical .wtns for one instance */
int cw_batch_write_wtns(cw_batch *b, uint32_t instance, const char *path);
/* same bytes into a caller buffer of 76 + 32*n_witness bytes (calculateWTNSBin, witness_calculator.js:212-276) */
int cw_batch_wtns_bytes(cw_batch *b, uint32_t instance, uint8_t *out, size_t cap, size_t *len);

/* ---- R1CS --------------------------------------------------------------------------------- */
/* constraints of the loaded circuit in witness numbering */
int cw_r1cs_from_circuit(const cw_circuit *c, cw_r1cs **out);
/* parse a .r1cs file (layout of constraint_writers/src/r1cs_writer.rs:93-101,49-72,246-269,328-341) */
int cw_r1cs_load(const char *path, cw_r1cs **out);
/* write it back in the reference's section order (constraint_list/src/r1cs_porting.rs:19-53); a count given as
 * CW_KEEP keeps the value the circuit / the loaded file carries */
#define CW_KEEP 0xFFFFFFFFu
int cw_r1cs_write(const cw_r1cs *r, const char *path, uint32_t n_pub_out, uint32_t n_pub_in, uint32_t n_prv_in);
int cw_r1cs_info(const cw_r1cs *r, uint64_t *n_wires, uint64_t *n_constraints, uint64_t *nnz, int *prime_id);
void cw_r1cs_destroy(cw_r1cs *r);
/* A.w o B.w == C.w for `batch` witnesses w[batch][n_wires][4] (canonical).  first_bad[i] = -1 if
 * instance i satisfies every constraint, else the smallest violated row.  New functionality: the
 * reference has no evaluator (constraint_writers/src/r1cs_reader.rs has no caller).
 * A device pointer must be 32-byte aligned (elements are read with 256-bit loads); CW_EINVAL otherwise. */
int cw_r1cs_check(cw_r1cs *r, const uint64_t *witness, int is_device_ptr, uint32_t batch, int device,
                  int64_t *first_bad, float *kernel_ms);

/* same, for witness rows `stride_elems` 32-byte elements apart (stride_elems >= n_wires) */
int cw_r1cs_check_strided(cw_r1cs *r, const uint64_t *witness, uint64_t stride_elems, int is_device_ptr, uint32_t batch,
                          int device, int64_t *first_bad, float *kernel_ms);

/* the witnesses of a batch where the tape left them (any tile layout, bit plane, reused temporaries): nothing is
 * copied or expanded, plane bits are read as bits, recomposition sums as words.  Runs on the batch's stream. */
int cw_r1cs_check_batch(cw_r1cs *r, cw_batch *b, int64_t *first_bad, float *kernel_ms);
/* how the check reads the constraints for one value layout (b: that batch's store; NULL: dense witness rows on `device`):
 * info = {general rows, integer rows - rows of small +-2^k terms decided over the integers unless a value they meet is
 * wide (csrc/r1cs_small.h; CW_R1CS_SMALL=0 turns them off) -, boolean rows checked on their own, compiled terms} */
int cw_r1cs_compiled_info(cw_r1cs *r, cw_batch *b, int device, uint64_t info[4]);
/* A.w, B.w, C.w of every constraint for instances [first, first + count) of a batch, left in device memory
 * ([count][n_constraints][4] uint64 each, canonical, 32-byte aligned) for the prover stage that follows witness
 * generation; asynchronous on the batch stream (cw_batch_sync).  One-instance tile layouts only. */
int cw_r1cs_eval_batch(cw_r1cs *r, cw_batch *b, uint32_t first, uint32_t count, uint64_t *a_dev, uint64_t *b_dev,
                       uint64_t *c_dev);

/* ---- multi-GPU: one process per GPU, independent inputs sharded over the ranks ---------------------------
 * The reference has no distributed mode (Circom_CalcWit is per-process state, calcwit.cpp:26-45).  Here rank 0
 * lowers the circuit and broadcasts the lowered form once; every rank runs its shard; witnesses are gathered in
 * packed form.  NCCL is resolved at run time (dlopen of libnccl.so.2, or CW_NCCL_LIB); without it these entry
 * points return CW_ENODEV and everything else works. */
typedef struct cw_comm cw_comm;
#define CW_COMM_ID_BYTES 128
/* ncclGetUniqueId: call on one rank, hand the bytes to the others through the host program's own channel */
int cw_comm_unique_id(uint8_t id[CW_COMM_ID_BYTES]);
/* ncclCommInitRank (collective over `world` processes); `device` = this rank's CUDA device */
int cw_comm_init(const uint8_t id[CW_COMM_ID_BYTES], int rank, int world, int device, cw_comm **out);
/* adopt a communicator the host program already has (ncclComm_t as void*); not destroyed by cw_comm_destroy */
int cw_comm_from_nccl(void *nccl_comm, int rank, int world, int device, cw_comm **out);
void cw_comm_destroy(cw_comm *c);
/* payload bytes this rank sent / received through the collectives below */
int cw_comm_stats(const cw_comm *c, uint64_t *bytes_sent, uint64_t *bytes_received);
/* the lowered circuit as a blob (instruction tape, constants, witness maps, function code, input tables, CSR):
 * cw_circuit_serialize with out = NULL returns the size */
int cw_circuit_serialize(const cw_circuit *c, uint8_t *out, size_t cap, size_t *len);
int cw_circuit_deserialize(const void *data, size_t len, cw_circuit **out);
/* ONE broadcast of the lowered circuit from `root`: *c is the root's circuit on the root and receives a new handle
 * on the other ranks (which never run the lowering) */
int cw_circuit_broadcast(cw_comm *cm, cw_circuit **c, int root);
/* packed records of instances [first, first + count) into caller-provided DEVICE memory (count * words * 4 bytes,
 * words = cw_circuit_pack_info info[0]); asynchronous on the batch stream */
int cw_batch_pack_device(cw_batch *b, uint32_t first, uint32_t count, uint32_t *dst_device);
/* gather of witness vectors on `root`: every rank packs instances [first, first + count) of its batch and sends the
 * records over NVLink (grouped ncclSend / ncclRecv on the batch stream).  Root: recv_device[world][count][words];
 * other ranks: send_scratch_device[count][words].  ms = device time of pack + transfer on this rank. */
int cw_batch_gather_witness_packed(cw_comm *cm, cw_batch *b, uint32_t first, uint32_t count, int root,
                                   uint32_t *recv_device, uint32_t *send_scratch_device, float *ms);
/* out[0] = instances with a failed assert, out[1] = instances with a runtime error, summed over all ranks */
int cw_status_allreduce(cw_comm *cm, cw_batch *b, uint64_t out[2]);

/* ---- file boundary (the consumers of these files: snarkjs, rapidsnark) ---------------------------------- */
/* the entries of a .wtns (layout main.cpp:288-334): out[n_witness][4] canonical limbs; out = NULL returns the count */
int cw_wtns_read(const char *path, int *prime_id, uint64_t *n_witness, uint64_t *out, size_t cap_entries);
/* A.w o B.w == C.w for a .wtns file against a .r1cs file: *first_bad = -1 or the smallest violated row */
int cw_r1cs_check_files(const char *r1cs_path, const char *wtns_path, int device, int64_t *first_bad);

/* ---- field library, batched (parity tests of the device Fr_* equivalents, fr.hpp:28-70) ------ */
/* r[i] = op(a[i], b[i], c[i]) for i < n on `device`; canonical in / canonical out; b, c may be NULL */
int cw_fr_batch_op(int prime_id, int op, const uint64_t *a, const uint64_t *b, const uint64_t *c,
                   uint64_t *r, size_t n, int device);
/* Montgomery-multiplication throughput probe: n independent chains of `iters` dependent multiplications;
 * returns device milliseconds */
int cw_fr_mul_bench(int prime_id, size_t n, int iters, int device, float *ms);

#ifdef __cplusplus
}
#endif
#endif
