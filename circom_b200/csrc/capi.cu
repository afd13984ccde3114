// C ABI (include/circom_b200.h) over the lowering (flatten.cpp), the formats (formats.cpp) and the
// sm_100a kernels (kernels.cuh).  There is no CPU execution path: every compute entry point
// returns CW_ENODEV when no CUDA device is present.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <emmintrin.h>
#include <nccl.h>

#include <cstdio>
#include <cstdlib>
#include <algorithm>
#include <chrono>
#include <condition_variable>
#include <cstring>
#include <functional>
#include <map>
#include <memory>
#include <mutex>
#include <thread>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/circom_b200.h"
#include "kernels.cuh"
#include "tape_calls.h"
#include "tape.h"
#include "hostpack.h"

using namespace cw;

namespace {

thread_local std::string g_err;
int fail(int code, const std::string &msg) {
    g_err = msg;
    return code;
}
#define CU(call)                                                                                       \
    do {                                                                                               \
        cudaError_t e_ = (call);                                                                       \
        if (e_ != cudaSuccess)                                                                         \
            return fail(CW_ECUDA, std::string(#call) + ": " + cudaGetErrorString(e_));                 \
    } while (0)

FrParams make_dev_params(const FieldParams &F) {
    FrParams p;
    memset(&p, 0, sizeof(p));
    auto split = [](u32 *dst, const U256 &v) {
        for (int i = 0; i < 4; ++i) {
            dst[2 * i] = (u32)v.v[i];
            dst[2 * i + 1] = (u32)(v.v[i] >> 32);
        }
    };
    split(p.q, F.q);
    split(p.half, F.half);
    split(p.r1, F.r1);
    split(p.r2, F.r2);
    U256 two = u256_from_u64(2), qm2;
    u256_sub(qm2, F.q, two);
    split(p.qm2, qm2);
    p.np32 = F.np32;
    p.qbits = F.qbits;
    // lboMask of the limb that holds the top bit; fr_mask_wrap clears the limbs above it (goldilocks: limb 1, all ones)
    p.top_mask = (F.qbits % 32 == 0) ? 0xFFFFFFFFu : ((1u << (F.qbits % 32)) - 1u);
    return p;
}

std::mutex g_dev_mutex;
std::map<int, bool> g_dev_ready;

int ensure_device(int device) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) {
        cudaGetLastError();
        return fail(CW_ENODEV, "no CUDA device available (circom_b200 has no CPU execution path)");
    }
    if (device < 0 || device >= n) return fail(CW_EINVAL, "bad device index");
    CU(cudaSetDevice(device));
    std::lock_guard<std::mutex> lk(g_dev_mutex);
    if (!g_dev_ready[device]) {
        FrParams h[N_PRIMES_DEV];
        static_assert(N_PRIMES_DEV == CW_N_PRIMES, "prime tables");
        for (int k = 0; k < N_PRIMES_DEV; ++k) h[k] = make_dev_params(make_field(k));
        CU(cudaMemcpyToSymbol(c_fr, h, sizeof(h)));
        CU(tape_calls_set_params(h, sizeof(h)));
        g_dev_ready[device] = true;
    }
    return CW_OK;
}

struct DevTape {
    uint4 *ops = nullptr;
    u32 *items = nullptr, *level_start = nullptr, *level_info = nullptr;
    bool has_slow = false;
    uint4 *heads = nullptr;  // first tape word of every work item
    uint4 *consts = nullptr;
    u32 *input_slot = nullptr, *fn_code = nullptr, *fn_info = nullptr, *call_tab = nullptr;
    u32 *wloc = nullptr;  // per witness entry: where its value lives (slot id, or OPD_BIT | plane position)
    // witness entries outside the bit plane by static size class (slot ids), for the packed device->host transfer
    u32 *pk_bit = nullptr, *pk_u64 = nullptr, *pk_full = nullptr;
};
struct DevR1cs {
    unsigned long long *row_ptr = nullptr;
    uint4 *terms = nullptr;  // per term {location, dictionary index, kind word, absorbed boolean row}
    uint4 *dictM = nullptr;
    u32 *perm = nullptr, *bool_loc = nullptr, *bool_row = nullptr;
    u32 *perm_small = nullptr;   // rows small by shape: decided over the integers (r1cs_small.h)
    uint2 *sgroups = nullptr, *srecs = nullptr;   // ... from a term list of their own
    u32 *sbrow = nullptr;
    u32 n_general = 0, n_bool = 0, n_small = 0;
    u32 mean_row_terms = 0;  // compiled terms per general row
    uint64_t n_terms = 0;
};

template <class T>
int upload(T **dst, const void *src, size_t bytes) {
    CU(cudaMalloc((void **)dst, bytes ? bytes : 16));
    if (bytes) CU(cudaMemcpy(*dst, src, bytes, cudaMemcpyHostToDevice));
    return CW_OK;
}

int env_int(const char *name, int dflt) {
    const char *s = getenv(name);
    return s && *s ? atoi(s) : dflt;
}

}  // namespace

// Packed-transfer layout from the classes the witness values were SEEN to have (narrower than the proven ones; kernels.cuh:
// witness_observe_kernel), with the device copies of its location lists.  One per circuit and device, replaced (never
// edited) when a batch shows a wider value; transfers hold a reference while they use it.
struct NarrowPack {
    PackLayout L;
    std::vector<uint8_t> cls;
    u32 *pk_bit = nullptr, *pk_u64 = nullptr, *pk_full = nullptr;
    ~NarrowPack() {
        cudaFree(pk_bit);
        cudaFree(pk_u64);
        cudaFree(pk_full);
    }
};

struct cw_circuit {
    Tape tape;
    mutable std::mutex mu;
    mutable std::mutex narrow_mu;   // serialises the (rare) observation passes
    mutable std::map<int, std::shared_ptr<NarrowPack>> narrow;   // guarded by mu
    mutable std::map<int, DevTape> dev;
    mutable PackLayout pack;
    mutable bool pack_ready = false;
    const PackLayout &pack_layout() const {
        std::lock_guard<std::mutex> lk(mu);
        if (!pack_ready) {
            build_pack_layout(tape, pack);
            pack_ready = true;
        }
        return pack;
    }
};

struct R1csKey {
    int device;
    const cw_circuit *layout;  // nullptr: dense witness rows (location = wire id)
    bool operator<(const R1csKey &o) const { return device != o.device ? device < o.device : layout < o.layout; }
};
struct cw_r1cs {
    R1csData data;
    FieldParams F;
    std::mutex mu;
    std::map<R1csKey, DevR1cs> dev;
    cw_r1cs *eval_twin = nullptr;  // the same constraints compiled without boolean-row special cases (cw_r1cs_eval_batch)
    bool no_bool_rows = false;
};

struct cw_batch {
    const cw_circuit *c = nullptr;
    int device = 0;
    u32 batch = 0, batch_padded = 0, bt_log2 = 0, threads = 256;
    cudaStream_t stream = nullptr;
    uint4 *slots = nullptr, *inputs_d = nullptr, *witness_d = nullptr;
    u32 *plane = nullptr;
    u32 *first_assert_d = nullptr;
    int *err_d = nullptr;
    unsigned long long *fb_d = nullptr;  // per-instance result of the R1CS check
    u32 *r1cs_wide_d = nullptr;          // bitmap of the integer rows handed to the general kernel (launch_r1cs)
    u32 r1cs_wide_rows = 0;
    DevTape dt;
    std::vector<uint64_t> host_inputs;  // [batch][n_inputs][4]
    std::vector<uint8_t> assigned;      // [batch][n_inputs]
    std::vector<u32> remaining;         // [batch]
    bool host_inputs_dirty = false;
    bool inputs_on_device = false;
    bool ran = false;
    bool dense_valid = false;  // witness_d holds the dense rows of the current run
    // packed transfer: two staging buffers (device + pinned host) so that the pack kernel and the copy of one
    // chunk overlap the host-side expansion of the previous one
    u32 *packed_d[2] = {nullptr, nullptr}, *packed_h[2] = {nullptr, nullptr};
    size_t packed_cap = 0;  // instances per staging buffer
    uint4 *dense_chunk_d = nullptr;
    size_t dense_chunk_cap = 0;
    int *pack_flag_d = nullptr;
    cudaEvent_t pack_ev[2] = {nullptr, nullptr};
    uint64_t last_d2h_bytes = 0;
    cudaEvent_t ev[3] = {nullptr, nullptr, nullptr};
    std::thread async_th;  // cw_batch_get_witness_async
    int async_rc = 0;
    std::string async_err;
    bool async_active = false;
    bool identity_layout() const {  // witness row i = the first n_witness slots of instance i's slot store
        const Tape &t = c->tape;
        return bt_log2 == 0 && t.n_bitwords == 0 && t.n_resident == t.n_witness;
    }
    StoreDev store() const {
        StoreDev S;
        S.slots = slots;
        S.plane = plane;
        S.n_slots = c->tape.n_slots;
        S.n_bitwords = c->tape.n_bitwords;
        S.bt_log2 = bt_log2;
        S.batch = batch;
        return S;
    }
};

static int get_dev_tape(const cw_circuit *c, int device, DevTape &out) {
    const PackLayout &L = c->pack_layout();
    std::lock_guard<std::mutex> lk(c->mu);
    auto it = c->dev.find(device);
    if (it != c->dev.end()) {
        out = it->second;
        return CW_OK;
    }
    const Tape &t = c->tape;
    DevTape d;
    int rc;
    if ((rc = upload(&d.ops, t.ops.data(), t.ops.size() * 4))) return rc;
    if ((rc = upload(&d.items, t.items.data(), t.items.size() * 4))) return rc;
    {
        std::vector<uint32_t> heads(t.n_items() * 4);
        for (size_t k = 0; k < t.n_items(); ++k) memcpy(&heads[k * 4], &t.ops[(size_t)t.items[k] * 4], 16);
        if ((rc = upload(&d.heads, heads.data(), heads.size() * 4))) return rc;
    }
    if ((rc = upload(&d.level_start, t.level_start.data(), t.level_start.size() * 4))) return rc;
    {
        // per level: how many calls close it (the lowering sorts the items of a level by opcode, CALL is the largest: the
        // kernel runs them after the other items) and whether it has INV / POW items (run in a pass of their own)
        std::vector<uint32_t> info(t.n_levels(), 0);
        for (size_t l = 0; l < t.n_levels(); ++l) {
            bool tail = true;
            for (uint32_t k = t.level_start[l + 1]; k-- > t.level_start[l];) {
                const uint32_t opc = t.ops[(size_t)t.items[k] * 4] & 0xFFu;
                const bool single = t.items[k + 1] - t.items[k] == 1;
                const bool is_call = opc == 45u && single;
                if (opc == 45u && !(single && tail)) return fail(CW_ESTATE, "internal: a call is not at the end of its level");
                if (is_call) ++info[l];
                else tail = false;
                for (uint32_t w = t.items[k]; w < t.items[k + 1]; ++w) {
                    const uint32_t o = t.ops[(size_t)w * 4] & 0xFFu;
                    if (o == 28u || o == 5u) {   // INV, POW
                        if (!single) return fail(CW_ESTATE, "internal: a fused work item contains INV / POW");
                        info[l] |= 0x80000000u;
                        d.has_slow = true;
                    }
                }
            }
        }
        if ((rc = upload(&d.level_info, info.data(), info.size() * 4))) return rc;
    }
    if ((rc = upload(&d.consts, t.consts.data(), t.consts.size() * 32))) return rc;
    if ((rc = upload(&d.input_slot, t.input_slot.data(), t.input_slot.size() * 4))) return rc;
    if ((rc = upload(&d.fn_code, t.fn_code.data(), t.fn_code.size() * 4))) return rc;
    if ((rc = upload(&d.fn_info, t.fn_info.data(), t.fn_info.size() * 4))) return rc;
    if ((rc = upload(&d.call_tab, t.call_tab.data(), t.call_tab.size() * 4))) return rc;
    if ((rc = upload(&d.wloc, t.witness_slot.data(), t.witness_slot.size() * 4))) return rc;
    if ((rc = upload(&d.pk_bit, L.bit_loc.data(), L.bit_loc.size() * 4))) return rc;
    if ((rc = upload(&d.pk_u64, L.u64_loc.data(), L.u64_loc.size() * 4))) return rc;
    if ((rc = upload(&d.pk_full, L.full_loc.data(), L.full_loc.size() * 4))) return rc;
    c->dev[device] = d;
    out = d;
    return CW_OK;
}

// builds of the interpreter: function calls (runtime tile size); fused work items (CW_FLAG_FUSE; runtime tile size, or
// a warp per op); one operator per work item, per bit-plane mode: one instance per tile / a warp per op (tile sizes
// fixed at compile time) / tile size as an argument
template <int PR, bool CALLS, bool BP, int BT, bool FU>
static void launch_tape_k(const TapeDev &tp, cw_batch *b, u32 tiles, u32 th) {
    static_assert(tape_acc_smem(CW_TAPE_LB) <= 48u * 1024u, "the accumulators of the widest CTA need an opt-in shared-memory size");
    tape_exec_kernel<PR, CALLS, BP, BT, FU><<<tiles, th, FU ? tape_acc_smem(th) : 0u, b->stream>>>(
        tp, b->slots, b->plane, b->bt_log2, b->first_assert_d, b->err_d, b->batch);
}
template <int PR>
static void launch_tape(const TapeDev &tp, cw_batch *b, u32 tiles, u32 th, bool calls, bool bp, bool fused) {
    if (calls) {  // the builds with the function machine: tape_calls.cu
        launch_tape_calls(PR, tp, b->slots, b->plane, b->bt_log2, b->first_assert_d, b->err_d, b->batch, tiles, th, bp, fused,
                          b->stream);
    } else if (fused) {  // (the bit-plane build also runs tapes without a plane: they contain no plane operands)
        if (b->bt_log2 == 5) launch_tape_k<PR, false, true, 5, true>(tp, b, tiles, th);
        else launch_tape_k<PR, false, true, -1, true>(tp, b, tiles, th);
    } else if (bp) {
        if (b->bt_log2 == 0) launch_tape_k<PR, false, true, 0, false>(tp, b, tiles, th);
        else if (b->bt_log2 == 5) launch_tape_k<PR, false, true, 5, false>(tp, b, tiles, th);
        else launch_tape_k<PR, false, true, -1, false>(tp, b, tiles, th);
    } else {
        if (b->bt_log2 == 0) launch_tape_k<PR, false, false, 0, false>(tp, b, tiles, th);
        else launch_tape_k<PR, false, false, -1, false>(tp, b, tiles, th);
    }
}

extern "C" {

int cw_version(void) { return 100; }
const char *cw_last_error(void) { return g_err.c_str(); }
int cw_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

int cw_circuit_load_mem(const void *data, size_t len, uint32_t flags, cw_circuit **out) {
    if (!data || !out) return fail(CW_EINVAL, "null argument");
    cw_circuit *c = new cw_circuit();
    try {
        lower_circuit((const uint8_t *)data, len, flags, c->tape);
    } catch (const std::exception &e) {
        delete c;
        return fail(CW_EFORMAT, e.what());
    }
    *out = c;
    return CW_OK;
}

int cw_circuit_load(const char *path, uint32_t flags, cw_circuit **out) {
    if (!path || !out) return fail(CW_EINVAL, "null argument");
    FILE *f = fopen(path, "rb");
    if (!f) return fail(CW_EIO, std::string("cannot open ") + path);
    fseek(f, 0, SEEK_END);
    long sz = ftell(f);
    fseek(f, 0, SEEK_SET);
    std::vector<uint8_t> buf(sz);
    size_t rd = sz ? fread(buf.data(), 1, sz, f) : 0;
    fclose(f);
    if ((long)rd != sz) return fail(CW_EIO, "short read");
    return cw_circuit_load_mem(buf.data(), buf.size(), flags, out);
}

void cw_circuit_destroy(cw_circuit *c) {
    if (!c) return;
    for (auto &kv : c->dev) {
        cudaSetDevice(kv.first);
        cudaFree(kv.second.ops);
        cudaFree(kv.second.items);
        cudaFree(kv.second.heads);
        cudaFree(kv.second.level_start);
        cudaFree(kv.second.level_info);
        cudaFree(kv.second.consts);
        cudaFree(kv.second.input_slot);
        cudaFree(kv.second.fn_code);
        cudaFree(kv.second.fn_info);
        cudaFree(kv.second.call_tab);
        cudaFree(kv.second.wloc);
        cudaFree(kv.second.pk_bit);
        cudaFree(kv.second.pk_u64);
        cudaFree(kv.second.pk_full);
    }
    delete c;
}

int cw_circuit_stats(const cw_circuit *c, cw_stats *o) {
    if (!c || !o) return fail(CW_EINVAL, "null argument");
    const Tape &t = c->tape;
    memset(o, 0, sizeof(*o));
    o->n_signals = t.n_signals;
    o->n_witness = t.n_witness;
    o->n_inputs = t.n_inputs;
    o->n_outputs = t.n_outputs;
    o->n_components = t.n_components;
    o->n_constants = t.consts.size();
    o->n_ir_ops = t.n_ir_ops;
    o->n_tape_ops = t.n_tape_ops();
    o->n_slots = t.n_slots;
    o->n_levels = t.n_levels();
    o->n_constraints = t.r1cs.n_constraints;
    o->n_nnz = t.r1cs.col.size();
    o->n_mul_ops = t.n_mul_ops;
    o->n_conv_ops = t.n_conv_ops;
    o->max_level_width = t.max_level_width;
    o->n_slot_operands = t.n_slot_operands;
    o->n_bitwords = t.n_bitwords;
    o->n_resident_slots = t.n_resident;
    o->n_values = t.n_values;
    o->n_items = t.n_items();
    o->n_stored = t.n_stored;
    return CW_OK;
}

int cw_circuit_prime(const cw_circuit *c, int *prime_id, uint64_t q[4]) {
    if (!c) return fail(CW_EINVAL, "null argument");
    if (prime_id) *prime_id = c->tape.F.prime_id;
    if (q) memcpy(q, c->tape.F.q.v, 32);
    return CW_OK;
}

uint32_t cw_get_main_input_signal_start(const cw_circuit *c) { return (uint32_t)c->tape.n_outputs + 1; }
uint32_t cw_get_main_input_signal_no(const cw_circuit *c) { return (uint32_t)c->tape.n_inputs; }
uint32_t cw_get_total_signal_no(const cw_circuit *c) { return (uint32_t)c->tape.n_signals; }
uint32_t cw_get_number_of_components(const cw_circuit *c) { return (uint32_t)c->tape.n_components; }
uint32_t cw_get_size_of_input_hashmap(const cw_circuit *c) { return (uint32_t)c->tape.hashmap.size(); }
uint32_t cw_get_size_of_witness(const cw_circuit *c) { return (uint32_t)c->tape.n_witness; }
uint32_t cw_get_size_of_constants(const cw_circuit *c) { return (uint32_t)c->tape.consts.size(); }

uint64_t cw_fnv1a(const char *name) { return fnv1a(name, strlen(name)); }

// getInputSignalHashPosition (calcwit.cpp:51-69)
static int hash_pos(const Tape &t, uint64_t h, size_t *pos) {
    size_t n = t.hashmap.size();
    size_t p = (size_t)(h % n);
    if (t.hashmap[p].hash != h || t.hashmap[p].signalid == 0) {
        size_t ini = p;
        p = (p + 1) % n;
        while (p != ini) {
            if (t.hashmap[p].hash == h && t.hashmap[p].signalid != 0) {
                *pos = p;
                return CW_OK;
            }
            if (t.hashmap[p].signalid == 0) return fail(CW_ENOTFOUND, "Signal not found");
            p = (p + 1) % n;
        }
        return fail(CW_ENOTFOUND, "Signals not found");
    }
    *pos = p;
    return CW_OK;
}

int cw_get_input_signal_size(const cw_circuit *c, uint64_t h, uint64_t *size) {
    size_t p;
    int rc = hash_pos(c->tape, h, &p);
    if (rc) return rc;
    *size = c->tape.hashmap[p].signalsize;
    return CW_OK;
}
int cw_get_input_signal_id(const cw_circuit *c, uint64_t h, uint64_t *id) {
    size_t p;
    int rc = hash_pos(c->tape, h, &p);
    if (rc) return rc;
    *id = c->tape.hashmap[p].signalid;
    return CW_OK;
}

int cw_circuit_tape_items(const cw_circuit *c, uint32_t *items) {
    if (!c || !items) return fail(CW_EINVAL, "null argument");
    memcpy(items, c->tape.items.data(), c->tape.items.size() * 4);
    return CW_OK;
}

int cw_circuit_tape(const cw_circuit *c, uint32_t *ops, uint32_t *level_start, uint32_t *witness_slot) {
    const Tape &t = c->tape;
    if (ops) memcpy(ops, t.ops.data(), t.ops.size() * 4);
    if (level_start) memcpy(level_start, t.level_start.data(), t.level_start.size() * 4);
    if (witness_slot) memcpy(witness_slot, t.witness_slot.data(), t.witness_slot.size() * 4);
    return CW_OK;
}

int cw_circuit_slot_census(const cw_circuit *c, uint64_t out[4]) {
    if (!c || !out) return fail(CW_EINVAL, "null argument");
    memcpy(out, c->tape.slot_census, sizeof(c->tape.slot_census));
    return CW_OK;
}

int cw_circuit_witness2signal(const cw_circuit *c, uint64_t *out) {
    if (!c || !out) return fail(CW_EINVAL, "null argument");
    memcpy(out, c->tape.witness2signal.data(), c->tape.witness2signal.size() * 8);
    return CW_OK;
}

int cw_circuit_write_dat(const cw_circuit *c, const char *path) {
    try {
        write_dat(c->tape, path);
    } catch (const std::exception &e) {
        return fail(CW_EIO, e.what());
    }
    return CW_OK;
}

int cw_circuit_functions(const cw_circuit *c, uint32_t *n, uint32_t *info) {
    if (!c || !n) return fail(CW_EINVAL, "null argument");
    *n = (uint32_t)(c->tape.fn_info.size() / 4);
    if (info) memcpy(info, c->tape.fn_info.data(), c->tape.fn_info.size() * 4);
    return CW_OK;
}

int cw_circuit_write_sym(const cw_circuit *c, const char *path) {
    if (!c || !path) return fail(CW_EINVAL, "null argument");
    if (c->tape.sym.empty()) return fail(CW_ESTATE, "the circuit description carries no symbols section");
    try {
        write_sym(c->tape, path);
    } catch (const std::exception &e) {
        return fail(CW_EIO, e.what());
    }
    return CW_OK;
}

// ---- batch ------------------------------------------------------------------------------------
int cw_batch_create(const cw_circuit *c, uint32_t batch, int device, cw_batch **out) {
    if (!c || !out || batch == 0) return fail(CW_EINVAL, "bad argument");
    if (c->tape.flags & CW_FLAG_HOST_ONLY) return fail(CW_ESTATE, "circuit was loaded with CW_FLAG_HOST_ONLY");
    int rc = ensure_device(device);
    if (rc) return rc;
    const Tape &t = c->tape;
    cw_batch *b = new cw_batch();
    b->c = c;
    b->device = device;
    b->batch = batch;
    // Tile size (instances side by side in the slot store).  Lanes along instances (32-instance tiles: a warp is one
    // op, every access coalesced, no divergence) need enough tiles to fill the GPU with CTAs; below that, lanes run
    // along the ops of a level (one-instance tiles).
    int bt = env_int("CW_BT_LOG2", -1);
    const uint64_t avg_w = t.n_levels() ? t.n_items() / t.n_levels() + 1 : 1;
    if (bt < 0) {
        bt = 0;
        if (batch >= 32u * 148u * 2u) bt = 5;   // (also with function calls: the 32 lanes run the same function body)
        else if (t.call_tab.empty())
            while (bt < 5 && (avg_w << bt) < 64 && (batch >> (bt + 1)) >= 296u) ++bt;  // very narrow tapes (Poseidon)
    }
    if (bt > 5) bt = 5;
    b->bt_log2 = (u32)bt;
    u32 btn = 1u << bt;
    b->batch_padded = (batch + btn - 1) / btn * btn;
    int th = env_int("CW_THREADS", 0);
    if (th <= 0) {
        // enough threads for a typical level: average width x tile, clamped to [64, 512]
        uint64_t avg = avg_w * btn;
        th = 64;
        while (th < 512 && (uint64_t)th < avg) th <<= 1;
        // many tiles per SM hide latency better than wide CTAs: keep <= ~1024 resident threads per SM
        // (measured on B200: batch 256 -> 512 threads, 512 -> 256, 1024 -> 128)
        u32 tiles = b->batch_padded >> bt;
        u32 per_sm = (tiles + 147) / 148;
        while (th > 64 && (u32)th * per_sm > 1024) th >>= 1;
        if (tiles < 148u) th = CW_TAPE_LB;  // fewer tiles than SMs: the widest CTA (wide levels finish in one pass; measured 6.5 vs 7.6 ms at 8 instances)
    }
    th = (th + 31) / 32 * 32;
    if (th > CW_TAPE_LB) th = CW_TAPE_LB;
    b->threads = (u32)th;
    size_t slot_bytes = (size_t)b->batch_padded * t.n_slots * 32;
    size_t plane_bytes = (size_t)b->batch_padded * t.n_bitwords * 4;
    size_t free_b = 0, total_b = 0;
    cudaMemGetInfo(&free_b, &total_b);
    size_t need = slot_bytes + plane_bytes + (size_t)batch * t.n_inputs * 32 + (64u << 20);
    if (need > free_b) {
        delete b;
        return fail(CW_ECUDA, "batch needs " + std::to_string(need >> 20) + " MiB of device memory, " +
                                  std::to_string(free_b >> 20) + " MiB free");
    }
    if ((rc = get_dev_tape(c, device, b->dt))) { delete b; return rc; }
    CU(cudaStreamCreateWithFlags(&b->stream, cudaStreamNonBlocking));
    CU(cudaMalloc((void **)&b->slots, slot_bytes));
    CU(cudaMalloc((void **)&b->plane, std::max<size_t>(plane_bytes, 16)));
    CU(cudaMalloc((void **)&b->inputs_d, std::max<size_t>((size_t)batch * t.n_inputs * 32, 32)));
    CU(cudaMalloc((void **)&b->first_assert_d, (size_t)batch * 4));
    CU(cudaMalloc((void **)&b->err_d, (size_t)batch * 4));
    CU(cudaMalloc((void **)&b->fb_d, (size_t)batch * 8));
    for (auto &e : b->ev) CU(cudaEventCreate(&e));
    for (auto &e : b->pack_ev) CU(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    b->host_inputs.assign((size_t)batch * t.n_inputs * 4, 0);
    b->assigned.assign((size_t)batch * t.n_inputs, 0);
    b->remaining.assign(batch, (u32)t.n_inputs);
    *out = b;
    return CW_OK;
}

static void join_async(cw_batch *b) {
    if (b->async_th.joinable()) b->async_th.join();
    b->async_active = false;
}

void cw_batch_destroy(cw_batch *b) {
    if (!b) return;
    join_async(b);
    cudaSetDevice(b->device);
    cudaFree(b->slots);
    cudaFree(b->plane);
    cudaFree(b->inputs_d);
    cudaFree(b->witness_d);
    cudaFree(b->dense_chunk_d);
    for (int k = 0; k < 2; ++k) {
        cudaFree(b->packed_d[k]);
        if (b->packed_h[k]) cudaFreeHost(b->packed_h[k]);
        if (b->pack_ev[k]) cudaEventDestroy(b->pack_ev[k]);
    }
    cudaFree(b->pack_flag_d);
    cudaFree(b->first_assert_d);
    cudaFree(b->err_d);
    cudaFree(b->fb_d);
    cudaFree(b->r1cs_wide_d);
    for (auto &e : b->ev)
        if (e) cudaEventDestroy(e);
    if (b->stream) cudaStreamDestroy(b->stream);
    delete b;
}

int cw_batch_layout(const cw_batch *b, uint32_t *bt_log2, uint32_t *threads, uint64_t *bytes_per_instance) {
    if (!b) return fail(CW_EINVAL, "null argument");
    if (bt_log2) *bt_log2 = b->bt_log2;
    if (threads) *threads = b->threads;
    if (bytes_per_instance) *bytes_per_instance = (uint64_t)b->c->tape.n_slots * 32 + (uint64_t)b->c->tape.n_bitwords * 4;
    return CW_OK;
}

int cw_batch_set_input(cw_batch *b, uint32_t inst, uint64_t h, uint32_t idx, const uint64_t limbs[4]) {
    if (!b || inst >= b->batch) return fail(CW_EINVAL, "bad instance");
    const Tape &t = b->c->tape;
    if (b->remaining[inst] == 0) return fail(CW_ESTATE, "No more signals to be assigned");
    size_t p;
    int rc = hash_pos(t, h, &p);
    if (rc) return rc;
    if (idx >= t.hashmap[p].signalsize) return fail(CW_EINVAL, "Input signal array access exceeds the size");
    uint64_t si = t.hashmap[p].signalid + idx;
    uint64_t k = si - (t.n_outputs + 1);
    if (si < t.n_outputs + 1 || k >= t.n_inputs) return fail(CW_EINVAL, "input signal outside the main inputs");
    if (b->assigned[(size_t)inst * t.n_inputs + k]) return fail(CW_ESTATE, "Signal assigned twice: " + std::to_string(si));
    U256 v;
    memcpy(v.v, limbs, 32);
    if (!(v < t.F.q)) return fail(CW_EINVAL, "input value not reduced modulo the field prime");
    memcpy(&b->host_inputs[((size_t)inst * t.n_inputs + k) * 4], limbs, 32);
    b->assigned[(size_t)inst * t.n_inputs + k] = 1;
    b->remaining[inst]--;
    b->host_inputs_dirty = true;
    return CW_OK;
}

int cw_batch_remaining_inputs(const cw_batch *b, uint32_t inst, uint32_t *rem) {
    if (!b || inst >= b->batch) return fail(CW_EINVAL, "bad instance");
    *rem = b->remaining[inst];
    return CW_OK;
}

int cw_batch_set_inputs(cw_batch *b, const uint64_t *inputs, int is_device_ptr) {
    if (!b || !inputs) return fail(CW_EINVAL, "null argument");
    if (b->async_active) return fail(CW_ESTATE, "a witness transfer of this batch is in flight (cw_batch_get_witness_wait)");
    const Tape &t = b->c->tape;
    CU(cudaSetDevice(b->device));
    size_t bytes = (size_t)b->batch * t.n_inputs * 32;
    CU(cudaMemcpyAsync(b->inputs_d, inputs, bytes, is_device_ptr ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice,
                       b->stream));
    std::fill(b->remaining.begin(), b->remaining.end(), 0u);
    b->host_inputs_dirty = false;
    b->inputs_on_device = true;
    return CW_OK;
}

int cw_batch_run(cw_batch *b) {
    if (!b) return fail(CW_EINVAL, "null argument");
    if (b->async_active) return fail(CW_ESTATE, "a witness transfer of this batch is in flight (cw_batch_get_witness_wait)");
    const Tape &t = b->c->tape;
    CU(cudaSetDevice(b->device));
    if (b->host_inputs_dirty || !b->inputs_on_device) {
        for (u32 i = 0; i < b->batch; ++i)
            if (b->remaining[i])
                return fail(CW_ESTATE, "Not all inputs have been set. Only " +
                                           std::to_string(t.n_inputs - b->remaining[i]) + " out of " +
                                           std::to_string(t.n_inputs) + " (instance " + std::to_string(i) + ")");
        CU(cudaMemcpyAsync(b->inputs_d, b->host_inputs.data(), b->host_inputs.size() * 8, cudaMemcpyHostToDevice,
                           b->stream));
        b->host_inputs_dirty = false;
        b->inputs_on_device = true;
    }
    TapeDev tp;
    tp.ops = b->dt.ops;
    tp.items = b->dt.items;
    tp.heads = b->dt.heads;
    tp.level_start = b->dt.level_start;
    tp.level_info = b->dt.level_info;
    tp.has_slow = b->dt.has_slow ? 1u : 0u;
    tp.consts = b->dt.consts;
    tp.n_levels = (u32)t.n_levels();
    tp.n_slots = t.n_slots;
    tp.input_slot = b->dt.input_slot;
    tp.fn_code = b->dt.fn_code;
    tp.fn_info = b->dt.fn_info;
    tp.call_tab = b->dt.call_tab;
    tp.n_inputs = (u32)t.n_inputs;
    tp.n_bitwords = t.n_bitwords;
    tp.prime = (u32)t.F.prime_id;
    // the 128-bit register machine computes over the integers and gives up when a value leaves 128 bits: right only for a
    // prime above 2^128 (every 256-bit one); goldilocks calls run on the full-width machine
    tp.vm_wide = (env_int("CW_VM_WIDE", 0) || t.F.qbits <= 128) ? 1u : 0u;
    CU(cudaMemsetAsync(b->first_assert_d, 0xFF, (size_t)b->batch * 4, b->stream));
    CU(cudaMemsetAsync(b->err_d, 0, (size_t)b->batch * 4, b->stream));
    CU(cudaEventRecord(b->ev[0], b->stream));
    {
        size_t total = (size_t)b->batch_padded * (t.n_inputs + 1);
        u32 grid = (u32)std::min<size_t>((total + 255) / 256, 148 * 8);
        stage_inputs_kernel<<<grid, 256, 0, b->stream>>>(tp, b->inputs_d, b->slots, b->batch, b->batch_padded, b->bt_log2);
    }
    u32 tiles = b->batch_padded >> b->bt_log2;
    if (tp.n_levels) {
        const bool calls = !t.call_tab.empty();
        const bool bp = t.n_bitwords != 0;
        const u32 th = calls ? std::min<u32>(b->threads, 256u) : b->threads;  // the interpreter build has a large frame
        const bool fused = t.n_items() != t.n_tape_ops();
        if (t.F.prime_id == 0) launch_tape<0>(tp, b, tiles, th, calls, bp, fused);
        else if (t.F.prime_id == 1) launch_tape<1>(tp, b, tiles, th, calls, bp, fused);
        else {  // the other 256-bit primes: one build (bit-plane capable, runtime tile size), prime index from tp.prime
            if (fused) return fail(CW_ESTATE, "CW_FLAG_FUSE is available for bn128 and bls12381");
            if (calls) launch_tape_calls(-1, tp, b->slots, b->plane, b->bt_log2, b->first_assert_d, b->err_d, b->batch, tiles, th,
                                         true, false, b->stream);
            else launch_tape_k<-1, false, true, -1, false>(tp, b, tiles, th);
        }
    }
    CU(cudaEventRecord(b->ev[1], b->stream));
    b->dense_valid = false;
    CU(cudaEventRecord(b->ev[2], b->stream));
    CU(cudaGetLastError());
    b->ran = true;
    return CW_OK;
}

int cw_batch_sync(cw_batch *b) {
    if (!b) return fail(CW_EINVAL, "null argument");
    CU(cudaSetDevice(b->device));
    CU(cudaStreamSynchronize(b->stream));
    return CW_OK;
}

int cw_batch_status(cw_batch *b, int32_t *status) {
    if (!b || !status) return fail(CW_EINVAL, "null argument");
    if (!b->ran) return fail(CW_ESTATE, "batch has not been run");
    CU(cudaSetDevice(b->device));
    std::vector<u32> fa(b->batch);
    std::vector<int> er(b->batch);
    CU(cudaMemcpyAsync(fa.data(), b->first_assert_d, (size_t)b->batch * 4, cudaMemcpyDeviceToHost, b->stream));
    CU(cudaMemcpyAsync(er.data(), b->err_d, (size_t)b->batch * 4, cudaMemcpyDeviceToHost, b->stream));
    CU(cudaStreamSynchronize(b->stream));
    for (u32 i = 0; i < b->batch; ++i) {
        if (er[i]) status[i] = -1;  // division by zero: the reference process aborts inside GMP
        else status[i] = fa[i] == 0xFFFFFFFFu ? 0 : (int32_t)(fa[i] + 1);
    }
    return CW_OK;
}

// dense witness rows of instances [first, first + count) into `dst` (device, 32-byte aligned), on the batch stream
static int expand_rows(cw_batch *b, u32 first, u32 count, uint4 *dst) {
    const Tape &t = b->c->tape;
    if (count == 0) return CW_OK;
    dim3 grid((u32)std::min<size_t>((t.n_witness + 255) / 256, 148 * 4), std::min<u32>(count, 65535u));
    witness_expand_kernel<<<grid, 256, 0, b->stream>>>(b->store(), b->dt.wloc, (u32)t.n_witness, first, count, dst);
    CU(cudaGetLastError());
    return CW_OK;
}

// contiguous [batch][n_witness] copy in device memory, for callers that want the reference's layout on the device
static int dense_witness(cw_batch *b) {
    if (b->dense_valid) return CW_OK;
    const Tape &t = b->c->tape;
    if (!b->witness_d) {
        size_t bytes = (size_t)b->batch * t.n_witness * 32, free_b = 0, total_b = 0;
        cudaMemGetInfo(&free_b, &total_b);
        if (bytes + (64u << 20) > free_b)
            return fail(CW_ECUDA, "dense witness rows of the whole batch need " + std::to_string(bytes >> 20) +
                                      " MiB of device memory (" + std::to_string(free_b >> 20) +
                                      " MiB free): use cw_batch_expand_witness on a range of instances");
        CU(cudaMalloc((void **)&b->witness_d, bytes));
    }
    int rc = expand_rows(b, 0, b->batch, b->witness_d);
    if (rc) return rc;
    b->dense_valid = true;
    return CW_OK;
}

int cw_batch_expand_witness(cw_batch *b, uint32_t first, uint32_t count, uint64_t *dst_device) {
    if (!b || !dst_device || (uint64_t)first + count > b->batch) return fail(CW_EINVAL, "bad argument");
    if (!b->ran) return fail(CW_ESTATE, "batch has not been run");
    if ((uintptr_t)dst_device & 31u) return fail(CW_EINVAL, "destination must be 32-byte aligned");
    CU(cudaSetDevice(b->device));
    return expand_rows(b, first, count, (uint4 *)dst_device);
}

// NUMA node the GPU hangs off (/sys/bus/pci/devices/<bus id>/numa_node), -1 if unknown
static int device_numa_node(int device) {
    char id[32] = {0};
    if (cudaDeviceGetPCIBusId(id, sizeof(id), device) != cudaSuccess) return -1;
    for (char *p = id; *p; ++p) *p = (char)tolower(*p);
    std::string path = std::string("/sys/bus/pci/devices/") + id + "/numa_node";
    FILE *f = fopen(path.c_str(), "r");
    if (!f) return -1;
    int node = -1;
    if (fscanf(f, "%d", &node) != 1) node = -1;
    fclose(f);
    return node;
}

static size_t pack_chunk_instances(const cw_batch *b, const PackLayout &L) {
    size_t mb = (size_t)std::max(8, env_int("CW_PACK_CHUNK_MB", 96));
    size_t n = std::max<size_t>(1, (mb << 20) / (L.words * 4));
    return std::min<size_t>(n, b->batch);
}

static int ensure_pack_buffers(cw_batch *b, const PackLayout &L) {
    if (b->packed_cap) return CW_OK;
    size_t n = pack_chunk_instances(b, L);
    for (int k = 0; k < 2; ++k) {
        CU(cudaMalloc((void **)&b->packed_d[k], n * L.words * 4));
        CU(cudaMallocHost((void **)&b->packed_h[k], n * L.words * 4));
    }
    CU(cudaMalloc((void **)&b->pack_flag_d, 4));
    b->packed_cap = n;
    return CW_OK;
}

// packed records of instances [first, first + count) into `dst_d` (device), on the batch stream; np: the layout of observed
// classes (else the proven one, whose location lists are part of the device tape)
static int pack_rows(cw_batch *b, const PackLayout &L, u32 first, u32 count, u32 *dst_d, const NarrowPack *np = nullptr) {
    const size_t items = L.n_plane_words + L.n_bit_words + L.u64_loc.size() + L.full_loc.size();
    dim3 grid((u32)std::max<size_t>(1, std::min<size_t>((items + 255) / 256, 148 * 4)), std::min<u32>(count, 65535u));
    witness_pack_kernel<<<grid, 256, 0, b->stream>>>(b->store(), np ? np->pk_bit : b->dt.pk_bit, (u32)L.bit_loc.size(),
                                                     np ? np->pk_u64 : b->dt.pk_u64, (u32)L.u64_loc.size(),
                                                     np ? np->pk_full : b->dt.pk_full, (u32)L.full_loc.size(), dst_d, L.words,
                                                     first, count, b->pack_flag_d);
    CU(cudaGetLastError());
    return CW_OK;
}

// Looks at the values of a finished batch and (re)builds the circuit's layout of observed classes for the batch's device:
// class = max(what earlier batches showed, what this one shows), never wider than the proven class.
static int observe_classes(cw_batch *b, std::shared_ptr<NarrowPack> prev, std::shared_ptr<NarrowPack> &out) {
    const cw_circuit *c = b->c;
    const Tape &t = c->tape;
    const size_t W = t.n_witness;
    std::lock_guard<std::mutex> guard(c->narrow_mu);
    {   // another transfer may have observed meanwhile: start from the newest
        std::lock_guard<std::mutex> lk(c->mu);
        auto it = c->narrow.find(b->device);
        if (it != c->narrow.end() && it->second != prev) prev = it->second;
    }
    // the entries worth looking at: outside the bit plane, proven class above "bit"
    std::vector<u32> loc, wit;
    for (size_t i = 0; i < W; ++i)
        if (!(t.witness_slot[i] & OPERAND_BIT) && t.wit_class[i] > 0) {
            loc.push_back(t.witness_slot[i]);
            wit.push_back((u32)i);
        }
    auto np = std::make_shared<NarrowPack>();
    np->cls.assign(t.wit_class.begin(), t.wit_class.end());
    if (!loc.empty()) {
        std::vector<u32> cls(loc.size(), 0);
        if (prev)
            for (size_t k = 0; k < loc.size(); ++k) cls[k] = prev->cls[wit[k]];
        u32 *loc_d = nullptr, *cls_d = nullptr;
        int rc;
        if ((rc = upload(&loc_d, loc.data(), loc.size() * 4))) return rc;
        if ((rc = upload(&cls_d, cls.data(), cls.size() * 4))) { cudaFree(loc_d); return rc; }
        const u32 n_tiles = (b->batch + (1u << b->bt_log2) - 1) >> b->bt_log2;
        const uint64_t items = (uint64_t)loc.size() << b->bt_log2;
        dim3 grid((u32)std::max<uint64_t>(1, std::min<uint64_t>((items + 255) / 256, 148 * 8)), std::min<u32>(n_tiles, 65535u));
        witness_observe_kernel<<<grid, 256, 0, b->stream>>>(b->store(), loc_d, (u32)loc.size(), cls_d);
        cudaError_t e = cudaMemcpyAsync(cls.data(), cls_d, cls.size() * 4, cudaMemcpyDeviceToHost, b->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(b->stream);
        cudaFree(loc_d);
        cudaFree(cls_d);
        if (e != cudaSuccess) return fail(CW_ECUDA, cudaGetErrorString(e));
        for (size_t k = 0; k < loc.size(); ++k) np->cls[wit[k]] = (uint8_t)std::min<u32>(cls[k], t.wit_class[wit[k]]);
    }
    build_pack_layout(t, np->L, np->cls.data());
    int rc;
    if ((rc = upload(&np->pk_bit, np->L.bit_loc.data(), np->L.bit_loc.size() * 4))) return rc;
    if ((rc = upload(&np->pk_u64, np->L.u64_loc.data(), np->L.u64_loc.size() * 4))) return rc;
    if ((rc = upload(&np->pk_full, np->L.full_loc.data(), np->L.full_loc.size() * 4))) return rc;
    {
        std::lock_guard<std::mutex> lk(c->mu);
        c->narrow[b->device] = np;
    }
    out = np;
    return CW_OK;
}

// Packed transfer: entries the lowering proved to be one bit / <= 64 bits cross PCIe as that, the host expands
// them to the canonical 32-byte rows (zero-extension only - no field arithmetic happens on the CPU).  The batch
// moves in chunks through two staging buffers: while the worker threads expand chunk k, the pack kernel and the
// copy of chunk k + 1 run on the GPU / the copy engine.  CW_PACKED_D2H=0 forces the dense copy.
static int get_witness_packed_with(cw_batch *b, uint64_t *out, const PackLayout &L, const PackLayout &Lstatic,
                                   const NarrowPack *np, bool *flagged);
static int get_witness_packed(cw_batch *b, uint64_t *out, bool *done) {
    const Tape &t = b->c->tape;
    const PackLayout &Lstatic = b->c->pack_layout();
    *done = false;
    if (env_int("CW_PACKED_D2H", 1) == 0) return CW_OK;
    int rc;
    // Classes observed at run time (CW_PACK_OBSERVE=0: proven classes only).  Values that are bits or limbs without the
    // lowering being able to prove it - every xor of a hash circuit - then cross PCIe as bits / 8 bytes.  The first
    // transfer of a circuit looks at its batch; the pack kernel re-checks every value, a batch that shows a wider value
    // widens the layout and is sent again.
    std::shared_ptr<NarrowPack> np;
    if (env_int("CW_PACK_OBSERVE", 1) != 0 && (!Lstatic.u64_loc.empty() || !Lstatic.full_loc.empty())) {
        {
            std::lock_guard<std::mutex> lk(b->c->mu);
            auto it = b->c->narrow.find(b->device);
            if (it != b->c->narrow.end()) np = it->second;
        }
        if (!np && (rc = observe_classes(b, nullptr, np))) return rc;
    }
    for (int attempt = 0;; ++attempt) {
        const PackLayout &L = np ? np->L : Lstatic;
        if (L.words * 4 * 2 > (size_t)t.n_witness * 32) return CW_OK;   // not worth it: dense copy
        bool flagged = false;
        if ((rc = get_witness_packed_with(b, out, L, Lstatic, np.get(), &flagged))) return rc;
        if (!flagged) break;
        if (!np || attempt > 0) return CW_OK;   // a value exceeded its PROVEN class (never expected): dense copy
        std::shared_ptr<NarrowPack> wider;
        if ((rc = observe_classes(b, np, wider))) return rc;
        np = wider;
    }
    *done = true;
    return CW_OK;
}

// one pass of the packed transfer with layout L (staging buffers are sized for the proven layout, the widest)
static int get_witness_packed_with(cw_batch *b, uint64_t *out, const PackLayout &L, const PackLayout &Lstatic,
                                   const NarrowPack *np, bool *flagged) {
    const Tape &t = b->c->tape;
    int rc = ensure_pack_buffers(b, Lstatic);
    if (rc) return rc;
    CU(cudaMemsetAsync(b->pack_flag_d, 0, 4, b->stream));
    const size_t W = t.n_witness, cap = b->packed_cap;
    const size_t n_chunks = (b->batch + cap - 1) / cap;
    Pool &pool = Pool::get(device_numa_node(b->device));
    auto expand_chunk = [&](size_t k) {
        const size_t first = k * cap, cnt = std::min(cap, b->batch - first);
        const uint32_t *src = b->packed_h[k & 1];
        // item key = instance index: the rows of instance i of `out` are always written by the same (pinned) worker
        pool.parallel_for(cnt, first, [&](size_t i) { expand_record(L, src + i * L.words, out + (first + i) * W * 4); });
    };
    for (size_t k = 0; k < n_chunks; ++k) {
        const size_t first = k * cap, cnt = std::min(cap, b->batch - first);
        // staging buffer k & 1 was consumed by the expansion of chunk k - 2, which finished before chunk k - 1 was waited for
        if ((rc = pack_rows(b, L, (u32)first, (u32)cnt, b->packed_d[k & 1], np))) return rc;
        CU(cudaMemcpyAsync(b->packed_h[k & 1], b->packed_d[k & 1], cnt * L.words * 4, cudaMemcpyDeviceToHost, b->stream));
        CU(cudaEventRecord(b->pack_ev[k & 1], b->stream));
        if (k > 0) {
            CU(cudaEventSynchronize(b->pack_ev[(k - 1) & 1]));
            expand_chunk(k - 1);
        }
    }
    int flag = 0;
    CU(cudaMemcpyAsync(&flag, b->pack_flag_d, 4, cudaMemcpyDeviceToHost, b->stream));
    CU(cudaStreamSynchronize(b->stream));
    if (flag) {   // a value exceeded its class: the rows written so far are overwritten by the next attempt
        *flagged = true;
        return CW_OK;
    }
    expand_chunk(n_chunks - 1);
    b->last_d2h_bytes = (uint64_t)b->batch * L.words * 4;
    return CW_OK;
}

static int get_witness_impl(cw_batch *b, uint64_t *out) {
    const Tape &t = b->c->tape;
    CU(cudaSetDevice(b->device));
    bool done = false;
    int rc = get_witness_packed(b, out, &done);
    if (rc) return rc;
    if (done) return CW_OK;
    b->last_d2h_bytes = (uint64_t)b->batch * t.n_witness * 32;
    if (b->identity_layout()) {  // rows are read in place: pitched device-to-host copy
        CU(cudaMemcpy2DAsync(out, (size_t)t.n_witness * 32, b->slots, (size_t)t.n_slots * 32, (size_t)t.n_witness * 32,
                             b->batch, cudaMemcpyDeviceToHost, b->stream));
        CU(cudaStreamSynchronize(b->stream));
        return CW_OK;
    }
    // dense rows, a bounded number of instances at a time
    const size_t row = (size_t)t.n_witness * 32;
    if (!b->dense_chunk_d) {
        size_t n = std::max<size_t>(1, std::min<size_t>(b->batch, ((size_t)512 << 20) / row));
        CU(cudaMalloc((void **)&b->dense_chunk_d, n * row));
        b->dense_chunk_cap = n;
    }
    for (size_t first = 0; first < b->batch; first += b->dense_chunk_cap) {
        const size_t cnt = std::min(b->dense_chunk_cap, b->batch - first);
        if ((rc = expand_rows(b, (u32)first, (u32)cnt, b->dense_chunk_d))) return rc;
        CU(cudaMemcpyAsync((uint8_t *)out + first * row, b->dense_chunk_d, cnt * row, cudaMemcpyDeviceToHost, b->stream));
        CU(cudaStreamSynchronize(b->stream));
    }
    return CW_OK;
}

int cw_batch_get_witness(cw_batch *b, uint64_t *out) {
    if (!b || !out) return fail(CW_EINVAL, "null argument");
    if (!b->ran) return fail(CW_ESTATE, "batch has not been run");
    if (b->async_active) return fail(CW_ESTATE, "a witness transfer of this batch is in flight (cw_batch_get_witness_wait)");
    return get_witness_impl(b, out);
}

// The same transfer on a helper thread: the caller may run OTHER batches (their own streams) meanwhile, so that the
// tape of batch k + 1 executes while the witnesses of batch k are packed, copied and expanded.
int cw_batch_get_witness_async(cw_batch *b, uint64_t *out) {
    if (!b || !out) return fail(CW_EINVAL, "null argument");
    if (!b->ran) return fail(CW_ESTATE, "batch has not been run");
    if (b->async_active) return fail(CW_ESTATE, "a witness transfer of this batch is already in flight");
    join_async(b);
    b->async_active = true;
    b->async_th = std::thread([b, out] {
        b->async_rc = get_witness_impl(b, out);
        b->async_err = g_err;  // (thread-local message of the helper thread)
    });
    return CW_OK;
}

int cw_batch_get_witness_wait(cw_batch *b) {
    if (!b) return fail(CW_EINVAL, "null argument");
    if (!b->async_active) return CW_OK;
    join_async(b);
    if (b->async_rc) return fail(b->async_rc, b->async_err);
    return CW_OK;
}

uint64_t cw_batch_last_d2h_bytes(const cw_batch *b) { return b ? b->last_d2h_bytes : 0; }

// The packed records themselves, for consumers that do not need 32-byte rows (layout: cw_circuit_pack_info)
int cw_batch_get_witness_packed(cw_batch *b, uint32_t *out_words) {
    if (!b || !out_words) return fail(CW_EINVAL, "null argument");
    if (!b->ran) return fail(CW_ESTATE, "batch has not been run");
    if (b->async_active) return fail(CW_ESTATE, "a witness transfer of this batch is in flight (cw_batch_get_witness_wait)");
    CU(cudaSetDevice(b->device));
    const PackLayout &L = b->c->pack_layout();
    int rc = ensure_pack_buffers(b, L);
    if (rc) return rc;
    CU(cudaMemsetAsync(b->pack_flag_d, 0, 4, b->stream));
    for (size_t first = 0; first < b->batch; first += b->packed_cap) {
        const size_t cnt = std::min(b->packed_cap, b->batch - first);
        if ((rc = pack_rows(b, L, (u32)first, (u32)cnt, b->packed_d[0]))) return rc;
        CU(cudaMemcpyAsync(out_words + first * L.words, b->packed_d[0], cnt * L.words * 4, cudaMemcpyDeviceToHost, b->stream));
        CU(cudaStreamSynchronize(b->stream));
    }
    int flag = 0;
    CU(cudaMemcpy(&flag, b->pack_flag_d, 4, cudaMemcpyDeviceToHost));
    if (flag) return fail(CW_ESTATE, "a witness value exceeds the width the lowering proved for it");
    return CW_OK;
}

int cw_batch_witness_device(cw_batch *b, const uint64_t **dptr) {
    if (!b || !dptr) return fail(CW_EINVAL, "null argument");
    if (!b->ran) return fail(CW_ESTATE, "batch has not been run");
    CU(cudaSetDevice(b->device));
    int rc = dense_witness(b);
    if (rc) return rc;
    *dptr = (const uint64_t *)b->witness_d;
    return CW_OK;
}

int cw_batch_witness_strided(cw_batch *b, const uint64_t **dptr, uint64_t *stride_elems) {
    if (!b || !dptr || !stride_elems) return fail(CW_EINVAL, "null argument");
    if (!b->ran) return fail(CW_ESTATE, "batch has not been run");
    if (b->identity_layout()) {
        *dptr = (const uint64_t *)b->slots;
        *stride_elems = b->c->tape.n_slots;
        return CW_OK;
    }
    int rc = cw_batch_witness_device(b, dptr);
    *stride_elems = b->c->tape.n_witness;
    return rc;
}

void *cw_batch_stream(cw_batch *b) { return b ? (void *)b->stream : nullptr; }

int cw_batch_last_ms(cw_batch *b, float *exec_ms, float *gather_ms) {
    if (!b || !b->ran) return fail(CW_ESTATE, "batch has not been run");
    CU(cudaSetDevice(b->device));
    CU(cudaEventSynchronize(b->ev[2]));
    if (exec_ms) CU(cudaEventElapsedTime(exec_ms, b->ev[0], b->ev[1]));
    if (gather_ms) *gather_ms = 0.f;  // no gather pass: witness entries are written in place by the tape
    return CW_OK;
}

int cw_batch_wtns_bytes(cw_batch *b, uint32_t inst, uint8_t *out, size_t cap, size_t *len) {
    if (!b || inst >= b->batch) return fail(CW_EINVAL, "bad instance");
    if (!b->ran) return fail(CW_ESTATE, "batch has not been run");
    const Tape &t = b->c->tape;
    const size_t n8 = field_bytes(t.F);
    size_t need = 44 + n8 + n8 * (size_t)t.n_witness;
    if (len) *len = need;
    if (!out) return CW_OK;
    if (cap < need) return fail(CW_EINVAL, "buffer too small");
    CU(cudaSetDevice(b->device));
    std::vector<uint64_t> w((size_t)t.n_witness * 4);
    uint4 *row = nullptr;
    CU(cudaMalloc((void **)&row, (size_t)t.n_witness * 32));
    int rc = expand_rows(b, inst, 1, row);
    if (!rc) {
        cudaError_t e = cudaMemcpyAsync(w.data(), row, (size_t)t.n_witness * 32, cudaMemcpyDeviceToHost, b->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(b->stream);
        if (e != cudaSuccess) rc = fail(CW_ECUDA, cudaGetErrorString(e));
    }
    cudaFree(row);
    if (rc) return rc;
    std::vector<uint8_t> bytes = wtns_bytes(t.F, w.data(), t.n_witness);
    memcpy(out, bytes.data(), need);
    return CW_OK;
}

int cw_batch_write_wtns(cw_batch *b, uint32_t inst, const char *path) {
    size_t need = 0;
    int rc = cw_batch_wtns_bytes(b, inst, nullptr, 0, &need);
    if (rc) return rc;
    std::vector<uint8_t> buf(need);
    if ((rc = cw_batch_wtns_bytes(b, inst, buf.data(), need, &need))) return rc;
    FILE *f = fopen(path, "wb");
    if (!f) return fail(CW_EIO, std::string("cannot open ") + path);
    size_t wr = fwrite(buf.data(), 1, need, f);
    fclose(f);
    return wr == need ? CW_OK : fail(CW_EIO, "short write");
}

// packed-record layout of the circuit: per witness entry (class << 30) | index - class 0: bit `index` of the plane
// section, 1: bit `index` of the extra-bit section, 2: u64 entry `index`, 3: full entry `index`; sections follow each
// other in that order; info = {words per instance, plane words, extra-bit words, u64 entries, full entries}
int cw_circuit_pack_info(const cw_circuit *c, uint64_t info[5], uint32_t *entry) {
    if (!c) return fail(CW_EINVAL, "null argument");
    const PackLayout &L = c->pack_layout();
    if (info) {
        info[0] = L.words;
        info[1] = L.n_plane_words;
        info[2] = L.n_bit_words;
        info[3] = L.u64_loc.size();
        info[4] = L.full_loc.size();
    }
    if (entry)
        for (const PackSeg &sg : L.segs)
            for (uint32_t j = 0; j < sg.count; ++j) entry[sg.start + j] = (sg.kind << 30) | (sg.src + j);
    return CW_OK;
}

// one packed record -> the n_witness canonical 32-byte rows of that instance (host memory; what cw_batch_get_witness
// does for every instance); `store_bits` 0 = widest vector stores of the CPU, or at most 128 / 256 / 512
int cw_circuit_expand_record(const cw_circuit *c, const uint32_t *record, uint64_t *rows, int store_bits) {
    if (!c || !record || !rows) return fail(CW_EINVAL, "null argument");
    expand_record(c->pack_layout(), record, rows, store_bits);
    return CW_OK;
}
const char *cw_host_expand_isa(void) { return expand_isa(); }
const char *cw_host_pool_info(void) { return Pool::get().describe(); }

// Host-side probe (no GPU): the expansion of `n_inst` packed records (all zero) into a freshly allocated row buffer on
// the worker pool, `reps` passes over the same buffer; mode 0 = expand_record, 1 = plain streaming fill of the same
// bytes (the memory system's ceiling for this access pattern), 2 = memset.  gbps[r] = bytes of rows written / time.
int cw_host_expand_bench(const cw_circuit *c, uint32_t n_inst, uint32_t reps, int mode, double *gbps) {
    if (!c || !gbps || !n_inst || !reps) return fail(CW_EINVAL, "bad argument");
    const PackLayout &L = c->pack_layout();
    const size_t W = c->tape.n_witness, row_bytes = W * 32;
    uint64_t *out = (uint64_t *)aligned_alloc(64, ((size_t)n_inst * row_bytes + 63) & ~(size_t)63);
    if (!out) return fail(CW_EINVAL, "out of host memory");
    std::vector<uint32_t> rec(L.words, 0);
    Pool &pool = Pool::get();
    for (uint32_t r = 0; r < reps; ++r) {
        auto t0 = std::chrono::steady_clock::now();
        pool.parallel_for(n_inst, 0, [&](size_t i) {
            uint64_t *dst = out + i * W * 4;
            if (mode == 0) expand_record(L, rec.data(), dst);
            else if (mode == 1) {
                const __m128i z = _mm_setzero_si128();
                for (size_t k = 0; k < W * 2; ++k) _mm_stream_si128((__m128i *)dst + k, z);
                _mm_sfence();
            } else memset(dst, 0, row_bytes);
        });
        double dt = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
        gbps[r] = (double)n_inst * row_bytes / dt / 1e9;
    }
    free(out);
    return CW_OK;
}

// ---- R1CS -------------------------------------------------------------------------------------
int cw_r1cs_from_circuit(const cw_circuit *c, cw_r1cs **out) {
    if (!c || !out) return fail(CW_EINVAL, "null argument");
    cw_r1cs *r = new cw_r1cs();
    r->data = c->tape.r1cs;
    r->F = c->tape.F;
    *out = r;
    return CW_OK;
}
int cw_r1cs_load(const char *path, cw_r1cs **out) {
    if (!path || !out) return fail(CW_EINVAL, "null argument");
    cw_r1cs *r = new cw_r1cs();
    try {
        read_r1cs(path, r->data);
    } catch (const std::exception &e) {
        delete r;
        return fail(CW_EFORMAT, e.what());
    }
    r->F = make_field(r->data.prime_id);
    *out = r;
    return CW_OK;
}
int cw_r1cs_write(const cw_r1cs *r, const char *path, uint32_t n_pub_out, uint32_t n_pub_in, uint32_t n_prv_in) {
    if (!r || !path) return fail(CW_EINVAL, "null argument");
    try {
        R1csData d = r->data;  // CW_KEEP: the count the circuit / the loaded file carries
        if (n_pub_out != CW_KEEP) d.n_pub_out = n_pub_out;
        if (n_pub_in != CW_KEEP) d.n_pub_in = n_pub_in;
        if (n_prv_in != CW_KEEP) d.n_prv_in = n_prv_in;
        write_r1cs(d, r->F, path);
    } catch (const std::exception &e) {
        return fail(CW_EIO, e.what());
    }
    return CW_OK;
}
int cw_r1cs_info(const cw_r1cs *r, uint64_t *n_wires, uint64_t *n_constraints, uint64_t *nnz, int *prime_id) {
    if (!r) return fail(CW_EINVAL, "null argument");
    if (n_wires) *n_wires = r->data.n_wires;
    if (n_constraints) *n_constraints = r->data.n_constraints;
    if (nnz) *nnz = r->data.col.size();
    if (prime_id) *prime_id = r->data.prime_id;
    return CW_OK;
}
void cw_r1cs_destroy(cw_r1cs *r) {
    if (!r) return;
    if (r->eval_twin) cw_r1cs_destroy(r->eval_twin);
    for (auto &kv : r->dev) {
        cudaSetDevice(kv.first.device);
        cudaFree(kv.second.row_ptr);
        cudaFree(kv.second.terms);
        cudaFree(kv.second.dictM);
        cudaFree(kv.second.perm);
        cudaFree(kv.second.perm_small);
        cudaFree(kv.second.sgroups);
        cudaFree(kv.second.srecs);
        cudaFree(kv.second.sbrow);
        cudaFree(kv.second.bool_loc);
        cudaFree(kv.second.bool_row);
    }
    delete r;
}

// The CSR compiled for one value layout (r1cs_compile.cpp), uploaded.
static int compile_r1cs(cw_r1cs *r, int device, const cw_circuit *layout, DevR1cs &d) {
    R1csCompiled h;
    try {
        compile_r1cs_host(r->data, r->F, layout ? &layout->tape : nullptr, r->no_bool_rows,
                          !r->no_bool_rows && env_int("CW_R1CS_SMALL", 1) != 0, h);
    } catch (const std::exception &e) {
        return fail(CW_EINVAL, e.what());
    }
    int rc;
    static_assert(sizeof(R1csTerm) == sizeof(uint4), "term records are read as uint4");
    d.n_general = (u32)h.perm.size();
    d.n_small = (u32)h.perm_small.size();
    d.n_bool = (u32)h.bool_loc.size();
    d.n_terms = h.n_terms;
    d.mean_row_terms = h.mean_row_terms;
    if ((rc = upload(&d.terms, h.terms.data(), h.terms.size() * sizeof(uint4)))) return rc;
    if ((rc = upload(&d.bool_loc, h.bool_loc.data(), h.bool_loc.size() * 4))) return rc;
    if ((rc = upload(&d.bool_row, h.bool_row.data(), h.bool_row.size() * 4))) return rc;
    if ((rc = upload(&d.row_ptr, h.row_ptr.data(), h.row_ptr.size() * 8))) return rc;
    if ((rc = upload(&d.dictM, h.dictM.data(), h.dictM.size() * 32))) return rc;
    if ((rc = upload(&d.perm, h.perm.data(), h.perm.size() * 4))) return rc;
    if ((rc = upload(&d.perm_small, h.perm_small.data(), h.perm_small.size() * 4))) return rc;
    static_assert(sizeof(R1csSmallRec) == sizeof(uint2), "integer-row records are read as uint2");
    if ((rc = upload(&d.sgroups, h.sgroups.data(), h.sgroups.size() * 4))) return rc;
    if ((rc = upload(&d.srecs, h.srecs.data(), h.srecs.size() * sizeof(uint2)))) return rc;
    if ((rc = upload(&d.sbrow, h.sbrow.data(), h.sbrow.size() * 4))) return rc;
    (void)device;
    return CW_OK;
}

static int get_dev_r1cs(cw_r1cs *r, int device, const cw_circuit *layout, DevR1cs &d) {
    std::lock_guard<std::mutex> lk(r->mu);
    R1csKey key{device, layout};
    auto it = r->dev.find(key);
    if (it != r->dev.end()) {
        d = it->second;
        return CW_OK;
    }
    int rc = compile_r1cs(r, device, layout, d);
    if (rc) return rc;
    r->dev[key] = d;
    return CW_OK;
}

struct R1csOut {
    uint4 *a = nullptr, *b = nullptr, *c = nullptr;
};

// launches on `stream`; fb_d[batch] must hold ~0 on entry; `wide` = (n_small + 31) / 32 + 1 words of scratch for the rows the
// integer-row kernel hands to the general one
static int launch_r1cs(cw_r1cs *r, const DevR1cs &d, const StoreDev &S, cudaStream_t stream, unsigned long long *fb_d,
                       const R1csOut *eval, u32 *wide) {
    const R1csData &R = r->data;
    R1csDev rd;
    rd.row_ptr = d.row_ptr;
    rd.terms = d.terms;
    rd.dictM = d.dictM;
    rd.perm = d.perm;
    rd.n_rows = d.n_general;
    rd.prime = (u32)R.prime_id;
    const u32 n_tiles = (S.batch + (1u << S.bt_log2) - 1) >> S.bt_log2;
    if (d.n_general) {
        const uint64_t items = (uint64_t)d.n_general << S.bt_log2;
        dim3 grid((u32)std::max<uint64_t>(1, std::min<uint64_t>((items + 255) / 256, 148 * 8)), std::min<u32>(n_tiles, 65535u));
        // long rows: many resident warps (48 registers); short rows: the unspilled build
        const bool lean = env_int("CW_R1CS_LEAN", d.mean_row_terms >= 12 ? 1 : 0) != 0;
        EvalOut eo;
        if (eval) { eo.a = eval->a; eo.b = eval->b; eo.c = eval->c; eo.m = R.n_constraints; }
#define CW_LAUNCH_R1CS(PR)                                                                              \
    do {                                                                                                \
        if (eval) r1cs_check_kernel<PR, 3, true, false><<<grid, 256, 0, stream>>>(rd, S, fb_d, eo, nullptr);       \
        else if (lean) r1cs_check_kernel<PR, 5, false, false><<<grid, 256, 0, stream>>>(rd, S, fb_d, eo, nullptr); \
        else r1cs_check_kernel<PR, 3, false, false><<<grid, 256, 0, stream>>>(rd, S, fb_d, eo, nullptr);           \
    } while (0)
        if (R.prime_id == 0) CW_LAUNCH_R1CS(0);
        else if (R.prime_id == 1) CW_LAUNCH_R1CS(1);
        else if (eval) r1cs_check_kernel<-1, 3, true, false><<<grid, 256, 0, stream>>>(rd, S, fb_d, eo, nullptr);
        else r1cs_check_kernel<-1, 3, false, false><<<grid, 256, 0, stream>>>(rd, S, fb_d, eo, nullptr);
#undef CW_LAUNCH_R1CS
    }
    if (d.n_small) {
        // rows that are small by shape: over the integers first; the rows in which a value turned out wide (bitmap) go
        // through the general kernel afterwards
        if (!wide || eval) return fail(CW_ESTATE, "integer rows need their scratch bitmap");
        CU(cudaMemsetAsync(wide, 0, (((size_t)d.n_small + 31) / 32 + 1) * 4, stream));
        rd.perm = d.perm_small;
        rd.n_rows = d.n_small;
        const uint64_t items = (uint64_t)d.n_small << S.bt_log2;
        dim3 grid((u32)std::max<uint64_t>(1, std::min<uint64_t>((items + 255) / 256, 148 * 8)), std::min<u32>(n_tiles, 65535u));
        R1csSmallDev sg;
        sg.groups = d.sgroups;
        sg.recs = d.srecs;
        sg.brow = d.sbrow;
        if (S.bt_log2 == 0) r1cs_small_kernel<true><<<grid, 256, 0, stream>>>(rd, sg, S, fb_d, wide);
        else r1cs_small_kernel<false><<<grid, 256, 0, stream>>>(rd, sg, S, fb_d, wide);
        EvalOut eo;
        if (R.prime_id == 0) r1cs_check_kernel<0, 3, false, true><<<grid, 256, 0, stream>>>(rd, S, fb_d, eo, wide);
        else if (R.prime_id == 1) r1cs_check_kernel<1, 3, false, true><<<grid, 256, 0, stream>>>(rd, S, fb_d, eo, wide);
        else r1cs_check_kernel<-1, 3, false, true><<<grid, 256, 0, stream>>>(rd, S, fb_d, eo, wide);
    }
    if (d.n_bool && !eval) {
        const uint64_t items = (uint64_t)d.n_bool << S.bt_log2;
        dim3 bgrid((u32)std::max<uint64_t>(1, std::min<uint64_t>((items + 255) / 256, 148 * 8)), std::min<u32>(n_tiles, 65535u));
        r1cs_bool_kernel<<<bgrid, 256, 0, stream>>>(d.bool_loc, d.bool_row, d.n_bool, S, fb_d);
    }
    CU(cudaGetLastError());
    return CW_OK;
}

int cw_r1cs_check(cw_r1cs *r, const uint64_t *witness, int is_device_ptr, uint32_t batch, int device,
                  int64_t *first_bad, float *kernel_ms) {
    if (!r) return fail(CW_EINVAL, "bad argument");
    return cw_r1cs_check_strided(r, witness, r->data.n_wires, is_device_ptr, batch, device, first_bad, kernel_ms);
}

// dense witness rows handed in by the caller (host or device memory)
int cw_r1cs_check_strided(cw_r1cs *r, const uint64_t *witness, uint64_t stride_elems, int is_device_ptr, uint32_t batch,
                          int device, int64_t *first_bad, float *kernel_ms) {
    if (!r || !witness || !first_bad || batch == 0 || stride_elems < r->data.n_wires || stride_elems >> 32)
        return fail(CW_EINVAL, "bad argument");
    if (is_device_ptr && ((uintptr_t)witness & 31u))
        return fail(CW_EINVAL, "device witness pointer must be 32-byte aligned (elements are read with 256-bit loads)");
    int rc = ensure_device(device);
    if (rc) return rc;
    DevR1cs d;
    if ((rc = get_dev_r1cs(r, device, nullptr, d))) return rc;
    const R1csData &R = r->data;
    const uint4 *w_d = (const uint4 *)witness;
    uint4 *tmp = nullptr;
    if (!is_device_ptr) {
        CU(cudaMalloc((void **)&tmp, (size_t)batch * R.n_wires * 32));
        CU(cudaMemcpy2D(tmp, (size_t)R.n_wires * 32, witness, (size_t)stride_elems * 32, (size_t)R.n_wires * 32, batch,
                        cudaMemcpyHostToDevice));
        w_d = tmp;
        stride_elems = R.n_wires;
    }
    unsigned long long *fb_d = nullptr;
    CU(cudaMalloc((void **)&fb_d, (size_t)batch * 8));
    CU(cudaMemset(fb_d, 0xFF, (size_t)batch * 8));
    StoreDev S;
    S.slots = w_d;
    S.plane = nullptr;
    S.n_slots = (u32)stride_elems;
    S.n_bitwords = 0;
    S.bt_log2 = 0;
    S.batch = batch;
    u32 *wide_d = nullptr;
    if (d.n_small) CU(cudaMalloc((void **)&wide_d, (((size_t)d.n_small + 31) / 32 + 1) * 4));
    cudaEvent_t e0, e1;
    CU(cudaEventCreate(&e0));
    CU(cudaEventCreate(&e1));
    CU(cudaEventRecord(e0));
    rc = launch_r1cs(r, d, S, nullptr, fb_d, nullptr, wide_d);
    CU(cudaEventRecord(e1));
    if (!rc) {
        std::vector<unsigned long long> fb(batch);
        CU(cudaMemcpy(fb.data(), fb_d, (size_t)batch * 8, cudaMemcpyDeviceToHost));
        float ms = 0;
        CU(cudaEventElapsedTime(&ms, e0, e1));
        if (kernel_ms) *kernel_ms = ms;
        for (u32 i = 0; i < batch; ++i) first_bad[i] = fb[i] == ~0ull ? -1 : (int64_t)fb[i];
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(fb_d);
    if (wide_d) cudaFree(wide_d);
    if (tmp) cudaFree(tmp);
    return rc;
}

// The witnesses of a batch where the tape left them (resident slots + bit plane, any tile layout): no dense rows
// are materialised, plane bits are read as bits, recomposition sums as words.  Runs on the batch's stream, behind
// the tape; the per-instance result buffer belongs to the batch (no allocation per call).
int cw_r1cs_check_batch(cw_r1cs *r, cw_batch *b, int64_t *first_bad, float *kernel_ms) {
    if (!r || !b || !first_bad) return fail(CW_EINVAL, "null argument");
    if (!b->ran) return fail(CW_ESTATE, "batch has not been run");
    if (r->data.prime_id != b->c->tape.F.prime_id) return fail(CW_EINVAL, "the R1CS and the batch use different primes");
    CU(cudaSetDevice(b->device));
    DevR1cs d;
    int rc = get_dev_r1cs(r, b->device, b->c, d);
    if (rc) return rc;
    cudaEvent_t e0, e1;
    CU(cudaEventCreate(&e0));
    CU(cudaEventCreate(&e1));
    CU(cudaMemsetAsync(b->fb_d, 0xFF, (size_t)b->batch * 8, b->stream));
    if (d.n_small > b->r1cs_wide_rows) {   // scratch of the integer rows: grows with the largest R1CS this batch has checked
        CU(cudaStreamSynchronize(b->stream));
        cudaFree(b->r1cs_wide_d);
        b->r1cs_wide_d = nullptr;
        b->r1cs_wide_rows = 0;
        CU(cudaMalloc((void **)&b->r1cs_wide_d, (((size_t)d.n_small + 31) / 32 + 1) * 4));
        b->r1cs_wide_rows = d.n_small;
    }
    CU(cudaEventRecord(e0, b->stream));
    rc = launch_r1cs(r, d, b->store(), b->stream, b->fb_d, nullptr, b->r1cs_wide_d);
    CU(cudaEventRecord(e1, b->stream));
    if (!rc) {
        std::vector<unsigned long long> fb(b->batch);
        CU(cudaMemcpyAsync(fb.data(), b->fb_d, (size_t)b->batch * 8, cudaMemcpyDeviceToHost, b->stream));
        CU(cudaStreamSynchronize(b->stream));
        float ms = 0;
        CU(cudaEventElapsedTime(&ms, e0, e1));
        if (kernel_ms) *kernel_ms = ms;
        for (u32 i = 0; i < b->batch; ++i) first_bad[i] = fb[i] == ~0ull ? -1 : (int64_t)fb[i];
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    return rc;
}

static int copy_text(const std::string &msg, char *buf, size_t cap, size_t *len) {
    if (len) *len = msg.size();
    if (buf && cap) {
        const size_t n = std::min(msg.size(), cap - 1);
        memcpy(buf, msg.data(), n);
        buf[n] = 0;
    }
    return CW_OK;
}

int cw_circuit_format_log(const cw_circuit *c, const uint64_t *witness, char *buf, size_t cap, size_t *len) {
    if (!c || !witness) return fail(CW_EINVAL, "null argument");
    return copy_text(format_log(c->tape, witness), buf, cap, len);
}

int cw_batch_log(cw_batch *b, uint32_t inst, char *buf, size_t cap, size_t *len) {
    if (!b || inst >= b->batch) return fail(CW_EINVAL, "bad instance");
    if (!b->ran) return fail(CW_ESTATE, "batch has not been run");
    const Tape &t = b->c->tape;
    if (t.log_args.empty()) return copy_text(std::string(), buf, cap, len);
    CU(cudaSetDevice(b->device));
    std::vector<uint64_t> w((size_t)t.n_witness * 4);
    uint4 *row = nullptr;
    CU(cudaMalloc((void **)&row, (size_t)t.n_witness * 32));
    int rc = expand_rows(b, inst, 1, row);       // (the dense row of one instance, as the .wtns writer fetches it)
    if (!rc) {
        cudaError_t e = cudaMemcpyAsync(w.data(), row, (size_t)t.n_witness * 32, cudaMemcpyDeviceToHost, b->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(b->stream);
        if (e != cudaSuccess) rc = fail(CW_ECUDA, cudaGetErrorString(e));
    }
    cudaFree(row);
    if (rc) return rc;
    return copy_text(format_log(t, w.data()), buf, cap, len);
}

int cw_circuit_assert_info(const cw_circuit *c, uint32_t assert_no, char *buf, size_t cap, size_t *len) {
    if (!c) return fail(CW_EINVAL, "null argument");
    const Tape &t = c->tape;
    if (assert_no >= t.assert_tid.size()) return fail(CW_EINVAL, "no such assert (or a circuit without its description: broadcast)");
    std::string msg = "Failed assert in template/function " + t.tmpl_names[t.assert_tid[assert_no]];
    if (!t.sym.empty()) {
        // the component whose signals start at assert_start: walk down from main by signal ranges (own signals first, then
        // the sub-components in creation order - the numbering of the whole description)
        std::string trace = "main";
        uint32_t tid = t.sym_main;
        uint64_t start = 1;   // (signal 0 is the constant one)
        const uint64_t want = t.assert_start[assert_no];
        while (start != want) {
            const Tape::SymTemplate &st = t.sym[tid];
            uint64_t off = start + st.n_own;
            bool down = false;
            for (size_t i = 0; i < st.subs.size(); ++i) {
                const uint64_t n = t.sym[st.subs[i]].total_signals;
                if (want >= off && want < off + n) {
                    trace += "." + st.sub[i];
                    tid = st.subs[i];
                    start = off;
                    down = true;
                    break;
                }
                off += n;
            }
            if (!down) return fail(CW_EINVAL, "assert site outside the component tree");
        }
        msg += ". Followed trace of components: " + trace;
    }
    if (len) *len = msg.size();
    if (buf && cap) {
        const size_t n = std::min(msg.size(), cap - 1);
        memcpy(buf, msg.data(), n);
        buf[n] = 0;
    }
    return CW_OK;
}

int cw_r1cs_compiled_info(cw_r1cs *r, cw_batch *b, int device, uint64_t info[4]) {
    if (!r || !info) return fail(CW_EINVAL, "null argument");
    int rc = b ? CW_OK : ensure_device(device);
    if (rc) return rc;
    if (b) CU(cudaSetDevice(b->device));
    DevR1cs d;
    if ((rc = get_dev_r1cs(r, b ? b->device : device, b ? b->c : nullptr, d))) return rc;
    info[0] = d.n_general;
    info[1] = d.n_small;
    info[2] = d.n_bool;
    info[3] = d.n_terms;
    return CW_OK;
}

// A.w, B.w, C.w of every constraint for instances [first, first + count) of a batch, left in device memory for a
// prover (the QAP evaluation / rapidsnark-style pipeline that follows witness generation): three arrays
// [count][n_constraints][4 x u64], canonical.  Rows the check treats specially (boolean rows) are evaluated like
// all others here.
int cw_r1cs_eval_batch(cw_r1cs *r, cw_batch *b, uint32_t first, uint32_t count, uint64_t *a_dev, uint64_t *b_dev,
                       uint64_t *c_dev) {
    if (!r || !b || !a_dev || !b_dev || !c_dev || (uint64_t)first + count > b->batch || count == 0)
        return fail(CW_EINVAL, "bad argument");
    if (((uintptr_t)a_dev | (uintptr_t)b_dev | (uintptr_t)c_dev) & 31u) return fail(CW_EINVAL, "outputs must be 32-byte aligned");
    if (!b->ran) return fail(CW_ESTATE, "batch has not been run");
    if (b->bt_log2 != 0) return fail(CW_ESTATE, "cw_r1cs_eval_batch needs a one-instance tile layout (CW_BT_LOG2=0)");
    CU(cudaSetDevice(b->device));
    // all rows through the general path: a layout key of its own (no boolean-row special cases)
    cw_r1cs *all = nullptr;
    {
        std::lock_guard<std::mutex> lk(r->mu);
        if (!r->eval_twin) {
            r->eval_twin = new cw_r1cs();
            r->eval_twin->data = r->data;
            r->eval_twin->F = r->F;
            r->eval_twin->no_bool_rows = true;
        }
        all = r->eval_twin;
    }
    DevR1cs d;
    int rc = get_dev_r1cs(all, b->device, b->c, d);
    if (rc) return rc;
    StoreDev S = b->store();
    S.slots += (size_t)first * S.n_slots * 2;
    S.plane += (size_t)first * S.n_bitwords;
    S.batch = count;
    R1csOut eo;
    eo.a = (uint4 *)a_dev;
    eo.b = (uint4 *)b_dev;
    eo.c = (uint4 *)c_dev;
    CU(cudaMemsetAsync(b->fb_d, 0xFF, (size_t)b->batch * 8, b->stream));
    return launch_r1cs(all, d, S, b->stream, b->fb_d, &eo, nullptr);
}

// readWitness side of the file boundary: the 32-byte entries of a .wtns (written by this library, the reference
// calculator or snarkjs); out = NULL returns the count only
int cw_wtns_read(const char *path, int *prime_id, uint64_t *n_witness, uint64_t *out, size_t cap_entries) {
    if (!path || !n_witness) return fail(CW_EINVAL, "null argument");
    std::vector<uint64_t> w;
    int pid = 0;
    try {
        read_wtns(path, pid, w);
    } catch (const std::exception &e) {
        return fail(CW_EFORMAT, e.what());
    }
    if (prime_id) *prime_id = pid;
    *n_witness = w.size() / 4;
    if (!out) return CW_OK;
    if (cap_entries < w.size() / 4) return fail(CW_EINVAL, "buffer too small");
    memcpy(out, w.data(), w.size() * 8);
    return CW_OK;
}

// A.w o B.w == C.w for a .wtns file against a .r1cs file (what `snarkjs wtns check` does): first_bad = -1 if every
// constraint holds, else the smallest violated row
int cw_r1cs_check_files(const char *r1cs_path, const char *wtns_path, int device, int64_t *first_bad) {
    if (!r1cs_path || !wtns_path || !first_bad) return fail(CW_EINVAL, "null argument");
    cw_r1cs *r = nullptr;
    int rc = cw_r1cs_load(r1cs_path, &r);
    if (rc) return rc;
    std::vector<uint64_t> w;
    int pid = 0;
    try {
        read_wtns(wtns_path, pid, w);
    } catch (const std::exception &e) {
        cw_r1cs_destroy(r);
        return fail(CW_EFORMAT, e.what());
    }
    if (pid != r->data.prime_id || w.size() / 4 != r->data.n_wires) {
        cw_r1cs_destroy(r);
        return fail(CW_EINVAL, "the witness and the constraint system do not match (prime or number of wires)");
    }
    rc = cw_r1cs_check(r, w.data(), 0, 1, device, first_bad, nullptr);
    cw_r1cs_destroy(r);
    return rc;
}

// ---- lowered circuit as a blob / multi-GPU plumbing -----------------------------------------------------------
int cw_circuit_serialize(const cw_circuit *c, uint8_t *out, size_t cap, size_t *len) {
    if (!c || !len) return fail(CW_EINVAL, "null argument");
    std::vector<uint8_t> blob;
    serialize_tape(c->tape, blob);
    *len = blob.size();
    if (!out) return CW_OK;
    if (cap < blob.size()) return fail(CW_EINVAL, "buffer too small");
    memcpy(out, blob.data(), blob.size());
    return CW_OK;
}

int cw_circuit_deserialize(const void *data, size_t len, cw_circuit **out) {
    if (!data || !out) return fail(CW_EINVAL, "null argument");
    cw_circuit *c = new cw_circuit();
    try {
        deserialize_tape((const uint8_t *)data, len, c->tape);
    } catch (const std::exception &e) {
        delete c;
        return fail(CW_EFORMAT, e.what());
    }
    *out = c;
    return CW_OK;
}

// packed records of instances [first, first + count) into caller-provided DEVICE memory (count * words * 4 bytes),
// asynchronously on the batch stream: what a gather to another GPU sends
int cw_batch_pack_device(cw_batch *b, uint32_t first, uint32_t count, uint32_t *dst_device) {
    if (!b || !dst_device || (uint64_t)first + count > b->batch) return fail(CW_EINVAL, "bad argument");
    if (!b->ran) return fail(CW_ESTATE, "batch has not been run");
    CU(cudaSetDevice(b->device));
    const PackLayout &L = b->c->pack_layout();
    if (!b->pack_flag_d) CU(cudaMalloc((void **)&b->pack_flag_d, 4));
    return pack_rows(b, L, first, count, dst_device);
}

// NCCL is resolved at run time (dlopen): the library loads and every single-GPU entry point works on machines
// without NCCL, and inside a process that already carries a copy (PyTorch's) that copy is the one used.
namespace {
struct NcclApi {
    void *h = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*Broadcast)(const void *, void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllReduce)(const void *, void *, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Send)(const void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Recv)(void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char *(*GetErrorString)(ncclResult_t) = nullptr;
};
NcclApi g_nccl;
std::mutex g_nccl_mu;

int load_nccl() {
    std::lock_guard<std::mutex> lk(g_nccl_mu);
    if (g_nccl.h) return CW_OK;
    void *h = nullptr;
    const char *env = getenv("CW_NCCL_LIB");
    for (const char *name : {env ? env : "libnccl.so.2", "libnccl.so.2", "libnccl.so"}) {
        h = dlopen(name, RTLD_NOW | RTLD_GLOBAL);
        if (h) break;
    }
    if (!h) return fail(CW_ENODEV, "NCCL is not available (libnccl.so.2 could not be loaded)");
    NcclApi a;
    a.h = h;
#define CW_SYM(field, sym)                                             \
    *(void **)(&a.field) = dlsym(h, sym);                              \
    if (!a.field) return fail(CW_ENODEV, std::string("NCCL symbol missing: ") + sym)
    CW_SYM(GetUniqueId, "ncclGetUniqueId");
    CW_SYM(CommInitRank, "ncclCommInitRank");
    CW_SYM(CommDestroy, "ncclCommDestroy");
    CW_SYM(Broadcast, "ncclBroadcast");
    CW_SYM(AllReduce, "ncclAllReduce");
    CW_SYM(Send, "ncclSend");
    CW_SYM(Recv, "ncclRecv");
    CW_SYM(GroupStart, "ncclGroupStart");
    CW_SYM(GroupEnd, "ncclGroupEnd");
    CW_SYM(GetErrorString, "ncclGetErrorString");
#undef CW_SYM
    g_nccl = a;
    return CW_OK;
}
#define NC(call)                                                                                           \
    do {                                                                                                   \
        ncclResult_t r_ = (call);                                                                          \
        if (r_ != ncclSuccess) return fail(CW_ECUDA, std::string(#call) + ": " + g_nccl.GetErrorString(r_)); \
    } while (0)
}  // namespace

struct cw_comm {
    ncclComm_t comm = nullptr;
    int rank = 0, world = 1, device = 0;
    bool owned = false;
    cudaStream_t stream = nullptr;
    uint64_t bytes_sent = 0, bytes_received = 0;  // payload bytes this rank moved through the data-path collectives
};

int cw_comm_unique_id(uint8_t id[CW_COMM_ID_BYTES]) {
    if (!id) return fail(CW_EINVAL, "null argument");
    int rc = load_nccl();
    if (rc) return rc;
    static_assert(sizeof(ncclUniqueId) == CW_COMM_ID_BYTES, "ncclUniqueId size");
    ncclUniqueId u;
    NC(g_nccl.GetUniqueId(&u));
    memcpy(id, &u, sizeof(u));
    return CW_OK;
}

int cw_comm_init(const uint8_t id[CW_COMM_ID_BYTES], int rank, int world, int device, cw_comm **out) {
    if (!id || !out || world < 1 || rank < 0 || rank >= world) return fail(CW_EINVAL, "bad argument");
    int rc = load_nccl();
    if (rc) return rc;
    if ((rc = ensure_device(device))) return rc;
    ncclUniqueId u;
    memcpy(&u, id, sizeof(u));
    cw_comm *c = new cw_comm();
    c->rank = rank;
    c->world = world;
    c->device = device;
    c->owned = true;
    ncclResult_t r = g_nccl.CommInitRank(&c->comm, world, u, rank);
    if (r != ncclSuccess) {
        delete c;
        return fail(CW_ECUDA, std::string("ncclCommInitRank: ") + g_nccl.GetErrorString(r));
    }
    CU(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    *out = c;
    return CW_OK;
}

int cw_comm_from_nccl(void *nccl_comm, int rank, int world, int device, cw_comm **out) {
    if (!nccl_comm || !out || world < 1 || rank < 0 || rank >= world) return fail(CW_EINVAL, "bad argument");
    int rc = load_nccl();
    if (rc) return rc;
    if ((rc = ensure_device(device))) return rc;
    cw_comm *c = new cw_comm();
    c->comm = (ncclComm_t)nccl_comm;
    c->rank = rank;
    c->world = world;
    c->device = device;
    CU(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    *out = c;
    return CW_OK;
}

void cw_comm_destroy(cw_comm *c) {
    if (!c) return;
    cudaSetDevice(c->device);
    if (c->stream) {
        cudaStreamSynchronize(c->stream);
        cudaStreamDestroy(c->stream);
    }
    if (c->owned && c->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(c->comm);
    delete c;
}

int cw_comm_stats(const cw_comm *c, uint64_t *bytes_sent, uint64_t *bytes_received) {
    if (!c) return fail(CW_EINVAL, "null argument");
    if (bytes_sent) *bytes_sent = c->bytes_sent;
    if (bytes_received) *bytes_received = c->bytes_received;
    return CW_OK;
}

// The lowered circuit of `root` (instruction tape, constants, witness maps, function code, input tables, R1CS in
// CSR form) on every rank: ONE NCCL broadcast of the size and one of the blob; only the root lowers.
int cw_circuit_broadcast(cw_comm *cm, cw_circuit **c, int root) {
    if (!cm || !c || root < 0 || root >= cm->world) return fail(CW_EINVAL, "bad argument");
    if (cm->rank == root && !*c) return fail(CW_EINVAL, "the root must pass its circuit");
    CU(cudaSetDevice(cm->device));
    std::vector<uint8_t> blob;
    if (cm->rank == root) serialize_tape((*c)->tape, blob);
    unsigned long long n = blob.size(), *n_d = nullptr;
    CU(cudaMalloc((void **)&n_d, 8));
    CU(cudaMemcpy(n_d, &n, 8, cudaMemcpyHostToDevice));
    NC(g_nccl.Broadcast(n_d, n_d, 8, ncclUint8, root, cm->comm, cm->stream));
    CU(cudaStreamSynchronize(cm->stream));
    CU(cudaMemcpy(&n, n_d, 8, cudaMemcpyDeviceToHost));
    cudaFree(n_d);
    uint8_t *buf_d = nullptr;
    CU(cudaMalloc((void **)&buf_d, n ? n : 16));
    if (cm->rank == root) CU(cudaMemcpy(buf_d, blob.data(), n, cudaMemcpyHostToDevice));
    NC(g_nccl.Broadcast(buf_d, buf_d, n, ncclUint8, root, cm->comm, cm->stream));
    CU(cudaStreamSynchronize(cm->stream));
    int rc = CW_OK;
    if (cm->rank != root) {
        blob.resize(n);
        CU(cudaMemcpy(blob.data(), buf_d, n, cudaMemcpyDeviceToHost));
        rc = cw_circuit_deserialize(blob.data(), blob.size(), c);
        cm->bytes_received += n;
    } else cm->bytes_sent += n * (uint64_t)(cm->world - 1);
    cudaFree(buf_d);
    return rc;
}

// Gather of witness vectors: every rank packs instances [first, first + count) of its batch on the device and sends
// the records to `root` over NVLink (grouped ncclSend / ncclRecv); on the root recv_device[r][count][words] holds
// rank r's records (its own are packed in place).  Packed records, not 32-byte rows: 30x fewer bytes for circuits
// of bit decompositions; the root expands what it needs (cw_circuit_pack_info).  ms = device time on the root /
// sender of pack + transfer.
int cw_batch_gather_witness_packed(cw_comm *cm, cw_batch *b, uint32_t first, uint32_t count, int root,
                                   uint32_t *recv_device, uint32_t *send_scratch_device, float *ms) {
    if (!cm || !b || root < 0 || root >= cm->world || (uint64_t)first + count > b->batch) return fail(CW_EINVAL, "bad argument");
    if (!b->ran) return fail(CW_ESTATE, "batch has not been run");
    if (cm->rank == root && !recv_device) return fail(CW_EINVAL, "the root needs a receive buffer");
    if (cm->rank != root && !send_scratch_device) return fail(CW_EINVAL, "senders need a scratch buffer of count * words * 4 bytes");
    CU(cudaSetDevice(b->device));
    const PackLayout &L = b->c->pack_layout();
    const size_t n = (size_t)count * L.words * 4;  // bytes per rank
    cudaEvent_t e0, e1;
    CU(cudaEventCreate(&e0));
    CU(cudaEventCreate(&e1));
    CU(cudaEventRecord(e0, b->stream));
    uint32_t *mine = cm->rank == root ? recv_device + (size_t)root * count * L.words : send_scratch_device;
    int rc = cw_batch_pack_device(b, first, count, mine);
    if (rc) return rc;
    NC(g_nccl.GroupStart());
    if (cm->rank == root) {
        for (int r = 0; r < cm->world; ++r)
            if (r != root) NC(g_nccl.Recv(recv_device + (size_t)r * count * L.words, n, ncclUint8, r, cm->comm, b->stream));
    } else {
        NC(g_nccl.Send(mine, n, ncclUint8, root, cm->comm, b->stream));
    }
    NC(g_nccl.GroupEnd());
    CU(cudaEventRecord(e1, b->stream));
    CU(cudaStreamSynchronize(b->stream));
    if (ms) CU(cudaEventElapsedTime(ms, e0, e1));
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    if (cm->rank == root) cm->bytes_received += n * (uint64_t)(cm->world - 1);
    else cm->bytes_sent += n;
    return CW_OK;
}

// all ranks learn whether any instance of any rank failed: out[0] = number of instances with a failed assert,
// out[1] = number with a runtime error, summed over the communicator (ncclAllReduce of two counters)
int cw_status_allreduce(cw_comm *cm, cw_batch *b, uint64_t out[2]) {
    if (!cm || !b || !out) return fail(CW_EINVAL, "null argument");
    std::vector<int32_t> st(b->batch);
    int rc = cw_batch_status(b, st.data());
    if (rc) return rc;
    unsigned long long h[2] = {0, 0}, *d = nullptr;
    for (int32_t s : st) {
        if (s > 0) ++h[0];
        else if (s < 0) ++h[1];
    }
    CU(cudaMalloc((void **)&d, 16));
    CU(cudaMemcpyAsync(d, h, 16, cudaMemcpyHostToDevice, b->stream));
    NC(g_nccl.AllReduce(d, d, 2, ncclUint64, ncclSum, cm->comm, b->stream));
    CU(cudaMemcpyAsync(h, d, 16, cudaMemcpyDeviceToHost, b->stream));
    CU(cudaStreamSynchronize(b->stream));
    cudaFree(d);
    out[0] = h[0];
    out[1] = h[1];
    return CW_OK;
}

// ---- field batch ops ---------------------------------------------------------------------------
int cw_fr_batch_op(int prime_id, int op, const uint64_t *a, const uint64_t *b, const uint64_t *c, uint64_t *r,
                   size_t n, int device) {
    if (!a || !r || prime_id < 0 || prime_id >= CW_N_PRIMES) return fail(CW_EINVAL, "bad argument");
    int rc = ensure_device(device);
    if (rc) return rc;
    uint4 *A = nullptr, *B = nullptr, *C = nullptr, *Rr = nullptr;
    int *err = nullptr;
    if ((rc = upload(&A, a, n * 32))) return rc;
    if (b && (rc = upload(&B, b, n * 32))) return rc;
    if (c && (rc = upload(&C, c, n * 32))) return rc;
    CU(cudaMalloc((void **)&Rr, n * 32 + 32));
    CU(cudaMalloc((void **)&err, 4));
    CU(cudaMemset(err, 0, 4));
    u32 grid = (u32)std::min<size_t>((n + 127) / 128, 148 * 16);
    if (!grid) grid = 1;
    if (prime_id == 0) fr_batch_op_kernel<0><<<grid, 128>>>(op, A, B, C, Rr, n, err, 0u);
    else if (prime_id == 1) fr_batch_op_kernel<1><<<grid, 128>>>(op, A, B, C, Rr, n, err, 1u);
    else fr_batch_op_kernel<-1><<<grid, 128>>>(op, A, B, C, Rr, n, err, (u32)prime_id);
    CU(cudaGetLastError());
    CU(cudaMemcpy(r, Rr, n * 32, cudaMemcpyDeviceToHost));
    int herr = 0;
    CU(cudaMemcpy(&herr, err, 4, cudaMemcpyDeviceToHost));
    cudaFree(A);
    cudaFree(B);
    cudaFree(C);
    cudaFree(Rr);
    cudaFree(err);
    return herr ? fail(CW_EINVAL, "division by zero in batch op") : CW_OK;
}

int cw_fr_mul_bench(int prime_id, size_t n, int iters, int device, float *ms) {
    if (prime_id < 0 || prime_id > 1 || !ms) return fail(CW_EINVAL, "the throughput probe is built for bn128 and bls12381");
    int rc = ensure_device(device);
    if (rc) return rc;
    std::vector<uint64_t> h(n * 4);
    uint64_t s = 0x9E3779B97F4A7C15ull;
    for (auto &x : h) {
        s ^= s << 13; s ^= s >> 7; s ^= s << 17;
        x = s;
    }
    for (size_t i = 0; i < n; ++i) h[4 * i + 3] &= 0x0FFFFFFFFFFFFFFFull;
    uint4 *d = nullptr;
    if ((rc = upload(&d, h.data(), n * 32))) return rc;
    cudaEvent_t e0, e1;
    CU(cudaEventCreate(&e0));
    CU(cudaEventCreate(&e1));
    u32 grid = (u32)((n + 255) / 256);
    for (int rep = 0; rep < 2; ++rep) {
        CU(cudaEventRecord(e0));
        if (prime_id == 0) fr_mul_bench_kernel<0><<<grid, 256>>>(d, n, iters);
        else fr_mul_bench_kernel<1><<<grid, 256>>>(d, n, iters);
        CU(cudaEventRecord(e1));
        CU(cudaEventSynchronize(e1));
    }
    CU(cudaEventElapsedTime(ms, e0, e1));
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    cudaFree(d);
    return CW_OK;
}

}  // extern "C"
