// Lowering: circuit description (.cb2c) -> flat, levelised instruction tape.
//
// This is the job a `cuda_elements` code producer does in place of
// Circuit::produce_c (compiler/src/circuit_design/circuit.rs:596-612): instead of
// printing one C++ function per template instance, the component tree is
// instantiated once and its field operations are emitted as a single SSA tape.
//
//   1. symbolic execution in the reference's run order: a sub-component body is
//      expanded when its last input is stored (store_bucket.rs:660-734,
//      template.rs:274-278), so the emission order is a valid schedule;
//   2. moves are removed by aliasing (Fr_copy of store_bucket.rs:607-646 becomes
//      slot renaming);
//   3. static representation inference: each value lives in canonical or
//      Montgomery form, decided here, replacing the reference's run-time
//      tri-state dispatch (generic/fr.cpp:416-533); a Montgomery product of a
//      Montgomery and a canonical operand is canonical for free, exactly the
//      mixed case of Fr_mul (generic/fr.cpp:449-465); conversions are cached;
//   4. dead values are dropped, ops are levelised (wavefronts), sorted by
//      (level, opcode) and slots renumbered so that the destination of tape
//      op i is slot n_pre + i.
#include <algorithm>
#include <bitset>
#include <cstdio>
#include <cstring>
#include <functional>
#include <stdexcept>
#include <unordered_map>

#include "../../include/circom_b200.h"
#include "tape.h"

namespace cw {

uint64_t fnv1a(const char *s, size_t n) {  // calcwit.cpp:17-24
    uint64_t h = 0xCBF29CE484222325ULL;
    for (size_t i = 0; i < n; ++i) {
        h ^= (uint64_t)(int64_t)(signed char)s[i];  // `u64(c)` of a (signed) char
        h *= 0x100000001B3ULL;
    }
    return h;
}

namespace {

enum { K_NONE = 0, K_OWN = 1, K_SUB = 2, K_CONST = 3, K_TMP = 4, K_ONE = 5 };
// FC canonical x; FM Montgomery x*R; FD "deferred" x*R^-1: the raw Montgomery product of two canonical
// operands.  Zero tests read any form; FD is converted (one product, like converting an input would
// have cost) only if a consumer needs the value itself.
enum Form { FC = 0, FM = 1, FD = 2 };

struct IrOp {
    uint32_t op;
    uint64_t d, a, b, c;
};
struct Term {
    uint64_t ref;
    uint32_t cid;
};
struct Tmpl {
    std::string name;
    uint32_t n_out, n_in, n_inter, n_tmp, n_own;
    std::vector<uint32_t> subs;
    std::vector<IrOp> ops;
    std::vector<uint32_t> lc_len;  // 3 per constraint
    std::vector<Term> terms;
    std::vector<uint8_t> tmp_zero_only;  // temporary is consumed by zero / non-zero tests only
    uint64_t total_signals = 0, total_components = 0;
};

inline int rk(uint64_t r) { return (int)(r >> 56); }
inline uint32_t rsub(uint64_t r) { return (uint32_t)((r >> 32) & 0xFFFFFF); }
inline uint32_t ridx(uint64_t r) { return (uint32_t)r; }

struct Reader {
    const uint8_t *p, *end;
    template <class T>
    T get() {
        if (p + sizeof(T) > end) throw std::runtime_error("cb2c: truncated");
        T v;
        memcpy(&v, p, sizeof(T));
        p += sizeof(T);
        return v;
    }
    const uint8_t *bytes(size_t n) {
        if (n > (size_t)(end - p)) throw std::runtime_error("cb2c: truncated");
        const uint8_t *r = p;
        p += n;
        return r;
    }
    size_t left() const { return (size_t)(end - p); }
    // a count read from the file must be backed by that many records of `bytes_each` bytes
    void expect(uint64_t count, uint64_t bytes_each) const {
        if (count * bytes_each > left()) throw std::runtime_error("cb2c: truncated (count exceeds the file)");
    }
    std::string str() {
        uint32_t n = get<uint32_t>();
        const uint8_t *b = bytes((size_t)(((uint64_t)n + 3) & ~3ull));  // (64-bit: n = 2^32 - 1 must not wrap to 0)
        return std::string((const char *)b, n);
    }
};

struct Val {
    uint32_t slot[3] = {NO_SLOT, NO_SLOT, NO_SLOT};  // provisional slot per representation (Form)
    int32_t cid = -1;                       // IR constant id if this value is a compile-time constant
    // static knowledge used by the peepholes
    uint16_t bits = 256;                    // the canonical integer is < 2^bits (256 = nothing known)
    uint8_t org_op = 0;                     // IR opcode that produced the value (0 = input / constant)
    int32_t org_a = -1, org_b = -1;         // its operand values
    // bit-field provenance (integer identities on the canonical value of `src`):
    //   fld_src >= 0 : value == (src >> fld_k) & (2^fld_m - 1)                (a field moved to position 0)
    //   bf_src  >= 0 : value == src & ((2^bf_len - 1) << bf_lo)               (a field left in place)
    // An in-place field may be *virtual* (no slot yet): sums of adjacent in-place fields of the same
    // source are again in-place fields, so `sum_i ((x >> i) & 1) << i` never materialises its terms.
    int32_t fld_src = -1, bf_src = -1;
    uint16_t fld_k = 0, fld_m = 0, bf_lo = 0, bf_len = 0;
};

// device-only opcodes (kernels.cuh / fr_device.cuh)
enum { DOP_BITS = 29, DOP_ASSERT_BOOL = 30, DOP_MULSMALL = 31, DOP_BITSIP = 32, DOP_ASSERT_FITS = 33,
       DOP_ADD_NR = 34, DOP_ADD128 = 35, DOP_MULSMALL128 = 36, DOP_MULSMALL192 = 37, DOP_SHRI = 38, DOP_SHLI = 39 };
inline bool c_is_immediate(uint32_t opcode) {
    return opcode == CW_OP_ASSERT || opcode == CW_OP_ASSERT_EQ || opcode == DOP_BITS || opcode == DOP_ASSERT_BOOL ||
           opcode == DOP_BITSIP || opcode == DOP_ASSERT_FITS;
}
inline bool is_assert_op(uint32_t opcode) {
    return opcode == CW_OP_ASSERT || opcode == CW_OP_ASSERT_EQ || opcode == DOP_ASSERT_BOOL || opcode == DOP_ASSERT_FITS;
}

inline size_t n_live_ops(const std::vector<uint8_t> &live, uint32_t n_pre, size_t n_prov) {
    size_t n = 0;
    for (size_t i = 0; i < n_prov; ++i) n += live[n_pre + i];
    return n;
}
// accumulators a fused sub-tree needs while it is evaluated (1: a chain)
inline int subtree_need(uint32_t i, const std::vector<uint32_t> &kid_a, const std::vector<uint32_t> &kid_b) {
    const uint32_t a = kid_a[i], b = kid_b[i];
    if (a == NO_SLOT && b == NO_SLOT) return 1;
    if (a == NO_SLOT) return subtree_need(b, kid_a, kid_b);
    if (b == NO_SLOT) return subtree_need(a, kid_a, kid_b);
    const int na = subtree_need(a, kid_a, kid_b), nb = subtree_need(b, kid_a, kid_b);
    return std::max(std::max(na, nb), std::min(na, nb) + 1);
}

// ---- copy coalescing in function bodies ---------------------------------------------------------------------------
// The producers write `x = e` as the expression into a temporary followed by a copy (the C++ producer's
// `Fr_add(&expaux[0], ..); Fr_copy(&lvar[x], &expaux[0]);`): a quarter of the instructions an interpreted call executes.
// When the temporary is written by the instruction just before the copy, dies with it, and no jump lands on the copy, the
// expression writes its destination directly and the copy disappears.  Returns the new instruction count.
static uint32_t coalesce_function_copies(uint32_t *code, uint32_t n_instr, uint32_t n_regs, const std::vector<uint32_t> &fn_params) {
    constexpr uint32_t MAXR = 192;
    if (n_regs > MAXR || n_instr < 2) return n_instr;
    using Set = std::bitset<MAXR>;
    enum { JMP = 40, JZ = 41, RET = 42, LOADX = 43, STOREX = 44, CALLF = 45, COPY = 24 };
    auto is_reg = [&](uint32_t o) { return !(o & 0xC0000000u) && o < n_regs; };
    Set pinned;
    std::vector<uint8_t> target(n_instr + 1, 0);
    for (uint32_t i = 0; i < n_instr; ++i) {
        const uint32_t *w = &code[5 * (size_t)i];
        uint32_t lo = 0, hi = 0;
        if (w[0] == LOADX) { lo = w[2] & 0x3FFFFFFFu; hi = w[4] & 0x3FFFFFFFu; }
        else if (w[0] == STOREX) { lo = w[2] & 0x3FFFFFFFu; hi = w[1] & 0x3FFFFFFFu; }
        else if (w[0] == RET && (w[3] & 0x3FFFFFFFu) > 1) { lo = w[2]; hi = lo + (w[3] & 0x3FFFFFFFu); }
        else if (w[0] == CALLF) {   // the argument registers are one block; several results too
            for (uint32_t r = w[3]; r < w[3] + fn_params[w[2] & 0x3FFFFFFFu] && r < n_regs; ++r) pinned.set(r);
            if ((w[4] & 0x3FFFFFFFu) > 1) { lo = w[1]; hi = lo + (w[4] & 0x3FFFFFFFu); }
        }
        for (uint32_t r = lo; r < hi && r < n_regs; ++r) pinned.set(r);
        if (w[0] == JMP) target[std::min(w[2] & 0x3FFFFFFFu, n_instr)] = 1;
        if (w[0] == JZ) target[std::min(w[3] & 0x3FFFFFFFu, n_instr)] = 1;
    }
    // liveness of the scalars (as in allocate_function_registers)
    std::vector<Set> use(n_instr), live_in(n_instr), live_out(n_instr);
    std::vector<int> def(n_instr, -1);
    auto add_use = [&](uint32_t i, uint32_t o) { if (is_reg(o) && !pinned.test(o)) use[i].set(o); };
    for (uint32_t i = 0; i < n_instr; ++i) {
        const uint32_t *w = &code[5 * (size_t)i];
        switch (w[0]) {
            case JMP: break;
            case JZ: add_use(i, w[2]); break;
            case RET: if ((w[3] & 0x3FFFFFFFu) <= 1) add_use(i, w[2]); break;
            case LOADX: add_use(i, w[3]); if (!pinned.test(w[1])) def[i] = (int)w[1]; break;
            case STOREX: add_use(i, w[3]); add_use(i, w[4]); break;
            case CALLF: if (!pinned.test(w[1])) def[i] = (int)w[1]; break;   // (arguments: pinned registers)
            default: add_use(i, w[2]); add_use(i, w[3]); add_use(i, w[4]); if (!pinned.test(w[1])) def[i] = (int)w[1];
        }
    }
    for (bool changed = true; changed;) {
        changed = false;
        for (uint32_t i = n_instr; i-- > 0;) {
            const uint32_t *w = &code[5 * (size_t)i];
            Set out;
            if (w[0] == JMP) out = live_in[w[2] & 0x3FFFFFFFu];
            else if (w[0] != RET) {
                if (i + 1 < n_instr) out = live_in[i + 1];
                if (w[0] == JZ) out |= live_in[w[3] & 0x3FFFFFFFu];
            }
            Set in = out;
            if (def[i] >= 0) in.reset((size_t)def[i]);
            in |= use[i];
            if (in != live_in[i] || out != live_out[i]) { live_in[i] = in; live_out[i] = out; changed = true; }
        }
    }
    std::vector<uint8_t> dead(n_instr, 0);
    for (uint32_t i = 1; i < n_instr; ++i) {
        uint32_t *c = &code[5 * (size_t)i], *p = &code[5 * (size_t)(i - 1)];
        if (c[0] != COPY || target[i] || dead[i - 1]) continue;
        const uint32_t t = c[2], d = c[1];
        if (!is_reg(t) || pinned.test(t) || t == d || def[i - 1] != (int)t || live_out[i].test(t)) continue;
        if (p[0] == JMP || p[0] == JZ || p[0] == RET || p[0] == STOREX) continue;   // (def[] is -1 for these anyway)
        p[1] = d;      // the producer writes the destination of the copy
        dead[i] = 1;
    }
    std::vector<uint32_t> newidx(n_instr + 1, 0);
    uint32_t n = 0;
    for (uint32_t i = 0; i < n_instr; ++i) { newidx[i] = n; n += !dead[i]; }
    newidx[n_instr] = n;
    if (n == n_instr) return n_instr;
    for (uint32_t i = 0; i < n_instr; ++i) {
        uint32_t *w = &code[5 * (size_t)i];
        if (w[0] == JMP) w[2] = 0x40000000u | newidx[w[2] & 0x3FFFFFFFu];
        if (w[0] == JZ) w[3] = 0x40000000u | newidx[w[3] & 0x3FFFFFFFu];
    }
    for (uint32_t i = 0; i < n_instr; ++i)
        if (!dead[i] && newidx[i] != i) memmove(&code[5 * (size_t)newidx[i]], &code[5 * (size_t)i], 20);
    return n;
}

// ---- register allocation for function bodies ---------------------------------------------------------------------
// A compiler-written function body gives every expression temporary its own register (the `expaux` of the C++ producer) and
// every variable its own slot; the interpreter keeps the registers of a call in the thread's local memory (32 bytes each,
// dynamically indexed), so the frame size is what a call costs: hundreds of concurrent calls per SM each touching a 3 KB frame
// live in L2 / DRAM instead of L1.  Scalars are therefore packed: liveness over the control-flow graph, interference, greedy
// colouring.  Registers that can be reached through a run-time index (LOADX / STOREX ranges [base, limit), array returns)
// are never shared: a range that contains parameters stays where it is, the others move behind the scalars as blocks.
// Parameters keep their registers (the caller stores the arguments there); a dead parameter's register is reused.
// Registers read before they are written rely on the zero-initialised frame: they stay live from the entry and may not
// share a register with a parameter.
static void allocate_function_registers(uint32_t *code, uint32_t n_instr, uint32_t n_params, uint32_t &n_regs,
                                        const std::vector<uint32_t> &fn_params) {
    constexpr uint32_t MAXR = 192;
    if (n_regs > MAXR || n_regs == 0 || n_instr == 0) return;
    using Set = std::bitset<MAXR>;
    auto is_reg = [](uint32_t o) { return !(o & 0xC0000000u); };
    enum { JMP = 40, JZ = 41, RET = 42, LOADX = 43, STOREX = 44, CALLF = 45 };
    // registers reachable through a run-time index
    Set pinned;
    for (uint32_t i = 0; i < n_instr; ++i) {
        const uint32_t *w = &code[5 * (size_t)i];
        uint32_t lo = 0, hi = 0;
        if (w[0] == LOADX) { lo = w[2] & 0x3FFFFFFFu; hi = w[4] & 0x3FFFFFFFu; }
        else if (w[0] == STOREX) { lo = w[2] & 0x3FFFFFFFu; hi = w[1] & 0x3FFFFFFFu; }
        else if (w[0] == RET && (w[3] & 0x3FFFFFFFu) > 1) { lo = w[2]; hi = lo + (w[3] & 0x3FFFFFFFu); }
        else if (w[0] == CALLF) {   // the argument registers are one block; several results too
            for (uint32_t r = w[3]; r < w[3] + fn_params[w[2] & 0x3FFFFFFFu] && r < n_regs; ++r) pinned.set(r);
            if ((w[4] & 0x3FFFFFFFu) > 1) { lo = w[1]; hi = lo + (w[4] & 0x3FFFFFFFu); }
        }
        for (uint32_t r = lo; r < hi && r < n_regs; ++r) pinned.set(r);
    }
    // per instruction: registers read / the register written, scalars only
    std::vector<Set> use(n_instr), live_in(n_instr), live_out(n_instr);
    std::vector<int> def(n_instr, -1);
    auto add_use = [&](uint32_t i, uint32_t o) { if (is_reg(o) && o < n_regs && !pinned.test(o)) use[i].set(o); };
    for (uint32_t i = 0; i < n_instr; ++i) {
        const uint32_t *w = &code[5 * (size_t)i];
        switch (w[0]) {
            case JMP: break;
            case JZ: add_use(i, w[2]); break;
            case RET: if ((w[3] & 0x3FFFFFFFu) <= 1) add_use(i, w[2]); break;
            case LOADX: add_use(i, w[3]); if (!pinned.test(w[1])) def[i] = (int)w[1]; break;
            case STOREX: add_use(i, w[3]); add_use(i, w[4]); break;
            case CALLF: if (!pinned.test(w[1])) def[i] = (int)w[1]; break;   // (arguments: pinned registers)
            default: add_use(i, w[2]); add_use(i, w[3]); add_use(i, w[4]); if (!pinned.test(w[1])) def[i] = (int)w[1];
        }
    }
    for (bool changed = true; changed;) {
        changed = false;
        for (uint32_t i = n_instr; i-- > 0;) {
            const uint32_t *w = &code[5 * (size_t)i];
            Set out;
            if (w[0] == JMP) { out = live_in[w[2] & 0x3FFFFFFFu]; }
            else if (w[0] == RET) {}
            else {
                if (i + 1 < n_instr) out = live_in[i + 1];
                if (w[0] == JZ) out |= live_in[w[3] & 0x3FFFFFFFu];
            }
            Set in = out;
            if (def[i] >= 0) in.reset((size_t)def[i]);
            in |= use[i];
            if (in != live_in[i] || out != live_out[i]) { live_in[i] = in; live_out[i] = out; changed = true; }
        }
    }
    // interference
    std::vector<Set> edge(n_regs);
    auto connect = [&](uint32_t a, uint32_t b) { if (a != b) { edge[a].set(b); edge[b].set(a); } };
    for (uint32_t i = 0; i < n_instr; ++i)
        if (def[i] >= 0)
            for (uint32_t r = 0; r < n_regs; ++r)
                if (live_out[i].test(r)) connect((uint32_t)def[i], r);
    for (uint32_t p = 0; p < n_params; ++p)   // the arguments are all written before the first instruction
        for (uint32_t r = 0; r < n_regs; ++r)
            if (!pinned.test(p) && !pinned.test(r) && (r < n_params || live_in[0].test(r))) connect(p, r);
    // which scalars exist at all (a register no instruction names needs no place)
    Set named;
    for (uint32_t i = 0; i < n_instr; ++i) { named |= use[i]; if (def[i] >= 0) named.set((size_t)def[i]); }
    // pinned ranges (maximal runs); a run that reaches into the parameters stays in place
    struct Run { uint32_t lo, hi; bool fixed; };
    std::vector<Run> runs;
    for (uint32_t r = 0; r < n_regs;) {
        if (!pinned.test(r)) { ++r; continue; }
        uint32_t e = r;
        while (e < n_regs && pinned.test(e)) ++e;
        runs.push_back({r, e, r < n_params});
        r = e;
    }
    std::vector<uint32_t> map(n_regs, 0xFFFFFFFFu);
    Set taken;   // places no scalar may use
    for (const Run &ru : runs)
        if (ru.fixed)
            for (uint32_t r = ru.lo; r < ru.hi; ++r) { map[r] = r; taken.set(r); }
    for (uint32_t p = 0; p < n_params; ++p)
        if (map[p] == 0xFFFFFFFFu) map[p] = p;
    uint32_t top = n_params;
    for (const Run &ru : runs)
        if (ru.fixed) top = std::max(top, ru.hi);
    for (uint32_t r = n_params; r < n_regs; ++r) {
        if (pinned.test(r) || !named.test(r)) continue;
        Set busy = taken;
        for (uint32_t o = 0; o < n_regs; ++o)
            if (edge[r].test(o) && map[o] != 0xFFFFFFFFu && !pinned.test(o)) busy.set(map[o]);
        uint32_t c = 0;
        while (c < MAXR && busy.test(c)) ++c;
        if (c >= MAXR) return;   // (cannot happen: the identity is a valid colouring)
        map[r] = c;
        top = std::max(top, c + 1);
    }
    for (const Run &ru : runs) {
        if (ru.fixed) continue;
        for (uint32_t r = ru.lo; r < ru.hi; ++r) map[r] = top + (r - ru.lo);
        top += ru.hi - ru.lo;
    }
    if (top > n_regs) return;    // (no gain; keep the original numbering)
    auto m = [&](uint32_t o) { return is_reg(o) && o < n_regs && map[o] != 0xFFFFFFFFu ? map[o] : o; };
    for (uint32_t i = 0; i < n_instr; ++i) {
        uint32_t *w = &code[5 * (size_t)i];
        switch (w[0]) {
            case JMP: break;
            case JZ: w[2] = m(w[2]); break;
            case RET: w[2] = m(w[2]); break;   // (an array return names its first register: pinned, mapped like the others)
            case LOADX: case STOREX: {
                const uint32_t base = w[2] & 0x3FFFFFFFu, lim = (w[0] == LOADX ? w[4] : w[1]) & 0x3FFFFFFFu;
                // base == limit (an empty range) names no register: any in-frame value will do
                const uint32_t nb = base < lim && base < n_regs ? map[base] : 0, nl = nb + (lim > base ? lim - base : 0);
                w[2] = 0x40000000u | nb;
                if (w[0] == LOADX) { w[1] = m(w[1]); w[3] = m(w[3]); w[4] = 0x40000000u | nl; }
                else { w[3] = m(w[3]); w[4] = m(w[4]); w[1] = 0x40000000u | nl; }
                break;
            }
            case CALLF: w[1] = m(w[1]); if (fn_params[w[2] & 0x3FFFFFFFu]) w[3] = m(w[3]); break;
            default: w[1] = m(w[1]); w[2] = m(w[2]); w[3] = m(w[3]); w[4] = m(w[4]);
        }
    }
    n_regs = std::max<uint32_t>(top, 1);
}

struct Lowerer {
    Tape &T;
    const FieldParams &F;
    uint32_t flags;
    std::vector<Tmpl> tm;
    std::vector<U256> ir_consts;
    std::vector<Val> vals;
    std::vector<int32_t> sig_vid;
    // provisional tape
    std::vector<uint32_t> pops;  // 4 words per op
    std::vector<uint32_t> pcalls;  // provisional call table: {function, n_args, arg operands..., n_extra, provisional slots of results 1..}
    std::vector<uint32_t> fn_min_ret;  // per function: the fewest values any of its RETs returns
    std::vector<uint32_t> fn_stack_regs, fn_stack_depth;  // per function: registers / frames of its deepest chain of calls
    std::vector<uint32_t> plevel;
    std::vector<uint32_t> slot_level;  // per provisional slot
    // constant table (raw patterns)
    std::vector<U256> consts;
    std::unordered_map<std::string, uint32_t> const_index;
    uint32_t n_pre = 0;
    uint64_t n_ir_ops = 0, n_conv = 0, n_asserts = 0, n_static_asserts = 0;
    int64_t max_log_string = -1;
    struct PendingLog { uint8_t kind; bool last; uint64_t idx; };   // kind 1: idx = global signal id until the witness exists
    std::vector<PendingLog> pending_logs;
    int32_t vid_one = -1;

    Lowerer(Tape &t, uint32_t fl) : T(t), F(t.F), flags(fl) {}

    uint32_t raw_const(const U256 &v) {
        std::string key((const char *)v.v, 32);
        auto it = const_index.find(key);
        if (it != const_index.end()) return it->second;
        uint32_t i = (uint32_t)consts.size();
        consts.push_back(v);
        const_index.emplace(std::move(key), i);
        return i;
    }
    uint32_t const_operand(int32_t cid, Form f) {
        const U256 &v = ir_consts[cid];
        return OPERAND_CONST | raw_const(f == FM ? F.to_mont(v) : v);
    }
    uint32_t operand_level(uint32_t o) const { return (o & OPERAND_CONST) || o == NO_SLOT ? 0 : slot_level[o]; }

    uint32_t emit(uint32_t opcode, uint32_t a, uint32_t b = NO_SLOT, uint32_t c = NO_SLOT, bool c_is_imm = false) {
        uint32_t slot = n_pre + (uint32_t)(pops.size() / 4);
        pops.push_back(opcode);
        pops.push_back(a);
        pops.push_back(b);
        pops.push_back(c);
        uint32_t l = std::max(operand_level(a), operand_level(b));
        if (!c_is_imm) l = std::max(l, operand_level(c));
        slot_level.push_back(l + 1);
        return slot;
    }
    int32_t new_val(uint32_t slot, Form f) {
        Val v;
        v.slot[f] = slot;
        vals.push_back(v);
        return (int32_t)vals.size() - 1;
    }
    bool is_virtual(int32_t vid) const {
        const Val &v = vals[vid];
        return v.cid < 0 && v.bf_src >= 0 && v.slot[FC] == NO_SLOT && v.slot[FM] == NO_SLOT && v.slot[FD] == NO_SLOT;
    }
    // a virtual in-place field gets its slot on first real use: one mask op on the source
    void materialise(int32_t vid) {
        if (!is_virtual(vid)) return;
        int32_t src = vals[vid].bf_src;
        uint32_t imm = (uint32_t)vals[vid].bf_lo | ((uint32_t)vals[vid].bf_len << 8);
        uint32_t s = emit(DOP_BITSIP, need(src, FC), NO_SLOT, imm, true);
        vals[vid].slot[FC] = s;
    }
    bool has(int32_t vid, Form f) const {
        return vals[vid].cid >= 0 || vals[vid].slot[f] != NO_SLOT || (f == FC && is_virtual(vid));
    }
    bool is_const(int32_t vid) const { return vals[vid].cid >= 0; }
    // operand holding `vid` in form `f` (FC or FM), converting (once) if necessary
    uint32_t need(int32_t vid, Form f) {
        materialise(vid);
        Val &v = vals[vid];
        if (v.cid >= 0) return const_operand(v.cid, f);
        if (v.slot[f] != NO_SLOT) return v.slot[f];
        uint32_t src = v.slot[1 - f];
        U256 k;
        if (src != NO_SLOT) {
            // to Montgomery: MontMul(x, R^2) = x*R ; to canonical: MontMul(xR, 1) = x
            k = (f == FM) ? F.r2 : u256_from_u64(1);
        } else {
            src = v.slot[FD];
            if (src == NO_SLOT) throw std::runtime_error("lowering: value without representation");
            // from x/R: MontMul(x/R, R^2) = x ; MontMul(x/R, R^3) = x*R
            k = (f == FC) ? F.r2 : F.mont_mul(F.r2, F.r2);
        }
        uint32_t s = emit(CW_OP_MUL, src, OPERAND_CONST | raw_const(k));
        ++n_conv;
        vals[vid].slot[f] = s;
        return s;
    }
    // operand for a zero / non-zero test: any representation will do
    uint32_t need_any(int32_t vid) {
        materialise(vid);
        const Val &v = vals[vid];
        if (v.cid >= 0) return const_operand(v.cid, FC);
        for (int f = 0; f < 3; ++f)
            if (v.slot[f] != NO_SLOT) return v.slot[f];
        throw std::runtime_error("lowering: value without representation");
    }
    bool is_const_zero(int32_t vid) const { return vals[vid].cid >= 0 && ir_consts[vals[vid].cid].is_zero(); }
    bool only_deferred(int32_t vid) const {
        const Val &v = vals[vid];
        return v.cid < 0 && v.slot[FC] == NO_SLOT && v.slot[FM] == NO_SLOT;
    }
    Form any_form(int32_t vid) const {
        const Val &v = vals[vid];
        if (v.cid >= 0) return FC;
        return v.slot[FM] != NO_SLOT ? FM : FC;  // a deferred-only value converts to canonical
    }
    // common form for an operation that needs both operands in the same representation
    Form common_form(int32_t x, int32_t y) const {
        bool xc = is_const(x), yc = is_const(y);
        if (xc && yc) return FC;
        if (xc) return any_form(y);
        if (yc) return any_form(x);
        int cost_m = !has(x, FM) + !has(y, FM), cost_c = !has(x, FC) + !has(y, FC);
        return cost_c < cost_m ? FC : FM;  // fewest conversions; ties stay in the Montgomery domain
    }

    uint32_t qb() const { return F.qbits; }
    uint32_t vbits(int32_t v) const { return v < 0 ? 0 : std::min<uint32_t>(vals[v].bits, qb()); }
    // value of a compile-time constant if it fits 64 bits
    bool const_u64(int32_t v, uint64_t &out) const {
        if (v < 0 || vals[v].cid < 0) return false;
        const U256 &c = ir_consts[vals[v].cid];
        if (c.v[1] | c.v[2] | c.v[3]) return false;
        out = c.v[0];
        return true;
    }
    static int u256_bitlen(const U256 &c) {
        for (int i = 255; i >= 0; --i)
            if ((c.v[i >> 6] >> (i & 63)) & 1) return i + 1;
        return 0;
    }
    // is the constant 2^m - 1 (m >= 1)?  /  2^k ?
    bool const_mask(int32_t v, uint32_t &m) const {
        if (v < 0 || vals[v].cid < 0) return false;
        U256 c = ir_consts[vals[v].cid], one = u256_from_u64(1), t;
        if (u256_add(t, c, one)) return false;
        int bl = u256_bitlen(t);
        if (bl < 2) return false;
        U256 p = u256_from_u64(0);
        p.v[(bl - 1) >> 6] = 1ull << ((bl - 1) & 63);
        if (!(p == t)) return false;
        m = (uint32_t)bl - 1;
        return true;
    }
    bool const_pow2(int32_t v, uint32_t &k) const {
        if (v < 0 || vals[v].cid < 0) return false;
        const U256 &c = ir_consts[vals[v].cid];
        int bl = u256_bitlen(c);
        if (bl < 1) return false;
        U256 p = u256_from_u64(0);
        p.v[(bl - 1) >> 6] = 1ull << ((bl - 1) & 63);
        if (!(p == c)) return false;
        k = (uint32_t)bl - 1;
        return true;
    }
    uint32_t range_of(uint32_t op, int32_t a, int32_t b) const {
        const uint32_t FULL = 256, lim = qb() - 1;
        uint32_t ba = vbits(a), bb = vbits(b);
        uint64_t k;
        switch (op) {
            case CW_OP_ADD: return std::max(ba, bb) + 1 <= lim ? std::max(ba, bb) + 1 : FULL;
            case CW_OP_MUL: return ba + bb <= lim ? ba + bb : FULL;
            case CW_OP_IDIV: return ba;
            case CW_OP_MOD: return std::min(ba, bb);
            // Fr_shr / Fr_shl reverse direction for amounts >= q - qbits ("negative" amounts,
            // generic/fr.cpp:2157-2173,2233-2249): `a >> b` is then a LEFT shift and can be qbits wide.  The
            // operand's width is only a bound of the result when the amount provably is a plain one: a constant
            // below qbits, or a value narrower than qbits - 1 bits (2^(qbits-2) < q - qbits for both primes).
            case CW_OP_SHR:
                if (const_u64(b, k)) return k < qb() ? (ba > k ? ba - (uint32_t)k : 0) : FULL;
                return (b >= 0 && !is_const(b) && bb + 2 <= qb()) ? ba : FULL;
            case CW_OP_SHL: return const_u64(b, k) && ba + k <= lim ? ba + (uint32_t)k : FULL;
            case CW_OP_BAND: return std::min(ba, bb);
            case CW_OP_BOR: case CW_OP_BXOR: return std::max(ba, bb) <= lim ? std::max(ba, bb) : FULL;
            case CW_OP_LEQ: case CW_OP_GEQ: case CW_OP_LT: case CW_OP_GT: case CW_OP_EQ: case CW_OP_NEQ:
            case CW_OP_LOR: case CW_OP_LAND: case CW_OP_LNOT: return 1;
            case CW_OP_SELECT: return std::max(ba, bb);
            default: return FULL;
        }
    }

    int32_t lower_op(uint32_t op, int32_t a, int32_t b, int32_t c, bool zero_test_only = false) {
        int32_t r = -1;
        size_t n_before = vals.size();
        if (!(flags & CW_FLAG_NO_PEEPHOLE)) r = peephole(op, a, b);
        if (r >= 0 && (size_t)r < n_before) return r;  // the result is an existing value (x * 1)
        if (r < 0) r = lower_op_plain(op, a, b, c, zero_test_only);
        Val &v = vals[r];
        v.bits = (uint16_t)range_of(op, a, b);
        v.org_op = (uint8_t)op;
        v.org_a = a;
        v.org_b = b;
        return r;
    }

    // pattern-directed replacements; each preserves the canonical value of the result exactly
    int32_t peephole(uint32_t op, int32_t a, int32_t b) {
        if (op == CW_OP_BAND) {
            // (x >> k) & (2^m - 1)  ->  bit-field extract;  x & (2^m - 1) likewise with k = 0
            uint32_t m;
            int32_t x = -1;
            if (const_mask(b, m)) x = a;
            else if (const_mask(a, m)) x = b;
            if (x >= 0 && !is_const(x) && m < qb()) {
                uint32_t k = 0;
                uint64_t kk;
                const Val &vx = vals[x];
                if (vx.org_op == CW_OP_SHR && const_u64(vx.org_b, kk) && kk < qb() && !is_const(vx.org_a)) {
                    k = (uint32_t)kk;
                    x = vx.org_a;
                }
                int32_t r = new_val(emit(DOP_BITS, need(x, FC), NO_SLOT, k | (m << 16), true), FC);
                vals[r].fld_src = x;
                vals[r].fld_k = (uint16_t)k;
                vals[r].fld_m = (uint16_t)m;
                if (k == 0) {  // a low field is already in place
                    vals[r].bf_src = x;
                    vals[r].bf_lo = 0;
                    vals[r].bf_len = (uint16_t)m;
                }
                return r;
            }
        }
        if (op == CW_OP_ADD && a >= 0 && b >= 0) {
            // adjacent in-place fields of one source add up to the covering field (no carries)
            const Val &va = vals[a], &vb = vals[b];
            if (va.bf_src >= 0 && va.bf_src == vb.bf_src && va.cid < 0 && vb.cid < 0) {
                const Val &lo = va.bf_lo <= vb.bf_lo ? va : vb, &hi = va.bf_lo <= vb.bf_lo ? vb : va;
                if ((uint32_t)lo.bf_lo + lo.bf_len == hi.bf_lo && (uint32_t)lo.bf_lo + lo.bf_len + hi.bf_len <= 256) {
                    Val nv;
                    nv.bf_src = va.bf_src;
                    nv.bf_lo = lo.bf_lo;
                    nv.bf_len = (uint16_t)(lo.bf_len + hi.bf_len);
                    vals.push_back(nv);  // virtual: materialised by need() if anything reads it
                    return (int32_t)vals.size() - 1;
                }
            }
        }
        if (op == CW_OP_MUL) {
            // x * 2^k with x*2^k < q known statically: a shift of the canonical value
            uint32_t k;
            int32_t x = -1;
            if (const_pow2(b, k)) x = a;
            else if (const_pow2(a, k)) x = b;
            if (x >= 0 && !is_const(x) && k == 0) return x;  // x * 1
            // x * 0 (polynomial evaluations at the point 0): the constant itself
            if (a >= 0 && b >= 0 && is_const(a) != is_const(b) && is_const_zero(is_const(a) ? a : b))
                return is_const(a) ? a : b;
            if (x >= 0 && !is_const(x) && vals[x].fld_src >= 0 && vals[x].fld_k == k && k + vals[x].fld_m <= 256) {
                Val nv;  // ((src >> k) & mask) << k  ==  src & (mask << k)
                nv.bf_src = vals[x].fld_src;
                nv.bf_lo = (uint16_t)k;
                nv.bf_len = vals[x].fld_m;
                vals.push_back(nv);
                return (int32_t)vals.size() - 1;
            }
            if (x >= 0 && !is_const(x) && has(x, FC) && vbits(x) + k <= qb() - 1) {
                U256 kc = u256_from_u64(k);
                return new_val(emit(CW_OP_SHL, need(x, FC), OPERAND_CONST | raw_const(kc)), FC);
            }
            // small * small with the integer product < q: plain product, no reduction
            // (one factor may be a constant: polynomial evaluation points, limb weights)
            if (a >= 0 && b >= 0 && !(is_const(a) && is_const(b)) && (is_const(a) || has(a, FC)) &&
                (is_const(b) || has(b, FC)) && vbits(a) + vbits(b) <= qb() - 1)
                return new_val(emit(DOP_MULSMALL, need(a, FC), need(b, FC)), FC);
        }
        return -1;
    }

    // `x & (2^m - 1) === x` (the recomposition check of a bit decomposition)  ->  x < 2^m
    bool try_assert_fits(int32_t a, int32_t b, uint32_t id) {
        for (int s = 0; s < 2; ++s) {
            int32_t f = s ? b : a, x = s ? a : b;
            const Val &vf = vals[f];
            if (vf.cid < 0 && vf.bf_src == x && vf.bf_lo == 0 && !is_const(x)) {
                if (vbits(x) <= vf.bf_len) { ++n_static_asserts; return true; }
                U256 m = u256_from_u64(vf.bf_len);
                emit(DOP_ASSERT_FITS, need(x, FC), OPERAND_CONST | raw_const(m), id, true);
                return true;
            }
        }
        return false;
    }

    // `x*(x-1) === 0`  ->  one boolean assert on x
    bool try_assert_bool(int32_t a, uint32_t id) {
        const Val &va = vals[a];
        if (va.org_op != CW_OP_MUL || va.org_a < 0 || va.org_b < 0) return false;
        for (int s = 0; s < 2; ++s) {
            int32_t x = s ? va.org_b : va.org_a, y = s ? va.org_a : va.org_b;
            const Val &vy = vals[y];
            uint64_t one;
            if (vy.org_op == CW_OP_SUB && vy.org_a == x && const_u64(vy.org_b, one) && one == 1 && !is_const(x)) {
                if (vbits(x) <= 1) { ++n_static_asserts; return true; }  // x is a bit by construction: cannot fail
                Form f = has(x, FC) ? FC : FM;
                U256 o = f == FC ? u256_from_u64(1) : F.r1;
                emit(DOP_ASSERT_BOOL, need(x, f), OPERAND_CONST | raw_const(o), id, true);
                return true;
            }
        }
        return false;
    }

    int32_t lower_op_plain(uint32_t op, int32_t a, int32_t b, int32_t c, bool zero_test_only) {
        switch (op) {
            case CW_OP_ADD:
            case CW_OP_SUB: {
                Form f = common_form(a, b);
                return new_val(emit(op, need(a, f), need(b, f)), f);
            }
            case CW_OP_NEG: {
                Form f = any_form(a);
                return new_val(emit(op, need(a, f)), f);
            }
            case CW_OP_MUL: {
                if (is_const(a) || is_const(b)) {
                    int32_t k = is_const(a) ? a : b, x = is_const(a) ? b : a;
                    if (is_const(x)) return new_val(emit(op, need(k, FM), need(x, FC)), FC);
                    Form f = any_form(x);
                    return new_val(emit(op, need(x, f), need(k, FM)), f);
                }
                if (has(a, FM) && has(b, FM)) return new_val(emit(op, need(a, FM), need(b, FM)), FM);
                if (has(a, FM)) return new_val(emit(op, need(a, FM), need(b, FC)), FC);
                if (has(b, FM)) return new_val(emit(op, need(a, FC), need(b, FM)), FC);
                if (zero_test_only && has(a, FC) && has(b, FC))
                    return new_val(emit(op, need(a, FC), need(b, FC)), FD);  // x*y/R is all a zero test needs
                return new_val(emit(op, need(a, FM), need(b, FC)), FC);
            }
            case CW_OP_DIV: {
                uint32_t inv = emit(CW_OP_INV, need(b, FM));
                int32_t iv = new_val(inv, FM);
                Form f = is_const(a) ? FC : any_form(a);
                return new_val(emit(CW_OP_MUL, need(a, f), need(iv, FM)), f);
            }
            case CW_OP_POW:
                return new_val(emit(op, need(a, FM), need(b, FC)), FM);
            case CW_OP_IDIV: case CW_OP_MOD: case CW_OP_SHL: case CW_OP_SHR:
            case CW_OP_BOR: case CW_OP_BAND: case CW_OP_BXOR:
            case CW_OP_LEQ: case CW_OP_GEQ: case CW_OP_LT: case CW_OP_GT:
                return new_val(emit(op, need(a, FC), need(b, FC)), FC);
            case CW_OP_BNOT:
                return new_val(emit(op, need(a, FC)), FC);
            case CW_OP_EQ:
            case CW_OP_NEQ: {
                if (is_const_zero(b)) return new_val(emit(op, need_any(a), need(b, FC)), FC);
                if (is_const_zero(a)) return new_val(emit(op, need(a, FC), need_any(b)), FC);
                Form f = common_form(a, b);
                return new_val(emit(op, need(a, f), need(b, f)), FC);
            }
            case CW_OP_LOR:
            case CW_OP_LAND:
                return new_val(emit(op, need_any(a), need_any(b)), FC);
            case CW_OP_LNOT:
                return new_val(emit(op, need_any(a)), FC);
            case CW_OP_SELECT: {
                Form f = common_form(a, b);
                return new_val(emit(op, need(a, f), need(b, f), need_any(c)), f);
            }
            default:
                throw std::runtime_error("lowering: unsupported opcode " + std::to_string(op));
        }
    }

    // ---- symbolic execution of the component tree -------------------------------------------
    struct Comp {
        uint32_t tid;
        uint64_t start;
        uint32_t counter;
        bool ran = false;
    };

    void run(Comp &c) {
        const Tmpl &t = tm[c.tid];
        c.ran = true;
        std::vector<int32_t> tmp(t.n_tmp, -1);
        std::vector<Comp> subs(t.subs.size());
        uint64_t off = c.start + t.n_own;
        for (size_t i = 0; i < t.subs.size(); ++i) {
            const Tmpl &st = tm[t.subs[i]];
            subs[i].tid = t.subs[i];
            subs[i].start = off;
            subs[i].counter = st.n_in;
            off += st.total_signals;
            if (st.n_in == 0) run(subs[i]);
        }
        auto load = [&](uint64_t r) -> int32_t {
            int32_t v = -1;
            switch (rk(r)) {
                case K_OWN: v = sig_vid[c.start + ridx(r)]; break;
                case K_SUB: v = sig_vid[subs[rsub(r)].start + ridx(r)]; break;
                case K_CONST: v = (int32_t)ridx(r); break;  // vids [0, n_consts) are the constants
                case K_TMP: v = tmp[ridx(r)]; break;
                case K_ONE: v = vid_one; break;
                default: return -1;
            }
            if (v < 0) throw std::runtime_error("lowering: read of unassigned value in template " + t.name);
            return v;
        };
        std::vector<int32_t> argstack;
        for (const IrOp &o : t.ops) {
            ++n_ir_ops;
            if (o.op == 46 /* ARG */) {
                argstack.push_back(load(o.a));
                continue;
            }
            if (o.op == 45 /* CALL */) {
                uint32_t fid = ridx(o.a), n = ridx(o.b);
                if ((size_t)fid * 4 + 3 >= T.fn_info.size() || n != T.fn_info[fid * 4 + 3] || n > argstack.size())
                    throw std::runtime_error("lowering: bad function call in " + t.name);
                // one tape op per call; arguments are read canonical, the result is canonical
                uint32_t off = (uint32_t)pcalls.size();
                pcalls.push_back(fid);
                pcalls.push_back(n);
                uint32_t lvl = 0;
                for (uint32_t k = 0; k < n; ++k) {
                    uint32_t opnd = need(argstack[argstack.size() - n + k], FC);
                    pcalls.push_back(opnd);
                    lvl = std::max(lvl, operand_level(opnd));
                }
                argstack.resize(argstack.size() - n);
                // `var r[k] = f(..)`: ONE call, k results.  Result 0 is the CALL's own value; every further result is a
                // pseudo-op (47) that owns a slot but no tape word - the call stores it through the call table
                const uint32_t n_res = rk(o.c) == K_NONE && ridx(o.c) > 1 ? ridx(o.c) : 1;
                if (rk(o.d) != K_TMP || (uint64_t)ridx(o.d) + n_res > tmp.size() || n_res > fn_min_ret[fid])
                    throw std::runtime_error("lowering: bad call destination in " + t.name);
                uint32_t slot = emit(45, NO_SLOT, NO_SLOT, NO_SLOT, true);
                pops[pops.size() - 3] = off;  // operand `a` is the call-table offset, not a slot
                slot_level.back() = lvl + 1;
                tmp[ridx(o.d)] = new_val(slot, FC);
                pcalls.push_back(n_res - 1);
                for (uint32_t k = 1; k < n_res; ++k) {
                    uint32_t s = emit(47, slot);
                    slot_level.back() = lvl + 1;   // written by the call itself
                    pcalls.push_back(s);
                    tmp[ridx(o.d) + k] = new_val(s, FC);
                }
                continue;
            }
            if (o.op == 29 /* LOG: nothing to execute - the argument is looked up in the witness afterwards */) {
                PendingLog pl;
                pl.last = ridx(o.c) != 0;
                switch (rk(o.a)) {
                    case K_NONE: pl.kind = 0; pl.idx = ridx(o.b); break;
                    case K_OWN: pl.kind = 1; pl.idx = c.start + ridx(o.a); break;
                    case K_SUB: pl.kind = 1; pl.idx = subs[rsub(o.a)].start + ridx(o.a); break;
                    case K_ONE: pl.kind = 1; pl.idx = 0; break;
                    default: pl.kind = 2; pl.idx = ridx(o.a); break;   // K_CONST
                }
                pending_logs.push_back(pl);
                continue;
            }
            if (o.op == CW_OP_ASSERT_EQ || o.op == CW_OP_ASSERT) {
                uint32_t id = (uint32_t)n_asserts++;
                T.assert_tid.push_back(c.tid);
                T.assert_start.push_back(c.start);
                if (flags & CW_FLAG_NO_ASSERTS) continue;
                if (o.op == CW_OP_ASSERT_EQ) {
                    int32_t a = load(o.a), b = load(o.b);
                    if (!(flags & CW_FLAG_NO_PEEPHOLE) && try_assert_fits(a, b, id)) continue;
                    if (!(flags & CW_FLAG_NO_PEEPHOLE) && is_const_zero(b) && try_assert_bool(a, id)) continue;
                    if (!(flags & CW_FLAG_NO_PEEPHOLE) && is_const_zero(a) && try_assert_bool(b, id)) continue;
                    if (is_const_zero(b)) emit(CW_OP_ASSERT_EQ, need_any(a), need(b, FC), id, true);
                    else if (is_const_zero(a)) emit(CW_OP_ASSERT_EQ, need(a, FC), need_any(b), id, true);
                    else {
                        Form f = common_form(a, b);
                        emit(CW_OP_ASSERT_EQ, need(a, f), need(b, f), id, true);
                    }
                } else {
                    int32_t a = load(o.a);
                    emit(CW_OP_ASSERT, need_any(a), NO_SLOT, id, true);
                }
                continue;
            }
            int32_t v;
            if (o.op == CW_OP_COPY) {
                v = load(o.a);  // a move is an alias
            } else {
                int32_t a = load(o.a), b = rk(o.b) ? load(o.b) : -1, cc = rk(o.c) ? load(o.c) : -1;
                v = lower_op(o.op, a, b, cc, rk(o.d) == K_TMP && t.tmp_zero_only[ridx(o.d)]);
            }
            switch (rk(o.d)) {
                case K_TMP: tmp[ridx(o.d)] = v; break;
                case K_OWN: {
                    uint64_t g = c.start + ridx(o.d);
                    if (sig_vid[g] >= 0) throw std::runtime_error("lowering: signal assigned twice in " + t.name);
                    sig_vid[g] = v;
                    break;
                }
                case K_SUB: {
                    Comp &sc = subs[rsub(o.d)];
                    const Tmpl &st = tm[sc.tid];
                    uint64_t g = sc.start + ridx(o.d);
                    if (sig_vid[g] >= 0) throw std::runtime_error("lowering: signal assigned twice in " + t.name);
                    sig_vid[g] = v;
                    uint32_t li = ridx(o.d);
                    if (li >= st.n_out && li < st.n_out + st.n_in) {
                        if (--sc.counter == 0) run(sc);
                    }
                    break;
                }
                default: throw std::runtime_error("lowering: bad destination");
            }
        }
        for (Comp &sc : subs)
            if (!sc.ran) throw std::runtime_error("lowering: sub-component of " + t.name + " never received all its inputs");
    }

    void collect_constraints(uint32_t tid, uint64_t start) {
        const Tmpl &t = tm[tid];
        std::vector<uint64_t> offs(t.subs.size());
        uint64_t off = start + t.n_own;
        for (size_t i = 0; i < t.subs.size(); ++i) {
            offs[i] = off;
            off += tm[t.subs[i]].total_signals;
        }
        R1csData &R = T.r1cs;
        size_t ti = 0;
        std::vector<std::pair<uint32_t, uint32_t>> row;
        for (size_t k = 0; k < t.lc_len.size(); ++k) {
            row.clear();
            for (uint32_t j = 0; j < t.lc_len[k]; ++j, ++ti) {
                const Term &tr = t.terms[ti];
                uint64_t g;
                switch (rk(tr.ref)) {
                    case K_OWN: g = start + ridx(tr.ref); break;
                    case K_SUB: g = offs[rsub(tr.ref)] + ridx(tr.ref); break;
                    case K_ONE: g = 0; break;
                    default: throw std::runtime_error("cb2c: bad constraint reference");
                }
                row.emplace_back((uint32_t)g, tr.cid);
            }
            std::sort(row.begin(), row.end());  // wire ids ascending (r1cs_writer.rs:59-60)
            for (auto &e : row) {
                R.col.push_back(e.first);
                R.coef.push_back(e.second);
            }
            R.row_ptr.push_back(R.col.size());
        }
        for (size_t i = 0; i < t.subs.size(); ++i) collect_constraints(t.subs[i], offs[i]);
    }

    // union-find over signals for the `signal = signal` eliminations; rewrites T.r1cs into witness numbering
    void simplify_constraints(uint64_t S, uint64_t n_fixed, std::vector<uint32_t> &sig2wit) {
        R1csData &R = T.r1cs;
        std::vector<uint32_t> parent(S);
        for (uint64_t i = 0; i < S; ++i) parent[i] = (uint32_t)i;
        auto find = [&](uint32_t x) {
            while (parent[x] != x) { parent[x] = parent[parent[x]]; x = parent[x]; }
            return x;
        };
        size_t m = (R.row_ptr.size() - 1) / 3;
        if (!(flags & CW_FLAG_O0)) {
            for (size_t r = 0; r < m; ++r) {
                uint64_t a0 = R.row_ptr[3 * r], b0 = R.row_ptr[3 * r + 1], c0 = R.row_ptr[3 * r + 2], c1 = R.row_ptr[3 * r + 3];
                if (b0 != a0 || c0 != b0 || c1 - c0 != 2) continue;
                uint32_t x = R.col[c0], y = R.col[c0 + 1];
                if (x == 0 || y == 0) continue;
                const U256 &cx = R.dict[R.coef[c0]], &cy = R.dict[R.coef[c0 + 1]];
                if (cx.is_zero() || !(F.addm(cx, cy).is_zero())) continue;
                uint32_t rx = find(x), ry = find(y);
                if (rx == ry) continue;
                if (rx > ry) std::swap(rx, ry);
                if (ry < n_fixed) continue;  // both classes contain a main input/output: keep the constraint
                parent[ry] = rx;             // representative = smallest signal id
            }
        }
        sig2wit.assign(S, 0);
        T.witness2signal.clear();
        for (uint64_t i = 0; i < S; ++i)
            if (find((uint32_t)i) == i) {
                sig2wit[i] = (uint32_t)T.witness2signal.size();
                T.witness2signal.push_back(i);
            }
        for (uint64_t i = 0; i < S; ++i) sig2wit[i] = sig2wit[find((uint32_t)i)];
        // rewrite rows: map columns, merge duplicates, drop zero terms and trivial rows
        std::vector<uint64_t> row_ptr(1, 0);
        std::vector<uint32_t> col, coef;
        col.reserve(R.col.size());
        coef.reserve(R.coef.size());
        std::unordered_map<std::string, uint32_t> dict_index;
        for (size_t i = 0; i < R.dict.size(); ++i) dict_index.emplace(std::string((const char *)R.dict[i].v, 32), (uint32_t)i);
        std::vector<std::pair<uint32_t, U256>> lc[3];
        for (size_t r = 0; r < m; ++r) {
            for (int k = 0; k < 3; ++k) {
                lc[k].clear();
                for (uint64_t i = R.row_ptr[3 * r + k]; i < R.row_ptr[3 * r + k + 1]; ++i)
                    lc[k].emplace_back(sig2wit[R.col[i]], R.dict[R.coef[i]]);
                std::sort(lc[k].begin(), lc[k].end(), [](const std::pair<uint32_t, U256> &x, const std::pair<uint32_t, U256> &y) { return x.first < y.first; });
                size_t o = 0;
                for (size_t i = 0; i < lc[k].size(); ++i) {
                    if (o && lc[k][o - 1].first == lc[k][i].first) lc[k][o - 1].second = F.addm(lc[k][o - 1].second, lc[k][i].second);
                    else lc[k][o++] = lc[k][i];
                }
                lc[k].resize(o);
                o = 0;
                for (size_t i = 0; i < lc[k].size(); ++i)
                    if (!lc[k][i].second.is_zero()) lc[k][o++] = lc[k][i];
                lc[k].resize(o);
            }
            if ((lc[0].empty() || lc[1].empty()) && lc[2].empty()) continue;  // 0 = 0
            for (int k = 0; k < 3; ++k) {
                for (auto &e : lc[k]) {
                    std::string key((const char *)e.second.v, 32);
                    auto it = dict_index.find(key);
                    uint32_t id;
                    if (it == dict_index.end()) {
                        id = (uint32_t)R.dict.size();
                        R.dict.push_back(e.second);
                        dict_index.emplace(std::move(key), id);
                    } else id = it->second;
                    col.push_back(e.first);
                    coef.push_back(id);
                }
                row_ptr.push_back(col.size());
            }
        }
        R.row_ptr.swap(row_ptr);
        R.col.swap(col);
        R.coef.swap(coef);
    }

    void parse(const uint8_t *data, size_t len) {
        Reader r{data, data + len};
        if (memcmp(r.bytes(4), "CB2C", 4)) throw std::runtime_error("cb2c: bad magic");
        uint32_t version = r.get<uint32_t>();
        if (version != 1) throw std::runtime_error("cb2c: unsupported version");
        uint32_t prime = r.get<uint32_t>(), n_consts = r.get<uint32_t>(), n_tm = r.get<uint32_t>();
        main_tid = r.get<uint32_t>();
        uint32_t n_names = r.get<uint32_t>();
        uint32_t n_funcs = r.get<uint32_t>();
        if (prime >= (uint32_t)CW_N_PRIMES) throw std::runtime_error("cb2c: unknown prime");
        T.F = make_field((int)prime);
        r.expect(n_consts, 32);
        r.expect(n_tm, 36);
        ir_consts.resize(n_consts);
        for (auto &c : ir_consts) {
            memcpy(c.v, r.bytes(32), 32);
            if (!(c < T.F.q)) throw std::runtime_error("cb2c: constant not reduced");
        }
        tm.resize(n_tm);
        for (uint32_t i = 0; i < n_tm; ++i) {
            Tmpl &t = tm[i];
            t.name = r.str();
            t.n_out = r.get<uint32_t>();
            t.n_in = r.get<uint32_t>();
            t.n_inter = r.get<uint32_t>();
            uint32_t n_sub = r.get<uint32_t>();
            t.n_tmp = r.get<uint32_t>();
            uint32_t n_ops = r.get<uint32_t>(), n_cons = r.get<uint32_t>(), n_terms = r.get<uint32_t>();
            if ((uint64_t)t.n_out + t.n_in + t.n_inter > (1u << 28) || t.n_tmp > (1u << 28))
                throw std::runtime_error("cb2c: template too large");
            t.n_own = t.n_out + t.n_in + t.n_inter;
            r.expect(n_sub, 4);
            r.expect(n_ops, 40);
            r.expect((uint64_t)n_cons * 3, 8);
            r.expect(n_terms, 16);
            t.subs.resize(n_sub);
            for (auto &s : t.subs) {
                s = r.get<uint32_t>();
                if (s >= i) throw std::runtime_error("cb2c: sub-component template must precede its user");
            }
            t.ops.resize(n_ops);
            for (auto &o : t.ops) {
                o.op = (uint32_t)r.get<uint64_t>();
                o.d = r.get<uint64_t>();
                o.a = r.get<uint64_t>();
                o.b = r.get<uint64_t>();
                o.c = r.get<uint64_t>();
            }
            t.lc_len.reserve(n_cons * 3);
            t.terms.reserve(n_terms);
            for (uint32_t k = 0; k < n_cons * 3; ++k) {
                uint32_t n = (uint32_t)r.get<uint64_t>();
                t.lc_len.push_back(n);
                for (uint32_t j = 0; j < n; ++j) {
                    Term tr;
                    tr.ref = r.get<uint64_t>();
                    tr.cid = (uint32_t)r.get<uint64_t>();
                    if (tr.cid >= n_consts) throw std::runtime_error("cb2c: bad coefficient id");
                    t.terms.push_back(tr);
                }
            }
            // The description is an untrusted file: every reference must stay inside the objects it names.
            auto check_ref = [&](uint64_t ref, bool may_be_none, bool is_dst) {
                bool ok = false;
                switch (rk(ref)) {
                    case K_NONE: ok = may_be_none; break;
                    case K_OWN: ok = ridx(ref) < t.n_own; break;
                    case K_SUB:
                        ok = rsub(ref) < t.subs.size() &&
                             ridx(ref) < (uint64_t)tm[t.subs[rsub(ref)]].n_out + tm[t.subs[rsub(ref)]].n_in;
                        break;
                    case K_CONST: ok = !is_dst && ridx(ref) < n_consts; break;
                    case K_TMP: ok = ridx(ref) < t.n_tmp; break;
                    case K_ONE: ok = !is_dst; break;
                    default: break;
                }
                if (!ok) throw std::runtime_error("cb2c: reference out of range in template " + t.name);
            };
            for (const IrOp &o : t.ops) {
                if (o.op == 46 /* ARG */) {
                    check_ref(o.a, false, false);
                } else if (o.op == 45 /* CALL */) {
                    if (rk(o.d) != K_TMP) throw std::runtime_error("cb2c: bad call destination in template " + t.name);
                    check_ref(o.d, false, true);
                    if (rk(o.c) == K_NONE && ridx(o.c) > 1 && (ridx(o.c) > 64 || (uint64_t)ridx(o.d) + ridx(o.c) > t.n_tmp))
                        throw std::runtime_error("cb2c: bad result count of a call in template " + t.name);
                } else if (o.op == 29 /* LOG */) {
                    const int k = rk(o.a);
                    if (k == K_TMP || rk(o.d) != K_NONE || rk(o.b) != K_NONE || rk(o.c) != K_NONE || ridx(o.c) > 1)
                        throw std::runtime_error("cb2c: bad log argument in template " + t.name + " (a signal, a constant or a string)");
                    check_ref(o.a, true, false);
                    if (k == K_NONE) max_log_string = std::max<int64_t>(max_log_string, (int64_t)ridx(o.b));
                } else {
                    if (o.op < CW_OP_MUL || o.op > CW_OP_INV) throw std::runtime_error("cb2c: unknown opcode in template " + t.name);
                    const bool is_assert = o.op == CW_OP_ASSERT || o.op == CW_OP_ASSERT_EQ;
                    int arity = 2;
                    switch (o.op) {
                        case CW_OP_NEG: case CW_OP_LNOT: case CW_OP_BNOT: case CW_OP_COPY: case CW_OP_INV: case CW_OP_ASSERT:
                            arity = 1;
                            break;
                        case CW_OP_SELECT: arity = 3; break;
                        default: break;
                    }
                    check_ref(o.d, is_assert, true);
                    check_ref(o.a, false, false);
                    check_ref(o.b, arity < 2, false);
                    check_ref(o.c, arity < 3, false);
                }
            }
            for (const Term &tr : t.terms) {
                const int k = rk(tr.ref);
                if (k != K_OWN && k != K_SUB && k != K_ONE) throw std::runtime_error("cb2c: bad constraint reference");
                check_ref(tr.ref, false, false);
            }
            // which temporaries feed only zero / non-zero tests (so a raw product x*y/R suffices)
            t.tmp_zero_only.assign(t.n_tmp, 1);
            auto is_zero_const = [&](uint64_t r) { return rk(r) == K_CONST && ridx(r) < n_consts && ir_consts[ridx(r)].is_zero(); };
            auto mark = [&](uint64_t r, bool zero_use) {
                if (rk(r) == K_TMP && ridx(r) < t.n_tmp && !zero_use) t.tmp_zero_only[ridx(r)] = 0;
            };
            for (const IrOp &o : t.ops) {
                switch (o.op) {
                    case CW_OP_ASSERT: case CW_OP_LNOT: case CW_OP_LAND: case CW_OP_LOR:
                        break;  // every operand is only tested for zero
                    case CW_OP_SELECT:
                        mark(o.a, false); mark(o.b, false);
                        break;
                    case CW_OP_ASSERT_EQ: case CW_OP_EQ: case CW_OP_NEQ:
                        mark(o.a, is_zero_const(o.b)); mark(o.b, is_zero_const(o.a));
                        break;
                    default:
                        mark(o.a, false); mark(o.b, false); mark(o.c, false);
                }
            }
            t.total_signals = t.n_own;
            t.total_components = 1;
            for (auto s : t.subs) {
                t.total_signals += tm[s].total_signals;
                t.total_components += tm[s].total_components;
                // a few nested templates can describe an astronomically large tree: stop before instantiating it
                if (t.total_signals > (1ull << 28) || t.total_components > (1ull << 26))
                    throw std::runtime_error("cb2c: circuit too large (more than 2^28 signals or 2^26 components)");
            }
        }
        if (main_tid >= n_tm) throw std::runtime_error("cb2c: bad main template");
        {
            // main-input name table: every name covers a run of the main component's input signals
            // (signal ids 1 + n_out ... n_out + n_in), no two names overlap
            const Tmpl &M = tm[main_tid];
            const uint64_t in_lo = 1 + (uint64_t)M.n_out, in_hi = in_lo + M.n_in;
            std::vector<uint8_t> covered(M.n_in, 0);
            for (uint32_t i = 0; i < n_names; ++i) {
                InputInfo in;
                in.name = r.str();
                in.signal_id = r.get<uint32_t>();
                in.size = r.get<uint32_t>();
                if (in.size < 1 || in.signal_id < in_lo || in.signal_id + in.size > in_hi)
                    throw std::runtime_error("cb2c: input name '" + in.name + "' lies outside the main inputs");
                for (uint64_t k = in.signal_id - in_lo; k < in.signal_id - in_lo + in.size; ++k)
                    if (covered[k]++) throw std::runtime_error("cb2c: input names overlap at '" + in.name + "'");
                in.hash = fnv1a(in.name.data(), in.name.size());
                T.inputs.push_back(in);
            }
        }
        // function bodies -> device register-machine code (fr_device.cuh: vm_run).  Untrusted like everything else
        // in the file: every register, array base, jump target and opcode is checked here, the interpreter then
        // only bounds-checks run-time indices.
        for (uint32_t i = 0; i < n_funcs; ++i) {
            r.str();
            uint32_t n_params = r.get<uint32_t>(), n_regs = r.get<uint32_t>(), n_instr = r.get<uint32_t>();
            if (n_regs > 192 || n_params > n_regs) throw std::runtime_error("cb2c: function needs too many registers");
            r.expect(n_instr, 40);
            T.fn_info.push_back((uint32_t)(T.fn_code.size() / 5));
            T.fn_info.push_back(n_instr);
            T.fn_info.push_back(n_regs);
            T.fn_info.push_back(n_params);
            uint32_t min_ret = 0xFFFFFFFFu;
            std::vector<uint32_t> callees;
            auto bad = [&](const char *what) { throw std::runtime_error(std::string("cb2c: function body: ") + what); };
            auto reg = [&](uint64_t w) -> uint32_t {   // a register
                if (rk(w) != K_TMP || ridx(w) >= n_regs) bad("bad register");
                return ridx(w);
            };
            auto val = [&](uint64_t w, bool may_be_none) -> uint32_t {   // a value operand: register, constant, or unused
                if (rk(w) == K_TMP) return reg(w);
                if (rk(w) == K_CONST) {
                    if (ridx(w) >= n_consts) bad("bad constant");
                    return OPERAND_CONST | raw_const(ir_consts[ridx(w)]);  // canonical
                }
                if (rk(w) != K_NONE || !may_be_none) bad("bad operand");
                return 0x40000000u;  // unused: the immediate 0
            };
            auto imm = [&](uint64_t w, uint32_t limit) -> uint32_t {     // an immediate below `limit`
                if (rk(w) != K_NONE || ridx(w) >= limit) bad("immediate out of range");
                return 0x40000000u | ridx(w);
            };
            for (uint32_t k = 0; k < n_instr; ++k) {
                uint64_t w[5];
                for (auto &x : w) x = r.get<uint64_t>();
                uint32_t op = (uint32_t)w[0], e[4] = {0x40000000u, 0x40000000u, 0x40000000u, 0x40000000u};
                if (w[0] >> 32) bad("unknown opcode");
                switch (op) {
                    case 40 /* JMP */: e[1] = imm(w[2], n_instr); break;
                    case 41 /* JZ */: e[1] = val(w[2], false); e[2] = imm(w[3], n_instr); break;
                    case 42 /* RET: a value, or (operand b = count > 1) `count` consecutive registers from register a */: {
                        e[1] = val(w[2], false);
                        const uint32_t cnt = rk(w[3]) == K_NONE && ridx(w[3]) > 1 ? ridx(w[3]) : 1;
                        if (cnt > 1 && (rk(w[2]) != K_TMP || cnt > 64 || (uint64_t)ridx(w[2]) + cnt > n_regs)) bad("bad array return");
                        e[2] = 0x40000000u | cnt;
                        min_ret = std::min(min_ret, cnt);
                        break;
                    }
                    // run-time indexed `var` arrays.  The producer may state the extent of the array behind the base (LOADX:
                    // operand c, STOREX: operand d; 0 / NONE = unknown, then up to the last register); the encoded word is the
                    // exclusive upper limit of the register index, checked by the interpreter at run time.
                    case 43 /* LOADX: d = regs[base + b] */: {
                        e[0] = reg(w[1]); e[1] = imm(w[2], n_regs); e[2] = val(w[3], false);
                        const uint32_t base = ridx(w[2]), ext = rk(w[4]) == K_NONE ? ridx(w[4]) : 0;
                        if (rk(w[4]) != K_NONE || (uint64_t)base + ext > n_regs) bad("bad array extent");
                        e[3] = 0x40000000u | (ext ? base + ext : n_regs);
                        break;
                    }
                    case 44 /* STOREX: regs[base + b] = c */: {
                        e[1] = imm(w[2], n_regs); e[2] = val(w[3], false); e[3] = val(w[4], false);
                        const uint32_t base = ridx(w[2]), ext = rk(w[1]) == K_NONE ? ridx(w[1]) : 0;
                        if (rk(w[1]) != K_NONE || (uint64_t)base + ext > n_regs) bad("bad array extent");
                        e[0] = 0x40000000u | (ext ? base + ext : n_regs);
                        break;
                    }
                    case 45 /* CALL of an earlier function: d <- f(registers b .. b + n_params - 1); c = result count */: {
                        if (rk(w[2]) != K_NONE || ridx(w[2]) >= i) bad("a function may only call functions with a smaller index");
                        const uint32_t f = ridx(w[2]), np = T.fn_info[4 * (size_t)f + 3];
                        const uint32_t want = rk(w[4]) == K_NONE && ridx(w[4]) > 1 ? ridx(w[4]) : 1;
                        if (rk(w[4]) != K_NONE || want > 64 || want > fn_min_ret[f]) bad("bad result count of a call");
                        e[0] = reg(w[1]);
                        if ((uint64_t)e[0] + want > n_regs) bad("call results run past the registers");
                        if (np) {
                            if (rk(w[3]) != K_TMP || (uint64_t)ridx(w[3]) + np > n_regs) bad("bad argument registers of a call");
                            e[2] = ridx(w[3]);
                        } else e[2] = 0;
                        e[1] = 0x40000000u | f;
                        e[3] = 0x40000000u | want;
                        callees.push_back(f);
                        break;
                    }
                    default:
                        if (op < CW_OP_MUL || op > CW_OP_INV || op == CW_OP_ASSERT || op == CW_OP_ASSERT_EQ) bad("unknown opcode");
                        e[0] = reg(w[1]);
                        e[1] = val(w[2], false);
                        e[2] = val(w[3], true);
                        e[3] = val(w[4], true);
                }
                T.fn_code.push_back(op);
                for (uint32_t x : e) T.fn_code.push_back(x);
            }
            fn_min_ret.push_back(min_ret == 0xFFFFFFFFu ? 1 : min_ret);
            if (!(flags & CW_FLAG_NO_PEEPHOLE)) {
                uint32_t *body = &T.fn_code[5 * (size_t)T.fn_info[4 * (size_t)i]];
                std::vector<uint32_t> fn_params;   // parameters of the functions defined so far (callees)
                for (size_t f = 0; f + 1 <= (size_t)i; ++f) fn_params.push_back(T.fn_info[4 * f + 3]);
                const uint32_t kept = coalesce_function_copies(body, n_instr, n_regs, fn_params);
                T.fn_code.resize(5 * ((size_t)T.fn_info[4 * (size_t)i] + kept));   // (this function's code is the tail of fn_code)
                T.fn_info[4 * (size_t)i + 1] = kept;
                uint32_t packed = n_regs;
                allocate_function_registers(&T.fn_code[5 * (size_t)T.fn_info[4 * (size_t)i]], kept, n_params, packed, fn_params);
                T.fn_info[4 * (size_t)i + 2] = packed;
            }
            // the deepest chain of nested calls below this function: registers and frames the interpreter needs
            uint32_t below_regs = 0, below_depth = 0;
            for (uint32_t f : callees) {
                below_regs = std::max(below_regs, fn_stack_regs[f]);
                below_depth = std::max(below_depth, fn_stack_depth[f]);
            }
            fn_stack_regs.push_back(T.fn_info[4 * (size_t)i + 2] + below_regs);
            fn_stack_depth.push_back(1 + below_depth);
            if (fn_stack_regs.back() > 192 || fn_stack_depth.back() > 9)   // (VM_MAX_REGS, VM_MAX_DEPTH + 1 of fr_device.cuh)
                throw std::runtime_error("cb2c: nested function calls need too many registers / frames");
        }
        // optional symbols section: "SYMS", then per template the names of its own signals and of its sub-components
        // (what the reference keeps in the DAG for sym_porting.rs).  Anything else after the functions is refused.
        // optional io-map section: "IOMP" - the compiler's TemplateInstanceIOMap (code_producers/src/components/mod.rs:4-10,47:
        // per template instance that sits in a component array of mixed templates, the list of its input / output
        // signals with offset, dimensions, element size, bus id).  The reference's generated code resolves `Mapped`
        // locations through it at run time (load_bucket.rs:264-322); here a producer has resolved them already, the map is
        // carried for the `.dat` only (c_code_generator.rs:681-735).
        // optional string table of log(): "LOGS", u32 count, count x str (printable ASCII without % \ ": the reference pastes the
        // text into a printf format, log_bucket.rs:128-137)
        if (r.left() >= 4 && !memcmp(r.p, "LOGS", 4)) {
            r.bytes(4);
            const uint32_t n_s = r.get<uint32_t>();
            r.expect(n_s, 4);
            for (uint32_t i = 0; i < n_s; ++i) {
                std::string x = r.str();
                if (x.empty() || x.size() > 4096) throw std::runtime_error("cb2c: bad log string");
                for (unsigned char ch : x)
                    if (ch < 0x20 || ch >= 0x7F || ch == '%' || ch == '\\' || ch == '"') throw std::runtime_error("cb2c: bad character in a log string");
                T.log_strings.push_back(std::move(x));
            }
        }
        if (max_log_string >= (int64_t)T.log_strings.size()) throw std::runtime_error("cb2c: log() names a string the file does not carry");
        if (r.left() >= 4 && !memcmp(r.p, "IOMP", 4)) {
            r.bytes(4);
            const uint32_t n_e = r.get<uint32_t>();
            if (n_e > n_tm) throw std::runtime_error("cb2c: io map names more templates than the file has");
            int64_t prev = -1;
            for (uint32_t e = 0; e < n_e; ++e) {
                const uint32_t tid = r.get<uint32_t>(), n_defs = r.get<uint32_t>();
                if (tid >= n_tm || (int64_t)tid <= prev) throw std::runtime_error("cb2c: io map entries must name templates in ascending order");
                prev = tid;
                const uint64_t n_io = (uint64_t)tm[tid].n_out + tm[tid].n_in;
                if (n_defs > n_io) throw std::runtime_error("cb2c: io map lists more signals than the template has inputs and outputs");
                std::vector<Tape::IoDef> defs(n_defs);
                for (Tape::IoDef &d : defs) {
                    d.offset = r.get<uint32_t>();
                    const uint32_t nl = r.get<uint32_t>();
                    if (nl > 32) throw std::runtime_error("cb2c: io map signal with more than 32 dimensions");
                    r.expect(nl, 4);
                    uint64_t elems = 1;
                    for (uint32_t k = 0; k < nl; ++k) {
                        d.lengths.push_back(r.get<uint32_t>());
                        elems *= d.lengths.back();
                        if (elems > n_io) throw std::runtime_error("cb2c: io map signal larger than its template");
                    }
                    d.size = r.get<uint32_t>();
                    d.bus_id = r.get<uint32_t>();
                    if (d.size < 1 || (uint64_t)d.offset + elems * d.size > n_io) throw std::runtime_error("cb2c: io map signal outside its template's inputs and outputs");
                }
                T.io_map.emplace_back(tid, std::move(defs));
            }
        }
        if (r.left()) {
            if (r.left() < 4 || memcmp(r.bytes(4), "SYMS", 4)) throw std::runtime_error("cb2c: unknown section after the functions");
            T.sym.resize(n_tm);
            auto name = [&]() {
                std::string s = r.str();
                if (s.empty() || s.size() > 4096) throw std::runtime_error("cb2c: bad symbol name");
                for (unsigned char ch : s)
                    if (ch < 0x21 || ch == ',' || ch == 0x7F) throw std::runtime_error("cb2c: bad character in a symbol name");
                return s;
            };
            for (uint32_t i = 0; i < n_tm; ++i) {
                Tape::SymTemplate &st = T.sym[i];
                st.n_own = tm[i].n_own;
                st.total_signals = tm[i].total_signals;
                st.subs = tm[i].subs;
                r.expect((uint64_t)st.n_own + st.subs.size(), 4);
                st.own.resize(st.n_own);
                for (auto &n : st.own) n = name();
                st.sub.resize(st.subs.size());
                for (auto &n : st.sub) n = name();
            }
            if (r.left()) throw std::runtime_error("cb2c: bytes after the symbols section");
            T.sym_main = main_tid;
        }
    }
    uint32_t main_tid = 0;

    void lower() {
        const Tmpl &M = tm[main_tid];
        uint64_t S = 1 + M.total_signals;
        if (S >= 0x7FFFFFFFull) throw std::runtime_error("circuit too large");
        T.n_signals = S;
        T.n_inputs = M.n_in;
        T.n_outputs = M.n_out;
        T.n_components = M.total_components;
        n_pre = 1 + M.n_in;
        // constants are vids [0, n_consts)
        vals.resize(ir_consts.size());
        for (size_t i = 0; i < ir_consts.size(); ++i) {
            vals[i].cid = (int32_t)i;
            vals[i].bits = (uint16_t)u256_bitlen(ir_consts[i]);
        }
        sig_vid.assign(S, -1);
        slot_level.assign(n_pre, 0);
        vid_one = new_val(0, FC);  // slot 0: the constant-one signal (calcwit.cpp:34)
        vals[vid_one].bits = 1;
        sig_vid[0] = vid_one;
        for (uint32_t i = 0; i < M.n_in; ++i) sig_vid[1 + M.n_out + i] = new_val(1 + i, FC);
        Comp mc;
        mc.tid = main_tid;
        mc.start = 1;
        mc.counter = 0;
        run(mc);

        // R1CS rows in signal numbering (component pre-order), then the witness list:
        //   --O0 : every signal, in signal order (dag/src/witness_producer.rs:3-19)
        //   default (the reference's --O1 core): constraints `c*x - c*y = 0` between two signals are
        //   removed by merging the signals (constraint_list/src/constraint_simplification.rs "signal = signal"
        //   eliminations); the witness keeps one representative per class, main inputs/outputs always stay.
        R1csData &R = T.r1cs;
        R.prime_id = F.prime_id;
        R.row_ptr.push_back(0);
        R.dict = ir_consts;
        collect_constraints(main_tid, 1);
        std::vector<uint32_t> sig2wit;
        simplify_constraints(S, 1 + M.n_out + M.n_in, sig2wit);
        uint64_t W = T.witness2signal.size();
        T.n_witness = W;
        R.n_wires = W;
        R.n_constraints = (R.row_ptr.size() - 1) / 3;
        R.n_pub_out = (uint32_t)M.n_out;
        R.n_pub_in = 0;
        R.n_prv_in = (uint32_t)M.n_in;
        // ---- witness values live IN the slot store: slot i (i < W) is witness entry i, canonical ---------
        // Each witness entry claims the slot of the op that produces its canonical value (so the tape
        // writes the witness rows directly and no gather pass exists); a second entry with the same
        // value, or a value only held in another representation, costs one move / conversion op.
        for (uint64_t i = 0; i < S; ++i)
            if (sig_vid[i] < 0) throw std::runtime_error("lowering: signal " + std::to_string(i) + " is never assigned");
        if (!pending_logs.empty()) {   // logged signals -> the witness entries that hold their values
            std::unordered_map<int32_t, uint32_t> entry_of_value;
            for (uint64_t i = 0; i < W; ++i) entry_of_value.emplace(sig_vid[T.witness2signal[i]], (uint32_t)i);
            std::unordered_map<std::string, uint32_t> const_at;
            auto log_const = [&](const U256 &v) {
                std::string key((const char *)v.v, 32);
                auto it = const_at.find(key);
                if (it != const_at.end()) return it->second;
                T.log_consts.push_back(v);
                return const_at.emplace(std::move(key), (uint32_t)T.log_consts.size() - 1).first->second;
            };
            for (const PendingLog &pl : pending_logs) {
                Tape::LogArg a;
                a.kind = pl.kind;
                a.last = pl.last ? 1 : 0;
                a.idx = (uint32_t)pl.idx;
                if (pl.kind == 2) a.idx = log_const(ir_consts[pl.idx]);
                if (pl.kind == 1) {
                    const int32_t v = sig_vid[pl.idx];
                    auto it = entry_of_value.find(v);
                    if (it != entry_of_value.end()) a.idx = it->second;
                    else if (vals[v].cid >= 0) { a.kind = 2; a.idx = log_const(ir_consts[vals[v].cid]); }
                    else throw std::runtime_error("lowering: log() of a signal whose value is not part of the witness");
                }
                T.log_args.push_back(a);
            }
        }
        std::vector<int64_t> claimed;  // provisional slot -> witness index
        std::vector<uint32_t> wsrc(W);
        auto grow = [&]() { claimed.resize(n_pre + pops.size() / 4, -1); };
        grow();
        for (uint64_t i = 0; i < W; ++i) {
            int32_t v = sig_vid[T.witness2signal[i]];
            uint32_t src;
            if (vals[v].cid >= 0) src = emit(CW_OP_COPY, const_operand(vals[v].cid, FC));  // constant signal
            else src = need(v, FC);
            grow();
            if (claimed[src] >= 0) {  // value already is another witness entry: one move
                src = emit(CW_OP_COPY, src);
                grow();
            }
            claimed[src] = (int64_t)i;
            wsrc[i] = src;
            // static size class of the entry (range analysis): 1 bit / <= 64 bits / full.  Used only to pack
            // the device->host transfer of witnesses; the pack kernel re-checks every value at run time.
            uint32_t wb = vbits(v);
            T.wit_bits.push_back((uint16_t)std::min<uint32_t>(wb, 256));
            if (wb <= 1) { T.pk_bit_wire.push_back((uint32_t)i); T.wit_class.push_back(0); }
            else if (wb <= 64) { T.pk_u64_wire.push_back((uint32_t)i); T.wit_class.push_back(1); }
            else { T.pk_full_wire.push_back((uint32_t)i); T.wit_class.push_back(2); }
        }
        size_t n_prov = pops.size() / 4;
        // static width of every provisional slot (range analysis; Montgomery / deferred images are full width)
        std::vector<uint16_t> slot_bits(n_pre + n_prov, 256);
        for (const Val &v : vals)
            if (v.cid < 0 && v.slot[FC] != NO_SLOT && v.slot[FC] < slot_bits.size())
                slot_bits[v.slot[FC]] = std::min<uint16_t>(slot_bits[v.slot[FC]], v.bits);
        // ---- width-typed operators ------------------------------------------------------------------------------
        // Where the range analysis proves an operator's canonical result narrow, the generic operator does work that
        // cannot change the result: the modular correction of an addition below q, the limbs of an integer product
        // above its width, the decoding of a constant shift amount (a 256-bit compare with q) and the reduction of a
        // left shift below q.  Those operators become typed ones whose opcode says what is known (fr_device.cuh); the
        // operands stay as they are.  Only the operators' own range analysis (Val::bits) is trusted here, not the
        // widths of witness entries, which the circuit's constraints state but a failing instance may break.
        if (!(flags & CW_FLAG_NO_TYPED)) {
            const uint32_t lim = qb() - 1;
            auto const_amount = [&](uint32_t o) {   // a constant operand below qbits
                if (o == NO_SLOT || !(o & OPERAND_CONST)) return false;
                const U256 &c = consts[o & ~OPERAND_CONST];
                return !(c.v[1] | c.v[2] | c.v[3]) && c.v[0] < qb();
            };
            for (size_t i = 0; i < n_prov; ++i) {
                uint32_t *o = &pops[i * 4];
                const uint32_t bits = slot_bits[n_pre + i];
                if (o[0] == CW_OP_ADD && bits <= lim) o[0] = bits <= 128 ? DOP_ADD128 : DOP_ADD_NR;
                else if (o[0] == DOP_MULSMALL && bits <= 192) o[0] = bits <= 128 ? DOP_MULSMALL128 : DOP_MULSMALL192;
                else if (o[0] == CW_OP_SHR && const_amount(o[2])) o[0] = DOP_SHRI;
                else if (o[0] == CW_OP_SHL && bits <= lim && const_amount(o[2])) o[0] = DOP_SHLI;
            }
        }
        for (uint64_t i = 0; i < W; ++i) {  // copies made for the witness carry their entry's width
            uint32_t wb = vbits(sig_vid[T.witness2signal[i]]);
            slot_bits[wsrc[i]] = std::min<uint16_t>(slot_bits[wsrc[i]], (uint16_t)wb);
        }
        std::vector<uint8_t> live(n_pre + n_prov, 0);
        for (uint64_t i = 0; i < W; ++i) live[wsrc[i]] = 1;
        // dead-value elimination (reverse sweep; provisional order is topological)
        for (size_t i = n_prov; i-- > 0;) {
            uint32_t *o = &pops[i * 4];
            bool is_assert = is_assert_op(o[0]);
            if (!is_assert && !live[n_pre + i]) continue;
            live[n_pre + i] = 1;
            if (o[0] == 45) {  // CALL: operands live in the call table
                uint32_t n = pcalls[o[1] + 1];
                for (uint32_t k = 0; k < n; ++k) {
                    uint32_t a = pcalls[o[1] + 2 + k];
                    if (!(a & OPERAND_CONST)) live[a] = 1;
                }
                continue;
            }
            for (int k = 1; k <= 3; ++k) {
                if (k == 3 && c_is_immediate(o[0])) break;
                if (o[k] != NO_SLOT && !(o[k] & OPERAND_CONST)) live[o[k]] = 1;
            }
        }
        // ---- op fusion ---------------------------------------------------------------------------------------
        // 70 % of the values of circom programs are read exactly once, by the next operation of the same
        // expression (`acc + a[i]*b[j]`, `(s >> 64) - OFF`, the trees of `+` the DSL builds).  Writing each of them
        // to the value store and reading it back costs two memory round trips and a level of the DAG per operator.
        // A value with ONE reader that is not a witness entry is therefore *fused* into its reader: the work item of
        // the reader first evaluates the producer(s) into one of two accumulator registers.  Trees are evaluated in
        // post order with at most two live accumulators (deeper sub-tree first; a second fused operand may only be a
        // chain), at most FUSE_MAX operators per work item.  The DAG gets shallower (levels are recomputed over the
        // groups) and narrower in memory traffic; each group still writes exactly one value (its root's).
        constexpr uint32_t FUSE_MAX = 24;
        std::vector<uint8_t> fusedf(n_prov, 0);          // op is evaluated inside its reader's work item
        std::vector<uint32_t> kid_a(n_prov, NO_SLOT), kid_b(n_prov, NO_SLOT);  // fused producers of operands a / b (op index)
        {
            std::vector<uint32_t> uses(n_pre + n_prov, 0), cons(n_pre + n_prov, NO_SLOT);
            std::vector<uint8_t> cons_pos(n_pre + n_prov, 0);
            for (size_t i = 0; i < n_prov; ++i) {
                if (!live[n_pre + i]) continue;
                const uint32_t *o = &pops[i * 4];
                if (o[0] == 45) {
                    uint32_t n = pcalls[o[1] + 1];
                    for (uint32_t k = 0; k < n; ++k) {
                        uint32_t x = pcalls[o[1] + 2 + k];
                        if (!(x & OPERAND_CONST)) uses[x] += 2;  // call arguments are read through the call table
                    }
                    continue;
                }
                for (int k = 1; k <= 3; ++k) {
                    if (k == 3 && c_is_immediate(o[0])) break;
                    if (o[k] == NO_SLOT || (o[k] & OPERAND_CONST)) continue;
                    ++uses[o[k]];
                    cons[o[k]] = (uint32_t)i;
                    cons_pos[o[k]] = (uint8_t)k;
                }
            }
            std::vector<uint8_t> need(n_prov, 1);
            std::vector<uint32_t> gsize(n_prov, 1);
            // (tapes with function calls keep one operator per work item: with the function machine in the build the fused
            // interpreter spills - measured 169.7 ms against 153.6 ms per 18,944 instances of the bench circuit with hints
            // computed by functions)
            const bool fuse_on = (flags & CW_FLAG_FUSE) && !(flags & CW_FLAG_NO_PEEPHOLE) && pcalls.empty();
            auto candidate = [&](uint32_t slot, size_t reader, int pos) -> bool {
                if (!fuse_on || slot == NO_SLOT || (slot & OPERAND_CONST) || slot < n_pre) return false;
                const size_t c = slot - n_pre;
                const uint32_t opc = pops[c * 4];
                if (uses[slot] != 1 || cons[slot] != reader || cons_pos[slot] != pos || claimed[slot] >= 0) return false;
                if (is_assert_op(opc) || opc == 45 || opc == 47 || opc == DOP_BITS || opc == CW_OP_COPY) return false;
                if (opc == CW_OP_INV || opc == CW_OP_POW) return false;   // (run in a pass of their own: items of one word)
                return true;
            };
            for (size_t i = 0; i < n_prov; ++i) {
                if (!live[n_pre + i]) continue;
                const uint32_t *o = &pops[i * 4];
                if (o[0] == 45 || o[0] == 47 || o[0] == CW_OP_INV || o[0] == CW_OP_POW) continue;
                uint32_t ka = candidate(o[1], i, 1) ? o[1] - n_pre : NO_SLOT;
                uint32_t kb = candidate(o[2], i, 2) ? o[2] - n_pre : NO_SLOT;
                if (ka != NO_SLOT && kb != NO_SLOT) {
                    // two fused operands: the shallower one must be a chain (one accumulator)
                    uint32_t deep = need[ka] >= need[kb] ? ka : kb, other = deep == ka ? kb : ka;
                    if (need[other] > 1 || gsize[ka] + gsize[kb] + 1 > FUSE_MAX) {
                        // keep the larger tree, give the other its own work item
                        uint32_t drop = gsize[ka] >= gsize[kb] ? kb : ka;
                        if (need[other] > 1) drop = other;
                        if (drop == ka) ka = NO_SLOT; else kb = NO_SLOT;
                    }
                }
                if (ka != NO_SLOT && kb == NO_SLOT && gsize[ka] + 1 > FUSE_MAX) ka = NO_SLOT;
                if (kb != NO_SLOT && ka == NO_SLOT && gsize[kb] + 1 > FUSE_MAX) kb = NO_SLOT;
                kid_a[i] = ka;
                kid_b[i] = kb;
                uint32_t sz = 1;
                uint8_t nd = 1;
                if (ka != NO_SLOT && kb != NO_SLOT) {
                    sz += gsize[ka] + gsize[kb];
                    nd = (uint8_t)std::max<int>(std::max(need[ka], need[kb]), std::min(need[ka], need[kb]) + 1);
                } else if (ka != NO_SLOT) { sz += gsize[ka]; nd = need[ka]; }
                else if (kb != NO_SLOT) { sz += gsize[kb]; nd = need[kb]; }
                gsize[i] = sz;
                need[i] = nd;
                if (ka != NO_SLOT) fusedf[ka] = 1;
                if (kb != NO_SLOT) fusedf[kb] = 1;
            }
        }
        // levels over the groups (a group reads the external operands of all its operators, writes its root's value)
        std::vector<uint32_t> glevel(n_pre + n_prov, 0);  // per provisional slot: level of the group that writes it
        std::vector<uint64_t> gsig(n_prov, 0);            // structure of the group's tree (orders similar work items together)
        uint32_t max_level = 0;
        size_t n_roots = 0;
        {
            std::vector<uint32_t> ext(n_prov, 0);  // highest level among the external operands of the sub-tree
            for (size_t i = 0; i < n_prov; ++i) {
                if (!live[n_pre + i]) continue;
                const uint32_t *o = &pops[i * 4];
                uint32_t e = 0;
                uint64_t sg = 1469598103934665603ull ^ o[0];
                if (o[0] == 47) {  // a further result of a call: written by the call's work item
                    glevel[n_pre + i] = glevel[o[1]];
                    continue;
                }
                if (o[0] == 45) {
                    uint32_t n = pcalls[o[1] + 1];
                    for (uint32_t k = 0; k < n; ++k) {
                        uint32_t x = pcalls[o[1] + 2 + k];
                        if (!(x & OPERAND_CONST)) e = std::max(e, glevel[x]);
                    }
                } else {
                    for (int k = 1; k <= 3; ++k) {
                        if (k == 3 && c_is_immediate(o[0])) break;
                        if (o[k] == NO_SLOT || (o[k] & OPERAND_CONST)) continue;
                        const uint32_t kid = k == 1 ? kid_a[i] : k == 2 ? kid_b[i] : NO_SLOT;
                        if (kid != NO_SLOT) {
                            e = std::max(e, ext[kid]);
                            sg = (sg * 1099511628211ull) ^ gsig[kid] ^ (uint64_t)k;
                        } else e = std::max(e, glevel[o[k]]);
                    }
                }
                ext[i] = e;
                gsig[i] = sg * 1099511628211ull;
                if (!fusedf[i]) {
                    glevel[n_pre + i] = e + 1;
                    max_level = std::max(max_level, e + 1);
                    ++n_roots;
                }
            }
        }
        // work items = group roots, sorted by (level, root opcode, tree structure)
        std::vector<uint32_t> order;
        order.reserve(n_roots);
        for (size_t i = 0; i < n_prov; ++i)
            if (live[n_pre + i] && !fusedf[i] && pops[i * 4] != 47) order.push_back((uint32_t)i);
        std::stable_sort(order.begin(), order.end(), [&](uint32_t x, uint32_t y) {
            uint32_t lx = glevel[n_pre + x], ly = glevel[n_pre + y];
            if (lx != ly) return lx < ly;
            if (pops[x * 4] != pops[y * 4]) return pops[x * 4] < pops[y * 4];
            return gsig[x] < gsig[y];
        });
        // final slots: witness entries first (slot = witness index), other values after them in tape order
        std::vector<uint32_t> remap(n_pre + n_prov, NO_SLOT);
        uint32_t next_tmp = (uint32_t)W;
        for (uint32_t i = 0; i < n_pre; ++i) {
            if (claimed[i] < 0) throw std::runtime_error("lowering: main input outside the witness");
            remap[i] = (uint32_t)claimed[i];
        }
        for (size_t r = 0; r < order.size(); ++r) {
            uint32_t p = n_pre + order[r];
            if (claimed[p] >= 0) remap[p] = (uint32_t)claimed[p];
            else if (!is_assert_op(pops[(size_t)order[r] * 4])) remap[p] = next_tmp++;
            if (pops[(size_t)order[r] * 4] == 45) {  // the further results of a call follow its first one
                const uint32_t *ct = &pcalls[pops[(size_t)order[r] * 4 + 1]];
                const uint32_t *ex = ct + 2 + ct[1];
                for (uint32_t k = 0; k < ex[0]; ++k) {
                    const uint32_t s = ex[1 + k];
                    if (!live[s]) continue;
                    remap[s] = claimed[s] >= 0 ? (uint32_t)claimed[s] : next_tmp++;
                }
            }
        }
        if (next_tmp >= DST_ACC) throw std::runtime_error("circuit too large for the packed tape word (2^24 slots)");
        T.ops.clear();
        T.ops.reserve(n_live_ops(live, n_pre, n_prov) * 4);
        T.items.clear();
        T.items.reserve(n_roots + 1);
        T.level_start.assign(max_level + 1, 0);
        T.n_mul_ops = 0;
        uint32_t prev_level = 0;
        // one operator as a tape word; operands that are fused producers read an accumulator
        auto word = [&](uint32_t i, uint32_t dstfield, int acc_a, int acc_b, uint32_t d[4]) {
            const uint32_t *o = &pops[(size_t)i * 4];
            d[0] = o[0] | (dstfield << 8);  // opcode in bits 0-7, destination in bits 8-31
            if (o[0] == 45) {
                uint32_t n = pcalls[o[1] + 1];
                d[1] = (uint32_t)T.call_tab.size();
                d[2] = d[3] = OPERAND_CONST;
                T.call_tab.push_back(pcalls[o[1]]);
                T.call_tab.push_back(n);
                for (uint32_t k = 0; k < n; ++k) {
                    uint32_t a = pcalls[o[1] + 2 + k];
                    T.call_tab.push_back((a & OPERAND_CONST) ? a : remap[a]);
                }
                const uint32_t *ex = &pcalls[o[1] + 2 + n];
                T.call_tab.push_back(ex[0]);
                for (uint32_t k = 0; k < ex[0]; ++k) T.call_tab.push_back(live[ex[1 + k]] ? remap[ex[1 + k]] : NO_SLOT);
                return;
            }
            for (int k = 1; k <= 3; ++k) {
                if (k == 3 && c_is_immediate(o[0])) d[k] = o[k];  // immediate: IR assert number / bit-field spec
                else if (o[k] == NO_SLOT) d[k] = OPERAND_CONST;  // unused operand: constant 0 (never read for its value)
                else if (o[k] & OPERAND_CONST) d[k] = o[k];
                else if (k == 1 && acc_a >= 0) d[k] = OPERAND_ACC | (uint32_t)acc_a;
                else if (k == 2 && acc_b >= 0) d[k] = OPERAND_ACC | (uint32_t)acc_b;
                else d[k] = remap[o[k]];
            }
        };
        // post-order emission of a fused sub-tree; its value ends in accumulator `target`
        std::function<void(uint32_t, int)> emit_sub = [&](uint32_t i, int target) {
            const uint32_t ka = kid_a[i], kb = kid_b[i];
            int acc_a = -1, acc_b = -1;
            if (ka != NO_SLOT && kb != NO_SLOT) {
                // the deeper sub-tree first (it may use both accumulators), then the chain into the other one
                const bool a_first = subtree_need(ka, kid_a, kid_b) >= subtree_need(kb, kid_a, kid_b);
                if (a_first) { emit_sub(ka, target); emit_sub(kb, target ^ 1); }
                else { emit_sub(kb, target); emit_sub(ka, target ^ 1); }
                acc_a = a_first ? target : (target ^ 1);
                acc_b = a_first ? (target ^ 1) : target;
            } else if (ka != NO_SLOT) { emit_sub(ka, target); acc_a = target; }
            else if (kb != NO_SLOT) { emit_sub(kb, target); acc_b = target; }
            uint32_t d[4];
            word(i, DST_ACC + (uint32_t)target, acc_a, acc_b, d);
            T.ops.insert(T.ops.end(), d, d + 4);
            if (pops[(size_t)i * 4] == CW_OP_MUL) ++T.n_mul_ops;
        };
        for (size_t r = 0; r < order.size(); ++r) {
            const uint32_t i = order[r];
            const uint32_t *o = &pops[(size_t)i * 4];
            const uint32_t lvl = glevel[n_pre + i];
            const uint32_t dst = is_assert_op(o[0]) ? 0u : remap[n_pre + i];
            const uint32_t ka = kid_a[i], kb = kid_b[i];
            const bool single = ka == NO_SLOT && kb == NO_SLOT;
            uint32_t d[4];
            if (single) {
                word(i, dst, -1, -1, d);
                // runs of single-bit extractions of one source into consecutive slots (the bits of a decomposition
                // are consecutive witness entries) become ONE tape op that writes the whole run: imm bits 24-31 hold
                // (run length - 1).  One thread fetches the source word once.
                if (o[0] == DOP_BITS && !(flags & CW_FLAG_NO_PEEPHOLE) && lvl == prev_level && !T.ops.empty() &&
                    T.items.back() == T.ops.size() / 4 - 1) {
                    uint32_t *p = &T.ops[T.ops.size() - 4];
                    if ((p[0] & 0xFFu) == DOP_BITS && p[1] == d[1] && ((p[3] >> 16) & 0xFFu) == 1u && ((d[3] >> 16) & 0xFFu) == 1u) {
                        uint32_t cnt = (p[3] >> 24) + 1u, pk = p[3] & 0xFFFFu, pdst = p[0] >> 8;
                        if (cnt < 32u && (d[3] & 0xFFFFu) == pk + cnt && dst == pdst + cnt) {
                            p[3] += 1u << 24;
                            continue;
                        }
                    }
                }
                T.items.push_back((uint32_t)(T.ops.size() / 4));
                T.ops.insert(T.ops.end(), d, d + 4);
            } else {
                T.items.push_back((uint32_t)(T.ops.size() / 4));
                int acc_a = -1, acc_b = -1;
                if (ka != NO_SLOT && kb != NO_SLOT) {
                    const bool a_first = subtree_need(ka, kid_a, kid_b) >= subtree_need(kb, kid_a, kid_b);
                    if (a_first) { emit_sub(ka, 0); emit_sub(kb, 1); }
                    else { emit_sub(kb, 0); emit_sub(ka, 1); }
                    acc_a = a_first ? 0 : 1;
                    acc_b = a_first ? 1 : 0;
                } else if (ka != NO_SLOT) { emit_sub(ka, 0); acc_a = 0; }
                else { emit_sub(kb, 0); acc_b = 0; }
                word(i, dst, acc_a, acc_b, d);
                T.ops.insert(T.ops.end(), d, d + 4);
            }
            prev_level = lvl;
            if (o[0] == CW_OP_MUL) ++T.n_mul_ops;
            T.level_start[lvl]++;  // work items per level (levels start at 1)
        }
        T.items.push_back((uint32_t)(T.ops.size() / 4));
        // prefix sums: level_start[l-1] = first work item of level l
        {
            std::vector<uint32_t> ls(max_level + 1, 0);
            uint32_t acc = 0;
            uint64_t widest = 0;
            for (uint32_t l = 1; l <= max_level; ++l) {
                ls[l - 1] = acc;
                widest = std::max<uint64_t>(widest, T.level_start[l]);
                acc += T.level_start[l];
            }
            ls[max_level] = acc;
            T.level_start.swap(ls);
            T.max_level_width = widest;
        }
        // Bit plane (CW_FLAG_BITPLANE).  The outputs of bit runs - the bits of range checks, 98 % of the witness
        // of limb-arithmetic circuits - leave the 32-byte slot store: a run of up to 32 bits becomes ONE 32-bit
        // word of a per-instance bit plane (one 4-byte store instead of 32 x 32 bytes; 32 x 32 bits per 128-byte
        // line instead of 4).  A reference to such a bit is OPERAND_BIT | (word * 32 + bit); the remaining slots
        // are renumbered densely, witness entry i is found through witness_slot[i].
        std::vector<uint32_t> newid;
        T.n_bitwords = 0;
        if (flags & CW_FLAG_BITPLANE) {
            std::vector<uint32_t> code(next_tmp, NO_SLOT);
            uint32_t n_words = 0;
            const size_t n_ops = T.ops.size() / 4;
            for (size_t i = 0; i < n_ops; ++i) {
                const uint32_t *o = &T.ops[i * 4];
                if ((o[0] & 0xFFu) != DOP_BITS || !(o[3] >> 24)) continue;
                const uint32_t run = (o[3] >> 24) + 1u, d0 = o[0] >> 8;
                for (uint32_t j = 0; j < run; ++j) code[d0 + j] = OPERAND_BIT | (n_words * 32u + j);
                ++n_words;
            }
            bool ok = n_words > 0 && n_words < (1u << 24);
            for (size_t i = 0; ok && i < n_ops; ++i) {  // a run whose source is itself a packed bit stays unsupported
                const uint32_t *o = &T.ops[i * 4];
                if ((o[0] & 0xFFu) == DOP_BITS && (o[3] >> 24) && !(o[1] & OPERAND_CONST) && code[o[1]] != NO_SLOT) ok = false;
            }
            for (uint32_t i = 0; ok && i < M.n_in + 1; ++i)
                if (code[remap[i]] != NO_SLOT) ok = false;
            if (next_tmp >= OPERAND_BIT) ok = false;
            if (ok) {
                newid.resize(next_tmp);
                uint32_t nw = 0;
                for (uint32_t s = 0; s < next_tmp; ++s) newid[s] = code[s] == NO_SLOT ? nw++ : code[s];
                uint32_t word = 0;
                for (size_t i = 0; i < n_ops; ++i) {
                    uint32_t *o = &T.ops[i * 4];
                    const uint32_t opc = o[0] & 0xFFu;
                    if (opc == DOP_BITS && (o[3] >> 24)) o[0] = opc | (word++ << 8);        // destination = bit-plane word
                    else if (!is_assert_op(opc) && (o[0] >> 8) < DST_ACC) o[0] = opc | (newid[o[0] >> 8] << 8);
                    if (opc == 45) continue;  // operand a is the call-table offset; the table is renumbered below
                    for (int k = 1; k <= 3; ++k) {
                        if (k == 3 && c_is_immediate(opc)) break;
                        if (!(o[k] & (OPERAND_CONST | OPERAND_ACC))) o[k] = newid[o[k]];
                    }
                }
                for (size_t i = 0; i < T.call_tab.size();) {  // {function, n_args, operands..., n_extra, destinations...}
                    const uint32_t n = T.call_tab[i + 1], nx = T.call_tab[i + 2 + n];
                    for (uint32_t k = 0; k < n + 1 + nx; ++k) {
                        if (k == n) continue;
                        uint32_t &e = T.call_tab[i + 2 + k];
                        if (!(e & OPERAND_CONST)) e = newid[e];   // (NO_SLOT, a dead result, has the constant bit)
                    }
                    i += 3 + n + nx;
                }
                T.n_bitwords = n_words;
                next_tmp = nw;
            }
        }
        // Slot reuse (CW_FLAG_REUSE).  Values that are not witness entries only live from their op to their last
        // reader; numbering every one of them keeps 386 k dead 32-byte values per instance for the bench circuit
        // while at most 25 k are live at any level.  Temporaries are therefore allocated like registers: an id is
        // released when the level of its last reader has completed (the interpreter's barrier) and handed out
        // again, most recently released first (still in cache).  Witness-resident slots are never reused.
        const uint32_t n_resident = newid.empty() ? (uint32_t)W : [&]() {
            uint32_t n = 0;
            for (uint64_t i = 0; i < W; ++i) n += !(newid[i] & OPERAND_BIT);
            return n;
        }();
        if (flags & CW_FLAG_REUSE) {
            const size_t n_ops = T.ops.size() / 4;
            const size_t n_lv = T.level_start.size() - 1;
            std::vector<uint32_t> last(next_tmp, 0), phys(next_tmp, NO_SLOT);
            auto is_tmp = [&](uint32_t o) { return !(o & (OPERAND_CONST | OPERAND_BIT | OPERAND_ACC)) && o >= n_resident; };
            for (size_t l = 0; l < n_lv; ++l)
                for (uint32_t i = T.items[T.level_start[l]]; i < T.items[T.level_start[l + 1]]; ++i) {
                    const uint32_t *o = &T.ops[(size_t)i * 4];
                    const uint32_t opc = o[0] & 0xFFu;
                    if (opc == 45) {
                        const uint32_t n = T.call_tab[o[1] + 1];
                        for (uint32_t k = 0; k < n; ++k)
                            if (is_tmp(T.call_tab[o[1] + 2 + k])) last[T.call_tab[o[1] + 2 + k]] = (uint32_t)l;
                        continue;
                    }
                    for (int k = 1; k <= 3; ++k) {
                        if (k == 3 && c_is_immediate(opc)) break;
                        if (is_tmp(o[k])) last[o[k]] = (uint32_t)l;
                    }
                }
            std::vector<std::vector<uint32_t>> release(n_lv + 1);  // physical ids that become free when level l starts
            std::vector<uint32_t> free_ids;
            uint32_t next_phys = n_resident;
            for (size_t l = 0; l < n_lv; ++l) {
                for (uint32_t p : release[l]) free_ids.push_back(p);
                for (uint32_t i = T.items[T.level_start[l]]; i < T.items[T.level_start[l + 1]]; ++i) {
                    uint32_t *o = &T.ops[(size_t)i * 4];
                    const uint32_t opc = o[0] & 0xFFu, d = o[0] >> 8;
                    if (is_assert_op(opc) || d >= DST_ACC) continue;
                    const uint32_t run = opc == DOP_BITS ? (o[3] >> 24) + 1u : 1u;
                    if (run > 1) {
                        if (T.n_bitwords || d < n_resident) continue;  // a word of the bit plane / witness entries
                        for (uint32_t j = 0; j < run; ++j) phys[d + j] = next_phys++;  // consecutive, never released
                        continue;
                    }
                    auto alloc = [&](uint32_t d) {
                        if (d < n_resident) return;
                        uint32_t p;
                        if (!free_ids.empty()) { p = free_ids.back(); free_ids.pop_back(); }
                        else p = next_phys++;
                        phys[d] = p;
                        // readers are in levels (l, last[d]]; a value nobody reads (the first result of a call whose
                        // other results are used) is released at once
                        release[std::min<size_t>(std::max<size_t>(last[d], l) + 1, n_lv)].push_back(p);
                    };
                    alloc(d);
                    if (opc == 45) {  // the further results of a call
                        const uint32_t *ex = &T.call_tab[o[1] + 2 + T.call_tab[o[1] + 1]];
                        for (uint32_t k = 0; k < ex[0]; ++k)
                            if (ex[1 + k] != NO_SLOT) alloc(ex[1 + k]);
                    }
                }
            }
            auto map = [&](uint32_t o) { return is_tmp(o) ? phys[o] : o; };
            for (size_t i = 0; i < n_ops; ++i) {
                uint32_t *o = &T.ops[i * 4];
                const uint32_t opc = o[0] & 0xFFu;
                if (!is_assert_op(opc) && !(opc == DOP_BITS && (o[3] >> 24) && T.n_bitwords) && (o[0] >> 8) >= n_resident &&
                    (o[0] >> 8) < DST_ACC)
                    o[0] = opc | (phys[o[0] >> 8] << 8);
                if (opc == 45) continue;
                for (int k = 1; k <= 3; ++k) {
                    if (k == 3 && c_is_immediate(opc)) break;
                    o[k] = map(o[k]);
                }
            }
            for (size_t i = 0; i < T.call_tab.size();) {
                const uint32_t n = T.call_tab[i + 1], nx = T.call_tab[i + 2 + n];
                for (uint32_t k = 0; k < n + 1 + nx; ++k)
                    if (k != n) T.call_tab[i + 2 + k] = map(T.call_tab[i + 2 + k]);
                i += 3 + n + nx;
            }
            next_tmp = next_phys;
        }
        T.n_resident = n_resident;
        {   // operand statistics
            T.n_slot_operands = 0;
            T.n_values = 0;
            T.n_stored = 0;
            const size_t n_ops = T.ops.size() / 4;
            for (size_t i = 0; i < n_ops; ++i) {
                const uint32_t *o = &T.ops[i * 4];
                const uint32_t opc = o[0] & 0xFFu;
                if (!is_assert_op(opc)) T.n_values += opc == DOP_BITS ? (o[3] >> 24) + 1u : 1u;  // (fused values included: S_w of 8(d))
                if (!is_assert_op(opc) && (o[0] >> 8) < DST_ACC) ++T.n_stored;
                if (opc == 45) {
                    const uint32_t *ex = &T.call_tab[o[1] + 2 + T.call_tab[o[1] + 1]];
                    for (uint32_t k = 0; k < ex[0]; ++k)
                        if (ex[1 + k] != NO_SLOT) { ++T.n_values; ++T.n_stored; }
                    continue;
                }
                for (int k = 1; k <= 3; ++k) {
                    if (k == 3 && c_is_immediate(opc)) break;
                    if (!(o[k] & (OPERAND_CONST | OPERAND_BIT | OPERAND_ACC))) ++T.n_slot_operands;
                }
            }
        }
        T.witness_slot.resize(W);
        for (uint64_t i = 0; i < W; ++i) T.witness_slot[i] = newid.empty() ? (uint32_t)i : newid[i];
        T.input_slot.resize(M.n_in);
        for (uint32_t i = 0; i < M.n_in; ++i) T.input_slot[i] = newid.empty() ? remap[1 + i] : newid[remap[1 + i]];
        if (remap[0] != 0) throw std::runtime_error("lowering: constant-one signal is not witness entry 0");
        T.consts = consts;
        if (T.consts.empty()) T.consts.push_back(u256_from_u64(0));
        T.dat_consts = ir_consts;
        // census of the value slots by static width (what narrow slots would store in 4 / 8 bytes, DESIGN.md 10.1)
        for (int k = 0; k < 4; ++k) T.slot_census[k] = 0;
        for (size_t i = 0; i < n_pre + n_prov; ++i) {
            if (remap[i] == NO_SLOT) continue;
            const uint16_t b = slot_bits[i];
            T.slot_census[b <= 1 ? 0 : b <= 32 ? 1 : b <= 64 ? 2 : 3]++;
        }
        T.n_pre = n_pre;
        T.n_slots = next_tmp;
        T.n_ir_ops = n_ir_ops;
        T.n_conv_ops = n_conv;
        T.n_asserts = n_asserts;
        T.flags = flags;
        for (const Tmpl &t : tm) T.tmpl_names.push_back(t.name);

        // input hash map, laid out as the reference's .dat (c_code_generator.rs:575-603)
        uint64_t hs = 256;
        while (hs < T.inputs.size()) hs <<= 1;  // get_input_hash_map_entry_size (c_elements/mod.rs:167-169)
        T.hashmap.assign(hs, HashEntry{0, 0, 0});
        for (const InputInfo &in : T.inputs) {
            uint64_t p = in.hash % hs;
            while (T.hashmap[p].signalid != 0) p = (p + 1) % hs;
            T.hashmap[p] = HashEntry{in.hash, in.signal_id, in.size};
        }

    }
};

}  // namespace

void lower_circuit(const uint8_t *data, size_t len, uint32_t flags, Tape &out) {
    Lowerer L(out, flags);
    L.parse(data, len);
    L.lower();
}

}  // namespace cw

// ---- the lowered circuit as one blob ---------------------------------------------------------------------
// What rank 0 broadcasts to the other GPUs' processes (instruction tape, constants, witness maps, function code,
// input tables and the R1CS in CSR form): they then skip the lowering.  Also usable as an on-disk cache.  The
// format is private to one build of the library ("CB2T" + a layout version), not an interchange format.
namespace cw {
namespace {
struct BlobW {
    std::vector<uint8_t> &o;
    void raw(const void *p, size_t n) { o.insert(o.end(), (const uint8_t *)p, (const uint8_t *)p + n); }
    template <class T> void pod(const T &v) { raw(&v, sizeof(T)); }
    template <class T> void vec(const std::vector<T> &v) {
        pod<uint64_t>(v.size());
        if (!v.empty()) raw(v.data(), v.size() * sizeof(T));
    }
    void str(const std::string &s) {
        pod<uint64_t>(s.size());
        raw(s.data(), s.size());
    }
};
struct BlobR {
    const uint8_t *p, *end;
    void raw(void *d, size_t n) {
        if (n > (size_t)(end - p)) throw std::runtime_error("lowered-circuit blob: truncated");
        memcpy(d, p, n);
        p += n;
    }
    template <class T> void pod(T &v) { raw(&v, sizeof(T)); }
    template <class T> void vec(std::vector<T> &v) {
        uint64_t n;
        pod(n);
        if (n > (uint64_t)(end - p) / sizeof(T)) throw std::runtime_error("lowered-circuit blob: bad length");
        v.resize(n);
        if (n) raw(v.data(), n * sizeof(T));
    }
    void str(std::string &s) {
        uint64_t n;
        pod(n);
        if (n > (uint64_t)(end - p)) throw std::runtime_error("lowered-circuit blob: bad length");
        s.assign((const char *)p, n);
        p += n;
    }
};
constexpr uint32_t BLOB_VERSION = 7;
}  // namespace

void serialize_tape(const Tape &t, std::vector<uint8_t> &out) {
    BlobW w{out};
    w.raw("CB2T", 4);
    w.pod<uint32_t>(BLOB_VERSION);
    w.pod<int32_t>(t.F.prime_id);
    w.pod(t.flags);
    const uint64_t nums[] = {t.n_signals, t.n_witness, t.n_inputs, t.n_outputs, t.n_components, t.n_ir_ops, t.n_mul_ops,
                             t.n_conv_ops, t.max_level_width, t.n_asserts, t.slot_census[0], t.slot_census[1],
                             t.slot_census[2], t.slot_census[3], t.n_slot_operands, t.n_values, t.n_resident, t.n_pre,
                             t.n_slots, t.n_bitwords, t.n_stored};
    w.pod<uint64_t>(sizeof(nums) / 8);
    w.raw(nums, sizeof(nums));
    w.vec(t.ops); w.vec(t.items); w.vec(t.level_start); w.vec(t.consts); w.vec(t.dat_consts); w.vec(t.witness_slot); w.vec(t.input_slot);
    w.vec(t.pk_bit_wire); w.vec(t.pk_u64_wire); w.vec(t.pk_full_wire); w.vec(t.wit_class); w.vec(t.wit_bits);
    w.vec(t.fn_code); w.vec(t.fn_info); w.vec(t.call_tab); w.vec(t.witness2signal);
    w.pod<uint64_t>(t.inputs.size());
    for (const InputInfo &in : t.inputs) {
        w.str(in.name);
        w.pod(in.hash); w.pod(in.signal_id); w.pod(in.size);
    }
    w.vec(t.hashmap);
    const R1csData &r = t.r1cs;
    w.pod<int32_t>(r.prime_id);
    w.pod(r.n_wires); w.pod(r.n_constraints);
    w.vec(r.row_ptr); w.vec(r.col); w.vec(r.coef); w.vec(r.dict);
    w.pod(r.n_pub_out); w.pod(r.n_pub_in); w.pod(r.n_prv_in);
}

void deserialize_tape(const uint8_t *data, size_t len, Tape &t) {
    BlobR r{data, data + len};
    char magic[4];
    r.raw(magic, 4);
    uint32_t ver;
    r.pod(ver);
    if (memcmp(magic, "CB2T", 4) || ver != BLOB_VERSION) throw std::runtime_error("lowered-circuit blob: bad magic / version");
    int32_t prime;
    r.pod(prime);
    if (prime < 0 || prime >= CW_N_PRIMES) throw std::runtime_error("lowered-circuit blob: unknown prime");
    t.F = make_field(prime);
    r.pod(t.flags);
    uint64_t n_nums;
    r.pod(n_nums);
    uint64_t nums[21];
    if (n_nums != 21) throw std::runtime_error("lowered-circuit blob: layout mismatch");
    r.raw(nums, sizeof(nums));
    t.n_signals = nums[0]; t.n_witness = nums[1]; t.n_inputs = nums[2]; t.n_outputs = nums[3]; t.n_components = nums[4];
    t.n_ir_ops = nums[5]; t.n_mul_ops = nums[6]; t.n_conv_ops = nums[7]; t.max_level_width = nums[8]; t.n_asserts = nums[9];
    for (int k = 0; k < 4; ++k) t.slot_census[k] = nums[10 + k];
    t.n_slot_operands = nums[14]; t.n_values = nums[15]; t.n_resident = (uint32_t)nums[16]; t.n_pre = (uint32_t)nums[17];
    t.n_slots = (uint32_t)nums[18]; t.n_bitwords = (uint32_t)nums[19]; t.n_stored = nums[20];
    r.vec(t.ops); r.vec(t.items); r.vec(t.level_start); r.vec(t.consts); r.vec(t.dat_consts); r.vec(t.witness_slot); r.vec(t.input_slot);
    r.vec(t.pk_bit_wire); r.vec(t.pk_u64_wire); r.vec(t.pk_full_wire); r.vec(t.wit_class); r.vec(t.wit_bits);
    r.vec(t.fn_code); r.vec(t.fn_info); r.vec(t.call_tab); r.vec(t.witness2signal);
    uint64_t n_in;
    r.pod(n_in);
    if (n_in > len) throw std::runtime_error("lowered-circuit blob: bad length");
    t.inputs.resize(n_in);
    for (InputInfo &in : t.inputs) {
        r.str(in.name);
        r.pod(in.hash); r.pod(in.signal_id); r.pod(in.size);
    }
    r.vec(t.hashmap);
    R1csData &R = t.r1cs;
    int32_t rp;
    r.pod(rp);
    R.prime_id = rp;
    r.pod(R.n_wires); r.pod(R.n_constraints);
    r.vec(R.row_ptr); r.vec(R.col); r.vec(R.coef); r.vec(R.dict);
    r.pod(R.n_pub_out); r.pod(R.n_pub_in); r.pod(R.n_prv_in);
    // consistency of what the kernels index with (the blob comes from another rank of the same job, not from a user,
    // but a short read or a version skew must not turn into out-of-bounds device accesses)
    if (t.ops.size() % 4 || t.level_start.empty() || t.items.empty() || t.level_start.back() != t.items.size() - 1 ||
        t.items.back() != t.ops.size() / 4 ||
        t.witness_slot.size() != t.n_witness || t.input_slot.size() != t.n_inputs || t.wit_class.size() != t.n_witness || t.wit_bits.size() != t.n_witness ||
        t.witness2signal.size() != t.n_witness || R.row_ptr.size() != 3 * R.n_constraints + 1 || R.col.size() != R.coef.size() ||
        (R.row_ptr.size() && R.row_ptr.back() != R.col.size()) || t.hashmap.empty())
        throw std::runtime_error("lowered-circuit blob: inconsistent");
}

}  // namespace cw
