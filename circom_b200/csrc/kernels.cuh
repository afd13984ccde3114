// sm_100a kernels: tape execution, input staging, witness gather, R1CS check, field batch ops.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "fr_device.cuh"
#include "r1cs_small.h"

namespace cw {

// Per-prime parameters live in constant memory so that modulus limbs are read as c[bank][imm]
// instruction operands (no registers, no loads).
// bn128 and bls12381 have kernel builds of their own (template PRIME = 0 / 1: the table index folds into the
// instruction); the other 256-bit primes share one build (PRIME = -1) that takes the index from its arguments.
constexpr int N_PRIMES_DEV = 8;
__constant__ FrParams c_fr[N_PRIMES_DEV];
#define CW_FR(PRIME, rt) c_fr[(PRIME) >= 0 ? (PRIME) : (int)(rt)]

// ---- value-slot storage ---------------------------------------------------------------------
// One instance tile holds BT = 1 << bt_log2 instances.  A slot (256-bit value) of a tile is two
// 16-byte halves, each stored for the BT instances contiguously:
//     uint4 index = (tile * n_slots + slot) * 2 * BT + half * BT + instance_in_tile
// so a (warp of) thread(s) working on BT instances of one op issues 128-bit loads over
// BT*16 contiguous bytes per half; with BT = 1 this is the plain 32-byte element (one DRAM sector).
// sm_100 moves a whole 32-byte element with one instruction (LDG/STG.E.ENL2.256): half the memory
// instructions and half the L1/L2 requests of a pair of 128-bit accesses.  32-byte alignment required.
__device__ __forceinline__ void ldg256(u32 *v, const void *p) {
    asm volatile("ld.global.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
                 : "l"(p)
                 : "memory");
}
__device__ __forceinline__ void ldg256_nc(u32 *v, const void *p) {  // data that no thread of the kernel writes
    asm("ld.global.nc.v8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
        : "l"(p));
}
__device__ __forceinline__ void stg256(void *p, const u32 *v) {
    asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "r"(v[0]), "r"(v[1]), "r"(v[2]),
                 "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
                 : "memory");
}

__device__ __forceinline__ void load_slot(u32 *v, const uint4 *__restrict__ tile_base, u32 slot, u32 bt_log2,
                                          u32 inst) {
    if (bt_log2 == 0) {  // one instance per tile: the element is contiguous
        ldg256(v, tile_base + ((size_t)slot << 1));
        return;
    }
    size_t i = ((size_t)slot << (bt_log2 + 1)) + inst;
    uint4 lo = tile_base[i];
    uint4 hi = tile_base[i + ((size_t)1 << bt_log2)];
    v[0] = lo.x; v[1] = lo.y; v[2] = lo.z; v[3] = lo.w;
    v[4] = hi.x; v[5] = hi.y; v[6] = hi.z; v[7] = hi.w;
}
__device__ __forceinline__ void store_slot(const u32 *v, uint4 *__restrict__ tile_base, u32 slot, u32 bt_log2,
                                           u32 inst) {
    if (bt_log2 == 0) {
        stg256(tile_base + ((size_t)slot << 1), v);
        return;
    }
    size_t i = ((size_t)slot << (bt_log2 + 1)) + inst;
    tile_base[i] = make_uint4(v[0], v[1], v[2], v[3]);
    tile_base[i + ((size_t)1 << bt_log2)] = make_uint4(v[4], v[5], v[6], v[7]);
}
__device__ __forceinline__ void load_const(u32 *v, const uint4 *__restrict__ consts, u32 idx) {
    uint4 lo = __ldg(&consts[2 * (size_t)idx]);
    uint4 hi = __ldg(&consts[2 * (size_t)idx + 1]);
    v[0] = lo.x; v[1] = lo.y; v[2] = lo.z; v[3] = lo.w;
    v[4] = hi.x; v[5] = hi.y; v[6] = hi.z; v[7] = hi.w;
}
constexpr u32 OPD_CONST = 0x80000000u, OPD_BIT = 0x20000000u, OPD_ACC = 0x10000000u, OPD_SLOT = 0x00FFFFFFu, OPD_BITPOS = 0x1FFFFFFFu;
constexpr u32 DST_ACC_DEV = 0x00FFFFFEu;  // destination field: accumulator 0 / 1 of a fused work item (tape.h DST_ACC)

// ---- the bit plane (CW_FLAG_BITPLANE) ----------------------------------------------------------------
// Bits produced by bit runs (the outputs of Num2Bits-style decompositions: most of the witness of limb
// arithmetic) are not 32-byte slots: a run of up to 32 bits is ONE 32-bit word.  Word w of instance li of a tile:
//     u32 index = (tile * n_bitwords + w) * BT + li
__device__ __forceinline__ u32 load_plane_bit(const u32 *__restrict__ plane_base, u32 pos, u32 bt_log2, u32 li) {
    return (plane_base[((size_t)(pos >> 5) << bt_log2) + li] >> (pos & 31u)) & 1u;
}

// operand of a tape op: constant-table entry, a bit of the bit plane, or a value slot
template <bool BP>
__device__ __forceinline__ void load_operand(u32 *v, u32 operand, const uint4 *__restrict__ tile_base,
                                             const u32 *__restrict__ plane_base, const uint4 *__restrict__ consts,
                                             u32 bt_log2, u32 li) {
    if (operand & OPD_CONST) {
        load_const(v, consts, operand & 0x7FFFFFFFu);
    } else if (BP && (operand & OPD_BIT)) {
        u256_set_u32(v, load_plane_bit(plane_base, operand & OPD_BITPOS, bt_log2, li));
    } else {
        load_slot(v, tile_base, operand & OPD_SLOT, bt_log2, li);
    }
}

__device__ __forceinline__ u32 u256_bitlen_dev(const u32 *a) {
    u32 n = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i)
        if (a[i]) n = 32u * i + (32u - __clz(a[i]));
    return n;
}

struct TapeDev {
    const uint4 *ops;          // {opcode | dst << 8, a, b, c}
    const u32 *items;          // n_items + 1: work item k = tape words [items[k], items[k+1]) evaluated by one thread
    const uint4 *heads;        // n_items: copy of the first tape word of every work item (fetched in parallel with items[])
    const u32 *level_start;    // n_levels + 1, indexes work items
    const uint4 *consts;       // 2 per constant
    const u32 *input_slot;     // slot of main input k
    const u32 *fn_code;        // register-machine code of the circuit's functions (5 words per instruction)
    const u32 *fn_info;        // per function {code offset, n_instr, n_regs, n_params}
    const u32 *call_tab;       // per call {function, n_args, arg operands..., n_extra, slots of results 1..n_extra}
    const u32 *level_info;     // per level: bits 0-30 how many of its LAST work items are calls, bit 31: it has INV / POW items
    u32 n_levels;
    u32 n_slots;
    u32 n_inputs;
    u32 n_bitwords;            // words of the bit plane per instance (0: no bit plane)
    u32 prime;                 // index into c_fr (read by the PRIME = -1 builds)
    u32 vm_wide;               // 1: calls skip the 128-bit register machine (CW_VM_WIDE=1, for measurements)
    u32 has_slow;              // the tape has INV / POW items at all
};

// (tape_calls.cu compiles only the interpreter builds with the function machine - ptxas gives up on one module with all
// builds - and defines CW_KERNELS_TAPE_ONLY: the non-template kernels must exist in one translation unit only)
#ifndef CW_KERNELS_TAPE_ONLY
// ---- inputs: inputs[batch][n_inputs][8 u32] canonical -> slots 1..n_inputs, slot 0 = 1 ----------
__global__ void stage_inputs_kernel(TapeDev tp, const uint4 *__restrict__ inputs, uint4 *__restrict__ slots,
                                    u32 batch, u32 batch_padded, u32 bt_log2) {
    size_t total = (size_t)batch_padded * (tp.n_inputs + 1);
    for (size_t w = blockIdx.x * (size_t)blockDim.x + threadIdx.x; w < total; w += (size_t)gridDim.x * blockDim.x) {
        u32 inst = (u32)(w % batch_padded);
        u32 k = (u32)(w / batch_padded);  // 0 = constant one, 1.. = input k-1
        u32 tile = inst >> bt_log2, li = inst & ((1u << bt_log2) - 1);
        uint4 *base = slots + (((size_t)tile * tp.n_slots) << (bt_log2 + 1));
        u32 v[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        if (k == 0) v[0] = 1;
        else if (inst < batch) {
            const uint4 *src = inputs + ((size_t)inst * tp.n_inputs + (k - 1)) * 2;
            uint4 lo = src[0], hi = src[1];
            v[0] = lo.x; v[1] = lo.y; v[2] = lo.z; v[3] = lo.w;
            v[4] = hi.x; v[5] = hi.y; v[6] = hi.z; v[7] = hi.w;
        }
        store_slot(v, base, k == 0 ? 0u : __ldg(&tp.input_slot[k - 1]), bt_log2, li);
    }
}

#endif  // CW_KERNELS_TAPE_ONLY

// ---- the tape interpreter ---------------------------------------------------------------------
// One CTA owns one tile of BT instances and walks the levels of the tape; within a level the work
// items (op, instance) are spread over the CTA's threads, instance fastest.  Values produced in
// level l are consumed in later levels by other threads of the same CTA only, so a CTA barrier
// per level is the only synchronisation (no grid-wide sync, tiles are independent).  With BT = 32 a warp
// is ONE op for 32 instances: no divergence, every slot access is 2 x 512 contiguous bytes, the tape word
// is a broadcast; with BT = 1 a warp is 32 ops of one instance (small batches: lanes along ops).
// A function call (circom `function` with run-time loops / branches): the thread copies the arguments into
// the callee's registers (local memory: they are indexed dynamically) and interprets the body.
// (TAG: one copy of the function per interpreter build - ptxas 12.9 crashes on a module in which several kernels share it)
// INV (600 division steps) and POW (a square-and-multiply ladder) are loops of hundreds of steps over many registers; the
// interpreter skips them in its hot loop and runs them afterwards, per level, through this function (one copy per build, TAG)
template <int PRIME, int TAG>
__device__ __noinline__ void exec_slow_op(u32 opcode, u32 *r, const u32 *a, const u32 *b, u32 prime_rt) {
    const FrParams &P = CW_FR(PRIME, prime_rt);
    if (opcode == OP_INV) fr_inv_mont(r, a, P);
    else fr_pow_mont(r, a, b, P);
}

template <int PRIME, bool BP, int TAG>
__device__ __noinline__ void exec_call(const TapeDev &tp, u32 call_off, uint4 *base, const u32 *plane_base,
                                       u32 bt_log2, u32 li, u32 *r, int *err) {
    const FrParams &P = CW_FR(PRIME, tp.prime);
    const u32 *ct = tp.call_tab + call_off;
    const u32 f = __ldg(&ct[0]), n_args = __ldg(&ct[1]);
    FnInfo fi;
    fi.code_off = __ldg(&tp.fn_info[4 * f]);
    fi.n_instr = __ldg(&tp.fn_info[4 * f + 1]);
    fi.n_regs = __ldg(&tp.fn_info[4 * f + 2]);
    fi.n_params = __ldg(&tp.fn_info[4 * f + 3]);
    u32 regs[VM_MAX_REGS * 8];
    for (u32 k = 0; k < n_args; ++k) {
        u32 v[8];
        load_operand<BP>(v, __ldg(&ct[2 + k]), base, plane_base, tp.consts, bt_log2, li);
        for (int j = 0; j < 8; ++j) regs[8 * k + j] = v[j];
    }
    int e = 0;
    u32 ret_base, ret_cnt;
    // first on the 128-bit machine (fr_device.cuh: half the frame, integer arithmetic); a value that leaves 128 bits
    // abandons that run and the call is repeated at full width
    const bool narrow = !tp.vm_wide && vm_run_narrow(tp.fn_code, tp.fn_info, f, regs, reinterpret_cast<const u32 *>(tp.consts), r,
                                                     e, ret_base, ret_cnt);
    if (!narrow) {
        for (u32 k = 0; k < fi.n_regs * 8; ++k) regs[k] = 0;
        for (u32 k = 0; k < n_args; ++k) {
            u32 v[8];
            load_operand<BP>(v, __ldg(&ct[2 + k]), base, plane_base, tp.consts, bt_log2, li);
            for (int j = 0; j < 8; ++j) regs[8 * k + j] = v[j];
        }
        e = 0;
        vm_run(tp.fn_code, tp.fn_info, f, regs, reinterpret_cast<const u32 *>(tp.consts), r, P, e, ret_base, ret_cnt);
    }
    // `var q[k] = f(..)`: results 1 .. k-1 go straight from the callee's registers to their slots (result 0 is `r`)
    const u32 n_extra = __ldg(&ct[2 + n_args]);
    for (u32 k = 0; k < n_extra; ++k) {
        const u32 d = __ldg(&ct[3 + n_args + k]);
        if (d == 0xFFFFFFFFu) continue;   // a result nobody reads
        if (k + 1 >= ret_cnt) { e = 2; continue; }
        u32 v[8];
        vm_result(v, regs, ret_base + k + 1, narrow);
        store_slot(v, base, d, bt_log2, li);
    }
    *err = e;
}

// ---- the accumulators of fused work items ----------------------------------------------------------------
// A fused work item keeps the values its inner words produce in two accumulators.  They live in shared memory, not
// in registers: 16 registers of accumulators, plus the selects between them that a register array indexed by a tape
// bit needs, pushed the fused interpreter over its 64-register budget into local-memory spills around every word.
// Layout [acc][half][thread] (uint4): a warp moves one 512-byte row per half, without bank conflicts.
__host__ __device__ constexpr unsigned tape_acc_smem(unsigned threads) { return 4u * threads * (unsigned)sizeof(uint4); }
__device__ __forceinline__ void load_acc(u32 *v, const uint4 *s_acc, u32 k) {
    const uint4 lo = s_acc[(2u * k) * blockDim.x + threadIdx.x], hi = s_acc[(2u * k + 1u) * blockDim.x + threadIdx.x];
    v[0] = lo.x; v[1] = lo.y; v[2] = lo.z; v[3] = lo.w;
    v[4] = hi.x; v[5] = hi.y; v[6] = hi.z; v[7] = hi.w;
}
__device__ __forceinline__ void store_acc(const u32 *v, uint4 *s_acc, u32 k) {
    s_acc[(2u * k) * blockDim.x + threadIdx.x] = make_uint4(v[0], v[1], v[2], v[3]);
    s_acc[(2u * k + 1u) * blockDim.x + threadIdx.x] = make_uint4(v[4], v[5], v[6], v[7]);
}

// HAS_CALLS selects the build that contains the function interpreter (more registers, a local-memory
// frame); tapes without calls - all circuits whose hints are straight-line - use the lean build.
// BP: the tape was lowered with a bit plane (bit runs write plane words, operands may be plane bits).
#ifndef CW_TAPE_LB
#define CW_TAPE_LB 512  // widest CTA of the interpreter (cw_batch_create clamps to it); with MINB it bounds the registers
#endif
#ifndef CW_TAPE_MINB
#define CW_TAPE_MINB 2  // 512 x 2: a 64-register budget (measured faster than 84 registers)
#endif
// BT >= 0 fixes the tile size at compile time (BT = 0, one instance per CTA: the slot address arithmetic then
// folds to `base + slot * 32`; BT = 5, a warp per op); BT < 0 takes it from the launch argument.
// FUSED: the tape has multi-word work items (CW_FLAG_FUSE); otherwise work item k IS tape word k and the item table,
// the accumulators and the inner loop disappear at compile time.
template <int PRIME, bool HAS_CALLS, bool BP, int BT, bool FUSED>
__global__ void __launch_bounds__(CW_TAPE_LB, CW_TAPE_MINB)
    tape_exec_kernel(TapeDev tp, uint4 *__restrict__ slots, u32 *__restrict__ plane, u32 bt_log2_arg,
                     u32 *__restrict__ first_assert, int *__restrict__ err, u32 batch) {
    const FrParams &P = CW_FR(PRIME, tp.prime);
    const u32 bt_log2 = BT >= 0 ? (u32)BT : bt_log2_arg;
    constexpr bool COOP = BT == 0 && !HAS_CALLS && !BP;  // warp-cooperative bit-run stores (needs blockDim % 32 == 0)
    const u32 tile = blockIdx.x;
    const u32 bt_mask = (1u << bt_log2) - 1;
    uint4 *base = slots + (((size_t)tile * tp.n_slots) << (bt_log2 + 1));
    u32 *plane_base = BP ? plane + (((size_t)tile * tp.n_bitwords) << bt_log2) : nullptr;
    // FUSED: the two accumulators of the thread's work item (tape_acc_smem bytes of dynamic shared memory)
    extern __shared__ uint4 s_acc[];
    u32 lb = tp.level_start[0];
    u32 le = tp.n_levels ? tp.level_start[1] : lb;
    // the first tape word of a thread's first work item of the next level is fetched before the barrier of the
    // current one, taking the memory round trips of the item table and the tape off the per-level critical path
    uint4 pre = make_uint4(0, 0, 0, 0);
    u32 pre_g0 = 0, pre_g1 = 0;
    if (threadIdx.x < ((le - lb) << bt_log2)) {
        if (FUSED) {
            pre_g0 = __ldg(&tp.items[lb + (threadIdx.x >> bt_log2)]);
            pre_g1 = __ldg(&tp.items[lb + (threadIdx.x >> bt_log2) + 1]);
            pre = __ldg(&tp.heads[lb + (threadIdx.x >> bt_log2)]);
        } else pre = __ldg(&tp.ops[lb + (threadIdx.x >> bt_log2)]);
    }
    for (u32 l = 0; l < tp.n_levels; ++l) {
        // Calls are the last work items of their level (the items of a level are sorted by opcode, CALL is the largest) and
        // run in a loop of their own after the others: the call site - an ABI call with a 6 KB frame - then does not sit
        // in the hot loop, whose values would otherwise have to survive it in memory.
        const u32 info = (HAS_CALLS || tp.has_slow) ? __ldg(&tp.level_info[l]) : 0u;
        const u32 n_calls = HAS_CALLS ? (info & 0x7FFFFFFFu) : 0u;
        const u32 n = (le - lb - n_calls) << bt_log2;
        const u32 le_next = (l + 1 < tp.n_levels) ? tp.level_start[l + 2] : le;
        // COOP (one instance per CTA): the warp walks the level together - lanes beyond the level's end idle in
        // the body - so that the bit runs of its lanes can be stored cooperatively afterwards
        for (u32 w0 = COOP ? (threadIdx.x & ~31u) : threadIdx.x; w0 < n; w0 += blockDim.x) {
            const u32 w = COOP ? w0 + (threadIdx.x & 31u) : w0;
            u32 run_dst = 0, run_n = 0, run_bits = 0;
            if (!COOP || w < n) {
            const u32 li = w & bt_mask;
            const u32 inst = (tile << bt_log2) + li;
            const bool first = w == threadIdx.x;
            u32 g0 = lb + (w >> bt_log2), g1 = g0 + 1u;   // !FUSED: work item k is tape word k
            if (FUSED) {
                g0 = first ? pre_g0 : __ldg(&tp.items[lb + (w >> bt_log2)]);
                g1 = first ? pre_g1 : __ldg(&tp.items[lb + (w >> bt_log2) + 1]);
            }
            uint4 nxt = pre;
            if (!first) {
                if (FUSED) nxt = __ldg(&tp.heads[lb + (w >> bt_log2)]);
                else nxt = __ldg(&tp.ops[g0]);
            }
            for (u32 k = g0; k < g1; ++k) {
            const uint4 opw = nxt;
            bool has_value = true;   // false: the word stored its results itself / has none (asserts)
            if (FUSED && k + 1 < g1) nxt = __ldg(&tp.ops[k + 1]);   // the next word of the item travels while this one executes
            const u32 opcode = opw.x & 0xFFu, dst = opw.x >> 8;
            u32 r[8];
            if (opcode == OP_BITS && ((opw.w >> 16) & 0xFFu) <= 32u && !(opw.y & (OPD_CONST | OPD_BIT | OPD_ACC))) {
                // narrow bit-field of a slot value: fetch only the one or two 32-bit words that hold it
                const u32 kk = opw.w & 0xFFFFu, m = (opw.w >> 16) & 0xFFu, run = (opw.w >> 24) + 1u;
                const u32 wd = kk >> 5, sh = kk & 31u;
                const bool two = sh + m + run - 1u > 32u && wd < 7u;
                u32 lo, hi = 0;
                {
                    const u32 *words = reinterpret_cast<const u32 *>(base);
                    const size_t src = (size_t)(opw.y & OPD_SLOT) << (bt_log2 + 1);
                    const u32 w1 = wd + 1u;
                    lo = words[((src + ((size_t)(wd >> 2) << bt_log2) + li) << 2) + (wd & 3u)];
                    if (two) hi = words[((src + ((size_t)(w1 >> 2) << bt_log2) + li) << 2) + (w1 & 3u)];
                }
                const unsigned long long window = (((unsigned long long)hi << 32) | lo) >> sh;
#pragma unroll
                for (int i = 1; i < 8; ++i) r[i] = 0;
                if (run > 1u) {
                    if (BP && tp.n_bitwords) {  // the run is ONE word of the bit plane (dst = word index): a single 4-byte store
                        // (a BP build may be handed a tape without a plane: then runs are slots, below)
                        plane_base[((size_t)dst << bt_log2) + li] =
                            (u32)window & (run >= 32u ? 0xFFFFFFFFu : ((1u << run) - 1u));
                    } else if (COOP) {  // `run` (<= 32) consecutive slots, one bit each: stored by the whole warp after the body
                        run_dst = dst;
                        run_n = run;
                        run_bits = (u32)window;
                    } else {
                        for (u32 j = 0; j < run; ++j) {
                            r[0] = (u32)(window >> j) & 1u;
                            store_slot(r, base, dst + j, bt_log2, li);
                        }
                    }
                    has_value = false;
                } else r[0] = (u32)window & (m >= 32u ? 0xFFFFFFFFu : ((1u << m) - 1u));
            } else {
                u32 a[8], b[8];
                if (FUSED && !(opw.y & OPD_CONST) && (opw.y & OPD_ACC)) load_acc(a, s_acc, opw.y & 1u);
                else load_operand<BP>(a, opw.y, base, plane_base, tp.consts, bt_log2, li);
                if (FUSED && !(opw.z & OPD_CONST) && (opw.z & OPD_ACC)) load_acc(b, s_acc, opw.z & 1u);
                else load_operand<BP>(b, opw.z, base, plane_base, tp.consts, bt_log2, li);
                if (opcode == OP_SELECT) {
                    u32 c[8];
                    load_operand<BP>(c, opw.w, base, plane_base, tp.consts, bt_log2, li);
                    bool t = !u256_is_zero(c);
#pragma unroll
                    for (int i = 0; i < 8; ++i) r[i] = t ? a[i] : b[i];
                } else if (opcode == OP_ASSERT_EQ || opcode == OP_ASSERT || opcode == OP_ASSERT_BOOL ||
                           opcode == OP_ASSERT_FITS) {
                    bool ok = opcode == OP_ASSERT_EQ     ? u256_eq(a, b)
                              : opcode == OP_ASSERT      ? !u256_is_zero(a)
                              : opcode == OP_ASSERT_BOOL ? (u256_is_zero(a) || u256_eq(a, b))
                                                         : (u256_bitlen_dev(a) <= b[0]);
                    if (!ok && inst < batch) atomicMin(&first_assert[inst], opw.w);
                    has_value = false;  // asserts have no destination value
                } else if (opcode == OP_INV || opcode == OP_POW) {
                    has_value = false;   // the slow operators of the level run after the others (below); never fused
                } else {
                    int e = 0;
                    fr_exec_t<false>(opcode, r, a, b, opw.w, P, e);
                    if (e && inst < batch) err[inst] = 1;
                }
            }
            if (has_value) {
                if (FUSED && dst >= DST_ACC_DEV) store_acc(r, s_acc, dst & 1u);
                else store_slot(r, base, dst, bt_log2, li);
            }
            }
            }
            if (COOP) {
                // Bit runs, warp-cooperatively: the slots of a run are consecutive, so lane j stores bit j and one
                // store instruction covers run * 32 contiguous bytes (whole 128-byte lines) - a lane streaming its
                // own run would touch one line per instruction and lane, 32 different lines per instruction.
                unsigned pending = __ballot_sync(0xFFFFFFFFu, run_n != 0u);
                const u32 lane = threadIdx.x & 31u;
                while (pending) {
                    const int src = __ffs(pending) - 1;
                    pending &= pending - 1u;
                    const u32 d = __shfl_sync(0xFFFFFFFFu, run_dst, src);
                    const u32 cnt = __shfl_sync(0xFFFFFFFFu, run_n, src);
                    const u32 bits = __shfl_sync(0xFFFFFFFFu, run_bits, src);
                    if (lane < cnt) {
                        u32 r[8] = {(bits >> lane) & 1u, 0u, 0u, 0u, 0u, 0u, 0u, 0u};
                        stg256(base + ((size_t)(d + lane) << 1), r);
                    }
                }
            }
        }
        if (info >> 31) {   // INV / POW items of this level (work items of one word)
            for (u32 w = threadIdx.x; w < n; w += blockDim.x) {
                const u32 li = w & bt_mask;
                const uint4 opw = __ldg(&tp.ops[FUSED ? __ldg(&tp.items[lb + (w >> bt_log2)]) : lb + (w >> bt_log2)]);
                const u32 opcode = opw.x & 0xFFu;
                if (opcode != OP_INV && opcode != OP_POW) continue;
                u32 a[8], b[8], r[8];
                load_operand<BP>(a, opw.y, base, plane_base, tp.consts, bt_log2, li);
                load_operand<BP>(b, opw.z, base, plane_base, tp.consts, bt_log2, li);
                exec_slow_op<PRIME, (HAS_CALLS ? 64 : 0) + (BP ? 32 : 0) + (BT + 1) * 2 + (FUSED ? 1 : 0)>(opcode, r, a, b, tp.prime);
                store_slot(r, base, opw.x >> 8, bt_log2, li);
            }
        }
        if (HAS_CALLS && n_calls) {
            const u32 cb = le - n_calls;   // (a call is a work item of one word: item k is tape word items[k])
            for (u32 w = threadIdx.x; w < (n_calls << bt_log2); w += blockDim.x) {
                const u32 li = w & bt_mask;
                const u32 inst = (tile << bt_log2) + li;
                const uint4 opw = __ldg(&tp.ops[FUSED ? __ldg(&tp.items[cb + (w >> bt_log2)]) : cb + (w >> bt_log2)]);
                u32 r[8];
                int e = 0;
                exec_call<PRIME, BP, BT * 2 + (FUSED ? 1 : 0)>(tp, opw.y, base, plane_base, bt_log2, li, r, &e);
                if (e && inst < batch) err[inst] = 1;
                store_slot(r, base, opw.x >> 8, bt_log2, li);
            }
        }
        if (threadIdx.x < ((le_next - le) << bt_log2)) {
            if (FUSED) {   // three independent loads: one round trip
                pre_g0 = __ldg(&tp.items[le + (threadIdx.x >> bt_log2)]);
                pre_g1 = __ldg(&tp.items[le + (threadIdx.x >> bt_log2) + 1]);
                pre = __ldg(&tp.heads[le + (threadIdx.x >> bt_log2)]);
            } else pre = __ldg(&tp.ops[le + (threadIdx.x >> bt_log2)]);
        }
        lb = le;
        le = le_next;
        __syncthreads();
    }
}

#ifndef CW_KERNELS_TAPE_ONLY
// ---- where the values of an instance live --------------------------------------------------------------
// The tape's value store (tile layout, optional bit plane) or - for witnesses handed in by a caller - a dense
// array of 32-byte rows (bt_log2 = 0, n_bitwords = 0, n_slots = row stride, location = wire id).
// A *location* is an operand word of the tape: OPD_BIT | (word * 32 + bit), or a slot id.
struct StoreDev {
    const uint4 *slots;
    const u32 *plane;
    u32 n_slots, n_bitwords, bt_log2, batch;
};
__device__ __forceinline__ const uint4 *store_tile(const StoreDev &S, u32 tile) {
    return S.slots + (((size_t)tile * S.n_slots) << (S.bt_log2 + 1));
}
__device__ __forceinline__ const u32 *store_plane(const StoreDev &S, u32 tile) {
    return S.plane + (((size_t)tile * S.n_bitwords) << S.bt_log2);
}
// (slot values of other kernels' output: read-only here, through the non-coherent path)
__device__ __forceinline__ void load_slot_nc(u32 *v, const uint4 *__restrict__ tile_base, u32 slot, u32 bt_log2, u32 li) {
    if (bt_log2 == 0) {
        ldg256_nc(v, tile_base + ((size_t)slot << 1));
        return;
    }
    size_t i = ((size_t)slot << (bt_log2 + 1)) + li;
    uint4 lo = __ldg(&tile_base[i]);
    uint4 hi = __ldg(&tile_base[i + ((size_t)1 << bt_log2)]);
    v[0] = lo.x; v[1] = lo.y; v[2] = lo.z; v[3] = lo.w;
    v[4] = hi.x; v[5] = hi.y; v[6] = hi.z; v[7] = hi.w;
}
__device__ __forceinline__ void load_loc(u32 *v, const StoreDev &S, const uint4 *__restrict__ tile_base,
                                         const u32 *__restrict__ plane_base, u32 loc, u32 li) {
    if (loc & OPD_BIT) {
        const u32 pos = loc & OPD_BITPOS;
        u256_set_u32(v, (__ldg(&plane_base[((size_t)(pos >> 5) << S.bt_log2) + li]) >> (pos & 31u)) & 1u);
    } else {
        load_slot_nc(v, tile_base, loc, S.bt_log2, li);
    }
}

// ---- dense witness rows on demand: out[i - first][w] = witness entry w of instance i, canonical 32 bytes ----
// The tape keeps the witness where it produced it (resident slots + bit plane); the reference's layout - W
// consecutive 32-byte elements per witness (calcwit.hpp:54-56, main.cpp:328-332) - is materialised only for
// consumers that ask for it (cw_batch_witness_device, .wtns, the plain device->host copy).
__global__ void witness_expand_kernel(StoreDev S, const u32 *__restrict__ wloc, u32 n_witness, u32 first, u32 count,
                                      uint4 *__restrict__ out) {
    const u32 bt_mask = (1u << S.bt_log2) - 1u;
    for (u32 i = blockIdx.y; i < count; i += gridDim.y) {
        const u32 inst = first + i, tile = inst >> S.bt_log2, li = inst & bt_mask;
        const uint4 *tb = store_tile(S, tile);
        const u32 *pb = store_plane(S, tile);
        uint4 *row = out + (size_t)i * n_witness * 2;
        for (u32 w = blockIdx.x * blockDim.x + threadIdx.x; w < n_witness; w += gridDim.x * blockDim.x) {
            u32 v[8];
            load_loc(v, S, tb, pb, __ldg(&wloc[w]), li);
            stg256(row + 2 * (size_t)w, v);
        }
    }
}

// ---- classes of the witness values as they ARE in a batch -----------------------------------------------------
// cls[k] = max over the instances of {0: the value of entry loc[k] is 0 or 1, 1: below 2^64, 2: wider} (merged into what
// cls already holds).  The packed transfer uses observed classes where they are narrower than the proven ones - the
// xor / majority outputs of hash circuits are bits that no range analysis proves - and re-checks every value it packs.
__global__ void __launch_bounds__(256) witness_observe_kernel(StoreDev S, const u32 *__restrict__ loc, u32 n, u32 *__restrict__ cls) {
    const u32 bt_mask = (1u << S.bt_log2) - 1u;
    const u32 n_tiles = (S.batch + bt_mask) >> S.bt_log2;
    const unsigned long long n_items = (unsigned long long)n << S.bt_log2;
    for (u32 tile = blockIdx.y; tile < n_tiles; tile += gridDim.y) {
        const uint4 *tb = store_tile(S, tile);
        for (unsigned long long w = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; w < n_items;
             w += (unsigned long long)gridDim.x * blockDim.x) {
            const u32 li = (u32)w & bt_mask, inst = (tile << S.bt_log2) + li;
            if (inst >= S.batch) continue;
            const u32 k = (u32)(w >> S.bt_log2);
            u32 x[8];
            load_slot_nc(x, tb, __ldg(&loc[k]), S.bt_log2, li);
            const u32 c = (x[2] | x[3] | x[4] | x[5] | x[6] | x[7]) ? 2u : ((x[1] | (x[0] & ~1u)) ? 1u : 0u);
            if (c > cls[k]) atomicMax(&cls[k], c);
        }
    }
}

// ---- packed witness for the device->host transfer -------------------------------------------------------
// Most witness entries of real circuits are bits or 64-bit limbs.  The lowering knows an upper bound of every
// entry's bit length (range analysis); entries proven to be one bit travel as one bit, entries proven <= 64 bits
// as 8 bytes, the rest as 32 bytes, and the host expands them back to the canonical 32-byte rows.  Per-instance
// packed record (32-bit words):
//     [the instance's bit plane, as it is][bits outside the plane, 32 per word][u64 entries][full entries]
// Values outside the plane are re-checked against their class: a violation raises `flag` and the caller falls
// back to the dense copy.  (Plane bits are single bits by construction.)
__global__ void witness_pack_kernel(StoreDev S, const u32 *__restrict__ bit_loc, u32 n_bits,
                                    const u32 *__restrict__ u64_loc, u32 n_u64, const u32 *__restrict__ full_loc,
                                    u32 n_full, u32 *__restrict__ packed, size_t words_per_inst, u32 first, u32 count,
                                    int *__restrict__ flag) {
    const u32 n_bit_words = (n_bits + 31u) >> 5;
    const size_t items = (size_t)S.n_bitwords + n_bit_words + n_u64 + n_full;
    const u32 bt_mask = (1u << S.bt_log2) - 1u;
    for (u32 i = blockIdx.y; i < count; i += gridDim.y) {
        const u32 inst = first + i, tile = inst >> S.bt_log2, li = inst & bt_mask;
        const uint4 *tb = store_tile(S, tile);
        const u32 *pb = store_plane(S, tile);
        u32 *out = packed + (size_t)i * words_per_inst;
        for (size_t it = blockIdx.x * (size_t)blockDim.x + threadIdx.x; it < items; it += (size_t)gridDim.x * blockDim.x) {
            if (it < S.n_bitwords) {
                out[it] = __ldg(&pb[(it << S.bt_log2) + li]);
                continue;
            }
            u32 *o = out + S.n_bitwords;
            size_t k = it - S.n_bitwords;
            if (k < n_bit_words) {
                u32 word = 0, bad = 0;
                const u32 j0 = (u32)k << 5;
#pragma unroll 4
                for (u32 j = 0; j < 32u; ++j) {
                    if (j0 + j < n_bits) {
                        u32 x[8];
                        load_slot_nc(x, tb, __ldg(&bit_loc[j0 + j]), S.bt_log2, li);
                        bad |= x[1] | x[2] | x[3] | x[4] | x[5] | x[6] | x[7] | (x[0] & ~1u);
                        word |= (x[0] & 1u) << j;
                    }
                }
                o[k] = word;
                if (bad) *flag = 1;
            } else if (k < (size_t)n_bit_words + n_u64) {
                const u32 e = (u32)(k - n_bit_words);
                u32 x[8];
                load_slot_nc(x, tb, __ldg(&u64_loc[e]), S.bt_log2, li);
                if (x[2] | x[3] | x[4] | x[5] | x[6] | x[7]) *flag = 1;
                o[n_bit_words + 2 * (size_t)e] = x[0];
                o[n_bit_words + 2 * (size_t)e + 1] = x[1];
            } else {
                const u32 e = (u32)(k - n_bit_words - n_u64);
                u32 x[8];
                load_slot_nc(x, tb, __ldg(&full_loc[e]), S.bt_log2, li);
                u32 *oo = o + n_bit_words + 2 * (size_t)n_u64 + 8 * (size_t)e;
#pragma unroll
                for (int q = 0; q < 8; ++q) oo[q] = x[q];
            }
        }
    }
}

// ---- R1CS check: A.w * B.w == C.w for every row and instance ------------------------------------
// Compiled CSR: row_ptr[3m+1] (A, B, C blocks per row) over 16-byte term records
//     {location of the wire's value, coefficient dictionary index, kind word, absorbed boolean row or ~0}
// kind word: bits 0-7  : 0 general (Montgomery product with dictM), 1 = +1, 2 = -1, 3 = +2^k, 4 = -2^k, with k in
//                        bits 8-15;  5 / 6 = +- RUN: `count` consecutive bits of ONE bit-plane word, whose
//                        coefficients are consecutive powers of two - the recomposition sums of range checks,
//                        65 terms in the file, are two such records: value = ((word >> first) & mask) << k,
//                        first in bits 16-20, count - 1 in bits 21-25, location = word index.
//
// Work decomposition: work item = (row, instance), instance fastest inside a tile, rows visited through `perm`,
// a host-side stable sort of the rows by structure (term counts and coefficient kinds).  With 32-instance tiles
// a warp is ONE row for 32 instances: the term records are broadcasts, the witness loads 512 contiguous bytes,
// nothing diverges but the data-dependent product skips; with one-instance tiles a warp is 32 rows of equal
// structure.  blockIdx.y walks the tiles.
//
// Arithmetic: +-1 coefficients are modular add/sub; +-2^k coefficients shift the witness value when
// the shifted value provably stays below q (runtime check of the value's bit length; a Montgomery
// product otherwise); the row product a*b is skipped when a or b is 0, 1 or -1.
struct R1csDev {
    const unsigned long long *row_ptr;
    const uint4 *terms;
    const uint4 *dictM;
    const u32 *perm;
    u32 n_rows;  // rows in perm
    u32 prime;   // index into c_fr (PRIME = -1 build)
};

// Lazy reduction: most terms of circom constraints are bits / small values times +-1 or +-2^k (boolean logic, the
// recomposition sums of range checks, carries).  Such a term is an integer below 2^112; the terms of one linear
// combination are summed as plain 128-bit integers (positive and negative coefficients apart) and enter the modular
// accumulator ONCE, instead of one 256-bit modular addition per term.
__device__ __forceinline__ void acc128_add(unsigned long long &lo, unsigned long long &hi, u32 v, u32 sh) {
    // (lo, hi) += v << sh, 0 <= sh <= 80
    unsigned long long l, h;
    if (sh < 64u) {
        l = (unsigned long long)v << sh;
        h = sh > 32u ? ((unsigned long long)v >> (64u - sh)) : 0ull;
    } else {
        l = 0ull;
        h = (unsigned long long)v << (sh - 64u);
    }
    lo += l;
    hi += h + (lo < l ? 1ull : 0ull);
}

template <int PRIME>
__device__ __forceinline__ void r1cs_lc(u32 *acc, const R1csDev &R, unsigned long long b, unsigned long long e,
                                        const StoreDev &S, const uint4 *__restrict__ tb, const u32 *__restrict__ pb,
                                        u32 li, const FrParams &P, unsigned long long *__restrict__ first_bad_inst) {
    u256_set_u32(acc, 0);
    unsigned long long plo = 0, phi = 0, nlo = 0, nhi = 0;
    // 2^16 terms below 2^112 cannot overflow 128 bits; the sum enters the accumulator unreduced, so it must stay below q
    // (every 256-bit prime; not goldilocks, whose terms take the modular path)
    const bool lazy = e - b < 65536ull && P.qbits > 130u;
    for (unsigned long long k = b; k < e; ++k) {
        const uint4 term = __ldg(&R.terms[k]);
        const u32 loc = term.x, ci = term.y, kw = term.z, brow = term.w;
        const u32 kd = kw & 0xFF, sh = (kw >> 8) & 0xFF;
        u32 x[8], t[8];
        bool neg = (kd == 2) || (kd == 4) || (kd == 6);
        if (kd >= 5) {
            // run of plane bits times consecutive powers of two: an integer below 2^(sh + count) < q
            const u32 first = (kw >> 16) & 31u, cnt = ((kw >> 21) & 31u) + 1u;
            const u32 word = (__ldg(&pb[((size_t)loc << S.bt_log2) + li]) >> first) & (cnt >= 32u ? 0xFFFFFFFFu : ((1u << cnt) - 1u));
            if (lazy && sh <= 80u) {
                if (neg) acc128_add(nlo, nhi, word, sh);
                else acc128_add(plo, phi, word, sh);
                continue;
            }
            const u32 wd = sh >> 5, s = sh & 31u;
            const u32 l = word << s, h = s ? (word >> (32u - s)) : 0u;
#pragma unroll
            for (int i = 0; i < 8; ++i) x[i] = ((u32)i == wd) ? l : (((u32)i == wd + 1u) ? h : 0u);
        } else {
            load_loc(x, S, tb, pb, loc, li);
            const u32 upper = x[1] | x[2] | x[3] | x[4] | x[5] | x[6] | x[7];
            // the boolean constraint x*(x-1) = 0 of this wire is checked here, while its value is in registers
            if (brow != 0xFFFFFFFFu && (upper || x[0] > 1u)) atomicMin(first_bad_inst, (unsigned long long)brow);
            if (lazy && !upper && kd >= 1u && (kd <= 2u || sh <= 80u)) {   // a 32-bit value times +-1 / +-2^sh
                if (neg) acc128_add(nlo, nhi, x[0], kd <= 2u ? 0u : sh);
                else acc128_add(plo, phi, x[0], kd <= 2u ? 0u : sh);
                continue;
            }
            if (kd >= 3) {
                if (!upper && sh + 32u < P.qbits) {  // x < 2^32: x * 2^sh < 2^(qbits-1) < q, placed without a reduction
                    const u32 wd = sh >> 5, s = sh & 31u;
                    const u32 l = x[0] << s, h = s ? (x[0] >> (32u - s)) : 0u;
#pragma unroll
                    for (int i = 0; i < 8; ++i) x[i] = ((u32)i == wd) ? l : (((u32)i == wd + 1u) ? h : 0u);
                } else if (u256_bitlen_dev(x) + sh < P.qbits) {   // x * 2^sh < 2^(qbits-1) < q : plain shift
                    u32 y[8];
                    u256_shl(y, x, sh);
                    u256_set(x, y);
                } else {
                    u32 cm[8], p[8];
                    load_const(cm, R.dictM, ci);
                    fr_mont_mul(p, cm, x, P);           // (cR) * x / R = c*x, sign included
                    u256_set(x, p);
                    neg = false;
                }
            } else if (kd == 0) {
                u32 cm[8], p[8];
                load_const(cm, R.dictM, ci);
                fr_mont_mul(p, cm, x, P);
                u256_set(x, p);
            }
        }
        if (neg) fr_sub(t, acc, x, P);
        else fr_add(t, acc, x, P);
        u256_set(acc, t);
    }
    if (plo | phi) {
        u32 v[8] = {(u32)plo, (u32)(plo >> 32), (u32)phi, (u32)(phi >> 32), 0u, 0u, 0u, 0u}, t[8];
        fr_add(t, acc, v, P);
        u256_set(acc, t);
    }
    if (nlo | nhi) {
        u32 v[8] = {(u32)nlo, (u32)(nlo >> 32), (u32)nhi, (u32)(nhi >> 32), 0u, 0u, 0u, 0u}, t[8];
        fr_sub(t, acc, v, P);
        u256_set(acc, t);
    }
}

// a * b == c for canonical a, b, c; the product is skipped for a or b in {0, 1, -1}
__device__ __forceinline__ bool r1cs_row_holds(const u32 *a, const u32 *b, const u32 *c, const FrParams &P) {
    bool ok;
    u32 ha = a[1] | a[2] | a[3] | a[4] | a[5] | a[6] | a[7];
    u32 hb = b[1] | b[2] | b[3] | b[4] | b[5] | b[6] | b[7];
    if ((!ha && a[0] == 0) || (!hb && b[0] == 0)) ok = u256_is_zero(c);
    else if (!ha && a[0] == 1) ok = u256_eq(b, c);
    else if (!hb && b[0] == 1) ok = u256_eq(a, c);
    else if (a[0] + 1u == P.q[0] && a[1] == P.q[1] && a[2] == P.q[2] && a[3] == P.q[3] && a[4] == P.q[4] &&
             a[5] == P.q[5] && a[6] == P.q[6] && a[7] == P.q[7]) {
        // a = -1: rows `out <== x*y` are stored as (-x) * y = -out (the reference's normal form), so a
        // bit-valued x = 1 lands here: -b == c
        u32 s[8];
        fr_add(s, b, c, P);
        ok = u256_is_zero(s);
    } else {
        u32 ab[8], c1[8];
        fr_mont_mul(ab, a, b, P);  // a*b/R
        fr_from_mont(c1, c, P);    // c/R
        ok = u256_eq(ab, c1);
    }
    return ok;
}

// MINB = CTAs per SM the register budget is cut for (r01 measurements on the bench circuit, long rows, bound by
// memory latency: 3 -> 16.4 ms, 4 -> 13.7 ms, 5 -> 13.0 ms, 6 -> 17.0 ms per 1024 instances; circuits of short
// rows prefer the unspilled build); the host picks by the mean row length.
// EVAL: also leave A.w, B.w, C.w of every row in device memory ([instance][row] 32-byte elements) for a prover
struct EvalOut {
    uint4 *a = nullptr, *b = nullptr, *c = nullptr;
    unsigned long long m = 0;  // rows per instance
};
// FILTER: the rows of R.perm are the integer rows (r1cs_small_kernel below); only those it marked in `filter` are decided
template <int PRIME, int MINB, bool EVAL, bool FILTER>
__global__ void __launch_bounds__(256, MINB) r1cs_check_kernel(R1csDev R, StoreDev S, unsigned long long *__restrict__ first_bad,
                                                         EvalOut out, const u32 *__restrict__ filter) {
    const FrParams &P = CW_FR(PRIME, R.prime);
    const u32 bt_mask = (1u << S.bt_log2) - 1u;
    const u32 n_tiles = (S.batch + bt_mask) >> S.bt_log2;
    const unsigned long long n_items = (unsigned long long)R.n_rows << S.bt_log2;
    for (u32 tile = blockIdx.y; tile < n_tiles; tile += gridDim.y) {
        const uint4 *tb = store_tile(S, tile);
        const u32 *pb = store_plane(S, tile);
        for (unsigned long long w = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; w < n_items;
             w += (unsigned long long)gridDim.x * blockDim.x) {
            const u32 li = (u32)w & bt_mask, inst = (tile << S.bt_log2) + li;
            if (inst >= S.batch) continue;
            if (FILTER) {
                if (!filter[(R.n_rows + 31u) >> 5]) return;   // the word after the bitmap: no row was marked at all
                const u32 k = (u32)(w >> S.bt_log2);
                if (!((filter[k >> 5] >> (k & 31u)) & 1u)) continue;   // (written by the kernel before this one: plain load)
            }
            const u32 row = __ldg(&R.perm[w >> S.bt_log2]);
            const unsigned long long p0 = __ldg(&R.row_ptr[3 * (size_t)row]), p1 = __ldg(&R.row_ptr[3 * (size_t)row + 1]),
                                     p2 = __ldg(&R.row_ptr[3 * (size_t)row + 2]), p3 = __ldg(&R.row_ptr[3 * (size_t)row + 3]);
            u32 a[8], b[8], c[8];
            r1cs_lc<PRIME>(a, R, p0, p1, S, tb, pb, li, P, &first_bad[inst]);
            r1cs_lc<PRIME>(b, R, p1, p2, S, tb, pb, li, P, &first_bad[inst]);
            r1cs_lc<PRIME>(c, R, p2, p3, S, tb, pb, li, P, &first_bad[inst]);
            if (EVAL) {
                const size_t o = ((size_t)inst * out.m + row) * 2;
                stg256(out.a + o, a);
                stg256(out.b + o, b);
                stg256(out.c + o, c);
            }
            if (!r1cs_row_holds(a, b, c, P)) atomicMin(&first_bad[inst], (unsigned long long)row);
        }
    }
}

// ---- integer rows (r1cs_small.h): rows that are small by shape, decided over the integers ----------------------
// Work item = (row of R.perm = the small rows, instance), as in r1cs_check_kernel; the rows are read from their own term
// list: groups of 32 rows with uniform term counts, 8-byte records interleaved inside a group (one-instance tiles: a warp
// is a group, a record load is one 256-byte line, the loops do not diverge; 32-instance tiles: a warp is one row).  Per
// term: the record, the value (32 bytes, or a plane word), a shift and a 64-bit add - no field arithmetic, six
// 64-bit accumulators instead of three 8-limb ones.  A value of 2^16 or more marks the row in `wide` (one bit per row of
// R.perm, whichever instance) and the general kernel decides it afterwards.
struct R1csSmallDev {
    const uint2 *groups;   // {first record, n0 | n1 << 8 | n2 << 16}
    const uint2 *recs;     // R1csSmallRec
    const u32 *brow;       // boolean row of a record with SM_BROW
};
template <bool BT0>
__global__ void __launch_bounds__(256, 6) r1cs_small_kernel(R1csDev R, R1csSmallDev G, StoreDev S, unsigned long long *__restrict__ first_bad,
                                                            u32 *__restrict__ wide) {
    const u32 bt_log2 = BT0 ? 0u : S.bt_log2;
    const u32 bt_mask = (1u << bt_log2) - 1u;
    const u32 n_tiles = (S.batch + bt_mask) >> bt_log2;
    const unsigned long long n_items = (unsigned long long)R.n_rows << bt_log2;
    for (u32 tile = blockIdx.y; tile < n_tiles; tile += gridDim.y) {
        const uint4 *tb = store_tile(S, tile);
        const u32 *pb = store_plane(S, tile);
        for (unsigned long long w = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; w < n_items;
             w += (unsigned long long)gridDim.x * blockDim.x) {
            const u32 li = (u32)w & bt_mask, inst = (tile << bt_log2) + li;
            if (inst >= S.batch) continue;
            const u32 k = (u32)(w >> bt_log2);
            const uint2 hdr = __ldg(&G.groups[k >> 5]);
            u32 at = hdr.x + (k & 31u);
            long long v[3];
            u32 is_wide = 0u;
#pragma unroll
            for (int blk = 0; blk < 3; ++blk) {
                const u32 n = (hdr.y >> (8 * blk)) & 0xFFu;
                unsigned long long pos = 0ull, neg = 0ull;
                for (u32 t = 0; t < n; ++t, at += 32u) {
                    const uint2 rec = __ldg(&G.recs[at]);
                    if (rec.x & (SM_RUN | SM_BIT)) {
                        if (rec.x & SM_RUN) {
                            r1cs_small_acc_run(pos, neg, rec.x, rec.y, __ldg(&pb[((size_t)(rec.x & SM_LOC) << bt_log2) + li]));
                        } else {
                            const u32 p = rec.x & SM_BITPOS;
                            r1cs_small_acc(pos, neg, is_wide, rec.x, rec.y, (__ldg(&pb[((size_t)(p >> 5) << bt_log2) + li]) >> (p & 31u)) & 1u, 0u);
                        }
                    } else {
                        u32 x[8];
                        load_slot_nc(x, tb, rec.x & OPD_SLOT, bt_log2, li);
                        const u32 upper = x[1] | x[2] | x[3] | x[4] | x[5] | x[6] | x[7];
                        // the boolean constraint x*(x-1) = 0 of this wire rides on the term, as in the general kernel
                        if ((rec.x & SM_BROW) && (upper || x[0] > 1u)) atomicMin(&first_bad[inst], (unsigned long long)__ldg(&G.brow[at]));
                        r1cs_small_acc(pos, neg, is_wide, rec.x, rec.y, x[0], upper);
                    }
                }
                v[blk] = (long long)(pos - neg);
            }
            if (is_wide) {
                atomicOr(&wide[k >> 5], 1u << (k & 31u));
                wide[(R.n_rows + 31u) >> 5] = 1u;   // "some row is marked" (every writer stores the same value)
            } else if (!r1cs_small_holds(v[0], v[1], v[2])) atomicMin(&first_bad[inst], (unsigned long long)__ldg(&R.perm[k]));
        }
    }
}

// boolean rows x*(x-1) = 0 that no general row absorbs: the witness value must be 0 or 1.  Work item = (boolean
// row, instance); the wires of consecutive boolean rows are consecutive witness entries.  (Rows whose wire is a
// bit of the bit plane are not listed at all: a stored bit is 0 or 1.)
__global__ void __launch_bounds__(256) r1cs_bool_kernel(const u32 *__restrict__ loc, const u32 *__restrict__ rows,
                                                        u32 n_bool, StoreDev S, unsigned long long *__restrict__ first_bad) {
    const u32 bt_mask = (1u << S.bt_log2) - 1u;
    const u32 n_tiles = (S.batch + bt_mask) >> S.bt_log2;
    const unsigned long long n_items = (unsigned long long)n_bool << S.bt_log2;
    for (u32 tile = blockIdx.y; tile < n_tiles; tile += gridDim.y) {
        const uint4 *tb = store_tile(S, tile);
        for (unsigned long long w = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; w < n_items;
             w += (unsigned long long)gridDim.x * blockDim.x) {
            const u32 li = (u32)w & bt_mask, inst = (tile << S.bt_log2) + li;
            if (inst >= S.batch) continue;
            const u32 k = (u32)(w >> S.bt_log2);
            u32 x[8];
            load_slot_nc(x, tb, __ldg(&loc[k]), S.bt_log2, li);
            const u32 rest = x[1] | x[2] | x[3] | x[4] | x[5] | x[6] | x[7];
            if (rest || x[0] > 1u) atomicMin(&first_bad[inst], (unsigned long long)__ldg(&rows[k]));
        }
    }
}

// ---- batched single field op (parity tests of the device Fr_* equivalents) ---------------------
// canonical in / canonical out; the kernel applies the same representation rules as the lowering
template <int PRIME>
__global__ void fr_batch_op_kernel(int op, const uint4 *__restrict__ A, const uint4 *__restrict__ B,
                                   const uint4 *__restrict__ C, uint4 *__restrict__ Rr, size_t n,
                                   int *__restrict__ err, u32 prime_rt) {
    const FrParams &P = CW_FR(PRIME, prime_rt);
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        u32 a[8], b[8] = {0, 0, 0, 0, 0, 0, 0, 0}, c[8] = {0, 0, 0, 0, 0, 0, 0, 0}, r[8];
        load_const(a, A, (u32)i);
        if (B) load_const(b, B, (u32)i);
        if (C) load_const(c, C, (u32)i);
        int e = 0;
        if (op == OP_MUL) {  // canonical x canonical: convert one side
            u32 am[8];
            fr_to_mont(am, a, P);
            fr_mont_mul(r, am, b, P);
        } else if (op == 2 /* DIV */) {
            u32 bm[8], im[8];
            fr_to_mont(bm, b, P);
            fr_inv_mont(im, bm, P);
            fr_mont_mul(r, im, a, P);
        } else if (op == OP_POW) {
            u32 am[8], rm[8];
            fr_to_mont(am, a, P);
            fr_pow_mont(rm, am, b, P);
            fr_from_mont(r, rm, P);
        } else if (op == OP_INV) {
            u32 am[8], rm[8];
            fr_to_mont(am, a, P);
            fr_inv_mont(rm, am, P);
            fr_from_mont(r, rm, P);
        } else if (op == OP_SELECT) {
            bool t = !u256_is_zero(c);
            for (int k = 0; k < 8; ++k) r[k] = t ? a[k] : b[k];
        } else {
            fr_exec((u32)op, r, a, b, 0, P, e);
        }
        if (e) err[0] = 1;
        Rr[2 * i] = make_uint4(r[0], r[1], r[2], r[3]);
        Rr[2 * i + 1] = make_uint4(r[4], r[5], r[6], r[7]);
    }
}

// ---- Montgomery-multiplication throughput probe ------------------------------------------------
template <int PRIME>
__global__ void fr_mul_bench_kernel(uint4 *__restrict__ data, size_t n, int iters) {
    const FrParams &P = c_fr[PRIME];
    size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
    if (i >= n) return;
    u32 x[8], y[8];
    load_const(x, data, (u32)i);
    u256_set(y, x);
    y[0] ^= 0x9E3779B9u & 0x0FFFFFFFu;
#pragma unroll 1
    for (int k = 0; k < iters; ++k) {
        u32 t[8];
        fr_mont_mul(t, x, y, P);
        u256_set(x, t);
    }
    data[2 * i] = make_uint4(x[0], x[1], x[2], x[3]);
    data[2 * i + 1] = make_uint4(x[4], x[5], x[6], x[7]);
}

#endif  // CW_KERNELS_TAPE_ONLY

}  // namespace cw
