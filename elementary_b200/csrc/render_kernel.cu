// render_kernel.cu — K1: the fused render-sequence kernel for sm_100a.
//
// Replaces, for every voice at once, the reference's per-block walk
//   GraphRenderSequence::process -> RootRenderSequence::process -> node->process(BlockContext)
//   (runtime/elem/GraphRenderSequence.h:268-309, :212-232)
//
// Work decomposition.  One warp owns one *voice tile* of L voices (L = 1..32, chosen by the host so that few
// voices still fill the machine) for the whole block.  The block is cut into sample tiles of T samples with
// E = L*T = 32*NITER elements; a node output for one tile is a shared-memory slot [T][L] (element e = t*L + v)
// — the reference's 2 KB-per-node block buffers never exist.  For each sample tile the warp interprets the
// compiled render program (program.h) op by op, warp-uniformly:
//   * stateless ops (chains of element-wise math, fades, table lookups, prewarp, svf coefficient math, delay
//     lines whose read head is outside the tile, ...) run with ALL 32 lanes over the E elements of the tile —
//     lanes are voices when L = 32 and consecutive samples of one voice when L = 1, the code is the same;
//   * true recurrences (phasor, svf tick, pole, biquad, ...) run serially over the T samples inside the lane that
//     owns the voice (lanes < L), state in registers, carried across tiles in the warp's shared-memory state
//     area and across blocks in HBM rows.
// So with few voices the time axis of everything that is not a recurrence is spread over the lanes, and with
// many voices every lane is a voice; results are identical either way because no floating-point operation is
// re-associated.  Tile geometry (NITER, log2 L) is a template parameter so that all slot addressing is
// immediate-offset arithmetic.
//
// Numerics: compiled with -fmad=false so a*b+c is two roundings exactly like the reference built with
// -ffp-contract=off; svf/svfshelf/mm1p/prewarp coefficient math is evaluated in double like the reference
// (filters/SVF.h:72-80); no -use_fast_math, no flush-to-zero.
//
// HBM layout (per voice group): rows[row][Vpad] f32 (params, scalar state; a double state is two rows viewed
// as double[Vpad]); delay rings / tap buffers [tile][pos][L] so the lanes of a warp touch one contiguous line.

#ifndef __CUDACC_RTC__
#include <cuda_runtime.h>
#endif
#include "rtc_compat.h"
#include "program.h"
#include "kernels.h"

namespace eb {

namespace {

constexpr float kEps = FLT_EPSILON;
#ifndef EB_SVF_SCAN_MAX_L
#define EB_SVF_SCAN_MAX_L 4      // tiles of up to this many voices run the svf tick as a warp scan (render_ops.inc, OP_SVF)
#endif
constexpr unsigned FULL = 0xFFFFFFFFu;

// Everything the interpreter touches per sample lives in the CTA's dynamic shared memory.  Addresses into it are kept as 32-bit
// element indices (SP), not 64-bit generic pointers: half the registers per address, 32-bit address arithmetic, and LDS/STS
// with immediate offsets — the kernel runs at a 64-register budget where every live pointer pair costs a spill or a
// re-computation (profiles/r01_o_*: a fifth of all instructions were re-materialised address arithmetic).
extern __shared__ __align__(16) float g_smem[];
struct SP {
    int i;
    __device__ __forceinline__ float& operator[](int k) const { return g_smem[i + k]; }
    __device__ __forceinline__ SP operator+(int d) const { return SP{i + d}; }
    __device__ __forceinline__ float* ptr() const { return g_smem + i; }
};

// ---- TMA (1-D bulk async copy) + mbarrier: stages a program's wavetable HBM -> shared memory once per CTA (SASS: UBLKCP)
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t) __cvta_generic_to_shared(p); }
// ---- cp.async (LDGSTS): global -> shared copies that do not hold up the issuing warp; completed by cp.async.wait_all
__device__ __forceinline__ void cp_async_4(uint32_t dst, const void* src) { asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst), "l"(src) : "memory"); }
__device__ __forceinline__ void cp_async_8(uint32_t dst, const void* src) { asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst), "l"(src) : "memory"); }

__device__ __forceinline__ void stage_table_tma(const float* src, int floats, float* dst, uint64_t* bar) {
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(bar)) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        const uint32_t bytes = (uint32_t) floats * 4u;
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
    }
    __syncthreads();            // the barrier is initialised before anyone polls it
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "TBL_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], 0;\n"
        "@P1 bra TBL_DONE;\n"
        "bra TBL_WAIT;\n"
        "TBL_DONE:\n"
        "}" ::"r"(smem_u32(bar)) : "memory");
}

// An operand is a shared-memory address plus strides: a slot advances 32 floats per element slice k and L floats
// per sample; a parameter row (one float per voice) has stride 0 in both.
struct Opnd {
    SP p;
    int stride;    // per element slice k (stateless ops)
    int tstride;   // per sample t (owner-lane recurrences)
};

#define LDE(o, k) ((o).p[(k) * (o).stride])
#define LDT(o, t) ((o).p[(t) * (o).tstride])
// the same read by ANY lane of the voice column (an operand pointer is set up for the owner lane = lane vlane of the column;
// parameter operands, stride 0, already point at the column)
#define LDC(o, t) ((o).p[(t) * (o).tstride + ((o).stride ? (vlane - lane) : 0)])
#ifndef EB_RECUR_BROADCAST
#define EB_RECUR_BROADCAST 0      /* narrow-tile recurrences: 0 = operands by shuffle from the lane that holds them, 1 = broadcast reads of the slots (A/B: profiles/r02_m_*) */
#endif
#ifndef EB_INTERP_PREFETCH
#define EB_INTERP_PREFETCH 0      /* interpreter loop: 1 = next op's header + operand words loaded while the current op runs (A/B: profiles/r02_m_*) */
#endif

__device__ __forceinline__ float clampf(float v, float lo, float hi) { return (v < lo) ? lo : ((hi < v) ? hi : v); }
__device__ __forceinline__ double clampd(double v, double lo, double hi) { return (v < lo) ? lo : ((hi < v) ? hi : v); }
__device__ __forceinline__ float stdmin(float a, float b) { return (b < a) ? b : a; }   // std::min
__device__ __forceinline__ float stdmax(float a, float b) { return (a < b) ? b : a; }   // std::max

// helpers/Change.h:12-32
__device__ __forceinline__ float change_tick(float& lastIn, float xn) {
    const float dt = xn - lastIn;
    lastIn = xn;
    return (dt > 0.0f) ? 1.0f : ((dt < 0.0f) ? -1.0f : 0.0f);
}

__device__ __forceinline__ double bits_to_double(uint32_t lo, uint32_t hi) {
    return __longlong_as_double((long long) ((uint64_t) lo | ((uint64_t) hi << 32)));
}

// Cold or bulky libm entry points are kept out of line: the kernel is one big interpreter and its instruction
// footprint decides how often warps stall on instruction fetch (ncu: stall_no_instruction).  sinf/tanhf and the
// cheap rounding/abs/sqrt ops stay inline.
__device__ __noinline__ double tan_f64(double x) { return tan(x); }
__device__ __noinline__ double pow_f64(double x, double y) { return pow(x, y); }
__device__ __noinline__ float cos_f32(float x) { return cosf(x); }
__device__ __noinline__ float tan_f32(float x) { return tanf(x); }
__device__ __noinline__ float asinh_f32(float x) { return asinhf(x); }
__device__ __noinline__ float log_f32(float x) { return logf(x); }
__device__ __noinline__ float log10_f32(float x) { return log10f(x); }
__device__ __noinline__ float log2_f32(float x) { return log2f(x); }
__device__ __noinline__ float exp_f32(float x) { return expf(x); }
__device__ __noinline__ float pow_f32(float x, float y) { return powf(x, y); }
__device__ __noinline__ float fmod_f32(float x, float y) { return fmodf(x, y); }
// Out-of-line twins of the math that is inline in the hot geometries, for the 128-sample one-voice tiles (NITER = 4, L = 1): there a
// FOR_K loop is four unrolled copies of its body, and the many-graphs launch is bound by instruction FETCH (about one instruction per
// clock and SM once the interpreter's hot set has outgrown the 32 KB L1.5 instruction cache) — four calls to one copy of sinf fetch
// a quarter of the instructions of four inlined copies.
__device__ __noinline__ float sin_f32_ool(float x) { return sinf(x); }
__device__ __noinline__ float tanh_f32_ool(float x) { return tanhf(x); }
__device__ __noinline__ double ddiv_ool(double a, double b) { return a / b; }

// 1/b and a/b in double to ~1 ulp: MUFU.RCP64H seed (rcp.approx.ftz.f64, >= 20 good bits) + two Newton steps (+ one residual
// correction for the quotient), 6-9 instructions instead of the ~30 of the IEEE-exact division sequence with its slow path.
// Only used inside the svf coefficient math, whose results are rounded to float at the output: an ulp of double (1e-16) is nine
// orders of magnitude below what a float sample resolves (same reasoning as the FMA contraction of the tick).  The profile
// (profiles/r01_o_*) had the three divisions of SVF.h:72-80 at 10 % of all instructions of a SUBSYNTH32 voice.
__device__ __forceinline__ double rcp_fast(double b) {
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(b));
    double e = fma(-b, r, 1.0);
    r = fma(r, e, r);
    e = fma(-b, r, 1.0);
    return fma(r, e, r);
}
__device__ __forceinline__ double div_fast(double a, double b) {
    const double r = rcp_fast(b);
    const double q = a * r;
    return fma(fma(-b, q, a), r, q);
}

// tan(x) for 0 <= x < pi/2, the only range the svf family ever asks for (fc is clamped to [20, sr/2.0001] before
// g = tan(pi*fc/sr), SVF.h:75).  Reduce to y in [0, pi/4] by the co-function identity and use 7-term Taylor sums
// for sin and cos: max relative error 5.2e-13 over the whole clamped range (checked against glibc tan on 3M points;
// 8 terms would give 1.8e-15) — nine orders of magnitude below what a float output sample can resolve — at half the
// instructions of the general-purpose tan(), with no branch and no argument-reduction slow path.
__device__ __forceinline__ double tan_quarter_wave(double x) {
    const bool big = x > 0.78539816339744831;
    const double y = big ? ((1.5707963267948966 - x) + 6.123233995736766e-17) : x;
    const double y2 = y * y;
    double s = 1.0 / 6227020800.0;                    // sin: y - y^3/3! + y^5/5! - ... + y^13/13!
    s = fma(s, y2, -1.0 / 39916800.0);
    s = fma(s, y2, 1.0 / 362880.0);
    s = fma(s, y2, -1.0 / 5040.0);
    s = fma(s, y2, 1.0 / 120.0);
    s = fma(s, y2, -1.0 / 6.0);
    s = fma(s * y2, y, y);                             // y + y^3 * poly(y^2)
    double c = 1.0 / 479001600.0;                      // cos: 1 - y^2/2! + ... + y^12/12!
    c = fma(c, y2, -1.0 / 3628800.0);
    c = fma(c, y2, 1.0 / 40320.0);
    c = fma(c, y2, -1.0 / 720.0);
    c = fma(c, y2, 1.0 / 24.0);
    c = fma(c, y2, -0.5);
    c = fma(c, y2, 1.0);
    return big ? div_fast(c, s) : div_fast(s, c);
}

// svf coefficients of one sample (SVF.h:72-80) out of line, for the 128-sample one-voice tiles (see sin_f32_ool): g, a1 = 1/(1 + g (g + k))
__device__ __noinline__ void svf_coefs_ool(double x, double kq, double& g, double& a1) {
    g = tan_quarter_wave(x);
    a1 = rcp_fast(fma(g, g + kq, 1.0));
}

// Math.h:30-57,128-188 — fn(x, y) for the binary and reducing node families
__device__ __forceinline__ float binary_apply(uint32_t fn, float x, float y) {
    switch (fn) {
        case F_ADD: return x + y;
        case F_SUB: return x - y;
        case F_MUL: return x * y;
        case F_DIV: return (y == 0.0f) ? 0.0f : x / y;
        case F_MOD: return fmod_f32(x, y);
        case F_MIN: return stdmin(x, y);
        case F_MAX: return stdmax(x, y);
        case F_LE:  return (x < y) ? 1.0f : 0.0f;
        case F_LEQ: return (x <= y) ? 1.0f : 0.0f;
        case F_GE:  return (x > y) ? 1.0f : 0.0f;
        case F_GEQ: return (x >= y) ? 1.0f : 0.0f;
        case F_POW: return (x < 0.0f && y != floorf(y)) ? 0.0f : pow_f32(x, y);
        case F_EQ:  return (fabsf(x - y) <= kEps) ? 1.0f : 0.0f;
        case F_AND: return (fabsf(1.0f - x) <= kEps && fabsf(1.0f - y) <= kEps) ? 1.0f : 0.0f;
        default:    return (fabsf(1.0f - x) <= kEps || fabsf(1.0f - y) <= kEps) ? 1.0f : 0.0f;
    }
}

__host__ __device__ constexpr int ilog2(int x) { return x <= 1 ? 0 : 1 + ilog2(x >> 1); }

} // namespace


// =========================================================================================================
// Sequencing / control nodes (SURVEY.md §8f N3).  They are rare in a render program and bulky, so each lives in
// its own out-of-line function: the interpreter's hot loop keeps its instruction footprint.  All of them are true
// recurrences (edge detectors + counters), run by the lane that owns the voice.
struct CtlCtx {
    float* sst;              // the warp's state area [row][L]
    const float* spar;       // the warp's parameter area [row][L]
    float* slots;            // the warp's slot area
    float* outT;             // owner lane, sample t: outT[t * L]
    const uint32_t* opnds;   // operand words, then immediates
    uint64_t ptr;
    long long sampleTime;    // of sample 0 of this tile
    uint32_t sidx, aux0, aux1, mode, nopnd;
    int cnt, s0, lane, vlane;
};

template <int L, int E>
__device__ __forceinline__ Opnd ctl_decode(const CtlCtx& c, uint32_t w) {
    Opnd o;
    const uint32_t idx = w & 0x3FFFFFFFu;
    if ((w >> 30) == K_SLOT) { o.p = SP{(int) (c.slots - g_smem) + (int) idx * E + c.lane}; o.stride = 32; o.tstride = L; }
    else { o.p = SP{(int) (c.spar - g_smem) + (int) idx * L + c.vlane}; o.stride = 0; o.tstride = 0; }
    return o;
}

#define ST(r) c.sst[(c.sidx + (r)) * L + c.lane]
#define STU(r) __float_as_uint(ST(r))
#define STI(r) __float_as_int(ST(r))

// Core.h:341-404 — OnceNode.  state: armed, gain, change.lastIn, isArmed (armed as loaded at the top of process())
template <int L, int E>
__device__ __noinline__ void ctl_once(const CtlCtx& c) {
    const Opnd x = ctl_decode<L, E>(c, __ldg(c.opnds));
    float armed = ST(0), gain = ST(1), last = ST(2), isArmed = ST(3);
    if (c.s0 == 0) isArmed = armed;                      // Core.h:370: one load per process() call
    for (int t = 0; t < c.cnt; ++t) {
        const float xin = LDT(x, t);
        const float delta = change_tick(last, xin);
        if (isArmed != 0.0f && delta > 0.5f) { gain = 1.0f; armed = 0.0f; }
        if (delta < -0.5f) gain = 0.0f;
        c.outT[t * L] = xin * gain;
    }
    ST(0) = armed; ST(1) = gain; ST(2) = last; ST(3) = isArmed;
}

// Core.h:407-573 — SequenceNode.  state: change.lastIn, resetChange.lastIn, holdValue, seqIndex, hasReceivedFirstPulse,
// generation of the sequence data last seen.  imm: [offset, generation].  mode: 1 hold, 2 loop, 4 reset input present.
template <int L, int E>
__device__ __noinline__ void ctl_seq(const CtlCtx& c) {
    const Opnd x = ctl_decode<L, E>(c, __ldg(c.opnds));
    const bool hasReset = (c.mode & 4u) != 0, hold = (c.mode & 1u) != 0, loop = (c.mode & 2u) != 0;
    const Opnd r = ctl_decode<L, E>(c, hasReset ? __ldg(c.opnds + 1) : make_operand(K_PARAM, 0));
    const uint32_t offset = __ldg(c.opnds + c.nopnd), codeGen = __ldg(c.opnds + c.nopnd + 1);
    const float* data = reinterpret_cast<const float*>(c.ptr);
    const uint32_t n = c.aux0;
    float last = ST(0), rlast = ST(1), holdv = ST(2);
    uint32_t idx = STU(3), first = STU(4), gen = STU(5);
    if (c.s0 == 0 && gen != codeGen) {                   // a new sequence was popped from the queue: Core.h:473-495
        idx = idx % n;
        if (first) holdv = __ldg(data + idx);
        gen = codeGen;
    }
    for (int t = 0; t < c.cnt; ++t) {
        const float in = LDT(x, t);
        const float reset = hasReset ? LDT(r, t) : 0.0f;
        if (change_tick(rlast, reset) > 0.5f) idx = offset;
        if (change_tick(last, in) > 0.5f) {
            holdv = __ldg(data + min(idx, n - 1));
            first = 1;
            if (++idx >= n && loop) idx = 0;
        }
        c.outT[t * L] = (idx < n) ? (hold ? holdv : holdv * in) : (hold ? holdv : 0.0f);
    }
    ST(0) = last; ST(1) = rlast; ST(2) = holdv;
    ST(3) = __uint_as_float(idx); ST(4) = __uint_as_float(first); ST(5) = __uint_as_float(gen);
}

// Seq2.h:87-148 — Seq2Node.  state: change.lastIn, resetChange.lastIn, edgeCount.  imm: [offset].
template <int L, int E>
__device__ __noinline__ void ctl_seq2(const CtlCtx& c) {
    const Opnd x = ctl_decode<L, E>(c, __ldg(c.opnds));
    const bool hasReset = (c.mode & 4u) != 0, hold = (c.mode & 1u) != 0, loop = (c.mode & 2u) != 0;
    const Opnd r = ctl_decode<L, E>(c, hasReset ? __ldg(c.opnds + 1) : make_operand(K_PARAM, 0));
    const unsigned long long offset = __ldg(c.opnds + c.nopnd);
    const float* data = reinterpret_cast<const float*>(c.ptr);
    const unsigned long long n = c.aux0;
    float last = ST(0), rlast = ST(1);
    uint32_t edge = STU(2);
    for (int t = 0; t < c.cnt; ++t) {
        const float in = LDT(x, t);
        const float reset = hasReset ? LDT(r, t) : 0.0f;
        if (change_tick(last, in) > 0.5f) edge++;
        if (change_tick(rlast, reset) > 0.5f) edge = 0;
        const unsigned long long idx = offset + edge;
        const float next = (idx < n) ? __ldg(data + idx)
                         : (loop ? __ldg(data + idx % n) : (hold ? __ldg(data + (n - 1)) : 0.0f));
        c.outT[t * L] = hold ? next : next * in;
    }
    ST(0) = last; ST(1) = rlast; ST(2) = __uint_as_float(edge);
}

// first index whose key is > t (std::map::upper_bound over the sorted key array)
template <typename K>
__device__ __forceinline__ int upper_bound_idx(const K* keys, int n, K t) {
    int lo = 0, hi = n;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (t < keys[mid]) hi = mid; else lo = mid + 1;
    }
    return lo;
}

// SparSeq2.h:69-128 — SparSeq2Node.  ptr = double time[n] then float value[n].  state: prevEvent, nextEvent (indices, n =
// end()), generation.  imm: [generation].  mode bit0 = interpolate.
template <int L, int E>
__device__ __noinline__ void ctl_sparseq2(const CtlCtx& c) {
    const Opnd x = ctl_decode<L, E>(c, __ldg(c.opnds));
    const int n = (int) c.aux0;
    const double* times = reinterpret_cast<const double*>(c.ptr);
    const float* values = reinterpret_cast<const float*>(times + n);
    const bool interp = (c.mode & 1u) != 0;
    const uint32_t codeGen = __ldg(c.opnds + c.nopnd);
    int prev = STI(0), next = STI(1);
    uint32_t gen = STU(2);
    if (c.s0 == 0 && gen != codeGen) { prev = n; next = n; gen = codeGen; }   // SparSeq2.h:77-86
    for (int i = 0; i < c.cnt; ++i) {
        const double t = (double) LDT(x, i);
        const bool update = (prev == n && next == n) || (prev != n && t <= (times[prev] + 1e-9)) || (next != n && t >= (times[next] - 1e-9));
        if (update) {
            next = upper_bound_idx<double>(times, n, t);
            prev = (next == 0) ? n : next - 1;
        }
        float y;
        if (prev == n) y = 0.0f;
        else if (next == n) y = values[prev];
        else {
            const double alpha = interp ? ((t - times[prev]) / (times[next] - times[prev])) : 0.0;
            y = values[prev] + (float) alpha * (values[next] - values[prev]);
        }
        c.outT[i * L] = y;
    }
    ST(0) = __int_as_float(prev); ST(1) = __int_as_float(next); ST(2) = __uint_as_float(gen);
}

// SparSeq.h:17-377 — SparSeqNode.  ptr = int32 tickTime[n] then float value[n] (0 = no sequence yet).
// state rows: 0 change.lastIn, 1 resetChange.lastIn, 2 edgeCount, 3 samplesSinceClockEdge, 4 holdValue (index, n = end()),
// 5/6 loopPoints, 7 pending flag, 8/9 pendingLoopPoints, 10 sequence generation seen, 11 loop-points generation seen,
// 12 tickTime (a local of process(), carried between the sample tiles of one call).
// imm: [offset, follow, interpolate, seqGen, loopGen, loopStart, loopEnd, tickInterval lo, hi].
struct SparSeqState { int edge, ls, le, pend, ps, pe; };

__device__ __forceinline__ int sparseq_tick_time(SparSeqState& s, int offset) {     // SparSeq.h:147-193
    int tick = offset + s.edge;
    const int ls = s.ls, le = s.le;
    if (ls > -1 && le > -1 && tick >= le) {
        const int dur = le - ls;
        if (dur > 0) {
            if (s.pend) {
                s.ls = s.ps; s.le = s.pe; s.pend = 0;
                const int nls = s.ls, nle = s.le;
                if (nls == -1 && nle == -1) return tick;
                if (nle - nls != 0) tick = nls + ((tick - le) % (nle - nls));
            } else {
                tick = ls + ((tick - le) % dur);
            }
            s.edge = tick - offset;
        }
    }
    return tick;
}

__device__ __forceinline__ int sparseq_find(const int* times, int n, int tick) {      // SparSeq.h:126-145
    if (n == 0) return 0;
    const int it = upper_bound_idx<int>(times, n, tick);
    if (it == 0) return (times[0] == 0) ? 0 : n;
    return it - 1;
}

template <int L, int E>
__device__ __noinline__ void ctl_sparseq(const CtlCtx& c) {
    const Opnd x = ctl_decode<L, E>(c, __ldg(c.opnds));
    const bool hasReset = (c.mode & 4u) != 0;
    const Opnd r = ctl_decode<L, E>(c, hasReset ? __ldg(c.opnds + 1) : make_operand(K_PARAM, 0));
    const uint32_t* imm = c.opnds + c.nopnd;
    const int offset = (int) __ldg(imm), follow = (int) __ldg(imm + 1), ho = (int) __ldg(imm + 2);
    const uint32_t seqGen = __ldg(imm + 3), loopGen = __ldg(imm + 4);
    const double spc = bits_to_double(__ldg(imm + 7), __ldg(imm + 8));
    const int n = (int) c.aux0;
    const bool hasSeq = c.ptr != 0;
    const int* times = reinterpret_cast<const int*>(c.ptr);
    const float* values = reinterpret_cast<const float*>(times + n);

    float last = ST(0), rlast = ST(1);
    SparSeqState s{STI(2), STI(5), STI(6), STI(7), STI(8), STI(9)};
    uint32_t since = STU(3);
    int holdIdx = STI(4), tick = STI(12);
    if (c.s0 == 0) {                                       // top of process(): SparSeq.h:209-257
        tick = sparseq_tick_time(s, offset);
        uint32_t sg = STU(10), lg = STU(11);
        if (sg != seqGen || lg != loopGen) {
            if (lg != loopGen) { s.pend = 1; s.ps = (int) __ldg(imm + 5); s.pe = (int) __ldg(imm + 6); }
            ST(10) = __uint_as_float(seqGen); ST(11) = __uint_as_float(loopGen);
            holdIdx = hasSeq ? sparseq_find(times, n, tick) : n;
        }
        if (s.pend) {
            const bool takeImmediately = (s.ls == -1 && s.le == -1) || !follow;
            if (takeImmediately) { s.ls = s.ps; s.le = s.pe; s.pend = 0; tick = sparseq_tick_time(s, offset); }
        }
    }
    if (!hasSeq) {
        for (int t = 0; t < c.cnt; ++t) c.outT[t * L] = 0.0f;
    } else {
        for (int i = 0; i < c.cnt; ++i) {
            since++;
            const float in = LDT(x, i);
            const float reset = hasReset ? LDT(r, i) : 0.0f;
            const bool trig = change_tick(last, in) > 0.5f;
            const bool rst = change_tick(rlast, reset) > 0.5f;
            if (rst) s.edge = 0;
            if (trig) {
                s.edge = rst ? 0 : s.edge + 1;
                since = 0;
                tick = sparseq_tick_time(s, offset);
                holdIdx = sparseq_find(times, n, tick);
            }
            float y;
            if (holdIdx == n) y = 0.0f;
            else if (ho == 1) {
                const int right = holdIdx + 1;
                if (right == n) y = values[holdIdx];
                else {
                    const int tl = times[holdIdx], tr = times[right];
                    const float lv = values[holdIdx], rv = values[right];
                    double alpha = (double) max(0, tick - tl) / (double) (tr - tl);
                    if (spc > 0.0) alpha += (fmin((double) since, spc) / spc) / (double) (tr - tl);
                    y = (float) ((double) lv + alpha * (double) (rv - lv));
                }
            } else y = values[holdIdx];
            c.outT[i * L] = y;
        }
    }
    ST(0) = last; ST(1) = rlast;
    ST(2) = __int_as_float(s.edge); ST(3) = __uint_as_float(since); ST(4) = __int_as_float(holdIdx);
    ST(5) = __int_as_float(s.ls); ST(6) = __int_as_float(s.le); ST(7) = __int_as_float(s.pend);
    ST(8) = __int_as_float(s.ps); ST(9) = __int_as_float(s.pe); ST(12) = __int_as_float(tick);
}

// Capture.h:22-58 — CaptureNode.  state rows: 0 change.lastIn, 1 scratchSize, 2 ring writePos, 3 ring readPos, 4 relayReady.
// ptr = this tile's [capacity + CAPTURE_SCRATCH][L] floats: ring, then the 128-sample scratch (Capture.h:96-98).
// The ring follows MultiChannelRingBuffer::write (MultiChannelRingBuffer.h:36-62): a write that does not fit clobbers
// and pushes the read pointer.
template <int L, int E>
__device__ __noinline__ void ctl_capture(const CtlCtx& c) {
    const Opnd g = ctl_decode<L, E>(c, __ldg(c.opnds));
    const Opnd x = ctl_decode<L, E>(c, __ldg(c.opnds + 1));
    const uint32_t cap = c.aux0, mask = cap - 1;
    float* ring = reinterpret_cast<float*>(c.ptr) + c.lane;      // position p: ring[p * L]
    float* scratch = ring + (size_t) cap * L;
    float last = ST(0);
    uint32_t ssize = STU(1), w = STU(2), r = STU(3), ready = STU(4);
    for (int i = 0; i < c.cnt; ++i) {
        const float gv = LDT(g, i), xv = LDT(x, i);
        const bool falling = change_tick(last, gv) < -0.5f;
        if (falling || ssize >= (uint32_t) CAPTURE_SCRATCH) {
            const uint32_t freeSlots = (r > w) ? (r - w) : (cap - (w - r));
            const bool moveRead = ssize >= freeSlots;
            for (uint32_t k = 0; k < ssize; ++k) ring[(size_t) ((w + k) & mask) * L] = scratch[(size_t) k * L];
            w = (w + ssize) & mask;
            if (moveRead) r = (w + 1) & mask;
            ssize = 0;
            if (falling) ready = 1;
        }
        if (gv != 0.0f) scratch[(size_t) (ssize++) * L] = xv;      // static_cast<bool>(float): anything but zero
        c.outT[i * L] = xv;
    }
    ST(0) = last; ST(1) = __uint_as_float(ssize); ST(2) = __uint_as_float(w); ST(3) = __uint_as_float(r); ST(4) = __uint_as_float(ready);
}
#undef ST
#undef STU
#undef STI

// A/B builds only (-DEB_OPPROF, tools/gpu/opprof.sh): cycles and dispatch count per opcode, accumulated by lane 0 of every warp of
// the interpreter — what the host's pipeline cost model (graph_host.cpp) is calibrated against.  Not compiled into the product library.
#ifdef EB_OPPROF
__device__ unsigned long long g_opprof[2 * 64];
#endif

// =========================================================================================================
// The whole per-tile interpreter; instantiated by the two thin __global__ wrappers at the end of this section.
// PIPE (many-groups launch of one-voice graphs only): this warp is stage `stage` of the P.pipeW-stage pipeline of ONE graph — the
// warps of the CTA share the graph's shared-memory area and hand sample tiles on through progress counters (see LaunchParams).
template <int NITER, int LOGL, bool PIPE = false>
__device__ __forceinline__ void render_tile(const LaunchParams& P, const int tile, const int perWarp, const long long sampleTime, const int outOffset,
                                            const int stage = 0) {
    constexpr int L = 1 << LOGL;          // voices per warp
    constexpr int E = 32 * NITER;         // elements per sample tile
    constexpr int T = E >> LOGL;          // samples per tile
    constexpr int LOGT = ilog2(T);
    constexpr int PER = 32 >> LOGL;       // samples of one voice inside one 32-element slice

    constexpr bool OOLM = (NITER == 4 && LOGL == 0);    // 128-sample one-voice tiles: heavy math through out-of-line copies (sin_f32_ool)
    const int warpInCta = threadIdx.x >> 5;
    const int lane = threadIdx.x & 31;

    const int vlane = lane & (L - 1);     // the voice column this lane works for
    const int voice = tile * L + vlane;   // may be a padding voice (>= nv): it owns storage but is never output
    const bool valid = voice < P.nv;
    const bool owner = lane < L;          // this lane runs the recurrences of `voice`
    const int tlane = lane >> LOGL;       // sample index of this lane's element inside slice 0

    const SP slots{PIPE ? 0 : warpInCta * perWarp};
    const SP outacc = slots + P.nSlots * E;
    const SP sst = outacc + P.nOut * E;
    const SP spar = sst + P.nStateRows * L;   // [nParams + 1][L], row 0 = zeros

    // pipeline bookkeeping (all constants when !PIPE)
    const int pipeW = PIPE ? max(1, P.pipeW) : 1;
    const bool firstStage = !PIPE || stage == 0, lastStage = !PIPE || stage == pipeW - 1;
    const int ringBase = (PIPE && pipeW > 1) ? P.pipeRingBase : 0x7FFFFFFF, pipeDepth = PIPE ? max(1, P.pipeDepth) : 1;
    volatile int* const progress = PIPE ? reinterpret_cast<volatile int*>(g_smem + perWarp) : nullptr;   // [MAX_PIPE] tiles finished per stage
    int ringOff = 0;                          // ring buffer of the current tile: tile index mod pipeDepth
    auto SLOTI = [&](int idx) -> int { if constexpr (PIPE) return idx + ((idx >= ringBase) ? ringOff : 0); else return idx; };
    (void) firstStage; (void) lastStage; (void) ringBase; (void) pipeDepth; (void) progress;

    auto decode = [&](uint32_t w) -> Opnd {
        Opnd o;
        const uint32_t idx = w & 0x3FFFFFFFu;
        if ((w >> 30) == K_SLOT) { o.p = slots + (SLOTI((int) idx) * E + lane); o.stride = 32; o.tstride = L; }
        else { o.p = spar + ((int) idx * L + vlane); o.stride = 0; o.tstride = 0; }
        return o;
    };

    // ---- state and parameter rows HBM -> shared memory (once per block), by the owner lanes ----
    // (a pipeline stage stages the state rows of ITS ops only; stage 0 also stages the parameters — the later stages read them after
    // their first hand-over from the stage before, which orders them behind these stores)
    const int stateBegin = (PIPE && pipeW > 1) ? (int) P.pipeState[stage] : 0;
    const int stateEnd = (PIPE && pipeW > 1) ? (int) P.pipeState[stage + 1] : P.nStateEntries;
    const int srowBegin = (PIPE && pipeW > 1) ? (int) P.pipeSrow[stage] : 0;
    if (!PIPE && P.k1Prefetch) {
        // Two dependent round trips in all: every lane loads one map entry, then the owner lanes issue all row copies back to back
        // as cp.async (LDGSTS) and wait once.  (A load-then-store loop waits for each row before it issues the next map load: with
        // the L2 cold that is some twenty HBM round trips per warp before the first sample.)  The one-voice pipeline kernel keeps the
        // plain loop: there this code costs spill loads inside the 64-register interpreter loop (BASELINE config 5 ran 5 % slower).
        const int nSt = stateEnd - stateBegin, nPar = firstStage ? P.nParams : 0;
        int srow = srowBegin;
        for (int c0 = 0; c0 < max(nSt, nPar); c0 += 32) {
            const uint32_t ms = (c0 + lane < nSt) ? __ldg(P.stateMap + stateBegin + c0 + lane) : STATE_PAD;
            const uint32_t mp = (c0 + lane < nPar) ? __ldg(P.paramMap + c0 + lane) : 0u;
            for (int j = 0, jn = min(32, nSt - c0); j < jn; ++j) {
                const uint32_t m = __shfl_sync(FULL, ms, j);
                if (m == STATE_PAD) { srow += 1; continue; }
                const size_t row = m & ~STATE_DOUBLE_FLAG;
                if (m & STATE_DOUBLE_FLAG) {
                    if (owner) cp_async_8(smem_u32(reinterpret_cast<double*>((sst + srow * L).ptr()) + lane),
                                          reinterpret_cast<const double*>(P.rows + row * P.Vpad) + voice);
                    srow += 2;
                } else {
                    if (owner) cp_async_4(smem_u32((sst + (srow * L + lane)).ptr()), P.rows + row * P.Vpad + voice);
                    srow += 1;
                }
            }
            for (int j = 0, jn = min(32, nPar - c0); j < jn; ++j) {
                const uint32_t m = __shfl_sync(FULL, mp, j);
                if (owner) cp_async_4(smem_u32((spar + ((c0 + j + 1) * L + lane)).ptr()), P.rows + (size_t) m * P.Vpad + voice);
            }
        }
        if (firstStage && owner) spar[lane] = 0.0f;
        asm volatile("cp.async.wait_all;" ::: "memory");
    } else if (owner) {
        int srow = srowBegin;
        for (int i = stateBegin; i < stateEnd; ++i) {
            const uint32_t m = __ldg(P.stateMap + i);
            if (m == STATE_PAD) { srow += 1; continue; }
            const size_t row = m & ~STATE_DOUBLE_FLAG;
            if (m & STATE_DOUBLE_FLAG) {
                const double* g = reinterpret_cast<const double*>(P.rows + row * P.Vpad);
                reinterpret_cast<double*>((sst + srow * L).ptr())[lane] = g[voice];
                srow += 2;
            } else {
                sst[srow * L + lane] = P.rows[row * P.Vpad + voice];
                srow += 1;
            }
        }
        if (firstStage) {
            spar[lane] = 0.0f;
            for (int i = 0; i < P.nParams; ++i)
                spar[(i + 1) * L + lane] = __ldg(P.rows + (size_t) __ldg(P.paramMap + i) * P.Vpad + voice);
        }
    }
    __syncwarp();

#define FOR_K(k) _Pragma("unroll") for (int k = 0; k < NITER; ++k)
#define T_OF(k) (tlane + (k) * PER)                       /* sample index of this lane's element in slice k */
#define FOR_OWNER(t) _Pragma("unroll 4") for (int t = 0; t < cnt; ++t)
    // recurrences walked by every lane of a voice column (narrow tiles, render_ops.inc OP_POLE): sample t = k * PER + j of the column
    // lives in register k of lane j * L + vlane
    // (the j loop stays ROLLED: the interpreter is instruction-fetch bound, 32 unrolled steps of shuffles run 3x slower than a rolled
    // loop that stays in the instruction cache — profiles/r02_j_opprof_config5_unrolled.txt)
#define FOR_TJ(k, j) _Pragma("unroll") for (int k = 0; k < NITER; ++k) _Pragma("unroll 4") for (int j = 0, jn_ = min(PER, cnt - k * PER); j < jn_; ++j)
#define FETCH_T(reg, j) __shfl_sync(FULL, (reg), (j) * L + vlane)

#ifdef EB_OPPROF
    const long long prof_tile0 = clock64();
#endif
    const int numSamples = P.numSamples;
    int tileIdx = 0;
    for (int s0 = 0; s0 < numSamples; s0 += T, ++tileIdx) {
        const int cnt = min(T, numSamples - s0);          // samples in this tile

        if constexpr (PIPE) {
            if (pipeW > 1) {
                // RAW: the stage before has finished this tile (transitively: every earlier stage has).  WAR: the ring buffer this tile
                // writes was last used pipeDepth tiles ago — the LAST stage must be through with that tile.  Bounded spins: a protocol
                // bug must end in wrong samples (the parity tests say so), never in a hung GPU.
                ringOff = tileIdx % pipeDepth;
                if (stage > 0) { for (int spins = 0; progress[stage - 1] <= tileIdx && spins < (1 << 22); ++spins) __nanosleep(20); }
                if (!lastStage && tileIdx >= pipeDepth) { for (int spins = 0; progress[pipeW - 1] <= tileIdx - pipeDepth && spins < (1 << 22); ++spins) __nanosleep(20); }
                __threadfence_block();
            }
        }
        if (lastStage) for (int i = lane; i < P.nOut * E; i += 32) outacc[i] = 0.0f;

#ifdef EB_SPEC_PROGRAM
        // ---- per-program specialisation (DESIGN.md §8; compiled only when a generated header defines the program as the
        // compile-time constant array eb::EB_SPEC_CODE, C++20): the same op bodies, but every header field and operand word
        // is a constant expression, so each `switch (opcode)` folds to its one case, slot addresses become immediates and chain
        // steps unroll — no dispatch, no decoding.  Device pointers (words 4/5 of a header) and the words that lanes index with
        // their own id (phasor runs, out-of-line control ops) are still read from the copy of the program in memory.
        {
            const uint32_t* const codeMem = P.code;
            auto run = [&]<int PC, int END>(auto&& self) -> void {
                if constexpr (PC < END) {
                    constexpr uint32_t opcode = EB_SPEC_CODE[PC] & 0xFF;
                    if constexpr (opcode != OP_END) {
                        constexpr struct { uint32_t x, y, z, w; } h0 = {EB_SPEC_CODE[PC], EB_SPEC_CODE[PC + 1], EB_SPEC_CODE[PC + 2], EB_SPEC_CODE[PC + 3]};
                        constexpr uint32_t nwords = (h0.x >> 8) & 0xFF, mode = h0.x >> 24;
                        constexpr uint32_t sidx = h0.y, aux0 = h0.z, aux1 = h0.w;
                        constexpr uint32_t count6 = EB_SPEC_CODE[PC + 6];
                        constexpr int NEXT0 = PC + (int) OP_HEADER_WORDS + (int) nwords;
                        if constexpr (opcode == OP_SEG) {
                            if ((P.runMask >> aux0) & 1u) self.template operator()<NEXT0, NEXT0 + (int) aux1>(self);
                            self.template operator()<NEXT0 + (int) aux1, END>(self);
                        } else {
                            __syncwarp();   // slot / state traffic of the previous op is visible to every lane
                            const SP out = slots + ((int) ((h0.x >> 16) & 0xFF) * E + lane);
                            const SP outT = out;
                            const uint64_t ptrbits = (uint64_t) __ldg(codeMem + PC + 4) | ((uint64_t) __ldg(codeMem + PC + 5) << 32);
                            const uint32_t* opnds = codeMem + PC + OP_HEADER_WORDS;
                            const uint32_t* pc = opnds + nwords;
                            (void) outT; (void) ptrbits; (void) opnds; (void) pc; (void) mode; (void) sidx; (void) count6;
#define OPWORD(i) (EB_SPEC_CODE[PC + (int) OP_HEADER_WORDS + (int) (i)])
#define CHAIN_FOR_STEPS(s) _Pragma("unroll") for (uint32_t s = 0; s < count6; ++s)
#define CHAIN_FN_WORD(s) (EB_SPEC_CODE[PC + (int) OP_HEADER_WORDS + 1 + 2 * (int) (s)])
#define CHAIN_OPND_WORD(s) (EB_SPEC_CODE[PC + (int) OP_HEADER_WORDS + 2 + 2 * (int) (s)])
#define CHAIN_NEXT(s) ((void) 0)
#define PC_ADVANCE(n) ((void) 0)
#define PC_SKIP_SEGMENT_IF(cond, n) ((void) 0)
#include "render_ops.inc"
#undef CHAIN_NEXT
#undef OPWORD
#undef CHAIN_FOR_STEPS
#undef CHAIN_FN_WORD
#undef CHAIN_OPND_WORD
#undef PC_ADVANCE
#undef PC_SKIP_SEGMENT_IF
                            constexpr int RUN_EXTRA = (opcode == OP_PHASOR && aux1 >= 1) ? (int) (aux1 - 1) * ((int) OP_HEADER_WORDS + 4) : 0;
                            self.template operator()<NEXT0 + RUN_EXTRA, END>(self);
                        }
                    }
                }
            };
            run.template operator()<0, EB_SPEC_CODE_LEN>(run);
        }
#else
#if EB_INTERP_PREFETCH
        // The interpreter loop is software-pipelined: the header (two 128-bit words) and the first four operand words of the NEXT op are
        // loaded while the current op executes, so that a dispatch does not begin with three dependent trips to memory (header ->
        // operand word -> slot).  Ops that move the program counter themselves (phasor runs, skipped segments) just reload.
        const uint32_t* pc = P.code + ((PIPE && pipeW > 1) ? P.pipeCode[stage] : 0u);
        uint4 h0 = __ldg(reinterpret_cast<const uint4*>(pc));
        uint4 h1 = __ldg(reinterpret_cast<const uint4*>(pc + 4));
        uint4 ow4 = __ldg(reinterpret_cast<const uint4*>(pc + 8));      // (behind the last op lie the END header's zero words: always readable)
        for (;;) {
            __syncwarp();   // slot / state traffic of the previous op is visible to every lane
            const uint32_t opcode = h0.x & 0xFF;
            if (opcode == OP_END) break;
            const uint32_t nwords = (h0.x >> 8) & 0xFF, mode = h0.x >> 24;
            const SP out = slots + (SLOTI((int) ((h0.x >> 16) & 0xFF)) * E + lane);    // element k of this lane: out[k * 32]
            const SP outT = out;                                         // owner lane, sample t: outT[t * L]
            const uint32_t sidx = h0.y, aux0 = h0.z, aux1 = h0.w;
            const uint64_t ptrbits = (uint64_t) h1.x | ((uint64_t) h1.y << 32);
            const uint32_t count6 = h1.z;
            const uint32_t* opnds = pc + OP_HEADER_WORDS;
            const uint4 ow = ow4;
            pc += OP_HEADER_WORDS + nwords;
            const uint32_t* const pcPrefetched = pc;
            const uint4 h0n = __ldg(reinterpret_cast<const uint4*>(pc));
            const uint4 h1n = __ldg(reinterpret_cast<const uint4*>(pc + 4));
            const uint4 ow4n = __ldg(reinterpret_cast<const uint4*>(pc + 8));

            // program-word access of the interpreter (render_ops.inc explains the contract)
#define OPWORD(i) (((i) == 0) ? ow.x : ((i) == 1) ? ow.y : ((i) == 2) ? ow.z : ((i) == 3) ? ow.w : __ldg(opnds + (i)))
#define CHAIN_FOR_STEPS(s) const uint32_t* sp = opnds + 1; uint32_t cfw_ = ow.y, cow_ = ow.z; for (uint32_t s = 0; s < count6; ++s, sp += 2)
#define CHAIN_FN_WORD(s) cfw_
#define CHAIN_OPND_WORD(s) cow_
#define CHAIN_NEXT(s) do { cfw_ = __ldg(sp + 2); cow_ = __ldg(sp + 3); } while (0)
#define PC_ADVANCE(n) pc += (n)
#define PC_SKIP_SEGMENT_IF(cond, n) if (cond) pc += (n)
#ifdef EB_OPPROF
            const long long prof_t0 = clock64();
#endif
#include "render_ops.inc"
#ifdef EB_OPPROF
            __syncwarp();
            if (lane == 0) { atomicAdd(&g_opprof[2 * (opcode & 63)], (unsigned long long) (clock64() - prof_t0)); atomicAdd(&g_opprof[2 * (opcode & 63) + 1], 1ull); }
#endif
#undef OPWORD
#undef CHAIN_FOR_STEPS
#undef CHAIN_FN_WORD
#undef CHAIN_OPND_WORD
#undef CHAIN_NEXT
#undef PC_ADVANCE
#undef PC_SKIP_SEGMENT_IF
            if (pc == pcPrefetched) { h0 = h0n; h1 = h1n; ow4 = ow4n; }
            else {
                h0 = __ldg(reinterpret_cast<const uint4*>(pc));
                h1 = __ldg(reinterpret_cast<const uint4*>(pc + 4));
                ow4 = __ldg(reinterpret_cast<const uint4*>(pc + 8));
            }
        }
#else
        const uint32_t* pc = P.code + ((PIPE && pipeW > 1) ? P.pipeCode[stage] : 0u);
        for (;;) {
            __syncwarp();   // slot / state traffic of the previous op is visible to every lane
            const uint4 h0 = __ldg(reinterpret_cast<const uint4*>(pc));
            const uint32_t opcode = h0.x & 0xFF;
            if (opcode == OP_END) break;
            const uint4 h1 = __ldg(reinterpret_cast<const uint4*>(pc + 4));
            const uint32_t nwords = (h0.x >> 8) & 0xFF, mode = h0.x >> 24;
            const SP out = slots + (SLOTI((int) ((h0.x >> 16) & 0xFF)) * E + lane);    // element k of this lane: out[k * 32]
            const SP outT = out;                                         // owner lane, sample t: outT[t * L]
            const uint32_t sidx = h0.y, aux0 = h0.z, aux1 = h0.w;
            const uint64_t ptrbits = (uint64_t) h1.x | ((uint64_t) h1.y << 32);
            const uint32_t count6 = h1.z;
            const uint32_t* opnds = pc + OP_HEADER_WORDS;
            pc += OP_HEADER_WORDS + nwords;

            // program-word access of the interpreter (render_ops.inc explains the contract)
#define OPWORD(i) __ldg(opnds + (i))
#define CHAIN_FOR_STEPS(s) const uint32_t* sp = opnds + 1; uint32_t cfw_ = __ldg(sp), cow_ = __ldg(sp + 1); for (uint32_t s = 0; s < count6; ++s, sp += 2)
#define CHAIN_FN_WORD(s) cfw_
#define CHAIN_OPND_WORD(s) cow_
#define CHAIN_NEXT(s) do { cfw_ = __ldg(sp + 2); cow_ = __ldg(sp + 3); } while (0)
#define PC_ADVANCE(n) pc += (n)
#define PC_SKIP_SEGMENT_IF(cond, n) if (cond) pc += (n)
#ifdef EB_OPPROF
            const long long prof_t0 = clock64();
#endif
#include "render_ops.inc"
#ifdef EB_OPPROF
            __syncwarp();
            if (lane == 0) { atomicAdd(&g_opprof[2 * (opcode & 63)], (unsigned long long) (clock64() - prof_t0)); atomicAdd(&g_opprof[2 * (opcode & 63) + 1], 1ull); }
#endif
#undef OPWORD
#undef CHAIN_FOR_STEPS
#undef CHAIN_FN_WORD
#undef CHAIN_OPND_WORD
#undef CHAIN_NEXT
#undef PC_ADVANCE
#undef PC_SKIP_SEGMENT_IF
        }
#endif   // EB_INTERP_PREFETCH
#endif   // EB_SPEC_PROGRAM

        if constexpr (PIPE) {
            if (pipeW > 1) {   // hand the tile on: slot / state stores first, then the counter
                __syncwarp();
                __threadfence_block();
                if (lane == 0) progress[stage] = tileIdx + 1;
            }
            if (!lastStage) continue;
        }
        // ---- tile epilogue: per-voice output and per-tile partial mix ----
        if (P.outVoice) {
            for (int ch = 0; ch < P.nOut; ++ch) {
                const SP a = outacc + ch * E;
                FOR_K(k) {
                    const int qq = lane + 32 * k;           // transposed: consecutive lanes = consecutive samples
                    const int v = qq >> LOGT, t = qq & (T - 1);
                    const int vv = tile * L + v;
                    if (t < cnt && vv < P.nv)
                        P.outVoice[((size_t) (P.voice0 + vv) * P.nOut + ch) * P.outStride + outOffset + s0 + t] = a[t * L + v];
                }
            }
        }
        if (P.mixPartial) {
            // sum over the voices of the tile in a fixed order (xor butterfly over the voice bits of the lane id)
            for (int ch = 0; ch < P.nOut; ++ch) {
                const SP a = outacc + (ch * E + lane);
                float* gp = P.mixPartial + ((size_t) (P.tileBase + tile) * P.nOut + ch) * P.blockSize + s0;
                FOR_K(k) {
                    const int t = T_OF(k);
                    float v = (valid && t < cnt) ? a[k * 32] : 0.0f;
                    _Pragma("unroll") for (int d = L >> 1; d > 0; d >>= 1) v += __shfl_xor_sync(FULL, v, d);
                    if (vlane == 0 && t < cnt) gp[t] = v;
                }
            }
        }
    }
    __syncwarp();

#ifdef EB_OPPROF
    if (lane == 0) { atomicAdd(&g_opprof[2 * 63], (unsigned long long) (clock64() - prof_tile0)); atomicAdd(&g_opprof[2 * 63 + 1], 1ull); }   // whole sample loop of one warp
#endif
    // ---- state rows shared memory -> HBM ----
    if (owner) {
        int srow = srowBegin;
        for (int i = stateBegin; i < stateEnd; ++i) {
            const uint32_t m = __ldg(P.stateMap + i);
            if (m == STATE_PAD) { srow += 1; continue; }
            const size_t row = m & ~STATE_DOUBLE_FLAG;
            if (m & STATE_DOUBLE_FLAG) {
                double* g = reinterpret_cast<double*>(P.rows + row * P.Vpad);
                g[voice] = reinterpret_cast<const double*>((sst + srow * L).ptr())[lane];
                srow += 2;
            } else {
                P.rows[row * P.Vpad + voice] = sst[srow * L + lane];
                srow += 1;
            }
        }
    }

    // ---- tap promotion (GraphRenderSequence.h:200-210,306-308): OP_PROMOTE records after the first OP_END ----
    // (the host never pipelines a program with taps; it also knows where the records start, so most programs skip this entirely)
    if (!(PIPE && pipeW > 1) && (!P.k1Prefetch || P.promoteAt >= 0)) {
        const uint32_t* pc = P.code;
        if (P.k1Prefetch) pc += P.promoteAt;
        else for (;;) {   // skip the main program
            const uint32_t w0 = __ldg(pc);
            pc += OP_HEADER_WORDS + ((w0 >> 8) & 0xFF);
            if ((w0 & 0xFF) == OP_END) break;
        }
        for (;;) {
            const uint4 h0 = __ldg(reinterpret_cast<const uint4*>(pc));
            if ((h0.x & 0xFF) != OP_PROMOTE) break;
            const uint4 h1 = __ldg(reinterpret_cast<const uint4*>(pc + 4));
            pc += OP_HEADER_WORDS;
            // only roots that are still the active target promote (RootRenderSequence::promoteTapBuffers)
            if (!((P.runMask >> (16 + h0.y)) & 1u)) continue;
            const uint64_t sb = (uint64_t) h0.z | ((uint64_t) h0.w << 32);
            const uint64_t db = (uint64_t) h1.x | ((uint64_t) h1.y << 32);
            const float* src = reinterpret_cast<const float*>(sb) + (size_t) tile * P.blockSize * L;
            float* dst = reinterpret_cast<float*>(db) + (size_t) tile * P.blockSize * L;
            for (int i = lane; i < numSamples * L; i += 32) dst[i] = src[i];
        }
    }
#undef FOR_K
#undef T_OF
#undef FOR_OWNER
#undef FOR_TJ
#undef FETCH_T
}

// Occupancy target (measured, profiles/r01_d_occupancy_ab.txt): the full-width geometry (L = 32, every lane a voice)
// is issue-latency bound and gains 20 % from 64-register / 8-CTA occupancy; the narrow geometries run few warps
// anyway and prefer the 128-register budget.
#ifndef EB_L32_MINBLOCKS
#define EB_L32_MINBLOCKS 8
#endif
#ifndef EB_L1_MINBLOCKS
#define EB_L1_MINBLOCKS 4
#endif
#ifndef EB_NARROW_MINBLOCKS
#define EB_NARROW_MINBLOCKS 4      /* 1 < L < 32; a specialised kernel may be compiled for 8 (64 registers): engine option "spec_minblocks" */
#endif
#define EB_BOUNDS __launch_bounds__(128, (LOGL == 5) ? EB_L32_MINBLOCKS : ((LOGL == 0) ? EB_L1_MINBLOCKS : EB_NARROW_MINBLOCKS))

// One voice group per launch: the descriptor travels in the constant bank.
template <int NITER, int LOGL>
__global__ void EB_BOUNDS render_block_kernel(const __grid_constant__ LaunchParams P, const int perWarp) {
    if (P.tableSmem >= 0)       // CTA-wide: one TMA bulk copy of the program's wavetable into shared memory, guarded by an mbarrier
        stage_table_tma(P.tableSrc, P.tableFloats, g_smem + P.tableSmem, reinterpret_cast<uint64_t*>(g_smem + P.tableSmem + P.tableFloats));
    const int tile = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (tile >= ((P.nv + (1 << LOGL) - 1) >> LOGL)) return;   // whole warp leaves together
    render_tile<NITER, LOGL>(P, tile, perWarp, P.sampleTime, 0);
}

// Many voice groups (different graphs) of the same tile geometry in ONE launch: warp w finds its group by binary
// search in the tile prefix table and reads that group's descriptor from global memory.  This is what makes
// thousands of small heterogeneous graphs (BASELINE config 5) run concurrently instead of one launch each.
template <int NITER, int LOGL>
__global__ void EB_BOUNDS render_groups_kernel(const LaunchParams* __restrict__ descs, const int* __restrict__ tileStart,
                                                const int nGroups, const int totalTiles, const int perWarp, const long long sampleTime, const int outOffset) {
    const int w = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (w >= totalTiles) return;
    int lo = 0, hi = nGroups - 1;                      // largest g with tileStart[g] <= w
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (__ldg(tileStart + mid) <= w) lo = mid; else hi = mid - 1;
    }
    render_tile<NITER, LOGL>(descs[lo], w - __ldg(tileStart + lo), perWarp, sampleTime, outOffset);   // the sample clock travels as an argument: the descriptors of a steady engine never change
}

// The same for one-voice graphs whose programs the host cut into pipeline stages (LaunchParams::pipeW): ONE CTA per graph, warp w of
// the CTA runs stage w.  A graph's recurrences are serial per sample and own a single lane, so one warp per graph is latency bound
// (profiles/r02_f_groups_ncu.txt: 0.08 instructions per cycle and warp at 8 warps per SM); with W stages W warps work on W different
// sample tiles of the same graph at once.  Programs that were not cut (pipeW <= 1) simply use warp 0.
template <int NITER>
__global__ void __launch_bounds__(32 * MAX_PIPE, 8) render_groups_pipe_kernel(const LaunchParams* __restrict__ descs, const int* __restrict__ tileStart,
                                                                              const int nGroups, const int totalTiles, const int perGraph,
                                                                              const long long sampleTime, const int outOffset) {
    const int w = blockIdx.x;                          // one-voice tiles: tile index == CTA index
    const int stage = threadIdx.x >> 5;
    if (threadIdx.x < MAX_PIPE) reinterpret_cast<volatile int*>(g_smem + perGraph)[threadIdx.x] = 0;   // progress counters
    __syncthreads();
    if (w >= totalTiles) return;
    int lo = 0, hi = nGroups - 1;                      // largest g with tileStart[g] <= w
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (__ldg(tileStart + mid) <= w) lo = mid; else hi = mid - 1;
    }
    const LaunchParams& P = descs[lo];
    if (stage >= max(1, P.pipeW)) return;              // (whole warps leave; no CTA-wide barrier follows)
    render_tile<NITER, 0, true>(P, w - __ldg(tileStart + lo), perGraph, sampleTime, outOffset, stage);
}

#ifndef __CUDACC_RTC__   // K2, K4 and the host launchers are not needed by a run-time compiled specialisation of K1
} // namespace eb
#include "spec_host.h"
namespace eb {
// ---- K2: deterministic reduction of the per-tile partial mixes: out[ch][s] = sum over tiles in a fixed order ----
// grid = (channel x 32-sample chunk, G tile groups).  Block (bx, g) sums the tiles of group g (32 tile lanes x 32 samples, four
// interleaved accumulators per lane so that independent loads are in flight), leaves its result in scratch[g]; the block that
// arrives last at the chunk's ticket counter adds the G group sums in group order.  The summation order is a function of
// (nTiles, G) only — never of which block happens to be last — so the mix is reproducible run to run.
__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) { asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory"); }

// Called by every CTA that has just written its part of the FINAL mix bus (all threads of the CTA): the part is already in hd.out;
// the CTA that arrives last at the `done` counter raises the host flag (data first: system-scope fences on both sides of the counter).
__device__ __forceinline__ void host_deliver_arrive(const HostDeliver& hd, unsigned int nCtas) {
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned int d = atomicAdd(hd.done, 1u);
        if (d == nCtas - 1) {
            *hd.done = 0;                                     // ready for the next block of audio
            __threadfence_system();
            st_release_sys(hd.flag, hd.seq);
        }
    }
}

__global__ void __launch_bounds__(1024) mix_reduce_kernel(const float* __restrict__ partial, float* __restrict__ out, float* __restrict__ scratch,
                                                          unsigned int* __restrict__ tickets, int nTiles, int nOut, int blockSize, int numSamples, const HostDeliver hd) {
    __shared__ float red[32][33];
    __shared__ bool last;
    const int sx = threadIdx.x & 31, gy = threadIdx.x >> 5;       // 32 samples x 32 tile lanes
    const int chunksPerCh = (blockSize + 31) / 32;
    const int ch = blockIdx.x / chunksPerCh;
    const int s = (blockIdx.x % chunksPerCh) * 32 + sx;
    const int G = gridDim.y, g = blockIdx.y;
    const int perGroup = ((nTiles + G - 1) / G + 31) / 32 * 32;   // tiles per group, a multiple of the 32 lanes
    const int tBegin = g * perGroup, tEnd = min(nTiles, tBegin + perGroup);
    float a0 = 0.0f, a1 = 0.0f, a2 = 0.0f, a3 = 0.0f;
    if (s < numSamples) {
        const size_t step = (size_t) 32 * nOut * blockSize;
        int t = tBegin + gy;
        const float* p = partial + ((size_t) t * nOut + ch) * blockSize + s;
        for (; t + 96 < tEnd; t += 128, p += 4 * step) { a0 += p[0]; a1 += p[step]; a2 += p[2 * step]; a3 += p[3 * step]; }
        for (; t < tEnd; t += 32, p += step) a0 += p[0];
    }
    red[gy][sx] = (a0 + a1) + (a2 + a3);
    __syncthreads();
    if (gy == 0) {
        float v = 0.0f;
        for (int k = 0; k < 32; ++k) v += red[k][sx];
        if (G == 1) { if (s < numSamples) { out[(size_t) ch * blockSize + s] = v; if (hd.out) hd.out[(size_t) ch * blockSize + s] = v; } }
        else if (s < numSamples) scratch[((size_t) g * nOut + ch) * blockSize + s] = v;
    }
    if (G == 1) {
        if (hd.out) host_deliver_arrive(hd, gridDim.x);
        return;
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned int ticket = atomicAdd(&tickets[blockIdx.x], 1u);
        last = (ticket == (unsigned int) G - 1);
        if (last) tickets[blockIdx.x] = 0;                        // ready for the next block of audio
    }
    __syncthreads();
    if (last && gy == 0 && s < numSamples) {
        __threadfence();
        float v = 0.0f;
        for (int k = 0; k < G; ++k) v += __ldcg(scratch + ((size_t) k * nOut + ch) * blockSize + s);
        out[(size_t) ch * blockSize + s] = v;
        if (hd.out) hd.out[(size_t) ch * blockSize + s] = v;
    }
    if (last && hd.out) host_deliver_arrive(hd, gridDim.x);   // `last` is uniform over the CTA: one finishing CTA per chunk
}

// =========================================================================================================
// host-side launchers (called from graph_host.cpp)

int render_niter_for(int tileWidth, int niterOverride) {
    // E = L*T = 32*NITER elements per sample tile (measured choices, profiles/r01_i_tile_samples_ab.txt):
    //   L >= 8 : E = 256 (T = 256/L);  L = 4 : T = 32;  L = 2 : T = 64 (fewer op dispatches per sample);  L = 1 : T = 32
    // L = 32 may also run with NITER = 4 (T = 4) for A/B runs.
    if (tileWidth == 32 && niterOverride == 4) return 4;
    if (tileWidth == 1 && niterOverride == 4) return 4;
    if (tileWidth == 2 && niterOverride == 8) return 8;       // L = 2, T = 128 (A/B: profiles/r02_q_*)       // L = 1, T = 128: four times fewer op dispatches per sample (A/B: profiles/r02_k_*)
    if (tileWidth >= 8) return 8;
    if (tileWidth == 4) return 4;
    return tileWidth == 2 ? 4 : 1;   // L = 1 keeps T = 32: with one voice per warp longer tiles push delay lines off their fast path (config 5)
}

size_t render_smem_bytes(int nSlots, int nOut, int nStateRows, int nParams, int warpsPerCta, int tileWidth, int niterOverride) {
    const int E = 32 * render_niter_for(tileWidth, niterOverride);
    const size_t perWarp = ((size_t) (nSlots + nOut) * E + (size_t) (nStateRows + nParams + 1) * tileWidth + 3) & ~(size_t) 3;
    return (size_t) warpsPerCta * perWarp * sizeof(float);
}

template <int NITER, int LOGL>
static cudaError_t launch_impl(const LaunchParams& P, int grid, int threads, size_t smem, cudaStream_t stream) {
    cudaError_t e = cudaFuncSetAttribute(render_block_kernel<NITER, LOGL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem);
    if (e != cudaSuccess) return e;
    // per-warp area = everything in front of the (optional) staged table
    const size_t warpArea = P.tableSmem >= 0 ? (size_t) P.tableSmem * sizeof(float) : smem;
    render_block_kernel<NITER, LOGL><<<grid, threads, smem, stream>>>(P, (int) (warpArea / sizeof(float) / (threads / 32)));
    return cudaGetLastError();
}

static cudaError_t launch_render_block_geometry(const LaunchParams& P, int L, int grid, int threads, size_t smem, int perWarpFloats, int niterOverride, cudaStream_t stream);

template <int NITER, int LOGL>
static cudaError_t launch_groups_impl(const LaunchParams* descs, const int* tileStart, int nGroups, int totalTiles,
                                      int grid, int threads, size_t smem, long long sampleTime, int outOffset, cudaStream_t stream) {
    cudaError_t e = cudaFuncSetAttribute(render_groups_kernel<NITER, LOGL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem);
    if (e != cudaSuccess) return e;
    render_groups_kernel<NITER, LOGL><<<grid, threads, smem, stream>>>(descs, tileStart, nGroups, totalTiles,
                                                                          (int) (smem / sizeof(float) / (threads / 32)), sampleTime, outOffset);
    return cudaGetLastError();
}

cudaError_t launch_render_block(const LaunchParams& P, int warpsPerCta, int niterOverride, cudaStream_t stream, const SpecKernel* spec) {
    const int L = P.tileWidth;
    const int nTiles = (P.nv + L - 1) / L;
    if (nTiles <= 0) return cudaSuccess;
    const int grid = (nTiles + warpsPerCta - 1) / warpsPerCta;
    const int threads = warpsPerCta * 32;
    size_t smem = render_smem_bytes(P.nSlots, P.nOut, P.nStateRows, P.nParams, warpsPerCta, L, niterOverride);
    LaunchParams Q = P;
    const int perWarpFloats = (int) (smem / sizeof(float) / warpsPerCta);
    if (Q.tableSrc && Q.tableFloats > 0 && Q.tableFloats <= TABLE_SMEM_MAX_FLOATS &&
        smem + (size_t) Q.tableFloats * 4 + 16 <= (size_t) 200 * 1024) {
        Q.tableSmem = perWarpFloats * warpsPerCta;            // behind the per-warp areas; 16-byte aligned (perWarp is a multiple of 4 floats)
        smem += (size_t) Q.tableFloats * 4 + 16;              // + the mbarrier
    } else { Q.tableSmem = -1; Q.tableSrc = nullptr; }
    if (spec && spec->function) return specialise_launch(*spec, Q, grid, threads, smem, perWarpFloats, stream);
    return launch_render_block_geometry(Q, L, grid, threads, smem, perWarpFloats, niterOverride, stream);
}

static cudaError_t launch_render_block_geometry(const LaunchParams& P, int L, int grid, int threads, size_t smem, int perWarpFloats, int niterOverride, cudaStream_t stream) {
    switch (L) {
        case 32: return render_niter_for(32, niterOverride) == 4 ? launch_impl<4, 5>(P, grid, threads, smem, stream)
                                                                  : launch_impl<8, 5>(P, grid, threads, smem, stream);
        case 16: return launch_impl<8, 4>(P, grid, threads, smem, stream);
        case 8:  return launch_impl<8, 3>(P, grid, threads, smem, stream);
        case 4:  return launch_impl<4, 2>(P, grid, threads, smem, stream);
        case 2:  return render_niter_for(2, niterOverride) == 8 ? launch_impl<8, 1>(P, grid, threads, smem, stream)
                                                                 : launch_impl<4, 1>(P, grid, threads, smem, stream);
        default: return render_niter_for(1, niterOverride) == 4 ? launch_impl<4, 0>(P, grid, threads, smem, stream)
                                                                : launch_impl<1, 0>(P, grid, threads, smem, stream);
    }
}

// descs / tileStart are DEVICE pointers; maxSlots etc. are the maxima over the groups (uniform shared-memory carve-up).
cudaError_t launch_render_groups(const LaunchParams* descs, const int* tileStart, int nGroups, int totalTiles, int tileWidth,
                                 int maxSlots, int nOut, int maxStateRows, int maxParams, int warpsPerCta, long long sampleTime, int outOffset, cudaStream_t stream,
                                 int niterOverride) {
    if (totalTiles <= 0) return cudaSuccess;
    const int grid = (totalTiles + warpsPerCta - 1) / warpsPerCta;
    const int threads = warpsPerCta * 32;
    if (tileWidth != 1) niterOverride = 0;       // the many-groups launch has the T = 128 variant for one-voice tiles only
    const size_t smem = render_smem_bytes(maxSlots, nOut, maxStateRows, maxParams, warpsPerCta, tileWidth, niterOverride);
    if (tileWidth == 1 && render_niter_for(1, niterOverride) == 4)
        return launch_groups_impl<4, 0>(descs, tileStart, nGroups, totalTiles, grid, threads, smem, sampleTime, outOffset, stream);
    switch (tileWidth) {
        case 32: return launch_groups_impl<8, 5>(descs, tileStart, nGroups, totalTiles, grid, threads, smem, sampleTime, outOffset, stream);
        case 16: return launch_groups_impl<8, 4>(descs, tileStart, nGroups, totalTiles, grid, threads, smem, sampleTime, outOffset, stream);
        case 8:  return launch_groups_impl<8, 3>(descs, tileStart, nGroups, totalTiles, grid, threads, smem, sampleTime, outOffset, stream);
        case 4:  return launch_groups_impl<4, 2>(descs, tileStart, nGroups, totalTiles, grid, threads, smem, sampleTime, outOffset, stream);
        case 2:  return launch_groups_impl<4, 1>(descs, tileStart, nGroups, totalTiles, grid, threads, smem, sampleTime, outOffset, stream);
        default: return launch_groups_impl<1, 0>(descs, tileStart, nGroups, totalTiles, grid, threads, smem, sampleTime, outOffset, stream);
    }
}

// One CTA of `stages` warps per one-voice graph (descs / tileStart are DEVICE pointers; the maxima size the per-graph shared memory).
cudaError_t launch_render_groups_pipe(const LaunchParams* descs, const int* tileStart, int nGroups, int totalTiles, int stages,
                                      int maxSlots, int nOut, int maxStateRows, int maxParams, long long sampleTime, int outOffset, cudaStream_t stream,
                                      int niterOverride) {
    if (totalTiles <= 0) return cudaSuccess;
    if (stages < 1) stages = 1;
    if (stages > MAX_PIPE) stages = MAX_PIPE;
    const size_t graphBytes = render_smem_bytes(maxSlots, nOut, maxStateRows, maxParams, 1, 1, niterOverride);
    const size_t smem = graphBytes + sizeof(int) * 8;              // + the progress counters
    const bool wide = render_niter_for(1, niterOverride) == 4;
    cudaError_t e = wide ? cudaFuncSetAttribute(render_groups_pipe_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem)
                         : cudaFuncSetAttribute(render_groups_pipe_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int) smem);
    if (e != cudaSuccess) return e;
    if (wide) render_groups_pipe_kernel<4><<<totalTiles, 32 * stages, smem, stream>>>(descs, tileStart, nGroups, totalTiles, (int) (graphBytes / sizeof(float)), sampleTime, outOffset);
    else render_groups_pipe_kernel<1><<<totalTiles, 32 * stages, smem, stream>>>(descs, tileStart, nGroups, totalTiles, (int) (graphBytes / sizeof(float)), sampleTime, outOffset);
    return cudaGetLastError();
}

cudaError_t launch_mix_reduce(const float* partial, float* out, float* scratch, unsigned int* tickets, int nTiles, int nOut, int blockSize,
                              int numSamples, cudaStream_t stream, HostDeliver hd) {
    const int chunksPerCh = (blockSize + 31) / 32;
    int G = (nTiles + 255) / 256;                 // ~8 tiles per lane per group; 4096 voices at L = 2 -> 8 groups x 16 chunks = 128 CTAs
    if (G > MIX_REDUCE_MAX_GROUPS) G = MIX_REDUCE_MAX_GROUPS;
    if (G < 1 || !scratch || !tickets) G = 1;
    mix_reduce_kernel<<<dim3(nOut * chunksPerCh, G), 1024, 0, stream>>>(partial, out, scratch, tickets, nTiles, nOut, blockSize, numSamples, hd);
    return cudaGetLastError();
}

// ---- K4: cross-GPU all-reduce of the mix bus over peer memory (see kernels.h) -------------------------------------------
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) { uint32_t v; asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory"); return v; }
__device__ __forceinline__ float ld_volatile_f32(const float* p) { float v; asm volatile("ld.volatile.global.f32 %0, [%1];" : "=f"(v) : "l"(p) : "memory"); return v; }

// grid = world - 1 CTAs.  CTA b PUSHES this rank's partial mix (PeerMix::own, left there by K2) into slot [parity][rank] of ONE peer —
// peer (rank + 1 + b) mod world, so at any moment every link carries one stream — as 8-byte (sample bits, epoch) pairs: a pair is its
// own arrival flag (8-byte stores are single transactions), so there is no fence and no flag store behind the data.  Then every CTA
// sums its 1/(world-1) share of the samples over the sources in rank order — its own partial from local memory, a remote one by
// polling the pair in its OWN buffer until it shows this epoch (bounded: a dead peer must not hang the GPU) — so every rank computes
// the bit-identical float sum.  Two parities: a rank can be one epoch ahead of a slow peer, never two (it needs the peer's pairs of
// epoch e+1, which the peer sends after finishing e).  count = 0 is a pure barrier through the flag words.
__device__ __forceinline__ void st_volatile_v2(uint2* p, uint32_t x, uint32_t y) { asm volatile("st.volatile.global.v2.u32 [%0], {%1, %2};" ::"l"(p), "r"(x), "r"(y) : "memory"); }
__device__ __forceinline__ uint2 ld_volatile_v2(const uint2* p) { uint2 v; asm volatile("ld.volatile.global.v2.u32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "l"(p) : "memory"); return v; }

__global__ void __launch_bounds__(256) mix_exchange_kernel(const PeerMix pm, float* __restrict__ mix, int count, uint32_t epoch, int* status, const HostDeliver hd) {
    const int tid = threadIdx.x, b = blockIdx.x, nb = gridDim.x;
    const int parity = (int) (epoch & 1u);
    if (count == 0) {   // barrier: raise my flag on one peer, wait for every peer's flag here
        const int p = (pm.rank + 1 + b) % pm.world;
        if (tid == 0) st_release_sys(pm.flag[p] + parity * MAX_PEERS + pm.rank, epoch);
        if (tid < pm.world && tid != pm.rank) {
            const uint32_t* f = pm.flag[pm.rank] + parity * MAX_PEERS + tid;
            const long long t0 = clock64();
            while (ld_acquire_sys(f) != epoch) {
                if (clock64() - t0 > 2000000000ll) { if (status) *status = 1; break; }   // ~1 s
                __nanosleep(32);
            }
        }
        return;
    }
    {   // 1. push (value, epoch) pairs
        const int p = (pm.rank + 1 + b) % pm.world;
        uint2* dst = pm.slot[p] + (size_t) (parity * MAX_PEERS + pm.rank) * pm.stride;
        for (int i = tid; i < count; i += blockDim.x) st_volatile_v2(dst + i, __float_as_uint(pm.own[i]), epoch);
    }
    // 2. sum this CTA's share of the samples over the sources in rank order
    const uint2* mine = pm.slot[pm.rank] + (size_t) parity * MAX_PEERS * pm.stride;               // [src rank][stride] in OUR buffer
    const int per = (count + nb - 1) / nb;
    const int i1 = min(count, (b + 1) * per);
    for (int i = b * per + tid; i < i1; i += blockDim.x) {
        float s = 0.0f;
        for (int src = 0; src < pm.world; ++src) {
            if (src == pm.rank) { s += pm.own[i]; continue; }
            const uint2* q = mine + (size_t) src * pm.stride + i;
            uint2 v = ld_volatile_v2(q);
            if (v.y != epoch) {
                const long long t0 = clock64();
                do {
                    if (clock64() - t0 > 2000000000ll) { if (status) *status = 1; break; }       // ~1 s
                    __nanosleep(20);
                    v = ld_volatile_v2(q);
                } while (v.y != epoch);
            }
            s += __uint_as_float(v.x);
        }
        mix[i] = s;
        if (hd.out) hd.out[i] = s;
    }
    if (hd.out) host_deliver_arrive(hd, nb);
}

// Per-opcode profile of an -DEB_OPPROF build: out[2 * opcode] = cycles, out[2 * opcode + 1] = dispatches; zeros in the product build.
cudaError_t debug_opprof_read(unsigned long long* out128, bool reset) {
#ifdef EB_OPPROF
    cudaError_t e = cudaMemcpyFromSymbol(out128, g_opprof, sizeof(unsigned long long) * 128);
    if (e == cudaSuccess && reset) { static const unsigned long long z[128] = {}; e = cudaMemcpyToSymbol(g_opprof, z, sizeof z); }
    return e;
#else
    for (int i = 0; i < 128; ++i) out128[i] = 0;
    (void) reset;
    return cudaSuccess;
#endif
}

cudaError_t launch_mix_exchange(const PeerMix& pm, float* mix, int count, uint32_t epoch, int* status, cudaStream_t stream, HostDeliver hd) {
    if (pm.world < 2) return cudaSuccess;
    mix_exchange_kernel<<<pm.world - 1, 256, 0, stream>>>(pm, mix, count, epoch, status, hd);
    return cudaGetLastError();
}

#endif   // __CUDACC_RTC__

} // namespace eb
