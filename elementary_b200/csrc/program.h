// program.h — the compiled "render program" shared by the host graph compiler (graph_host.cpp) and the
// fused device kernel (render_kernel.cu).
//
// The reference turns its node graph into a GraphRenderSequence: a topologically sorted list of closures,
// each calling one GraphNode::process() over a whole block with one 2 KB buffer per node output
// (runtime/elem/GraphRenderSequence.h:107-187,212-232; Runtime.h:521-577).  Here the same sorted list is
// lowered to a flat array of 32-bit words that ONE kernel interprets, warp-uniformly, for every voice tile:
//
//   op := header (8 words, 16-byte aligned so it is fetched with two 128-bit loads)
//           [w0 = opcode | nWords<<8 | outSlot<<16 | mode<<24]   nWords = operand words that follow (padded to x4)
//           [w1 = state index (row inside the warp's shared-memory state area) or 0xFFFFFFFF]
//           [w2 = aux0] [w3 = aux1] [w4, w5 = 64-bit device pointer] [w6 = logical operand / step count] [w7 = 0]
//         operand words            operand = kind<<30 | index
//
// Node outputs live in shared-memory "slots" ([T samples][L voices] floats per warp, liveness-allocated by the
// host), not in per-node block buffers.  `const`/`sr` nodes never execute: their per-voice value is a parameter
// row, staged once per block into the warp's shared-memory parameter area and read like a slot with stride 0.
// Runs of stateless element-wise nodes (sin, mul, add, le, ...) whose intermediate has a single consumer are
// fused by the host into one OP_CHAIN: the intermediate never leaves registers.
#pragma once
#include "rtc_compat.h"

namespace eb {

enum Opcode : uint32_t {
    OP_END = 0,
    OP_SEG,        // root sub-sequence header: aux0 = root index, aux1 = words to skip when the root is not running
    OP_FILL0,      // out = 0 (node lacked the inputs it needs: Core.h:125-126 and friends)
    OP_COPY,       // out = in0 (IdentityNode with a child, analysis pass-through)
    OP_LOADIN,     // out = host input channel aux0 (IdentityNode leaf / leaf-node host inputs, GraphRenderSequence.h:126-135)
    OP_CHAIN,      // acc = operand0; then w6 steps (fn word, operand word): unary/binary/reducing math (Math.h:9-89)
    OP_PHASOR,     // Core.h:85-136 (WithReset=false)
    OP_SPHASOR,    // Core.h:85-136 (WithReset=true)
    OP_COUNTER,    // Core.h:183-215
    OP_ACCUM,      // Core.h:218-248
    OP_LATCH,      // Core.h:250-286
    OP_MAXHOLD,    // Core.h:288-339
    OP_RAND,       // Noise.h:9-43
    OP_POLE,       // Filters.h:13-39
    OP_ENV,        // Filters.h:46-79
    OP_BIQUAD,     // Filters.h:87-120
    OP_PREWARP,    // filters/MultiMode1p.h:9-37
    OP_MM1P,       // filters/MultiMode1p.h:39-113
    OP_SVF,        // filters/SVF.h:18-121
    OP_SVFSHELF,   // filters/SVFShelf.h:20-126
    OP_Z,          // Delays.h:15-39
    OP_DELAY,      // Delays.h:51-169
    OP_SDELAY,     // Delays.h:177-272
    OP_TABLE,      // Table.h:16-76
    OP_BLEP,       // Oscillators.h:19-94, mode = 0 saw / 1 square / 2 triangle
    OP_TAPIN,      // Feedback.h:20-57
    OP_TAPOUT,     // Feedback.h:59-131
    OP_ROOT,       // Core.h:15-83 + helpers/GainFade.h:56-72, aux0 = root index
    OP_STOREBUF,   // stage boundary: in0 -> global per-voice block buffer (ptr), used around `convolve`
    OP_LOADBUF,    // stage boundary: global per-voice block buffer (ptr) -> out
    OP_PROMOTE,    // after the first OP_END: tap promotion record (w1 = root index, w2/w3 = src, w4/w5 = dst)
    // ---- sequencing / control nodes (SURVEY.md §8f N3) ----
    OP_ONCE,       // Core.h:341-404
    OP_SEQ,        // Core.h:407-573  (ptr = float[aux0] sequence; imm: offset, generation; mode bit0 hold, bit1 loop, bit2 has reset input)
    OP_SEQ2,       // Seq2.h:35-166   (same encoding, no generation)
    OP_SPARSEQ,    // SparSeq.h:17-377 (ptr = int32 tickTime[aux0] then float value[aux0]; imm block see graph_host.cpp)
    OP_SPARSEQ2,   // SparSeq2.h:17-141 (ptr = double time[aux0] then float value[aux0]; imm: generation; mode bit0 interpolate)
    OP_TIME,       // wasm/SampleTime.h:12-24 (LaunchParams::sampleTime)
    OP_METRO,      // wasm/Metro.h:10-71 ((aux0,aux1) = bits of double(intervalSamps))
    // ---- analysis nodes (SURVEY.md §8f N4): audio passes through, a per-voice record feeds processQueuedEvents ----
    OP_METER,      // Analyzers.h:20-69    state: min, max, readouts pushed since the host last drained them
    OP_SNAPSHOT,   // Analyzers.h:77-136   state: z, latest value, readouts pushed
    OP_SCOPE,      // Analyzers.h:146-255, wasm/FFT.h:17-139  ptr = ring [tile][aux1][SCOPE_RING][L]; aux0 = index of the write position in LaunchParams::dyn
    OP_CAPTURE,    // Capture.h:14-103     ptr = [tile][aux0 + CAPTURE_SCRATCH][L] (ring then scratch); state: lastIn, scratchSize, w, r, ready
    // ---- device node types registered at run time (elem_b200_register_node_type; reference: Runtime::registerNodeType, Runtime.h:105-106) ----
    OP_CUSTOM,     // aux0 = registered type index, aux1 = state floats; operands, then one immediate word: bits of float(sr).  Has a body
                   // only in a kernel specialised for the program (spec_host.h): the body text is compiled by NVRTC
    OP_COUNT_
};

// Chain step function codes (one table for the unary, binary and reducing node families of Math.h).
enum ChainFn : uint32_t {
    // unary: DefaultNodeTypes.h:54-67
    F_SIN = 0, F_COS, F_TAN, F_TANH, F_ASINH, F_LN, F_LOG10, F_LOG2, F_CEIL, F_FLOOR, F_ROUND, F_SQRT, F_EXP, F_ABS,
    // binary reducing: DefaultNodeTypes.h:80-86
    F_ADD = 16, F_SUB, F_MUL, F_DIV, F_MOD, F_MIN, F_MAX,
    // binary: DefaultNodeTypes.h:70-77
    F_LE = 32, F_LEQ, F_GE, F_GEQ, F_POW, F_EQ, F_AND, F_OR,
};
constexpr uint32_t CHAIN_REVERSED = 0x100;   // step computes fn(operand, acc) instead of fn(acc, operand)
inline bool chain_fn_is_unary(uint32_t fn) { return (fn & 0xFF) < 16; }

enum OperandKind : uint32_t { K_SLOT = 0, K_PARAM = 1, K_ZERO = 2 };

constexpr uint32_t OP_HEADER_WORDS = 8;
constexpr uint32_t NO_STATE = 0xFFFFFFFFu;
constexpr uint32_t STATE_DOUBLE_FLAG = 0x80000000u;   // stateMap entry: two consecutive rows holding double[Vpad]
constexpr uint32_t STATE_PAD = 0x7FFFFFFFu;           // stateMap entry: one unused shared-memory row (keeps doubles 8-byte aligned)
constexpr int MAX_ROOTS = 16;
constexpr int MAX_OUT_CHANNELS = 8;
constexpr int MAX_SLOTS = 255;
constexpr int MAX_PIPE = 4;                 // stages of the warp pipeline of one graph (LaunchParams::pipeW)
constexpr int MAX_DYN = 16;                 // per-launch dynamic scalars (ring positions the host mirrors)
constexpr int SCOPE_RING = 8192;            // MultiChannelRingBuffer default capacity (MultiChannelRingBuffer.h:17), 4 channels (Analyzers.h:149)
constexpr int SCOPE_CHANNELS = 4;
constexpr int CAPTURE_SCRATCH = 128;        // Capture.h:97

inline uint32_t make_w0(uint32_t opcode, uint32_t nWords, uint32_t outSlot, uint32_t mode) {
    return (opcode & 0xFF) | ((nWords & 0xFF) << 8) | ((outSlot & 0xFF) << 16) | ((mode & 0xFF) << 24);
}
#ifdef __CUDACC__
__host__ __device__
#endif
inline uint32_t make_operand(uint32_t kind, uint32_t index) { return (kind << 30) | (index & 0x3FFFFFFFu); }

// Per-block dynamic root state (host mirrors GainFade, helpers/GainFade.h:56-72): the fade ramp of a block is a
// pure function of (gain at block start, step, target), so it is passed by value with the launch.
struct RootDyn {
    float gain0;
    float step;
    float target;
    int   channel;   // root "channel" prop; <0 or >= nOut => contributes nothing (GraphRenderSequence.h:214-219)
};

// One launch = one voice group (topology class).
struct LaunchParams {
    const uint32_t* code;        // program words (device, 16-byte aligned)
    const uint32_t* stateMap;    // [nStateEntries] global row index (| STATE_DOUBLE_FLAG) or STATE_PAD
    const uint32_t* paramMap;    // [nParams] global row index of shared-memory parameter row i+1 (row 0 is zeros)
    float*          rows;        // group row storage: rows[row * Vpad + voice]
    const float*    inShared;    // [nIn][inStride] host inputs shared by all voices (or null)
    const float*    inVoice;     // [voice][nIn][inStride] per-voice inputs (or null)
    float*          outVoice;    // [voice][nOut][outStride] per-voice outputs (or null = mix only)
    float*          mixPartial;  // [tile][nOut][blockSize] per-tile partial mix (or null)
    int nStateEntries;
    int nStateRows;              // shared-memory state rows per warp
    int nParams;                 // parameter rows per warp (excluding the zero row)
    int nSlots;
    int Vpad;
    int nv;                      // voices in the group
    int voice0;                  // first global voice index of the group (outVoice/inVoice indexing)
    int tileWidth;               // L: voices per warp (power of two <= 32)
    int numSamples;
    int blockSize;
    int nIn;
    int nOut;
    int inStride;
    int outStride;
    int tileBase;                // index of this group's first tile in mixPartial
    uint32_t runMask;            // bit r: root r's sub-sequence runs this block; bit 16+r: root r promotes its taps
    long long sampleTime;        // int64 sample clock of this block's first sample (*userData of Runtime::process: wasm/Main.cpp:206-217)
    RootDyn roots[MAX_ROOTS];
    uint32_t dyn[MAX_DYN];
    // One wavetable of the program staged into shared memory by a TMA bulk copy at kernel start (single-group launches only):
    // OP_TABLE ops whose table pointer equals tableSrc read shared memory at float index tableSmem instead of global memory.
    const float* tableSrc;       // device copy of the resource (16-byte aligned, padded to a multiple of 16 bytes), or null
    int tableFloats;             // padded length in floats
    int tableSmem;               // float index of the staged copy in the CTA's dynamic shared memory, or -1
    // Stage pipeline (render_groups_pipe_kernel; one-voice groups, BASELINE config 5): the host cut the program into pipeW contiguous
    // stages; pipeW warps of ONE CTA share the graph's shared-memory area, warp w runs stage w, one sample tile behind warp w - 1.
    // Values crossing a stage boundary live in ring slots (pipeDepth buffers, buffer = tile index mod pipeDepth).  0 / 1 = not pipelined.
    int pipeW;
    int pipeRingBase;            // slot indices >= pipeRingBase are ring slots
    int pipeDepth;
    uint32_t pipeCode[MAX_PIPE];            // word offset of stage w's code behind `code`
    unsigned short pipeState[MAX_PIPE + 1]; // stage w owns stateMap entries [pipeState[w], pipeState[w + 1])
    unsigned short pipeSrow[MAX_PIPE];      // first shared-memory state row of stage w
    int promoteAt;               // word offset of the first OP_PROMOTE record behind `code`, -1 = the program has none
    // Engine option "k1_prefetch" (default 1).  The kernel chooses its latency-hiding paths (prologue rows staged by cp.async outside
    // the one-voice pipeline kernel, delay ring reads of a tile issued together, no program walk to find the tap promotion records) from what it sees: parameter-row delay
    // lengths and their distance from the tile's writes.  0 forces the plain paths those fall back to; it is a reference for tests
    // and A/B runs, not a tuning knob — both compute the same bits.
    int k1Prefetch;
};
constexpr int TABLE_SMEM_MAX_FLOATS = 8192;   // tables up to 32 KB are staged

} // namespace eb
