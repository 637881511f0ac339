// graph_host.h — host side of the B200 engine: the part of elem::Runtime (runtime/elem/Runtime.h:40-577) that
// is NOT the per-block walk: node table, instruction interpreter, DFS topological sort, root activation and
// fades, garbage collection, shared resources — plus what is new here: voice groups, device storage and the
// compilation of the sorted node list into a render program (program.h) for the fused kernel.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <map>
#include <memory>
#include <mutex>
#include <set>
#include <string>
#include <unordered_map>
#include <vector>

#include "kernels.h"
#include "program.h"
#include "value.h"

namespace eb {

// Same numbering as elem::ReturnCode (runtime/elem/Types.h:51-60); negative values are ours (CUDA failures).
namespace rc {
constexpr int Ok = 0, UnknownNodeType = 1, NodeNotFound = 2, NodeAlreadyExists = 3, NodeTypeAlreadyExists = 4,
              InvalidPropertyType = 5, InvalidPropertyValue = 6, InvariantViolation = 7, InvalidInstructionFormat = 8;
constexpr int CudaError = -1, BadArgument = -2;
}

enum class NodeKind : uint8_t {
    In, Unary, Binary, Reduce, Root, Const, Sr, Phasor, SPhasor, Counter, Accum, Latch, MaxHold, Rand,
    Delay, SDelay, Z, Pole, Env, Biquad, Prewarp, MM1p, Svf, SvfShelf, TapIn, TapOut, Table, Blep, Convolve,
    PassThrough,  // analysis nodes whose events are not produced: audio passes through
    Once, Seq, Seq2, SparSeq, SparSeq2, Time, Metro,  // sequencing / control nodes (SURVEY.md §8f N3)
    Meter, Snapshot, Scope, Capture, Fft,             // analysis nodes feeding processQueuedEvents (SURVEY.md §8f N4)
    Custom                                            // a device node type registered at run time (registerNodeType)
};

// A read-only device array owned jointly by the node that uploaded it and by every compiled program that points at it
// (sequence data of seq/seq2/sparseq/sparseq2: the reference hands such data to the audio thread through a
// RefCountedPool + SPSC queue, Core.h:447-466).
struct DeviceArray {
    void* d = nullptr;
    size_t bytes = 0, count = 0;
    bool planOnly = false;
    ~DeviceArray();
};

struct Inlet { int32_t source; int32_t channel; };

// Float mirror of helpers/GainFade.h:16-121 (only what RootNode uses).
struct GainFade {
    float current = 0.0f, target = 1.0f, step = 0.0f, inStep = 0.0f, outStep = 0.0f;
    void init(double sr);
    void setFadeInMs(double sr, double ms);
    void setFadeOutMs(double sr, double ms);
    void fadeIn()  { target = 1.0f; updateStep(); }
    void fadeOut() { target = 0.0f; updateStep(); }
    bool on() const { return target > 0.5f; }
    bool settled() const;
    void advance(int numSamples);   // what GainFade::process does to currentGain after a block
    void updateStep() { step = (current > target) ? outStep : inStep; }
};

struct Resource {
    std::string name;
    std::vector<std::vector<float>> channels;   // host copy (always float: AudioBufferResource.h:13-24)
    float* dChannel0 = nullptr;                 // device copy of channel 0 (padded with zeros to a multiple of 16 bytes: TMA bulk copies)
    size_t numSamples = 0;
};

struct ConvolverState;   // convolve.h
struct SpecKernel;       // spec_host.h
struct SpecJob;

struct Node {
    int32_t id = 0;
    NodeKind kind = NodeKind::Const;
    uint32_t fn = 0;                 // UnaryFn / BinaryFn / ReduceFn / blep mode
    std::string typeName;
    std::vector<Inlet> inlets;
    std::map<std::string, Value> props;

    int paramRow = -1;               // const / sr: per-voice parameter row
    int stateRow = -1;               // first scalar state row (even-aligned when it holds doubles)
    int mode = 0;                    // svf / svfshelf / mm1p mode
    int channel = 0;                 // in.channel, root.channel (-1 default for root)
    GainFade fade;                   // root
    int size = 0, length = 0;        // delay / sdelay
    bool ringDirty = true;           // (re)allocate + zero + reset writeIndex at next compile (Delays.h:92-95)
    float* ring = nullptr;
    size_t ringFloats = 0;
    uint32_t holdSamples = 0xFFFFFFFFu;   // maxhold
    std::string tapName;
    float* tapPrivate = nullptr;     // tapOut private delayBuffer
    std::shared_ptr<Resource> resource;   // table / convolve
    bool resourceDirty = false;
    std::shared_ptr<ConvolverState> conv;
    // seq / seq2 / sparseq / sparseq2 (Core.h:411-466, Seq2.h:39-84, SparSeq.h:40-124, SparSeq2.h:20-56)
    std::shared_ptr<DeviceArray> seqData;
    uint32_t seqGen = 0, loopGen = 0;
    bool seqHold = false, seqLoop = true, follow = false;
    uint64_t seqOffset = 0;
    int32_t loopStart = -1, loopEnd = -1, interpolate = 0;
    double tickIntervalSamples = 0.0;
    int64_t intervalSamps = 0;       // metro (wasm/Metro.h:24-34)
    // event side (SURVEY.md §8f N4).  Ring positions that evolve identically for every voice of the group are mirrored
    // on the host: scope's MultiChannelRingBuffer read/write positions (MultiChannelRingBuffer.h:36-96), metro's
    // eventFlag/lastOut (Metro.h:47-52).  capture's relayBuffer (Capture.h:62-72) is a host vector per voice.
    uint32_t scopeR = 0, scopeW = 0;
    bool metroFlag = false; float metroLastOut = 0.0f;
    std::vector<std::vector<float>> relay;
    std::vector<float> window;       // fft: Blackman-Harris window of the current size (wasm/FFT.h:49-62)
};

struct Program {
    std::vector<uint32_t> code;
    std::vector<uint32_t> stateMap;
    std::vector<uint32_t> paramMap;       // shared-memory parameter row i+1 <- global row paramMap[i]
    int nOps = 0;
    int nStateRows = 0;
    int nSlots = 1;
    int nIn = 0;
    bool usesHostInputs = false;
    std::vector<int32_t> rootIds;         // root index -> node id
    std::vector<int32_t> nodeIds;         // every node referenced (gc liveness)
    uint32_t* dCode = nullptr;
    uint32_t* dStateMap = nullptr;
    uint32_t* dParamMap = nullptr;
    bool planOnly = false;
    // warp pipeline of a one-voice program (LaunchParams::pipeW ...): filled by compile() when the program was cut
    int pipeW = 1, pipeRingBase = 0, pipeDepth = 1;
    uint32_t pipeCode[MAX_PIPE] = {0, 0, 0, 0};
    unsigned short pipeState[MAX_PIPE + 1] = {0, 0, 0, 0, 0}, pipeSrow[MAX_PIPE] = {0, 0, 0, 0};
    // K1 stages: stage k interprets code[stages[k].codeOffset ...]; after it the convolvers of that stage run (K3)
    struct Conv { int32_t node; float* in; float* out; int inChannel; };   // inChannel >= 0: K3 reads host input channel inChannel directly (no staging copy)
    struct Stage { uint32_t codeOffset = 0; std::vector<Conv> convolves; bool empty = false;   // empty: no K1 work in this stage
                   int promoteAt = -1; };   // LaunchParams::promoteAt of the stage's launch (relative to codeOffset)
    std::vector<Stage> stages;
    // `convolve -> root`: the last stage would only reload the convolver's output and apply the root — K3 does that in its epilogue
    // (convolve.h ConvEpilogue) and the stage's K1 launch is skipped.  fusedConvStage < 0: not fused.
    int fusedConvStage = -1, fusedConvIndex = 0, fusedRoot = 0;
    std::vector<float*> blockBuffers;     // [Vpad][blockSize] HBM buffers carrying values across stages
    std::vector<std::shared_ptr<DeviceArray>> pinned;   // device arrays the code points at
    struct EvNode { int32_t node; int root; };
    std::vector<EvNode> evNodes;          // event-emitting nodes in render order (GraphRenderSequence.h:189-198 walks nodeList)
    std::vector<int32_t> dynNodes;        // LaunchParams::dyn[i] belongs to node dynNodes[i]
    bool hasCustom = false;               // uses a registered device node type: only a specialised kernel can run it
    std::shared_ptr<SpecJob> specJob;     // K1 being / having been specialised for this program (option "specialize"); the interpreter runs until it is loaded
    const float* stagedTable = nullptr; int stagedTableFloats = 0;   // the wavetable K1 stages into shared memory with TMA (first `table` node that fits)
    ~Program();
};

struct Group {
    int v0 = 0, nv = 0, Vpad = 0;
    int tileWidth = 0;                    // L, fixed at first compile
    std::unordered_map<int32_t, Node> nodes;
    std::set<int32_t> currentRoots;
    float* dRows = nullptr;
    int rowsCap = 0, rowsUsed = 0;
    std::map<std::string, float*> tapShared;
    std::shared_ptr<Program> pending, active;
    bool codeDirty = false;               // a property that is baked into the program changed: recompile at the next process()
    std::vector<std::shared_ptr<Program>> superseded;   // queued but never run (rseqQueue, Runtime.h:133,277-285): still pin their nodes for gc
    int nTiles() const { return tileWidth ? (nv + tileWidth - 1) / tileWidth : 0; }
};

struct EngineOptions {
    int tileWidth = 0;            // 0 = choose per group from the voice count
    int warpsPerCta = 0;          // 0 = choose
    int targetTiles = 2048;       // shrink the tile width until about this many warps exist (measured optimum, profiles/)
    bool targetTilesSet = false;  // the option was given explicitly: no automatic choice (see Engine::midRangeDense)
    int niter = 0;                // 0 = default elements-per-lane per tile; 4 selects the T = 4 variant for L = 32
    bool batchGroups = true;      // launch all single-stage voice groups of one tile geometry together
    bool fuseChains = true;       // fold runs of element-wise nodes into one OP_CHAIN
    int specialize = 0;           // spec_host.h: NVRTC-compile K1 against each small single-stage program; 1 = on the compile-queue thread
                                  // (the interpreter serves meanwhile), 2 = wait for the compiler at COMMIT (benchmarks, parity runs)
    int specializeMaxWords = 512; // programs longer than this keep the interpreter (compile time grows with the unrolled program)
    bool fuseConvRoot = true;     // `convolve -> root`: root gain + per-voice output + partial mix in K3's epilogue, no K1 launch for the last stage
    int pipelineStages = 4;       // one-voice groups in the many-groups launch: cut the program into this many pipeline stages, one warp each
                                  // (render_groups_pipe_kernel; 0 / 1 = off).  Bit-identical to one warp per graph; worth 7 % on BASELINE
                                  // config 5 (0.77 against 0.83 ms per block, profiles/r02_o_*, r02_s_*) — per-op time grows with the number
                                  // of resident warps, so the gain is far from the stage count (DESIGN.md section 4)
    int specMinBlocks = 0;        // > 0: specialised kernels of the narrow geometries (1 < L < 32) are compiled for this many CTAs per SM (8 = 64 registers)
    bool specializeStrict = false; // a failed specialisation is an error (COMMIT returns 7 / process -1) instead of a silent stay on the interpreter
    bool k1Prefetch = true;       // LaunchParams::k1Prefetch: false forces K1's plain paths (the bit-identical reference of tests and A/B runs)
};

class Engine {
public:
    Engine(double sampleRate, int blockSize, int numVoices, int device);
    ~Engine();

    int applyInstructions(int voiceBegin, int voiceEnd, const char* json, size_t len);
    int setPropertyPerVoice(int32_t nodeId, const char* key, const double* values, int voiceBegin, int count);
    // Instruction-stream ingestion at scale (SURVEY.md §8f N2).  applyBinary: the SAME instruction stream in the binary encoding
    // documented in include/elem_b200.h (no text to parse: ids are int32, numbers float64, strings length-prefixed), decoded into the
    // same in-memory batch and run through the same interpreter — identical semantics and return codes.  setConstTable: a per-voice
    // property TABLE, values[p][count] float32 row-major -> `value` of const node nodeIds[p] for voices [voiceBegin, voiceBegin +
    // count): nProps copies straight from the caller's table, no per-value conversion, no JSON.
    int applyBinary(int voiceBegin, int voiceEnd, const void* data, size_t bytes);
    int setConstTable(const int32_t* nodeIds, int nProps, const float* values, int voiceBegin, int count);
    int addSharedResource(const char* name, const float* const* chans, size_t nCh, size_t nSamples);
    void pruneSharedResources();
    std::vector<std::string> listSharedResources() const;
    int gc(int voice, std::vector<int32_t>& pruned);
    void reset();

    // Runtime::process shape: planar host buffers; inputs broadcast to every voice; out = mix bus.
    int process(const float* const* in, size_t nIn, float* const* out, size_t nOut, size_t numSamples, const int64_t* sampleTime = nullptr);
    // Voice-major host buffers: in[voice][nIn][n] (may be null), out[voice][nOut][n] (may be null), mix (may be null).
    int processVoices(const float* in, size_t nIn, float* outVoices, float* mix, size_t nOut, size_t numSamples);
    // Device-resident: no host I/O, no synchronisation; used for throughput timing and by processVoices/process.
    int enqueueBlock(size_t nIn, size_t nOut, size_t numSamples, bool perVoiceIn, bool materialise, bool mix, bool allReduce = false);
    int synchronize();
    // Offline rendering (BASELINE config 5: minutes of audio per graph, nobody listening): numBlocks blocks of every voice, per-voice
    // output, no mix bus, no host round trip per block — blocks are enqueued back to back, the kernels write straight into chunk buffers
    // of `chunkBlocks` blocks ([voice][nOut][chunk] on the device), and finished chunks travel to hostOut[voice][nOut][numBlocks *
    // blockSize] on a copy stream while the next chunk renders.  The reference does the same job with OfflineRenderer.process in a loop.
    int renderOffline(size_t nOut, size_t numBlocks, float* hostOut, size_t chunkBlocks);

    // Cross-GPU mix bus (SURVEY.md §8e): peerExport() allocates this rank's exchange buffer and returns its CUDA IPC handle
    // (64 bytes); peerAttach() maps the buffers of all ranks (handles = world x 64 bytes, in rank order).  Afterwards
    // enqueueBlock(..., allReduce = true) leaves the sum over all ranks in the mix bus of every rank (K4, kernels.h).
    int peerExport(void* handleOut64);
    int peerAttach(int rank, int world, const void* handles);
    int peerStatus();   // 0 = ok, 1 = a peer did not answer within the spin bound
    int setOption(const char* key, double value);
    // Runtime::registerNodeType (Runtime.h:105-106,480-487) for a fused-kernel engine: a new node type is DEVICE code — the body of
    //   float node(float* s /* numState persistent floats per voice, zero-initialised */, const float* in /* numInputs samples */, float sr)
    // as CUDA C++ text, evaluated once per sample.  It is compiled (NVRTC) into the kernel specialised for every render program that
    // uses the type; numState = 0 makes it element-wise (all lanes), otherwise it runs in the lane that owns the voice.  Returns
    // NodeTypeAlreadyExists (4) for a builtin or already registered name, like the reference.
    int registerNodeType(const char* type, int numInputs, int numState, const char* body);
    bool hasNodeType(const char* type) const;
    void setStream(cudaStream_t s);
    float* mixDevicePtr() { return dMix_; }
    float* voiceOutDevicePtr() { return dOutVoice_; }
    float* voiceInDevicePtr(size_t nIn);
    float* sharedInDevicePtr(size_t nIn);
    std::string lastError() const { Lock lk(mu_); return lastError_; }
    int numVoices() const { return numVoices_; }
    int blockSize() const { return blockSize_; }
    uint64_t kernelLaunches() const { Lock lk(mu_); return launches_; }
    // The int64 sample clock handed to nodes through BlockContext::userData (wasm/Main.cpp:206-217, Metro.h:44,
    // SampleTime.h:19).  process() takes it from *userData when given; otherwise the engine counts samples itself.
    // Runtime::processQueuedEvents (Runtime.h:64,438-446): events of the voices [vb, ve); cb(type, event JSON, voice).
    typedef void (*EventFn)(const char* type, const char* json, int voice, void* user);
    int processQueuedEvents(int vb, int ve, EventFn cb, void* user);
    void setCurrentTime(int64_t t) { Lock lk(mu_); sampleTime_ = t; }
    int64_t currentTime() const { Lock lk(mu_); return sampleTime_; }
    // Sum of the device durations (ms) of the K1 render kernels launched since the last call, measured with
    // CUDA events recorded on the launching stream (option "time_kernels" = 1). Synchronises the stream.
    double takeKernelTimeMs(uint64_t* count);
    // K3 time/count gathered by the same takeKernelTimeMs() call
    double lastConvolveTimeMs(uint64_t* count) const { Lock lk(mu_); if (count) *count = lastConvCount_; return lastConvMs_; }
    // per kernel kind (0 = K1 render, 1 = K2 mix reduce, 2 = K3 convolve, 3 = K4 mix exchange): summed ms and launch counts of the same call
    void lastKernelTimes(double ms[4], uint64_t counts[4]) const { Lock lk(mu_); for (int i = 0; i < 4; ++i) { ms[i] = lastKindMs_[i]; counts[i] = lastKindCount_[i]; } }
    // A cross-GPU barrier on the render stream (K4 with an empty payload): returns once every rank's stream has reached it.
    int peerBarrier();
    std::string describe() const;
    // Runtime::snapshot() (Runtime.h:110,490-499): {"0x<node id, 8 hex digits>": {props...}, ...} of the voice group containing `voice`
    // (per-voice capable props report the value last set for the group's highest addressed voice, like any other prop the last write).
    std::string snapshot(int voice) const;
    // The encoded render program (program.h) of the voice group containing `voice` — the newest compiled one.  Introspection:
    // tests, and the input of per-program kernel specialisation (DESIGN.md §8).
    std::vector<uint32_t> programWords(int voice) const;
    // Compile (not load, not run) the specialised K1 of the voice group containing `voice`: returns the cubin size or -1, the
    // NVRTC log in `log`.  Works without a GPU (NVRTC is a pure compiler): the CPU test-suite uses it.
    long specializeDryRun(int voice, std::string& log);

private:
    // Threading contract of the boundary (Runtime.h:133,204,277-285: one control thread + one render thread, concurrently): every
    // public entry point takes this lock for its host-side work.  process()/processVoices() hold it only while they ENQUEUE the block
    // (tens of microseconds) and wait for the GPU without it, so the control thread works while a block renders; a control call
    // holds it while it mutates the node table / compiles (NVRTC never runs under it in "specialize" = 1 mode).  Recursive because
    // public methods call each other.
    mutable std::recursive_mutex mu_;
    typedef std::lock_guard<std::recursive_mutex> Lock;
    bool planDryRun_ = false;     // plan-only engines: enqueueBlock runs ALL its host logic and skips only the CUDA calls (thread-safety tests)
    double sr_;
    int blockSize_, numVoices_, device_;
    cudaStream_t stream_ = nullptr;
    bool ownStream_ = true;
    EngineOptions opt_;
    std::vector<std::unique_ptr<Group>> groups_;
    std::map<std::string, std::shared_ptr<Resource>> resources_;
    struct CustomType { std::string name, body; int nIn = 0, nState = 0; };
    std::vector<CustomType> customTypes_;
    std::string customSource() const;     // the generated device text of all registered types (part of the specialisation key)
    std::string lastError_;
    uint64_t launches_ = 0;
    int64_t sampleTime_ = 0;
    bool timeKernels_ = false;
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> timedEvents_, timedConvEvents_, timedMixEvents_, timedXchgEvents_, eventPool_;
    double lastConvMs_ = 0.0; uint64_t lastConvCount_ = 0;
    double lastKindMs_[4] = {0, 0, 0, 0}; uint64_t lastKindCount_[4] = {0, 0, 0, 0};   // K1, K2, K3, K4 of the latest takeKernelTimeMs()
    std::pair<cudaEvent_t, cudaEvent_t> timedBegin();

    // I/O staging
    float* dMix_ = nullptr;          // [MAX_OUT][blockSize]
    float* dMixScratch_ = nullptr;   // K2 group sums [MIX_REDUCE_MAX_GROUPS][MAX_OUT][blockSize]
    unsigned int* dMixTickets_ = nullptr;
    float* dPartial_ = nullptr; size_t partialFloats_ = 0;
    float* dOutVoice_ = nullptr; size_t outVoiceFloats_ = 0;
    float* dInVoice_ = nullptr; size_t inVoiceFloats_ = 0;
    float* dInShared_ = nullptr; size_t inSharedFloats_ = 0;
    float* hPinned_ = nullptr; size_t pinnedFloats_ = 0;
    // Host delivery of the mix bus (kernels.h HostDeliver): mapped pinned [MAX_OUT][blockSize] floats + the sequence word behind them.
    // process() arms it for the block it enqueues and polls the word instead of D2H copy + stream synchronize.
    float* hMixHost_ = nullptr; float* dMixHostAlias_ = nullptr;
    volatile uint32_t* hMixFlag_ = nullptr; uint32_t* dMixFlagAlias_ = nullptr;
    unsigned int* dDeliverDone_ = nullptr;
    uint32_t deliverSeq_ = 0;
    bool hostDeliver_ = true, processAllReduce_ = true;   // options "host_deliver", "process_allreduce"
    bool deliverArmed_ = false, deliverLaunched_ = false;
    HostDeliver takeDeliver();
    float* offlineDev_[2] = {nullptr, nullptr}; float* offlinePinned_[2] = {nullptr, nullptr}; size_t offlineChunkFloats_ = 0;   // renderOffline chunk buffers, kept across calls
    size_t curNOut_ = 0;
    struct BatchBuffers { LaunchParams* dDescs = nullptr; int* dTileStart = nullptr; size_t capGroups = 0; std::vector<char> lastDescs; };
    std::map<int, BatchBuffers> batch_;   // per tile width
    // Steady-state fast path for engines made of many batched voice groups (BASELINE config 5: 1250 graphs): when the last block found
    // every group steady — no queued program, nothing dirty, all root fades settled, no event mirrors to advance — and the call has the
    // same shape, the next block re-launches the cached buckets (the descriptors on the device are still right; the sample clock is a
    // kernel argument) without walking the groups.  Any instruction batch, gc, option or resource change invalidates it.
    struct SteadyBucket { int L, nGroups, totalTiles, maxSlots, maxState, maxParams, wpc, pipeStages, key; };
    static constexpr int PIPE_BUCKET = 1000;   // bucket key = tile width (+ PIPE_BUCKET for pipelined one-voice programs)
    std::vector<SteadyBucket> steadyBuckets_;
    bool steadyValid_ = false;
    size_t steadyKey_[6] = {0, 0, 0, 0, 0, 0};
    int steadyTiles_ = 0;
    float* offlineOut_ = nullptr; int offlineStride_ = 0, offlineOffset_ = 0;   // renderOffline: where materialised outputs go instead of dOutVoice_

    // K4 state
    void* dExchange_ = nullptr; size_t exchangeBytes_ = 0; size_t exchangeFlagOffset_ = 0, exchangeOwnOffset_ = 0;
    PeerMix peer_{}; bool peerAttached_ = false; uint32_t peerEpoch_ = 0; int* dPeerStatus_ = nullptr;
    std::vector<void*> peerMapped_;

    bool planOnly_ = false;
    bool cuda(cudaError_t e, const char* what);
    cudaError_t dmalloc(void** p, size_t bytes);
    void dfree(void* p);
    cudaError_t dmemset(void* p, int v, size_t bytes);
    cudaError_t dmemcpy(void* dst, const void* src, size_t bytes, cudaMemcpyKind kind);
    cudaError_t dmemcpySync(void* dst, const void* src, size_t bytes, cudaMemcpyKind kind);
    void dsync();
    void dsetdev();
    int fail(int code, const std::string& msg) { lastError_ = msg; return code; }

    // instruction interpreter (Runtime.h:170-433)
    int applyToGroup(Group& g, const std::vector<Value>& batch, int vb, int ve);
    int applyBatch(int vb, int ve, const std::vector<Value>& batch);
    int createNode(Group& g, const Value& id, const Value& type);
    int appendChild(Group& g, const Value& parent, const Value& child, const Value& chan);
    int setProperty(Group& g, const Value& id, const Value& key, const Value& val, int vb, int ve);
    int activateRoots(Group& g, const Value& roots);
    int nodeSetProperty(Group& g, Node& n, const std::string& key, const Value& val, int vb, int ve);
    bool isValueOnlyBatch(const std::vector<Value>& batch, int vb, int ve);
    int splitGroupsAt(int v);
    // 8192 <= voices < 131072 with specialised kernels: twice the warps (about 4096) from narrow-geometry kernels compiled for 8 CTAs per
    // SM (64 registers) — 6-18 % faster than ~2048 warps at 110 registers (profiles/r02_aa_midrange_voices_ab.txt)
    bool midRangeDense(int nv) const { return opt_.specialize > 0 && !opt_.targetTilesSet && opt_.tileWidth == 0 && opt_.specMinBlocks == 0 && nv >= 8192; }

    // storage
    int allocRows(Group& g, int count, bool evenAlign, int& row);
    int fillRow(Group& g, int row, int vb, int ve, float value);
    int fillRowBits(Group& g, int row, int vb, int ve, uint32_t bits);
    int ensureResourceOnDevice(Resource& r);
    int uploadArray(std::shared_ptr<DeviceArray>& out, const void* data, size_t bytes, size_t count);

    // compile (Runtime.h:521-577 + GraphRenderSequence.h:107-187)
    int compile(Group& g, int nIn, std::shared_ptr<Program>& out);
    void traverse(Group& g, std::set<int32_t>& visited, std::vector<int32_t>& order, int32_t n);
    int chooseTileWidth(int nv) const;
    int ensureBuffers(size_t nIn, size_t nOut, bool perVoiceIn, bool materialise);
    friend struct Compiler;
};

} // namespace eb
