// graph_host.cpp — see graph_host.h.  Reference behaviour mirrored here is cited inline as file:line of
// /root/reference (runtime/elem/...).
#include "graph_host.h"

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstring>
#include <functional>
#include <list>
#include <sstream>
#include <thread>

#include "convolve.h"
#include "kernels.h"
#include "spec_host.h"

namespace eb {

static inline void cpuRelax() {
#if defined(__x86_64__) || defined(__i386__)
    __builtin_ia32_pause();
#elif defined(__aarch64__)
    asm volatile("yield" ::: "memory");
#endif
}

// ---------------------------------------------------------------------------------------------------------
// GainFade mirror (helpers/GainFade.h)
static double msToStep(double sr, double ms) { return ms > 1e-6 ? 1.0 / (sr * ms / 1000.0) : 1.0; }   // :10-12

void GainFade::init(double sr) {            // GainFade(sr, 20, 20, 0.0, 1.0)  Core.h:80, GainFade.h:18-24
    current = 0.0f; target = 1.0f; step = 0.0f; inStep = 0.0f; outStep = 0.0f;
    setFadeInMs(sr, 20.0);
    setFadeOutMs(sr, 20.0);
}
void GainFade::setFadeInMs(double sr, double ms) { inStep = (float) msToStep(sr, ms); updateStep(); }              // :74-77
void GainFade::setFadeOutMs(double sr, double ms) { outStep = (float) ((double) -1.0f * msToStep(sr, ms)); updateStep(); }   // :79-82
bool GainFade::settled() const { return std::fabs(target - current) <= 1e-6f; }                                     // :102-104
void GainFade::advance(int n) {                                                                                  // :56-72
    if (current == target) return;
    float v = current + step * (float) n;
    current = v < 0.0f ? 0.0f : (v > 1.0f ? 1.0f : v);
}


// ---------------------------------------------------------------------------------------------------------
// Device-memory shims.  In "plan-only" mode (device == -1; used by the CPU test-suite to exercise the host
// logic: instruction interpreter, return codes, gc, compilation) they fall back to host memory so that the
// graph compiler can run without a GPU.  Plan-only engines can NOT render: every process call fails loudly.
static void rawFree(void* p, bool plan) { if (!p) return; if (plan) std::free(p); else cudaFree(p); }

cudaError_t Engine::dmalloc(void** p, size_t bytes) {
    if (planOnly_) { *p = std::calloc(1, bytes ? bytes : 1); return *p ? cudaSuccess : cudaErrorMemoryAllocation; }
    return cudaMalloc(p, bytes);
}
void Engine::dfree(void* p) { rawFree(p, planOnly_); }
cudaError_t Engine::dmemset(void* p, int v, size_t bytes) {
    if (planOnly_) { std::memset(p, v, bytes); return cudaSuccess; }
    return cudaMemsetAsync(p, v, bytes, stream_);
}
cudaError_t Engine::dmemcpy(void* dst, const void* src, size_t bytes, cudaMemcpyKind kind) {
    if (planOnly_) { std::memmove(dst, src, bytes); return cudaSuccess; }
    return cudaMemcpyAsync(dst, src, bytes, kind, stream_);
}
cudaError_t Engine::dmemcpySync(void* dst, const void* src, size_t bytes, cudaMemcpyKind kind) {
    if (planOnly_) { std::memmove(dst, src, bytes); return cudaSuccess; }
    cudaError_t e = cudaMemcpyAsync(dst, src, bytes, kind, stream_);
    if (e != cudaSuccess) return e;
    return cudaStreamSynchronize(stream_);
}
void Engine::dsync() { if (!planOnly_ && stream_) cudaStreamSynchronize(stream_); }
void Engine::dsetdev() { if (!planOnly_) cudaSetDevice(device_); }
void Engine::setStream(cudaStream_t s) {
    Lock lk(mu_);
    if (planOnly_) return;
    if (ownStream_ && stream_) { cudaStreamSynchronize(stream_); cudaStreamDestroy(stream_); }
    stream_ = s; ownStream_ = false;
}

// ---------------------------------------------------------------------------------------------------------
Program::~Program() {
    if (dCode) rawFree(dCode, planOnly);      // stateMap / paramMap live in the same allocation
    for (float* p : blockBuffers) rawFree(p, planOnly);
}

DeviceArray::~DeviceArray() { if (d) rawFree(d, planOnly); }

struct TypeInfo { NodeKind kind; uint32_t fn; int stateRows; bool evenAlign; };

// Registered builtin names: DefaultNodeTypes.h:53-143 (+ "convolve", "metro", "time": wasm/Main.cpp:47-61).  Types that
// are out of scope (SURVEY.md §2d: sample*, mc.*) are deliberately absent and yield UnknownNodeType like any
// unregistered name (Runtime.h:304-305).
static const std::unordered_map<std::string, TypeInfo>& typeTable() {
    static const std::unordered_map<std::string, TypeInfo> t = {
        {"in", {NodeKind::In, 0, 0, false}},
        {"sin", {NodeKind::Unary, F_SIN, 0, false}}, {"cos", {NodeKind::Unary, F_COS, 0, false}},
        {"tan", {NodeKind::Unary, F_TAN, 0, false}}, {"tanh", {NodeKind::Unary, F_TANH, 0, false}},
        {"asinh", {NodeKind::Unary, F_ASINH, 0, false}}, {"ln", {NodeKind::Unary, F_LN, 0, false}},
        {"log", {NodeKind::Unary, F_LOG10, 0, false}}, {"log2", {NodeKind::Unary, F_LOG2, 0, false}},
        {"ceil", {NodeKind::Unary, F_CEIL, 0, false}}, {"floor", {NodeKind::Unary, F_FLOOR, 0, false}},
        {"round", {NodeKind::Unary, F_ROUND, 0, false}}, {"sqrt", {NodeKind::Unary, F_SQRT, 0, false}},
        {"exp", {NodeKind::Unary, F_EXP, 0, false}}, {"abs", {NodeKind::Unary, F_ABS, 0, false}},
        {"le", {NodeKind::Binary, F_LE, 0, false}}, {"leq", {NodeKind::Binary, F_LEQ, 0, false}},
        {"ge", {NodeKind::Binary, F_GE, 0, false}}, {"geq", {NodeKind::Binary, F_GEQ, 0, false}},
        {"pow", {NodeKind::Binary, F_POW, 0, false}}, {"eq", {NodeKind::Binary, F_EQ, 0, false}},
        {"and", {NodeKind::Binary, F_AND, 0, false}}, {"or", {NodeKind::Binary, F_OR, 0, false}},
        {"add", {NodeKind::Reduce, F_ADD, 0, false}}, {"sub", {NodeKind::Reduce, F_SUB, 0, false}},
        {"mul", {NodeKind::Reduce, F_MUL, 0, false}}, {"div", {NodeKind::Reduce, F_DIV, 0, false}},
        {"mod", {NodeKind::Reduce, F_MOD, 0, false}}, {"min", {NodeKind::Reduce, F_MIN, 0, false}},
        {"max", {NodeKind::Reduce, F_MAX, 0, false}},
        {"root", {NodeKind::Root, 0, 0, false}}, {"const", {NodeKind::Const, 0, 0, false}},
        {"sr", {NodeKind::Sr, 0, 0, false}},
        {"phasor", {NodeKind::Phasor, 0, 1, false}}, {"sphasor", {NodeKind::SPhasor, 0, 2, false}},
        {"counter", {NodeKind::Counter, 0, 1, false}}, {"accum", {NodeKind::Accum, 0, 2, false}},
        {"latch", {NodeKind::Latch, 0, 2, false}}, {"maxhold", {NodeKind::MaxHold, 0, 3, false}},
        {"rand", {NodeKind::Rand, 0, 1, false}},
        {"delay", {NodeKind::Delay, 0, 1, false}}, {"sdelay", {NodeKind::SDelay, 0, 1, false}},
        {"z", {NodeKind::Z, 0, 1, false}},
        {"pole", {NodeKind::Pole, 0, 1, false}}, {"env", {NodeKind::Env, 0, 1, false}},
        {"biquad", {NodeKind::Biquad, 0, 2, false}}, {"prewarp", {NodeKind::Prewarp, 0, 0, false}},
        {"mm1p", {NodeKind::MM1p, 0, 2, true}}, {"svf", {NodeKind::Svf, 0, 4, true}},
        {"svfshelf", {NodeKind::SvfShelf, 0, 4, true}},
        {"tapIn", {NodeKind::TapIn, 0, 0, false}}, {"tapOut", {NodeKind::TapOut, 0, 0, false}},
        {"table", {NodeKind::Table, 0, 0, false}},
        {"blepsaw", {NodeKind::Blep, 0, 2, false}}, {"blepsquare", {NodeKind::Blep, 1, 2, false}},
        {"bleptriangle", {NodeKind::Blep, 2, 2, false}},
        {"convolve", {NodeKind::Convolve, 0, 0, false}},
        {"once", {NodeKind::Once, 0, 4, false}}, {"seq", {NodeKind::Seq, 0, 6, false}},
        {"seq2", {NodeKind::Seq2, 0, 3, false}}, {"sparseq", {NodeKind::SparSeq, 0, 13, false}},
        {"sparseq2", {NodeKind::SparSeq2, 0, 3, false}},
        {"time", {NodeKind::Time, 0, 0, false}}, {"metro", {NodeKind::Metro, 0, 0, false}},
        {"meter", {NodeKind::Meter, 0, 3, false}}, {"snapshot", {NodeKind::Snapshot, 0, 3, false}},
        {"scope", {NodeKind::Scope, 0, 0, false}}, {"capture", {NodeKind::Capture, 0, 5, false}},
        {"fft", {NodeKind::Fft, 0, 0, false}},
    };
    return t;
}

static int bitceil(int n) {   // helpers/BitUtils.h:9
    if ((n & (n - 1)) == 0) return n;
    int o = 1;
    while (o < n) o <<= 1;
    return o;
}

// ---------------------------------------------------------------------------------------------------------
Engine::Engine(double sampleRate, int blockSize, int numVoices, int device)
    : sr_(sampleRate), blockSize_(blockSize), numVoices_(numVoices), device_(device) {
    if (numVoices_ < 1) numVoices_ = 1;
    planOnly_ = device_ < 0;
    if (!planOnly_) {
        cuda(cudaSetDevice(device_), "cudaSetDevice");
        cuda(cudaStreamCreateWithFlags(&stream_, cudaStreamNonBlocking), "cudaStreamCreate");
    }
    auto g = std::make_unique<Group>();
    g->v0 = 0; g->nv = numVoices_; g->Vpad = (numVoices_ + 31) / 32 * 32;
    groups_.push_back(std::move(g));
    cuda(dmalloc((void**) &dMix_, sizeof(float) * MAX_OUT_CHANNELS * blockSize_), "cudaMalloc mix");
    if (dMix_) cuda(dmemset(dMix_, 0, sizeof(float) * MAX_OUT_CHANNELS * blockSize_), "memset mix");
    if (!planOnly_) {
        const size_t tick = (size_t) MAX_OUT_CHANNELS * ((blockSize_ + 31) / 32);
        cuda(cudaMalloc((void**) &dMixScratch_, sizeof(float) * MIX_REDUCE_MAX_GROUPS * MAX_OUT_CHANNELS * blockSize_), "cudaMalloc mix scratch");
        cuda(cudaMalloc((void**) &dMixTickets_, sizeof(unsigned int) * tick), "cudaMalloc mix tickets");
        if (dMixTickets_) cuda(cudaMemsetAsync(dMixTickets_, 0, sizeof(unsigned int) * tick, stream_), "memset mix tickets");
        // mapped pinned mix bus + sequence word (HostDeliver); a failure here only disables the fast hand-over
        const size_t mixFloats = (size_t) MAX_OUT_CHANNELS * blockSize_;
        if (cudaHostAlloc((void**) &hMixHost_, sizeof(float) * mixFloats + 64, cudaHostAllocMapped) == cudaSuccess) {
            std::memset(hMixHost_, 0, sizeof(float) * mixFloats + 64);
            hMixFlag_ = reinterpret_cast<volatile uint32_t*>(hMixHost_ + mixFloats);
            void* d = nullptr;
            if (cudaHostGetDevicePointer(&d, hMixHost_, 0) == cudaSuccess && cudaMalloc((void**) &dDeliverDone_, sizeof(unsigned int)) == cudaSuccess) {
                dMixHostAlias_ = static_cast<float*>(d);
                dMixFlagAlias_ = reinterpret_cast<uint32_t*>(dMixHostAlias_ + mixFloats);
                cudaMemsetAsync(dDeliverDone_, 0, sizeof(unsigned int), stream_);
            } else { cudaFreeHost(hMixHost_); hMixHost_ = nullptr; hMixFlag_ = nullptr; }
        } else { hMixHost_ = nullptr; cudaGetLastError(); }
    }
}

static void freeGroupStorage(Group& g, bool plan) {
    for (auto& kv : g.nodes) {
        if (kv.second.ring) rawFree(kv.second.ring, plan);
        if (kv.second.tapPrivate) rawFree(kv.second.tapPrivate, plan);
    }
    for (auto& kv : g.tapShared) if (kv.second) rawFree(kv.second, plan);
    if (g.dRows) rawFree(g.dRows, plan);
}

Engine::~Engine() {
    dsetdev();
    dsync();
    for (auto& g : groups_) freeGroupStorage(*g, planOnly_);
    groups_.clear();
    for (auto& kv : resources_) if (kv.second->dChannel0) dfree(kv.second->dChannel0);
    for (void* m : peerMapped_) cudaIpcCloseMemHandle(m);
    if (dExchange_) cudaFree(dExchange_);
    if (dPeerStatus_) cudaFree(dPeerStatus_);
    if (dMix_) dfree(dMix_);
    if (dMixScratch_) cudaFree(dMixScratch_);
    if (dMixTickets_) cudaFree(dMixTickets_);
    if (dPartial_) dfree(dPartial_);
    if (dOutVoice_) dfree(dOutVoice_);
    if (dInVoice_) dfree(dInVoice_);
    if (dInShared_) dfree(dInShared_);
    if (hPinned_ && !planOnly_) cudaFreeHost(hPinned_);
    if (hMixHost_) cudaFreeHost(hMixHost_);
    for (int i = 0; i < 2; ++i) { if (offlineDev_[i]) cudaFree(offlineDev_[i]); if (offlinePinned_[i]) cudaFreeHost(offlinePinned_[i]); }
    if (dDeliverDone_) cudaFree(dDeliverDone_);
    for (auto& kv : batch_) { if (kv.second.dDescs) dfree(kv.second.dDescs); if (kv.second.dTileStart) dfree(kv.second.dTileStart); }
    for (auto* l : {&timedEvents_, &timedMixEvents_, &timedConvEvents_, &timedXchgEvents_})
        for (auto& ev : *l) { cudaEventDestroy(ev.first); cudaEventDestroy(ev.second); }
    for (auto& ev : eventPool_) { cudaEventDestroy(ev.first); cudaEventDestroy(ev.second); }
    if (ownStream_ && stream_) cudaStreamDestroy(stream_);
}

bool Engine::cuda(cudaError_t e, const char* what) {
    if (e == cudaSuccess) return true;
    lastError_ = std::string(what) + ": " + cudaGetErrorString(e);
    return false;
}

int Engine::setOption(const char* key, double value) {
    Lock lk(mu_);
    steadyValid_ = false;
    const std::string k(key);
    if (k == "tile_width") { opt_.tileWidth = (int) value; }
    else if (k == "warps_per_cta") { opt_.warpsPerCta = (int) value; }
    else if (k == "target_tiles") { opt_.targetTiles = (int) value; opt_.targetTilesSet = true; }
    else if (k == "niter") { opt_.niter = (int) value; }
    else if (k == "batch_groups") { opt_.batchGroups = value != 0; }
    else if (k == "fuse_chains") { opt_.fuseChains = value != 0; }
    else if (k == "specialize") { opt_.specialize = (int) value; }
    else if (k == "specialize_max_words") { opt_.specializeMaxWords = (int) value; }
    else if (k == "specialize_strict") { opt_.specializeStrict = value != 0; }
    else if (k == "spec_minblocks") { opt_.specMinBlocks = (int) value; }
    else if (k == "k1_prefetch") { opt_.k1Prefetch = value != 0; }
    else if (k == "time_kernels") { timeKernels_ = value != 0 && !planOnly_; }
    else if (k == "fuse_conv_root") { opt_.fuseConvRoot = value != 0; }
    else if (k == "pipeline_stages") { opt_.pipelineStages = std::max(0, std::min((int) value, (int) MAX_PIPE)); }
    else if (k == "host_deliver") { hostDeliver_ = value != 0; }
    else if (k == "process_allreduce") { processAllReduce_ = value != 0; }
    else if (k == "plan_dry_run") { planDryRun_ = value != 0 && planOnly_; }
    else return rc::BadArgument;
    return rc::Ok;
}

std::string Engine::describe() const {
    Lock lk(mu_);
    std::ostringstream os;
    os << "{\"voices\":" << numVoices_ << ",\"groups\":[";
    bool first = true;
    for (auto& g : groups_) {
        if (!first) os << ",";
        first = false;
        os << "{\"v0\":" << g->v0 << ",\"nv\":" << g->nv << ",\"tile_width\":" << g->tileWidth << ",\"nodes\":" << g->nodes.size();
        if (g->pending || g->active) {
            auto& p = g->pending ? g->pending : g->active;
            os << ",\"slots\":" << p->nSlots << ",\"state_rows\":" << p->nStateRows << ",\"params\":" << p->paramMap.size() << ",\"ops\":" << p->nOps << ",\"code_words\":" << p->code.size()
               << ",\"promote_at\":" << (p->stages.empty() ? -1 : p->stages.back().promoteAt)
               << ",\"roots\":" << p->rootIds.size() << ",\"pipeline_stages\":" << p->pipeW;
            if (p->specJob) {
                const int st = p->specJob->state.load(std::memory_order_acquire);
                os << ",\"spec_state\":" << st << ",\"spec_cubin_bytes\":" << (st > 0 ? p->specJob->kernel.cubin.size() : 0);
                if (st == 2) os << ",\"spec_regs\":" << p->specJob->kernel.numRegs << ",\"spec_local_bytes\":" << p->specJob->kernel.localBytes;
                if (st < 0) {   // the compiler / loader log, JSON-escaped
                    os << ",\"spec_log\":\"";
                    for (char c : p->specJob->log) {
                        if (c == '"' || c == '\\') os << '\\' << c;
                        else if (c == '\n') os << "\\n";
                        else if ((unsigned char) c >= 0x20) os << c;
                    }
                    os << "\"";
                }
            }
        }
        os << "}";
    }
    os << "]}";
    return os.str();
}

std::string Engine::snapshot(int voice) const {
    Lock lk(mu_);
    std::string o = "{";
    for (auto& g : groups_) {
        if (voice < g->v0 || voice >= g->v0 + g->nv) continue;
        std::map<int32_t, const Node*> sorted;
        for (auto& kv : g->nodes) sorted[kv.first] = &kv.second;
        bool first = true;
        for (auto& kv : sorted) {
            char key[24];
            std::snprintf(key, sizeof key, "\"0x%08x\":", (unsigned) kv.first);    // nodeIdToHex, Types.h:16-27
            if (!first) o += ',';
            first = false;
            o += key;
            Value props = Value::object();
            for (auto& p : kv.second->props) props.asObject()[p.first] = p.second;
            writeJson(o, props);
        }
        break;
    }
    return o + "}";
}

long Engine::specializeDryRun(int voice, std::string& log) {
    Lock lk(mu_);
    for (auto& g : groups_) {
        if (voice < g->v0 || voice >= g->v0 + g->nv) continue;
        auto& p = g->pending ? g->pending : g->active;
        if (!p) { log = "no compiled program for this voice"; return -1; }
        if (p->stages.size() > 1) { log = "multi-stage programs (convolve) are not specialised"; return -1; }
        SpecKernel k;
        if (!specialise_compile(p->code, g->tileWidth, opt_.niter, customSource(), k, log, opt_.specMinBlocks)) return -1;
        return (long) k.cubin.size();
    }
    log = "voice out of range";
    return -1;
}

std::vector<uint32_t> Engine::programWords(int voice) const {
    Lock lk(mu_);
    for (auto& g : groups_) {
        if (voice < g->v0 || voice >= g->v0 + g->nv) continue;
        auto& p = g->pending ? g->pending : g->active;
        if (p) return p->code;
    }
    return {};
}

// ---------------------------------------------------------------------------------------------------------
// storage
int Engine::allocRows(Group& g, int count, bool evenAlign, int& row) {
    int start = g.rowsUsed;
    if (evenAlign && (start & 1)) ++start;
    const int need = start + count;
    if (need > g.rowsCap) {
        int cap = std::max(64, g.rowsCap * 2);
        while (cap < need) cap *= 2;
        float* nb = nullptr;
        if (!cuda(dmalloc((void**) &nb, sizeof(float) * (size_t) cap * g.Vpad), "cudaMalloc rows")) return rc::CudaError;
        if (!cuda(dmemset(nb, 0, sizeof(float) * (size_t) cap * g.Vpad), "memset rows")) return rc::CudaError;
        if (g.dRows) {
            if (!cuda(dmemcpy(nb, g.dRows, sizeof(float) * (size_t) g.rowsUsed * g.Vpad, cudaMemcpyDeviceToDevice), "copy rows")) return rc::CudaError;
            dsync();
            dfree(g.dRows);
        }
        g.dRows = nb;
        g.rowsCap = cap;
    }
    row = start;
    g.rowsUsed = need;
    return rc::Ok;
}

int Engine::fillRowBits(Group& g, int row, int vb, int ve, uint32_t bits) {
    if (row < 0) return rc::Ok;
    const int n = ve - vb;
    if (n <= 0) return rc::Ok;
    uint32_t* p = reinterpret_cast<uint32_t*>(g.dRows + (size_t) row * g.Vpad + vb);
    if (bits == 0) return cuda(dmemset(p, 0, sizeof(float) * n), "memset row") ? rc::Ok : rc::CudaError;
    // cudaMemcpyAsync from PAGEABLE host memory returns once the source has been copied to the driver's staging buffer (CUDA runtime
    // API, "API synchronization behavior"): tmp may die right after the call, no stream synchronisation needed — a graph with fifty
    // consts used to cost fifty of them (config 5 set-up: 1250 graphs).
    std::vector<uint32_t> tmp((size_t) n, bits);
    if (!cuda(dmemcpy(p, tmp.data(), sizeof(uint32_t) * n, cudaMemcpyHostToDevice), "fill row")) return rc::CudaError;
    return rc::Ok;
}

int Engine::fillRow(Group& g, int row, int vb, int ve, float value) {
    uint32_t bits;
    std::memcpy(&bits, &value, 4);
    return fillRowBits(g, row, vb, ve, bits);
}

int Engine::ensureResourceOnDevice(Resource& r) {
    if (r.dChannel0 || r.numSamples == 0) return rc::Ok;
    const size_t padded = (r.numSamples + 3) / 4 * 4;
    if (!cuda(dmalloc((void**) &r.dChannel0, sizeof(float) * padded), "cudaMalloc resource")) return rc::CudaError;
    if (!cuda(dmemset(r.dChannel0, 0, sizeof(float) * padded), "memset resource")) return rc::CudaError;
    if (!cuda(dmemcpySync(r.dChannel0, r.channels[0].data(), sizeof(float) * r.numSamples, cudaMemcpyHostToDevice), "upload resource")) return rc::CudaError;
    return rc::Ok;
}

int Engine::uploadArray(std::shared_ptr<DeviceArray>& out, const void* data, size_t bytes, size_t count) {
    auto a = std::make_shared<DeviceArray>();
    a->planOnly = planOnly_; a->bytes = bytes; a->count = count;
    if (!cuda(dmalloc(&a->d, std::max<size_t>(bytes, 16)), "cudaMalloc sequence data")) return rc::CudaError;
    if (bytes && !cuda(dmemcpySync(a->d, data, bytes, cudaMemcpyHostToDevice), "upload sequence data")) return rc::CudaError;
    out = a;   // programs compiled against the previous array keep it alive until they are released
    return rc::Ok;
}

int Engine::addSharedResource(const char* name, const float* const* chans, size_t nCh, size_t nSamples) {
    Lock lk(mu_);
    // insert-only: SharedResource.h:44-46 (emplace fails on an existing key)
    if (resources_.count(name)) return 0;
    auto r = std::make_shared<Resource>();
    r->name = name;
    r->numSamples = nSamples;
    for (size_t c = 0; c < nCh; ++c) r->channels.emplace_back(chans[c], chans[c] + nSamples);   // copied in: AudioBufferResource.h:13-24
    if (nCh == 0) r->numSamples = 0;
    resources_[name] = r;
    return 1;
}

void Engine::pruneSharedResources() {
    Lock lk(mu_);   // SharedResource.h:93-101: drop entries nobody else references
    dsync();
    for (auto it = resources_.begin(); it != resources_.end();) {
        if (it->second.use_count() == 1) {
            if (it->second->dChannel0) dfree(it->second->dChannel0);
            it = resources_.erase(it);
        } else ++it;
    }
}

std::vector<std::string> Engine::listSharedResources() const {
    Lock lk(mu_);
    std::vector<std::string> out;
    for (auto& kv : resources_) out.push_back(kv.first);
    return out;
}

// ---------------------------------------------------------------------------------------------------------
// instruction interpreter
static bool toInt32(const Value& v, int32_t& out) {
    if (!v.isNumber()) return false;
    out = static_cast<int32_t>(v.asNumber());   // Runtime.h:299
    return true;
}

// builtin or registered: kind, fn (registered types: their index), state rows
static bool lookupType(const std::string& name, const std::vector<std::pair<std::string, int>>& custom, TypeInfo& out) {
    auto it = typeTable().find(name);
    if (it != typeTable().end()) { out = it->second; return true; }
    for (size_t i = 0; i < custom.size(); ++i)
        if (custom[i].first == name) { out = TypeInfo{NodeKind::Custom, (uint32_t) i, custom[i].second, false}; return true; }
    return false;
}

int Engine::registerNodeType(const char* type, int numInputs, int numState, const char* body) {
    Lock lk(mu_);
    if (!type || !body || numInputs < 0 || numInputs > 8 || numState < 0 || numState > 8) return fail(rc::BadArgument, "registerNodeType: 0..8 inputs, 0..8 state floats");
    if (hasNodeType(type)) return rc::NodeTypeAlreadyExists;     // Runtime.h:482-483
    customTypes_.push_back(CustomType{type, body, numInputs, numState});
    return rc::Ok;
}

bool Engine::hasNodeType(const char* type) const {
    Lock lk(mu_);
    if (typeTable().count(type)) return true;
    for (auto& c : customTypes_) if (c.name == type) return true;
    return false;
}

std::string Engine::customSource() const {
    if (customTypes_.empty()) return std::string();
    std::ostringstream os;
    os << "#define EB_CUSTOM_NODES 1\nnamespace eb {\n";
    for (size_t i = 0; i < customTypes_.size(); ++i)
        os << "// registered node type \"" << customTypes_[i].name << "\"\n__device__ __forceinline__ float eb_custom_" << i
           << "(float* s, const float* in, const float sr) {\n" << customTypes_[i].body << "\n}\n";
    os << "template <int ID> __device__ __forceinline__ float eb_custom_call(float* s, const float* in, const float sr) {\n";
    for (size_t i = 0; i < customTypes_.size(); ++i) os << "    if constexpr (ID == " << i << ") return eb_custom_" << i << "(s, in, sr);\n";
    os << "    return 0.0f;\n}\n}\n";
    return os.str();
}

int Engine::createNode(Group& g, const Value& a1, const Value& a2) {   // Runtime.h:294-313
    int32_t id;
    if (!toInt32(a1, id) || !a2.isString()) return rc::InvalidInstructionFormat;
    std::vector<std::pair<std::string, int>> custom;
    for (auto& c : customTypes_) custom.push_back({c.name, c.nState});
    TypeInfo ti;
    if (!lookupType(a2.asString(), custom, ti)) return rc::UnknownNodeType;
    struct { TypeInfo second; } holder{ti};
    auto* it = &holder;
    if (g.nodes.count(id)) return rc::NodeAlreadyExists;

    Node n;
    n.id = id;
    n.kind = it->second.kind;
    n.fn = it->second.fn;
    n.typeName = a2.asString();
    if (it->second.stateRows > 0) {
        int r = allocRows(g, it->second.stateRows, it->second.evenAlign, n.stateRow);
        if (r != rc::Ok) return r;
    }
    switch (n.kind) {
        case NodeKind::Const: {   // Core.h:166 default 1
            int r = allocRows(g, 1, false, n.paramRow);
            if (r != rc::Ok) return r;
            if ((r = fillRow(g, n.paramRow, 0, g.nv, 1.0f)) != rc::Ok) return r;
        } break;
        case NodeKind::Sr: {      // Core.h:173-180
            int r = allocRows(g, 1, false, n.paramRow);
            if (r != rc::Ok) return r;
            if ((r = fillRow(g, n.paramRow, 0, g.nv, (float) sr_)) != rc::Ok) return r;
        } break;
        case NodeKind::Root: n.fade.init(sr_); n.channel = -1; break;          // Core.h:80-82
        case NodeKind::Delay: n.size = blockSize_; n.ringDirty = true; break;  // Delays.h:56
        case NodeKind::SDelay: n.length = blockSize_; n.size = bitceil(blockSize_ + blockSize_); n.ringDirty = true; break;   // Delays.h:183,197-198
        case NodeKind::SparSeq: {   // SparSeq.h:353,342-345: edgeCount = -1, loopPoints = {-1, -1}
            for (int k : {2, 5, 6}) { int r = fillRowBits(g, n.stateRow + k, 0, g.Vpad, 0xFFFFFFFFu); if (r != rc::Ok) return r; }
        } break;
        case NodeKind::Metro: n.intervalSamps = static_cast<int64_t>(std::max(2.0, 1000.0 * 0.001 * sr_)); break;   // Metro.h:14-18
        case NodeKind::Scope:   // Analyzers.h:147-153: the constructor sets both props
            n.props["channels"] = Value::number(1); n.props["size"] = Value::number(512);
            n.size = SCOPE_CHANNELS * SCOPE_RING; break;
        case NodeKind::Capture: n.size = bitceil((int) (size_t) sr_) + CAPTURE_SCRATCH; break;   // Capture.h:17
        case NodeKind::Fft: {   // wasm/FFT.h:18-26: ring of one channel, default size 1024 set through setProperty
            n.size = SCOPE_RING;
            Node& ref = g.nodes.emplace(id, std::move(n)).first->second;
            return nodeSetProperty(g, ref, "size", Value::number(1024), 0, g.nv);
        }
        default: break;
    }
    g.nodes.emplace(id, std::move(n));
    return rc::Ok;
}

int Engine::appendChild(Group& g, const Value& a1, const Value& a2, const Value& a3) {   // Runtime.h:336-366
    int32_t parent, child, chan;
    if (!toInt32(a1, parent) || !toInt32(a2, child) || !toInt32(a3, chan)) return rc::InvalidInstructionFormat;
    auto p = g.nodes.find(parent);
    if (p == g.nodes.end()) return rc::NodeNotFound;
    if (!g.nodes.count(child)) return rc::NodeNotFound;
    p->second.inlets.push_back(Inlet{child, chan});
    return rc::Ok;
}

int Engine::nodeSetProperty(Group& g, Node& n, const std::string& key, const Value& val, int vb, int ve) {
    // vb/ve are group-relative voice bounds; only per-voice capable props honour a sub-range.
    switch (n.kind) {
        case NodeKind::Const:
            if (key == "value") {   // Core.h:142-152
                if (!val.isNumber()) return rc::InvalidPropertyType;
                int r = fillRow(g, n.paramRow, vb, ve, (float) val.asNumber());
                if (r != rc::Ok) return r;
            }
            break;
        case NodeKind::Root:        // Core.h:33-64
            if (key == "active") {
                if (!val.isBool()) return rc::InvalidPropertyType;
                if (val.asBool()) n.fade.fadeIn(); else n.fade.fadeOut();
            }
            if (key == "channel") {
                if (!val.isNumber()) return rc::InvalidInstructionFormat;   // reference throws bad_variant_access here
                n.channel = static_cast<int>(val.asNumber());
            }
            if (key == "fadeInMs") {
                if (!val.isNumber()) return rc::InvalidPropertyType;
                n.fade.setFadeInMs(sr_, val.asNumber());
            }
            if (key == "fadeOutMs") {
                if (!val.isNumber()) return rc::InvalidPropertyType;
                n.fade.setFadeOutMs(sr_, val.asNumber());
            }
            break;
        case NodeKind::In:          // Math.h:95-105
            if (key == "channel") {
                if (!val.isNumber()) return rc::InvalidPropertyType;
                n.channel = static_cast<int>(val.asNumber());
                g.codeDirty = true;
            }
            break;
        case NodeKind::Svf:         // filters/SVF.h:30-46
            if (key == "mode") {
                if (!val.isString()) return rc::InvalidPropertyType;
                const std::string& m = val.asString();
                if (m == "lowpass") n.mode = 0; if (m == "bandpass") n.mode = 1; if (m == "highpass") n.mode = 2;
                if (m == "notch") n.mode = 3; if (m == "allpass") n.mode = 4;
                g.codeDirty = true;
            }
            break;
        case NodeKind::SvfShelf:    // filters/SVFShelf.h:30-44
            if (key == "mode") {
                if (!val.isString()) return rc::InvalidPropertyType;
                const std::string& m = val.asString();
                if (m == "lowshelf") n.mode = 0; if (m == "highshelf") n.mode = 1; if (m == "bell" || m == "peak") n.mode = 2;
                g.codeDirty = true;
            }
            break;
        case NodeKind::MM1p:        // filters/MultiMode1p.h:50-65
            if (key == "mode") {
                if (!val.isString()) return rc::InvalidPropertyType;
                const std::string& m = val.asString();
                if (m == "lowpass") n.mode = 0; if (m == "highpass") n.mode = 2; if (m == "allpass") n.mode = 4;
                g.codeDirty = true;
            }
            break;
        case NodeKind::Delay:       // Delays.h:59-76
            if (key == "size") {
                if (!val.isNumber()) return rc::InvalidPropertyType;
                n.size = std::max(0, static_cast<int>(val.asNumber()));
                n.ringDirty = true; g.codeDirty = true;
            }
            break;
        case NodeKind::SDelay:      // Delays.h:188-206
            if (key == "size") {
                if (!val.isNumber()) return rc::InvalidPropertyType;
                n.length = std::max(0, static_cast<int>(val.asNumber()));
                n.size = bitceil(n.length + blockSize_);
                n.ringDirty = true; g.codeDirty = true;
            }
            break;
        case NodeKind::MaxHold:     // Core.h:292-303
            if (key == "hold") {
                if (!val.isNumber()) return rc::InvalidPropertyType;
                const double h = sr_ * 0.001 * val.asNumber();
                n.holdSamples = static_cast<uint32_t>(h); g.codeDirty = true;
            }
            break;
        case NodeKind::Rand:        // Noise.h:13-23
            if (key == "seed") {
                if (!val.isNumber()) return rc::InvalidPropertyType;
                int r = fillRowBits(g, n.stateRow, vb, ve, static_cast<uint32_t>(val.asNumber()));
                if (r != rc::Ok) return r;
            }
            break;
        case NodeKind::TapIn:
        case NodeKind::TapOut:      // Feedback.h:24-38,71-85
            if (key == "name") {
                if (!val.isString()) return rc::InvalidPropertyType;
                n.tapName = val.asString(); g.codeDirty = true;
            }
            break;
        case NodeKind::Table:       // Table.h:20-34
        case NodeKind::Convolve:    // wasm/Convolve.h:35-56
            if (key == "path") {
                if (!val.isString()) return rc::InvalidPropertyType;
                auto it = resources_.find(val.asString());
                if (it == resources_.end()) return rc::InvalidPropertyValue;
                n.resource = it->second;
                n.resourceDirty = true; g.codeDirty = true;
            }
            break;

        case NodeKind::Once:        // Core.h:345-361: the prop can arm but never disarm
            if (key == "arm") {
                if (!val.isBool()) return rc::InvalidPropertyType;
                if (val.asBool()) { int r = fillRow(g, n.stateRow, vb, ve, 1.0f); if (r != rc::Ok) return r; }
            }
            break;
        case NodeKind::Seq:         // Core.h:411-466
        case NodeKind::Seq2:        // Seq2.h:39-84
            if (key == "hold") { if (!val.isBool()) return rc::InvalidPropertyType; n.seqHold = val.asBool(); g.codeDirty = true; }
            if (key == "loop") { if (!val.isBool()) return rc::InvalidPropertyType; n.seqLoop = val.asBool(); g.codeDirty = true; }
            if (key == "offset") {
                if (!val.isNumber()) return rc::InvalidPropertyType;
                if (val.asNumber() < 0.0) return rc::InvalidPropertyValue;
                n.seqOffset = static_cast<uint64_t>(val.asNumber()); g.codeDirty = true;
            }
            if (key == "seq") {
                if (!val.isArray()) return rc::InvalidPropertyType;
                std::vector<float> data;
                for (auto& e : val.asArray()) {
                    if (!e.isNumber()) return rc::InvalidInstructionFormat;   // the reference throws bad_variant_access here
                    data.push_back((float) e.asNumber());
                }
                int r = uploadArray(n.seqData, data.data(), data.size() * sizeof(float), data.size());
                if (r != rc::Ok) return r;
                ++n.seqGen; g.codeDirty = true;
            }
            break;
        case NodeKind::SparSeq:     // SparSeq.h:40-124
            if (key == "offset") {
                if (!val.isNumber()) return rc::InvalidPropertyType;
                if (val.asNumber() < 0.0) return rc::InvalidPropertyValue;
                n.seqOffset = static_cast<uint64_t>(val.asNumber()); g.codeDirty = true;
            }
            if (key == "loop") {
                if (val.isNull() || (val.isBool() && !val.asBool())) { n.loopStart = -1; n.loopEnd = -1; }
                else {
                    if (!val.isArray()) return rc::InvalidPropertyType;
                    auto& pts = val.asArray();
                    if (pts.size() < 2 || !pts[0].isNumber() || !pts[1].isNumber()) return rc::InvalidInstructionFormat;
                    n.loopStart = static_cast<int32_t>(pts[0].asNumber()); n.loopEnd = static_cast<int32_t>(pts[1].asNumber());
                }
                ++n.loopGen; g.codeDirty = true;
            }
            if (key == "follow") { if (!val.isBool()) return rc::InvalidPropertyType; n.follow = val.asBool(); g.codeDirty = true; }
            if (key == "interpolate") { if (!val.isNumber()) return rc::InvalidPropertyType; n.interpolate = static_cast<int32_t>(val.asNumber()); g.codeDirty = true; }
            if (key == "tickInterval") {
                if (!val.isNumber()) return rc::InvalidPropertyType;
                if (val.asNumber() < 0.0) return rc::InvalidPropertyValue;
                n.tickIntervalSamples = sr_ * val.asNumber(); g.codeDirty = true;
            }
            if (key == "seq") {   // std::map<int32_t, float>::insert keeps the FIRST value of a duplicated tick time (SparSeq.h:111)
                if (!val.isArray()) return rc::InvalidPropertyType;
                std::map<int32_t, float> m;
                for (auto& e : val.asArray()) {
                    if (!e.isObject()) return rc::InvalidInstructionFormat;
                    auto& o = e.asObject();
                    auto v = o.find("value"), t = o.find("tickTime");
                    if (v == o.end() || t == o.end() || !v->second.isNumber() || !t->second.isNumber()) return rc::InvalidInstructionFormat;
                    m.insert({static_cast<int32_t>(t->second.asNumber()), (float) v->second.asNumber()});
                }
                std::vector<char> blob(m.size() * 8);
                size_t i = 0;
                for (auto& kv : m) { std::memcpy(blob.data() + 4 * i, &kv.first, 4); std::memcpy(blob.data() + 4 * (m.size() + i), &kv.second, 4); ++i; }
                int r = uploadArray(n.seqData, blob.data(), blob.size(), m.size());
                if (r != rc::Ok) return r;
                ++n.seqGen; g.codeDirty = true;
            }
            break;
        case NodeKind::SparSeq2:    // SparSeq2.h:20-56
            if (key == "seq") {
                if (!val.isArray()) return rc::InvalidPropertyType;
                std::map<double, float> m;
                for (auto& e : val.asArray()) {
                    if (!e.isObject()) return rc::InvalidInstructionFormat;
                    auto& o = e.asObject();
                    auto v = o.find("value"), t = o.find("time");
                    if (v == o.end() || t == o.end() || !v->second.isNumber() || !t->second.isNumber()) return rc::InvalidInstructionFormat;
                    m.insert({t->second.asNumber(), (float) v->second.asNumber()});
                }
                std::vector<char> blob(m.size() * 12);
                size_t i = 0;
                for (auto& kv : m) { std::memcpy(blob.data() + 8 * i, &kv.first, 8); std::memcpy(blob.data() + 8 * m.size() + 4 * i, &kv.second, 4); ++i; }
                int r = uploadArray(n.seqData, blob.data(), blob.size(), m.size());
                if (r != rc::Ok) return r;
                ++n.seqGen; g.codeDirty = true;
            }
            if (key == "interpolate") { if (!val.isNumber()) return rc::InvalidPropertyType; n.interpolate = static_cast<int32_t>(val.asNumber()); g.codeDirty = true; }
            break;
        case NodeKind::Scope:       // Analyzers.h:155-179
            if (key == "size") {
                if (!val.isNumber()) return rc::InvalidPropertyType;
                if (val.asNumber() < 256 || val.asNumber() > 8192) return rc::InvalidPropertyValue;
            }
            if (key == "channels") {
                if (!val.isNumber()) return rc::InvalidPropertyType;
                if (val.asNumber() < 0 || val.asNumber() > 4) return rc::InvalidPropertyValue;
            }
            if (key == "name" && !val.isString()) return rc::InvalidPropertyType;
            break;
        case NodeKind::Fft:         // wasm/FFT.h:32-71
            if (key == "size") {
                if (!val.isNumber()) return rc::InvalidPropertyType;
                const int size = static_cast<int>(val.asNumber());
                if (!(size > 0 && (size & (size - 1)) == 0) || size < 256 || size > 8192) return rc::InvalidPropertyValue;
                n.window.resize((size_t) size);
                for (int i = 0; i < size; ++i) {   // Blackman-Harris in the reference's mixed float/double arithmetic (FFT.h:49-62)
                    const float a0 = 0.35875f, a1 = 0.48829f, a2 = 0.14128f, a3 = 0.01168f;
                    const float pi = 3.1415926535897932385f;
                    const float t1 = (float) (a1 * std::cos(2.0 * pi * (i / (double) (size - 1))));
                    const float t2 = (float) (a2 * std::cos(4.0 * pi * (i / (double) (size - 1))));
                    const float t3 = (float) (a3 * std::cos(6.0 * pi * (i / (double) (size - 1))));
                    n.window[(size_t) i] = a0 - t1 + t2 - t3;
                }
            }
            if (key == "name" && !val.isString()) return rc::InvalidPropertyType;
            break;
        case NodeKind::Metro:       // wasm/Metro.h:20-37
            if (key == "interval") {
                if (!val.isNumber()) return rc::InvalidPropertyType;
                if (0 >= val.asNumber()) return rc::InvalidPropertyValue;
                n.intervalSamps = static_cast<int64_t>(std::max(2.0, val.asNumber() * 0.001 * sr_)); g.codeDirty = true;
            }
            break;
        default: break;
    }
    n.props[key] = val;   // GraphNode.h:60-63
    return rc::Ok;
}

int Engine::setProperty(Group& g, const Value& a1, const Value& a2, const Value& v, int vb, int ve) {   // Runtime.h:316-333
    int32_t id;
    if (!toInt32(a1, id) || !a2.isString()) return rc::InvalidInstructionFormat;
    auto it = g.nodes.find(id);
    if (it == g.nodes.end()) return rc::NodeNotFound;
    return nodeSetProperty(g, it->second, a2.asString(), v, vb, ve);
}

int Engine::activateRoots(Group& g, const Value& roots) {   // Runtime.h:369-433
    if (!roots.isArray()) return rc::InvalidInstructionFormat;
    std::set<int32_t> active;
    for (auto& v : roots.asArray()) {
        int32_t id;
        if (!toInt32(v, id)) return rc::InvalidInstructionFormat;
        auto it = g.nodes.find(id);
        if (it == g.nodes.end()) return rc::NodeNotFound;
        if (it->second.kind == NodeKind::Root) {
            nodeSetProperty(g, it->second, "active", Value::boolean(true), 0, g.nv);
            active.insert(id);
        }
    }
    for (int32_t id : g.currentRoots) {
        auto it = g.nodes.find(id);
        if (it == g.nodes.end() || it->second.kind != NodeKind::Root) continue;
        Node& n = it->second;
        if (!active.count(id)) nodeSetProperty(g, n, "active", Value::boolean(false), 0, g.nv);
        if (n.fade.on() || !n.fade.settled()) active.insert(id);   // stillRunning(): Core.h:28-31
    }
    g.currentRoots.swap(active);
    return rc::Ok;
}

int Engine::applyToGroup(Group& g, const std::vector<Value>& batch, int vb, int ve) {   // Runtime.h:170-218
    bool shouldRebuild = false;
    for (auto& next : batch) {
        if (!next.isArray()) return rc::InvalidInstructionFormat;
        auto& ar = next.asArray();
        if (ar.empty() || !ar[0].isNumber()) return rc::InvalidInstructionFormat;
        const int cmd = static_cast<int>(ar[0].asNumber());
        int res = rc::Ok;
        // the reference indexes ar[1..3] unchecked; a short instruction is undefined behaviour there, an
        // InvalidInstructionFormat here.
        auto need = [&](size_t n) { return ar.size() >= n; };
        switch (cmd) {
            case 0: res = need(3) ? createNode(g, ar[1], ar[2]) : rc::InvalidInstructionFormat; break;
            case 3: res = need(4) ? setProperty(g, ar[1], ar[2], ar[3], vb, ve) : rc::InvalidInstructionFormat; break;
            case 2: res = need(4) ? appendChild(g, ar[1], ar[2], ar[3]) : rc::InvalidInstructionFormat; break;
            case 4:
                res = need(2) ? activateRoots(g, ar[1]) : rc::InvalidInstructionFormat;
                shouldRebuild = true;
                break;
            case 5:
                if (shouldRebuild) {
                    std::shared_ptr<Program> p;
                    res = compile(g, g.active ? g.active->nIn : (g.pending ? g.pending->nIn : 0), p);
                    if (res == rc::Ok) {                // rseqQueue.push(buildRenderSequence())
                        if (g.pending) g.superseded.push_back(g.pending);
                        g.pending = p;
                    }
                }
                break;
            default: break;
        }
        if (res != rc::Ok) return res;   // no rollback: Runtime.h:211-214
    }
    return rc::Ok;
}

bool Engine::isValueOnlyBatch(const std::vector<Value>& batch, int vb, int ve) {
    // A batch made only of SET_PROPERTY on per-voice-capable props (const.value, rand.seed, once.arm) never changes the
    // structure of a group, so it may address any sub-range of voices without splitting the group.
    for (auto& ins : batch) {
        if (!ins.isArray()) return false;
        auto& ar = ins.asArray();
        if (ar.size() < 4 || !ar[0].isNumber() || static_cast<int>(ar[0].asNumber()) != 3) return false;
        int32_t id;
        if (!toInt32(ar[1], id) || !ar[2].isString() || !(ar[3].isNumber() || ar[3].isBool())) return false;
        for (auto& g : groups_) {
            if (g->v0 >= ve || g->v0 + g->nv <= vb) continue;
            auto it = g->nodes.find(id);
            if (it == g->nodes.end()) return false;
            const bool ok = (it->second.kind == NodeKind::Const && ar[2].asString() == "value" && ar[3].isNumber()) ||
                            (it->second.kind == NodeKind::Rand && ar[2].asString() == "seed" && ar[3].isNumber()) ||
                            (it->second.kind == NodeKind::Once && ar[2].asString() == "arm" && ar[3].isBool());
            if (!ok) return false;
        }
    }
    return true;
}

int Engine::splitGroupsAt(int v) {
    if (v <= 0 || v >= numVoices_) return rc::Ok;
    for (size_t i = 0; i < groups_.size(); ++i) {
        Group& g = *groups_[i];
        if (v <= g.v0 || v >= g.v0 + g.nv) continue;
        auto ng = std::make_unique<Group>();
        const int cut = v - g.v0;                       // first voice (group-relative) that moves to the new group
        ng->v0 = v; ng->nv = g.nv - cut; ng->Vpad = (ng->nv + 31) / 32 * 32;
        if (g.nodes.empty() && !g.dRows) {              // nothing to migrate
            g.nv = cut; g.Vpad = (g.nv + 31) / 32 * 32;
            groups_.insert(groups_.begin() + i + 1, std::move(ng));
            return rc::Ok;
        }
        // ---- the group is live: the voices [cut, nv) leave with a copy of the graph and THEIR device state -------
        // (dynamic graph updates at voice scale, SURVEY.md §8f N1: afterwards each half can be re-wired independently,
        // every voice keeping its phases, filter memories, delay lines and taps, like a Runtime of its own would.)
        const int L = g.tileWidth;
        if (L > 0 && cut % L != 0)
            return fail(rc::InvariantViolation, "voice groups can only be cut on a voice-tile boundary (multiple of the group's tile width)");
        dsync();
        ng->tileWidth = L;
        ng->currentRoots = g.currentRoots;
        // rows: column slice of every row; a double state is a row PAIR viewed as double[Vpad], sliced as doubles
        ng->rowsCap = g.rowsCap; ng->rowsUsed = g.rowsUsed;
        if (g.dRows && g.rowsCap > 0) {
            if (!cuda(dmalloc((void**) &ng->dRows, sizeof(float) * (size_t) ng->rowsCap * ng->Vpad), "cudaMalloc rows (split)")) return rc::CudaError;
            if (!cuda(dmemset(ng->dRows, 0, sizeof(float) * (size_t) ng->rowsCap * ng->Vpad), "memset rows (split)")) return rc::CudaError;
            std::vector<char> isDoublePair((size_t) g.rowsUsed + 2, 0);
            for (auto& kv : g.nodes) {
                const Node& n = kv.second;
                if (n.kind == NodeKind::Custom) continue;     // registered types keep float state only
                const auto& ti = typeTable().at(n.typeName);
                if (ti.evenAlign && n.stateRow >= 0) for (int k = 0; k < ti.stateRows; k += 2) isDoublePair[(size_t) n.stateRow + k] = 1;
            }
            for (int r = 0; r < g.rowsUsed; ++r) {
                if (isDoublePair[(size_t) r]) {
                    const float* src = g.dRows + (size_t) r * g.Vpad + (size_t) 2 * cut;
                    if (!cuda(dmemcpy(ng->dRows + (size_t) r * ng->Vpad, src, sizeof(double) * ng->nv, cudaMemcpyDeviceToDevice), "copy double row (split)")) return rc::CudaError;
                    ++r;   // the pair's second row is part of the same double array
                } else {
                    if (!cuda(dmemcpy(ng->dRows + (size_t) r * ng->Vpad, g.dRows + (size_t) r * g.Vpad + cut, sizeof(float) * ng->nv, cudaMemcpyDeviceToDevice), "copy row (split)")) return rc::CudaError;
                }
            }
        }
        // tile-structured buffers [tile][pos][L]: the moving voices are a contiguous run of tiles
        const size_t tile0 = L > 0 ? (size_t) cut / L : 0;
        const size_t newTiles = L > 0 ? (size_t) (ng->nv + L - 1) / L : 0;
        auto cloneTiles = [&](const float* src, size_t perTileFloats, float** dst) -> bool {
            *dst = nullptr;
            if (!src || newTiles == 0 || perTileFloats == 0) return true;
            const size_t n = newTiles * perTileFloats;
            if (!cuda(dmalloc((void**) dst, sizeof(float) * n), "cudaMalloc tile buffer (split)")) return false;
            return cuda(dmemcpy(*dst, src + tile0 * perTileFloats, sizeof(float) * n, cudaMemcpyDeviceToDevice), "copy tile buffer (split)");
        };
        for (auto& kv : g.tapShared) {
            float* d = nullptr;
            if (!cloneTiles(kv.second, (size_t) blockSize_ * L, &d)) return rc::CudaError;
            ng->tapShared[kv.first] = d;
        }
        for (auto& kv : g.nodes) {
            Node n = kv.second;   // host-side copy: props, inlets, fades, resource handles, row indices (same layout)
            n.ring = nullptr; n.tapPrivate = nullptr;
            if (!kv.second.relay.empty()) {   // capture relay buffers follow their voices
                n.relay.assign(kv.second.relay.begin() + std::min<size_t>(cut, kv.second.relay.size()), kv.second.relay.end());
                kv.second.relay.resize(std::min<size_t>(cut, kv.second.relay.size()));
            }
            if (kv.second.ring) {
                if (!cloneTiles(kv.second.ring, (size_t) kv.second.size * L, &n.ring)) return rc::CudaError;
                n.ringFloats = newTiles * (size_t) kv.second.size * L;
            }
            if (kv.second.tapPrivate && !cloneTiles(kv.second.tapPrivate, (size_t) blockSize_ * L, &n.tapPrivate)) return rc::CudaError;
            if (kv.second.conv) {
                auto cs = std::make_shared<ConvolverState>();
                std::string err;
                if (!convolver_clone_range(*kv.second.conv, cut, ng->nv, *cs, stream_, err)) return fail(rc::CudaError, err);
                n.conv = cs;
                kv.second.conv->nv = cut;   // the old state keeps its (now partly unused) storage
            }
            ng->nodes.emplace(kv.first, std::move(n));
        }
        const bool hadActive = (bool) g.active, hadPending = (bool) g.pending;
        const int nIn = g.active ? g.active->nIn : (g.pending ? g.pending->nIn : 0);
        g.nv = cut;   // Vpad (the row stride) and the tile buffers of the old group stay as allocated
        Group* ngp = ng.get();
        groups_.insert(groups_.begin() + i + 1, std::move(ng));
        if (hadActive || hadPending) {   // the moved voices keep rendering the same sequence, now through their own program
            std::shared_ptr<Program> p;
            int rcode = compile(*ngp, nIn, p);
            if (rcode != rc::Ok) return rcode;
            if (hadActive && !hadPending) ngp->active = p; else ngp->pending = p;
        }
        return rc::Ok;
    }
    return rc::Ok;
}

int Engine::applyInstructions(int vb, int ve, const char* json, size_t len) {
    Value doc;
    bool parsed = true;
    std::string parseError;
    try {
        doc = parseJson(json, len);           // outside the lock: the render thread never waits for a JSON parse
    } catch (const std::exception& e) {   // the reference throws here (JSON.h:146-154); the C ABI maps it to a code
        parsed = false; parseError = e.what();
    }
    Lock lk(mu_);
    dsetdev();
    if (vb < 0) vb = 0;
    if (ve < 0 || ve > numVoices_) ve = numVoices_;
    if (vb >= ve) return fail(rc::BadArgument, "empty voice range");
    if (!parsed) return fail(rc::InvalidInstructionFormat, parseError);
    lastError_.clear();
    if (!doc.isArray()) return fail(rc::InvalidInstructionFormat, "batch is not an array");
    return applyBatch(vb, ve, doc.asArray());
}

int Engine::applyBatch(int vb, int ve, const std::vector<Value>& batch) {
    steadyValid_ = false;
    if (!isValueOnlyBatch(batch, vb, ve)) {
        int r = splitGroupsAt(vb);
        if (r != rc::Ok) return r;
        if ((r = splitGroupsAt(ve)) != rc::Ok) return r;
    }
    for (auto& g : groups_) {
        const int b = std::max(vb, g->v0), e = std::min(ve, g->v0 + g->nv);
        if (b >= e) continue;
        int r = applyToGroup(*g, batch, b - g->v0, e - g->v0);
        if (r != rc::Ok) { if (lastError_.empty()) lastError_ = "instruction failed"; return r; }
    }
    return rc::Ok;
}

// Binary instruction batch (include/elem_b200.h "binary batch format"): little-endian, unaligned.
namespace {
struct BinReader {
    const unsigned char* p; const unsigned char* end; bool ok = true;
    template <typename T> T get() { T v{}; if ((size_t) (end - p) < sizeof(T)) { ok = false; return v; } std::memcpy(&v, p, sizeof(T)); p += sizeof(T); return v; }
    std::string str(size_t n) { if ((size_t) (end - p) < n) { ok = false; return std::string(); } std::string s(reinterpret_cast<const char*>(p), n); p += n; return s; }
};
}

int Engine::applyBinary(int vb, int ve, const void* data, size_t bytes) {
    BinReader r{static_cast<const unsigned char*>(data), static_cast<const unsigned char*>(data) + bytes};
    if (r.get<uint32_t>() != 0x49324245u /* "EB2I" */ || r.get<uint32_t>() != 1u) { Lock lk(mu_); return fail(rc::InvalidInstructionFormat, "binary batch: bad magic or version"); }
    const uint32_t count = r.get<uint32_t>();
    std::vector<Value> batch;
    batch.reserve(count);
    for (uint32_t i = 0; i < count && r.ok; ++i) {          // decoded outside the lock, like the JSON text
        Value ins = Value::array();
        auto& a = ins.asArray();
        const uint8_t op = r.get<uint8_t>();
        a.push_back(Value::number(op));
        switch (op) {
            case 0: { const int32_t id = r.get<int32_t>(); const uint16_t n = r.get<uint16_t>(); a.push_back(Value::number(id)); a.push_back(Value::string(r.str(n))); } break;
            case 2: { for (int k = 0; k < 3; ++k) a.push_back(Value::number(r.get<int32_t>())); } break;
            case 3: {
                const int32_t id = r.get<int32_t>(); const uint16_t n = r.get<uint16_t>();
                a.push_back(Value::number(id)); a.push_back(Value::string(r.str(n)));
                const uint8_t vt = r.get<uint8_t>();
                switch (vt) {
                    case 0: a.push_back(Value::null()); break;
                    case 1: a.push_back(Value::boolean(r.get<uint8_t>() != 0)); break;
                    case 2: a.push_back(Value::number(r.get<double>())); break;
                    case 3: { const uint32_t len = r.get<uint32_t>(); a.push_back(Value::string(r.str(len))); } break;
                    case 4: { const uint32_t len = r.get<uint32_t>(); Value arr = Value::array(); arr.asArray().reserve(len);
                              for (uint32_t k = 0; k < len && r.ok; ++k) arr.asArray().push_back(Value::number(r.get<float>())); a.push_back(arr); } break;
                    case 5: { const uint32_t len = r.get<uint32_t>(); const std::string js = r.str(len);      // anything else travels as JSON text
                              try { a.push_back(parseJson(js.data(), js.size())); } catch (const std::exception&) { r.ok = false; } } break;
                    default: r.ok = false; break;
                }
            } break;
            case 4: { const uint32_t n = r.get<uint32_t>(); Value roots = Value::array(); for (uint32_t k = 0; k < n && r.ok; ++k) roots.asArray().push_back(Value::number(r.get<int32_t>())); a.push_back(roots); } break;
            case 5: break;
            default: r.ok = false; break;
        }
        batch.push_back(std::move(ins));
    }
    Lock lk(mu_);
    dsetdev();
    if (!r.ok) return fail(rc::InvalidInstructionFormat, "binary batch: truncated or malformed");
    if (vb < 0) vb = 0;
    if (ve < 0 || ve > numVoices_) ve = numVoices_;
    if (vb >= ve) return fail(rc::BadArgument, "empty voice range");
    lastError_.clear();
    return applyBatch(vb, ve, batch);
}

int Engine::setConstTable(const int32_t* nodeIds, int nProps, const float* values, int vb, int count) {
    Lock lk(mu_);
    dsetdev();
    if (vb < 0 || count < 0 || vb + count > numVoices_ || nProps < 0) return fail(rc::BadArgument, "voice range out of bounds");
    for (auto& gp : groups_) {
        Group& g = *gp;
        const int b = std::max(vb, g.v0), e = std::min(vb + count, g.v0 + g.nv);
        if (b >= e) continue;
        for (int p = 0; p < nProps; ++p) {
            auto it = g.nodes.find(nodeIds[p]);
            if (it == g.nodes.end()) return rc::NodeNotFound;
            Node& n = it->second;
            if (n.kind != NodeKind::Const) return fail(rc::InvalidPropertyType, "property table rows must address const nodes");
            const float* src = values + (size_t) p * count + (b - vb);
            if (!cuda(dmemcpy(g.dRows + (size_t) n.paramRow * g.Vpad + (b - g.v0), src, sizeof(float) * (size_t) (e - b), cudaMemcpyHostToDevice), "property table upload")) return rc::CudaError;
            n.props["value"] = Value::number(src[e - b - 1]);
        }
    }
    return rc::Ok;
}

int Engine::setPropertyPerVoice(int32_t nodeId, const char* key, const double* values, int vb, int count) {
    Lock lk(mu_);
    // Vectorised SET_PROPERTY (SURVEY.md §8f N2): values[i] goes to voice vb+i. Same semantics as `count`
    // single-voice [3,id,key,value] batches, without `count` JSON parses.
    dsetdev();
    if (vb < 0 || count < 0 || vb + count > numVoices_) return fail(rc::BadArgument, "voice range out of bounds");
    const std::string k(key);
    for (auto& gp : groups_) {
        Group& g = *gp;
        const int b = std::max(vb, g.v0), e = std::min(vb + count, g.v0 + g.nv);
        if (b >= e) continue;
        auto it = g.nodes.find(nodeId);
        if (it == g.nodes.end()) return rc::NodeNotFound;
        Node& n = it->second;
        int row;
        std::vector<uint32_t> bits((size_t) (e - b));
        if (n.kind == NodeKind::Const && k == "value") {
            row = n.paramRow;
            for (int v = b; v < e; ++v) { float f = (float) values[v - vb]; std::memcpy(&bits[v - b], &f, 4); }
        } else if (n.kind == NodeKind::Rand && k == "seed") {
            row = n.stateRow;
            for (int v = b; v < e; ++v) bits[v - b] = static_cast<uint32_t>(values[v - vb]);
        } else return fail(rc::InvalidPropertyType, "property is not per-voice capable");
        if (!cuda(dmemcpy(g.dRows + (size_t) row * g.Vpad + (b - g.v0), bits.data(), sizeof(uint32_t) * bits.size(), cudaMemcpyHostToDevice), "per-voice prop upload")) return rc::CudaError;   // pageable source: staged before the call returns
        n.props[k] = Value::number(values[e - 1 - vb]);
    }
    return rc::Ok;
}

int Engine::gc(int voice, std::vector<int32_t>& pruned) {
    Lock lk(mu_);   // Runtime.h:221-272
    pruned.clear();
    for (auto& gp : groups_) {
        Group& g = *gp;
        if (voice < g.v0 || voice >= g.v0 + g.nv) continue;
        std::set<int32_t> live;
        if (g.active) live.insert(g.active->nodeIds.begin(), g.active->nodeIds.end());
        if (g.pending) live.insert(g.pending->nodeIds.begin(), g.pending->nodeIds.end());
        for (auto& q : g.superseded) live.insert(q->nodeIds.begin(), q->nodeIds.end());
        dsync();
        for (auto it = g.nodes.begin(); it != g.nodes.end();) {
            if (!live.count(it->first)) {
                pruned.push_back(it->first);
                if (it->second.ring) dfree(it->second.ring);
                if (it->second.tapPrivate) dfree(it->second.tapPrivate);
                it = g.nodes.erase(it);
            } else ++it;
        }
    }
    std::sort(pruned.begin(), pruned.end());
    return rc::Ok;
}

void Engine::reset() {
    Lock lk(mu_);
    // Runtime.h:449-458: only SampleNode does anything on reset() in the reference; no in-scope node does.
}

// ---------------------------------------------------------------------------------------------------------
// compile: sorted node list -> render program
int Engine::chooseTileWidth(int nv) const {
    if (opt_.tileWidth > 0) {
        int L = 1;
        while (L * 2 <= std::min(32, opt_.tileWidth)) L *= 2;
        return L;
    }
    const int target = midRangeDense(nv) ? 4096 : opt_.targetTiles;
    int L = 32;
    while (L > 1 && (nv + L - 1) / L < target) L >>= 1;
    return L;
}

void Engine::traverse(Group& g, std::set<int32_t>& visited, std::vector<int32_t>& order, int32_t n) {   // Runtime.h:503-518
    if (visited.count(n)) return;
    // A cycle would recurse forever in the reference; break it by marking the node before descending when we
    // see it again on the stack (front ends never emit cycles).
    static thread_local std::set<int32_t> onStack;
    if (onStack.count(n)) return;
    onStack.insert(n);
    auto it = g.nodes.find(n);
    if (it != g.nodes.end())
        for (auto& in : it->second.inlets) traverse(g, visited, order, in.source);
    onStack.erase(n);
    order.push_back(n);
    visited.insert(n);
}

struct Compiler {
    Engine& E;
    Group& g;
    int nIn;
    Program& prog;

    struct PendingOp {
        uint32_t opcode = 0, mode = 0, state = NO_STATE, aux0 = 0, aux1 = 0;
        uint64_t ptr = 0;
        int32_t outNode = 0;               // node whose output this op produces (0x7fffffff+k for temporaries)
        std::vector<std::pair<uint32_t, int32_t>> operands;   // (kind, node id | param row)
        struct Step { uint32_t fn; uint32_t kind; int32_t ref; };   // OP_CHAIN: acc = fn(acc, operand) / fn(acc)
        std::vector<Step> steps;
        std::vector<uint32_t> imm;         // raw immediate words behind the operands (control nodes)
        int segment = 0;                   // root sub-sequence the op belongs to
        bool dead = false;                 // absorbed into a later chain
        bool isSeg = false;
        int segRoot = 0;
        size_t segEndOp = 0;
    };
    std::vector<PendingOp> ops;
    std::vector<std::pair<int, int32_t>> promotes;   // (root index, tapOut node id)
    int32_t tempCounter = 0;

    int32_t newTemp() { return INT32_MIN + (++tempCounter); }

    static void putDouble(PendingOp& op, double d) {
        uint64_t b;
        std::memcpy(&b, &d, 8);
        op.aux0 = (uint32_t) b; op.aux1 = (uint32_t) (b >> 32);
    }
    static uint32_t fbits(float f) { uint32_t b; std::memcpy(&b, &f, 4); return b; }

    std::pair<uint32_t, int32_t> operandFor(const Inlet& in) {
        auto it = g.nodes.find(in.source);
        if (it == g.nodes.end() || in.channel != 0) return {K_ZERO, 0};
        const Node& c = it->second;
        if (c.kind == NodeKind::Const || c.kind == NodeKind::Sr) return {K_PARAM, c.paramRow};
        return {K_SLOT, c.id};
    }

    int emitNode(Node& n, int rootIndex);
};

int Compiler::emitNode(Node& n, int rootIndex) {
    if (n.kind == NodeKind::Const || n.kind == NodeKind::Sr) return rc::Ok;   // folded into PARAM operands

    const bool leaf = n.inlets.empty();
    const bool sourceNode = n.kind == NodeKind::Rand || n.kind == NodeKind::TapIn || n.kind == NodeKind::Time || n.kind == NodeKind::Metro;
    if (leaf && !sourceNode) prog.usesHostInputs = true;
    // Inputs as the node's process() sees them: children, or — for a leaf — the host input channels
    // (GraphRenderSequence.h:126-135).
    std::vector<std::pair<uint32_t, int32_t>> inputs;
    if (!leaf) {
        for (auto& in : n.inlets) inputs.push_back(operandFor(in));
    } else if (n.kind != NodeKind::In && !sourceNode) {
        for (int ch = 0; ch < nIn; ++ch) {
            PendingOp ld;
            ld.opcode = OP_LOADIN; ld.aux0 = (uint32_t) ch; ld.outNode = newTemp();
            ops.push_back(ld);
            inputs.push_back({K_SLOT, ld.outNode});
            prog.usesHostInputs = true;
        }
    }
    const int numCh = leaf ? nIn : (int) n.inlets.size();

    bool evNode = n.kind == NodeKind::Metro;
    PendingOp op;
    op.outNode = n.id;
    op.state = (n.stateRow >= 0) ? (uint32_t) n.stateRow : NO_STATE;   // rewritten to a smem index later
    auto zeros = [&]() { op.opcode = OP_FILL0; op.state = NO_STATE; op.operands.clear(); };
    auto take = [&](int k) { op.operands.assign(inputs.begin(), inputs.begin() + k); };

    switch (n.kind) {
        case NodeKind::In: {   // Math.h:107-122
            const int ch = n.channel;
            if (ch < 0 || ch >= numCh) { zeros(); break; }
            if (leaf) { op.opcode = OP_LOADIN; op.aux0 = (uint32_t) ch; prog.usesHostInputs = true; }
            else { op.opcode = OP_COPY; op.operands = {operandFor(n.inlets[ch])}; }
        } break;
        // Math.h:9-89 — element-wise nodes become one-node chains; fuseChains() merges runs of them
        case NodeKind::Unary:
            if (numCh < 1) { zeros(); break; }
            op.opcode = OP_CHAIN; take(1); op.steps.push_back({n.fn, K_ZERO, 0});
            break;
        case NodeKind::Binary:
            if (numCh < 2) { zeros(); break; }
            op.opcode = OP_CHAIN; take(1); op.steps.push_back({n.fn, inputs[1].first, inputs[1].second});
            break;
        case NodeKind::Reduce:   // left fold over the children in order (Math.h:71-84)
            if (numCh < 1) { zeros(); break; }
            op.opcode = OP_CHAIN; take(1);
            for (int j = 1; j < numCh; ++j) op.steps.push_back({n.fn, inputs[j].first, inputs[j].second});
            break;
        case NodeKind::Root:
            op.opcode = OP_ROOT; op.aux0 = (uint32_t) rootIndex;
            if (numCh >= 1) take(1);
            break;
        case NodeKind::Phasor:
            if (numCh < 1) { zeros(); break; }
            op.opcode = OP_PHASOR; op.aux0 = fbits(1.0f / (float) E.sr_); take(1);   // Core.h:90
            break;
        case NodeKind::SPhasor:
            if (numCh < 2) { zeros(); break; }
            op.opcode = OP_SPHASOR; op.aux0 = fbits(1.0f / (float) E.sr_); take(2);
            break;
        case NodeKind::Counter: if (numCh < 1) { zeros(); break; } op.opcode = OP_COUNTER; take(1); break;
        case NodeKind::Accum: if (numCh < 2) { zeros(); break; } op.opcode = OP_ACCUM; take(2); break;
        case NodeKind::Latch: if (numCh < 2) { zeros(); break; } op.opcode = OP_LATCH; take(2); break;
        case NodeKind::MaxHold: if (numCh < 2) { zeros(); break; } op.opcode = OP_MAXHOLD; op.aux0 = n.holdSamples; take(2); break;
        case NodeKind::Rand: op.opcode = OP_RAND; break;
        case NodeKind::Pole: if (numCh < 2) { zeros(); break; } op.opcode = OP_POLE; take(2); break;
        case NodeKind::Env: if (numCh < 3) { zeros(); break; } op.opcode = OP_ENV; take(3); break;
        case NodeKind::Biquad: if (numCh < 6) { zeros(); break; } op.opcode = OP_BIQUAD; take(6); break;
        case NodeKind::Prewarp: if (numCh < 1) { zeros(); break; } op.opcode = OP_PREWARP; putDouble(op, 1.0 / E.sr_); take(1); break;
        case NodeKind::MM1p: if (numCh < 2) { zeros(); break; } op.opcode = OP_MM1P; op.mode = (uint32_t) n.mode; take(2); break;
        case NodeKind::Svf: if (numCh < 3) { zeros(); break; } op.opcode = OP_SVF; op.mode = (uint32_t) n.mode; putDouble(op, E.sr_); take(3); break;
        case NodeKind::SvfShelf: if (numCh < 4) { zeros(); break; } op.opcode = OP_SVFSHELF; op.mode = (uint32_t) n.mode; putDouble(op, E.sr_); take(4); break;
        case NodeKind::Z: if (numCh < 1) { zeros(); break; } op.opcode = OP_Z; take(1); break;
        case NodeKind::Blep:
            if (numCh < 1) { zeros(); break; }
            op.opcode = OP_BLEP; op.mode = n.fn; op.aux0 = fbits((float) E.sr_); take(1);
            break;
        case NodeKind::PassThrough: if (numCh < 1) { zeros(); break; } op.opcode = OP_COPY; take(1); break;
        case NodeKind::Custom: {   // a registered device node type: missing inputs give zeros like every builtin
            const auto& ct = E.customTypes_[n.fn];
            if (numCh < ct.nIn) { zeros(); break; }
            op.opcode = OP_CUSTOM; op.aux0 = n.fn; op.aux1 = (uint32_t) ct.nState; take(ct.nIn);
            op.imm = {fbits((float) E.sr_)};
            prog.hasCustom = true;
        } break;


        // ---- sequencing / control nodes (SURVEY.md §8f N3) ----
        case NodeKind::Once: if (numCh < 1) { zeros(); break; } op.opcode = OP_ONCE; take(1); break;
        case NodeKind::Seq:
        case NodeKind::Seq2: {   // Core.h:497-500, Seq2.h:100-103: zeros without a trigger input or a sequence
            if (numCh < 1 || !n.seqData || n.seqData->count == 0) { zeros(); break; }
            op.opcode = n.kind == NodeKind::Seq ? OP_SEQ : OP_SEQ2;
            take(std::min(numCh, 2));
            op.mode = (n.seqHold ? 1u : 0u) | (n.seqLoop ? 2u : 0u) | (numCh > 1 ? 4u : 0u);
            op.aux0 = (uint32_t) n.seqData->count; op.ptr = (uint64_t) (uintptr_t) n.seqData->d;
            op.imm = {(uint32_t) std::min<uint64_t>(n.seqOffset, 0xFFFFFFFFu), n.seqGen};
            prog.pinned.push_back(n.seqData);
        } break;
        case NodeKind::SparSeq: {   // SparSeq.h:259-262: zeros without a trigger input; the loop-point logic still runs without a sequence
            if (numCh < 1) { zeros(); break; }
            op.opcode = OP_SPARSEQ;
            take(std::min(numCh, 2));
            op.mode = (numCh > 1 ? 4u : 0u);
            if (n.seqData) { op.aux0 = (uint32_t) n.seqData->count; op.ptr = (uint64_t) (uintptr_t) n.seqData->d; prog.pinned.push_back(n.seqData); }
            uint64_t tb; std::memcpy(&tb, &n.tickIntervalSamples, 8);
            op.imm = {(uint32_t) n.seqOffset, n.follow ? 1u : 0u, (uint32_t) n.interpolate, n.seqGen, n.loopGen,
                      (uint32_t) n.loopStart, (uint32_t) n.loopEnd, (uint32_t) tb, (uint32_t) (tb >> 32)};
        } break;
        case NodeKind::SparSeq2: {  // SparSeq2.h:90-91
            if (numCh < 1 || !n.seqData || n.seqData->count == 0) { zeros(); break; }
            op.opcode = OP_SPARSEQ2; take(1);
            op.mode = (n.interpolate == 1) ? 1u : 0u;
            op.aux0 = (uint32_t) n.seqData->count; op.ptr = (uint64_t) (uintptr_t) n.seqData->d;
            op.imm = {n.seqGen};
            prog.pinned.push_back(n.seqData);
        } break;
        case NodeKind::Time: op.opcode = OP_TIME; break;                                     // wasm/SampleTime.h:16-23
        case NodeKind::Metro: op.opcode = OP_METRO; putDouble(op, (double) n.intervalSamps); break;   // wasm/Metro.h:39-55


        // ---- analysis nodes (SURVEY.md §8f N4) ----
        case NodeKind::Meter: if (numCh < 1) { zeros(); break; } op.opcode = OP_METER; take(1); evNode = true; break;
        case NodeKind::Snapshot: if (numCh < 2) { zeros(); break; } op.opcode = OP_SNAPSHOT; take(2); evNode = true; break;
        case NodeKind::Scope:
        case NodeKind::Fft:
        case NodeKind::Capture: {
            evNode = true;
            const size_t floats = (size_t) g.nTiles() * g.tileWidth * (size_t) n.size;
            if (!n.ring) {
                if (!E.cuda(E.dmalloc((void**) &n.ring, sizeof(float) * floats), "cudaMalloc analysis ring")) return rc::CudaError;
                if (!E.cuda(E.dmemset(n.ring, 0, sizeof(float) * floats), "memset analysis ring")) return rc::CudaError;
                n.ringFloats = floats;
            }
            if (n.kind == NodeKind::Scope || n.kind == NodeKind::Fft) {
                if (numCh < 1) { zeros(); break; }
                const int ringCh = n.kind == NodeKind::Scope ? (int) SCOPE_CHANNELS : 1;
                op.opcode = OP_SCOPE; take(std::min(numCh, ringCh)); op.aux1 = (uint32_t) ringCh;
                if (prog.dynNodes.size() >= (size_t) MAX_DYN) return E.fail(rc::InvariantViolation, "more than 16 scope nodes in one graph");
                op.aux0 = (uint32_t) prog.dynNodes.size();
                prog.dynNodes.push_back(n.id);
            } else {
                if (numCh < 2) { zeros(); break; }
                op.opcode = OP_CAPTURE; take(2);
                op.aux0 = (uint32_t) (n.size - CAPTURE_SCRATCH);
            }
            op.ptr = (uint64_t) (uintptr_t) n.ring;
        } break;

        case NodeKind::Delay: {   // Delays.h:92-106
            const size_t tiles = (size_t) g.nTiles() * g.tileWidth;
            if (n.ringDirty) {
                E.dsync();
                if (n.ring) { E.dfree(n.ring); n.ring = nullptr; }
                n.ringFloats = (size_t) n.size * tiles;
                if (n.ringFloats) {
                    if (!E.cuda(E.dmalloc((void**) &n.ring, sizeof(float) * n.ringFloats), "cudaMalloc delay ring")) return rc::CudaError;
                    if (!E.cuda(E.dmemset(n.ring, 0, sizeof(float) * n.ringFloats), "memset ring")) return rc::CudaError;
                }
                int r = E.fillRowBits(g, n.stateRow, 0, g.nv, 0);   // writeIndex = 0
                if (r != rc::Ok) return r;
                n.ringDirty = false;
            }
            if (numCh < 3) { zeros(); break; }
            op.opcode = OP_DELAY; op.aux0 = (uint32_t) n.size; op.ptr = (uint64_t) (uintptr_t) n.ring; take(3);
        } break;

        case NodeKind::SDelay: {  // Delays.h:221-245
            const size_t tiles = (size_t) g.nTiles() * g.tileWidth;
            if (n.ringDirty) {
                E.dsync();
                if (n.ring) { E.dfree(n.ring); n.ring = nullptr; }
                n.ringFloats = (size_t) n.size * tiles;
                if (n.ringFloats) {
                    if (!E.cuda(E.dmalloc((void**) &n.ring, sizeof(float) * n.ringFloats), "cudaMalloc sdelay ring")) return rc::CudaError;
                    if (!E.cuda(E.dmemset(n.ring, 0, sizeof(float) * n.ringFloats), "memset ring")) return rc::CudaError;
                }
                int r = E.fillRowBits(g, n.stateRow, 0, g.nv, 0);
                if (r != rc::Ok) return r;
                n.ringDirty = false;
            }
            if (numCh < 1 || n.size == 0) { zeros(); break; }
            op.opcode = OP_SDELAY; op.aux0 = (uint32_t) n.size; op.aux1 = (uint32_t) n.length; op.ptr = (uint64_t) (uintptr_t) n.ring; take(1);
        } break;

        case NodeKind::Table: {   // Table.h:44-57
            if (numCh == 0 || !n.resource || n.resource->numSamples == 0) { zeros(); break; }
            int r = E.ensureResourceOnDevice(*n.resource);
            if (r != rc::Ok) return r;
            op.opcode = OP_TABLE; op.aux0 = (uint32_t) n.resource->numSamples; op.ptr = (uint64_t) (uintptr_t) n.resource->dChannel0; take(1);
            if (!prog.stagedTable && n.resource->numSamples <= (size_t) TABLE_SMEM_MAX_FLOATS) {
                prog.stagedTable = n.resource->dChannel0;
                prog.stagedTableFloats = (int) ((n.resource->numSamples + 3) / 4 * 4);
            }
        } break;

        case NodeKind::TapIn:
        case NodeKind::TapOut: {
            const size_t floats = (size_t) g.nTiles() * g.tileWidth * E.blockSize_;
            float* shared = nullptr;
            if (!n.tapName.empty()) {   // Feedback.h:29-33: created on first request by either side
                auto it = g.tapShared.find(n.tapName);
                if (it == g.tapShared.end()) {
                    if (!E.cuda(E.dmalloc((void**) &shared, sizeof(float) * floats), "cudaMalloc tap")) return rc::CudaError;
                    if (!E.cuda(E.dmemset(shared, 0, sizeof(float) * floats), "memset tap")) return rc::CudaError;
                    g.tapShared[n.tapName] = shared;
                } else shared = it->second;
            }
            if (n.kind == NodeKind::TapIn) {
                if (!shared) { zeros(); break; }
                op.opcode = OP_TAPIN; op.ptr = (uint64_t) (uintptr_t) shared;
            } else {
                if (!n.tapPrivate) {
                    if (!E.cuda(E.dmalloc((void**) &n.tapPrivate, sizeof(float) * floats), "cudaMalloc tapOut")) return rc::CudaError;
                    if (!E.cuda(E.dmemset(n.tapPrivate, 0, sizeof(float) * floats), "memset tapOut")) return rc::CudaError;
                }
                if (shared) promotes.push_back({rootIndex, n.id});
                if (numCh < 1) { zeros(); break; }
                op.opcode = OP_TAPOUT; op.ptr = (uint64_t) (uintptr_t) n.tapPrivate; take(1);
            }
        } break;

        case NodeKind::Convolve: {   // wasm/Convolve.h:58-85: zeros without an input or a loaded IR
            if (numCh == 0 || !n.resource) { zeros(); break; }
            if (n.resourceDirty || !n.conv) {   // a new `path` makes a fresh convolver (Convolve.h:45-51)
                auto cs = std::make_shared<ConvolverState>();
                const auto& ch0 = n.resource->channels.empty() ? std::vector<float>() : n.resource->channels[0];
                std::string err;
                if (!convolver_init(*cs, ch0.data(), ch0.size(), g.nv, E.planOnly_, E.stream_, err)) return E.fail(rc::CudaError, err);
                n.conv = cs;
                n.resourceDirty = false;
            }
            op.opcode = 0xF0; take(1);   // OP_HOST_CONV: lowered to STOREBUF + K3 + LOADBUF by the stage pass
        } break;

        default: zeros(); break;
    }
    if (evNode) prog.evNodes.push_back({n.id, rootIndex});
    ops.push_back(std::move(op));
    return rc::Ok;
}

int Engine::compile(Group& g, int nIn, std::shared_ptr<Program>& out) {
    auto prog = std::make_shared<Program>();
    prog->planOnly = planOnly_;
    prog->nIn = nIn;
    g.codeDirty = false;
    if (g.tileWidth == 0) g.tileWidth = chooseTileWidth(g.nv);

    // Root order: Runtime.h:544-559 — iterate currentRoots ascending; active roots are pushed to the FRONT,
    // inactive (fading out) ones to the back.
    std::list<int32_t> sortedRoots;
    for (int32_t id : g.currentRoots) {
        auto it = g.nodes.find(id);
        if (it == g.nodes.end() || it->second.kind != NodeKind::Root) continue;
        auto ap = it->second.props.find("active");
        const bool isActive = ap != it->second.props.end() && ap->second.isBool() && ap->second.asBool();
        if (isActive) sortedRoots.push_front(id); else sortedRoots.push_back(id);
    }
    if (sortedRoots.size() > (size_t) MAX_ROOTS) return fail(rc::InvariantViolation, "more than 16 simultaneous roots");

    Compiler C{*this, g, nIn, *prog};
    std::set<int32_t> visited;
    for (int32_t rid : sortedRoots) {
        const int r = (int) prog->rootIds.size();
        prog->rootIds.push_back(rid);
        std::vector<int32_t> order;
        traverse(g, visited, order, rid);
        Compiler::PendingOp seg;
        seg.isSeg = true; seg.opcode = OP_SEG; seg.segRoot = r; seg.segment = r;
        const size_t segIdx = C.ops.size();
        C.ops.push_back(seg);
        for (int32_t nid : order) {
            auto it = g.nodes.find(nid);
            if (it == g.nodes.end()) continue;
            prog->nodeIds.push_back(nid);
            const size_t before = C.ops.size();
            int rcode = C.emitNode(it->second, r);
            if (rcode != rc::Ok) return rcode;
            for (size_t k = before; k < C.ops.size(); ++k) C.ops[k].segment = r;
        }
        C.ops[segIdx].segEndOp = C.ops.size();
    }
    auto& ops = C.ops;
    using Step = Compiler::PendingOp::Step;

    auto forEachSlotUse = [](const Compiler::PendingOp& op, const std::function<void(int32_t)>& f) {
        for (auto& o : op.operands) if (o.first == K_SLOT) f(o.second);
        for (auto& st : op.steps) if (!chain_fn_is_unary(st.fn) && st.kind == K_SLOT) f(st.ref);
    };

    // ---- chain fusion -------------------------------------------------------------------------------------
    // An element-wise node whose output has exactly one use, by a later element-wise node of the same root
    // sub-sequence, is folded into its consumer: as the head of the consumer's chain when it is the first
    // operand, or — for the other operands of a fold — by ending the producer's chain with the reversed step
    // fn(running value, acc).  Every node is still evaluated exactly once, with the same operand values in the
    // same left-fold order (Math.h:71-84), so results are bit-identical; only the evaluation ORDER of
    // independent stateless nodes changes, and the intermediates stay in registers.
    if (opt_.fuseChains) {
        std::unordered_map<int32_t, int> uses;
        for (auto& op : ops) if (!op.isSeg) forEachSlotUse(op, [&](int32_t id) { ++uses[id]; });
        std::unordered_map<int32_t, size_t> producer;   // value id -> index of the (still open) chain producing it
        std::vector<Compiler::PendingOp> outOps;
        std::vector<size_t> segHeaderAt(prog->rootIds.size(), 0);
        int32_t& tempCounter = C.tempCounter;
        for (size_t i = 0; i < ops.size(); ++i) {
            Compiler::PendingOp op = ops[i];
            if (op.isSeg) { segHeaderAt[op.segRoot] = outOps.size(); outOps.push_back(op); continue; }
            if (op.opcode != OP_CHAIN) { outOps.push_back(op); continue; }
            auto absorbable = [&](uint32_t kind, int32_t ref) -> long {
                if (kind != K_SLOT) return -1;
                auto u = uses.find(ref);
                if (u == uses.end() || u->second != 1) return -1;
                auto p = producer.find(ref);
                if (p == producer.end()) return -1;
                const auto& pop = outOps[p->second];
                if (pop.dead || pop.opcode != OP_CHAIN || pop.segment != op.segment) return -1;
                return (long) p->second;
            };
            // head: the first operand's producer continues into this chain
            Compiler::PendingOp cur = op;
            cur.steps.clear();
            {
                long pi = absorbable(op.operands[0].first, op.operands[0].second);
                if (pi >= 0) {
                    cur.operands = outOps[pi].operands;
                    cur.steps = outOps[pi].steps;
                    outOps[pi].dead = true;
                }
            }
            for (const Step& st : op.steps) {
                long pi = chain_fn_is_unary(st.fn) ? -1 : absorbable(st.kind, st.ref);
                if (pi < 0 || cur.steps.size() + outOps[pi].steps.size() > 200) { cur.steps.push_back(st); continue; }
                // flush the running value to a temporary, then restart from the absorbed producer and finish
                // with the reversed step: value = fn(running, producer)
                uint32_t runKind = cur.operands[0].first;
                int32_t runRef = cur.operands[0].second;
                if (!cur.steps.empty()) {
                    Compiler::PendingOp flushed = cur;
                    flushed.outNode = INT32_MIN + (++tempCounter);
                    flushed.state = NO_STATE;
                    outOps.push_back(flushed);
                    runKind = K_SLOT; runRef = flushed.outNode;
                }
                cur.operands = outOps[pi].operands;
                cur.steps = outOps[pi].steps;
                outOps[pi].dead = true;
                cur.steps.push_back({st.fn | CHAIN_REVERSED, runKind, runRef});
            }
            if (cur.steps.size() > 120) {   // keep every op's operand block within 255 words
                // split: flush the first 100 steps into a temporary and continue from it
                while (cur.steps.size() > 120) {
                    Compiler::PendingOp head = cur;
                    head.steps.assign(cur.steps.begin(), cur.steps.begin() + 100);
                    head.outNode = INT32_MIN + (++tempCounter);
                    outOps.push_back(head);
                    cur.operands = {{K_SLOT, head.outNode}};
                    cur.steps.erase(cur.steps.begin(), cur.steps.begin() + 100);
                }
            }
            producer[cur.outNode] = outOps.size();
            outOps.push_back(cur);
        }
        // drop absorbed ops, fix segment ends
        std::vector<Compiler::PendingOp> compact;
        std::vector<size_t> segStart(prog->rootIds.size(), 0);
        for (auto& op : outOps) {
            if (op.dead) continue;
            if (op.isSeg) segStart[op.segRoot] = compact.size();
            compact.push_back(op);
        }
        for (size_t r = 0; r < segStart.size(); ++r) {
            size_t end = compact.size();
            for (size_t k = segStart[r] + 1; k < compact.size(); ++k) if (compact[k].isSeg) { end = k; break; }
            compact[segStart[r]].segEndOp = end;
        }
        ops.swap(compact);

        // ---- re-schedule each root sub-sequence to shorten live ranges -----------------------------------------
        // Depth-first from the sinks of the segment, visiting the operand with the larger sub-tree first
        // (Sethi-Ullman order).  Any topological order gives the same results — every op is a function of its
        // operand values and its own private state only — but this one keeps a 64-partial additive voice at 3
        // live slots instead of 65.
        std::vector<Compiler::PendingOp> sched;
        size_t i0 = 0;
        while (i0 < ops.size()) {
            const size_t segBegin = i0;                       // ops[segBegin] is the OP_SEG header
            const size_t segEnd = ops[segBegin].segEndOp;
            std::unordered_map<int32_t, size_t> prodIdx;      // value id -> op index inside this segment
            for (size_t k = segBegin + 1; k < segEnd; ++k) prodIdx[ops[k].outNode] = k;
            std::vector<std::vector<size_t>> deps(segEnd - segBegin);
            std::vector<int> consumers(segEnd - segBegin, 0);
            for (size_t k = segBegin + 1; k < segEnd; ++k)
                forEachSlotUse(ops[k], [&](int32_t id) {
                    auto p = prodIdx.find(id);
                    if (p != prodIdx.end() && p->second != k) { deps[k - segBegin].push_back(p->second); ++consumers[p->second - segBegin]; }
                });
            std::vector<long> weight(segEnd - segBegin, -1);
            std::function<long(size_t)> subtree = [&](size_t k) -> long {
                long& w = weight[k - segBegin];
                if (w >= 0) return w;
                w = 1;
                for (size_t d : deps[k - segBegin]) w += subtree(d);
                return w;
            };
            std::vector<char> done(segEnd - segBegin, 0);
            const size_t headerAt = sched.size();
            sched.push_back(ops[segBegin]);
            std::function<void(size_t)> emit = [&](size_t k) {
                if (done[k - segBegin]) return;
                done[k - segBegin] = 1;
                std::vector<size_t> ds = deps[k - segBegin];
                std::stable_sort(ds.begin(), ds.end(), [&](size_t a, size_t b) { return subtree(a) > subtree(b); });
                for (size_t d : ds) emit(d);
                sched.push_back(ops[k]);
            };
            for (size_t k = segBegin + 1; k < segEnd; ++k) if (consumers[k - segBegin] == 0) emit(k);
            for (size_t k = segBegin + 1; k < segEnd; ++k) emit(k);   // anything unreachable (cannot happen) keeps its place
            sched[headerAt].segEndOp = sched.size();
            i0 = segEnd;
        }
        ops.swap(sched);

        // ---- group independent constant-frequency phasors into runs ----------------------------------------------
        // A phasor fed by a parameter depends on nothing, so it may run anywhere in its segment.  With L < 32 voices
        // per warp only L lanes work in a recurrence; a run of R <= 32/L such phasors is executed by R lane groups
        // in one serial loop (render_kernel.cu, OP_PHASOR with aux1 = R).  Followers are pulled forward to sit
        // right behind the leader; the look-ahead is bounded so live ranges stay short.
        bool staged = false;   // programs cut into stages (convolve) insert spill ops between ops: keep them ungrouped
        for (auto& op : ops) if (op.opcode == 0xF0) staged = true;
        const int maxRun = staged ? 1 : std::min(8, 32 / std::max(1, g.tileWidth));
        auto isParamPhasor = [](const Compiler::PendingOp& op) {
            return !op.isSeg && op.opcode == OP_PHASOR && op.operands.size() == 1 && op.operands[0].first != K_SLOT;
        };
        for (size_t i = 0; i < ops.size(); ++i) {
            if (!isParamPhasor(ops[i]) || ops[i].aux1 != 0 || ops[i].mode == 1) continue;
            size_t segEnd = ops.size();
            for (size_t k = i + 1; k < ops.size(); ++k) if (ops[k].isSeg) { segEnd = k; break; }
            uint32_t run = 1;
            for (size_t j = i + 1; j < segEnd && j < i + 1 + (size_t) 4 * maxRun && (int) run < maxRun; ++j) {
                if (!isParamPhasor(ops[j]) || ops[j].mode == 1) continue;
                Compiler::PendingOp follower = ops[j];
                follower.mode = 1;                     // marks "member of a run" (never dispatched on its own)
                ops.erase(ops.begin() + (long) j);
                ops.insert(ops.begin() + (long) (i + run), follower);
                ++run;
            }
            ops[i].aux1 = run;                         // run length, 1 = a lone constant-frequency phasor
        }
    }

    // ---- stages: a `convolve` node is a whole-block operation (K3) that cannot live inside the sample-tiled
    // interpreter, so the program is cut into K1 stages around it.  Values that cross a stage boundary travel
    // through per-voice block buffers in HBM (OP_STOREBUF / OP_LOADBUF); root ops always run in the last stage.
    constexpr uint32_t OP_HOST_CONV = 0xF0;   // host-only pseudo opcode emitted for Convolve nodes
    std::vector<std::vector<Compiler::PendingOp>> stageOps;
    bool hasConv = false;
    for (auto& op : ops) if (op.opcode == OP_HOST_CONV) hasConv = true;
    if (!hasConv) {
        stageOps.push_back(ops);
    } else {
        std::unordered_map<int32_t, int> stageOfValue;       // stage in which the value becomes available to K1
        std::unordered_map<int32_t, const Compiler::PendingOp*> producerOp;
        int lastStage = 0;
        std::vector<int> stageOfOp(ops.size(), 0);
        for (size_t i = 0; i < ops.size(); ++i) {
            auto& op = ops[i];
            if (op.isSeg) continue;
            int st = 0;
            forEachSlotUse(op, [&](int32_t id) { auto it = stageOfValue.find(id); if (it != stageOfValue.end()) st = std::max(st, it->second); });
            stageOfOp[i] = st;
            stageOfValue[op.outNode] = (op.opcode == OP_HOST_CONV) ? st + 1 : st;
            lastStage = std::max(lastStage, stageOfValue[op.outNode]);
        }
        for (size_t i = 0; i < ops.size(); ++i) if (!ops[i].isSeg && ops[i].opcode == OP_ROOT) stageOfOp[i] = lastStage;
        const int nStages = lastStage + 1;
        const size_t blockFloats = (size_t) g.Vpad * blockSize_;
        auto newBlockBuffer = [&]() -> float* {
            float* p = nullptr;
            if (!cuda(dmalloc((void**) &p, sizeof(float) * blockFloats), "cudaMalloc stage buffer")) return nullptr;
            dmemset(p, 0, sizeof(float) * blockFloats);
            prog->blockBuffers.push_back(p);
            return p;
        };
        // buffers: one per convolve node (in, out) and one per ordinary value that crosses stages
        std::unordered_map<int32_t, float*> spillOf;         // value id -> HBM block buffer holding it
        prog->stages.resize(nStages);
        for (size_t i = 0; i < ops.size(); ++i) {
            auto& op = ops[i];
            if (op.isSeg || op.opcode != OP_HOST_CONV) continue;
            Node& n = g.nodes.at(op.outNode);
            // A convolver fed straight by a host input channel (`convolve(in)`) reads that channel where it lies: no K1 staging
            // copy, and — when nothing else lives in the stage — no K1 launch at all for it.
            int inChannel = -1;
            if (op.operands.size() == 1 && op.operands[0].first == K_SLOT) {
                for (size_t j = 0; j < i; ++j)
                    if (!ops[j].isSeg && ops[j].outNode == op.operands[0].second && ops[j].opcode == OP_LOADIN) inChannel = (int) ops[j].aux0;
            }
            float* inB = inChannel >= 0 ? nullptr : newBlockBuffer();
            float* outB = newBlockBuffer();
            if ((inChannel < 0 && !inB) || !outB) return rc::CudaError;
            prog->stages[stageOfOp[i]].convolves.push_back({n.id, inB, outB, inChannel});
            spillOf[op.outNode] = outB;
            op.ptr = (uint64_t) (uintptr_t) inB;
            if (inChannel >= 0) op.mode = 1;      // marks "no STOREBUF needed"
        }
        // LOADINs whose only consumers are bypassed convolvers are dead
        {
            std::unordered_map<int32_t, int> otherUses;
            for (auto& op : ops) {
                if (op.isSeg || (op.opcode == OP_HOST_CONV && op.mode == 1)) continue;
                forEachSlotUse(op, [&](int32_t id) { ++otherUses[id]; });
            }
            for (auto& op : ops)
                if (!op.isSeg && op.opcode == OP_LOADIN && !otherUses.count(op.outNode)) {
                    bool feedsBypass = false;
                    for (auto& c : ops) if (!c.isSeg && c.opcode == OP_HOST_CONV && c.mode == 1 && c.operands[0].second == op.outNode) feedsBypass = true;
                    if (feedsBypass) op.dead = true;
                }
        }
        // which values are read in a later stage than the one that produces them?
        std::unordered_map<int32_t, int> producedIn;
        for (size_t i = 0; i < ops.size(); ++i) if (!ops[i].isSeg) producedIn[ops[i].outNode] = (ops[i].opcode == OP_HOST_CONV) ? -1 : stageOfOp[i];
        for (size_t i = 0; i < ops.size(); ++i) {
            if (ops[i].isSeg) continue;
            forEachSlotUse(ops[i], [&](int32_t id) {
                auto p = producedIn.find(id);
                if (p == producedIn.end() || p->second < 0) return;
                if (p->second < stageOfOp[i] && !spillOf.count(id)) spillOf[id] = nullptr;   // allocate below
            });
        }
        for (auto& kv : spillOf) if (!kv.second) { kv.second = newBlockBuffer(); if (!kv.second) return rc::CudaError; }

        stageOps.assign(nStages, {});
        for (int st = 0; st < nStages; ++st) {
            auto& out = stageOps[st];
            size_t i = 0;
            while (i < ops.size()) {
                const size_t segBegin = i, segEnd = ops[i].segEndOp;
                const size_t headerAt = out.size();
                out.push_back(ops[segBegin]);
                std::unordered_map<int32_t, int32_t> loaded;   // value id -> temp id loaded in this stage+segment
                for (size_t k = segBegin + 1; k < segEnd; ++k) {
                    if (stageOfOp[k] != st || ops[k].dead) continue;
                    Compiler::PendingOp op = ops[k];
                    // reload operands that were produced in an earlier stage (or by a convolver)
                    auto fix = [&](uint32_t& kind, int32_t& ref) {
                        if (kind != K_SLOT) return;
                        auto p = producedIn.find(ref);
                        if (p == producedIn.end()) return;
                        if (p->second >= 0 && p->second >= st) return;
                        auto l = loaded.find(ref);
                        if (l == loaded.end()) {
                            Compiler::PendingOp ld;
                            ld.opcode = OP_LOADBUF; ld.segment = op.segment; ld.outNode = INT32_MIN + (++C.tempCounter);
                            ld.ptr = (uint64_t) (uintptr_t) spillOf.at(ref);
                            out.push_back(ld);
                            l = loaded.emplace(ref, ld.outNode).first;
                        }
                        ref = l->second;
                    };
                    for (auto& o : op.operands) fix(o.first, o.second);
                    for (auto& stp : op.steps) if (!chain_fn_is_unary(stp.fn)) fix(stp.kind, stp.ref);
                    if (op.opcode == OP_HOST_CONV && op.mode == 1) continue;   // reads the host input channel directly
                    if (op.opcode == OP_HOST_CONV) {          // stage the convolver input
                        op.opcode = OP_STOREBUF; op.state = NO_STATE; op.outNode = INT32_MIN + (++C.tempCounter);
                        out.push_back(op);
                        continue;
                    }
                    out.push_back(op);
                    auto sp = spillOf.find(op.outNode);
                    if (sp != spillOf.end()) {                // the value is needed by a later stage
                        Compiler::PendingOp stb;
                        stb.opcode = OP_STOREBUF; stb.segment = op.segment; stb.outNode = INT32_MIN + (++C.tempCounter);
                        stb.operands = {{K_SLOT, op.outNode}};
                        stb.ptr = (uint64_t) (uintptr_t) sp->second;
                        out.push_back(stb);
                    }
                }
                out[headerAt].segEndOp = out.size();
                i = segEnd;
            }
            bool anyWork = false;
            for (auto& op : out) if (!op.isSeg) anyWork = true;
            prog->stages[st].empty = !anyWork;
        }
        // `convolve -> root` (a reverb send, BASELINE config 4): the last stage is [LOADBUF conv.out][ROOT of it] and nothing else
        if (opt_.fuseConvRoot && g.tileWidth == 1 && nStages >= 2 && prog->rootIds.size() == 1 && C.promotes.empty()) {
            const auto& lastOps = stageOps[nStages - 1];
            std::vector<const Compiler::PendingOp*> body;
            for (auto& op : lastOps) if (!op.isSeg) body.push_back(&op);
            if (body.size() == 2 && body[0]->opcode == OP_LOADBUF && body[1]->opcode == OP_ROOT && body[1]->operands.size() == 1 &&
                body[1]->operands[0].first == K_SLOT && body[1]->operands[0].second == body[0]->outNode) {
                for (int st = 0; st < nStages - 1 && prog->fusedConvStage < 0; ++st)
                    for (size_t ci = 0; ci < prog->stages[st].convolves.size(); ++ci)
                        if ((uint64_t) (uintptr_t) prog->stages[st].convolves[ci].out == body[0]->ptr) {
                            prog->fusedConvStage = st; prog->fusedConvIndex = (int) ci; prog->fusedRoot = (int) body[1]->aux0;
                            break;
                        }
            }
        }
    }

    // ---- warp pipeline for one-voice groups (BASELINE config 5: thousands of different graphs, one voice each) ----------------
    // With one voice per warp every recurrence owns a single lane and the warp is latency bound.  The op list (one root sub-sequence,
    // already in its final order) is cut into W contiguous stages of about equal cost; render_groups_pipe_kernel gives each stage its
    // own warp, and the warps work on consecutive sample tiles of the same graph at the same time.  A value that crosses a cut lives in
    // a ring slot with W buffers (tile index mod W), everything else in slots private to its stage.  Same ops, same order of evaluation
    // per value: bit-identical output (tests/test_parity_gpu.py::test_pipelined_groups_equal_the_unpipelined_path).
    std::vector<int> pipeStageOf;            // per op of stageOps[0]; empty = not pipelined
    {
        const bool batchedGroup = groups_.size() > 1 && opt_.batchGroups;
        int W = std::min(opt_.pipelineStages, (int) MAX_PIPE);
        bool ok = W > 1 && batchedGroup && g.tileWidth == 1 && stageOps.size() == 1 && prog->rootIds.size() == 1 && C.promotes.empty() &&
                  prog->evNodes.empty() && prog->dynNodes.empty() && !prog->hasCustom;
        auto& sops = stageOps[0];
        auto costOf = [](const Compiler::PendingOp& op) -> long {     // cycles of one 32-sample tile at L = 1, dispatch included: measured per
            switch (op.opcode) {                                          // opcode with the cycle-counter build (profiles/r02_k_opprof_config5.txt)
                case OP_CHAIN: {
                    long c = 350;
                    for (auto& st : op.steps) {
                        const uint32_t fn = st.fn & 0xFF;
                        if (fn <= F_EXP && fn != F_CEIL && fn != F_FLOOR && fn != F_ROUND && fn != F_SQRT && fn != F_ABS) c += 450;
                        else if (fn == F_DIV || fn == F_MOD || fn == F_POW) c += 150;
                        else c += 60;
                    }
                    return c;
                }
                case OP_PHASOR: return op.mode == 1 ? 0 : 1850;          // a run costs what its leader costs
                case OP_SPHASOR: return 2200;
                case OP_COUNTER: case OP_ACCUM: case OP_LATCH: case OP_MAXHOLD: return 1500;
                case OP_RAND: return 450;
                case OP_POLE: return 1850;
                case OP_ENV: return 2000;
                case OP_BIQUAD: return 2600;
                case OP_PREWARP: return 1350;
                case OP_MM1P: return 6800;
                case OP_SVF: return 3450;
                case OP_SVFSHELF: return 4500;
                case OP_BLEP: return 2500;
                case OP_DELAY: return 3300;
                case OP_SDELAY: case OP_TABLE: return 800;
                case OP_Z: return 700;
                case OP_ROOT: return 1100;
                default: return 300;
            }
        };
        if (ok) {
            for (size_t i = 0; i < sops.size() && ok; ++i) {
                const auto& op = sops[i];
                if (op.isSeg) { ok = (i == 0); continue; }
                switch (op.opcode) {
                    case OP_FILL0: case OP_COPY: case OP_CHAIN: case OP_PHASOR: case OP_SPHASOR: case OP_COUNTER: case OP_ACCUM: case OP_LATCH:
                    case OP_MAXHOLD: case OP_RAND: case OP_POLE: case OP_ENV: case OP_BIQUAD: case OP_PREWARP: case OP_MM1P: case OP_SVF:
                    case OP_SVFSHELF: case OP_Z: case OP_DELAY: case OP_SDELAY: case OP_TABLE: case OP_BLEP: case OP_ROOT: break;
                    default: ok = false;
                }
            }
        }
        if (ok) {
            // units: an op, or a phasor run (leader + its followers), which must stay together
            std::vector<std::pair<size_t, size_t>> units;     // [first op, one past the last op)
            std::vector<long> ucost;
            for (size_t i = 1; i < sops.size();) {
                size_t j = i + 1;
                if (sops[i].opcode == OP_PHASOR && sops[i].aux1 > 1) j = i + sops[i].aux1;
                long c = 0;
                for (size_t k = i; k < j && k < sops.size(); ++k) c += costOf(sops[k]);
                units.push_back({i, std::min(j, sops.size())});
                ucost.push_back(c);
                i = j;
            }
            const int n = (int) units.size();
            if (n < 2 * W) ok = false;
            if (ok) {
                // linear partition: minimise the most expensive stage (O(n^2 W), n <= a few hundred)
                std::vector<long> pre(n + 1, 0);
                for (int i = 0; i < n; ++i) pre[i + 1] = pre[i] + ucost[i];
                const long INF = (long) 1 << 60;
                std::vector<std::vector<long>> best(W + 1, std::vector<long>(n + 1, INF));
                std::vector<std::vector<int>> cut(W + 1, std::vector<int>(n + 1, 0));
                best[0][0] = 0;
                for (int w = 1; w <= W; ++w)
                    for (int i = w; i <= n; ++i)
                        for (int j = w - 1; j < i; ++j) {
                            if (best[w - 1][j] >= INF) continue;
                            const long c = std::max(best[w - 1][j], pre[i] - pre[j]);
                            if (c < best[w][i]) { best[w][i] = c; cut[w][i] = j; }
                        }
                std::vector<int> bounds(W + 1, 0);
                bounds[W] = n;
                for (int w = W; w >= 1; --w) bounds[w - 1] = cut[w][bounds[w]];
                pipeStageOf.assign(sops.size(), 0);
                for (int w = 0; w < W; ++w)
                    for (int u = bounds[w]; u < bounds[w + 1]; ++u)
                        for (size_t k = units[u].first; k < units[u].second; ++k) pipeStageOf[k] = w;
                for (size_t i = 1; i < sops.size(); ++i)          // roots write the graph's output accumulator: last stage only
                    if (sops[i].opcode == OP_ROOT && pipeStageOf[i] != W - 1) { pipeStageOf.clear(); break; }
                if (!pipeStageOf.empty()) { prog->pipeW = W; prog->pipeDepth = W; }
            }
        }
    }

    // ---- per stage: slot allocation by liveness (an output slot is never the slot of one of its own inputs),
    //      then encoding ----
    std::unordered_map<uint32_t, uint32_t> smemIndexOfRow;
    int nStateRows = 0;
    auto mapState = [&](Node& n) -> uint32_t {
        if (n.stateRow < 0) return NO_STATE;
        auto it = smemIndexOfRow.find((uint32_t) n.stateRow);
        if (it != smemIndexOfRow.end()) return it->second;
        const TypeInfo ti = n.kind == NodeKind::Custom ? TypeInfo{NodeKind::Custom, n.fn, customTypes_[n.fn].nState, false} : typeTable().at(n.typeName);
        if (ti.evenAlign && (nStateRows & 1)) {   // keep doubles 8-byte aligned in shared memory
            prog->stateMap.push_back(STATE_PAD);
            nStateRows += 1;
        }
        const uint32_t idx = (uint32_t) nStateRows;
        if (ti.evenAlign) {
            for (int k = 0; k < ti.stateRows; k += 2) prog->stateMap.push_back(((uint32_t) n.stateRow + k) | STATE_DOUBLE_FLAG);
        } else {
            for (int k = 0; k < ti.stateRows; ++k) prog->stateMap.push_back((uint32_t) n.stateRow + k);
        }
        nStateRows += ti.stateRows;
        smemIndexOfRow[(uint32_t) n.stateRow] = idx;
        return idx;
    };
    std::unordered_map<int32_t, uint32_t> smemParamOfRow;
    int nSlotsMax = 1;
    prog->nOps = 0;
    if (prog->stages.empty()) prog->stages.resize(1);
    for (size_t stg = 0; stg < stageOps.size(); ++stg) {
        auto& sops = stageOps[stg];
        prog->stages[stg].codeOffset = (uint32_t) prog->code.size();

        std::vector<int> outSlot(sops.size(), 0);
        int nSlots = 0;
        bool piped = !pipeStageOf.empty() && stg == 0;
        if (piped) {
            // ring values: read in a later pipeline stage than the one that produces them
            const int W = prog->pipeW;
            std::unordered_map<int32_t, int> prodStage, ringOf;
            for (size_t i = 0; i < sops.size(); ++i) if (!sops[i].isSeg) prodStage[sops[i].outNode] = pipeStageOf[i];
            int nRing = 0;
            for (size_t i = 0; i < sops.size(); ++i) {
                if (sops[i].isSeg) continue;
                forEachSlotUse(sops[i], [&](int32_t id) {
                    auto ps = prodStage.find(id);
                    if (ps != prodStage.end() && ps->second < pipeStageOf[i] && !ringOf.count(id)) ringOf[id] = nRing++;
                });
            }
            // private slots: liveness inside each stage, every stage in its own index range
            int privBase = 0;
            for (int w = 0; w < W; ++w) {
                std::unordered_map<int32_t, size_t> lastUse;
                for (size_t i = 0; i < sops.size(); ++i)
                    if (!sops[i].isSeg && pipeStageOf[i] == w) forEachSlotUse(sops[i], [&](int32_t id) { lastUse[id] = i; });
                std::unordered_map<int32_t, int> slotOf;
                std::vector<int> freeSlots;
                int local = 0;
                for (size_t i = 0; i < sops.size(); ++i) {
                    auto& op = sops[i];
                    if (op.isSeg || pipeStageOf[i] != w) continue;
                    auto rg = ringOf.find(op.outNode);
                    if (rg != ringOf.end()) {
                        outSlot[i] = -(rg->second + 1);                      // placed behind the private ranges below
                    } else {
                        int sl;
                        if (!freeSlots.empty()) { sl = freeSlots.back(); freeSlots.pop_back(); }
                        else sl = local++;
                        outSlot[i] = privBase + sl;
                        slotOf[op.outNode] = sl;
                    }
                    forEachSlotUse(op, [&](int32_t id) {
                        auto lu = lastUse.find(id);
                        auto so = slotOf.find(id);
                        if (lu != lastUse.end() && lu->second == i && so != slotOf.end()) { freeSlots.push_back(so->second); slotOf.erase(so); }
                    });
                    if (rg == ringOf.end() && !lastUse.count(op.outNode)) {
                        auto so = slotOf.find(op.outNode);
                        if (so != slotOf.end()) { freeSlots.push_back(so->second); slotOf.erase(so); }
                    }
                }
                privBase += local;
            }
            const int ringBase = std::max(privBase, 1);
            nSlots = ringBase + nRing * prog->pipeDepth;
            if (nSlots >= MAX_SLOTS) {                                       // does not fit the 8-bit slot field: keep the program in one piece
                piped = false; pipeStageOf.clear(); prog->pipeW = 1; prog->pipeDepth = 1;
            } else {
                for (size_t i = 0; i < sops.size(); ++i) if (outSlot[i] < 0) outSlot[i] = ringBase + (-outSlot[i] - 1) * prog->pipeDepth;
                prog->pipeRingBase = ringBase;
            }
        }
        if (!piped) {
        std::unordered_map<int32_t, size_t> lastUse;
        for (size_t i = 0; i < sops.size(); ++i)
            if (!sops[i].isSeg) forEachSlotUse(sops[i], [&](int32_t id) { lastUse[id] = i; });
        std::unordered_map<int32_t, int> slotOf;
        std::vector<int> freeSlots;
        nSlots = 0;
        for (size_t i = 0; i < sops.size(); ++i) {
            auto& op = sops[i];
            if (op.isSeg) continue;
            int s;
            if (!freeSlots.empty()) { s = freeSlots.back(); freeSlots.pop_back(); }
            else s = nSlots++;
            if (s >= MAX_SLOTS) return fail(rc::InvariantViolation, "graph needs more than 255 live intermediates");
            outSlot[i] = s;
            slotOf[op.outNode] = s;
            forEachSlotUse(op, [&](int32_t id) {   // free inputs whose last consumer is this op
                auto lu = lastUse.find(id);
                auto so = slotOf.find(id);
                if (lu != lastUse.end() && lu->second == i && so != slotOf.end()) {
                    freeSlots.push_back(so->second);
                    slotOf.erase(so);
                }
            });
            // an output nobody reads (root buffers, dangling nodes) is dead immediately
            if (!lastUse.count(op.outNode)) { freeSlots.push_back(s); slotOf.erase(op.outNode); }
        }
        }
        nSlotsMax = std::max(nSlotsMax, nSlots);

        std::unordered_map<int32_t, int> producerSlot;   // every value is produced exactly once per stage
        for (size_t i = 0; i < sops.size(); ++i) if (!sops[i].isSeg) producerSlot[sops[i].outNode] = outSlot[i];
        auto encodeOperand = [&](uint32_t kind, int32_t ref) -> uint32_t {
            if (kind == K_SLOT) {
                auto ps = producerSlot.find(ref);
                if (ps == producerSlot.end()) return make_operand(K_PARAM, 0);   // never produced: reads as zero
                return make_operand(K_SLOT, (uint32_t) ps->second);
            }
            if (kind == K_PARAM) {
                auto it = smemParamOfRow.find(ref);
                if (it == smemParamOfRow.end()) {
                    prog->paramMap.push_back((uint32_t) ref);
                    it = smemParamOfRow.emplace(ref, (uint32_t) prog->paramMap.size()).first;   // 1-based
                }
                return make_operand(K_PARAM, it->second);
            }
            return make_operand(K_PARAM, 0);
        };
        auto opWords = [&](const Compiler::PendingOp& op) -> size_t {
            if (op.isSeg) return OP_HEADER_WORDS;
            size_t n = op.operands.size() + 2 * op.steps.size() + op.imm.size();
            return OP_HEADER_WORDS + ((n + 3) & ~(size_t) 3);
        };
        auto emitSeg = [&](int segRoot, size_t skipWords) {
            prog->code.push_back(make_w0(OP_SEG, 0, 0, 0));
            prog->code.push_back(NO_STATE);
            prog->code.push_back((uint32_t) segRoot);
            prog->code.push_back((uint32_t) skipWords);
            for (int k = 0; k < 4; ++k) prog->code.push_back(0);
        };
        auto emitOp = [&](const Compiler::PendingOp& op, int slot) -> int {
            ++prog->nOps;
            uint32_t st = NO_STATE;
            if (op.state != NO_STATE) {
                auto it = g.nodes.find(op.outNode);
                if (it != g.nodes.end()) st = mapState(it->second);
            }
            const size_t nOperandWords = opWords(op) - OP_HEADER_WORDS;
            if (nOperandWords > 255) return fail(rc::InvariantViolation, "operand block of one op exceeds 255 words");
            prog->code.push_back(make_w0(op.opcode, (uint32_t) nOperandWords, (uint32_t) slot, op.mode));
            prog->code.push_back(st);
            prog->code.push_back(op.aux0);
            prog->code.push_back(op.aux1);
            prog->code.push_back((uint32_t) op.ptr);
            prog->code.push_back((uint32_t) (op.ptr >> 32));
            prog->code.push_back((uint32_t) (op.opcode == OP_CHAIN ? op.steps.size() : op.operands.size()));
            prog->code.push_back(0);
            size_t written = 0;
            for (auto& o : op.operands) { prog->code.push_back(encodeOperand(o.first, o.second)); ++written; }
            for (auto& stp : op.steps) {
                prog->code.push_back(stp.fn);
                prog->code.push_back(chain_fn_is_unary(stp.fn) ? 0u : encodeOperand(stp.kind, stp.ref));
                written += 2;
            }
            for (uint32_t w : op.imm) { prog->code.push_back(w); ++written; }
            for (; written < nOperandWords; ++written) prog->code.push_back(0);
            return rc::Ok;
        };
        if (piped) {
            // one code section per pipeline stage: [SEG header][the stage's ops][END]; state rows in stage order
            const uint32_t base = prog->stages[stg].codeOffset;
            for (int w = 0; w < prog->pipeW; ++w) {
                prog->pipeCode[w] = (uint32_t) prog->code.size() - base;
                prog->pipeState[w] = (unsigned short) prog->stateMap.size();
                prog->pipeSrow[w] = (unsigned short) nStateRows;
                size_t words = 0;
                for (size_t i = 1; i < sops.size(); ++i) if (pipeStageOf[i] == w) words += opWords(sops[i]);
                emitSeg(sops[0].segRoot, words);
                for (size_t i = 1; i < sops.size(); ++i) {
                    if (pipeStageOf[i] != w) continue;
                    int r = emitOp(sops[i], outSlot[i]);
                    if (r != rc::Ok) return r;
                }
                for (int k = 0; k < 8; ++k) prog->code.push_back(k == 0 ? make_w0(OP_END, 0, 0, 0) : 0u);
            }
            for (int w = prog->pipeW; w <= MAX_PIPE; ++w) prog->pipeState[w] = (unsigned short) prog->stateMap.size();
        } else {
        std::vector<size_t> wordOffset(sops.size() + 1, 0);
        for (size_t i = 0; i < sops.size(); ++i) wordOffset[i + 1] = wordOffset[i] + opWords(sops[i]);
        for (size_t i = 0; i < sops.size(); ++i) {
            auto& op = sops[i];
            if (op.isSeg) { emitSeg(op.segRoot, wordOffset[op.segEndOp] - wordOffset[i + 1]); continue; }
            int r = emitOp(op, outSlot[i]);
            if (r != rc::Ok) return r;
        }
        }
        for (int k = 0; k < 8; ++k) prog->code.push_back(k == 0 ? make_w0(OP_END, 0, 0, 0) : 0u);
        if (stg + 1 == stageOps.size()) {   // tap promotion records live behind the last stage only
            for (auto& pr : C.promotes) {
                Node& n = g.nodes.at(pr.second);
                float* dst = g.tapShared[n.tapName];
                const uint64_t sb = (uint64_t) (uintptr_t) n.tapPrivate, db = (uint64_t) (uintptr_t) dst;
                prog->code.push_back(make_w0(OP_PROMOTE, 0, 0, 0));
                prog->code.push_back((uint32_t) pr.first);
                prog->code.push_back((uint32_t) sb); prog->code.push_back((uint32_t) (sb >> 32));
                prog->code.push_back((uint32_t) db); prog->code.push_back((uint32_t) (db >> 32));
                prog->code.push_back(0); prog->code.push_back(0);
            }
        }
        for (int k = 0; k < 8; ++k) prog->code.push_back(k == 0 ? make_w0(OP_END, 0, 0, 0) : 0u);
    }
    prog->nStateRows = (nStateRows + 1) & ~1;
    prog->nSlots = nSlotsMax;
    for (auto& st : prog->stages) {   // K1's tap promotion records: directly behind the stage's first OP_END, if there are any
        size_t pc = st.codeOffset;
        while (pc < prog->code.size() && (prog->code[pc] & 0xFF) != OP_END) pc += OP_HEADER_WORDS + ((prog->code[pc] >> 8) & 0xFF);
        pc += OP_HEADER_WORDS;
        st.promoteAt = (pc < prog->code.size() && (prog->code[pc] & 0xFF) == OP_PROMOTE) ? (int) (pc - st.codeOffset) : -1;
    }

    // ---- upload: code, stateMap and paramMap in ONE allocation; the copies are stream-ordered in front of the first launch and their
    // sources are members of the Program, so nothing has to be waited for here ----
    {
        const size_t codeW = (prog->code.size() + 3) & ~(size_t) 3, smW = (prog->stateMap.size() + 3) & ~(size_t) 3, pmW = prog->paramMap.size();
        if (!cuda(dmalloc((void**) &prog->dCode, sizeof(uint32_t) * (codeW + smW + pmW + 4)), "cudaMalloc program")) return rc::CudaError;
        if (!cuda(dmemcpy(prog->dCode, prog->code.data(), sizeof(uint32_t) * prog->code.size(), cudaMemcpyHostToDevice), "upload code")) return rc::CudaError;
        if (!prog->stateMap.empty()) {
            prog->dStateMap = prog->dCode + codeW;
            if (!cuda(dmemcpy(prog->dStateMap, prog->stateMap.data(), sizeof(uint32_t) * prog->stateMap.size(), cudaMemcpyHostToDevice), "upload stateMap")) return rc::CudaError;
        }
        if (!prog->paramMap.empty()) {
            prog->dParamMap = prog->dCode + codeW + smW;
            if (!cuda(dmemcpy(prog->dParamMap, prog->paramMap.data(), sizeof(uint32_t) * prog->paramMap.size(), cudaMemcpyHostToDevice), "upload paramMap")) return rc::CudaError;
        }
    }
    // Per-program specialisation of K1 (spec_host.h).  Not for groups that render through the batched many-groups launch (that
    // kernel is the interpreter by construction: one launch serves different programs), not for multi-stage programs.
    const bool batched = groups_.size() > 1 && opt_.batchGroups && !prog->hasCustom;
    if (prog->hasCustom) {
        // Registered device node types exist only inside a kernel compiled for the program: specialisation is mandatory and
        // synchronous, whatever the "specialize" option says, and a body that does not compile fails the COMMIT.
        if (prog->stages.size() > 1) return fail(rc::InvariantViolation, "a registered node type cannot share a graph with convolve");
        prog->specJob = specialise_request(prog->code, g.tileWidth, opt_.niter, device_, customSource());
        specialise_wait(*prog->specJob);
        if (prog->specJob->state.load(std::memory_order_acquire) < 0)
            return fail(rc::InvariantViolation, "registered node type failed to compile: " + prog->specJob->log);
    } else if (opt_.specialize && !batched && prog->stages.size() <= 1 && (int) prog->code.size() <= opt_.specializeMaxWords) {
        prog->specJob = specialise_request(prog->code, g.tileWidth, opt_.niter, device_, std::string(), midRangeDense(g.nv) ? 8 : opt_.specMinBlocks);   // NVRTC on the compile-queue thread
        if (opt_.specialize >= 2) {                                                          // synchronous mode: wait for the compiler here
            specialise_wait(*prog->specJob);
            if (prog->specJob->state.load(std::memory_order_acquire) < 0 && opt_.specializeStrict)
                return fail(rc::InvariantViolation, "K1 specialisation failed: " + prog->specJob->log);
        }
    }
    out = prog;
    return rc::Ok;
}

// ---------------------------------------------------------------------------------------------------------
// process
int Engine::ensureBuffers(size_t nIn, size_t nOut, bool perVoiceIn, bool materialise) {
    size_t tiles = 0;
    for (auto& g : groups_) tiles += (size_t) g->nTiles();
    const size_t pf = std::max<size_t>(1, tiles) * nOut * blockSize_;
    if (pf > partialFloats_) {
        dsync();
        if (dPartial_) dfree(dPartial_);
        if (!cuda(dmalloc((void**) &dPartial_, sizeof(float) * pf), "cudaMalloc partial")) return rc::CudaError;
        dmemset(dPartial_, 0, sizeof(float) * pf);
        partialFloats_ = pf;
    }
    if (materialise && !offlineOut_) {
        const size_t of = (size_t) numVoices_ * nOut * blockSize_;
        if (of > outVoiceFloats_) {
            dsync();
            if (dOutVoice_) dfree(dOutVoice_);
            if (!cuda(dmalloc((void**) &dOutVoice_, sizeof(float) * of), "cudaMalloc voice out")) return rc::CudaError;
            outVoiceFloats_ = of;
        }
    }
    if (perVoiceIn && nIn) { if (!voiceInDevicePtr(nIn)) return rc::CudaError; }
    else if (nIn) { if (!sharedInDevicePtr(nIn)) return rc::CudaError; }
    return rc::Ok;
}

float* Engine::voiceInDevicePtr(size_t nIn) {
    Lock lk(mu_);
    const size_t f = (size_t) numVoices_ * nIn * blockSize_;
    if (f > inVoiceFloats_) {
        dsync();
        if (dInVoice_) dfree(dInVoice_);
        dInVoice_ = nullptr;
        if (!cuda(dmalloc((void**) &dInVoice_, sizeof(float) * f), "cudaMalloc voice in")) return nullptr;
        dmemset(dInVoice_, 0, sizeof(float) * f);
        inVoiceFloats_ = f;
    }
    return dInVoice_;
}

float* Engine::sharedInDevicePtr(size_t nIn) {
    Lock lk(mu_);
    const size_t f = nIn * blockSize_;
    if (f > inSharedFloats_) {
        dsync();
        if (dInShared_) dfree(dInShared_);
        dInShared_ = nullptr;
        if (!cuda(dmalloc((void**) &dInShared_, sizeof(float) * f), "cudaMalloc shared in")) return nullptr;
        dmemset(dInShared_, 0, sizeof(float) * f);
        inSharedFloats_ = f;
    }
    return dInShared_;
}

int Engine::enqueueBlock(size_t nIn, size_t nOut, size_t numSamples, bool perVoiceIn, bool materialise, bool mix, bool allReduce) {
    Lock lk(mu_);
    // A plan-only engine cannot render.  With option "plan_dry_run" it still walks the whole host side of a block — program swap,
    // recompiles, descriptors, fades, event mirrors — and skips exactly the CUDA calls: the thread-safety tests (TSAN, no GPU) use it.
    if (planOnly_ && !planDryRun_) return fail(rc::CudaError, "plan-only runtime (no CUDA device): rendering is impossible, there is no CPU fallback");
    const bool dry = planOnly_;
    dsetdev();
    if (numSamples > (size_t) blockSize_ || nOut > (size_t) MAX_OUT_CHANNELS) return fail(rc::BadArgument, "numSamples > blockSize or too many output channels");

    const size_t key[6] = {nIn, nOut, numSamples, (size_t) perVoiceIn, (size_t) materialise | ((size_t) (uintptr_t) offlineOut_ << 1), (size_t) mix | ((size_t) offlineStride_ << 1)};
    if (steadyValid_ && !dry && std::memcmp(key, steadyKey_, sizeof key) == 0) {
        for (auto& sb : steadyBuckets_) {
            BatchBuffers& bb = batch_[sb.key];
            auto ev = timedBegin();
            if (!cuda(sb.pipeStages >= 1
                          ? launch_render_groups_pipe(bb.dDescs, bb.dTileStart, sb.nGroups, sb.totalTiles, sb.pipeStages, sb.maxSlots, (int) nOut, sb.maxState, sb.maxParams, sampleTime_, offlineOut_ ? offlineOffset_ : 0, stream_, opt_.niter)
                          : launch_render_groups(bb.dDescs, bb.dTileStart, sb.nGroups, sb.totalTiles, sb.L, sb.maxSlots, (int) nOut, sb.maxState, sb.maxParams, sb.wpc, sampleTime_, offlineOut_ ? offlineOffset_ : 0, stream_, opt_.niter),
                      "render groups kernel launch")) return rc::CudaError;
            if (timeKernels_) { cudaEventRecord(ev.second, stream_); timedEvents_.push_back(ev); }
            ++launches_;
        }
        if (mix) {
            auto ev = timedBegin();
            if (!cuda(launch_mix_reduce(dPartial_, dMix_, dMixScratch_, dMixTickets_, steadyTiles_, (int) nOut, blockSize_, (int) numSamples, stream_, takeDeliver()), "mix reduce launch")) return rc::CudaError;
            if (timeKernels_) { cudaEventRecord(ev.second, stream_); timedMixEvents_.push_back(ev); }
            ++launches_;
        }
        curNOut_ = nOut;
        sampleTime_ += (int64_t) numSamples;
        return rc::Ok;
    }
    bool allSteady = !(allReduce && peerAttached_ && peer_.world > 1), allBatched = true;

    // Runtime::process: swap in the newest render sequence (Runtime.h:277-285); recompile when the number of
    // host input channels a leaf node sees has changed.
    for (auto& gp : groups_) {
        Group& g = *gp;
        if (g.pending) { g.active = g.pending; g.pending.reset(); g.superseded.clear(); }
        if (g.active && g.codeDirty) {
            // A property that is baked into the program (svf.mode, delay.size, seq data, ...) was set after the last
            // COMMIT: the reference's nodes pick such changes up at the top of their next process() through atomics
            // and SPSC queues (e.g. Delays.h:92-95, Core.h:470-495); here the sequence is recompiled.
            std::shared_ptr<Program> p;
            int r = compile(g, (int) nIn, p);
            if (r != rc::Ok) return r;
            g.active = p;
        }
        if (g.active && g.active->nIn != (int) nIn) {
            if (g.active->usesHostInputs) {   // leaf nodes see the host channels: GraphRenderSequence.h:126-135
                std::shared_ptr<Program> p;
                int r = compile(g, (int) nIn, p);
                if (r != rc::Ok) return r;
                g.active = p;
            } else g.active->nIn = (int) nIn;
        }
    }
    int r = ensureBuffers(nIn, nOut, perVoiceIn, materialise);
    if (r != rc::Ok) return r;

    int tileBase = 0;
    std::map<int, std::vector<LaunchParams>> buckets;   // tile width -> single-stage groups launched together
    for (auto& gp : groups_) {
        Group& g = *gp;
        const int nTiles = g.nTiles();
        if (!g.active || nTiles == 0) { allSteady = false; }
        if (!g.active || nTiles == 0) {
            // no render sequence yet: outputs are silence (Runtime.h:287-289 leaves the host buffers untouched;
            // we define the voice's contribution as zero)
            if (nTiles && mix) dmemset(dPartial_ + (size_t) tileBase * nOut * blockSize_, 0, sizeof(float) * (size_t) nTiles * nOut * blockSize_);
            if (materialise && dOutVoice_ && !offlineOut_) dmemset(dOutVoice_ + (size_t) g.v0 * nOut * blockSize_, 0, sizeof(float) * (size_t) g.nv * nOut * blockSize_);
            tileBase += nTiles;
            continue;
        }
        Program& p = *g.active;
        LaunchParams P{};
        P.code = p.dCode;
        P.stateMap = p.dStateMap;
        P.paramMap = p.dParamMap;
        P.nParams = (int) p.paramMap.size();
        P.rows = g.dRows;
        P.inShared = (!perVoiceIn && nIn) ? dInShared_ : nullptr;
        P.inVoice = (perVoiceIn && nIn) ? dInVoice_ : nullptr;
        float* const voiceOut = offlineOut_ ? offlineOut_ : dOutVoice_;
        P.outVoice = materialise ? voiceOut : nullptr;
        P.mixPartial = mix ? dPartial_ : nullptr;
        P.nStateEntries = (int) p.stateMap.size();
        P.nStateRows = p.nStateRows;
        P.nSlots = p.nSlots;
        P.Vpad = g.Vpad;
        P.nv = g.nv;
        P.voice0 = g.v0;
        P.tileWidth = g.tileWidth;
        P.numSamples = (int) numSamples;
        P.blockSize = blockSize_;
        P.nIn = (int) nIn;
        P.nOut = (int) nOut;
        P.inStride = blockSize_;
        P.outStride = offlineOut_ ? offlineStride_ : blockSize_;
        P.tileBase = tileBase;
        uint32_t runMask = 0;
        for (size_t ri = 0; ri < p.rootIds.size(); ++ri) {
            auto it = g.nodes.find(p.rootIds[ri]);
            if (it == g.nodes.end()) continue;
            Node& rn = it->second;
            const bool stillRunning = rn.fade.on() || !rn.fade.settled();                     // Core.h:28-31
            const bool chanOk = rn.channel >= 0 && (size_t) rn.channel < nOut;                // GraphRenderSequence.h:214-219
            if (stillRunning && chanOk) runMask |= (1u << ri);
            if (rn.fade.on()) runMask |= (1u << (16 + ri));                                   // promoteTapBuffers: :200-205
            P.roots[ri] = RootDyn{rn.fade.current, rn.fade.step, rn.fade.target, rn.channel};
            if (rn.fade.current != rn.fade.target) allSteady = false;        // the descriptor changes while a root fades
        }
        if (!p.evNodes.empty() || !p.dynNodes.empty() || g.codeDirty || g.pending) allSteady = false;
        P.runMask = runMask;
        P.sampleTime = sampleTime_;
        P.tableSrc = p.stagedTable; P.tableFloats = p.stagedTableFloats; P.tableSmem = -1;   // the launcher places it (single-group launches)
        P.pipeW = p.pipeW; P.pipeRingBase = p.pipeRingBase; P.pipeDepth = p.pipeDepth;
        P.k1Prefetch = opt_.k1Prefetch ? 1 : 0;
        for (int w = 0; w < MAX_PIPE; ++w) { P.pipeCode[w] = p.pipeCode[w]; P.pipeSrow[w] = p.pipeSrow[w]; }
        for (int w = 0; w <= MAX_PIPE; ++w) P.pipeState[w] = p.pipeState[w];
        for (size_t di = 0; di < p.dynNodes.size(); ++di) {
            auto it = g.nodes.find(p.dynNodes[di]);
            if (it != g.nodes.end()) P.dyn[di] = it->second.scopeW;
        }
        for (auto& ev : p.evNodes) {       // host mirrors of what is identical for every voice of the group
            if (!((runMask >> ev.root) & 1u)) continue;
            auto it = g.nodes.find(ev.node);
            if (it == g.nodes.end()) continue;
            Node& en = it->second;
            if ((en.kind == NodeKind::Scope || en.kind == NodeKind::Fft) && (en.inlets.empty() ? nIn : en.inlets.size()) >= 1) {          // MultiChannelRingBuffer::write, :36-62
                const uint32_t mask = SCOPE_RING - 1, w = en.scopeW, r = en.scopeR, n = (uint32_t) numSamples;
                const uint32_t freeSlots = (r > w) ? (r - w) : ((uint32_t) SCOPE_RING - (w - r));
                en.scopeW = (w + n) & mask;
                if (n >= freeSlots) en.scopeR = (en.scopeW + 1) & mask;
            } else if (en.kind == NodeKind::Metro) {                        // Metro.h:44-55
                const double is = (double) en.intervalSamps;
                for (size_t i = 0; i < numSamples; ++i) {
                    const double t = (double) (sampleTime_ + (int64_t) i) / is;
                    const float nextOut = (float) ((t - std::floor(t)) < 0.5);
                    if (en.metroLastOut < 0.5f && nextOut >= 0.5f) en.metroFlag = true;
                    en.metroLastOut = nextOut;
                }
            }
        }

        // launch geometry: spread warps over the SMs first, then stack them
        int wpc = opt_.warpsPerCta;
        if (wpc <= 0) wpc = nTiles >= 148 * 8 ? 4 : (nTiles >= 148 * 4 ? 2 : 1);
        const size_t perWarp = render_smem_bytes(p.nSlots, (int) nOut, p.nStateRows, (int) p.paramMap.size(), 1, g.tileWidth, opt_.niter);
        while (wpc > 1 && perWarp * wpc > 200 * 1024) wpc >>= 1;
        if (perWarp > 220 * 1024) return fail(rc::InvariantViolation, "graph state does not fit in shared memory");
        const size_t nStages = std::max<size_t>(1, p.stages.size());
        if (nStages == 1 && groups_.size() > 1 && opt_.batchGroups && !p.hasCustom) {
            // heterogeneous voice groups: collect single-stage groups per tile geometry and launch each bucket once
            P.code = p.dCode + (p.stages.empty() ? 0 : p.stages[0].codeOffset);
            P.promoteAt = p.stages.empty() ? -1 : p.stages[0].promoteAt;
            // one-voice groups launch through the pipeline kernel (programs that were not cut simply use warp 0 of their CTA): one
            // launch for all of them whether or not every program could be cut
            const int bkey = g.tileWidth + ((p.pipeW > 1 || (g.tileWidth == 1 && opt_.pipelineStages > 1)) ? PIPE_BUCKET : 0);
            buckets[bkey].push_back(P);
            buckets[bkey].back().sampleTime = 0;      // the many-groups kernel takes the clock as an argument: descriptors stay equal block to block
        } else
        for (size_t stg = 0; stg < nStages; ++stg) {
            allBatched = false;
            const bool last = stg + 1 == nStages;
            P.code = p.dCode + (p.stages.empty() ? 0 : p.stages[stg].codeOffset);
            P.promoteAt = p.stages.empty() ? -1 : p.stages[stg].promoteAt;
            P.outVoice = (last && materialise) ? voiceOut + (offlineOut_ ? offlineOffset_ : 0) : nullptr;   // outputs and taps belong to the last stage
            P.mixPartial = (last && mix) ? dPartial_ : nullptr;
            std::pair<cudaEvent_t, cudaEvent_t> ev{nullptr, nullptr};
            if (timeKernels_) {
                if (!eventPool_.empty()) { ev = eventPool_.back(); eventPool_.pop_back(); }
                else { cudaEventCreate(&ev.first); cudaEventCreate(&ev.second); }
                cudaEventRecord(ev.first, stream_);
            }
            const bool emptyStage = !p.stages.empty() && ((p.stages[stg].empty && !last) || (last && p.fusedConvStage >= 0));   // fused: K3's epilogue did the root
            if (!emptyStage) {
                const SpecKernel* spec = nullptr;
                if (p.specJob) {   // the cubin arrived: load it on this thread (its CUDA context is current), a matter of milliseconds
                    const int st = specialise_ensure_loaded(*p.specJob);
                    if (st == 2) spec = &p.specJob->kernel;
                    else if (st < 0 && (opt_.specializeStrict || p.hasCustom)) return fail(rc::CudaError, "K1 specialisation failed: " + p.specJob->log);
                }
                if (!dry && !cuda(launch_render_block(P, wpc, opt_.niter, stream_, spec), "render kernel launch")) return rc::CudaError;
                ++launches_;
            }
            if (timeKernels_) { cudaEventRecord(ev.second, stream_); timedEvents_.push_back(ev); }
            if (p.stages.empty()) continue;
            // K3: the convolvers fed by this stage (ConvolutionNode::process, wasm/Convolve.h:58-85); a call longer
            // than what is left of the current 512-sample partition is cut like FFTConvolver.cpp:155-203 does
            for (size_t cvi = 0; cvi < p.stages[stg].convolves.size(); ++cvi) {
                auto& cv = p.stages[stg].convolves[cvi];
                auto it = g.nodes.find(cv.node);
                if (it == g.nodes.end() || !it->second.conv) continue;
                ConvolverState& cs = *it->second.conv;
                ConvEpilogue epi;
                if (p.fusedConvStage == (int) stg && p.fusedConvIndex == (int) cvi) {
                    const RootDyn& rd = P.roots[p.fusedRoot];
                    epi.active = true;
                    epi.running = ((runMask >> p.fusedRoot) & 1u) != 0;
                    epi.gain0 = rd.gain0; epi.step = rd.step; epi.target = rd.target; epi.channel = rd.channel;
                    epi.nOut = (int) nOut; epi.blockSize = blockSize_;
                    epi.mixPartial = mix ? dPartial_ : nullptr; epi.tileBase = tileBase;
                    epi.outVoice = materialise ? voiceOut + (offlineOut_ ? offlineOffset_ : 0) : nullptr;
                    epi.voice0 = g.v0; epi.outStride = P.outStride; epi.outOffset = 0;
                }
                int offset = 0;
                while (offset < (int) numSamples) {
                    const int n = cs.partitions == 0 ? (int) numSamples - offset
                                                     : std::min((int) numSamples - offset, CONV_BLOCK - cs.fill);
                    std::pair<cudaEvent_t, cudaEvent_t> ev3{nullptr, nullptr};
                    if (timeKernels_) {
                        if (!eventPool_.empty()) { ev3 = eventPool_.back(); eventPool_.pop_back(); }
                        else { cudaEventCreate(&ev3.first); cudaEventCreate(&ev3.second); }
                        cudaEventRecord(ev3.first, stream_);
                    }
                    const float* cin = cv.in;
                    int cinStride = blockSize_;
                    if (cv.inChannel >= 0) {   // straight from the host input buffers: per-voice [voice][nIn][blockSize] or shared [nIn][blockSize]
                        if (perVoiceIn) { cin = dInVoice_ + ((size_t) g.v0 * nIn + cv.inChannel) * blockSize_; cinStride = (int) nIn * blockSize_; }
                        else { cin = dInShared_ + (size_t) cv.inChannel * blockSize_; cinStride = 0; }
                    }
                    if (!dry && !cuda(convolver_process_chunk(cs, cin, cinStride, cv.out, blockSize_, offset, n, stream_, epi), "convolver launch")) return rc::CudaError;
                    if (dry) { offset += n; continue; }
                    if (timeKernels_) { cudaEventRecord(ev3.second, stream_); timedConvEvents_.push_back(ev3); }
                    ++launches_;
                    offset += n;
                }
            }
        }

        for (size_t ri = 0; ri < p.rootIds.size(); ++ri) {
            if (!(runMask & (1u << ri))) continue;
            auto it = g.nodes.find(p.rootIds[ri]);
            if (it != g.nodes.end()) it->second.fade.advance((int) numSamples);
        }
        tileBase += nTiles;
    }
    steadyBuckets_.clear();
    for (auto& kv : buckets) {
        auto& descs = kv.second;
        const int L = kv.first % PIPE_BUCKET;
        std::vector<int> tileStart(descs.size());
        int total = 0, maxSlots = 1, maxState = 0, maxParams = 0, pipeStages = 0;
        for (size_t i = 0; i < descs.size(); ++i) {
            tileStart[i] = total;
            total += (descs[i].nv + L - 1) / L;
            maxSlots = std::max(maxSlots, descs[i].nSlots);
            maxState = std::max(maxState, descs[i].nStateRows);
            maxParams = std::max(maxParams, descs[i].nParams);
            if (kv.first >= PIPE_BUCKET) pipeStages = std::max(pipeStages, std::max(1, descs[i].pipeW));
        }
        // descriptors change only while roots fade or when graphs change: re-upload only then
        BatchBuffers& bb = batch_[kv.first];
        const size_t dbytes = descs.size() * sizeof(LaunchParams), tbytes = tileStart.size() * sizeof(int);
        if (bb.capGroups < descs.size()) {
            dsync();
            if (bb.dDescs) dfree(bb.dDescs);
            if (bb.dTileStart) dfree(bb.dTileStart);
            bb.capGroups = descs.size() * 2;
            if (!cuda(dmalloc((void**) &bb.dDescs, bb.capGroups * sizeof(LaunchParams)), "cudaMalloc group descriptors")) return rc::CudaError;
            if (!cuda(dmalloc((void**) &bb.dTileStart, bb.capGroups * sizeof(int)), "cudaMalloc tile table")) return rc::CudaError;
            bb.lastDescs.clear();
        }
        if (!dry && (bb.lastDescs.size() != dbytes || std::memcmp(bb.lastDescs.data(), descs.data(), dbytes) != 0)) {
            if (!cuda(cudaMemcpyAsync(bb.dDescs, descs.data(), dbytes, cudaMemcpyHostToDevice, stream_), "upload group descriptors")) return rc::CudaError;
            if (!cuda(cudaMemcpyAsync(bb.dTileStart, tileStart.data(), tbytes, cudaMemcpyHostToDevice, stream_), "upload tile table")) return rc::CudaError;
            bb.lastDescs.assign(reinterpret_cast<const char*>(descs.data()), reinterpret_cast<const char*>(descs.data()) + dbytes);
        }
        int wpc = opt_.warpsPerCta;
        if (wpc <= 0) wpc = total >= 148 * 8 ? 4 : (total >= 148 * 4 ? 2 : 1);
        while (wpc > 1 && render_smem_bytes(maxSlots, (int) nOut, maxState, maxParams, wpc, L, L == 1 ? opt_.niter : 0) > 200 * 1024) wpc >>= 1;
        std::pair<cudaEvent_t, cudaEvent_t> ev{nullptr, nullptr};
        if (timeKernels_) {
            if (!eventPool_.empty()) { ev = eventPool_.back(); eventPool_.pop_back(); }
            else { cudaEventCreate(&ev.first); cudaEventCreate(&ev.second); }
            cudaEventRecord(ev.first, stream_);
        }
        steadyBuckets_.push_back(SteadyBucket{L, (int) descs.size(), total, maxSlots, maxState, maxParams, wpc, pipeStages, kv.first});
        if (!dry && !cuda(pipeStages >= 1
                              ? launch_render_groups_pipe(bb.dDescs, bb.dTileStart, (int) descs.size(), total, pipeStages, maxSlots, (int) nOut, maxState, maxParams, sampleTime_, offlineOut_ ? offlineOffset_ : 0, stream_, opt_.niter)
                              : launch_render_groups(bb.dDescs, bb.dTileStart, (int) descs.size(), total, L, maxSlots, (int) nOut, maxState, maxParams, wpc, sampleTime_, offlineOut_ ? offlineOffset_ : 0, stream_, opt_.niter),
                  "render groups kernel launch")) return rc::CudaError;
        if (timeKernels_) { cudaEventRecord(ev.second, stream_); timedEvents_.push_back(ev); }
        ++launches_;
    }
    // With the cross-GPU sum behind it, K2 leaves this rank's partial mix in PeerMix::own (K4 pushes it to the peers from there and
    // writes the total to the mix bus): no staging copy, no in-place hazard between K4's CTAs.
    const bool exchange = mix && allReduce && peerAttached_ && peer_.world > 1;
    float* mixOut = dMix_;
    if (exchange) {
        ++peerEpoch_;
        mixOut = peer_.own;
    }
    if (mix) {
        if (tileBase > 0) {
            auto ev = timedBegin();
            if (!dry && !cuda(launch_mix_reduce(dPartial_, mixOut, dMixScratch_, dMixTickets_, tileBase, (int) nOut, blockSize_, (int) numSamples, stream_, exchange ? HostDeliver{} : takeDeliver()), "mix reduce launch")) return rc::CudaError;
            if (timeKernels_) { cudaEventRecord(ev.second, stream_); timedMixEvents_.push_back(ev); }
            ++launches_;
        } else {
            dmemset(mixOut, 0, sizeof(float) * nOut * blockSize_);
        }
    }
    if (exchange) {   // K4: the cross-GPU sum of the mix bus, in the same stream
        auto ev = timedBegin();
        if (!cuda(launch_mix_exchange(peer_, dMix_, (int) (nOut * blockSize_), peerEpoch_, dPeerStatus_, stream_, takeDeliver()), "mix exchange launch")) return rc::CudaError;
        if (timeKernels_) { cudaEventRecord(ev.second, stream_); timedXchgEvents_.push_back(ev); }
        ++launches_;
    }
    steadyValid_ = allSteady && allBatched && !buckets.empty() && !dry;
    std::memcpy(steadyKey_, key, sizeof key);
    steadyTiles_ = tileBase;
    curNOut_ = nOut;
    sampleTime_ += (int64_t) numSamples;   // wasm/Main.cpp:217
    return rc::Ok;
}

HostDeliver Engine::takeDeliver() {
    HostDeliver hd;
    if (!deliverArmed_ || !hMixHost_ || planOnly_) return hd;
    deliverArmed_ = false;
    deliverLaunched_ = true;
    hd.out = dMixHostAlias_; hd.flag = dMixFlagAlias_; hd.done = dDeliverDone_; hd.seq = ++deliverSeq_;
    return hd;
}

std::pair<cudaEvent_t, cudaEvent_t> Engine::timedBegin() {
    std::pair<cudaEvent_t, cudaEvent_t> ev{nullptr, nullptr};
    if (!timeKernels_) return ev;
    if (!eventPool_.empty()) { ev = eventPool_.back(); eventPool_.pop_back(); }
    else { cudaEventCreate(&ev.first); cudaEventCreate(&ev.second); }
    cudaEventRecord(ev.first, stream_);
    return ev;
}

int Engine::peerBarrier() {
    Lock lk(mu_);
    if (planOnly_ || !peerAttached_ || peer_.world <= 1) return rc::Ok;
    dsetdev();
    if (!cuda(launch_mix_exchange(peer_, dMix_, 0, ++peerEpoch_, dPeerStatus_, stream_), "peer barrier launch")) return rc::CudaError;
    return rc::Ok;
}

double Engine::takeKernelTimeMs(uint64_t* count) {
    Lock lk(mu_);
    if (planOnly_) { if (count) *count = 0; return 0.0; }
    cudaStreamSynchronize(stream_);
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>>* lists[4] = {&timedEvents_, &timedMixEvents_, &timedConvEvents_, &timedXchgEvents_};
    for (int k = 0; k < 4; ++k) {
        lastKindMs_[k] = 0.0; lastKindCount_[k] = lists[k]->size();
        for (auto& ev : *lists[k]) {
            float ms = 0.0f;
            if (cudaEventElapsedTime(&ms, ev.first, ev.second) == cudaSuccess) lastKindMs_[k] += ms;
            eventPool_.push_back(ev);
        }
        lists[k]->clear();
    }
    lastConvMs_ = lastKindMs_[2]; lastConvCount_ = lastKindCount_[2];
    if (count) *count = lastKindCount_[0];
    return lastKindMs_[0];
}

int Engine::renderOffline(size_t nOut, size_t numBlocks, float* hostOut, size_t chunkBlocks) {
    Lock lk(mu_);
    if (planOnly_) return fail(rc::CudaError, "plan-only runtime (no CUDA device): rendering is impossible, there is no CPU fallback");
    if (!hostOut || nOut == 0 || nOut > (size_t) MAX_OUT_CHANNELS) return fail(rc::BadArgument, "renderOffline: bad arguments");
    dsetdev();
    const size_t bs = (size_t) blockSize_, rows = (size_t) numVoices_ * nOut;
    size_t C = chunkBlocks ? chunkBlocks : 8;
    while (C > 1 && rows * C * bs * sizeof(float) > ((size_t) 256 << 20)) C >>= 1;          // two chunk buffers of at most 256 MiB each
    if (C > numBlocks) C = std::max<size_t>(1, numBlocks);
    // Chunk buffers: two on the device (rendered into back to back) and two PINNED on the host.  The user's buffer is pageable and
    // strided ([row][numBlocks * bs]); a 2-D copy straight into it would be staged by the driver row by row, synchronously.  So a chunk
    // leaves the device as ONE contiguous async copy into pinned memory on the copy stream, and this thread scatters the previous
    // chunk's rows into the user's buffer while the GPU renders the next one.  The buffers are kept across calls.
    const size_t chunkFloats = rows * C * bs;
    if (chunkFloats > offlineChunkFloats_) {
        dsync();
        for (int i = 0; i < 2; ++i) {
            if (offlineDev_[i]) cudaFree(offlineDev_[i]);
            if (offlinePinned_[i]) cudaFreeHost(offlinePinned_[i]);
            offlineDev_[i] = nullptr; offlinePinned_[i] = nullptr;
        }
        offlineChunkFloats_ = 0;
        for (int i = 0; i < 2; ++i) {
            if (!cuda(cudaMalloc((void**) &offlineDev_[i], chunkFloats * sizeof(float)), "cudaMalloc offline chunk")) return rc::CudaError;
            if (!cuda(cudaMallocHost((void**) &offlinePinned_[i], chunkFloats * sizeof(float)), "cudaMallocHost offline chunk")) return rc::CudaError;
        }
        offlineChunkFloats_ = chunkFloats;
    }
    cudaStream_t copyStream = nullptr;
    cudaEvent_t rendered[2] = {nullptr, nullptr}, copied[2] = {nullptr, nullptr};
    int rcode = rc::Ok;
    for (int i = 0; i < 2; ++i) {
        cudaMemsetAsync(offlineDev_[i], 0, chunkFloats * sizeof(float), stream_);               // voices without a render sequence stay silent
        cudaEventCreateWithFlags(&rendered[i], cudaEventDisableTiming);
        cudaEventCreateWithFlags(&copied[i], cudaEventDisableTiming);
    }
    cudaStreamCreateWithFlags(&copyStream, cudaStreamNonBlocking);
    steadyValid_ = false;
    struct Pending { bool valid = false; size_t chunk = 0, blocks = 0; int slot = 0; } prev;
    auto scatter = [&](const Pending& pc) {          // pinned chunk [row][C * bs] -> user rows
        if (!pc.valid) return;
        if (!cuda(cudaEventSynchronize(copied[pc.slot]), "wait for an offline chunk")) { rcode = rc::CudaError; return; }
        const size_t width = pc.blocks * bs;
        for (size_t r = 0; r < rows; ++r)
            std::memcpy(hostOut + r * numBlocks * bs + pc.chunk * C * bs, offlinePinned_[pc.slot] + r * C * bs, width * sizeof(float));
    };
    for (size_t b = 0; b < numBlocks && rcode == rc::Ok; ++b) {
        const size_t chunk = b / C, inChunk = b % C;
        const int slot = (int) (chunk & 1);
        if (inChunk == 0 && chunk >= 2) cudaStreamWaitEvent(stream_, copied[slot], 0);          // the chunk two back has left this device buffer
        offlineOut_ = offlineDev_[slot]; offlineStride_ = (int) (C * bs); offlineOffset_ = (int) (inChunk * bs);
        rcode = enqueueBlock(0, nOut, bs, false, true, false);
        const bool lastOfChunk = inChunk + 1 == C || b + 1 == numBlocks;
        if (rcode == rc::Ok && lastOfChunk) {
            // the pinned buffer of this slot was scattered when chunk - 1 was enqueued (below), i.e. before this copy is issued
            cudaEventRecord(rendered[slot], stream_);
            cudaStreamWaitEvent(copyStream, rendered[slot], 0);
            if (!cuda(cudaMemcpyAsync(offlinePinned_[slot], offlineDev_[slot], chunkFloats * sizeof(float), cudaMemcpyDeviceToHost, copyStream), "D2H offline chunk")) rcode = rc::CudaError;
            cudaEventRecord(copied[slot], copyStream);
            Pending cur; cur.valid = true; cur.chunk = chunk; cur.blocks = inChunk + 1; cur.slot = slot;
            scatter(prev);                                                                      // overlaps with the GPU rendering what was just enqueued
            prev = cur;
        }
    }
    scatter(prev);
    offlineOut_ = nullptr; offlineStride_ = 0; offlineOffset_ = 0; steadyValid_ = false;
    cudaStreamSynchronize(stream_);
    if (copyStream) { cudaStreamSynchronize(copyStream); cudaStreamDestroy(copyStream); }
    for (int i = 0; i < 2; ++i) { if (rendered[i]) cudaEventDestroy(rendered[i]); if (copied[i]) cudaEventDestroy(copied[i]); }
    return rcode;
}

int Engine::synchronize() {
    if (planOnly_) return rc::Ok;
    const cudaError_t e = cudaStreamSynchronize(stream_);     // no lock while waiting for the GPU
    if (e == cudaSuccess) return rc::Ok;
    Lock lk(mu_);
    cuda(e, "stream synchronize");
    return rc::CudaError;
}

int Engine::process(const float* const* in, size_t nIn, float* const* out, size_t nOut, size_t numSamples, const int64_t* sampleTime) {
    float* hOut = nullptr;
    uint32_t waitSeq = 0;
    bool polled = false;
    {
        Lock lk(mu_);   // held while the block is ENQUEUED; the wait for the GPU below runs without it (the control thread may work meanwhile)
        if (planOnly_) return fail(rc::CudaError, "plan-only runtime (no CUDA device): rendering is impossible, there is no CPU fallback");
        dsetdev();
        if (sampleTime) sampleTime_ = *sampleTime;   // BlockContext::userData as the wasm host passes it (wasm/Main.cpp:206-215)
        if (numSamples > (size_t) blockSize_) return fail(rc::BadArgument, "numSamples > blockSize");
        const size_t need = (nIn + nOut) * blockSize_;
        if (need > pinnedFloats_) {
            if (hPinned_) { dsync(); cudaFreeHost(hPinned_); }
            if (!cuda(cudaMallocHost(&hPinned_, sizeof(float) * need), "cudaMallocHost")) return rc::CudaError;
            pinnedFloats_ = need;
        }
        if (nIn) {
            float* d = sharedInDevicePtr(nIn);
            if (!d) return rc::CudaError;
            for (size_t c = 0; c < nIn; ++c) std::memcpy(hPinned_ + c * blockSize_, in[c], sizeof(float) * numSamples);
            if (!cuda(dmemcpy(d, hPinned_, sizeof(float) * nIn * blockSize_, cudaMemcpyHostToDevice), "H2D inputs")) return rc::CudaError;
        }
        // With peers attached every rank's process() returns the mix of ALL ranks (K4), like one Runtime over all the voices would.
        deliverArmed_ = hostDeliver_ && nOut > 0 && hMixHost_ != nullptr;
        deliverLaunched_ = false;
        int r = enqueueBlock(nIn, nOut, numSamples, false, false, true, processAllReduce_ && peerAttached_ && peer_.world > 1);
        deliverArmed_ = false;
        if (r != rc::Ok) return r;
        if (deliverLaunched_) {
            hOut = hMixHost_;
            waitSeq = deliverSeq_;
            polled = true;
        } else {
            hOut = hPinned_ + nIn * blockSize_;
            if (nOut) {
                if (!cuda(dmemcpy(hOut, dMix_, sizeof(float) * nOut * blockSize_, cudaMemcpyDeviceToHost), "D2H mix")) return rc::CudaError;
            }
        }
    }
    if (polled) {
        // The kernel that finishes the mix bus has stored it into mapped host memory and raises the sequence word behind it: poll that
        // word (no D2H copy launch, no stream synchronize wake-up).  A failed launch never raises it — the stream is queried every
        // ~20 us so that an error (or a finished stream) ends the wait.
        using clk = std::chrono::steady_clock;
        auto lastQuery = clk::now();
        for (;;) {
            if (*hMixFlag_ == waitSeq) break;
            for (int k = 0; k < 32; ++k) cpuRelax();
            const auto now = clk::now();
            if (now - lastQuery > std::chrono::microseconds(20)) {
                lastQuery = now;
                const cudaError_t q = cudaStreamQuery(stream_);
                if (q == cudaErrorNotReady) continue;
                if (q != cudaSuccess) { Lock lk(mu_); cuda(q, "stream query while waiting for the mix bus"); return rc::CudaError; }
                if (*hMixFlag_ == waitSeq) break;
                Lock lk(mu_);
                return fail(rc::CudaError, "the render stream finished without delivering the mix bus");
            }
        }
        std::atomic_thread_fence(std::memory_order_acquire);
    } else {
        int r = synchronize();
        if (r != rc::Ok) return r;
    }
    // hPinned_ belongs to the render thread: only process() (re)allocates it
    for (size_t c = 0; c < nOut; ++c) std::memcpy(out[c], hOut + c * blockSize_, sizeof(float) * numSamples);
    return rc::Ok;
}

int Engine::processVoices(const float* in, size_t nIn, float* outVoices, float* mix, size_t nOut, size_t numSamples) {
    {
        Lock lk(mu_);
        if (planOnly_) return fail(rc::CudaError, "plan-only runtime (no CUDA device): rendering is impossible, there is no CPU fallback");
        dsetdev();
        if (numSamples > (size_t) blockSize_) return fail(rc::BadArgument, "numSamples > blockSize");
        const bool perVoiceIn = in != nullptr && nIn > 0;
        if (perVoiceIn) {
            float* d = voiceInDevicePtr(nIn);
            if (!d) return rc::CudaError;
            // host layout [voice][nIn][numSamples] -> device [voice][nIn][blockSize]
            if (!cuda(cudaMemcpy2DAsync(d, sizeof(float) * blockSize_, in, sizeof(float) * numSamples, sizeof(float) * numSamples,
                                        (size_t) numVoices_ * nIn, cudaMemcpyHostToDevice, stream_), "H2D voice inputs")) return rc::CudaError;
        }
        int r = enqueueBlock(nIn, nOut, numSamples, perVoiceIn, outVoices != nullptr, mix != nullptr);
        if (r != rc::Ok) return r;
        if (outVoices) {
            if (!cuda(cudaMemcpy2DAsync(outVoices, sizeof(float) * numSamples, dOutVoice_, sizeof(float) * blockSize_, sizeof(float) * numSamples,
                                        (size_t) numVoices_ * nOut, cudaMemcpyDeviceToHost, stream_), "D2H voice outputs")) return rc::CudaError;
        }
        if (mix) {
            if (!cuda(cudaMemcpy2DAsync(mix, sizeof(float) * numSamples, dMix_, sizeof(float) * blockSize_, sizeof(float) * numSamples,
                                        nOut, cudaMemcpyDeviceToHost, stream_), "D2H mix")) return rc::CudaError;
        }
    }
    return synchronize();
}

} // namespace eb
