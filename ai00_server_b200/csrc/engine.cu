// b200rwkv engine: model build from `.st`, per-step kernel schedule, state ops, C ABI.
// Host side is plain C++ (the reference's engine, web-rwkv, is compiled Rust; no Rust toolchain
// exists in this image) — see include/b200rwkv.h for the reference call site of every entry.
#include "../../include/b200rwkv.h"

#include <unistd.h>

#include <algorithm>
#include <condition_variable>
#include <functional>
#include <thread>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <stdexcept>
#include <string>
#include <vector>

#include "gemm.cuh"
#include "qgemm.cuh"
#include "pre6.cuh"
#include "sample.cuh"
#include "misc.cuh"
#include "mix.cuh"
#ifdef B200RWKV_DEBUG
#include "streamtest.cuh"
#endif
#include "wkv.cuh"

namespace b200 {

// =========================================================================================
// errors
// =========================================================================================
struct Error : std::runtime_error {
    int code;
    Error(int c, const std::string& m) : std::runtime_error(m), code(c) {}
};
#define CK(call)                                                                                         \
    do {                                                                                                 \
        cudaError_t e_ = (call);                                                                         \
        if (e_ != cudaSuccess)                                                                           \
            throw Error(B200RWKV_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_) + " @" +   \
                                               __FILE__ + ":" + std::to_string(__LINE__) + watchdog_report()); \
    } while (0)
#define REQUIRE(cond, code, msg)                 \
    do {                                         \
        if (!(cond)) throw Error((code), (msg)); \
    } while (0)

static thread_local std::string g_err;

// Bring-up switches exist only in the debug build (-DB200RWKV_DEBUG, `python -m ai00_server_b200.build --debug` ->
// libb200rwkv_dbg.so): the product library ignores the environment entirely.
static inline const char* dbg_env(const char* name) {
#ifdef B200RWKV_DEBUG
    return getenv(name);
#else
    (void)name;
    return nullptr;
#endif
}

// watchdog record in mapped pinned host memory (see common.cuh)
static unsigned* g_wd_host = nullptr;
static void watchdog_setup() {
    if (g_wd_host) { memset(g_wd_host, 0, 64); return; }
    unsigned* h = nullptr;
    if (cudaHostAlloc(&h, 64, cudaHostAllocMapped | cudaHostAllocPortable) != cudaSuccess) return;
    memset(h, 0, 64);
    g_wd_host = h;
}
static std::string watchdog_report() {
    if (!g_wd_host || (g_wd_host[0] >> 16) != 0xDEADu) return "";
    char buf[256];
    snprintf(buf, sizeof buf, " [device watchdog: code=%u block=%u thread=%u a0=0x%x a1=%u a2=%u]", g_wd_host[0] & 0xFFFFu, g_wd_host[1],
             g_wd_host[2], g_wd_host[3], g_wd_host[4], g_wd_host[5]);
    return buf;
}

// =========================================================================================
// safetensors reader (header = u64 LE length + JSON object; tensor bytes follow)
// =========================================================================================
struct StTensor {
    std::string name;
    std::string dtype;
    std::vector<int64_t> shape;
    const uint8_t* data = nullptr;
    size_t nbytes = 0;
    int64_t numel() const {
        int64_t n = 1;
        for (auto d : shape) n *= d;
        return n;
    }
};

class StFile {
public:
    std::map<std::string, StTensor> tensors;

    StFile(const uint8_t* buf, size_t len) {
        REQUIRE(buf && len >= 8, B200RWKV_ERR_INVALID, "safetensors: buffer too small");
        uint64_t hlen = 0;
        memcpy(&hlen, buf, 8);
        REQUIRE(hlen <= len - 8, B200RWKV_ERR_INVALID, "safetensors: bad header length");
        s_ = reinterpret_cast<const char*>(buf + 8);
        n_ = (size_t)hlen;
        i_ = 0;
        const uint8_t* base = buf + 8 + hlen;
        const size_t data_len = len - 8 - hlen;
        ws();
        expect('{');
        ws();
        if (peek() == '}') return;
        for (;;) {
            ws();
            std::string key = str();
            ws();
            expect(':');
            ws();
            if (key == "__metadata__") {
                skip_value();
            } else {
                StTensor t;
                size_t b = 0, e = 0;
                expect('{');
                for (;;) {
                    ws();
                    std::string k = str();
                    ws();
                    expect(':');
                    ws();
                    if (k == "dtype") t.dtype = str();
                    else if (k == "shape") {
                        auto v = int_array();
                        t.shape.assign(v.begin(), v.end());
                    } else if (k == "data_offsets") {
                        auto v = int_array();
                        REQUIRE(v.size() == 2, B200RWKV_ERR_INVALID, "safetensors: data_offsets");
                        b = (size_t)v[0];
                        e = (size_t)v[1];
                    } else skip_value();
                    ws();
                    if (peek() == ',') { ++i_; continue; }
                    expect('}');
                    break;
                }
                REQUIRE(b <= e && e <= data_len, B200RWKV_ERR_INVALID, "safetensors: tensor out of bounds: " + key);
                t.data = base + b;
                t.nbytes = e - b;
                // byte length must equal dtype size x shape product (overflow-checked): every later size check trusts numel()
                const size_t esz = dtype_size(t.dtype);
                REQUIRE(esz > 0, B200RWKV_ERR_INVALID, "safetensors: unknown dtype '" + t.dtype + "' of " + key);
                REQUIRE(t.shape.size() <= 8, B200RWKV_ERR_INVALID, "safetensors: too many dimensions: " + key);
                uint64_t ne = 1;
                for (int64_t d : t.shape) {
                    REQUIRE(d >= 0 && (d == 0 || ne <= (uint64_t)1 << 40) && (uint64_t)d <= ((uint64_t)1 << 40), B200RWKV_ERR_INVALID,
                            "safetensors: bad shape of " + key);
                    ne *= (uint64_t)d;
                }
                REQUIRE(ne <= ((uint64_t)1 << 44) && ne * esz == (uint64_t)t.nbytes, B200RWKV_ERR_INVALID,
                        "safetensors: byte length of " + key + " does not match dtype x shape");
                t.name = key;
                tensors.emplace(std::move(key), std::move(t));
            }
            ws();
            if (peek() == ',') { ++i_; continue; }
            expect('}');
            break;
        }
    }
    const StTensor* find(const std::string& name) const {
        auto it = tensors.find(name);
        return it == tensors.end() ? nullptr : &it->second;
    }
    const StTensor& get(const std::string& name) const {
        auto* t = find(name);
        REQUIRE(t, B200RWKV_ERR_INVALID, "missing tensor: " + name);
        REQUIRE(t->dtype == "F16", B200RWKV_ERR_UNSUPPORTED, "tensor " + name + " is " + t->dtype + ", expected F16");
        return *t;
    }

    static size_t dtype_size(const std::string& d) {
        if (d == "F16" || d == "BF16" || d == "I16" || d == "U16") return 2;
        if (d == "F32" || d == "I32" || d == "U32") return 4;
        if (d == "F64" || d == "I64" || d == "U64") return 8;
        if (d == "I8" || d == "U8" || d == "BOOL" || d == "F8_E4M3" || d == "F8_E5M2") return 1;
        return 0;
    }
    // dimension i of a tensor that must have exactly `rank` dimensions (0 = any rank > i)
    static int64_t dim(const StTensor& t, size_t i, const std::string& name, size_t rank = 0) {
        REQUIRE((rank == 0 || t.shape.size() == rank) && i < t.shape.size(), B200RWKV_ERR_INVALID, "unexpected rank of tensor " + name);
        REQUIRE(t.shape[i] > 0 && t.shape[i] <= (int64_t)1 << 30, B200RWKV_ERR_INVALID, "bad dimension of tensor " + name);
        return t.shape[i];
    }
    int64_t dim(const std::string& name, size_t i, size_t rank = 0) const { return dim(get(name), i, name, rank); }

private:
    const char* s_;
    size_t n_, i_;
    int depth_ = 0;
    char peek() { return i_ < n_ ? s_[i_] : '\0'; }
    void ws() { while (i_ < n_ && (s_[i_] == ' ' || s_[i_] == '\n' || s_[i_] == '\t' || s_[i_] == '\r')) ++i_; }
    void expect(char c) {
        REQUIRE(peek() == c, B200RWKV_ERR_INVALID, std::string("safetensors: expected '") + c + "'");
        ++i_;
    }
    std::string str() {
        expect('"');
        std::string out;
        while (i_ < n_ && s_[i_] != '"') {
            if (s_[i_] == '\\' && i_ + 1 < n_) {
                ++i_;
                char c = s_[i_];
                if (c == 'n') out.push_back('\n');
                else if (c == 't') out.push_back('\t');
                else if (c == 'u') { i_ += 4; out.push_back('?'); }
                else out.push_back(c);
            } else out.push_back(s_[i_]);
            ++i_;
        }
        expect('"');
        return out;
    }
    std::vector<int64_t> int_array() {
        std::vector<int64_t> v;
        expect('[');
        ws();
        if (peek() == ']') { ++i_; return v; }
        for (;;) {
            ws();
            int64_t x = 0;
            bool any = false;
            while (i_ < n_ && s_[i_] >= '0' && s_[i_] <= '9') { x = x * 10 + (s_[i_] - '0'); ++i_; any = true; }
            REQUIRE(any, B200RWKV_ERR_INVALID, "safetensors: expected integer");
            v.push_back(x);
            ws();
            if (peek() == ',') { ++i_; continue; }
            expect(']');
            break;
        }
        return v;
    }
    struct DepthGuard {
        int& d;
        explicit DepthGuard(int& d_) : d(d_) { ++d; }
        ~DepthGuard() { --d; }
    };
    void skip_value() {
        DepthGuard dg(depth_);
        REQUIRE(depth_ <= 64, B200RWKV_ERR_INVALID, "safetensors: header nested too deeply");
        ws();
        char c = peek();
        if (c == '"') { (void)str(); return; }
        if (c == '{' || c == '[') {
            const char close = (c == '{') ? '}' : ']';
            ++i_;
            ws();
            if (peek() == close) { ++i_; return; }
            for (;;) {
                ws();
                if (c == '{') { (void)str(); ws(); expect(':'); }
                skip_value();
                ws();
                if (peek() == ',') { ++i_; continue; }
                expect(close);
                return;
            }
        }
        while (i_ < n_ && s_[i_] != ',' && s_[i_] != '}' && s_[i_] != ']') ++i_;
    }
};

// Mirror of web-rwkv `Loader::info` (reference lib.rs:587): version and dims from names/shapes.
static b200rwkv_info derive_info(const StFile& st) {
    b200rwkv_info o;
    memset(&o, 0, sizeof(o));
    o.num_vocab = (int)st.dim("emb.weight", 0, 2);
    o.num_emb = (int)st.dim("emb.weight", 1, 2);
    int L = 0;
    while (st.find("blocks." + std::to_string(L) + ".ln1.weight")) ++L;
    REQUIRE(L > 0, B200RWKV_ERR_INVALID, "no blocks.*.ln1.weight tensors");
    o.num_layer = L;
    o.num_hidden = (int)st.dim("blocks.0.ffn.key.weight", 0, 2);
    if (st.find("blocks.0.att.r_k")) {
        o.version = 7;
        o.num_head = (int)st.dim("blocks.0.att.r_k", 0, 2);
        o.head_size = (int)st.dim("blocks.0.att.r_k", 1, 2);
        o.time_decay_adapter = (int)st.dim("blocks.0.att.w1", 0, 2);
    } else if (st.find("blocks.0.att.time_mix_w1")) {
        o.version = 6;
        o.num_head = (int)st.dim("blocks.0.att.time_first", 0, 2);
        o.head_size = (int)st.dim("blocks.0.att.time_first", 1, 2);
        o.time_mix_adapter = (int)st.dim("blocks.0.att.time_mix_w1", 0, 2) / 5;
        o.time_decay_adapter = (int)st.dim("blocks.0.att.time_decay_w1", 0, 2);
    } else if (st.find("blocks.0.att.ln_x.weight") && st.find("blocks.0.att.gate.weight")) {
        o.version = 5;
        REQUIRE(st.get("blocks.0.att.time_first").shape.size() == 2, B200RWKV_ERR_UNSUPPORTED, "v5.0 (scalar time_first) is not supported");
        o.num_head = (int)st.dim("blocks.0.att.time_first", 0, 2);
        o.head_size = (int)st.dim("blocks.0.att.time_first", 1, 2);
    } else {
        throw Error(B200RWKV_ERR_UNSUPPORTED, "unsupported model version (RWKV v5.1/5.2, v6, v7 are supported)");
    }
    return o;
}

static float st_elem_f32(const StTensor& t, size_t i) {
    if (t.dtype == "F16") return __half2float(reinterpret_cast<const __half*>(t.data)[i]);
    if (t.dtype == "F32") { float v; memcpy(&v, t.data + i * 4, 4); return v; }
    if (t.dtype == "BF16") { uint32_t u = (uint32_t)reinterpret_cast<const uint16_t*>(t.data)[i] << 16; float v; memcpy(&v, &u, 4); return v; }
    throw Error(B200RWKV_ERR_UNSUPPORTED, "tensor " + t.name + " is " + t.dtype + ", expected F16 / F32 / BF16");
}

// `vN::read_state` (reference lib.rs:378-389) and `State::init` with a state-tuned model (run.rs:477, lib.rs:452-462):
// `blocks.{l}.att.time_state` [H, N, N] (transposed by the converter, convert_safetensors.py:101, crates/converter/src/main.rs:20)
// -> the host state tensor [L][N+2][C]: row 1+i, column h*N+j <- time_state[h][i][j]; shift rows zero.
// Returns false (and leaves `out` empty) when the file carries no time_state.
static bool state_from_st(const StFile& st, int L, int H, int N, int C, std::vector<float>& out) {
    if (!st.find("blocks.0.att.time_state")) return false;
    out.assign((size_t)L * (N + 2) * C, 0.f);
    for (int l = 0; l < L; ++l) {
        const std::string name = "blocks." + std::to_string(l) + ".att.time_state";
        const StTensor* ts = st.find(name);
        REQUIRE(ts, B200RWKV_ERR_INVALID, "missing tensor: " + name);
        REQUIRE(ts->numel() == (int64_t)H * N * N, B200RWKV_ERR_INVALID, "time_state must be [num_head, head_size, head_size]: " + name);
        for (int h = 0; h < H; ++h)
            for (int i = 0; i < N; ++i)
                for (int j = 0; j < N; ++j)
                    out[((size_t)l * (N + 2) + 1 + i) * C + h * N + j] = st_elem_f32(*ts, ((size_t)h * N + i) * N + j);
    }
    return true;
}

// =========================================================================================
// engine
// =========================================================================================
static inline int cdiv(int a, int b) { return (a + b - 1) / b; }
static inline int rup(int a, int b) { return cdiv(a, b) * b; }

enum KClass { KC_GEMM = 0, KC_WKV = 1, KC_LN = 2, KC_OTHER = 3 };

struct GemmLaunch {
    GemmParams p;
    int grid = 0;
    int grid_wide = 0;         // grid of steps with >= 64 tokens: whole tiles per CTA (see make_launch)
    int total_tiles = 0;
    size_t weight_bytes = 0;   // algorithmic (unpadded) weight bytes streamed (f16, or codes + block parameters)
    int qtype = QT_NONE;       // weight format of every segment of the launch (qgemm.cuh)
    bool forced = false;       // grid fixed by the caller (static split-K: tiles x slices CTAs)
};

struct SegDesc {
    const StTensor* t = nullptr;
    int64_t slice = -1;        // leading-dim index for 3-D tensors
    int n0 = 0, N = 0, k0 = 0, K = 0;
    GemmSeg proto;             // A, out_mode, act, bias, out, ldo, grp, grp_stride, aux*
    SegDesc() { memset(&proto, 0, sizeof(proto)); }
};

struct A16Buf {
    __half* p = nullptr;
    int kq = 0;                // k32 blocks per m-tile (padded K / 32)
    size_t halves_per_matrix = 0;
};

struct Layer {
    LnMixParams ln1, ln2;
    std::vector<GemmLaunch> pre;    // launches between LN1 and WKV
    int wd2_index = -1;             // v6: index in `pre` of the decay-LoRA stage-2 launch (skipped when the WKV kernel evaluates it in place)
    WkvParams wkv;
    GemmLaunch o;
    std::vector<GemmLaunch> ffn;    // launches after LN2
    // v6 decode front half as one launch (pre6.cuh): row-major copies of the ddlerp LoRA weights
    const __half* w1_raw = nullptr;
    const __half* w2_raw = nullptr;
    const float* mu5[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
};

struct Profiler {
    struct Rec { int cls; cudaEvent_t a, b; };
    std::vector<Rec> recs;
};

// CachedItem {state, output} on the device (run.rs:199-205).  `row`: the slot had a kept logits row when the snapshot was taken;
// recorded on every tensor-parallel rank (only rank 0 holds the row itself) so that checks of it agree across ranks.
struct Snapshot { float* buf = nullptr; float* logits = nullptr; size_t bytes = 0; bool row = false; };

}  // namespace b200

using namespace b200;

// In-process tensor parallelism (b200rwkv_create_ex with num_devices > 1): the handle the host holds is rank 0's engine; it
// owns the other ranks and one worker thread per rank.  Every SPMD entry point fans out to all ranks CONCURRENTLY (the ranks'
// kernels rendezvous with each other over NVLink, so one thread issuing rank after rank would deadlock on its first
// stream synchronisation) and returns rank 0's result: the reference's single `Runtime` object (run.rs:1230-1234).
struct Group {
    std::vector<b200rwkv_engine*> ranks;      // [world]; ranks[0] is the handle itself
    std::vector<std::thread> workers;         // ranks 1..world-1 (rank 0's share runs on the calling thread)
    std::mutex m;
    std::condition_variable cv;
    std::function<int32_t(int)> job;
    uint64_t gen = 0;
    int pending = 0;
    bool stop = false;
    std::vector<int32_t> status;
    std::vector<std::string> errs;
    std::mutex call_mu;                       // one fan-out at a time

    void start(int world);
    void shutdown();
    int32_t spmd(const std::function<int32_t(int)>& fn);
};

struct b200rwkv_engine {
    std::unique_ptr<Group> group;             // set on rank 0 of an in-process tensor-parallel engine
    b200rwkv_info info;
    int dev = 0, rank = 0, world = 1, num_sms = 148;
    int S = 0, chunk = 0, maxT = A16_MAX_ROWS, precision = 0;      // steps of up to 128 tokens
    int L = 0, C = 0, F = 0, V = 0, H = 0, N = 64, Cl = 0, Hl = 0, Fl = 0, Vl = 0;
    bool use_graph = true, use_pdl = true;
    int split_att = 1, split_ffn = 1;
    // tensor parallel: one symmetric comm block per rank (partials, gate block, logits shard, flags)
    uint8_t* comm_base = nullptr;
    size_t comm_bytes = 0, off_part_att = 0, off_part_ffn = 0, off_rr = 0, off_logits = 0, off_flags = 0;
    uint8_t* peer_base[8] = {nullptr};
    bool peer_ipc[8] = {false};       // peer_base[q] was opened with cudaIpcOpenMemHandle (closed in the destructor)
    bool connected = false;
    TpBar tpbar;
    unsigned* d_epoch = nullptr;
    cudaStream_t stream = nullptr, sm_stream = nullptr;
    std::vector<void*> allocs;
    size_t weight_bytes_total = 0;

    // model
    __half* emb = nullptr;
    EmbedParams embed;
    std::vector<Layer> layers;
    LnOutParams lnout;
    GemmLaunch head;

    // state
    float *att_shift = nullptr, *ffn_shift = nullptr, *wkv_state = nullptr, *d_api = nullptr;
    std::vector<float> init_state;     // API layout, empty => zeros
    std::map<uint64_t, Snapshot> snaps;
    uint64_t next_snap = 1;

    // activations
    float *x_a = nullptr, *x_b = nullptr, *xx1 = nullptr, *sx1 = nullptr, *xx2 = nullptr;
    float *f_r = nullptr, *f_k = nullptr, *f_v = nullptr, *f_g = nullptr, *f_w = nullptr, *f_a = nullptr, *f_nu = nullptr,
          *f_vfirst = nullptr, *f_rr = nullptr, *part_att = nullptr, *part_ffn = nullptr, *d_logits = nullptr, *d_hidden = nullptr;
    A16Buf a_x[6], a_lora[5], a_out, a_kk, a_head;
    float* gemm_ws = nullptr;
    size_t gemm_ws_floats = 0;

    // step plumbing
    static constexpr int META_RING = 4;
    cudaEvent_t meta_ev[META_RING] = {nullptr, nullptr, nullptr, nullptr};
    bool hidden_keep = false;          // b200rwkv_keep_hidden: accumulate the hidden rows of every token of an infer call
    float* d_hidden_all = nullptr;
    size_t hidden_cap_rows = 0;
    int hidden_rows = 0;
    int *d_meta = nullptr, *h_meta = nullptr;
    int* d_meta_all = nullptr;
    size_t meta_ints = 0;
    std::map<int, cudaGraphExec_t> graphs;
    std::map<int, long long> graph_launches;   // kernels per captured step graph
    long long launch_total = 0;                // kernels launched by this engine's steps since creation
    long long launches_last_step = 0;
    // the most recent step of b200rwkv_infer (b200rwkv_debug_read): tokens, output rows, token rows of the A16 operands and
    // of the head's operand, split (hi + lo) operands
    int last_T = 0, last_R = 0, last_th = 16, last_th_rows = 16;
    bool last_split = false;

    // softmax
    float *sm_in = nullptr, *sm_out = nullptr;
    int sm_rows_cap = 0;

    // sampling front half (sample.cuh): last logits row of every slot, candidate scratch, staging blobs
    float* d_keep = nullptr;                 // [S][V] (rank 0)
    std::vector<char> keep_valid;            // slot has a logits row (guarded by keep_mu)
    std::mutex keep_mu;
    cudaEvent_t step_done = nullptr;         // recorded on `stream` after every step: the sampling stream waits on it
    float* tk_cand_x = nullptr; unsigned* tk_cand_id = nullptr; float2* tk_stats = nullptr;
    unsigned* tk_out_id = nullptr; float* tk_out_p = nullptr;
    uint8_t *tk_dev = nullptr, *tk_host = nullptr;
    size_t tk_cap = 0;
    void enqueue_keep(cudaStream_t s, int MTR);
    void sample_topk(int nrows, const int32_t* slots, const int32_t* pen_off, const uint32_t* pen_tok, const float* pen_val,
                     const uint32_t* allow_bits, const int32_t* bias_off, const uint32_t* bias_tok, const float* bias_val,
                     int top_k, uint32_t* ids_out, float* probs_out);

    // scoring (b200rwkv_infer_score, rank 0): (row, target, destination) lists travel in their own pinned ring, separate
    // from the step metadata; log-probabilities collect in d_logp and go to the host once per call
    static constexpr int SCORE_RING = 4;
    ScoreItem *h_score = nullptr, *d_score = nullptr;
    int score_cap = 0;                       // items per ring buffer: max(maxT, S)
    cudaEvent_t score_ev[SCORE_RING] = {nullptr, nullptr, nullptr, nullptr};
    float* d_logp = nullptr;
    size_t logp_floats = 0;
    void enqueue_score(const std::vector<ScoreItem>& items, int seq);

    std::mutex mu, sm_mu;

    // LoRA files blended into the projection weights while they are uploaded (borrowed during build only)
    struct LoraSrc { const StFile* st; float alpha; };
    std::vector<LoraSrc> loras;
    void check_loras(const StFile& model) const;
    void blend_loras(const StTensor& t);

    // temp upload buffer during build
    __half* d_tmp = nullptr;
    size_t d_tmp_bytes = 0;
    const StTensor* d_tmp_holds = nullptr;

    ~b200rwkv_engine();
    void* dalloc(size_t bytes, bool zero = true);
    void build(const StFile& st);
    const __half* upload_tmp(const StTensor& t);
    float* vec_f32(const StFile& st, const std::string& name, size_t off, size_t count, float scale = 1.f, float bias = 0.f);
    A16Buf a16_alloc(int K, int nmat = 1);
    GemmLaunch make_launch(std::vector<SegDesc>& segs, int force_grid = 0, int qtype = QT_NONE);
    int quant_layers = 0, quant_type = QT_NONE;     // the first `quant_layers` layers hold Int8 / NF4 projection matrices
    bool q_ts = true;                               // expanded weights go to tensor memory (qgemm.cuh); false = reference variant
    int pick_split(int K, int tiles) const;
    void finalize_tp();
    template <typename P, typename... X>
    void launch_k(void (*kern)(P, X...), dim3 grid, dim3 block, size_t smem, const P& params, int cls, cudaStream_t s, Profiler* prof,
                  X... extra);
    bool fold_wd2 = false;
    unsigned step_seq = 0;        // step sequence number uploaded as meta[4]
    bool split_on = false;        // precision 1: split (hi + lo f16) projection operands, every step decode-shaped
    bool split_act = false;
    int prefetch_blocks = 16;     // L2 prefetch depth (32 KB blocks per CTA) into the next projection launch
    bool fused_pre = true, ln_cluster = true;     // decode-shaped cluster kernels of pre6.cuh
    bool fused_pre_ok = false, ln_cluster_ok = false;
    unsigned* pre_gbar = nullptr;
    int launch_cluster = 0;                       // consumed by the next launch_k
    // profiling aid (B200RWKV_STEP_TRACE=1): 8 globaltimer stamps of CTA 0 per launch of the per-op chain
    unsigned long long* d_step_trace = nullptr;
    std::vector<int> step_trace_types;
    static constexpr int STEP_TRACE_MAX = 1024;
    static constexpr int STEP_TRACE_ROW = 512;     // 8 stamps of CTA 0 + {SM id, last MMA, exit} of every projection CTA
    bool trace_capture = false;                    // stamps are wired into the launches being enqueued / captured right now
    std::vector<long long> step_trace_bytes;       // algorithmic weight bytes of each traced projection launch
    unsigned long long* tr_next(int label) {
        if (!d_step_trace || !trace_capture || launches_last_step >= STEP_TRACE_MAX) return nullptr;
        if ((int)step_trace_types.size() <= launches_last_step) step_trace_types.resize(launches_last_step + 1);
        step_trace_types[launches_last_step] = label;
        return d_step_trace + (size_t)STEP_TRACE_ROW * launches_last_step;
    }
    void launch_gemm(const GemmLaunch& g, int MT, cudaStream_t s, Profiler* prof, bool split = false);
    void enqueue_step(cudaStream_t s, int MT, int MTR, Profiler* prof);
    bool pre_skipped(const Layer& ly, int gi, int MT) const;
    void run_step(int MT, int MTR);
    int fill_meta(int* m, const std::vector<int>& slots, const std::vector<int>& counts, const std::vector<const uint32_t*>& toks,
                  const std::vector<int>& outmode /*0 none,1 last,2 full*/, int* R_out);
    void infer(int nslot, const int32_t* slot, const int32_t* ntok, const uint32_t* tokens, const int32_t* option,
               float* logits_out, size_t cap, int32_t* rows_out, float* logp_out = nullptr, size_t logp_cap = 0, bool scoring = false);
    void state_xform(int slot, bool import, float* snap = nullptr);
};

b200rwkv_engine::~b200rwkv_engine() {
    cudaSetDevice(dev);
    cudaDeviceSynchronize();
    for (auto& kv : graphs) cudaGraphExecDestroy(kv.second);
    for (auto& kv : snaps) { cudaFree(kv.second.buf); if (kv.second.logits) cudaFree(kv.second.logits); }
    for (int q = 0; q < 8; ++q)
        if (peer_ipc[q] && peer_base[q]) cudaIpcCloseMemHandle(peer_base[q]);
    for (void* p : allocs) cudaFree(p);
    if (d_tmp) cudaFree(d_tmp);          // only still set when build() threw
    if (sm_in) cudaFree(sm_in);
    if (sm_out) cudaFree(sm_out);
    if (h_meta) cudaFreeHost(h_meta);
    if (tk_dev) cudaFree(tk_dev);
    if (tk_host) cudaFreeHost(tk_host);
    if (h_score) cudaFreeHost(h_score);
    if (d_score) cudaFree(d_score);
    if (d_logp) cudaFree(d_logp);
    for (auto& ev : score_ev) if (ev) cudaEventDestroy(ev);
    if (step_done) cudaEventDestroy(step_done);
    for (auto& ev : meta_ev) if (ev) cudaEventDestroy(ev);
    if (d_hidden_all) cudaFree(d_hidden_all);
    if (stream) cudaStreamDestroy(stream);
    if (sm_stream) cudaStreamDestroy(sm_stream);
}

// scratch device allocation released on every exit path
struct DevTmp {
    void* p = nullptr;
    explicit DevTmp(size_t bytes) {
        cudaError_t e_ = cudaMalloc(&p, std::max<size_t>(bytes, 16));
        if (e_ != cudaSuccess) throw Error(B200RWKV_ERR_CUDA, std::string("cudaMalloc (scratch): ") + cudaGetErrorString(e_));
    }
    ~DevTmp() { if (p) cudaFree(p); }
    DevTmp(const DevTmp&) = delete;
    DevTmp& operator=(const DevTmp&) = delete;
};

void* b200rwkv_engine::dalloc(size_t bytes, bool zero) {
    void* p = nullptr;
    bytes = std::max<size_t>(bytes, 16);
    CK(cudaMalloc(&p, bytes));
    allocs.push_back(p);
    if (zero) CK(cudaMemset(p, 0, bytes));
    return p;
}

const __half* b200rwkv_engine::upload_tmp(const StTensor& t) {
    if (d_tmp_holds != &t) {
        REQUIRE(t.nbytes <= d_tmp_bytes, B200RWKV_ERR_INVALID, "internal: temp buffer too small");
        CK(cudaMemcpy(d_tmp, t.data, t.nbytes, cudaMemcpyHostToDevice));
        d_tmp_holds = &t;
        blend_loras(t);
    }
    return d_tmp;
}

static bool ends_with(const std::string& s, const std::string& suf) {
    return s.size() >= suf.size() && s.compare(s.size() - suf.size(), suf.size(), suf) == 0;
}

// Every `<base>.lora.0/.lora.1` pair of a LoRA file must address a projection matrix this engine blends (the matrices that
// go through upload_tmp); anything else is refused loudly rather than ignored.
void b200rwkv_engine::check_loras(const StFile& model) const {
    static const char* ok[] = {".att.receptance", ".att.key", ".att.value", ".att.gate", ".att.output", ".ffn.key", ".ffn.value", ".ffn.receptance"};
    for (const LoraSrc& lo : loras) {
        int pairs = 0;
        for (auto& kv : lo.st->tensors) {
            const std::string& n = kv.first;
            if (ends_with(n, ".lora.1")) continue;
            if (!ends_with(n, ".lora.0")) {
                REQUIRE(!model.find(n), B200RWKV_ERR_UNSUPPORTED, "LoRA file carries a full tensor (" + n + "): only low-rank pairs on projection matrices are blended");
                continue;
            }
            const std::string base = n.substr(0, n.size() - 7);
            bool good = (base == "head");
            for (const char* o : ok) good = good || ends_with(base, o);
            REQUIRE(good && model.find(base + ".weight"), B200RWKV_ERR_UNSUPPORTED, "LoRA on " + base + " is not supported (projection matrices only)");
            REQUIRE(lo.st->find(base + ".lora.1"), B200RWKV_ERR_INVALID, "LoRA file: " + base + ".lora.1 is missing");
            ++pairs;
        }
        REQUIRE(pairs > 0, B200RWKV_ERR_INVALID, "LoRA file holds no <name>.lora.0 / <name>.lora.1 pairs");
    }
}

void b200rwkv_engine::blend_loras(const StTensor& t) {
    if (loras.empty() || !ends_with(t.name, ".weight") || t.shape.size() != 2) return;
    const std::string base = t.name.substr(0, t.name.size() - 7);
    const int out = (int)t.shape[0], in = (int)t.shape[1];
    for (const LoraSrc& lo : loras) {
        const StTensor* a = lo.st->find(base + ".lora.0");
        const StTensor* b = lo.st->find(base + ".lora.1");
        if (!a || !b) continue;
        REQUIRE(a->dtype == "F16" && b->dtype == "F16", B200RWKV_ERR_UNSUPPORTED, "LoRA tensors must be F16: " + base);
        REQUIRE(a->shape.size() == 2 && b->shape.size() == 2 && b->shape[0] == out && a->shape[0] == in && a->shape[1] == b->shape[1] &&
                    a->shape[1] >= 1 && a->shape[1] <= 4096,
                B200RWKV_ERR_INVALID, "LoRA shapes do not match " + t.name + " (expected lora.0 [in, r], lora.1 [out, r])");
        const int r = (int)a->shape[1];
        DevTmp da(a->nbytes), db(b->nbytes);
        CK(cudaMemcpy(da.p, a->data, a->nbytes, cudaMemcpyHostToDevice));
        CK(cudaMemcpy(db.p, b->data, b->nbytes, cudaMemcpyHostToDevice));
        lora_blend_kernel<<<148 * 8, 256>>>(d_tmp, (const __half*)db.p, (const __half*)da.p, out, in, r, lo.alpha);
        CK(cudaGetLastError());
        CK(cudaDeviceSynchronize());
    }
}

float* b200rwkv_engine::vec_f32(const StFile& st, const std::string& name, size_t off, size_t count, float scale, float bias) {
    const StTensor& t = st.get(name);
    REQUIRE((size_t)t.numel() >= off + count, B200RWKV_ERR_INVALID, "tensor too small: " + name);
    float* d = (float*)dalloc(count * 4, false);
    DevTmp tmp(count * 2);
    CK(cudaMemcpy(tmp.p, t.data + off * 2, count * 2, cudaMemcpyHostToDevice));
    f16_to_f32_kernel<<<cdiv((int)count, 256), 256>>>((const __half*)tmp.p, d, count, scale, bias);
    CK(cudaGetLastError());
    CK(cudaDeviceSynchronize());
    return d;
}

A16Buf b200rwkv_engine::a16_alloc(int K, int nmat) {
    A16Buf b;
    const int Kp = rup(K, GEMM_BK);          // whole 128-wide k blocks, zero padded
    b.kq = Kp / 32;
    b.halves_per_matrix = (size_t)(Kp / GEMM_BK) * A16_KB_HALVES;
    b.p = (__half*)dalloc(b.halves_per_matrix * 2 * nmat, true);
    return b;
}

GemmLaunch b200rwkv_engine::make_launch(std::vector<SegDesc>& segs, int force_grid, int qtype) {
    REQUIRE(!segs.empty() && (int)segs.size() <= GEMM_MAX_SEG, B200RWKV_ERR_INVALID, "internal: bad segment count");
    GemmLaunch g;
    memset(&g.p, 0, sizeof(g.p));
    g.qtype = qtype;
    g.forced = force_grid > 0;
    g.p.qvar = 1;
    if (const char* v = dbg_env("B200RWKV_QVAR")) g.p.qvar = atoi(v);
    const size_t blk_bytes = (size_t)q_block_bytes(qtype);
    int blk = 0, tile = 0, kbmax = 0;
    for (size_t i = 0; i < segs.size(); ++i) {
        SegDesc& d = segs[i];
        GemmSeg& sg = g.p.seg[i];
        sg = d.proto;
        // A16 outputs are written as whole 16-byte chunks of 8 rows (gemm.cuh epilogue)
        REQUIRE(sg.out_mode == OUT_F32 || (d.N % 8 == 0 && sg.grp % 8 == 0), B200RWKV_ERR_UNSUPPORTED,
                "LoRA ranks / hidden size must be multiples of 8");
        sg.KB = cdiv(d.K, GEMM_BK);
        sg.tiles = cdiv(d.N, GEMM_BN);
        sg.N = d.N;
        sg.blk_begin = blk;
        sg.tile_begin = tile;
        blk += sg.tiles * sg.KB;
        tile += sg.tiles;
        kbmax = std::max(kbmax, sg.KB);
        if (qtype == QT_NONE) g.weight_bytes += (size_t)d.N * d.K * 2;
        else {
            // quantisation blocks are runs of 128 (Int8) / 64 (NF4) consecutive inputs of one output row of the FULL matrix
            REQUIRE(d.K % GEMM_BK == 0 && d.k0 % GEMM_BK == 0, B200RWKV_ERR_UNSUPPORTED,
                    "quantised projections need input dimensions that are multiples of 128");
            g.weight_bytes += qtype == QT_INT8 ? (size_t)d.N * d.K + (size_t)d.N * (d.K / 128) * 4
                                               : (size_t)d.N * d.K / 2 + (size_t)d.N * (d.K / 64) * 2;
        }
    }
    g.p.nseg = (int)segs.size();
    g.p.total_blocks = blk;
    g.total_tiles = tile;
    uint8_t* W = (uint8_t*)dalloc((size_t)blk * blk_bytes, false);
    g.p.W = W;
    for (size_t i = 0; i < segs.size(); ++i) {
        SegDesc& d = segs[i];
        const GemmSeg& sg = g.p.seg[i];
        const StTensor& t = *d.t;
        const __half* src = upload_tmp(t);
        int ld;
        if (d.slice >= 0) {
            REQUIRE(t.shape.size() == 3, B200RWKV_ERR_INVALID, "internal: slice of non-3D tensor");
            ld = (int)t.shape[2];
            src += (size_t)d.slice * t.shape[1] * t.shape[2];
            REQUIRE(d.slice < t.shape[0] && d.n0 + d.N <= t.shape[1] && d.k0 + d.K <= t.shape[2], B200RWKV_ERR_INVALID, "weight shape mismatch");
        } else {
            REQUIRE(t.shape.size() == 2, B200RWKV_ERR_INVALID, "internal: expected 2-D weight");
            ld = (int)t.shape[1];
            REQUIRE(d.n0 + d.N <= t.shape[0] && d.k0 + d.K <= t.shape[1], B200RWKV_ERR_INVALID, "weight shape mismatch");
        }
        if (qtype != QT_NONE) {
            const size_t nwarp = (size_t)sg.tiles * sg.KB * GEMM_BN;
            const int grid = (int)std::min<size_t>((nwarp + 7) / 8, 148 * 32);
            uint8_t* dstq = W + (size_t)sg.blk_begin * blk_bytes;
            if (qtype == QT_INT8) quantize_weight_kernel<QT_INT8><<<grid, 256>>>(src, ld, d.n0, d.k0, d.N, sg.tiles, sg.KB, dstq);
            else quantize_weight_kernel<QT_NF4><<<grid, 256>>>(src, ld, d.n0, d.k0, d.N, sg.tiles, sg.KB, dstq);
            CK(cudaGetLastError());
            CK(cudaDeviceSynchronize());
            continue;
        }
        const size_t nchunk = (size_t)sg.tiles * sg.KB * (GEMM_WBYTES / 16);
        const int grid = (int)std::min<size_t>((nchunk + 255) / 256, 148 * 16);
        repack_weight_kernel<<<grid, 256>>>(src, ld, d.n0, d.k0, d.N, d.K, sg.tiles, sg.KB,
                                            reinterpret_cast<uint4*>(W + (size_t)sg.blk_begin * GEMM_WBYTES));
        CK(cudaGetLastError());
        CK(cudaDeviceSynchronize());   // d_tmp is reused by the next upload
    }
    g.grid = std::max(1, std::min(num_sms, std::max(tile, cdiv(blk, 4))));
    g.grid = std::min(g.grid, blk);
    if (force_grid > 0) g.grid = std::min(force_grid, blk);
    else {
        // Whole tiles per CTA whenever that keeps >= 3/4 of the SMs streaming: no cross-CTA fix-up in the tail, and
        // (measured, profiles/r01_findings.md §7) grids of <= 16 CTAs per GPC finish together while 144-148 CTAs skew
        // by 25 % because the 18/20-SM GPCs share the same GPC bandwidth as the 16-SM ones.
        if (tile <= num_sms && tile * 4 >= num_sms * 3) g.grid = tile;
        else if (tile > num_sms)
            for (int cand = num_sms; cand * 4 >= num_sms * 3; --cand)
                if (tile % cand == 0) { g.grid = cand; break; }
    }
    // Steps of 64 / 128 tokens: a partial accumulator tile is 32 / 64 KB per contributor, and the last arriver of a cut tile
    // spends tens of microseconds summing them (measured: 3B K+R at 128 tokens, last MMA at 9-15 us, slowest CTA exits at
    // 82 us; profiles/r02_steptrace_prefill128_3b.log).  Those steps run whole tiles per CTA, even if that leaves SMs idle.
    g.grid_wide = g.grid;
    if (force_grid <= 0) {
        if (tile <= num_sms) g.grid_wide = tile;
        else
            for (int cand = num_sms; cand * 2 >= num_sms; --cand)        // several whole tiles per CTA; else keep stream-K
                if (tile % cand == 0) { g.grid_wide = cand; break; }
    }
    const int per_cta = std::max(1, blk / g.grid);
    g.p.max_contrib = cdiv(kbmax, per_cta) + 1;
    g.p.counters = (unsigned*)dalloc((size_t)tile * 4, true);
    g.p.nrows = d_meta;   // T by default
    g.p.w_lbo = GEMM_W_LBO; g.p.w_sbo = GEMM_W_SBO; g.p.a_lbo = GEMM_A_LBO; g.p.a_sbo = GEMM_A_SBO;
    gemm_ws_floats = std::max(gemm_ws_floats, (size_t)tile * g.p.max_contrib * (size_t)maxT * GEMM_BN);
    weight_bytes_total += g.weight_bytes;
    return g;
}

template <typename P, typename... X>
void b200rwkv_engine::launch_k(void (*kern)(P, X...), dim3 grid, dim3 block, size_t smem, const P& params, int cls, cudaStream_t s,
                               Profiler* prof, X... extra) {
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    cudaLaunchAttribute at[2];
    int na = 0;
    if (launch_cluster > 0) {
        at[na].id = cudaLaunchAttributeClusterDimension;
        at[na].val.clusterDim.x = (unsigned)launch_cluster;
        at[na].val.clusterDim.y = 1;
        at[na].val.clusterDim.z = 1;
        ++na;
        launch_cluster = 0;
    }
    if (use_pdl && !prof) {
        at[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
        at[na].val.programmaticStreamSerializationAllowed = 1;
        ++na;
    }
    cfg.attrs = at;
    cfg.numAttrs = na;
    cudaEvent_t ea = nullptr, eb = nullptr;
    if (prof) {
        CK(cudaEventCreate(&ea));
        CK(cudaEventCreate(&eb));
        CK(cudaEventRecord(ea, s));
    }
    CK(cudaLaunchKernelEx(&cfg, kern, params, extra...));
    if (prof) {
        CK(cudaEventRecord(eb, s));
        prof->recs.push_back({cls, ea, eb});
    }
    ++launches_last_step;
}

void b200rwkv_engine::launch_gemm(const GemmLaunch& g, int MT, cudaStream_t s, Profiler* prof, bool split) {
    if (g.qtype != QT_NONE) {
        REQUIRE(!split, B200RWKV_ERR_UNSUPPORTED, "internal: quantised projections run with f16 activations");
        const int grid = MT >= 4 ? g.grid_wide : g.grid;
#define QLAUNCH(MT_, QT_) launch_k(qgemm_kernel<MT_, QT_, true>, dim3(grid), dim3(QGEMM_THREADS), QGemmCfg<MT_, QT_, true>::SMEM_BYTES, g.p, KC_GEMM, s, prof)
        if (!q_ts && MT == 1) {      // reference variant (expanded weights through shared memory), decode shape only
            if (g.qtype == QT_INT8) launch_k(qgemm_kernel<1, QT_INT8, false>, dim3(grid), dim3(QGEMM_THREADS), QGemmCfg<1, QT_INT8, false>::SMEM_BYTES, g.p, KC_GEMM, s, prof);
            else launch_k(qgemm_kernel<1, QT_NF4, false>, dim3(grid), dim3(QGEMM_THREADS), QGemmCfg<1, QT_NF4, false>::SMEM_BYTES, g.p, KC_GEMM, s, prof);
        } else if (g.qtype == QT_INT8) {
            switch (MT) { case 1: QLAUNCH(1, QT_INT8); break; case 2: QLAUNCH(2, QT_INT8); break; case 4: QLAUNCH(4, QT_INT8); break; default: QLAUNCH(8, QT_INT8); break; }
        } else {
            switch (MT) { case 1: QLAUNCH(1, QT_NF4); break; case 2: QLAUNCH(2, QT_NF4); break; case 4: QLAUNCH(4, QT_NF4); break; default: QLAUNCH(8, QT_NF4); break; }
        }
#undef QLAUNCH
        return;
    }
    // RING 2 = one stage less than fits, so the small kernels around a projection can share its SMs (findings r1 §7)
    switch (MT) {
        case 1:
            if (split) launch_k(gemm_kernel<2, 2, true>, dim3(g.grid), dim3(GEMM_THREADS), GemmCfg<2, 2>::SMEM_BYTES, g.p, KC_GEMM, s, prof);
            else launch_k(gemm_kernel<1, 2>, dim3(g.grid), dim3(GEMM_THREADS), GemmCfg<1, 2>::SMEM_BYTES, g.p, KC_GEMM, s, prof);
            break;
        case 2: launch_k(gemm_kernel<2>, dim3(g.grid), dim3(GEMM_THREADS), GemmCfg<2>::SMEM_BYTES, g.p, KC_GEMM, s, prof); break;
        case 4: launch_k(gemm_kernel<4>, dim3(g.grid_wide), dim3(GEMM_THREADS), GemmCfg<4>::SMEM_BYTES, g.p, KC_GEMM, s, prof); break;
        default: launch_k(gemm_kernel<8>, dim3(g.grid_wide), dim3(GEMM_THREADS), GemmCfg<8>::SMEM_BYTES, g.p, KC_GEMM, s, prof); break;
    }
}

// static split-K factor of a row-parallel projection: the S <= 8 / world (partial buffers the LN stages sum) that cuts K
// into whole 128-wide blocks, gives every CTA whole tiles and puts the most SMs to work.  (Measured, round 2: with the
// old cap of 4 the 3B channel-mix value projection ran on 40 CTAs, 22 us for 43 MB; 7 slices -> 140 CTAs.)
int b200rwkv_engine::pick_split(int K, int tiles) const {
    if (dbg_env("B200RWKV_NOSPLIT")) return 1;
    const int kb = K / GEMM_BK;
    if (K % GEMM_BK != 0) return 1;
    int best = 1;
    for (int S = 2; S <= 8 / world; ++S)
        if (kb % S == 0 && tiles * S <= num_sms) best = S;
    return best;
}

// -----------------------------------------------------------------------------------------
// model build
// -----------------------------------------------------------------------------------------
void b200rwkv_engine::build(const StFile& st) {
    info = derive_info(st);
    check_loras(st);
    L = info.num_layer; C = info.num_emb; F = info.num_hidden; V = info.num_vocab; H = info.num_head; N = info.head_size;
    REQUIRE(N == 64, B200RWKV_ERR_UNSUPPORTED, "head_size must be 64");
    REQUIRE(H * N == C, B200RWKV_ERR_UNSUPPORTED, "num_head * head_size must equal num_emb");
    REQUIRE(C % 64 == 0 && C <= 8192, B200RWKV_ERR_UNSUPPORTED, "num_emb must be a multiple of 64 and <= 8192");
    REQUIRE(H % world == 0 && F % (8 * world) == 0 && V % world == 0, B200RWKV_ERR_UNSUPPORTED,
            "heads / hidden / vocab do not shard evenly over the tensor-parallel world");
    Cl = C / world; Hl = H / world; Fl = F / world; Vl = V / world;
    const int ver = info.version;
    const int c0 = rank * Cl, f0 = rank * Fl, v0 = rank * Vl;

    CK(cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&sm_stream, cudaStreamNonBlocking));
    CK(cudaFuncSetAttribute(gemm_kernel<1, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, GemmCfg<1, 2>::SMEM_BYTES));
    CK(cudaFuncSetAttribute(gemm_kernel<2, 2, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, GemmCfg<2, 2>::SMEM_BYTES));
    CK(cudaFuncSetAttribute(gemm_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, GemmCfg<2>::SMEM_BYTES));
    CK(cudaFuncSetAttribute(gemm_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, GemmCfg<4>::SMEM_BYTES));
    CK(cudaFuncSetAttribute(gemm_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, GemmCfg<8>::SMEM_BYTES));
    if (quant_layers > 0 && quant_type != QT_NONE) {
        REQUIRE(quant_type == QT_INT8 || quant_type == QT_NF4, B200RWKV_ERR_UNSUPPORTED, "quant_type must be Int8 or NF4 (SF4 is not implemented)");
        REQUIRE(world == 1, B200RWKV_ERR_UNSUPPORTED, "quantised layers are single-GPU in this version");
        REQUIRE(precision == 0, B200RWKV_ERR_UNSUPPORTED, "quantised layers run with precision 0 (f16 operands)");
#define QATTR(MT_, QT_) CK(cudaFuncSetAttribute(qgemm_kernel<MT_, QT_, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, QGemmCfg<MT_, QT_, true>::SMEM_BYTES))
        QATTR(1, QT_INT8); QATTR(2, QT_INT8); QATTR(4, QT_INT8); QATTR(8, QT_INT8);
        QATTR(1, QT_NF4); QATTR(2, QT_NF4); QATTR(4, QT_NF4); QATTR(8, QT_NF4);
        CK(cudaFuncSetAttribute(qgemm_kernel<1, QT_INT8, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, QGemmCfg<1, QT_INT8, false>::SMEM_BYTES));
        CK(cudaFuncSetAttribute(qgemm_kernel<1, QT_NF4, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, QGemmCfg<1, QT_NF4, false>::SMEM_BYTES));
        if (const char* v = dbg_env("B200RWKV_QTS")) q_ts = atoi(v) != 0;
#undef QATTR
    }
    {   // prefill steps of up to 128 tokens: per-token decay rows of a slot live in dynamic shared memory
        const int wkv_smem_max = 96 * 1024;
        CK(cudaFuncSetAttribute(wkv_kernel<5>, cudaFuncAttributeMaxDynamicSharedMemorySize, wkv_smem_max));
        CK(cudaFuncSetAttribute(wkv_kernel<6>, cudaFuncAttributeMaxDynamicSharedMemorySize, wkv_smem_max));
        CK(cudaFuncSetAttribute(wkv_kernel<7>, cudaFuncAttributeMaxDynamicSharedMemorySize, wkv_smem_max));
        CK(cudaFuncSetAttribute(wkv_kernel<5, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, wkv_smem_max));
        CK(cudaFuncSetAttribute(wkv_kernel<6, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, wkv_smem_max));
        CK(cudaFuncSetAttribute(wkv_kernel<7, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, wkv_smem_max));
    }
    if (precision == 1) split_act = true;         // f32-activation mode (web-rwkv `Bundle::<f32>`): no activation is rounded to f16
    if (const char* v = dbg_env("B200RWKV_PREFETCH_BLOCKS")) prefetch_blocks = std::max(0, atoi(v));
    if (const char* v = dbg_env("B200RWKV_FUSED_PRE")) fused_pre = atoi(v) != 0;
    if (const char* v = dbg_env("B200RWKV_LN_CLUSTER")) ln_cluster = atoi(v) != 0;

    // ---- step metadata ----
    meta_ints = MetaView::ints(maxT, S);
    d_meta = (int*)dalloc(meta_ints * 4);
    CK(cudaMallocHost(&h_meta, meta_ints * 4 * META_RING));
    memset(h_meta, 0, meta_ints * 4 * META_RING);
    for (auto& ev : meta_ev) CK(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    MetaView mv{d_meta, maxT, S};

    // ---- temp upload buffer: largest tensor ----
    for (auto& kv : st.tensors) d_tmp_bytes = std::max(d_tmp_bytes, kv.second.nbytes);
    CK(cudaMalloc(&d_tmp, d_tmp_bytes));

    // ---- state ----
    att_shift = (float*)dalloc((size_t)L * S * C * 4);
    ffn_shift = (float*)dalloc((size_t)L * S * C * 4);
    wkv_state = (float*)dalloc((size_t)L * S * Hl * N * N * 4);
    d_api = (float*)dalloc((size_t)L * (N + 2) * C * 4);
    state_from_st(st, L, H, N, C, init_state);      // State::init() with a state-tuned model; empty otherwise

    // ---- activations ----
    const size_t TC = (size_t)maxT * C, TCl = (size_t)maxT * Cl;
    x_a = (float*)dalloc(TC * 4); x_b = (float*)dalloc(TC * 4);
    xx1 = (float*)dalloc(TC * 4); sx1 = (float*)dalloc(TC * 4); xx2 = (float*)dalloc(TC * 4);
    f_r = (float*)dalloc(TCl * 4); f_k = (float*)dalloc(TCl * 4); f_v = (float*)dalloc(TCl * 4); f_g = (float*)dalloc(TCl * 4);
    f_w = (float*)dalloc(TCl * 4); f_a = (float*)dalloc(TCl * 4); f_nu = (float*)dalloc(TCl * 4); f_vfirst = (float*)dalloc(TCl * 4);
    {
        auto al = [](size_t x) { return (x + 255) & ~(size_t)255; };
        off_part_att = 0;
        off_part_ffn = al(off_part_att + TC * 4 * 8);       // up to 8 split-K slices each
        off_rr = al(off_part_ffn + TC * 4 * 8);
        off_logits = al(off_rr + TCl * 4);
        off_flags = al(off_logits + (size_t)maxT * Vl * 4);
        comm_bytes = al(off_flags + 256);
        comm_base = (uint8_t*)dalloc(comm_bytes, true);
        part_att = (float*)(comm_base + off_part_att);
        part_ffn = (float*)(comm_base + off_part_ffn);
        f_rr = (float*)(comm_base + off_rr);
        d_logits = (float*)(comm_base + off_logits);
        d_epoch = (unsigned*)dalloc(16, true);
        pre_gbar = (unsigned*)dalloc(256, true);
        if (dbg_env("B200RWKV_STEP_TRACE")) {
            d_step_trace = (unsigned long long*)dalloc((size_t)STEP_TRACE_MAX * STEP_TRACE_ROW * 8, true);
            trace_capture = true;
        }
        ln_cluster_ok = ln_cluster && C % (4 * PRE_CLUSTER) == 0 && C / (4 * PRE_CLUSTER) <= PRE_THREADS;
        split_on = split_act && ln_cluster_ok;
        REQUIRE(precision != 1 || split_on, B200RWKV_ERR_UNSUPPORTED, "precision 1 needs num_emb to be a multiple of 32 and <= 8192");
    }
    const int S_att = pick_split(Cl, cdiv(C, GEMM_BN)), S_ffn = pick_split(Fl, cdiv(C, GEMM_BN));
    split_att = S_att; split_ffn = S_ffn;
    d_hidden = (float*)dalloc(TC * 4);
    CK(cudaEventCreateWithFlags(&step_done, cudaEventDisableTiming));
    keep_valid.assign(S, 0);
    if (rank == 0) {
        d_keep = (float*)dalloc((size_t)S * V * 4);
        const int nseg = cdiv(V, TOPK_SEG);
        if (nseg <= TOPK_MAX_SEGS) {       // larger vocabularies: b200rwkv_sample_topk answers UNSUPPORTED
            tk_cand_x = (float*)dalloc((size_t)S * nseg * TOPK_MAX * 4);
            tk_cand_id = (unsigned*)dalloc((size_t)S * nseg * TOPK_MAX * 4);
            tk_stats = (float2*)dalloc((size_t)S * nseg * 8);
            tk_out_id = (unsigned*)dalloc((size_t)S * TOPK_MAX * 4);
            tk_out_p = (float*)dalloc((size_t)S * TOPK_MAX * 4);
        }
    }
    for (int i = 0; i < 6; ++i) a_x[i] = a16_alloc(C);
    a_out = a16_alloc(Cl);
    a_kk = a16_alloc(Fl);
    a_head = a16_alloc(C);

    // ---- embedding + ln0 ----
    {
        const StTensor& e = st.get("emb.weight");
        emb = (__half*)dalloc(e.nbytes, false);
        CK(cudaMemcpy(emb, e.data, e.nbytes, cudaMemcpyHostToDevice));
        embed.emb = emb; embed.C = C; embed.V = V; embed.meta = mv;
        embed.ln_w = vec_f32(st, "blocks.0.ln0.weight", 0, C);
        embed.ln_b = vec_f32(st, "blocks.0.ln0.bias", 0, C);
        embed.x_out = x_a;
    }

    auto base_ln = [&](LnMixParams& p) {
        memset(&p, 0, sizeof(p));
        p.C = C; p.meta = mv; p.kq_tile = C / 32;
    };
    auto f32_seg = [&](const StTensor& t, int n0, int Nn, int k0, int K, const A16Buf& ab, float* out, int ldo, int act,
                       const float* bias, int a_koff = 0, int a_mat = 0) {
        SegDesc d;
        d.t = &t; d.n0 = n0; d.N = Nn; d.k0 = k0; d.K = K;
        REQUIRE(a_koff % GEMM_BK == 0, B200RWKV_ERR_INVALID, "internal: split-K slices start on k-block boundaries");
        d.proto.A = ab.p + (size_t)a_mat * ab.halves_per_matrix + (size_t)(a_koff / GEMM_BK) * A16_KB_HALVES; d.proto.a_k8 = ab.kq * 4;
        d.proto.out_mode = OUT_F32; d.proto.act = act; d.proto.bias = bias; d.proto.out = out; d.proto.ldo = ldo;
        return d;
    };
    auto a16_seg = [&](const StTensor& t, int n0, int Nn, int k0, int K, const A16Buf& ab, const A16Buf& dst, int act,
                       const float* bias) {
        SegDesc d;
        d.t = &t; d.n0 = n0; d.N = Nn; d.k0 = k0; d.K = K;
        d.proto.A = ab.p; d.proto.a_k8 = ab.kq * 4;
        d.proto.out_mode = OUT_A16; d.proto.act = act; d.proto.bias = bias; d.proto.out = dst.p; d.proto.ldo = dst.kq;
        return d;
    };

    layers.resize(L);
    for (int l = 0; l < L; ++l) {
        Layer& ly = layers[l];
        const std::string b = "blocks." + std::to_string(l) + ".";
        const std::string a = b + "att.", f = b + "ffn.";
        float* att_sh = att_shift + (size_t)l * S * C;
        float* ffn_sh = ffn_shift + (size_t)l * S * C;
        // `quant`: the eight projection matrices of the first layers are quantised, adapters / LoRA matrices stay f16 -- so a
        // launch that mixed both kinds (R/K/V/G + decay LoRA, v7 R/K/V + adapters) goes out as two in those layers
        const int lq = (l < quant_layers) ? quant_type : QT_NONE;

        // ---------------- LN1 (+ residual update from the previous layer's channel mix) ----------------
        LnMixParams& n1 = ly.ln1;
        base_ln(n1);
        n1.x_in = (l == 0) ? x_a : x_b;
        n1.x_out = x_a;
        if (l > 0) {
            n1.n_parts = S_ffn;
            for (int sp = 0; sp < S_ffn; ++sp) n1.parts[sp] = part_ffn + (size_t)sp * TC;
            if (ver != 7) { n1.n_gate = 1; n1.gate_cl = Cl; n1.gates[0] = f_rr; }
            n1.commit_dst = ffn_shift + (size_t)(l - 1) * S * C;
            n1.commit_src = xx2;
        }
        n1.ln_w = vec_f32(st, b + "ln1.weight", 0, C);
        n1.ln_b = vec_f32(st, b + "ln1.bias", 0, C);
        n1.shift_state = att_sh;
        n1.xx_out = xx1;

        WkvParams& wk = ly.wkv;
        memset(&wk, 0, sizeof(wk));
        wk.version = ver; wk.ld = Cl; wk.meta = mv; wk.H = Hl;
        wk.state = wkv_state + (size_t)l * S * Hl * N * N;
        wk.r = f_r; wk.k = f_k; wk.v = f_v; wk.g = f_g;
        wk.lnx_w = vec_f32(st, a + "ln_x.weight", c0, Cl);
        wk.lnx_b = vec_f32(st, a + "ln_x.bias", c0, Cl);
        wk.out = a_out.p; wk.kq_tile = a_out.kq;

        const StTensor& Wr = st.get(a + "receptance.weight");
        const StTensor& Wk = st.get(a + "key.weight");
        const StTensor& Wv = st.get(a + "value.weight");
        const StTensor& Wo = st.get(a + "output.weight");

        if (ver == 6) {
            const int Dm = info.time_mix_adapter, Dd = info.time_decay_adapter;
            if (l == 0) {
                a_lora[0] = a16_alloc(Dm, 5);   // tanh(W1 xxx), five groups
                a_lora[1] = a16_alloc(Dd);      // tanh(Wd1 xw)
            }
            n1.n_mix = 1;
            n1.mu[0] = vec_f32(st, a + "time_mix_x", 0, C);
            n1.mix_out[0] = a_x[5].p;           // xxx
            n1.sx_out = sx1;
            // W1: [5*Dm, C]
            {
                std::vector<SegDesc> sv;
                SegDesc d = a16_seg(st.get(a + "time_mix_w1"), 0, 5 * Dm, 0, C, a_x[5], a_lora[0], ACT_TANH, nullptr);
                d.proto.grp = Dm;
                d.proto.grp_stride = (int)a_lora[0].halves_per_matrix;
                sv.push_back(d);
                ly.pre.push_back(make_launch(sv));
            }
            // W2: [5, C, Dm]; order w,k,v,r,g (SURVEY.md App. A)
            {
                static const char* names[5] = {"time_mix_w", "time_mix_k", "time_mix_v", "time_mix_r", "time_mix_g"};
                std::vector<SegDesc> sv;
                for (int i = 0; i < 5; ++i) {
                    SegDesc d;
                    d.t = &st.get(a + "time_mix_w2"); d.slice = i; d.n0 = 0; d.N = C; d.k0 = 0; d.K = Dm;
                    d.proto.A = a_lora[0].p + (size_t)i * a_lora[0].halves_per_matrix;
                    d.proto.a_k8 = a_lora[0].kq * 4;
                    d.proto.out_mode = OUT_LERP_A16; d.proto.act = ACT_NONE;
                    d.proto.out = a_x[i].p; d.proto.ldo = a_x[i].kq;
                    d.proto.aux0 = xx1; d.proto.aux1 = sx1; d.proto.aux2 = vec_f32(st, a + names[i], 0, C); d.proto.ld_aux = C;
                    sv.push_back(d);
                }
                ly.pre.push_back(make_launch(sv));
            }
            {   // the raw copies below are indexed with these exact shapes
                const StTensor& w1 = st.get(a + "time_mix_w1");
                const StTensor& w2 = st.get(a + "time_mix_w2");
                const StTensor& d2 = st.get(a + "time_decay_w2");
                REQUIRE(w1.shape.size() == 2 && w1.shape[0] == 5 * Dm && w1.shape[1] == C, B200RWKV_ERR_INVALID, "time_mix_w1 must be [5*Dm, C]");
                REQUIRE(w2.shape.size() == 3 && w2.shape[0] == 5 && w2.shape[1] == C && w2.shape[2] == Dm, B200RWKV_ERR_INVALID,
                        "time_mix_w2 must be [5, C, Dm]");
                REQUIRE(d2.shape.size() == 2 && d2.shape[0] == C && d2.shape[1] == Dd, B200RWKV_ERR_INVALID, "time_decay_w2 must be [C, Dd]");
            }
            if (fused_pre && (Dm == 32 || Dm == 64) && C % 128 == 0 && C <= PRE_MAX_C) {
                auto upload_raw = [&](const StTensor& t) {
                    __half* d = (__half*)dalloc(t.nbytes, false);
                    CK(cudaMemcpy(d, t.data, t.nbytes, cudaMemcpyHostToDevice));
                    return d;
                };
                ly.w1_raw = upload_raw(st.get(a + "time_mix_w1"));
                ly.w2_raw = upload_raw(st.get(a + "time_mix_w2"));
                for (int i = 0; i < 5; ++i) ly.mu5[i] = ly.pre[1].p.seg[i].aux2;
                fused_pre_ok = true;
            }
            // R,K,V,G (column parallel by head) + decay LoRA stage 1 (replicated)
            {
                std::vector<SegDesc> sv;
                sv.push_back(f32_seg(Wr, c0, Cl, 0, C, a_x[3], f_r, Cl, ACT_NONE, nullptr));
                sv.push_back(f32_seg(Wk, c0, Cl, 0, C, a_x[1], f_k, Cl, ACT_NONE, nullptr));
                sv.push_back(f32_seg(Wv, c0, Cl, 0, C, a_x[2], f_v, Cl, ACT_NONE, nullptr));
                sv.push_back(f32_seg(st.get(a + "gate.weight"), c0, Cl, 0, C, a_x[4], f_g, Cl, ACT_SILU, nullptr));
                if (lq != QT_NONE) {
                    // the small f16 launch goes first: it occupies a handful of SMs, and behind it the quantised launch is
                    // already resident on the others filling its ring (programmatic dependent launch)
                    std::vector<SegDesc> sd;
                    sd.push_back(a16_seg(st.get(a + "time_decay_w1"), 0, Dd, 0, C, a_x[0], a_lora[1], ACT_TANH, nullptr));
                    ly.pre.push_back(make_launch(sd));
                    ly.pre.push_back(make_launch(sv, 0, lq));
                } else {
                    sv.push_back(a16_seg(st.get(a + "time_decay_w1"), 0, Dd, 0, C, a_x[0], a_lora[1], ACT_TANH, nullptr));
                    ly.pre.push_back(make_launch(sv));
                }
            }
            // decay LoRA stage 2: w = exp(-exp(time_decay + Wd2 d))
            {
                std::vector<SegDesc> sv;
                sv.push_back(f32_seg(st.get(a + "time_decay_w2"), c0, Cl, 0, Dd, a_lora[1], f_w, Cl, ACT_EXPNEGEXP,
                                     vec_f32(st, a + "time_decay", c0, Cl)));
                ly.wd2_index = (int)ly.pre.size();
                ly.pre.push_back(make_launch(sv));
            }
            if (Dd <= 128 && Dd % 8 == 0 && !dbg_env("B200RWKV_NOFOLD")) {
                // k-major copy of this rank's time_decay_w2 rows, one contiguous [Dd][64] slice per head: the WKV
                // kernels evaluate the decay LoRA stage 2 themselves (one launch / phase less per layer)
                const StTensor& t = st.get(a + "time_decay_w2");
                const __half* src = reinterpret_cast<const __half*>(t.data);
                std::vector<__half> tmp((size_t)Hl * Dd * 64);
                for (int h = 0; h < Hl; ++h)
                    for (int k = 0; k < Dd; ++k)
                        for (int c = 0; c < 64; ++c) tmp[((size_t)h * Dd + k) * 64 + c] = src[(size_t)(c0 + h * 64 + c) * Dd + k];
                __half* dw = (__half*)dalloc(tmp.size() * 2, false);
                CK(cudaMemcpy(dw, tmp.data(), tmp.size() * 2, cudaMemcpyHostToDevice));
                wk.wd2t = dw;
                wk.decay_bias = ly.pre[ly.wd2_index].p.seg[0].bias;
                wk.d1 = a_lora[1].p;
                wk.d1_kq = a_lora[1].kq;
                wk.Dd = Dd;
                fold_wd2 = true;
            }
            wk.w = f_w;
            wk.u = vec_f32(st, a + "time_first", c0, Cl);
        } else if (ver == 5) {
            // x_* = xx*mix + prev*(1-mix) == xx + (prev-xx)*(1-mix)
            static const char* names[4] = {"time_mix_k", "time_mix_v", "time_mix_r", "time_mix_g"};
            n1.n_mix = 4;
            for (int i = 0; i < 4; ++i) {
                n1.mu[i] = vec_f32(st, a + names[i], 0, C, -1.f, 1.f);
                n1.mix_out[i] = a_x[1 + i].p;     // k,v,r,g -> a_x[1..4]
            }
            std::vector<SegDesc> sv;
            sv.push_back(f32_seg(Wr, c0, Cl, 0, C, a_x[3], f_r, Cl, ACT_NONE, nullptr));
            sv.push_back(f32_seg(Wk, c0, Cl, 0, C, a_x[1], f_k, Cl, ACT_NONE, nullptr));
            sv.push_back(f32_seg(Wv, c0, Cl, 0, C, a_x[2], f_v, Cl, ACT_NONE, nullptr));
            sv.push_back(f32_seg(st.get(a + "gate.weight"), c0, Cl, 0, C, a_x[4], f_g, Cl, ACT_SILU, nullptr));
            ly.pre.push_back(make_launch(sv, 0, lq));
            {
                const StTensor& td = st.get(a + "time_decay");
                REQUIRE(td.numel() == C, B200RWKV_ERR_UNSUPPORTED, "v5 time_decay must be [H, N]");
                float* d = (float*)dalloc((size_t)Cl * 4, false);
                DevTmp tmp((size_t)Cl * 2);
                CK(cudaMemcpy(tmp.p, td.data + (size_t)c0 * 2, (size_t)Cl * 2, cudaMemcpyHostToDevice));
                decay_table_kernel<<<cdiv(Cl, 256), 256>>>((const __half*)tmp.p, d, Cl);
                CK(cudaDeviceSynchronize());
                wk.w_static = d;
            }
            wk.u = vec_f32(st, a + "time_first", c0, Cl);
        } else {
            // v7: six static lerps r,w,k,v,a,g -> a_x[0..5]
            static const char* names[6] = {"x_r", "x_w", "x_k", "x_v", "x_a", "x_g"};
            const int Dw = (int)st.dim(a + "w1", 0, 2), Da = (int)st.dim(a + "a1", 0, 2), Dg = (int)st.dim(a + "g1", 0, 2);
            const std::string v1n = L > 1 ? "blocks.1.att.v1" : "blocks.0.att.v1";
            const int Dv = st.find(v1n) ? (int)st.dim(v1n, 0, 2) : 32;
            if (l == 0) {
                a_lora[0] = a16_alloc(Dw); a_lora[1] = a16_alloc(Da); a_lora[2] = a16_alloc(Dv); a_lora[3] = a16_alloc(Dg);
            }
            n1.n_mix = 6;
            for (int i = 0; i < 6; ++i) {
                n1.mu[i] = vec_f32(st, a + names[i], 0, C);
                n1.mix_out[i] = a_x[i].p;
            }
            {
                std::vector<SegDesc> sv;
                sv.push_back(f32_seg(Wr, c0, Cl, 0, C, a_x[0], f_r, Cl, ACT_NONE, nullptr));
                sv.push_back(f32_seg(Wk, c0, Cl, 0, C, a_x[2], f_k, Cl, ACT_NONE, nullptr));
                sv.push_back(f32_seg(Wv, c0, Cl, 0, C, a_x[3], f_v, Cl, ACT_NONE, nullptr));
                std::vector<SegDesc> sq;
                if (lq != QT_NONE) sq.swap(sv);          // quantised R/K/V go out as their own launch, after the f16 adapters
                sv.push_back(a16_seg(st.get(a + "w1"), 0, Dw, 0, C, a_x[1], a_lora[0], ACT_TANH, nullptr));
                sv.push_back(a16_seg(st.get(a + "a1"), 0, Da, 0, C, a_x[4], a_lora[1], ACT_NONE, nullptr));
                if (l > 0) sv.push_back(a16_seg(st.get(a + "v1"), 0, Dv, 0, C, a_x[3], a_lora[2], ACT_NONE, nullptr));
                sv.push_back(a16_seg(st.get(a + "g1"), 0, Dg, 0, C, a_x[5], a_lora[3], ACT_SIGMOID, nullptr));
                ly.pre.push_back(make_launch(sv));
                if (lq != QT_NONE) ly.pre.push_back(make_launch(sq, 0, lq));
            }
            {
                std::vector<SegDesc> sv;
                sv.push_back(f32_seg(st.get(a + "w2"), c0, Cl, 0, Dw, a_lora[0], f_w, Cl, ACT_V7DECAY, vec_f32(st, a + "w0", c0, Cl)));
                sv.push_back(f32_seg(st.get(a + "a2"), c0, Cl, 0, Da, a_lora[1], f_a, Cl, ACT_SIGMOID, vec_f32(st, a + "a0", c0, Cl)));
                if (l > 0)
                    sv.push_back(f32_seg(st.get(a + "v2"), c0, Cl, 0, Dv, a_lora[2], f_nu, Cl, ACT_SIGMOID, vec_f32(st, a + "v0", c0, Cl)));
                sv.push_back(f32_seg(st.get(a + "g2"), c0, Cl, 0, Dg, a_lora[3], f_g, Cl, ACT_NONE, nullptr));
                ly.pre.push_back(make_launch(sv));
            }
            wk.w = f_w; wk.a = f_a; wk.nu = f_nu; wk.v_first = f_vfirst; wk.layer0 = (l == 0);
            wk.k_k = vec_f32(st, a + "k_k", c0, Cl);
            wk.k_a = vec_f32(st, a + "k_a", c0, Cl);
            wk.r_k = vec_f32(st, a + "r_k", c0, Cl);
        }

        // ---------------- output projection (row parallel) -> partial ----------------
        {
            // row-parallel: K is cut into `S_att` static slices, one partial buffer each (summed by the
            // next LN stage in fixed order); with tiles * S CTAs every CTA owns whole tiles: no fix-up
            std::vector<SegDesc> sv;
            for (int sp = 0; sp < S_att; ++sp)
                sv.push_back(f32_seg(Wo, 0, C, c0 + sp * (Cl / S_att), Cl / S_att, a_out, part_att + (size_t)sp * TC, C, ACT_NONE,
                                     nullptr, sp * (Cl / S_att)));
            ly.o = make_launch(sv, S_att > 1 ? cdiv(C, GEMM_BN) * S_att : 0, lq);
        }

        // ---------------- LN2 ----------------
        LnMixParams& n2 = ly.ln2;
        base_ln(n2);
        n2.x_in = x_a; n2.x_out = x_b;
        n2.n_parts = S_att;
        for (int sp = 0; sp < S_att; ++sp) n2.parts[sp] = part_att + (size_t)sp * TC;
        n2.ln_w = vec_f32(st, b + "ln2.weight", 0, C);
        n2.ln_b = vec_f32(st, b + "ln2.bias", 0, C);
        n2.shift_state = ffn_sh;
        n2.xx_out = xx2;
        n2.commit_dst = att_sh; n2.commit_src = xx1;
        const StTensor& Fk = st.get(f + "key.weight");
        const StTensor& Fv = st.get(f + "value.weight");
        if (ver == 7) {
            n2.n_mix = 1;
            n2.mu[0] = vec_f32(st, f + "x_k", 0, C);
            n2.mix_out[0] = a_x[0].p;
            std::vector<SegDesc> sv;
            sv.push_back(a16_seg(Fk, f0, Fl, 0, C, a_x[0], a_kk, ACT_RELU2, nullptr));
            ly.ffn.push_back(make_launch(sv, 0, lq));
        } else {
            n2.n_mix = 2;
            if (ver == 6) {
                n2.mu[0] = vec_f32(st, f + "time_mix_k", 0, C);
                n2.mu[1] = vec_f32(st, f + "time_mix_r", 0, C);
            } else {
                n2.mu[0] = vec_f32(st, f + "time_mix_k", 0, C, -1.f, 1.f);
                n2.mu[1] = vec_f32(st, f + "time_mix_r", 0, C, -1.f, 1.f);
            }
            n2.mix_out[0] = a_x[0].p;
            n2.mix_out[1] = a_x[1].p;
            std::vector<SegDesc> sv;
            sv.push_back(a16_seg(Fk, f0, Fl, 0, C, a_x[0], a_kk, ACT_RELU2, nullptr));
            sv.push_back(f32_seg(st.get(f + "receptance.weight"), c0, Cl, 0, C, a_x[1], f_rr, Cl, ACT_SIGMOID, nullptr));
            ly.ffn.push_back(make_launch(sv, 0, lq));
        }
        {
            std::vector<SegDesc> sv;
            for (int sp = 0; sp < S_ffn; ++sp)
                sv.push_back(f32_seg(Fv, 0, C, f0 + sp * (Fl / S_ffn), Fl / S_ffn, a_kk, part_ffn + (size_t)sp * TC, C, ACT_NONE,
                                     nullptr, sp * (Fl / S_ffn)));
            ly.ffn.push_back(make_launch(sv, S_ffn > 1 ? cdiv(C, GEMM_BN) * S_ffn : 0, lq));
        }
    }

    // ---------------- ln_out + head ----------------
    memset(&lnout, 0, sizeof(lnout));
    lnout.x_in = x_b; lnout.C = C; lnout.meta = mv;
    lnout.n_parts = S_ffn;
    for (int sp = 0; sp < S_ffn; ++sp) lnout.parts[sp] = part_ffn + (size_t)sp * TC;
    if (ver != 7) { lnout.n_gate = 1; lnout.gate_cl = Cl; lnout.gates[0] = f_rr; }
    lnout.ln_w = vec_f32(st, "ln_out.weight", 0, C);
    lnout.ln_b = vec_f32(st, "ln_out.bias", 0, C);
    lnout.head_in = a_head.p; lnout.kq_tile = a_head.kq;
    lnout.commit_dst = ffn_shift + (size_t)(L - 1) * S * C;
    lnout.commit_src = xx2;
    lnout.hidden_out = d_hidden;
    {
        std::vector<SegDesc> sv;
        sv.push_back(f32_seg(st.get("head.weight"), v0, Vl, 0, C, a_head, d_logits, Vl, ACT_NONE, nullptr));
        head = make_launch(sv);
        head.p.nrows = d_meta + 2;    // R
    }

    gemm_ws = (float*)dalloc(gemm_ws_floats * 4, false);
    for (auto& ly : layers) {
        for (auto& g : ly.pre) g.p.ws = gemm_ws;
        ly.o.p.ws = gemm_ws;
        for (auto& g : ly.ffn) g.p.ws = gemm_ws;
    }
    head.p.ws = gemm_ws;

    if (world == 1) {
        peer_base[0] = comm_base;
        finalize_tp();
    }
    CK(cudaDeviceSynchronize());
    CK(cudaFree(d_tmp));
    d_tmp = nullptr;
}

// -----------------------------------------------------------------------------------------
// Tensor parallel wiring: every LN stage sums the partial projections of ALL ranks (rank-major,
// then split-K slice: the same fixed order on every rank, so the replicated residual stream stays
// bit-identical across ranks) straight out of the peers' comm blocks, and takes the channel-mix
// gate block-wise from the rank that owns those columns.
// -----------------------------------------------------------------------------------------
void b200rwkv_engine::finalize_tp() {
    const size_t TC = (size_t)maxT * C;
    const int ver = info.version;
    auto parts_of = [&](size_t off, int S, const float** dst) {
        int n = 0;
        for (int q = 0; q < world; ++q)
            for (int sp = 0; sp < S; ++sp) dst[n++] = (const float*)(peer_base[q] + off) + (size_t)sp * TC;
        return n;
    };
    auto gates_of = [&](const float** dst) {
        for (int q = 0; q < world; ++q) dst[q] = (const float*)(peer_base[q] + off_rr);
    };
    for (int l = 0; l < L; ++l) {
        Layer& ly = layers[l];
        if (l > 0) {
            ly.ln1.n_parts = parts_of(off_part_ffn, split_ffn, ly.ln1.parts);
            if (ver != 7) { ly.ln1.n_gate = world; ly.ln1.gate_cl = Cl; gates_of(ly.ln1.gates); }
        }
        ly.ln2.n_parts = parts_of(off_part_att, split_att, ly.ln2.parts);
    }
    lnout.n_parts = parts_of(off_part_ffn, split_ffn, lnout.parts);
    if (ver != 7) { lnout.n_gate = world; lnout.gate_cl = Cl; gates_of(lnout.gates); }
    memset(&tpbar, 0, sizeof(tpbar));
    for (int q = 0; q < world; ++q) tpbar.flags[q] = (unsigned*)(peer_base[q] + off_flags);
    tpbar.epoch = d_epoch;
    tpbar.rank = rank;
    tpbar.world = world;
    connected = true;
}

// -----------------------------------------------------------------------------------------
// one forward step over the tokens described by d_meta
// -----------------------------------------------------------------------------------------
bool b200rwkv_engine::pre_skipped(const Layer& ly, int gi, int MT) const {
    if (fold_wd2 && gi == ly.wd2_index) return true;                 // the WKV kernel evaluates the decay LoRA stage 2
    return fused_pre_ok && MT == 1 && ly.w1_raw && gi < 2;           // the front-half kernel holds both ddlerp LoRA stages
}

void b200rwkv_engine::enqueue_step(cudaStream_t s, int MT, int MTR, Profiler* prof) {
    launches_last_step = 0;
    const int rows = MT * 16;
    // token rows of this step's A16 operands (common.cuh): every producer and consumer of the step uses the same value
    const int th = (split_on && MT == 1) ? 32 : 16 * MT;
    const int th_rows = (split_on && MT == 1) ? 32 : 16 * MTR;        // the head's operand holds output rows
    // projection launches of this step in stream order: each one prefetches the head of the next into L2 (the last one
    // wraps around to the first launch of the next step)
    std::vector<const GemmLaunch*> seq;
    if (prefetch_blocks > 0) {
        for (int l = 0; l < L; ++l) {
            const Layer& ly = layers[l];
            for (int gi = 0; gi < (int)ly.pre.size(); ++gi)
                if (!pre_skipped(ly, gi, MT)) seq.push_back(&ly.pre[gi]);
            seq.push_back(&ly.o);
            for (auto& g : ly.ffn) seq.push_back(&g);
        }
        if (MTR > 0) seq.push_back(&head);
    }
    size_t seq_pos = 0;
    auto launch_gemm_chained = [&](const GemmLaunch& g, int mt) {
        GemmLaunch g2 = g;
        if (d_step_trace && trace_capture) {
            g2.p.trace = tr_next(1000000 + (int)(g.weight_bytes >> 20));
            if ((long long)step_trace_bytes.size() <= launches_last_step) step_trace_bytes.resize(launches_last_step + 1, 0);
            step_trace_bytes[launches_last_step] = (long long)g.weight_bytes;
        }
        if (!seq.empty()) {
            REQUIRE(seq_pos < seq.size() && seq[seq_pos] == &g, B200RWKV_ERR_INVALID, "internal: projection launch order");
            const GemmLaunch& nx = *seq[(seq_pos + 1) % seq.size()];
            ++seq_pos;
            g2.p.next_W = nx.qtype == QT_NONE ? nx.p.W : nullptr;     // the L2 prefetch walks 32 KB f16 blocks
            g2.p.next_blocks = nx.p.total_blocks;
            g2.p.next_grid = mt >= 4 ? nx.grid_wide : nx.grid;
            g2.p.prefetch_blocks = prefetch_blocks;
        }
        for (int i = 0; i < g2.p.nseg; ++i)
            if (g2.p.seg[i].out_mode != OUT_F32) g2.p.seg[i].ldo = th;      // A16 outputs feed a projection of this step
        launch_gemm(g2, mt, s, prof, split_on && MT == 1);      // split operands only when the whole step is decode-shaped
    };
    auto gemm = [&](const GemmLaunch& g) { launch_gemm_chained(g, MT); };
    launch_k(embed_ln0_kernel, dim3(rows), dim3(LN_THREADS), 0, embed, KC_LN, s, prof);
    auto launch_ln = [&](const LnMixParams& lp0) {
        LnMixParams lp = lp0;
        lp.trace = tr_next(0);
        lp.kq_tile = th;
        if (ln_cluster_ok && MT == 1) {
            launch_cluster = PRE_CLUSTER;
            if (split_on) launch_k(ln_mix_cluster_kernel<true>, dim3(PRE_GRID), dim3(PRE_THREADS), 0, lp, KC_LN, s, prof);
            else launch_k(ln_mix_cluster_kernel<false>, dim3(PRE_GRID), dim3(PRE_THREADS), 0, lp, KC_LN, s, prof);
        } else {
            launch_k(ln_mix_kernel, dim3(rows), dim3(LN_THREADS), 0, lp, KC_LN, s, prof);
        }
    };
    const int wkv_slots = std::min(S, rows);
    for (int l = 0; l < L; ++l) {
        Layer& ly = layers[l];
        const bool fused = fused_pre_ok && MT == 1 && ly.w1_raw;
        if (fused) {
            // LN1 + token shift + ddlerp LoRA (W1, tanh, W2, lerps) in one launch
            Pre6Params q;
            memset(&q, 0, sizeof(q));
            q.ln = ly.ln1;
            q.ln.trace = tr_next(6);
            q.ln.kq_tile = th;
            q.W1 = ly.w1_raw; q.W2 = ly.w2_raw;
            for (int j = 0; j < 5; ++j) { q.mu[j] = ly.mu5[j]; q.out[j] = a_x[j].p; }
            q.lora = a_lora[0].p; q.lora_stride = (int)a_lora[0].halves_per_matrix; q.lora_kq = a_lora[0].kq;
            q.Dm = info.time_mix_adapter;
            q.gbar = pre_gbar;
            launch_cluster = PRE_CLUSTER;
            if (split_on) {
                if (q.Dm == 32) launch_k(pre6_kernel<2, true>, dim3(PRE_GRID), dim3(PRE_THREADS), 0, q, KC_LN, s, prof);
                else launch_k(pre6_kernel<4, true>, dim3(PRE_GRID), dim3(PRE_THREADS), 0, q, KC_LN, s, prof);
            } else {
                if (q.Dm == 32) launch_k(pre6_kernel<2, false>, dim3(PRE_GRID), dim3(PRE_THREADS), 0, q, KC_LN, s, prof);
                else launch_k(pre6_kernel<4, false>, dim3(PRE_GRID), dim3(PRE_THREADS), 0, q, KC_LN, s, prof);
            }
        } else {
            launch_ln(ly.ln1);
        }
        for (int gi = 0; gi < (int)ly.pre.size(); ++gi)
            if (!pre_skipped(ly, gi, MT)) gemm(ly.pre[gi]);
        {
            // decays / staged rows are sized by the step shape: a slot cannot hold more tokens than the step
            WkvParams wp = ly.wkv;
            wp.trace = tr_next(2);
            wp.kq_tile = th; wp.d1_kq = th;
            const bool sp = split_on && MT == 1;
            const size_t sm_b = wkv_smem_bytes(info.version, fold_wd2, info.time_decay_adapter, rows, sp);
            switch (info.version * 2 + (sp ? 1 : 0)) {
                case 10: launch_k(wkv_kernel<5>, dim3(Hl, wkv_slots), dim3(WKV_SA_THREADS), sm_b, wp, KC_WKV, s, prof, rows); break;
                case 11: launch_k(wkv_kernel<5, true>, dim3(Hl, wkv_slots), dim3(WKV_SA_THREADS), sm_b, wp, KC_WKV, s, prof, rows); break;
                case 12: launch_k(wkv_kernel<6>, dim3(Hl, wkv_slots), dim3(WKV_SA_THREADS), sm_b, wp, KC_WKV, s, prof, rows); break;
                case 13: launch_k(wkv_kernel<6, true>, dim3(Hl, wkv_slots), dim3(WKV_SA_THREADS), sm_b, wp, KC_WKV, s, prof, rows); break;
                case 14: launch_k(wkv_kernel<7>, dim3(Hl, wkv_slots), dim3(WKV_SA_THREADS), sm_b, wp, KC_WKV, s, prof, rows); break;
                default: launch_k(wkv_kernel<7, true>, dim3(Hl, wkv_slots), dim3(WKV_SA_THREADS), sm_b, wp, KC_WKV, s, prof, rows); break;
            }
        }
        gemm(ly.o);
        if (world > 1) launch_k(tp_barrier_kernel, dim3(1), dim3(32), 0, tpbar, KC_OTHER, s, prof);
        launch_ln(ly.ln2);
        for (auto& g : ly.ffn) gemm(g);
        if (world > 1) launch_k(tp_barrier_kernel, dim3(1), dim3(32), 0, tpbar, KC_OTHER, s, prof);
    }
    {
        LnOutParams lo = lnout;
        lo.kq_tile = th_rows;
        if (split_on && MT == 1) launch_k(ln_out_kernel<true>, dim3(rows), dim3(LN_THREADS), 0, lo, KC_LN, s, prof);
        else launch_k(ln_out_kernel<false>, dim3(rows), dim3(LN_THREADS), 0, lo, KC_LN, s, prof);
    }
    if (MTR > 0) launch_gemm_chained(head, MTR);
    if (world > 1) launch_k(tp_barrier_kernel, dim3(1), dim3(32), 0, tpbar, KC_OTHER, s, prof);
}

static inline int mt_bucket(int rows) { return rows <= 16 ? 1 : (rows <= 32 ? 2 : (rows <= 64 ? 4 : 8)); }

// last logits row of every slot of this step -> keep[slot] (rank 0 gathers the vocabulary shards); see sample.cuh
void b200rwkv_engine::enqueue_keep(cudaStream_t s, int MTR) {
    if (MTR <= 0 || rank != 0 || !d_keep || Vl % 4 != 0) return;
    KeepParams kp;
    memset(&kp, 0, sizeof(kp));
    for (int q = 0; q < world; ++q) kp.shard[q] = (const float*)(peer_base[q] + off_logits);
    kp.world = world; kp.Vl = Vl; kp.V = V;
    kp.meta = MetaView{d_meta, maxT, S};
    kp.keep = d_keep;
    launch_k(keep_rows_kernel, dim3(MTR * 16, KEEP_CHUNKS), dim3(KEEP_THREADS), 0, kp, KC_OTHER, s, nullptr);
}

void b200rwkv_engine::run_step(int MT, int MTR) {
    // recorded here, not in enqueue_step: a replayed graph does not enqueue again (same formulas as enqueue_step)
    last_split = split_on && MT == 1;
    last_th = last_split ? 32 : 16 * MT;
    last_th_rows = last_split ? 32 : 16 * MTR;
    if (!use_graph) {
        enqueue_step(stream, MT, MTR, nullptr);
        enqueue_keep(stream, MTR);
        launch_total += launches_last_step;
        return;
    }
    const int key = MT * 8 + MTR;
    auto it = graphs.find(key);
    if (it == graphs.end()) {
        cudaGraph_t g = nullptr;
        CK(cudaStreamBeginCapture(stream, cudaStreamCaptureModeThreadLocal));
        try {
            enqueue_step(stream, MT, MTR, nullptr);
            enqueue_keep(stream, MTR);
        } catch (...) {
            cudaStreamEndCapture(stream, &g);
            if (g) cudaGraphDestroy(g);
            throw;
        }
        CK(cudaStreamEndCapture(stream, &g));
        cudaGraphExec_t ge = nullptr;
        CK(cudaGraphInstantiate(&ge, g, 0));
        CK(cudaGraphDestroy(g));
        it = graphs.emplace(key, ge).first;
        graph_launches[key] = launches_last_step;
    }
    CK(cudaGraphLaunch(it->second, stream));
    launch_total += graph_launches[key];         // kernels of THIS graph, not of whichever was captured last
}

// fills one step's metadata; returns T
int b200rwkv_engine::fill_meta(int* m, const std::vector<int>& slots, const std::vector<int>& counts,
                               const std::vector<const uint32_t*>& toks, const std::vector<int>& outmode, int* R_out) {
    MetaView mv{m, maxT, S};
    int* tok = const_cast<int*>(mv.tok());
    int* tslot = const_cast<int*>(mv.tok_slot());
    int* tprev = const_cast<int*>(mv.tok_prev());
    int* tlast = const_cast<int*>(mv.tok_last());
    int* otok = const_cast<int*>(mv.out_tok());
    int* torow = const_cast<int*>(mv.tok_outrow());
    int* sid = const_cast<int*>(mv.slot_id());
    int* sstart = const_cast<int*>(mv.slot_start());
    int* scount = const_cast<int*>(mv.slot_count());
    int T = 0, R = 0;
    for (size_t i = 0; i < slots.size(); ++i) {
        sid[i] = slots[i];
        sstart[i] = T;
        scount[i] = counts[i];
        for (int j = 0; j < counts[i]; ++j, ++T) {
            tok[T] = (int)toks[i][j];
            tslot[T] = slots[i];
            tprev[T] = (j == 0) ? -1 : T - 1;
            tlast[T] = (j == counts[i] - 1) ? 1 : 0;
            const bool out = (outmode[i] == 2) || (outmode[i] == 1 && j == counts[i] - 1);
            torow[T] = out ? R : -1;
            if (out) otok[R++] = T;
        }
    }
    m[0] = T; m[1] = (int)slots.size(); m[2] = R;
    m[4] = (int)++step_seq;   // identical on every rank (SPMD): epoch base of the folded rendezvous
    *R_out = R;
    return T;
}

void b200rwkv_engine::enqueue_score(const std::vector<ScoreItem>& items, int seq) {
    // pinned ring: a host buffer is rewritten only after the copy that read it has completed; the device list is reused in
    // stream order
    const int rb = seq % SCORE_RING;
    if (seq >= SCORE_RING) CK(cudaEventSynchronize(score_ev[rb]));
    ScoreItem* h = h_score + (size_t)rb * score_cap;
    memcpy(h, items.data(), items.size() * sizeof(ScoreItem));
    CK(cudaMemcpyAsync(d_score, h, items.size() * sizeof(ScoreItem), cudaMemcpyHostToDevice, stream));
    CK(cudaEventRecord(score_ev[rb], stream));
    ScoreParams sp;
    memset(&sp, 0, sizeof(sp));
    for (int q = 0; q < world; ++q) sp.shard[q] = (const float*)(peer_base[q] + off_logits);
    sp.world = world; sp.Vl = Vl; sp.V = V;
    sp.keep = d_keep; sp.items = d_score; sp.logp = d_logp;
    score_rows_kernel<<<(unsigned)items.size(), SCORE_THREADS, 0, stream>>>(sp);
    CK(cudaGetLastError());
    ++launch_total;
}

void b200rwkv_engine::infer(int nslot, const int32_t* slot, const int32_t* ntok, const uint32_t* tokens, const int32_t* option,
                            float* logits_out, size_t cap, int32_t* rows_out, float* logp_out, size_t logp_cap, bool scoring) {
    REQUIRE(nslot >= 0 && (nslot == 0 || (slot && ntok && option)), B200RWKV_ERR_INVALID, "infer: null argument");
    REQUIRE(connected, B200RWKV_ERR_INVALID, "tensor-parallel engine is not connected (b200rwkv_tp_connect)");
    // SCORE / SCORE_KEPT entries (b200rwkv_infer_score only) step like FULL; their rows are scored on the device, not copied
    const int opt_max = scoring ? B200RWKV_OPTION_SCORE_KEPT : B200RWKV_OPTION_NONE;
    auto is_score = [&](int i) { return option[i] == B200RWKV_OPTION_SCORE || option[i] == B200RWKV_OPTION_SCORE_KEPT; };
    std::vector<char> seen(S, 0);
    size_t total_rows = 0, total_tok = 0, total_score = 0;
    for (int i = 0; i < nslot; ++i) {
        REQUIRE(slot[i] >= 0 && slot[i] < S, B200RWKV_ERR_STATE, "infer: slot out of range");
        REQUIRE(!seen[slot[i]], B200RWKV_ERR_INVALID, "infer: duplicate slot in one call");
        seen[slot[i]] = 1;
        REQUIRE(ntok[i] >= 0, B200RWKV_ERR_INVALID, "infer: negative token count");
        REQUIRE(option[i] >= B200RWKV_OPTION_LAST && option[i] <= opt_max, B200RWKV_ERR_INVALID, "infer: bad option");
        const int r = (option[i] == B200RWKV_OPTION_FULL) ? ntok[i] : ((option[i] == B200RWKV_OPTION_LAST && ntok[i] > 0) ? 1 : 0);
        if (rows_out) rows_out[i] = r;
        total_rows += (size_t)r;
        total_tok += (size_t)ntok[i];
        if (is_score(i)) total_score += (size_t)ntok[i];
    }
    for (int i = 0; i < nslot; ++i) {
        if (option[i] != B200RWKV_OPTION_SCORE_KEPT) continue;
        REQUIRE(Vl % 4 == 0, B200RWKV_ERR_UNSUPPORTED, "infer_score: this engine keeps no logits rows (num_vocab / world is not a multiple of 4)");
        std::lock_guard<std::mutex> lk(keep_mu);
        REQUIRE(keep_valid[slot[i]], B200RWKV_ERR_STATE, "infer_score: SCORE_KEPT on slot " + std::to_string(slot[i]) + ", which has no kept logits row");
    }
    // tensor parallel: rank 0 writes logp_out; another rank checks it only when given it (in-process ranks all are)
    if (total_score > 0 && (rank == 0 || logp_out))
        REQUIRE(logp_out && logp_cap >= total_score, B200RWKV_ERR_INVALID, "infer_score: logp buffer missing or too small");
    REQUIRE(total_tok == 0 || tokens, B200RWKV_ERR_INVALID, "infer: null tokens");
    for (size_t i = 0; i < total_tok; ++i)
        REQUIRE(tokens[i] < (uint32_t)V, B200RWKV_ERR_INVALID, "infer: token id " + std::to_string(tokens[i]) + " is outside the vocabulary");
    const bool do_score = total_score > 0 && rank == 0;
    if (do_score) {
        if (!h_score) {
            score_cap = std::max(maxT, S);
            CK(cudaMallocHost(&h_score, (size_t)SCORE_RING * score_cap * sizeof(ScoreItem)));
            d_score = (ScoreItem*)dalloc((size_t)score_cap * sizeof(ScoreItem));
            for (auto& ev : score_ev) CK(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
        }
        if (total_score > logp_floats) {
            if (d_logp) { CK(cudaFree(d_logp)); d_logp = nullptr; logp_floats = 0; }
            const size_t want = std::max<size_t>(total_score, 4096);
            CK(cudaMalloc(&d_logp, want * 4));
            logp_floats = want;
        }
    }
    const bool want_logits = (rank == 0);          // tensor parallel: rank 0 gathers all vocabulary shards
    REQUIRE(!want_logits || !logits_out || total_rows * (size_t)V <= cap || total_rows == 0, B200RWKV_ERR_INVALID, "infer: logits buffer too small");
    // logits_out == NULL: the rows stay in HBM (b200rwkv_sample_topk reads the last row of every slot from there)
    const bool copy_logits = want_logits && logits_out != nullptr;
    // f32-activation mode runs every step decode-shaped (<= 16 tokens): the split-operand kernels are the 16-token ones
    const int step_cap = std::min(chunk, split_on ? 16 : maxT);
    // Step packing: every step shares its token budget evenly over the entries that still have tokens (web-rwkv shares the
    // chunk "fairly across slots", SURVEY.md A4; results do not depend on the cut).  Many slots with one token each keep
    // the WKV kernels wide (one CTA per head and slot) where a single slot with 64 tokens would run them 40 CTAs wide.
    std::vector<size_t> base(nslot + 1, 0), row_base(nslot + 1, 0);
    std::vector<int> pos(nslot, 0), rows_done(nslot, 0);
    for (int i = 0; i < nslot; ++i) {
        base[i + 1] = base[i] + (size_t)ntok[i];
        const int r = (option[i] == B200RWKV_OPTION_FULL) ? ntok[i] : ((option[i] == B200RWKV_OPTION_LAST && ntok[i] > 0) ? 1 : 0);
        row_base[i + 1] = row_base[i] + (size_t)r;
    }
    std::vector<size_t> lbase(nslot + 1, 0);      // where each scoring entry's log-probabilities start in logp_out
    for (int i = 0; i < nslot; ++i) lbase[i + 1] = lbase[i] + (is_score(i) ? (size_t)ntok[i] : 0);
    int score_seq = 0;
    if (do_score) {
        // first token of a SCORE_KEPT entry: scored against the slot's kept row as it stands before any step of this call
        std::vector<ScoreItem> first;
        for (int i = 0; i < nslot; ++i)
            if (option[i] == B200RWKV_OPTION_SCORE_KEPT && ntok[i] > 0) first.push_back({-(slot[i] + 1), tokens[base[i]], (int)lbase[i], 0});
        if (!first.empty()) {
            std::lock_guard<std::mutex> lk(keep_mu);
            enqueue_score(first, score_seq++);
        }
    }
    if (hidden_keep && total_tok > hidden_cap_rows) {
        if (d_hidden_all) { CK(cudaFree(d_hidden_all)); d_hidden_all = nullptr; hidden_cap_rows = 0; }
        const size_t want = std::max<size_t>(total_tok, 256);
        CK(cudaMalloc(&d_hidden_all, want * C * 4));
        hidden_cap_rows = want;
    }
    hidden_rows = 0;
    int step_no = 0;
    for (;;) {
        int n_active = 0;
        for (int i = 0; i < nslot; ++i) n_active += (pos[i] < ntok[i]);
        if (n_active == 0) break;
        std::vector<int> s_entry, s_slots, s_counts, s_out;
        std::vector<const uint32_t*> s_toks;
        // at least WKV_STAGE_TOK tokens per slot and step while prompts are long: a WKV CTA then loads and stores its 16 KB
        // of state once per four tokens (staged path) and a step touches a quarter of the slots' states
        const int quota = std::max(WKV_STAGE_TOK, step_cap / n_active);
        int used = 0;
        for (int i = 0; i < nslot && used < step_cap; ++i) {
            const int remain = ntok[i] - pos[i];
            if (remain <= 0) continue;
            const int take = std::min({remain, quota, step_cap - used});
            s_entry.push_back(i);
            s_counts.push_back(take);
            used += take;
        }
        for (size_t j = 0; j < s_entry.size() && used < step_cap; ++j) {      // left-over budget, in entry order
            const int i = s_entry[j];
            const int extra = std::min(ntok[i] - pos[i] - s_counts[j], step_cap - used);
            s_counts[j] += extra;
            used += extra;
        }
        for (size_t j = 0; j < s_entry.size(); ++j) {
            const int i = s_entry[j];
            s_slots.push_back(slot[i]);
            s_toks.push_back(tokens + base[i] + pos[i]);
            const bool finishes = (pos[i] + s_counts[j] == ntok[i]);
            s_out.push_back((option[i] == B200RWKV_OPTION_FULL || is_score(i)) ? 2 : ((finishes && option[i] == B200RWKV_OPTION_LAST) ? 1 : 0));
        }
        // pinned metadata ring: a buffer is rewritten only after the copy that read it has completed
        const int mb = step_no % META_RING;
        if (step_no >= META_RING) CK(cudaEventSynchronize(meta_ev[mb]));
        int* hm = h_meta + (size_t)mb * meta_ints;
        int R = 0;
        const int T = fill_meta(hm, s_slots, s_counts, s_toks, s_out, &R);
        last_T = T;
        last_R = R;
        CK(cudaMemcpyAsync(d_meta, hm, meta_ints * 4, cudaMemcpyHostToDevice, stream));
        CK(cudaEventRecord(meta_ev[mb], stream));
        run_step(mt_bucket(T), R > 0 ? mt_bucket(R) : 0);
        if (do_score) {
            // the target of a row is the next token of the same entry -- the first token of the entry's next step when the
            // packer cut its run here; an entry's last row has none.  Launched after the step, outside its graph.
            std::vector<ScoreItem> items;
            int r0 = 0;
            for (size_t j = 0; j < s_entry.size(); ++j) {
                const int i = s_entry[j];
                if (is_score(i))
                    for (int k = 0; k < s_counts[j]; ++k) {
                        const size_t p = (size_t)pos[i] + k;
                        if (p + 1 < (size_t)ntok[i]) items.push_back({r0 + k, tokens[base[i] + p + 1], (int)(lbase[i] + p + 1), 0});
                    }
                r0 += s_out[j] == 2 ? s_counts[j] : (s_out[j] == 1 ? 1 : 0);
            }
            if (!items.empty()) enqueue_score(items, score_seq++);
        }
        if (hidden_keep) {       // hidden rows of every token of this call (b200rwkv_last_hidden), in entry order
            int t0 = 0;
            for (size_t j = 0; j < s_entry.size(); ++j) {
                const int i = s_entry[j];
                CK(cudaMemcpyAsync(d_hidden_all + (base[i] + pos[i]) * (size_t)C, d_hidden + (size_t)t0 * C, (size_t)s_counts[j] * C * 4,
                                   cudaMemcpyDeviceToDevice, stream));
                t0 += s_counts[j];
            }
        }
        CK(cudaEventRecord(step_done, stream));
        if (R > 0) {
            std::lock_guard<std::mutex> lk(keep_mu);
            for (size_t i = 0; i < s_slots.size(); ++i)
                if (s_out[i] != 0) keep_valid[s_slots[i]] = 1;
        }
        if (R > 0 && copy_logits) {
            // rows of this step sit in entry order in d_logits; an entry's rows land at its own place of the entry-major
            // output, runs that are contiguous on both sides go out as one copy
            int r0 = 0;
            size_t j = 0;
            while (j < s_entry.size()) {
                const int i = s_entry[j];
                if (is_score(i)) { r0 += s_counts[j]; ++j; continue; }     // scored on the device, never copied
                int nr = s_out[j] == 2 ? s_counts[j] : (s_out[j] == 1 ? 1 : 0);
                if (nr == 0) { ++j; continue; }
                const size_t dst = row_base[i] + (size_t)rows_done[i];
                int run = nr;
                rows_done[i] += nr;
                size_t k = j + 1;
                while (k < s_entry.size()) {
                    const int i2 = s_entry[k];
                    if (is_score(i2)) break;                                  // its rows sit between: the source run ends
                    const int nr2 = s_out[k] == 2 ? s_counts[k] : (s_out[k] == 1 ? 1 : 0);
                    if (nr2 == 0) { ++k; continue; }
                    if (row_base[i2] + (size_t)rows_done[i2] != dst + (size_t)run) break;
                    rows_done[i2] += nr2;
                    run += nr2;
                    ++k;
                }
                float* o = logits_out + dst * (size_t)V;
                if (world == 1) {
                    CK(cudaMemcpyAsync(o, d_logits + (size_t)r0 * V, (size_t)run * V * 4, cudaMemcpyDeviceToHost, stream));
                } else {
                    for (int q = 0; q < world; ++q)      // column block q of every row, straight from rank q's shard
                        CK(cudaMemcpy2DAsync(o + (size_t)q * Vl, (size_t)V * 4, peer_base[q] + off_logits + (size_t)r0 * Vl * 4,
                                             (size_t)Vl * 4, (size_t)Vl * 4, run, cudaMemcpyDeviceToHost, stream));
                }
                r0 += run;
                j = k;
            }
        }      // (the next step's head projection is ordered after these copies by the stream)
        for (size_t j = 0; j < s_entry.size(); ++j) pos[s_entry[j]] += s_counts[j];
        ++step_no;
    }
    if (do_score) CK(cudaMemcpyAsync(logp_out, d_logp, total_score * 4, cudaMemcpyDeviceToHost, stream));
    CK(cudaStreamSynchronize(stream));
    if (do_score)
        for (int i = 0; i < nslot; ++i)
            if (option[i] == B200RWKV_OPTION_SCORE && ntok[i] > 0) logp_out[lbase[i]] = NAN;     // x0 has no preceding row
    if (hidden_keep) hidden_rows = (int)total_tok;
}

// GPU sampling front half (sample.cuh).  Runs on the softmax stream under the softmax mutex: the reference samples from the
// task that owns softmax (run.rs:1237), concurrently with the infer task; the per-slot rows it reads are only rewritten by a
// step that contains the slot, which the host cannot submit before this call returned the slot's token.
void b200rwkv_engine::sample_topk(int nrows, const int32_t* slots, const int32_t* pen_off, const uint32_t* pen_tok, const float* pen_val,
                                  const uint32_t* allow_bits, const int32_t* bias_off, const uint32_t* bias_tok, const float* bias_val,
                                  int top_k, uint32_t* ids_out, float* probs_out) {
    REQUIRE(rank == 0, B200RWKV_ERR_INVALID, "sample_topk: only rank 0 holds the gathered logits");
    REQUIRE(tk_cand_x, B200RWKV_ERR_UNSUPPORTED, "sample_topk: num_vocab > 65536 is not supported");
    REQUIRE(nrows >= 1 && nrows <= S && slots && ids_out && probs_out, B200RWKV_ERR_INVALID, "sample_topk: bad argument");
    REQUIRE(top_k >= 1 && top_k <= TOPK_MAX, B200RWKV_ERR_INVALID, "sample_topk: top_k must be in [1, 128]");
    {
        std::lock_guard<std::mutex> lk(keep_mu);
        std::vector<char> seen(S, 0);
        for (int i = 0; i < nrows; ++i) {
            REQUIRE(slots[i] >= 0 && slots[i] < S, B200RWKV_ERR_STATE, "sample_topk: slot out of range");
            REQUIRE(!seen[slots[i]], B200RWKV_ERR_INVALID, "sample_topk: duplicate slot");
            seen[slots[i]] = 1;
            REQUIRE(keep_valid[slots[i]], B200RWKV_ERR_STATE, "sample_topk: slot " + std::to_string(slots[i]) + " has produced no logits row yet");
        }
    }
    const int npen = pen_off ? pen_off[nrows] : 0, nbias = bias_off ? bias_off[nrows] : 0;
    REQUIRE(npen >= 0 && nbias >= 0 && (npen == 0 || (pen_tok && pen_val)) && (nbias == 0 || (bias_tok && bias_val)), B200RWKV_ERR_INVALID,
            "sample_topk: bad adjustment lists");
    for (int i = 0; i < nrows; ++i) {
        REQUIRE(!pen_off || (pen_off[i] >= 0 && pen_off[i] <= pen_off[i + 1]), B200RWKV_ERR_INVALID, "sample_topk: penalty offsets must ascend");
        REQUIRE(!bias_off || (bias_off[i] >= 0 && bias_off[i] <= bias_off[i + 1]), B200RWKV_ERR_INVALID, "sample_topk: bias offsets must ascend");
    }
    const size_t words = (size_t)(V + 31) / 32;
    auto al = [](size_t x) { return (x + 15) & ~(size_t)15; };
    // one staging blob: slot[n] | pen_off[n+1] | bias_off[n+1] | pen_tok | pen_val | bias_tok | bias_val | allow
    const size_t o_slot = 0, o_po = al(o_slot + (size_t)nrows * 4), o_bo = al(o_po + (size_t)(nrows + 1) * 4),
                 o_pt = al(o_bo + (size_t)(nrows + 1) * 4), o_pv = al(o_pt + (size_t)npen * 4), o_bt = al(o_pv + (size_t)npen * 4),
                 o_bv = al(o_bt + (size_t)nbias * 4), o_al = al(o_bv + (size_t)nbias * 4),
                 total = al(o_al + (allow_bits ? (size_t)nrows * words * 4 : 0));
    if (total > tk_cap) {
        if (tk_dev) { CK(cudaFree(tk_dev)); tk_dev = nullptr; }
        if (tk_host) { CK(cudaFreeHost(tk_host)); tk_host = nullptr; }
        tk_cap = 0;
        const size_t want = std::max<size_t>(total * 2, 1 << 20);
        CK(cudaMalloc(&tk_dev, want));
        CK(cudaMallocHost(&tk_host, want));
        tk_cap = want;
    }
    std::vector<int32_t> zeros(nrows + 1, 0);
    memcpy(tk_host + o_slot, slots, (size_t)nrows * 4);
    memcpy(tk_host + o_po, pen_off ? pen_off : zeros.data(), (size_t)(nrows + 1) * 4);
    memcpy(tk_host + o_bo, bias_off ? bias_off : zeros.data(), (size_t)(nrows + 1) * 4);
    if (npen) { memcpy(tk_host + o_pt, pen_tok, (size_t)npen * 4); memcpy(tk_host + o_pv, pen_val, (size_t)npen * 4); }
    if (nbias) { memcpy(tk_host + o_bt, bias_tok, (size_t)nbias * 4); memcpy(tk_host + o_bv, bias_val, (size_t)nbias * 4); }
    if (allow_bits) memcpy(tk_host + o_al, allow_bits, (size_t)nrows * words * 4);
    CK(cudaStreamWaitEvent(sm_stream, step_done, 0));
    CK(cudaMemcpyAsync(tk_dev, tk_host, total, cudaMemcpyHostToDevice, sm_stream));
    TopkParams tp;
    memset(&tp, 0, sizeof(tp));
    tp.keep = d_keep; tp.V = V; tp.nseg = cdiv(V, TOPK_SEG);
    tp.slot = (const int*)(tk_dev + o_slot);
    tp.pen_off = (const int*)(tk_dev + o_po); tp.pen_tok = (const unsigned*)(tk_dev + o_pt); tp.pen_val = (const float*)(tk_dev + o_pv);
    tp.bias_off = (const int*)(tk_dev + o_bo); tp.bias_tok = (const unsigned*)(tk_dev + o_bt); tp.bias_val = (const float*)(tk_dev + o_bv);
    tp.allow = allow_bits ? (const unsigned*)(tk_dev + o_al) : nullptr;
    tp.cand_x = tk_cand_x; tp.cand_id = tk_cand_id; tp.stats = tk_stats;
    tp.top_k = top_k; tp.out_id = tk_out_id; tp.out_p = tk_out_p;
    topk_segment_kernel<<<dim3(tp.nseg, nrows), TOPK_SEG_THREADS, 0, sm_stream>>>(tp);
    CK(cudaGetLastError());
    topk_merge_kernel<<<nrows, TOPK_MERGE_THREADS, 0, sm_stream>>>(tp);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(ids_out, tk_out_id, (size_t)nrows * top_k * 4, cudaMemcpyDeviceToHost, sm_stream));
    CK(cudaMemcpyAsync(probs_out, tk_out_p, (size_t)nrows * top_k * 4, cudaMemcpyDeviceToHost, sm_stream));
    CK(cudaStreamSynchronize(sm_stream));
}

// API layout <-> device layout for a live slot (snap == nullptr) or a snapshot record [L][C | Hl*N*N | C]
void b200rwkv_engine::state_xform(int slot, bool import, float* snap) {
    StateXform x;
    const size_t W = (size_t)Hl * N * N;
    x.api = d_api;
    if (snap) {
        const size_t rec = 2 * (size_t)C + W;
        x.att = snap; x.wkv = snap + C; x.ffn = snap + C + W;
        x.att_ls = x.wkv_ls = x.ffn_ls = rec;
    } else {
        x.att = att_shift + (size_t)slot * C; x.att_ls = (size_t)S * C;
        x.ffn = ffn_shift + (size_t)slot * C; x.ffn_ls = (size_t)S * C;
        x.wkv = wkv_state + (size_t)slot * W; x.wkv_ls = (size_t)S * W;
    }
    x.L = L; x.C = C; x.Hl = Hl; x.h0 = rank * Hl; x.transpose = (info.version != 7);
    const size_t total = (size_t)L * (N + 2) * C;
    const int grid = (int)std::min<size_t>((total + 255) / 256, 148 * 32);
    if (import) state_xform_kernel<true><<<grid, 256, 0, stream>>>(x);
    else state_xform_kernel<false><<<grid, 256, 0, stream>>>(x);
    CK(cudaGetLastError());
}

// =========================================================================================
// in-process tensor-parallel group
// =========================================================================================
void Group::start(int world) {
    status.assign(world, 0);
    errs.assign(world, "");
    for (int r = 1; r < world; ++r)
        workers.emplace_back([this, r]() {
            uint64_t seen = 0;
            for (;;) {
                std::function<int32_t(int)> fn;
                {
                    std::unique_lock<std::mutex> lk(m);
                    cv.wait(lk, [&] { return stop || gen != seen; });
                    if (stop) return;
                    seen = gen;
                    fn = job;
                }
                int32_t st;
                try {
                    st = fn(r);
                } catch (const std::exception& ex) {
                    g_err = ex.what();
                    st = B200RWKV_ERR_INVALID;
                }
                {
                    std::lock_guard<std::mutex> lk(m);
                    status[r] = st;
                    errs[r] = st < 0 ? g_err : std::string();
                    --pending;
                }
                cv.notify_all();
            }
        });
}

void Group::shutdown() {
    {
        std::lock_guard<std::mutex> lk(m);
        stop = true;
    }
    cv.notify_all();
    for (auto& t : workers) t.join();
    workers.clear();
}

// run fn(rank) on every rank at once; the first failure (lowest rank) is what the caller sees
int32_t Group::spmd(const std::function<int32_t(int)>& fn) {
    std::lock_guard<std::mutex> call(call_mu);
    {
        std::lock_guard<std::mutex> lk(m);
        job = fn;
        pending = (int)workers.size();
        ++gen;
    }
    cv.notify_all();
    int32_t st0;
    try {
        st0 = fn(0);
    } catch (const std::exception& ex) {
        g_err = ex.what();
        st0 = B200RWKV_ERR_INVALID;
    }
    {
        std::unique_lock<std::mutex> lk(m);
        cv.wait(lk, [&] { return pending == 0; });
    }
    if (st0 < 0) return st0;
    for (size_t r = 1; r < status.size(); ++r)
        if (status[r] < 0) {
            g_err = "rank " + std::to_string(r) + ": " + errs[r];
            return status[r];
        }
    return st0;
}

// =========================================================================================
// C ABI
// =========================================================================================
// Error text is thread-local: the reference makes engine calls from two tasks (infer / softmax, run.rs:1232-1237) and a
// per-engine string would race between them.  b200rwkv_last_error() returns the message of the calling thread's last failure.
#define API_BEGIN(e)                            \
    std::string* errp_ = &g_err;                \
    (void)(e);                                  \
    try {
#define API_END                                  \
    }                                            \
    catch (const Error& ex) {                    \
        *errp_ = ex.what();                      \
        return ex.code;                          \
    }                                            \
    catch (const std::exception& ex) {           \
        *errp_ = ex.what();                      \
        return B200RWKV_ERR_INVALID;             \
    }                                            \
    catch (...) {                                \
        *errp_ = "unknown exception";            \
        return B200RWKV_ERR_INVALID;             \
    }                                            \
    return B200RWKV_OK;

extern "C" {

int32_t b200rwkv_info_from_st(const uint8_t* st, size_t len, b200rwkv_info* out) {
    API_BEGIN((b200rwkv_engine*)nullptr)
    REQUIRE(out, B200RWKV_ERR_INVALID, "null out");
    StFile f(st, len);
    *out = derive_info(f);
    API_END
}

struct LoraArg { const uint8_t* st; size_t len; float alpha; };

static int32_t create_rank(const uint8_t* st, size_t len, int32_t device, int32_t max_batch, int32_t token_chunk_size,
                           int32_t precision, int32_t rank, int32_t world, const std::vector<LoraArg>& lora, b200rwkv_engine** out,
                           int32_t quant_layers = 0, int32_t quant_type = 0) {
    API_BEGIN((b200rwkv_engine*)nullptr)
    REQUIRE(out, B200RWKV_ERR_INVALID, "null out");
    *out = nullptr;
    REQUIRE(precision == 0 || precision == 1, B200RWKV_ERR_INVALID, "precision must be 0 (fp16) or 1 (fp32)");
    REQUIRE(max_batch >= 1 && max_batch <= 1024, B200RWKV_ERR_INVALID, "max_batch out of range");
    REQUIRE(token_chunk_size >= 1, B200RWKV_ERR_INVALID, "token_chunk_size must be >= 1");
    REQUIRE(world >= 1 && world <= 8 && rank >= 0 && rank < world, B200RWKV_ERR_INVALID, "bad rank/world");
    int ndev = 0;
    cudaError_t ce = cudaGetDeviceCount(&ndev);
    REQUIRE(ce == cudaSuccess && ndev > 0, B200RWKV_ERR_CUDA,
            std::string("no CUDA device (there is no CPU fallback): ") + cudaGetErrorString(ce));
    REQUIRE(device >= 0 && device < ndev, B200RWKV_ERR_INVALID, "device ordinal out of range");
    CK(cudaSetDevice(device));
    watchdog_setup();
    if (g_wd_host) {
        unsigned* dptr = nullptr;
        CK(cudaHostGetDevicePointer(&dptr, g_wd_host, 0));
        CK(cudaMemcpyToSymbol(g_watchdog, &dptr, sizeof(dptr)));
    }
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    REQUIRE(prop.major == 10, B200RWKV_ERR_UNSUPPORTED,
            "this library is built for sm_100a (B200) only; found sm_" + std::to_string(prop.major) + std::to_string(prop.minor));
    StFile f(st, len);
    std::vector<std::unique_ptr<StFile>> lora_files;
    std::unique_ptr<b200rwkv_engine> e(new b200rwkv_engine());
    for (const LoraArg& la : lora) {
        REQUIRE(la.st && la.len > 8, B200RWKV_ERR_INVALID, "null LoRA image");
        lora_files.emplace_back(new StFile(la.st, la.len));
        e->loras.push_back({lora_files.back().get(), la.alpha});
    }
    e->dev = device; e->rank = rank; e->world = world; e->num_sms = prop.multiProcessorCount;
    e->S = max_batch; e->chunk = token_chunk_size; e->precision = precision;
    REQUIRE(quant_layers >= 0 && quant_type >= 0, B200RWKV_ERR_INVALID, "bad quant_layers / quant_type");
    e->quant_layers = quant_type == QT_NONE ? 0 : quant_layers;
    e->quant_type = quant_layers == 0 ? (int)QT_NONE : quant_type;
    if (const char* v = dbg_env("B200RWKV_GRAPH")) e->use_graph = atoi(v) != 0;
    if (const char* v = dbg_env("B200RWKV_PDL")) e->use_pdl = atoi(v) != 0;
    e->build(f);
    e->loras.clear();            // the LoRA images are only borrowed during the build
    *out = e.release();
    API_END
}

int32_t b200rwkv_create_tp(const uint8_t* st, size_t len, int32_t device, int32_t max_batch, int32_t token_chunk_size,
                           int32_t precision, int32_t rank, int32_t world, b200rwkv_engine** out) {
    return create_rank(st, len, device, max_batch, token_chunk_size, precision, rank, world, {}, out);
}

int32_t b200rwkv_create(const uint8_t* st, size_t len, int32_t device, int32_t max_batch, int32_t token_chunk_size,
                        int32_t precision, b200rwkv_engine** out) {
    return create_rank(st, len, device, max_batch, token_chunk_size, precision, 0, 1, {}, out);
}

struct TpHandle {            // wire format of the 128-byte blob
    cudaIpcMemHandle_t ipc;  // 64 bytes
    int32_t rank, world;
    uint64_t comm_bytes;
    int32_t pid;
    int32_t device;
};
static_assert(sizeof(TpHandle) <= B200RWKV_TP_HANDLE_BYTES, "handle blob too large");

int32_t b200rwkv_tp_export(b200rwkv_engine* e, uint8_t* handle_out) {
    API_BEGIN(e)
    REQUIRE(e && handle_out, B200RWKV_ERR_INVALID, "null argument");
    CK(cudaSetDevice(e->dev));
    TpHandle h;
    memset(&h, 0, sizeof(h));
    CK(cudaIpcGetMemHandle(&h.ipc, e->comm_base));
    h.rank = e->rank; h.world = e->world; h.comm_bytes = e->comm_bytes; h.pid = (int32_t)getpid(); h.device = e->dev;
    memset(handle_out, 0, B200RWKV_TP_HANDLE_BYTES);
    memcpy(handle_out, &h, sizeof(h));
    API_END
}

int32_t b200rwkv_tp_connect(b200rwkv_engine* e, const uint8_t* handles) {
    API_BEGIN(e)
    REQUIRE(e && handles, B200RWKV_ERR_INVALID, "null argument");
    REQUIRE(!e->connected || e->world == 1, B200RWKV_ERR_INVALID, "already connected");
    std::lock_guard<std::mutex> lk(e->mu);
    CK(cudaSetDevice(e->dev));
    for (int q = 0; q < e->world; ++q) {
        TpHandle h;
        memcpy(&h, handles + (size_t)q * B200RWKV_TP_HANDLE_BYTES, sizeof(h));
        REQUIRE(h.rank == q && h.world == e->world && h.comm_bytes == e->comm_bytes, B200RWKV_ERR_INVALID,
                "tp_connect: handle blobs are not rank-ordered or come from a different model/world");
        if (q == e->rank) {
            e->peer_base[q] = e->comm_base;
        } else {
            void* p = nullptr;
            CK(cudaIpcOpenMemHandle(&p, h.ipc, cudaIpcMemLazyEnablePeerAccess));
            e->peer_base[q] = (uint8_t*)p;
            e->peer_ipc[q] = true;
        }
    }
    e->finalize_tp();
    CK(cudaDeviceSynchronize());
    API_END
}

// In-process variant (all ranks live in this process, e.g. tests with several ranks on one GPU, or a
// host that owns every GPU of the box as in SURVEY.md §8b): exchange the comm-block pointers directly.
int32_t b200rwkv_tp_connect_local(b200rwkv_engine** engines, int32_t n) {
    API_BEGIN((b200rwkv_engine*)nullptr)
    REQUIRE(engines && n >= 1 && n <= 8, B200RWKV_ERR_INVALID, "bad argument");
    for (int i = 0; i < n; ++i)
        REQUIRE(engines[i] && engines[i]->world == n && engines[i]->rank == i && engines[i]->comm_bytes == engines[0]->comm_bytes,
                B200RWKV_ERR_INVALID, "tp_connect_local: engines must be rank-ordered ranks of one world");
    for (int i = 0; i < n; ++i) {
        b200rwkv_engine* e = engines[i];
        CK(cudaSetDevice(e->dev));
        for (int q = 0; q < n; ++q) {
            if (engines[q]->dev != e->dev) {
                int can = 0;
                CK(cudaDeviceCanAccessPeer(&can, e->dev, engines[q]->dev));
                REQUIRE(can, B200RWKV_ERR_CUDA, "no peer access between the devices");
                cudaError_t pe = cudaDeviceEnablePeerAccess(engines[q]->dev, 0);
                if (pe != cudaSuccess && pe != cudaErrorPeerAccessAlreadyEnabled) CK(pe);
                (void)cudaGetLastError();
            }
            e->peer_base[q] = engines[q]->comm_base;
        }
        e->finalize_tp();
        CK(cudaDeviceSynchronize());
    }
    API_END
}

void b200rwkv_destroy(b200rwkv_engine* e) {
    if (!e) return;
    if (e->group) {
        std::unique_ptr<Group> g = std::move(e->group);
        g->shutdown();
        for (size_t r = 1; r < g->ranks.size(); ++r) delete g->ranks[r];
    }
    delete e;
}

int32_t b200rwkv_get_info(b200rwkv_engine* e, b200rwkv_info* out) {
    API_BEGIN(e)
    REQUIRE(e && out, B200RWKV_ERR_INVALID, "null argument");
    *out = e->info;
    API_END
}

static int32_t rank_infer(b200rwkv_engine* e, int32_t nslot, const int32_t* slot, const int32_t* ntok, const uint32_t* tokens,
                       const int32_t* option, float* logits_out, size_t logits_cap, int32_t* rows_out, float* logp_out = nullptr,
                       size_t logp_cap = 0, bool scoring = false) {
    API_BEGIN(e)
    REQUIRE(e, B200RWKV_ERR_INVALID, "null engine");
    std::lock_guard<std::mutex> lk(e->mu);
    CK(cudaSetDevice(e->dev));
    e->infer(nslot, slot, ntok, tokens, option, logits_out, logits_cap, rows_out, logp_out, logp_cap, scoring);
    API_END
}

int32_t b200rwkv_state_shape(b200rwkv_engine* e, int64_t shape[4]) {
    API_BEGIN(e)
    REQUIRE(e && shape, B200RWKV_ERR_INVALID, "null argument");
    shape[0] = e->C; shape[1] = e->N + 2; shape[2] = e->L; shape[3] = 1;
    API_END
}

int32_t b200rwkv_state_init(b200rwkv_engine* e, float* out) {
    API_BEGIN(e)
    REQUIRE(e && out, B200RWKV_ERR_INVALID, "null argument");
    const size_t n = (size_t)e->L * (e->N + 2) * e->C;
    if (e->init_state.empty()) memset(out, 0, n * 4);
    else memcpy(out, e->init_state.data(), n * 4);
    API_END
}

static int32_t rank_state_load(b200rwkv_engine* e, int32_t slot, const float* in) {
    API_BEGIN(e)
    REQUIRE(e && in, B200RWKV_ERR_INVALID, "null argument");
    REQUIRE(slot >= 0 && slot < e->S, B200RWKV_ERR_STATE, "slot out of range");
    std::lock_guard<std::mutex> lk(e->mu);
    CK(cudaSetDevice(e->dev));
    const size_t n = (size_t)e->L * (e->N + 2) * e->C;
    CK(cudaMemcpyAsync(e->d_api, in, n * 4, cudaMemcpyHostToDevice, e->stream));
    e->state_xform(slot, true);
    CK(cudaStreamSynchronize(e->stream));
    API_END
}

static int32_t rank_state_back(b200rwkv_engine* e, int32_t slot, float* out) {
    API_BEGIN(e)
    REQUIRE(e && out, B200RWKV_ERR_INVALID, "null argument");
    REQUIRE(slot >= 0 && slot < e->S, B200RWKV_ERR_STATE, "slot out of range");
    std::lock_guard<std::mutex> lk(e->mu);
    CK(cudaSetDevice(e->dev));
    const size_t n = (size_t)e->L * (e->N + 2) * e->C;
    e->state_xform(slot, false);
    CK(cudaMemcpyAsync(out, e->d_api, n * 4, cudaMemcpyDeviceToHost, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    API_END
}

// device-side snapshot: [L][C | Hl*N*N | C]
static void snapshot_copy(b200rwkv_engine* e, int slot, float* buf, bool to_snapshot) {
    const size_t C = e->C, W = (size_t)e->Hl * e->N * e->N, S = e->S, L = e->L;
    const size_t rec = 2 * C + W;
    struct Part { float* dev; size_t width; size_t off; };
    Part parts[3] = {{e->att_shift + (size_t)slot * C, C, 0}, {e->wkv_state + (size_t)slot * W, W, C}, {e->ffn_shift + (size_t)slot * C, C, C + W}};
    for (auto& p : parts) {
        if (to_snapshot)
            CK(cudaMemcpy2DAsync(buf + p.off, rec * 4, p.dev, S * p.width * 4, p.width * 4, L, cudaMemcpyDeviceToDevice, e->stream));
        else
            CK(cudaMemcpy2DAsync(p.dev, S * p.width * 4, buf + p.off, rec * 4, p.width * 4, L, cudaMemcpyDeviceToDevice, e->stream));
    }
}

// allocate a snapshot record (+ a logits row when this rank keeps them)
static Snapshot snapshot_alloc(b200rwkv_engine* e, bool with_logits) {
    Snapshot sn;
    const size_t rec = 2 * (size_t)e->C + (size_t)e->Hl * e->N * e->N;
    sn.bytes = rec * e->L * 4;
    CK(cudaMalloc(&sn.buf, sn.bytes));
    if (with_logits) {
        cudaError_t ce = cudaMalloc(&sn.logits, (size_t)e->V * 4);
        if (ce != cudaSuccess) { cudaFree(sn.buf); CK(ce); }
        sn.bytes += (size_t)e->V * 4;
    }
    return sn;
}

static int32_t rank_state_read(b200rwkv_engine* e, int32_t slot, uint64_t* snapshot_id) {
    API_BEGIN(e)
    REQUIRE(e && snapshot_id, B200RWKV_ERR_INVALID, "null argument");
    REQUIRE(slot >= 0 && slot < e->S, B200RWKV_ERR_STATE, "slot out of range");
    std::lock_guard<std::mutex> lk(e->mu);
    CK(cudaSetDevice(e->dev));
    bool row, has_row;
    {
        std::lock_guard<std::mutex> lk2(e->keep_mu);
        row = e->keep_valid[slot];
        has_row = e->d_keep && row;
    }
    Snapshot sn = snapshot_alloc(e, has_row);
    sn.row = row;
    try {
        snapshot_copy(e, slot, sn.buf, true);
        // the slot's last logits row travels with the state (CachedItem.output, run.rs:199-205): a cache hit can be sampled
        // on the device without re-running the last token
        if (has_row) CK(cudaMemcpyAsync(sn.logits, e->d_keep + (size_t)slot * e->V, (size_t)e->V * 4, cudaMemcpyDeviceToDevice, e->stream));
        CK(cudaStreamSynchronize(e->stream));
    } catch (...) {
        cudaFree(sn.buf);
        if (sn.logits) cudaFree(sn.logits);
        throw;
    }
    const uint64_t id = e->next_snap++;
    e->snaps[id] = sn;
    *snapshot_id = id;
    API_END
}

static int32_t rank_state_write(b200rwkv_engine* e, int32_t slot, uint64_t snapshot_id) {
    API_BEGIN(e)
    REQUIRE(e, B200RWKV_ERR_INVALID, "null engine");
    REQUIRE(slot >= 0 && slot < e->S, B200RWKV_ERR_STATE, "slot out of range");
    std::lock_guard<std::mutex> lk(e->mu);
    auto it = e->snaps.find(snapshot_id);
    REQUIRE(it != e->snaps.end(), B200RWKV_ERR_STATE, "unknown snapshot id");
    CK(cudaSetDevice(e->dev));
    snapshot_copy(e, slot, it->second.buf, false);
    if (e->d_keep && it->second.logits)
        CK(cudaMemcpyAsync(e->d_keep + (size_t)slot * e->V, it->second.logits, (size_t)e->V * 4, cudaMemcpyDeviceToDevice, e->stream));
    CK(cudaEventRecord(e->step_done, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    {
        std::lock_guard<std::mutex> lk2(e->keep_mu);
        e->keep_valid[slot] = it->second.row ? 1 : 0;       // rank 0: the snapshot holds the row exactly when `row` is set
    }
    API_END
}

static int32_t rank_state_free(b200rwkv_engine* e, uint64_t snapshot_id) {
    API_BEGIN(e)
    REQUIRE(e, B200RWKV_ERR_INVALID, "null engine");
    std::lock_guard<std::mutex> lk(e->mu);
    auto it = e->snaps.find(snapshot_id);
    REQUIRE(it != e->snaps.end(), B200RWKV_ERR_STATE, "unknown snapshot id");
    CK(cudaSetDevice(e->dev));
    CK(cudaFree(it->second.buf));
    if (it->second.logits) CK(cudaFree(it->second.logits));
    e->snaps.erase(it);
    API_END
}

// ---- device-resident state cache (SURVEY.md §8f-4): snapshots <-> host tensors, without passing through a slot ----
static int32_t rank_snapshot_back(b200rwkv_engine* e, uint64_t snapshot_id, float* state_out, float* logits_out) {
    API_BEGIN(e)
    REQUIRE(e && (state_out || logits_out), B200RWKV_ERR_INVALID, "null argument");
    std::lock_guard<std::mutex> lk(e->mu);
    auto it = e->snaps.find(snapshot_id);
    REQUIRE(it != e->snaps.end(), B200RWKV_ERR_STATE, "unknown snapshot id");
    CK(cudaSetDevice(e->dev));
    if (state_out) {
        const size_t n = (size_t)e->L * (e->N + 2) * e->C;
        e->state_xform(0, false, it->second.buf);
        CK(cudaMemcpyAsync(state_out, e->d_api, n * 4, cudaMemcpyDeviceToHost, e->stream));
    }
    if (logits_out) {
        REQUIRE(it->second.logits, B200RWKV_ERR_STATE, "snapshot holds no logits row");
        CK(cudaMemcpyAsync(logits_out, it->second.logits, (size_t)e->V * 4, cudaMemcpyDeviceToHost, e->stream));
    }
    CK(cudaStreamSynchronize(e->stream));
    API_END
}

static int32_t rank_snapshot_load(b200rwkv_engine* e, const float* state_in, const float* logits_in, uint64_t* snapshot_id) {
    API_BEGIN(e)
    REQUIRE(e && state_in && snapshot_id, B200RWKV_ERR_INVALID, "null argument");
    std::lock_guard<std::mutex> lk(e->mu);
    CK(cudaSetDevice(e->dev));
    Snapshot sn = snapshot_alloc(e, logits_in != nullptr && e->d_keep != nullptr);
    sn.row = logits_in != nullptr;
    try {
        const size_t n = (size_t)e->L * (e->N + 2) * e->C;
        CK(cudaMemcpyAsync(e->d_api, state_in, n * 4, cudaMemcpyHostToDevice, e->stream));
        e->state_xform(0, true, sn.buf);
        if (sn.logits) CK(cudaMemcpyAsync(sn.logits, logits_in, (size_t)e->V * 4, cudaMemcpyHostToDevice, e->stream));
        CK(cudaStreamSynchronize(e->stream));
    } catch (...) {
        cudaFree(sn.buf);
        if (sn.logits) cudaFree(sn.logits);
        throw;
    }
    const uint64_t id = e->next_snap++;
    e->snaps[id] = sn;
    *snapshot_id = id;
    API_END
}

int32_t b200rwkv_cache_stats(b200rwkv_engine* e, int64_t* num_snapshots, int64_t* bytes_used, int64_t* bytes_free) {
    API_BEGIN(e)
    REQUIRE(e, B200RWKV_ERR_INVALID, "null engine");
    std::lock_guard<std::mutex> lk(e->mu);
    CK(cudaSetDevice(e->dev));
    int64_t used = 0;
    for (auto& kv : e->snaps) used += (int64_t)kv.second.bytes;
    size_t fr = 0, tot = 0;
    CK(cudaMemGetInfo(&fr, &tot));
    if (num_snapshots) *num_snapshots = (int64_t)e->snaps.size();
    if (bytes_used) *bytes_used = used;
    if (bytes_free) *bytes_free = (int64_t)fr;
    API_END
}

// `vN::read_state(&context, &info, reader)` (reference lib.rs:378-389; `.state` files and InputState::File, run.rs:403-437):
// host only.  out: [L][N+2][C] f32 in the web-rwkv state layout.
int32_t b200rwkv_read_state(const b200rwkv_info* info, const uint8_t* st, size_t len, float* out) {
    API_BEGIN((b200rwkv_engine*)nullptr)
    REQUIRE(info && out, B200RWKV_ERR_INVALID, "null argument");
    REQUIRE(info->num_layer > 0 && info->num_head > 0 && info->head_size > 0 && info->num_emb == info->num_head * info->head_size,
            B200RWKV_ERR_INVALID, "bad model info");
    StFile f(st, len);
    std::vector<float> v;
    REQUIRE(state_from_st(f, info->num_layer, info->num_head, info->head_size, info->num_emb, v), B200RWKV_ERR_INVALID,
            "no blocks.*.att.time_state tensors in this file");
    memcpy(out, v.data(), v.size() * 4);
    API_END
}

int32_t b200rwkv_softmax(b200rwkv_engine* e, int32_t rows, const float* in, float* out) {
    API_BEGIN(e)
    REQUIRE(e && (rows == 0 || (in && out)) && rows >= 0, B200RWKV_ERR_INVALID, "bad argument");
    if (rows == 0) return B200RWKV_OK;
    std::lock_guard<std::mutex> lk(e->sm_mu);
    CK(cudaSetDevice(e->dev));
    if (rows > e->sm_rows_cap) {
        if (e->sm_in) { CK(cudaFree(e->sm_in)); CK(cudaFree(e->sm_out)); e->sm_in = e->sm_out = nullptr; }
        CK(cudaMalloc(&e->sm_in, (size_t)rows * e->V * 4));
        CK(cudaMalloc(&e->sm_out, (size_t)rows * e->V * 4));
        e->sm_rows_cap = rows;
    }
    const size_t bytes = (size_t)rows * e->V * 4;
    CK(cudaMemcpyAsync(e->sm_in, in, bytes, cudaMemcpyHostToDevice, e->sm_stream));
    softmax_kernel<<<rows, 1024, 0, e->sm_stream>>>(e->sm_in, e->sm_out, e->V);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(out, e->sm_out, bytes, cudaMemcpyDeviceToHost, e->sm_stream));
    CK(cudaStreamSynchronize(e->sm_stream));
    API_END
}

int32_t b200rwkv_sample_topk(b200rwkv_engine* e, int32_t nrows, const int32_t* slots, const int32_t* penalty_offset,
                             const uint32_t* penalty_token, const float* penalty_value, const uint32_t* allow_bits,
                             const int32_t* bias_offset, const uint32_t* bias_token, const float* bias_value, int32_t top_k,
                             uint32_t* ids_out, float* probs_out) {
    API_BEGIN(e)
    REQUIRE(e, B200RWKV_ERR_INVALID, "null engine");
    std::lock_guard<std::mutex> lk(e->sm_mu);
    CK(cudaSetDevice(e->dev));
    e->sample_topk(nrows, slots, penalty_offset, penalty_token, penalty_value, allow_bits, bias_offset, bias_token, bias_value, top_k,
                   ids_out, probs_out);
    API_END
}

int32_t b200rwkv_host_alloc(size_t bytes, void** out) {
    API_BEGIN((b200rwkv_engine*)nullptr)
    REQUIRE(out, B200RWKV_ERR_INVALID, "null out");
    CK(cudaMallocHost(out, bytes));
    API_END
}

void b200rwkv_host_free(void* p) {
    if (p) cudaFreeHost(p);
}

static void build_decode_metas(b200rwkv_engine* e, int nslot, const int32_t* slot, const uint32_t* tokens, int nsteps,
                               std::vector<int>& all) {
    all.assign((size_t)nsteps * e->meta_ints, 0);
    std::vector<int> s_slots(slot, slot + nslot), s_counts(nslot, 1), s_out(nslot, 1);
    std::vector<const uint32_t*> s_toks(nslot);
    for (size_t i = 0; i < (size_t)nsteps * nslot; ++i)
        REQUIRE(tokens[i] < (uint32_t)e->V, B200RWKV_ERR_INVALID, "token id outside the vocabulary");
    for (int st = 0; st < nsteps; ++st) {
        for (int i = 0; i < nslot; ++i) s_toks[i] = tokens + (size_t)st * nslot + i;
        int R = 0;
        e->fill_meta(all.data() + (size_t)st * e->meta_ints, s_slots, s_counts, s_toks, s_out, &R);
    }
}

static int32_t rank_bench_decode(b200rwkv_engine* e, int32_t nslot, const int32_t* slot, const uint32_t* tokens, int32_t warmup,
                              int32_t steps, int32_t flush_l2, float* ms_out, int64_t* launches_out, float* step_ms_out) {
    API_BEGIN(e)
    REQUIRE(e && slot && tokens && ms_out, B200RWKV_ERR_INVALID, "null argument");
    REQUIRE(nslot >= 1 && nslot <= e->S && nslot <= e->maxT && steps >= 1 && warmup >= 0, B200RWKV_ERR_INVALID, "bad argument");
    for (int i = 0; i < nslot; ++i) REQUIRE(slot[i] >= 0 && slot[i] < e->S, B200RWKV_ERR_STATE, "slot out of range");
    std::lock_guard<std::mutex> lk(e->mu);
    CK(cudaSetDevice(e->dev));
    const int nsteps = warmup + steps;
    std::vector<int> all;
    build_decode_metas(e, nslot, slot, tokens, nsteps, all);
    long long launches_before = 0;
    int* d_all = nullptr;
    CK(cudaMalloc(&d_all, all.size() * 4));
    CK(cudaMemcpy(d_all, all.data(), all.size() * 4, cudaMemcpyHostToDevice));
    void* flush = nullptr;
    const size_t flush_bytes = 256u << 20;
    if (flush_l2) CK(cudaMalloc(&flush, flush_bytes));
    cudaEvent_t ea, eb;
    CK(cudaEventCreate(&ea));
    CK(cudaEventCreate(&eb));
    std::vector<cudaEvent_t> marks;            // per-step boundaries (optional): the distribution of the step time
    if (step_ms_out) {
        marks.resize(steps);
        for (auto& m : marks) CK(cudaEventCreate(&m));
    }
    const int MT = mt_bucket(nslot);
    for (int st = 0; st < nsteps; ++st) {
        if (st == warmup) {
            CK(cudaStreamSynchronize(e->stream));
            CK(cudaEventRecord(ea, e->stream));
            launches_before = e->launch_total;
        }
        if (flush) CK(cudaMemsetAsync(flush, st & 0xff, flush_bytes, e->stream));
        CK(cudaMemcpyAsync(e->d_meta, d_all + (size_t)st * e->meta_ints, e->meta_ints * 4, cudaMemcpyDeviceToDevice, e->stream));
        e->run_step(MT, MT);
        if (step_ms_out && st >= warmup) CK(cudaEventRecord(marks[st - warmup], e->stream));
    }
    CK(cudaEventRecord(eb, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    {
        // every step kept each slot's logits row in HBM (enqueue_keep): readable as after b200rwkv_infer(logits_out = NULL)
        std::lock_guard<std::mutex> lk2(e->keep_mu);
        for (int i = 0; i < nslot; ++i) e->keep_valid[slot[i]] = 1;
    }
    CK(cudaEventElapsedTime(ms_out, ea, eb));
    for (int i = 0; i < (int)marks.size(); ++i) {
        CK(cudaEventElapsedTime(step_ms_out + i, i == 0 ? ea : marks[i - 1], marks[i]));
    }
    for (auto& m : marks) cudaEventDestroy(m);
    if (launches_out) *launches_out = (int64_t)(e->launch_total - launches_before);
    CK(cudaEventDestroy(ea));
    CK(cudaEventDestroy(eb));
    if (flush) CK(cudaFree(flush));
    CK(cudaFree(d_all));
    API_END
}

static int32_t rank_profile_step(b200rwkv_engine* e, int32_t nslot, const int32_t* slot, const uint32_t* tokens, float ms[4],
                              int32_t launches[4], int64_t* gemm_weight_bytes) {
    API_BEGIN(e)
    REQUIRE(e && slot && tokens && ms && launches, B200RWKV_ERR_INVALID, "null argument");
    REQUIRE(nslot >= 1 && nslot <= e->S && nslot <= e->maxT, B200RWKV_ERR_INVALID, "bad argument");
    std::lock_guard<std::mutex> lk(e->mu);
    CK(cudaSetDevice(e->dev));
    std::vector<int> all;
    build_decode_metas(e, nslot, slot, tokens, 1, all);
    CK(cudaMemcpyAsync(e->d_meta, all.data(), e->meta_ints * 4, cudaMemcpyHostToDevice, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    Profiler prof;
    const int MT = mt_bucket(nslot);
    e->enqueue_step(e->stream, MT, MT, &prof);
    CK(cudaStreamSynchronize(e->stream));
    for (int i = 0; i < 4; ++i) { ms[i] = 0.f; launches[i] = 0; }
    for (auto& r : prof.recs) {
        float t = 0.f;
        CK(cudaEventElapsedTime(&t, r.a, r.b));
        ms[r.cls] += t;
        launches[r.cls] += 1;
        cudaEventDestroy(r.a);
        cudaEventDestroy(r.b);
    }
    if (gemm_weight_bytes) *gemm_weight_bytes = (int64_t)e->weight_bytes_total;
    API_END
}

// In-situ timeline of a graph-replayed decode step: every launch of the step writes globaltimer stamps (CTA 0: entry, past
// griddepcontrol.wait, exit; projections: exit of EVERY CTA).  A launch's window is [released by griddepcontrol.wait, last CTA
// exit]: with programmatic dependent launch a kernel is resident long before it may touch its inputs, so CUDA events around
// launches (b200rwkv_profile_step) over-count; windows of consecutive launches cannot overlap (the wait returns only when the
// previous grid has completed), so their sum is <= the step.  Averages over `reps` replays of a traced copy of the step graph.
static int32_t rank_profile_insitu(b200rwkv_engine* e, int32_t nslot, const int32_t* slot, const uint32_t* tokens, int32_t reps,
                                int32_t cap, int32_t* n_out, int32_t* types, double* start_us, double* end_us, int64_t* bytes,
                                double* step_us) {
    API_BEGIN(e)
    REQUIRE(e && slot && tokens && n_out && types && start_us && end_us && bytes && step_us && reps >= 1 && cap >= 1, B200RWKV_ERR_INVALID,
            "bad argument");
    REQUIRE(nslot >= 1 && nslot <= e->S && nslot <= e->maxT, B200RWKV_ERR_INVALID, "bad argument");
    std::lock_guard<std::mutex> lk(e->mu);
    CK(cudaSetDevice(e->dev));
    if (!e->d_step_trace) e->d_step_trace = (unsigned long long*)e->dalloc((size_t)b200rwkv_engine::STEP_TRACE_MAX * b200rwkv_engine::STEP_TRACE_ROW * 8, true);
    std::vector<int> all;
    build_decode_metas(e, nslot, slot, tokens, 1, all);
    CK(cudaMemcpyAsync(e->d_meta, all.data(), e->meta_ints * 4, cudaMemcpyHostToDevice, e->stream));
    const int MT = mt_bucket(nslot);
    // traced copy of the step graph (the production graphs carry null trace pointers)
    const bool was = e->trace_capture;
    e->trace_capture = true;
    e->step_trace_types.clear();
    e->step_trace_bytes.clear();
    cudaGraph_t g = nullptr;
    cudaGraphExec_t ge = nullptr;
    CK(cudaStreamBeginCapture(e->stream, cudaStreamCaptureModeThreadLocal));
    try {
        e->enqueue_step(e->stream, MT, MT, nullptr);
    } catch (...) {
        cudaStreamEndCapture(e->stream, &g);
        if (g) cudaGraphDestroy(g);
        e->trace_capture = was;
        throw;
    }
    e->trace_capture = was;
    CK(cudaStreamEndCapture(e->stream, &g));
    CK(cudaGraphInstantiate(&ge, g, 0));
    CK(cudaGraphDestroy(g));
    const int n = (int)e->step_trace_types.size();
    const size_t row = b200rwkv_engine::STEP_TRACE_ROW;
    std::vector<unsigned long long> h((size_t)n * row);
    std::vector<double> s_acc(n, 0.0), e_acc(n, 0.0);
    double step_acc = 0.0;
    e->step_trace_bytes.resize(n, 0);
    for (int r = 0; r < reps + 1; ++r) {        // first replay is warm-up
        CK(cudaMemsetAsync(e->d_step_trace, 0, (size_t)n * row * 8, e->stream));
        build_decode_metas(e, nslot, slot, tokens, 1, all);      // a fresh step sequence number: the folded rendezvous keys on it
        CK(cudaMemcpyAsync(e->d_meta, all.data(), e->meta_ints * 4, cudaMemcpyHostToDevice, e->stream));
        CK(cudaGraphLaunch(ge, e->stream));
        CK(cudaStreamSynchronize(e->stream));
        if (r == 0) continue;
        CK(cudaMemcpy(h.data(), e->d_step_trace, (size_t)n * row * 8, cudaMemcpyDeviceToHost));
        unsigned long long t0 = ~0ull, t1 = 0;
        for (int i = 0; i < n; ++i) {
            const unsigned long long* q = h.data() + (size_t)i * row;
            if (q[0] && q[0] < t0) t0 = q[0];
        }
        for (int i = 0; i < n; ++i) {
            const unsigned long long* q = h.data() + (size_t)i * row;
            const bool gemm = e->step_trace_types[i] >= 1000000;
            unsigned long long st = gemm ? q[2] : q[1], en = q[7];
            if (gemm)
                for (int c = 0; c < e->num_sms && 8 + 3 * c + 2 < (int)row; ++c) en = std::max(en, q[8 + 3 * c + 2]);
            if (!st || !en) continue;
            s_acc[i] += (double)(st - t0) * 1e-3;
            e_acc[i] += (double)(en - t0) * 1e-3;
            t1 = std::max(t1, en);
        }
        step_acc += (double)(t1 - t0) * 1e-3;
    }
    cudaGraphExecDestroy(ge);
    int m = 0;
    for (int i = 0; i < n && m < cap; ++i) {
        if (e_acc[i] <= 0.0) continue;
        types[m] = e->step_trace_types[i];
        start_us[m] = s_acc[i] / reps;
        end_us[m] = e_acc[i] / reps;
        bytes[m] = e->step_trace_bytes[i];
        ++m;
    }
    *n_out = m;
    *step_us = step_acc / reps;
    API_END
}

// Operator-level entry for the parity tests: the load-time quantiser (qgemm.cuh) on one matrix, un-tiled on the host into plain
// row-major codes and per-block parameters so that oracle/quant_numpy.py can be compared bit for bit.
int32_t b200rwkv_op_quantize(int32_t device, int32_t quant_type, int32_t N, int32_t K, const uint16_t* w_f16, uint8_t* codes,
                             uint16_t* p0, uint16_t* p1) {
    API_BEGIN((b200rwkv_engine*)nullptr)
    REQUIRE(quant_type == QT_INT8 || quant_type == QT_NF4, B200RWKV_ERR_UNSUPPORTED, "quant_type must be Int8 or NF4");
    REQUIRE(N >= 1 && K >= GEMM_BK && K % GEMM_BK == 0 && (size_t)N * K <= ((size_t)1 << 31) && w_f16 && codes && p0, B200RWKV_ERR_INVALID, "bad argument");
    REQUIRE(quant_type == QT_NF4 || p1, B200RWKV_ERR_INVALID, "Int8 needs p1 (scales)");
    CK(cudaSetDevice(device));
    const int tiles = cdiv(N, GEMM_BN), KB = K / GEMM_BK;
    const size_t blk = (size_t)q_block_bytes(quant_type), total = (size_t)tiles * KB * blk;
    DevTmp src((size_t)N * K * 2), dst(total);
    CK(cudaMemcpy(src.p, w_f16, (size_t)N * K * 2, cudaMemcpyHostToDevice));
    const size_t nwarp = (size_t)tiles * KB * GEMM_BN;
    const int grid = (int)std::min<size_t>((nwarp + 7) / 8, 148 * 32);
    if (quant_type == QT_INT8) quantize_weight_kernel<QT_INT8><<<grid, 256>>>((const __half*)src.p, K, 0, 0, N, tiles, KB, (uint8_t*)dst.p);
    else quantize_weight_kernel<QT_NF4><<<grid, 256>>>((const __half*)src.p, K, 0, 0, N, tiles, KB, (uint8_t*)dst.p);
    CK(cudaGetLastError());
    CK(cudaDeviceSynchronize());
    std::vector<uint8_t> h(total);
    CK(cudaMemcpy(h.data(), dst.p, total, cudaMemcpyDeviceToHost));
    for (int n = 0; n < N; ++n) {
        const int tile = n / GEMM_BN, r = n % GEMM_BN;
        for (int kb = 0; kb < KB; ++kb) {
            const uint8_t* b = h.data() + ((size_t)tile * KB + kb) * blk;
            if (quant_type == QT_INT8) {
                for (int k = 0; k < GEMM_BK; ++k) codes[(size_t)n * K + kb * GEMM_BK + k] = b[(size_t)((k >> 4) * GEMM_BN + r) * 16 + (k & 15)];
                uint16_t pr[2];
                memcpy(pr, b + GEMM_BN * GEMM_BK + r * 4, 4);
                p1[(size_t)n * KB + kb] = pr[0];      // scale
                p0[(size_t)n * KB + kb] = pr[1];      // min
            } else {
                for (int k = 0; k < GEMM_BK; ++k) {
                    const uint8_t by = b[(size_t)((k >> 5) * GEMM_BN + r) * 16 + ((k & 31) >> 1)];
                    codes[(size_t)n * K + kb * GEMM_BK + k] = (k & 1) ? (by >> 4) : (by & 15);
                }
                uint16_t pr[2];
                memcpy(pr, b + GEMM_BN * GEMM_BK / 2 + r * 4, 4);
                p0[(size_t)n * (2 * KB) + 2 * kb] = pr[0];
                p0[(size_t)n * (2 * KB) + 2 * kb + 1] = pr[1];
            }
        }
    }
    API_END
}

// Operator-level entry for the parity tests: ONE launch of the WKV kernel (recurrence + GroupNorm + bonus + gate) on caller
// supplied head vectors and state, no model around it.  This is how the committed fla fixtures (tests/golden/wkv6_fla.npz,
// wkv7_fla.npz: independent pins of the recurrences) reach the CUDA kernels.
int32_t b200rwkv_op_wkv(int32_t device, int32_t version, int32_t T, int32_t H, const float* r, const float* k, const float* v,
                        const float* w, const float* u, const float* a, const float* k_k, const float* k_a, const float* r_k,
                        const float* g, const float* lnx_w, const float* lnx_b, float* state, float* out) {
    API_BEGIN((b200rwkv_engine*)nullptr)
    REQUIRE(version == 5 || version == 6 || version == 7, B200RWKV_ERR_UNSUPPORTED, "version must be 5, 6 or 7");
    REQUIRE(T >= 1 && T <= 64 && H >= 1 && H <= 1024 && r && k && v && w && state && out, B200RWKV_ERR_INVALID, "bad argument");
    REQUIRE(version == 7 ? (a && k_k && k_a && r_k) : (u != nullptr), B200RWKV_ERR_INVALID, "missing per-version operand");
    CK(cudaSetDevice(device));
    const int Cc = H * 64;
    const size_t TC = (size_t)T * Cc;
    std::vector<DevTmp*> keep;
    struct Guard { std::vector<DevTmp*>& v; ~Guard() { for (auto* p : v) delete p; } } guard{keep};
    auto up = [&](const float* h, size_t n, float fill) -> float* {
        keep.push_back(new DevTmp(n * 4));
        float* d = (float*)keep.back()->p;
        if (h) CK(cudaMemcpy(d, h, n * 4, cudaMemcpyHostToDevice));
        else {
            std::vector<float> tmp(n, fill);
            CK(cudaMemcpy(d, tmp.data(), n * 4, cudaMemcpyHostToDevice));
        }
        return d;
    };
    const int maxT = 64, maxS = 1;
    std::vector<int> meta(MetaView::ints(maxT, maxS), 0);
    meta[0] = T; meta[1] = 1; meta[2] = 0;
    for (int t = 0; t < T; ++t) {
        meta[8 + maxT + t] = 0;                       // tok_slot
        meta[8 + 2 * maxT + t] = t == 0 ? -1 : t - 1; // tok_prev
        meta[8 + 3 * maxT + t] = t == T - 1;          // tok_last
        meta[8 + 5 * maxT + t] = -1;                  // tok_outrow
    }
    meta[8 + 6 * maxT] = 0; meta[8 + 6 * maxT + maxS] = 0; meta[8 + 6 * maxT + 2 * maxS] = T;
    keep.push_back(new DevTmp(meta.size() * 4));
    int* d_meta = (int*)keep.back()->p;
    CK(cudaMemcpy(d_meta, meta.data(), meta.size() * 4, cudaMemcpyHostToDevice));
    WkvParams p;
    memset(&p, 0, sizeof(p));
    p.version = version; p.ld = Cc; p.meta = MetaView{d_meta, maxT, maxS}; p.H = H;
    p.state = up(state, (size_t)H * 64 * 64, 0.f);
    p.r = up(r, TC, 0.f); p.k = up(k, TC, 0.f); p.v = up(v, TC, 0.f); p.g = up(g, TC, 1.f);
    if (version == 5) p.w_static = up(w, Cc, 0.f); else p.w = up(w, TC, 0.f);
    p.lnx_w = up(lnx_w, Cc, 1.f); p.lnx_b = up(lnx_b, Cc, 0.f);
    if (version != 7) p.u = up(u, Cc, 0.f);
    else {
        p.a = up(a, TC, 0.f); p.nu = up(nullptr, TC, 0.f); p.v_first = up(nullptr, TC, 0.f); p.layer0 = 1;
        p.k_k = up(k_k, Cc, 0.f); p.k_a = up(k_a, Cc, 0.f); p.r_k = up(r_k, Cc, 0.f);
    }
    const size_t halves = (size_t)(rup(Cc, GEMM_BK) / GEMM_BK) * A16_KB_HALVES;
    keep.push_back(new DevTmp(halves * 2));
    p.out = (__half*)keep.back()->p;
    p.kq_tile = 64;                       // token rows of the A16 output: any value >= T the reader below agrees on
    CK(cudaMemset(p.out, 0, halves * 2));
    const size_t smem = wkv_smem_bytes(version, false, 0, maxT);
    switch (version) {
        case 5: wkv_kernel<5><<<dim3(H, 1), WKV_SA_THREADS, smem>>>(p, maxT); break;
        case 6: wkv_kernel<6><<<dim3(H, 1), WKV_SA_THREADS, smem>>>(p, maxT); break;
        default: wkv_kernel<7><<<dim3(H, 1), WKV_SA_THREADS, smem>>>(p, maxT); break;
    }
    CK(cudaGetLastError());
    CK(cudaDeviceSynchronize());
    std::vector<__half> ho(halves);
    CK(cudaMemcpy(ho.data(), p.out, halves * 2, cudaMemcpyDeviceToHost));
    for (int t = 0; t < T; ++t)
        for (int c = 0; c < Cc; ++c) out[(size_t)t * Cc + c] = __half2float(ho[a16_index(t, c, 64)]);
    CK(cudaMemcpy(state, p.state, (size_t)H * 64 * 64 * 4, cudaMemcpyDeviceToHost));
    API_END
}

int32_t b200rwkv_launch_count(b200rwkv_engine* e, int64_t* total) {
    API_BEGIN(e)
    REQUIRE(e && total, B200RWKV_ERR_INVALID, "null argument");
    std::lock_guard<std::mutex> lk(e->mu);
    *total = (int64_t)e->launch_total;
    API_END
}

int32_t b200rwkv_keep_hidden(b200rwkv_engine* e, int32_t enable) {
    API_BEGIN(e)
    REQUIRE(e, B200RWKV_ERR_INVALID, "null engine");
    std::lock_guard<std::mutex> lk(e->mu);
    e->hidden_keep = enable != 0;
    e->hidden_rows = 0;
    API_END
}

// returns the number of rows written (negative status on error)
int32_t b200rwkv_last_hidden(b200rwkv_engine* e, float* out, size_t cap) {
    int32_t rows = 0;
    const int32_t st = [&]() -> int32_t {
        API_BEGIN(e)
        REQUIRE(e && out, B200RWKV_ERR_INVALID, "null argument");
        std::lock_guard<std::mutex> lk(e->mu);
        CK(cudaSetDevice(e->dev));
        CK(cudaStreamSynchronize(e->stream));
        const bool all = e->hidden_keep && e->d_hidden_all;
        rows = all ? e->hidden_rows : e->last_T;
        const size_t n = (size_t)rows * e->C;
        REQUIRE(n <= cap, B200RWKV_ERR_INVALID, "hidden buffer too small");
        if (n) CK(cudaMemcpy(out, all ? e->d_hidden_all : e->d_hidden, n * 4, cudaMemcpyDeviceToHost));
        API_END
    }();
    return st < 0 ? st : rows;
}

// Test aid: copy a named internal activation buffer of the most recent step of b200rwkv_infer to the host as f32 row-major
// [rows, cols]; returns cols and stores rows (the step's tokens; output rows for `a_head`), or a negative status.  A16 buffers
// of a split-operand step hold hi values in token rows 0..15 and lo values in rows 16..31: they are returned as hi + lo, the
// value the projection consumes (exact in f32).  Not used on the product path.
int32_t b200rwkv_debug_read(b200rwkv_engine* e, const char* name, float* out, size_t cap, int32_t* rows_out) {
    if (!e || !name || !out || !rows_out) return B200RWKV_ERR_INVALID;
    std::string* errp_ = &g_err;
    try {
        std::lock_guard<std::mutex> lk(e->mu);
        CK(cudaSetDevice(e->dev));
        CK(cudaStreamSynchronize(e->stream));
        const std::string n(name);
        const int T = std::max(e->last_T, 1);
        struct F { const char* n; float* p; int cols; };
        const F fs[] = {{"x_a", e->x_a, e->C}, {"x_b", e->x_b, e->C}, {"xx1", e->xx1, e->C}, {"sx1", e->sx1, e->C}, {"xx2", e->xx2, e->C},
                        {"r", e->f_r, e->Cl}, {"k", e->f_k, e->Cl}, {"v", e->f_v, e->Cl}, {"g", e->f_g, e->Cl}, {"w", e->f_w, e->Cl},
                        {"a", e->f_a, e->Cl}, {"nu", e->f_nu, e->Cl}, {"rr", e->f_rr, e->Cl}, {"part_att", e->part_att, e->C},
                        {"part_ffn", e->part_ffn, e->C}, {"hidden", e->d_hidden, e->C}};
        for (const F& f : fs)
            if (n == f.n) {
                REQUIRE((size_t)T * f.cols <= cap, B200RWKV_ERR_INVALID, "debug buffer too small");
                CK(cudaMemcpy(out, f.p, (size_t)T * f.cols * 4, cudaMemcpyDeviceToHost));
                const int nsum = (n == "part_att") ? e->split_att : (n == "part_ffn" ? e->split_ffn : 1);
                std::vector<float> tmp((size_t)T * f.cols);
                for (int sp = 1; sp < nsum; ++sp) {       // split-K partials: sum the slices
                    CK(cudaMemcpy(tmp.data(), f.p + (size_t)sp * e->maxT * e->C, tmp.size() * 4, cudaMemcpyDeviceToHost));
                    for (size_t i = 0; i < tmp.size(); ++i) out[i] += tmp[i];
                }
                *rows_out = T;
                return f.cols;
            }
        struct A { std::string n; const A16Buf* b; int cols; int mat; };
        std::vector<A> as;
        for (int i = 0; i < 6; ++i) as.push_back({"a_x" + std::to_string(i), &e->a_x[i], e->C, 0});
        for (int i = 0; i < 5; ++i)
            for (int m = 0; m < 5; ++m) as.push_back({"a_lora" + std::to_string(i) + "_" + std::to_string(m), &e->a_lora[i], e->a_lora[i].kq * 32, m});
        as.push_back({"a_out", &e->a_out, e->Cl, 0});
        as.push_back({"a_kk", &e->a_kk, e->Fl, 0});
        as.push_back({"a_head", &e->a_head, e->C, 0});
        for (const A& a : as)
            if (n == a.n && a.b->p) {
                const bool head = (n == "a_head");        // the head's operand holds output rows (R), not tokens
                const int rows = head ? e->last_R : T, th = head ? e->last_th_rows : e->last_th;
                REQUIRE((size_t)rows * a.cols <= cap, B200RWKV_ERR_INVALID, "debug buffer too small");
                std::vector<__half> h(a.b->halves_per_matrix);
                CK(cudaMemcpy(h.data(), a.b->p + (size_t)a.mat * a.b->halves_per_matrix, h.size() * 2, cudaMemcpyDeviceToHost));
                for (int t = 0; t < rows; ++t)
                    for (int c = 0; c < a.cols; ++c) {
                        float v = __half2float(h[a16_index(t, c, th)]);
                        if (e->last_split) v += __half2float(h[a16_index(t + 16, c, th)]);
                        out[(size_t)t * a.cols + c] = v;
                    }
                *rows_out = rows;
                return a.cols;
            }
        throw Error(B200RWKV_ERR_INVALID, "unknown debug buffer: " + n);
    } catch (const Error& ex) {
        *errp_ = ex.what();
        return ex.code;
    } catch (const std::exception& ex) {
        *errp_ = ex.what();
        return B200RWKV_ERR_INVALID;
    } catch (...) {
        *errp_ = "unknown exception";
        return B200RWKV_ERR_INVALID;
    }
}

// Test aid: the projection launches a step of MT token tiles runs for layer `layer` (-1: the head, at MT output-row tiles), in
// stream order; one record of B200RWKV_PLAN_INTS int32 each (layout in include/b200rwkv.h).  Returns the number of launches.
static_assert(B200RWKV_PLAN_INTS == 8 + 5 * GEMM_MAX_SEG, "plan record layout");
int32_t b200rwkv_debug_plan(b200rwkv_engine* e, int32_t layer, int32_t mt, int32_t* out, size_t cap) {
    int32_t count = 0;
    const int32_t st = [&]() -> int32_t {
        API_BEGIN(e)
        REQUIRE(e && out, B200RWKV_ERR_INVALID, "null argument");
        REQUIRE(layer >= -1 && layer < e->L, B200RWKV_ERR_INVALID, "debug_plan: layer out of range");
        REQUIRE(mt == 1 || mt == 2 || mt == 4 || mt == 8, B200RWKV_ERR_INVALID, "debug_plan: mt must be 1, 2, 4 or 8");
        std::lock_guard<std::mutex> lk(e->mu);
        std::vector<const GemmLaunch*> gs;
        if (layer < 0) {
            gs.push_back(&e->head);
        } else {
            const Layer& ly = e->layers[layer];
            for (int gi = 0; gi < (int)ly.pre.size(); ++gi)
                if (!e->pre_skipped(ly, gi, mt)) gs.push_back(&ly.pre[gi]);
            gs.push_back(&ly.o);
            for (auto& g : ly.ffn) gs.push_back(&g);
        }
        REQUIRE(gs.size() * B200RWKV_PLAN_INTS <= cap, B200RWKV_ERR_INVALID, "debug_plan: buffer too small");
        for (const GemmLaunch* g : gs) {
            int32_t* r = out + (size_t)count * B200RWKV_PLAN_INTS;
            memset(r, 0, B200RWKV_PLAN_INTS * 4);
            r[0] = mt >= 4 ? g->grid_wide : g->grid;         // launch_gemm: split-operand decode steps run `grid` too
            r[1] = g->grid; r[2] = g->grid_wide; r[3] = g->p.total_blocks; r[4] = g->p.max_contrib; r[5] = g->qtype;
            r[6] = g->forced ? 1 : 0; r[7] = g->p.nseg;
            for (int i = 0; i < g->p.nseg; ++i) {
                const GemmSeg& sg = g->p.seg[i];
                int32_t* q = r + 8 + 5 * i;
                q[0] = sg.KB; q[1] = sg.tiles; q[2] = sg.N; q[3] = sg.out_mode; q[4] = sg.act;
            }
            ++count;
        }
        API_END
    }();
    return st < 0 ? st : count;
}

// Profiling aid: the raw stamp rows of the most recent traced replay (b200rwkv_profile_insitu): one row of 512 uint64 per
// launch -- [0..7] globaltimer stamps of CTA 0 (entry, past griddepcontrol.wait, phase marks, exit), then {SM id, last MMA
// issued, exit} of every projection CTA (or {entry, released, phase 1 done} of every CTA of the RWKV-6 front-half kernel).
int32_t b200rwkv_debug_trace(b200rwkv_engine* e, uint64_t* out, size_t cap, int32_t* types, int32_t* nphase) {
    API_BEGIN(e)
    REQUIRE(e && out && types && nphase, B200RWKV_ERR_INVALID, "null argument");
    REQUIRE(e->d_step_trace && !e->step_trace_types.empty(), B200RWKV_ERR_INVALID, "no trace: call b200rwkv_profile_insitu first");
    std::lock_guard<std::mutex> lk(e->mu);
    const size_t nl = e->step_trace_types.size();
    const size_t row = b200rwkv_engine::STEP_TRACE_ROW;
    REQUIRE(cap >= nl * row, B200RWKV_ERR_INVALID, "trace buffer too small");
    CK(cudaSetDevice(e->dev));
    CK(cudaStreamSynchronize(e->stream));
    CK(cudaMemcpy(out, e->d_step_trace, nl * row * 8, cudaMemcpyDeviceToHost));
    for (size_t i = 0; i < nl; ++i) types[i] = e->step_trace_types[i];
    *nphase = (int32_t)nl;
    API_END
}

// Profiling aid: time one projection launch class in isolation, round-robin over the layers so
// every launch streams cold weights.  which: 0.. = index into the pre-WKV launches, 10 = output
// projection, 20/21 = channel-mix launches, 30 = head.  Returns ms per launch and weight bytes.
int32_t b200rwkv_debug_gemm_time(b200rwkv_engine* e, int32_t which, int32_t reps, float* ms_out, int64_t* bytes_out,
                                 uint64_t* trace_out /* [L][8] stamps of CTA 0 for the last round, or null */) {
    API_BEGIN(e)
    REQUIRE(e && ms_out && bytes_out && reps >= 1, B200RWKV_ERR_INVALID, "bad argument");
    std::lock_guard<std::mutex> lk(e->mu);
    CK(cudaSetDevice(e->dev));
    auto pick = [&](int l) -> const GemmLaunch& {
        Layer& ly = e->layers[l % e->L];
        if (which == 30) return e->head;
        if (which >= 20) { REQUIRE(which - 20 < (int)ly.ffn.size(), B200RWKV_ERR_INVALID, "no such launch"); return ly.ffn[which - 20]; }
        if (which == 10) return ly.o;
        REQUIRE(which < (int)ly.pre.size(), B200RWKV_ERR_INVALID, "no such launch");
        return ly.pre[which];
    };
    // a valid 16-token meta so row masks are full
    std::vector<int> m(e->meta_ints, 0);
    m[0] = 16; m[1] = std::min(16, e->S); m[2] = 16;
    CK(cudaMemcpy(e->d_meta, m.data(), e->meta_ints * 4, cudaMemcpyHostToDevice));
    cudaEvent_t a, b;
    CK(cudaEventCreate(&a));
    CK(cudaEventCreate(&b));
    const int n = reps * e->L;
    unsigned long long* d_tr = nullptr;
    if (trace_out) { CK(cudaMalloc(&d_tr, (size_t)e->L * 16 * 8)); CK(cudaMemset(d_tr, 0, (size_t)e->L * 16 * 8)); }
    for (int i = 0; i < e->L; ++i) e->launch_gemm(pick(i), 1, e->stream, nullptr);
    CK(cudaEventRecord(a, e->stream));
    for (int i = 0; i < n; ++i) {
        GemmLaunch g = pick(i);
        if (d_tr && i >= n - e->L) g.p.trace = d_tr + (size_t)(i % e->L) * 16;
        e->launch_gemm(g, 1, e->stream, nullptr);
    }
    CK(cudaEventRecord(b, e->stream));
    CK(cudaStreamSynchronize(e->stream));
    if (d_tr) { CK(cudaMemcpy(trace_out, d_tr, (size_t)e->L * 16 * 8, cudaMemcpyDeviceToHost)); CK(cudaFree(d_tr)); }
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, a, b));
    *ms_out = ms / n;
    *bytes_out = (int64_t)pick(0).weight_bytes;
    API_END
}

#ifdef B200RWKV_DEBUG
// Streaming micro-benchmark (see streamtest.cuh).  kind 0: vector loads; kind 1: bulk-TMA ring.
int32_t b200rwkv_debug_stream(int32_t device, int32_t kind, double gbytes, int32_t stage_bytes, int32_t nstage, int32_t use_hint,
                              int32_t consumer, int32_t split, int32_t producers, int32_t reps, float* ms_out) {
    int32_t extra = 0;
    if (stage_bytes % 16384 != 0 && stage_bytes > 16384) { extra = stage_bytes % 16384; }
    API_BEGIN((b200rwkv_engine*)nullptr)
    REQUIRE(ms_out && reps >= 1, B200RWKV_ERR_INVALID, "bad argument");
    CK(cudaSetDevice(device));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    const int G = prop.multiProcessorCount;
    size_t per_cta = (size_t)(gbytes * 1e9 / G);
    per_cta = per_cta / stage_bytes * stage_bytes;
    const size_t total = per_cta * G;
    uint8_t* buf = nullptr;
    unsigned* sink = nullptr;
    CK(cudaMalloc(&buf, total + 1024));
    CK(cudaMalloc(&sink, 4));
    CK(cudaMemset(buf, 0, total));
    cudaEvent_t a, b;
    CK(cudaEventCreate(&a));
    CK(cudaEventCreate(&b));
    StreamParams sp;
    sp.src = buf; sp.bytes_per_cta = per_cta; sp.stage_bytes = stage_bytes; sp.nstage = nstage; sp.use_hint = use_hint;
    sp.consumer = consumer; sp.split = split; sp.producers = producers; sp.extra = extra;
    const size_t smem = (size_t)nstage * stage_bytes + 2 * nstage * 8 + 64;
    if (kind == 1) CK(cudaFuncSetAttribute(stream_ring_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    for (int r = 0; r < reps + 1; ++r) {
        if (r == 1) CK(cudaEventRecord(a));
        if (kind == 0) stream_ldg_kernel<<<G * 8, 256>>>(reinterpret_cast<const uint4*>(buf), total / 16, sink);
        else stream_ring_kernel<<<G, 128, smem>>>(sp);
        CK(cudaGetLastError());
    }
    CK(cudaEventRecord(b));
    CK(cudaDeviceSynchronize());
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, a, b));
    *ms_out = ms / reps;
    CK(cudaFree(buf));
    CK(cudaFree(sink));
    API_END
}

// L2 prefetch micro-benchmark (streamtest.cuh): per rep { flush L2 by streaming another buffer; prefetch kernel (+ idle);
// timed streaming kernel }.  ms_out[0] = streaming kernel alone (events around it), ms_out[1] = prefetch + idle + stream.
int32_t b200rwkv_debug_prefetch(int32_t device, double mbytes, int32_t consumers, int32_t pf_grid, int32_t skip, int32_t nblk,
                                int32_t mode, double idle_us, int32_t reps, float* ms_out) {
    API_BEGIN((b200rwkv_engine*)nullptr)
    REQUIRE(ms_out && reps >= 1 && consumers >= 1 && pf_grid >= 1, B200RWKV_ERR_INVALID, "bad argument");
    CK(cudaSetDevice(device));
    const int stage = 32768, nstage = 5;
    size_t per_cta = (size_t)(mbytes * 1e6 / consumers) / stage * stage;
    const size_t total = per_cta * consumers;
    const size_t flush_bytes = (size_t)148 * stage * 64;       // ~310 MB through the same ring kernel
    uint8_t *buf = nullptr, *fl = nullptr;
    CK(cudaMalloc(&buf, total + 1024));
    CK(cudaMalloc(&fl, flush_bytes + 1024));
    CK(cudaMemset(buf, 0, total));
    CK(cudaMemset(fl, 0, flush_bytes));
    const size_t smem = (size_t)nstage * stage + 2 * nstage * 8 + 64;
    CK(cudaFuncSetAttribute(stream_ring_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    StreamParams sp;
    memset(&sp, 0, sizeof(sp));
    sp.src = buf; sp.bytes_per_cta = per_cta; sp.stage_bytes = stage; sp.nstage = nstage; sp.use_hint = 1; sp.split = 1; sp.producers = 1;
    StreamParams fp = sp;
    fp.src = fl; fp.bytes_per_cta = (size_t)stage * 64;
    cudaEvent_t a, b, c;
    CK(cudaEventCreate(&a)); CK(cudaEventCreate(&b)); CK(cudaEventCreate(&c));
    double s0 = 0, s1 = 0;
    for (int r = 0; r < reps + 1; ++r) {
        stream_ring_kernel<<<148, 128, smem>>>(fp);
        CK(cudaEventRecord(a));
        prefetch_probe_kernel<<<pf_grid, 128>>>(buf, per_cta, consumers, skip, nblk, mode, (unsigned long long)(idle_us * 1e3));
        CK(cudaEventRecord(b));
        stream_ring_kernel<<<consumers, 128, smem>>>(sp);
        CK(cudaEventRecord(c));
        CK(cudaDeviceSynchronize());
        CK(cudaGetLastError());
        float m0 = 0.f, m1 = 0.f;
        CK(cudaEventElapsedTime(&m0, b, c));
        CK(cudaEventElapsedTime(&m1, a, c));
        if (r > 0) { s0 += m0; s1 += m1; }
    }
    ms_out[0] = (float)(s0 / reps);
    ms_out[1] = (float)(s1 / reps);
    CK(cudaFree(buf)); CK(cudaFree(fl));
    cudaEventDestroy(a); cudaEventDestroy(b); cudaEventDestroy(c);
    API_END
}

// tcgen05.mma rate of one instruction shape (streamtest.cuh): cycles[0] = issue loop, cycles[1] = until retired, for n MMAs.
int32_t b200rwkv_debug_mma_rate(int32_t device, int32_t M, int32_t N, int32_t a_in_tmem, int32_t n, int64_t* cycles) {
    API_BEGIN((b200rwkv_engine*)nullptr)
    REQUIRE((M == 64 || M == 128) && N >= 16 && N <= 256 && N % 16 == 0 && n >= 1 && cycles, B200RWKV_ERR_INVALID, "bad argument");
    CK(cudaSetDevice(device));
    const size_t smem = 32768 + 65536 + 64;
    CK(cudaFuncSetAttribute(mma_rate_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    DevTmp out(16);
    for (int r = 0; r < 2; ++r) {          // first launch warms the instruction cache
        mma_rate_kernel<<<1, 128, smem>>>(M, N, a_in_tmem, n, (long long*)out.p);
        CK(cudaGetLastError());
        CK(cudaDeviceSynchronize());
    }
    long long h[2];
    CK(cudaMemcpy(h, out.p, 16, cudaMemcpyDeviceToHost));
    cycles[0] = h[0]; cycles[1] = h[1];
    API_END
}
#endif   // B200RWKV_DEBUG

// ---- exported SPMD entries: one rank, or all ranks of an in-process tensor-parallel engine at once ----
#define RANKS(e, call_r) ((e) && (e)->group ? (e)->group->spmd([&](int r_) -> int32_t { b200rwkv_engine* er = (e)->group->ranks[r_]; (void)er; return call_r; }) : [&]() -> int32_t { b200rwkv_engine* er = (e); const int r_ = 0; (void)r_; return call_r; }())

int32_t b200rwkv_infer(b200rwkv_engine* e, int32_t nslot, const int32_t* slot, const int32_t* ntok, const uint32_t* tokens,
                       const int32_t* option, float* logits_out, size_t logits_cap, int32_t* rows_out) {
    return RANKS(e, rank_infer(er, nslot, slot, ntok, tokens, option, r_ == 0 ? logits_out : nullptr, r_ == 0 ? logits_cap : 0,
                               r_ == 0 ? rows_out : nullptr));
}
int32_t b200rwkv_infer_score(b200rwkv_engine* e, int32_t nslot, const int32_t* slot, const int32_t* ntok, const uint32_t* tokens,
                             const int32_t* option, float* logits_out, size_t logits_cap, int32_t* rows_out, float* logp_out,
                             size_t logp_cap) {
    // every in-process rank is handed logp_out so that its argument checks agree with rank 0's; only rank 0 writes it
    return RANKS(e, rank_infer(er, nslot, slot, ntok, tokens, option, r_ == 0 ? logits_out : nullptr, r_ == 0 ? logits_cap : 0,
                               r_ == 0 ? rows_out : nullptr, logp_out, logp_cap, true));
}
int32_t b200rwkv_state_load(b200rwkv_engine* e, int32_t slot, const float* in) { return RANKS(e, rank_state_load(er, slot, in)); }

// head-sharded state: every rank exports the WKV rows of its own heads (zeros elsewhere); the shift rows are replicated
static void merge_state_columns(const b200rwkv_engine* lead, float* out, const float* part, int r) {
    const int C = lead->C, N = lead->N, Cl = lead->Cl;
    for (int l = 0; l < lead->L; ++l)
        for (int row = 1; row <= N; ++row) {
            const size_t o = ((size_t)l * (N + 2) + row) * C + (size_t)r * Cl;
            memcpy(out + o, part + o, (size_t)Cl * 4);
        }
}
int32_t b200rwkv_state_back(b200rwkv_engine* e, int32_t slot, float* out) {
    if (!e || !e->group) return rank_state_back(e, slot, out);
    const size_t n = (size_t)e->L * (e->N + 2) * e->C;
    std::vector<std::vector<float>> part(e->group->ranks.size());
    for (size_t r = 1; r < part.size(); ++r) part[r].resize(n);
    const int32_t st = e->group->spmd([&](int r) { return rank_state_back(e->group->ranks[r], slot, r == 0 ? out : part[r].data()); });
    if (st < 0 || !out) return st;
    for (size_t r = 1; r < part.size(); ++r) merge_state_columns(e, out, part[r].data(), (int)r);
    return st;
}
int32_t b200rwkv_state_read(b200rwkv_engine* e, int32_t slot, uint64_t* snapshot_id) {
    if (!e || !e->group) return rank_state_read(e, slot, snapshot_id);
    // every rank snapshots its shard; the ranks' id counters advance in lockstep, so the ids agree
    std::vector<uint64_t> ids(e->group->ranks.size(), 0);
    const int32_t st = e->group->spmd([&](int r) { return rank_state_read(e->group->ranks[r], slot, &ids[r]); });
    if (st < 0) return st;
    for (uint64_t id : ids)
        if (id != ids[0]) { g_err = "internal: snapshot ids diverged across ranks"; return B200RWKV_ERR_STATE; }
    if (snapshot_id) *snapshot_id = ids[0];
    return st;
}
int32_t b200rwkv_state_write(b200rwkv_engine* e, int32_t slot, uint64_t id) { return RANKS(e, rank_state_write(er, slot, id)); }
int32_t b200rwkv_state_free(b200rwkv_engine* e, uint64_t id) { return RANKS(e, rank_state_free(er, id)); }
int32_t b200rwkv_snapshot_back(b200rwkv_engine* e, uint64_t id, float* state_out, float* logits_out) {
    if (!e || !e->group) return rank_snapshot_back(e, id, state_out, logits_out);
    const size_t n = (size_t)e->L * (e->N + 2) * e->C;
    std::vector<std::vector<float>> part(e->group->ranks.size());
    for (size_t r = 1; r < part.size(); ++r) part[r].resize(state_out ? n : 0);
    const int32_t st = e->group->spmd([&](int r) {
        if (r == 0) return rank_snapshot_back(e, id, state_out, logits_out);
        return state_out ? rank_snapshot_back(e->group->ranks[r], id, part[r].data(), nullptr) : (int32_t)B200RWKV_OK;
    });
    if (st < 0 || !state_out) return st;
    for (size_t r = 1; r < part.size(); ++r) merge_state_columns(e, state_out, part[r].data(), (int)r);
    return st;
}
int32_t b200rwkv_snapshot_load(b200rwkv_engine* e, const float* state_in, const float* logits_in, uint64_t* snapshot_id) {
    if (!e || !e->group) return rank_snapshot_load(e, state_in, logits_in, snapshot_id);
    std::vector<uint64_t> ids(e->group->ranks.size(), 0);
    // every rank records whether a row came with the state; only rank 0 keeps rows and reads logits_in
    const int32_t st = e->group->spmd([&](int r) { return rank_snapshot_load(e->group->ranks[r], state_in, logits_in, &ids[r]); });
    if (st < 0) return st;
    for (uint64_t id : ids)
        if (id != ids[0]) { g_err = "internal: snapshot ids diverged across ranks"; return B200RWKV_ERR_STATE; }
    if (snapshot_id) *snapshot_id = ids[0];
    return st;
}
int32_t b200rwkv_bench_decode(b200rwkv_engine* e, int32_t nslot, const int32_t* slot, const uint32_t* tokens, int32_t warmup,
                              int32_t steps, int32_t flush_l2, float* ms_out, int64_t* launches_out, float* step_ms_out) {
    if (!e || !e->group) return rank_bench_decode(e, nslot, slot, tokens, warmup, steps, flush_l2, ms_out, launches_out, step_ms_out);
    const size_t W = e->group->ranks.size();
    std::vector<float> ms(W, 0.f);
    std::vector<int64_t> ln(W, 0);
    const int32_t st = e->group->spmd([&](int r) {
        return rank_bench_decode(e->group->ranks[r], nslot, slot, tokens, warmup, steps, flush_l2, &ms[r], &ln[r], r == 0 ? step_ms_out : nullptr);
    });
    if (st < 0) return st;
    if (ms_out) *ms_out = *std::max_element(ms.begin(), ms.end());        // a step is done when the slowest rank is
    if (launches_out) *launches_out = ln[0];
    return st;
}
int32_t b200rwkv_profile_step(b200rwkv_engine* e, int32_t nslot, const int32_t* slot, const uint32_t* tokens, float ms[4],
                              int32_t launches[4], int64_t* gemm_weight_bytes) {
    if (!e || !e->group) return rank_profile_step(e, nslot, slot, tokens, ms, launches, gemm_weight_bytes);
    const size_t W = e->group->ranks.size();
    std::vector<float> m4(4 * W);
    std::vector<int32_t> l4(4 * W);
    std::vector<int64_t> wb(W);
    const int32_t st = e->group->spmd([&](int r) { return rank_profile_step(e->group->ranks[r], nslot, slot, tokens, &m4[4 * r], &l4[4 * r], &wb[r]); });
    if (st < 0) return st;
    for (int i = 0; i < 4; ++i) { ms[i] = m4[i]; launches[i] = l4[i]; }
    if (gemm_weight_bytes) *gemm_weight_bytes = wb[0];
    return st;
}
int32_t b200rwkv_profile_insitu(b200rwkv_engine* e, int32_t nslot, const int32_t* slot, const uint32_t* tokens, int32_t reps,
                                int32_t cap, int32_t* n_out, int32_t* types, double* start_us, double* end_us, int64_t* bytes,
                                double* step_us) {
    if (!e || !e->group) return rank_profile_insitu(e, nslot, slot, tokens, reps, cap, n_out, types, start_us, end_us, bytes, step_us);
    const size_t W = e->group->ranks.size();
    std::vector<std::vector<int32_t>> ty(W, std::vector<int32_t>(cap));
    std::vector<std::vector<double>> su(W, std::vector<double>(cap)), eu(W, std::vector<double>(cap));
    std::vector<std::vector<int64_t>> by(W, std::vector<int64_t>(cap));
    std::vector<int32_t> nn(W, 0);
    std::vector<double> sus(W, 0.0);
    const int32_t st = e->group->spmd([&](int r) {
        if (r == 0) return rank_profile_insitu(e, nslot, slot, tokens, reps, cap, n_out, types, start_us, end_us, bytes, step_us);
        return rank_profile_insitu(e->group->ranks[r], nslot, slot, tokens, reps, cap, &nn[r], ty[r].data(), su[r].data(), eu[r].data(), by[r].data(), &sus[r]);
    });
    return st;
}
#undef RANKS

// Replaces `ModelBuilder...build_vN()` + `Bundle::new` + `TokioRuntime::new` (lib.rs:484-497) with everything the reference's
// ReloadRequest carries for this path: devices (one engine object owning all tensor-parallel ranks, SURVEY.md §8b), LoRA files
// (lib.rs:466-485), precision (lib.rs:493).
int32_t b200rwkv_create_ex(const uint8_t* st, size_t len, const b200rwkv_options* opt, b200rwkv_engine** out) {
    if (!out || !opt) { g_err = "null argument"; return B200RWKV_ERR_INVALID; }
    *out = nullptr;
    if (opt->struct_bytes != sizeof(b200rwkv_options)) { g_err = "b200rwkv_options.struct_bytes does not match this library"; return B200RWKV_ERR_INVALID; }
    const int world = opt->num_devices <= 0 ? 1 : opt->num_devices;
    if (!(world == 1 || world == 2 || world == 4 || world == 8)) { g_err = "num_devices must be 1, 2, 4 or 8"; return B200RWKV_ERR_INVALID; }
    if (opt->num_lora < 0 || opt->num_lora > B200RWKV_MAX_LORA) { g_err = "bad num_lora"; return B200RWKV_ERR_INVALID; }
    std::vector<LoraArg> lora;
    for (int i = 0; i < opt->num_lora; ++i) lora.push_back({opt->lora_st[i], opt->lora_len[i], opt->lora_alpha[i]});
    const int dev0 = opt->num_devices <= 0 ? 0 : opt->devices[0];
    if (world == 1)
        return create_rank(st, len, dev0, opt->max_batch, opt->token_chunk_size, opt->precision, 0, 1, lora, out, opt->quant_layers, opt->quant_type);
    if (opt->quant_layers > 0 && opt->quant_type != B200RWKV_QUANT_NONE) { g_err = "quantised layers are single-GPU in this version"; return B200RWKV_ERR_UNSUPPORTED; }
    for (int r = 0; r < world; ++r)
        for (int q = 0; q < r; ++q)
            if (opt->devices[r] == opt->devices[q]) { g_err = "devices must be distinct"; return B200RWKV_ERR_INVALID; }
    // build all ranks concurrently (each uploads and re-tiles its own shard), then wire them
    std::unique_ptr<Group> g(new Group());
    g->ranks.assign(world, nullptr);
    g->start(world);
    const int32_t st_build = g->spmd([&](int r) {
        return create_rank(st, len, opt->devices[r], opt->max_batch, opt->token_chunk_size, opt->precision, r, world, lora, &g->ranks[r]);
    });
    int32_t rc = st_build;
    if (rc >= 0) rc = b200rwkv_tp_connect_local(g->ranks.data(), world);
    if (rc < 0) {
        const std::string msg = g_err;
        g->shutdown();
        for (auto* p : g->ranks) delete p;
        g_err = msg;
        return rc;
    }
    b200rwkv_engine* lead = g->ranks[0];
    lead->group = std::move(g);
    *out = lead;
    return B200RWKV_OK;
}

const char* b200rwkv_last_error(b200rwkv_engine* e) { (void)e; return g_err.c_str(); }

}  // extern "C"
