// Launch layer of the WIDE tcgen05 channel half (mmx_chan_wide.cuh): 80 <= max(H, ch) <= 128 -- K4 (AMASS-shaped MlpMixer,
// H = 128) and the H = 128 cells of the large-batch sweep.  Called from mmx_api_mlp_tc5.cu's channel dispatch.
//
// Workspace: the prep kernel's output (W1' and W2 split into bf16 hi / lo planes in the operand layout, b1') lives in a
// device buffer owned by the library, ONE PER (device, weight matrix): keyed by the fc1 weight pointer, so two streams that
// run the same block concurrently write identical bytes and different blocks never share a buffer.  Buffers are allocated on
// first use (cudaMalloc: not legal while a stream capture is under way -- run the step once eagerly first, as TrainStep does)
// and live until the process ends (captured CUDA graphs hold their addresses, so they are never freed: 129 KB per distinct fc1
// weight matrix the process ever runs).
#include "mmx_launch.cuh"

#if defined(MMX_HOST_EMU)
int mmx_chan_wide_run(bool, int, const void*, void*) { return fail(MMX_E_UNSUPPORTED, "no tensor cores in the emulator"); }
#else
#include <mutex>
#include <unordered_map>

#include "mmx_chan_wide.cuh"

using namespace mmx;

static int wide_workspace(const float* key, uint8_t** out) {
    struct KeyHash {
        size_t operator()(const std::pair<int, const void*>& k) const { return std::hash<const void*>()(k.second) ^ ((size_t)k.first * 0x9E3779B97F4A7C15ull); }
    };
    static std::unordered_map<std::pair<int, const void*>, uint8_t*, KeyHash> pool;
    static std::mutex mu;
    int dev = 0;
    cudaGetDevice(&dev);
    std::lock_guard<std::mutex> lk(mu);
    auto it = pool.find({dev, key});
    if (it != pool.end()) { *out = it->second; return MMX_OK; }
    void* p = nullptr;
    cudaError_t e = cudaMalloc(&p, chanw::kWsBytes);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(MMX_E_CUDA, "wide channel half: workspace allocation failed (%s); if a CUDA graph is being captured, run the step once eagerly first",
                    cudaGetErrorString(e));
    }
    pool[{dev, key}] = (uint8_t*)p;
    *out = (uint8_t*)p;
    return MMX_OK;
}

template <int ACT, int VEC, int KP>
static int run_wide(bool bwd, const chan::ChanArgs& c, void* stream) {
    const DevInfo di = dev_info();
    const chan::Geo g = chan::make_geo(c.T, c.H, VEC);
    const size_t smem = chanw::wide_smem<KP>(g, bwd).total;
    if (smem > (size_t)di.max_smem) return fail(MMX_E_UNSUPPORTED, "wide channel half: tile does not fit shared memory (H=%d ch=%d)", c.H, c.ch);
    uint8_t* ws = nullptr;
    int rc = wide_workspace(c.w1, &ws);
    if (rc) return rc;
    if ((rc = launch_kernel(chanw::chan_prep_kernel<KP>, KP <= 64 ? 8 : 32, 256, 0, stream, kPdl, c, ws))) return rc;
    const int ntiles = (c.B + g.seq_per_tile - 1) / g.seq_per_tile;
    // KP = 128: 512 TMEM columns, ~205 KB shared -> one CTA per SM; KP = 64: 256 columns, < 100 KB -> two CTAs per SM
    const int per_sm = KP <= 64 ? ctas_per_sm(di, smem, 2) : 1;
    const int grid = balanced_grid(ntiles, di.sms * per_sm);
    const uint8_t* wsc = ws;
    return launch_kernel(bwd ? chanw::chan_wide_bwd_kernel<ACT, VEC, KP> : chanw::chan_wide_fwd_kernel<ACT, VEC, KP>, grid, tc5::kCtaThreads, smem,
                         stream, kPdl, c, wsc);
}

template <int KP>
static int run_wide_kp(bool bwd, int act, const chan::ChanArgs& c, void* stream) {
    const bool vec4 = (c.H & 3) == 0;
    if (act == MMX_ACT_GELU) return vec4 ? run_wide<ACT_GELU, 4, KP>(bwd, c, stream) : run_wide<ACT_GELU, 2, KP>(bwd, c, stream);
    return vec4 ? run_wide<ACT_MISH, 4, KP>(bwd, c, stream) : run_wide<ACT_MISH, 2, KP>(bwd, c, stream);
}

// act: MMX_ACT_*; args: const chan::ChanArgs*.  Operand width 64 (H, ch <= 64: two CTAs per SM) or 128.
int mmx_chan_wide_run(bool bwd, int act, const void* args, void* stream) {
    const chan::ChanArgs& c = *static_cast<const chan::ChanArgs*>(args);
    if ((c.H & 1) || (c.ch & 1) || c.H > chanw::KPW || c.ch > chanw::KPW) return fail(MMX_E_UNSUPPORTED, "wide channel half: H, ch even and <= %d", chanw::KPW);
    if (c.H <= 64 && c.ch <= 64) return run_wide_kp<64>(bwd, act, c, stream);
    return run_wide_kp<128>(bwd, act, c, stream);
}
#endif
