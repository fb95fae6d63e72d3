// C-ABI glue: globals, error reporting, conv entry points and kernel selection.
#include "conv_internal.cuh"
#include <mutex>

namespace sae {

thread_local char g_err[512] = "";
std::atomic<int64_t> g_launches{0};

int sm_count() {
    static int n = 0;
    static std::once_flag once;
    std::call_once(once, [] {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess) dev = 0;
        cudaDeviceProp prop;
        if (cudaGetDeviceProperties(&prop, dev) == cudaSuccess) n = prop.multiProcessorCount;
        if (n <= 0) n = 148;
    });
    return n;
}

float* det_workspace(size_t nfloats) {
    constexpr int kMaxDevices = 64;
    static std::mutex mu;
    static float* buf[kMaxDevices] = {};
    static size_t cap[kMaxDevices] = {};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= kMaxDevices) {
        fail(SAE_E_CUDA, "deterministic-reduction workspace: no current device");
        return nullptr;
    }
    std::lock_guard<std::mutex> lock(mu);
    if (cap[dev] < nfloats) {
        // Allocated on first use, at least 64 MB: enough for every reduction of the default 256x256 training step.  The eager
        // half-steps that precede a graph capture size it; a capture that needed more would fail at cudaMalloc, and graphs.py
        // then runs that half-step eagerly.
        size_t want = nfloats + nfloats / 4;
        if (want < ((size_t)16 << 20)) want = (size_t)16 << 20;
        void* p = nullptr;
        cudaError_t e = cudaMalloc(&p, want * sizeof(float));
        if (e != cudaSuccess) {
            cudaGetLastError();
            fail(SAE_E_CUDA, "deterministic-reduction workspace of %zu bytes: %s", want * sizeof(float), cudaGetErrorString(e));
            return nullptr;
        }
        buf[dev] = static_cast<float*>(p);     // the previous buffer stays allocated: captured graphs may still use it
        cap[dev] = want;
    }
    return buf[dev];
}

constexpr int DR_COLS = 32, DR_MAX_ROWS = 8;

// grid = (column blocks, part groups), block = (32, rows).  Group g sums parts [g * per, min(parts, (g + 1) * per)): row r takes
// every rows-th part from g * per + r, then row 0 adds the rows in order.  With ws2 the group sums go to ws2[g * n + c],
// otherwise (one group) they are added to the destination.
__global__ void det_reduce_kernel(const float* __restrict__ ws, int64_t n, int parts, int per, float* __restrict__ ws2,
                                  float* a, int64_t n_a, float* b) {
    __shared__ float red[DR_MAX_ROWS][DR_COLS + 1];
    const int64_t col = (int64_t)blockIdx.x * DR_COLS + threadIdx.x;
    const int b0 = (int)blockIdx.y * per;
    const int b1 = min(b0 + per, parts);
    float s = 0.f;
    if (col < n)
        for (int k = b0 + (int)threadIdx.y; k < b1; k += (int)blockDim.y) s += ws[(int64_t)k * n + col];
    red[threadIdx.y][threadIdx.x] = s;
    __syncthreads();
    if (threadIdx.y != 0 || col >= n) return;
    float t = red[0][threadIdx.x];
    for (int r = 1; r < (int)blockDim.y; ++r) t += red[r][threadIdx.x];
    if (ws2 != nullptr) {
        ws2[(int64_t)blockIdx.y * n + col] = t;
        return;
    }
    float* dst = col < n_a ? (a ? a + col : nullptr) : (b ? b + (col - n_a) : nullptr);
    if (dst) *dst += t;
}

static int det_groups(int64_t n, int parts) {
    // many parts over few columns (per-block bias sums): a first pass over part groups fills the machine
    if (parts <= 64) return 1;
    const int64_t col_blocks = (n + DR_COLS - 1) / DR_COLS;
    int64_t g = ((int64_t)sm_count() * 4 + col_blocks - 1) / col_blocks;
    if (g > parts / 32) g = parts / 32;
    return g < 1 ? 1 : (int)g;
}

size_t det_reduce_floats(int64_t n, int parts) {
    const int g = det_groups(n, parts);
    return (size_t)parts * n + (g > 1 ? (size_t)g * n : 0);
}

int det_reduce(float* a, int64_t n_a, float* b, const float* ws, int64_t n, int parts, cudaStream_t st) {
    if (n <= 0 || parts <= 0) return SAE_OK;
    int g = det_groups(n, parts);
    const int per = (parts + g - 1) / g;
    g = (parts + per - 1) / per;
    const unsigned col_blocks = (unsigned)((n + DR_COLS - 1) / DR_COLS);
    if (g > 1) {
        float* ws2 = const_cast<float*>(ws) + (int64_t)parts * n;
        det_reduce_kernel<<<dim3(col_blocks, (unsigned)g), dim3(DR_COLS, DR_MAX_ROWS), 0, st>>>(ws, n, parts, per, ws2, a, n_a, b);
        int rc = check_launch("det_reduce (groups)");
        if (rc) return rc;
        ws = ws2;
        parts = g;
    }
    const unsigned rows = (unsigned)(parts < DR_MAX_ROWS ? parts : DR_MAX_ROWS);
    det_reduce_kernel<<<dim3(col_blocks, 1), dim3(DR_COLS, rows), 0, st>>>(ws, n, parts, parts, nullptr, a, n_a, b);
    return check_launch("det_reduce");
}

static int validate_geom(const sae_conv_geom* g, const char* who) {
    if (!g) return fail(SAE_E_INVALID, "%s: null geometry", who);
    if (g->N < 0 || g->H <= 0 || g->W <= 0 || g->C <= 0 || g->K <= 0 || g->R <= 0 || g->S <= 0 || g->P <= 0 ||
        g->Q <= 0 || g->stride <= 0)
        return fail(SAE_E_INVALID, "%s: non-positive dimension", who);
    // the last output row/column must start inside the padded input
    if ((int64_t)(g->P - 1) * g->stride - g->pad_t + g->R - 1 < 0 || (int64_t)(g->Q - 1) * g->stride - g->pad_l + g->S - 1 < 0)
        return fail(SAE_E_INVALID, "%s: inconsistent P/Q", who);
    return SAE_OK;
}

}  // namespace sae

using namespace sae;

extern "C" int sae_abi_version(void) { return SAE_ABI_VERSION; }
extern "C" const char* sae_last_error(void) { return g_err; }
extern "C" int64_t sae_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }
extern "C" int sae_tcgen05_available(void) { return tc_available() ? 1 : 0; }

extern "C" int sae_conv2d_query_impl(const sae_conv_geom* g, int dir) {
    if (validate_geom(g, "query_impl") != SAE_OK) return SAE_E_INVALID;
    if (!tc_available()) return 1;
    bool ok = dir == 0 ? tc_fprop_eligible(g) : dir == 1 ? tc_dgrad_eligible(g) : tc_wgrad_eligible(g);
    return ok ? 2 : 1;
}

extern "C" int sae_conv2d_fprop(const float* x, const float* w, float* y, const sae_conv_geom* g,
                                const sae_conv_epilogue* epi, int impl, void* stream) {
    int rc = validate_geom(g, "conv2d_fprop");
    if (rc) return rc;
    if (g->N == 0) return SAE_OK;
    if (!x || !w || !y) return fail(SAE_E_INVALID, "conv2d_fprop: null pointer");
    cudaStream_t st = (cudaStream_t)stream;
    EpiParams e = make_epi(epi);
    const bool tc_ok = tc_available() && tc_fprop_eligible(g);
    if (impl == 2 && !tc_ok) return fail(SAE_E_UNSUPPORTED, "conv2d_fprop: shape not eligible for the tcgen05 kernel");
    if (impl != 1 && tc_ok) return tc_fprop(x, w, y, g, e, st);
    GatherParams p;
    p.N = g->N; p.OH = g->P; p.OW = g->Q; p.IH = g->H; p.IW = g->W; p.Cs = g->C; p.R = g->R; p.S = g->S;
    p.SY = g->stride; p.DY = 1; p.OFFY = -g->pad_t; p.OFFX = -g->pad_l; p.DIV = 1;
    p.Ncol = g->K; p.K = g->R * g->S * g->C; p.M = (int64_t)g->N * g->P * g->Q;
    return conv_gather_dispatch(x, w, y, p, e, st);
}

extern "C" int sae_conv2d_dgrad(const float* dy, const float* wt, float* dx, const sae_conv_geom* g,
                                const sae_conv_epilogue* epi, int impl, void* stream) {
    int rc = validate_geom(g, "conv2d_dgrad");
    if (rc) return rc;
    if (g->N == 0) return SAE_OK;
    if (!dy || !wt || !dx) return fail(SAE_E_INVALID, "conv2d_dgrad: null pointer");
    cudaStream_t st = (cudaStream_t)stream;
    EpiParams e = make_epi(epi);
    const bool tc_ok = tc_available() && tc_dgrad_eligible(g);
    if (impl == 2 && !tc_ok) return fail(SAE_E_UNSUPPORTED, "conv2d_dgrad: shape not eligible for the tcgen05 kernel");
    if (impl != 1 && tc_ok) return tc_dgrad(dy, wt, dx, g, e, st);
    GatherParams p;
    p.N = g->N; p.OH = g->H; p.OW = g->W; p.IH = g->P; p.IW = g->Q; p.Cs = g->K; p.R = g->R; p.S = g->S;
    p.SY = 1; p.DY = -1; p.OFFY = g->pad_t; p.OFFX = g->pad_l; p.DIV = g->stride;
    p.Ncol = g->C; p.K = g->R * g->S * g->K; p.M = (int64_t)g->N * g->H * g->W;
    return conv_gather_dispatch(dy, wt, dx, p, e, st);
}

extern "C" int sae_conv2d_wgrad(const float* dy, const float* x, float* dw, const sae_conv_geom* g,
                                int impl, void* stream) {
    int rc = validate_geom(g, "conv2d_wgrad");
    if (rc) return rc;
    if (g->N == 0) return SAE_OK;
    if (!dy || !x || !dw) return fail(SAE_E_INVALID, "conv2d_wgrad: null pointer");
    cudaStream_t st = (cudaStream_t)stream;
    const bool tc_ok = tc_available() && tc_wgrad_eligible(g);
    if (impl == 2 && !tc_ok) return fail(SAE_E_UNSUPPORTED, "conv2d_wgrad: shape not eligible for the tcgen05 kernel");
    if (impl != 1 && tc_ok) return tc_wgrad(dy, x, dw, g, st);
    return conv_wgrad_generic(dy, x, dw, g, st);
}

// ---- style-modulated convolution with per-sample filters (no modulated copy of the activation) --------------------------
extern "C" int sae_conv2d_query_modulated(const sae_conv_geom* g) {
    if (validate_geom(g, "query_modulated") != SAE_OK) return 0;
    return (tc_available() && tc_per_sample_eligible(g, 0) && tc_per_sample_eligible(g, 1) && tc_wgrad_modulated_eligible(g)) ? 1 : 0;
}

extern "C" int sae_conv2d_fprop_per_sample(const float* x, const float* w_nkrsc, float* y, const sae_conv_geom* g,
                                           const sae_conv_epilogue* epi, void* stream) {
    int rc = validate_geom(g, "conv2d_fprop_per_sample");
    if (rc) return rc;
    if (g->N == 0) return SAE_OK;
    if (!x || !w_nkrsc || !y) return fail(SAE_E_INVALID, "conv2d_fprop_per_sample: null pointer");
    if (!tc_available()) return fail(SAE_E_UNSUPPORTED, "conv2d_fprop_per_sample: needs the tcgen05 path");
    return tc_conv_per_sample(x, w_nkrsc, y, g, 0, make_epi(epi), (cudaStream_t)stream);
}

extern "C" int sae_conv2d_dgrad_per_sample(const float* dy, const float* w_ncrsk, float* dx, const sae_conv_geom* g,
                                           const sae_conv_epilogue* epi, void* stream) {
    int rc = validate_geom(g, "conv2d_dgrad_per_sample");
    if (rc) return rc;
    if (g->N == 0) return SAE_OK;
    if (!dy || !w_ncrsk || !dx) return fail(SAE_E_INVALID, "conv2d_dgrad_per_sample: null pointer");
    if (!tc_available()) return fail(SAE_E_UNSUPPORTED, "conv2d_dgrad_per_sample: needs the tcgen05 path");
    return tc_conv_per_sample(dy, w_ncrsk, dx, g, 1, make_epi(epi), (cudaStream_t)stream);
}

extern "C" int sae_conv2d_wgrad_modulated(const float* dy, const float* x, const float* s, const float* w_krsc, float* dw, float* ds,
                                          const sae_conv_geom* g, void* stream) {
    int rc = validate_geom(g, "conv2d_wgrad_modulated");
    if (rc) return rc;
    if (g->N == 0) return SAE_OK;
    if (!dy || !x || !s || !w_krsc || !dw || !ds) return fail(SAE_E_INVALID, "conv2d_wgrad_modulated: null pointer");
    if (!tc_available()) return fail(SAE_E_UNSUPPORTED, "conv2d_wgrad_modulated: needs the tcgen05 path");
    return tc_wgrad_modulated(dy, x, s, w_krsc, dw, ds, g, (cudaStream_t)stream);
}
