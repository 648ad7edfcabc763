// extern "C" surface of libcfp (declared in include/cfp.h): argument validation, workspace
// partitioning and the per-layer launch sequences.  No device allocation, no synchronisation,
// no global mutable state (the error message is thread-local).
#include <algorithm>
#include <climits>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <atomic>
#include <mutex>
#include <string>
#include <vector>
#include "cfp_common.cuh"
#include "cfp_internal.h"

namespace cfp {

ErrorState& tls_error() {
    static thread_local ErrorState e = {{0}};
    return e;
}
int fail(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(tls_error().msg, sizeof(tls_error().msg), fmt, ap);
    va_end(ap);
    return 1;
}
static thread_local int tl_pdl = -1;      // -1: default (on unless CFP_NO_PDL is set); 0 / 1: cfp_set_pdl
bool pdl_enabled() {
    static const bool env_on = getenv("CFP_NO_PDL") == nullptr;
    return tl_pdl < 0 ? env_on : (tl_pdl != 0 && env_on);
}
int sm_count() {
    static thread_local int cached_dev = -1, cached = 0;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 148;
    if (dev != cached_dev) {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
        cached_dev = dev;
        cached = n;
    }
    return cached;
}
// Launch accounting and the optional event profiler (cfp_profile_*), process-wide: a training step enqueues its forward
// from the caller's thread and its backward from autograd's device thread, and both belong in one count / one profile.
// When profiling is on, one CUDA event is recorded on the call's stream after every kernel launch and one at the start of
// every API call; a kernel's time is the gap to the previous event (meaningful when the profiled calls share one in-order
// stream).  The call-start marker keeps the time the device idles between two calls of a launch-bound caller (small
// batches through Python: ~20 us per call) out of the next kernel's figure; on a saturated stream it fires right behind
// the previous kernel and changes nothing.
struct ProfileState {
    std::mutex mu;
    std::atomic<int64_t> launches{0};
    std::atomic<bool> profiling{false};
    cudaEvent_t first = nullptr;
    std::vector<std::pair<const char*, cudaEvent_t>> events;
};
static ProfileState& pstate() {
    static ProfileState p;
    return p;
}
static thread_local cudaStream_t tl_stream = nullptr;
static void begin_call(void* stream) {
    tl_stream = (cudaStream_t)stream;
    ProfileState& p = pstate();
    if (p.profiling.load(std::memory_order_relaxed)) {
        cudaEvent_t ev;
        cudaEventCreate(&ev);
        cudaEventRecord(ev, tl_stream);
        std::lock_guard<std::mutex> lk(p.mu);
        p.events.emplace_back(nullptr, ev);          // marker: not a kernel
    }
}
int check_launch(const char* what) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail("%s launch failed: %s", what, cudaGetErrorString(e));
    ProfileState& p = pstate();
    p.launches.fetch_add(1, std::memory_order_relaxed);
    if (p.profiling.load(std::memory_order_relaxed)) {
        cudaEvent_t ev;
        cudaEventCreate(&ev);
        cudaEventRecord(ev, tl_stream);
        std::lock_guard<std::mutex> lk(p.mu);
        p.events.emplace_back(what, ev);
    }
    return 0;
}

static inline size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

WsLayout ws_layout(int B, int H, int W, int C, int ws, int large_kernel, int dtype, const cfp_geom* g) {
    WsLayout L{};
    const size_t es = elem_size(dtype);
    const int Z = g ? g->zone_num * g->zone_num : 64;
    const size_t nwin = ws > 0 ? (size_t)((H + ws - 1) / ws) * ((W + ws - 1) / ws) : 0;
    const size_t zone_state = (size_t)B * Z * ((size_t)C * (C / 4) + C);      // hist2image / DAPM, 4 heads
    const size_t win_state = (size_t)B * nwin * ((size_t)C * (C / 8) + C);    // LSA / GSA, 8 heads
    size_t off = 0;
    L.kv = off;
    L.kv_bytes = align256((zone_state > win_state ? zone_state : win_state) * sizeof(float));
    off += L.kv_bytes;
    L.tok_bytes = align256((size_t)B * H * W * C * es);
    L.tok_a = off; off += L.tok_bytes;
    L.tok_b = off; off += L.tok_bytes;
    L.sr = off;
    L.sr_bytes = ws > 0 ? align256((size_t)B * (H / ws) * (W / ws) * C * sizeof(float)) : 0;
    off += L.sr_bytes;
    L.canvas = off;
    L.canvas_bytes = (g && g->interpolate) ? align256((size_t)B * Z * g->p1 * g->p2 * C * es) : 0;
    off += L.canvas_bytes;
    L.planes = off;
    L.planes_bytes = (dtype == CFP_BF16 && large_kernel > 0) ? align256(dwconv_tc_plane_bytes(B, H, W, C, large_kernel)) : 0;
    off += L.planes_bytes;
    L.total = off;
    return L;
}

static int check_common(const void* p, int B, int H, int W, int C, int dtype) {
    CFP_REQUIRE(p != nullptr, "null device pointer");
    CFP_REQUIRE(B > 0 && H > 0 && W > 0, "bad shape B=%d H=%d W=%d", B, H, W);
    CFP_REQUIRE(C == 32 || C == 64 || C == 128, "unsupported embedding_dim C=%d (decoder.py:90-94 uses 32/64/128)", C);
    CFP_REQUIRE(dtype == CFP_F32 || dtype == CFP_BF16, "unsupported dtype %d", dtype);
    return 0;
}
// Rows of the zone canvas must map one-to-one onto the zone rectangle (fusion.py:112-120,157): with no padding the
// reference's pad_mask is all ones (fusion.py:119-120), so nothing of the canvas may overhang the map.
static int check_canvas(const cfp_geom* g, int H, int W) {
    int top = g->sy_wo < 0 ? -g->sy_wo : 0, left = g->sx_wo < 0 ? -g->sx_wo : 0;
    int bot = g->ey_wo > H ? g->ey_wo - H : 0, right = g->ex_wo > W ? g->ex_wo - W : 0;
    if (g->pad_h == 0 && g->pad_w == 0) top = left = bot = right = 0;
    CFP_REQUIRE(g->tzh - top - bot == g->ry1 - g->ry0 && g->tzw - left - right == g->rx1 - g->rx0,
                "in-image canvas cells do not match the zone rectangle (the reference's index_put fails here too)");
    return 0;
}
static int check_geom(const cfp_geom* g, int H, int W) {
    CFP_REQUIRE(g != nullptr, "null geometry");
    CFP_REQUIRE(g->zone_num > 0 && g->p1 > 0 && g->p2 > 0 && g->tzh > 0 && g->tzw > 0, "degenerate zone geometry");
    CFP_REQUIRE(0 <= g->ry0 && g->ry0 <= g->ry1 && g->ry1 <= H && 0 <= g->rx0 && g->rx0 <= g->rx1 && g->rx1 <= W,
                "zone rectangle [%d:%d,%d:%d] outside the %dx%d map", g->ry0, g->ry1, g->rx0, g->rx1, H, W);
    CFP_REQUIRE(g->interpolate || (g->tzh == g->zone_num * g->p1 && g->tzw == g->zone_num * g->p2),
                "canvas %dx%d != zone_num*patch and interpolate flag not set", g->tzh, g->tzw);
    return 0;
}

}  // namespace cfp

using namespace cfp;

extern "C" {

CFP_API int cfp_version(void) { return CFP_ABI_VERSION; }
CFP_API const char* cfp_last_error(void) { return tls_error().msg; }

// One workspace serves every entry point of a level.  cfp_twins_fwd / cfp_lkpm_fwd take no geometry and lay the
// workspace out for the default 64 zones, cfp_d2i_fwd / cfp_dapm_fwd for zone_num^2: the size handed out covers both
// (with fewer than 64 zones - the reference's 6x6 training layout - the geometry-less layout is the larger one and
// those two calls used to refuse the workspace).
CFP_API size_t cfp_workspace_bytes(int B, int H, int W, int C, int ws, int large_kernel, int dtype, const cfp_geom* g) {
    const size_t with_g = ws_layout(B, H, W, C, ws, large_kernel, dtype, g).total;
    const size_t without = ws_layout(B, H, W, C, ws, large_kernel, dtype, nullptr).total;
    return with_g > without ? with_g : without;
}

CFP_API int cfp_geometry_from_rects(const float* rects, int B, int Z, int max_width, int H, int W, cfp_geom* out) {
    CFP_REQUIRE(rects && out, "null pointer");
    CFP_REQUIRE(B > 0 && Z > 0 && H > 0 && W > 0, "bad shape B=%d Z=%d H=%d W=%d", B, Z, H, W);
    CFP_REQUIRE(max_width > 0 && 640 % max_width == 0, "max_resolution[1]=%d does not divide 640 (fusion.py:41)", max_width);
    const int cps = 640 / max_width;                        // conv_patch_size: 4 / 8 / 16
    CFP_REQUIRE(cps == 4 || cps == 8 || cps == 16, "patch_info has no entry for cell size %d (utils/dataloader.py:25)", cps);
    int zn = (int)std::sqrt((double)Z);                     // int(math.sqrt(Z)), utils/dataloader.py:14
    while ((zn + 1) * (zn + 1) <= Z) ++zn;
    while (zn * zn > Z) --zn;
    int pad_h = INT_MIN, pad_w = INT_MIN, p1 = INT_MIN, p2 = INT_MIN;
    int sy_wo = INT_MAX, sx_wo = INT_MAX, ey_wo = INT_MIN, ex_wo = INT_MIN;
    const float fc = (float)cps;
    for (int b = 0; b < B; ++b) {                           // per frame (dataloader.py:15-38), then max / min over the batch
        const float* r = rects + (size_t)b * Z * 4;
        float hgt = -INFINITY, wid = -INFINITY, up = 0.f, left = 0.f, down = 0.f, right = 0.f;
        float y0min = INFINITY, x0min = INFINITY, y1max = -INFINITY, x1max = -INFINITY;
        for (int z = 0; z < Z; ++z) {
            const float y0 = r[4 * z], x0 = r[4 * z + 1], y1 = r[4 * z + 2], x1 = r[4 * z + 3];
            CFP_REQUIRE(std::isfinite(y0) && std::isfinite(x0) && std::isfinite(y1) && std::isfinite(x1) &&
                        fabsf(y0) < 1e6f && fabsf(x0) < 1e6f && fabsf(y1) < 1e6f && fabsf(x1) < 1e6f,
                        "rect_data[%d][%d] is not a finite pixel rectangle", b, z);
            hgt = fmaxf(hgt, y1 - y0);
            wid = fmaxf(wid, x1 - x0);
            up = fmaxf(up, fabsf(fminf(y0, 0.f)));
            left = fmaxf(left, fabsf(fminf(x0, 0.f)));
            down = fmaxf(down, fmaxf(y1, 480.f) - 480.f);   // the canvas is hard-coded 480 x 640 (dataloader.py:20-23)
            right = fmaxf(right, fmaxf(x1, 640.f) - 640.f);
            y0min = fminf(y0min, y0 / fc);                  // float32 divisions, truncated toward zero below
            x0min = fminf(x0min, x0 / fc);
            y1max = fmaxf(y1max, y1 / fc);
            x1max = fmaxf(x1max, x1 / fc);
        }
        const int over_h = (int)fmaxf(up, down), over_w = (int)fmaxf(left, right);
        const int ih = (int)hgt, iw = (int)wid;
        auto ceil_div = [](int a, int d) { return a >= 0 ? (a + d - 1) / d : -((-a) / d); };   // math.ceil(a / d)
        pad_h = std::max(pad_h, ceil_div(over_h, cps));
        pad_w = std::max(pad_w, ceil_div(over_w, cps));
        p1 = std::max(p1, ceil_div(ih, cps));
        p2 = std::max(p2, ceil_div(iw, cps));
        sy_wo = std::min(sy_wo, (int)y0min);
        sx_wo = std::min(sx_wo, (int)x0min);
        ey_wo = std::max(ey_wo, (int)y1max);
        ex_wo = std::max(ex_wo, (int)x1max);
    }
    cfp_geom g{};
    g.zone_num = zn; g.pad_h = pad_h; g.pad_w = pad_w; g.p1 = p1; g.p2 = p2;
    g.sy_wo = sy_wo; g.sx_wo = sx_wo; g.ey_wo = ey_wo; g.ex_wo = ex_wo;
    const int sy = sy_wo + pad_h, ey = ey_wo + pad_h, sx = sx_wo + pad_w, ex = ex_wo + pad_w;   // fusion.py:79-82
    g.tzh = ey - sy; g.tzw = ex - sx;
    g.interpolate = (g.tzh != p1 * zn || g.tzw != p2 * zn) ? 1 : 0;                               // fusion.py:83-84
    auto clip = [](int v, int top) { return v < 0 ? 0 : (v > top ? top : v); };
    g.ry0 = clip(sy_wo, H); g.ry1 = clip(ey_wo, H); g.rx0 = clip(sx_wo, W); g.rx1 = clip(ex_wo, W);   // fusion.py:104
    *out = g;
    // what the reference's own forward needs to be well defined (fusion.py:136-138,157)
    CFP_REQUIRE(sy >= 0 && sx >= 0 && ey <= H + 2 * pad_h && ex <= W + 2 * pad_w,
                "zone canvas [%d:%d,%d:%d] leaves the padded %dx%d map", sy, ey, sx, ex, H + 2 * pad_h, W + 2 * pad_w);
    CFP_REQUIRE(g.tzh > 0 && g.tzw > 0, "empty zone canvas");
    return check_canvas(&g, H, W);
}

CFP_API int cfp_hist_encoder_fwd(const float* hist, void* out32, void* out64, void* out128, int64_t rows,
                         const cfp_hist_w* w, int dtype, void* stream) {
    begin_call(stream);
    CFP_REQUIRE(hist && out32 && out64 && out128 && w, "null pointer");
    CFP_REQUIRE(dtype == CFP_F32 || dtype == CFP_BF16, "unsupported dtype %d", dtype);
    if (rows == 0) return 0;
    CFP_REQUIRE(rows > 0 && rows < ((int64_t)1 << 31) * 32, "bad row count");
    return hist_encoder(hist, out32, out64, out128, rows, *w, dtype, (cudaStream_t)stream);
}

CFP_API int cfp_zone_masks(const uint8_t* mask, uint8_t* zone_mask, uint8_t* hist_mask, uint8_t* pad_mask, int B, int H,
                   int W, const cfp_geom* g, void* stream) {
    begin_call(stream);
    CFP_REQUIRE(mask && zone_mask && hist_mask && pad_mask, "null pointer");
    if (int e = check_geom(g, H, W)) return e;
    return zone_masks(mask, zone_mask, hist_mask, pad_mask, B, H, W, *g, (cudaStream_t)stream);
}

CFP_API int cfp_posenc_tokens_fwd(const void* x_nchw, const float* pos, void* tokens, int B, int C, int H, int W, int pos_h,
                          int pos_w, int oy, int ox, int dtype, void* stream) {
    begin_call(stream);
    CFP_REQUIRE(x_nchw && pos && tokens, "null pointer");
    CFP_REQUIRE(B > 0 && B <= 65535 && C > 0 && H > 0 && W > 0, "bad shape");
    CFP_REQUIRE(oy >= 0 && ox >= 0 && ox + W <= pos_w && oy + H <= pos_h,
                "positional-encoding crop [%d:%d,%d:%d] outside the %dx%d table", oy, oy + H, ox, ox + W, pos_h, pos_w);
    CFP_REQUIRE(dtype == CFP_F32 || dtype == CFP_BF16, "unsupported dtype %d", dtype);
    return posenc_tokens(x_nchw, pos, tokens, B, C, H, W, pos_w, oy, ox, dtype, (cudaStream_t)stream);
}

CFP_API int cfp_posenc_tokens_crop_fwd(const void* x_nchw, const float* pos, void* tokens, int B, int C, int H, int W, int pos_h,
                                       int pos_w, const int* crop, int dtype, void* stream) {
    begin_call(stream);
    CFP_REQUIRE(x_nchw && pos && tokens && crop, "null pointer");
    CFP_REQUIRE(B > 0 && B <= 65535 && C > 0 && H > 0 && W > 0, "bad shape");
    CFP_REQUIRE(W <= pos_w && H <= pos_h, "feature map %dx%d larger than the %dx%d positional-encoding table", H, W, pos_h, pos_w);
    CFP_REQUIRE(dtype == CFP_F32 || dtype == CFP_BF16, "unsupported dtype %d", dtype);
    return posenc_tokens(x_nchw, pos, tokens, B, C, H, W, pos_w, 0, 0, dtype, (cudaStream_t)stream, crop);
}

CFP_API int cfp_tokens_to_nchw(const void* tokens, void* out_nchw, int B, int C, int H, int W, int dtype, void* stream) {
    begin_call(stream);
    CFP_REQUIRE(tokens && out_nchw, "null pointer");
    CFP_REQUIRE(B > 0 && B <= 65535 && C > 0 && H > 0 && W > 0, "bad shape");
    CFP_REQUIRE(dtype == CFP_F32 || dtype == CFP_BF16, "unsupported dtype %d", dtype);
    return tokens_to_nchw(tokens, out_nchw, B, C, H, W, dtype, (cudaStream_t)stream);
}

CFP_API int cfp_d2i_fwd(void* feat0, const void* emb, const void* zone_tok, const float* pos2, const uint8_t* mask, int B,
                int H, int W, int C, int S, const cfp_geom* g, const cfp_loftr_w* w, int assign, void* workspace,
                size_t workspace_bytes, int dtype, void* stream) {
    begin_call(stream);
    if (int e = check_common(feat0, B, H, W, C, dtype)) return e;
    if (int e = check_geom(g, H, W)) return e;
    CFP_REQUIRE(emb && zone_tok && pos2 && mask && w && workspace, "null pointer");
    CFP_REQUIRE(S > 0, "zone_sample_num must be positive");
    if (int e = check_canvas(g, H, W)) return e;
    WsLayout L = ws_layout(B, H, W, C, 0, 0, dtype, g);
    CFP_REQUIRE(workspace_bytes >= L.total, "workspace too small: %zu < %zu", workspace_bytes, L.total);
    return d2i(feat0, emb, zone_tok, pos2, mask, B, H, W, C, S, *g, *w, assign, (char*)workspace, L, dtype,
               (cudaStream_t)stream);
}

CFP_API int cfp_dapm_fwd(void* feat0, int B, int H, int W, int C, const cfp_geom* g, const cfp_dapm_w* w, void* workspace,
                 size_t workspace_bytes, int dtype, void* stream) {
    begin_call(stream);
    if (int e = check_common(feat0, B, H, W, C, dtype)) return e;
    if (int e = check_geom(g, H, W)) return e;
    CFP_REQUIRE(w && workspace, "null pointer");
    CFP_REQUIRE(B <= 65535, "B too large for grid.z");
    WsLayout L = ws_layout(B, H, W, C, 0, 0, dtype, g);
    CFP_REQUIRE(workspace_bytes >= L.kv_bytes + 2 * L.tok_bytes, "workspace too small: %zu < %zu", workspace_bytes,
                L.kv_bytes + 2 * L.tok_bytes);
    char* ws = (char*)workspace;
    cudaStream_t st = (cudaStream_t)stream;
    void* msg_map = ws + L.tok_a;     // written only outside the zone rectangle; read as zero inside
    void* mid = ws + L.tok_b;
    if (int e = dapm_attention(feat0, msg_map, B, H, W, C, *g, w->attn, ws, L, dtype, st)) return e;
    if (dtype == CFP_BF16) {     // tensor-core implicit GEMM (k_conv_tc.cu)
        CFP_REQUIRE(w->conv1_pk && w->conv2_pk, "bf16 DAPM needs the packed tensor-core weights (conv*_pk)");
        if (int e = conv3x3_tc(feat0, msg_map, w->conv1_pk, w->shift1, nullptr, mid, B, H, W, C, g->ry0, g->ry1,
                               g->rx0, g->rx1, st)) return e;
        return conv3x3_tc(mid, nullptr, w->conv2_pk, w->shift2, feat0, feat0, B, H, W, C, 0, 0, 0, 0, st);
    }
    if (int e = conv3x3(feat0, msg_map, w->conv1_t, w->shift1, nullptr, mid, B, H, W, C, g->ry0, g->ry1, g->rx0,
                        g->rx1, dtype, st)) return e;
    return conv3x3(mid, nullptr, w->conv2_t, w->shift2, feat0, feat0, B, H, W, C, 0, 0, 0, 0, dtype, st);
}

CFP_API int cfp_lkpm_fwd(void* feat0, int B, int H, int W, int C, const cfp_lkpm_w* w, void* workspace, size_t workspace_bytes,
                 int dtype, void* stream) {
    begin_call(stream);
    if (int e = check_common(feat0, B, H, W, C, dtype)) return e;
    CFP_REQUIRE(w && workspace, "null pointer");
    WsLayout L = ws_layout(B, H, W, C, 0, w->ksize, dtype, nullptr);
    CFP_REQUIRE(workspace_bytes >= L.total, "workspace too small: %zu < %zu", workspace_bytes, L.total);
    char* ws = (char*)workspace;
    cudaStream_t st = (cudaStream_t)stream;
    void* y = ws + L.tok_a;
    if (dtype == CFP_BF16) {
        // k >= 15: Toeplitz GEMM on the tensor pipe (k_dwconv_tc.cu); its planar output feeds the MLP directly.  At k = 7 the
        // Toeplitz kernel measured a wash against the stencil, which stays.
        if (w->ksize >= 15) {
            const void* planar = nullptr;
            int pitch = 0;
            if (int e = dwconv_tc(feat0, &planar, &pitch, B, H, W, C, w->ksize, w->dw_toep, w->dw_shift, ws + L.planes, st)) return e;
            return lkpm_mlp_tc(feat0, planar, (int64_t)B * H * W, H * W, W, pitch, C, *w, st);
        }
        if (int e = dwconv_bn_relu(feat0, y, B, H, W, C, w->ksize, w->dw_t, w->dw_shift, dtype, st)) return e;
        return lkpm_mlp_tc(feat0, y, (int64_t)B * H * W, 0, 0, 0, C, *w, st);
    }
    if (int e = dwconv_bn_relu(feat0, y, B, H, W, C, w->ksize, w->dw_t, w->dw_shift, dtype, st)) return e;
    return lkpm_mlp(feat0, y, (int64_t)B * H * W, C, *w, dtype, st);
}

static int twins_call(void* feat0, void* out_nchw, int B, int H, int W, int C, const cfp_twins_w* w, void* workspace,
                      size_t workspace_bytes, int dtype, void* stream);
CFP_API int cfp_twins_fwd(void* feat0, int B, int H, int W, int C, const cfp_twins_w* w, void* workspace,
                  size_t workspace_bytes, int dtype, void* stream) {
    begin_call(stream);
    return twins_call(feat0, nullptr, B, H, W, C, w, workspace, workspace_bytes, dtype, stream);
}
CFP_API int cfp_twins_nchw_fwd(void* feat0, void* out_nchw, int B, int H, int W, int C, const cfp_twins_w* w, void* workspace,
                       size_t workspace_bytes, int dtype, void* stream) {
    begin_call(stream);
    CFP_REQUIRE(out_nchw != nullptr && out_nchw != feat0, "out_nchw must be a separate NCHW map");
    return twins_call(feat0, out_nchw, B, H, W, C, w, workspace, workspace_bytes, dtype, stream);
}
static int twins_call(void* feat0, void* out_nchw, int B, int H, int W, int C, const cfp_twins_w* w, void* workspace,
                      size_t workspace_bytes, int dtype, void* stream) {
    if (int e = check_common(feat0, B, H, W, C, dtype)) return e;
    CFP_REQUIRE(w && workspace, "null pointer");
    CFP_REQUIRE(w->ws > 1, "window size must be > 1 (transformer.py:79)");
    CFP_REQUIRE(C % 8 == 0, "dim %d should be divided by num_heads 8 (transformer.py:81)", C);
    CFP_REQUIRE(H >= w->ws && W >= w->ws, "%dx%d map smaller than the %dx%d sub-sampling kernel (the reference's sr conv "
                "fails here too, transformer.py:144)", H, W, w->ws, w->ws);
    WsLayout L = ws_layout(B, H, W, C, w->ws, 0, dtype, nullptr);
    CFP_REQUIRE(workspace_bytes >= L.total, "workspace too small: %zu < %zu", workspace_bytes, L.total);
    return twins(feat0, out_nchw, B, H, W, C, *w, (char*)workspace, L, dtype, (cudaStream_t)stream);
}

// ---------------------------------------------------------------- training-step building blocks (fp32)
CFP_API int cfp_tr_gemm(const float* a, int64_t a_rs, int64_t a_cs, const float* b, int64_t b_rs, int64_t b_cs, float* c,
                        int64_t c_rs, int M, int N, int K, const float* bias, int accumulate, void* stream) {
    begin_call(stream);
    CFP_REQUIRE(a && b && c, "null pointer");
    return tr_gemm(a, a_rs, a_cs, b, b_rs, b_cs, c, c_rs, M, N, K, bias, accumulate, (cudaStream_t)stream);
}
CFP_API int cfp_tr_colsum(const float* x, float* out, int64_t rows, int C, void* stream) {
    begin_call(stream);
    CFP_REQUIRE(x && out && rows > 0 && C > 0, "bad arguments");
    return tr_colsum(x, out, rows, C, (cudaStream_t)stream);
}
CFP_API int cfp_tr_bn_stats(const float* x, int64_t rows, int C, float eps, float momentum, float* mean, float* rstd,
                            float* running_mean, float* running_var, float* scratch, void* stream) {
    begin_call(stream);
    CFP_REQUIRE(x && mean && rstd && scratch, "null pointer");
    return tr_bn_stats(x, rows, C, eps, momentum, mean, rstd, running_mean, running_var, scratch, (cudaStream_t)stream);
}
CFP_API int cfp_tr_bn_apply(const float* x, const float* mean, const float* rstd, const float* gamma, const float* beta,
                            float* y, int64_t rows, int C, int relu, void* stream) {
    begin_call(stream);
    CFP_REQUIRE(x && mean && rstd && gamma && beta && y, "null pointer");
    return tr_bn_apply(x, mean, rstd, gamma, beta, y, rows, C, relu, (cudaStream_t)stream);
}
CFP_API int cfp_tr_bn_bwd(const float* dy, const float* x, const float* mean, const float* rstd, const float* gamma,
                          const float* beta, float* dx, float* dgamma, float* dbeta, int64_t rows, int C, int relu, void* stream) {
    begin_call(stream);
    CFP_REQUIRE(dy && x && mean && rstd && gamma && beta && dx && dgamma && dbeta, "null pointer");
    return tr_bn_bwd(dy, x, mean, rstd, gamma, beta, dx, dgamma, dbeta, rows, C, relu, (cudaStream_t)stream);
}
CFP_API int cfp_tr_ln_fwd(const float* x, const float* g, const float* b, float* y, int64_t rows, int C, float eps, void* stream) {
    begin_call(stream);
    CFP_REQUIRE(x && g && b && y, "null pointer");
    return tr_ln_fwd(x, g, b, y, rows, C, eps, (cudaStream_t)stream);
}
CFP_API int cfp_tr_ln_bwd(const float* x, const float* g, const float* dy, float* dx, float* dg, float* db, int64_t rows, int C,
                          float eps, void* stream) {
    begin_call(stream);
    CFP_REQUIRE(x && g && dy && dx && dg && db, "null pointer");
    return tr_ln_bwd(x, g, dy, dx, dg, db, rows, C, eps, (cudaStream_t)stream);
}
CFP_API int cfp_tr_ew(const float* a, const float* b, float* out, int64_t n, int op, void* stream) {
    begin_call(stream);
    CFP_REQUIRE(a && out, "null pointer");
    return tr_ew(a, b, out, n, op, (cudaStream_t)stream);
}
CFP_API int cfp_tr_gather_rows(const float* src, const int* idx, float* out, int64_t n, int C, void* stream) {
    begin_call(stream);
    CFP_REQUIRE(src && idx && out && n >= 0, "bad arguments");
    return tr_gather_rows(src, idx, out, n, C, (cudaStream_t)stream);
}
CFP_API int cfp_tr_scatter_add_rows(const float* src, const int* idx, const float* base, float* out, int64_t n, int64_t base_rows,
                                    int C, void* stream) {
    begin_call(stream);
    CFP_REQUIRE(src && idx && base && out && n >= 0 && base_rows > 0 && C > 0, "bad arguments");
    return tr_scatter_add_rows(src, idx, base, out, n, base_rows, C, (cudaStream_t)stream);
}
CFP_API int cfp_tr_attn_reduce(const float* a, const float* b, const float* w, float* kv, float* as, int G, int R, int C, int nh,
                               void* stream) {
    begin_call(stream);
    CFP_REQUIRE(a && b && kv && as, "null pointer");
    return tr_attn_reduce(a, b, w, kv, as, G, R, C, nh, (cudaStream_t)stream);
}
CFP_API int cfp_tr_attn_apply(const float* x, const float* kv, float* out, int G, int R, int C, int nh, int transpose, void* stream) {
    begin_call(stream);
    CFP_REQUIRE(x && kv && out, "null pointer");
    return tr_attn_apply(x, kv, out, G, R, C, nh, transpose, (cudaStream_t)stream);
}
CFP_API int cfp_tr_head_dot(const float* a, const float* b, float* out, int64_t rows, int C, int nh, int rows_per_group, float eps,
                            void* stream) {
    begin_call(stream);
    CFP_REQUIRE(a && b && out, "null pointer");
    return tr_head_dot(a, b, out, rows, C, nh, rows_per_group, eps, (cudaStream_t)stream);
}
CFP_API int cfp_tr_rowop(const float* a, const float* s, const float* b, float* out, int64_t rows, int C, int nh, int rows_per_group,
                         int op, void* stream) {
    begin_call(stream);
    CFP_REQUIRE(a && out, "null pointer");
    return tr_rowop(a, s, b, out, rows, C, nh, rows_per_group, op, (cudaStream_t)stream);
}
CFP_API int cfp_tr_dwconv(const float* in, float* out, int B, int H, int W, int C, int ksize, const float* taps_t,
                          const float* shift, int relu, void* stream) {
    begin_call(stream);
    CFP_REQUIRE(in && out && taps_t && shift, "null pointer");
    CFP_REQUIRE(B > 0 && H > 0 && W > 0, "bad shape");
    return dwconv_bn_relu(in, out, B, H, W, C, ksize, taps_t, shift, CFP_F32, (cudaStream_t)stream, relu);
}
CFP_API int cfp_tr_dwconv_wgrad(const float* x, const float* dy, float* dw, int B, int H, int W, int C, int ksize, void* stream) {
    begin_call(stream);
    CFP_REQUIRE(x && dy && dw, "null pointer");
    CFP_REQUIRE(B > 0 && H > 0 && W > 0, "bad shape");
    return tr_dwconv_wgrad(x, dy, dw, B, H, W, C, ksize, (cudaStream_t)stream);
}

CFP_API int cfp_tr_sumsq(const float* x, int64_t n, float scale, float* out, void* stream) {
    begin_call(stream);
    CFP_REQUIRE(out && (x || n == 0) && n >= 0, "bad arguments");
    return tr_sumsq(x, n, scale, out, (cudaStream_t)stream);
}
CFP_API int cfp_tr_adamw(float* p, const float* g, float* m, float* v, int64_t n, const int64_t* seg_end, const float* seg_lr,
                         int nseg, float beta1, float beta2, float eps, float weight_decay, int step, float grad_scale,
                         const float* sumsq, float max_norm, void* stream) {
    begin_call(stream);
    CFP_REQUIRE(p && g && m && v && seg_end && seg_lr && n >= 0, "bad arguments");
    return tr_adamw(p, g, m, v, n, seg_end, seg_lr, nseg, beta1, beta2, eps, weight_decay, step, grad_scale, sumsq, max_norm,
                    (cudaStream_t)stream);
}

// ---------------------------------------------------------------- input side (f3) and loss / metrics (f4)
CFP_API int cfp_zone_hist(const float* dep, int B, int H, int W, int sy, int sx, int ph, int pw, int zone_num, int nbins,
                          float max_distance, const double* centres, float* fh, uint8_t* mask, int* hist_out, void* stream) {
    begin_call(stream);
    CFP_REQUIRE(dep && centres && fh && mask, "null pointer");
    CFP_REQUIRE(B > 0 && H > 0 && W > 0, "bad shape");
    return zone_hist(dep, B, H, W, sy, sx, ph, pw, zone_num, nbins, max_distance, centres, fh, mask, hist_out, (cudaStream_t)stream);
}
CFP_API int cfp_zone_samples(const float* fh, const uint8_t* mask, float* out, int64_t zones, int S, const float* w0,
                             const float* w1, int mode, void* stream) {
    begin_call(stream);
    CFP_REQUIRE(fh && mask && out, "null pointer");
    return zone_samples(fh, mask, out, zones, S, w0, w1, mode, (cudaStream_t)stream);
}
CFP_API int cfp_silog_fwd(const float* pred, const float* target, const uint8_t* mask, int B, int h, int w, int H, int W,
                          int interpolate, double* scratch, float* loss, void* stream) {
    begin_call(stream);
    CFP_REQUIRE(pred && target && scratch && loss, "null pointer");
    return silog_fwd(pred, target, mask, B, h, w, H, W, interpolate, scratch, loss, (cudaStream_t)stream);
}
CFP_API int cfp_silog_bwd(const float* pred, const float* target, const uint8_t* mask, int B, int h, int w, int H, int W,
                          int interpolate, const double* scratch, float grad_out, float* grad_pred, void* stream) {
    begin_call(stream);
    CFP_REQUIRE(pred && target && scratch && grad_pred, "null pointer");
    return silog_bwd(pred, target, mask, B, h, w, H, W, interpolate, scratch, grad_out, grad_pred, (cudaStream_t)stream);
}
CFP_API int cfp_depth_metrics(const float* gt, const float* pred, const uint8_t* valid, int64_t n, double* scratch, double* out,
                              void* stream) {
    begin_call(stream);
    CFP_REQUIRE(gt && pred && scratch && out, "null pointer");
    return depth_metrics(gt, pred, valid, n, scratch, out, (cudaStream_t)stream);
}

// ---------------------------------------------------------------- decoder shell (f1) and adaptive-bins head (f2)
CFP_API int cfp_conv_fwd(const void* in, int B, int H, int W, int cin, int cout, int ksize, int kchunk, const void* w_tc,
                         const float* shift, float leaky_slope, void* out, int out_pitch, int out_coff, void* stream) {
    begin_call(stream);
    CFP_REQUIRE(in && w_tc && shift && out, "null pointer");
    CFP_REQUIRE(ksize == 1 || ksize == 3, "kernel size %d (1 and 3 are served)", ksize);
    return conv_gen_tc(in, cin, kchunk, ksize * ksize, w_tc, shift, leaky_slope, out, out_pitch, out_coff, B, H, W, cout, (cudaStream_t)stream);
}
CFP_API int cfp_upsample_concat(const void* lo, int h, int w, int c_lo, int lo_pitch, const float* skip, int c_skip, void* out, int B,
                                int H, int W, int c_out, void* stream) {
    begin_call(stream);
    CFP_REQUIRE(out, "null pointer");
    return upsample_concat(lo, h, w, c_lo, lo_pitch, skip, c_skip, out, B, H, W, c_out, (cudaStream_t)stream);
}
CFP_API int cfp_posenc_tokens_nhwc_fwd(const void* x, int x_pitch, const float* pos, void* tokens, int B, int C, int H, int W,
                                       int pos_h, int pos_w, int oy, int ox, void* stream) {
    begin_call(stream);
    CFP_REQUIRE(x && pos && tokens, "null pointer");
    CFP_REQUIRE(B > 0 && C > 0 && H > 0 && W > 0, "bad shape");
    CFP_REQUIRE(oy >= 0 && ox >= 0 && ox + W <= pos_w && oy + H <= pos_h,
                "positional-encoding crop [%d:%d,%d:%d] outside the %dx%d table", oy, oy + H, ox, ox + W, pos_h, pos_w);
    return posenc_tokens_nhwc(x, x_pitch, pos, tokens, B, C, H, W, pos_w, oy, ox, (cudaStream_t)stream);
}
CFP_API int cfp_copy_channels(const void* src, int src_pitch, void* dst, int dst_pitch, int coff, int C, int64_t rows, void* stream) {
    begin_call(stream);
    CFP_REQUIRE(src && dst && rows >= 0, "bad arguments");
    return copy_channels(src, src_pitch, dst, dst_pitch, coff, C, rows, (cudaStream_t)stream);
}
CFP_API int cfp_head_bins(const void* x, int pitch, int B, int npix, int E, const float* wc, const float* w0, const float* b0,
                          const float* w2, const float* b2, const float* w4, const float* b4, int hidden, int n_bins, float min_val,
                          float max_val, float* mean_scratch, float* edges, float* centres, void* stream) {
    begin_call(stream);
    CFP_REQUIRE(x && wc && w0 && b0 && w2 && b2 && w4 && b4 && mean_scratch && edges && centres, "null pointer");
    if (int e = channel_mean(x, pitch, E, B, npix, mean_scratch, (cudaStream_t)stream)) return e;
    return head_regressor(mean_scratch, wc, w0, b0, w2, b2, w4, b4, B, E, hidden, n_bins, min_val, max_val, edges, centres,
                          (cudaStream_t)stream);
}
CFP_API int cfp_head_expect(const void* x, int pitch, int B, int npix, const void* w_tc, const float* bias, const float* centres,
                            int n_bins, float* pred, float* prob, void* stream) {
    begin_call(stream);
    CFP_REQUIRE(x && w_tc && bias && centres && pred, "null pointer");
    return head_expect_tc(x, pitch, B, npix, w_tc, bias, centres, n_bins, pred, prob, (cudaStream_t)stream);
}

// the exact fp32 engine of the same stages (k_dec_f32.cu)
CFP_API int cfp_conv_f32_fwd(const float* in, int B, int H, int W, int cin, int cout, int ksize, const float* w, const float* shift,
                             float leaky_slope, float* out, int out_pitch, int out_coff, void* stream) {
    begin_call(stream);
    CFP_REQUIRE(in && w && shift && out, "null pointer");
    CFP_REQUIRE(ksize == 1 || ksize == 3, "kernel size %d (1 and 3 are served)", ksize);
    return conv_f32(in, cin, ksize * ksize, w, shift, leaky_slope, out, out_pitch, out_coff, B, H, W, cout, (cudaStream_t)stream);
}
CFP_API int cfp_upsample_concat_f32(const float* lo, int h, int w, int c_lo, int lo_pitch, const float* skip, int c_skip, float* out, int B,
                                    int H, int W, int c_out, void* stream) {
    begin_call(stream);
    CFP_REQUIRE(out, "null pointer");
    return upsample_concat_f32(lo, h, w, c_lo, lo_pitch, skip, c_skip, out, B, H, W, c_out, (cudaStream_t)stream);
}
CFP_API int cfp_posenc_tokens_nhwc_f32_fwd(const float* x, int x_pitch, const float* pos, float* tokens, int B, int C, int H, int W,
                                           int pos_h, int pos_w, int oy, int ox, void* stream) {
    begin_call(stream);
    CFP_REQUIRE(x && pos && tokens, "null pointer");
    CFP_REQUIRE(B > 0 && C > 0 && H > 0 && W > 0, "bad shape");
    CFP_REQUIRE(oy >= 0 && ox >= 0 && ox + W <= pos_w && oy + H <= pos_h,
                "positional-encoding crop [%d:%d,%d:%d] outside the %dx%d table", oy, oy + H, ox, ox + W, pos_h, pos_w);
    return posenc_tokens_nhwc_f32(x, x_pitch, pos, tokens, B, C, H, W, pos_w, oy, ox, (cudaStream_t)stream);
}
CFP_API int cfp_copy_channels_f32(const float* src, int src_pitch, float* dst, int dst_pitch, int coff, int C, int64_t rows, void* stream) {
    begin_call(stream);
    CFP_REQUIRE(src && dst && rows >= 0, "bad arguments");
    return copy_channels_f32(src, src_pitch, dst, dst_pitch, coff, C, rows, (cudaStream_t)stream);
}
CFP_API int cfp_head_bins_f32(const float* x, int pitch, int B, int npix, int E, const float* wc, const float* w0, const float* b0,
                              const float* w2, const float* b2, const float* w4, const float* b4, int hidden, int n_bins, float min_val,
                              float max_val, float* mean_scratch, float* edges, float* centres, void* stream) {
    begin_call(stream);
    CFP_REQUIRE(x && wc && w0 && b0 && w2 && b2 && w4 && b4 && mean_scratch && edges && centres, "null pointer");
    if (int e = channel_mean_f32(x, pitch, E, B, npix, mean_scratch, (cudaStream_t)stream)) return e;
    return head_regressor(mean_scratch, wc, w0, b0, w2, b2, w4, b4, B, E, hidden, n_bins, min_val, max_val, edges, centres,
                          (cudaStream_t)stream);
}
CFP_API int cfp_head_expect_f32(const float* x, int pitch, int B, int npix, const float* w_t, const float* bias, const float* centres,
                                int n_bins, float* pred, float* prob, void* stream) {
    begin_call(stream);
    CFP_REQUIRE(x && w_t && bias && centres && pred, "null pointer");
    return head_expect_f32(x, pitch, B, npix, w_t, bias, centres, n_bins, pred, prob, (cudaStream_t)stream);
}

CFP_API int cfp_selftest_umma(const void* a, const void* b, float* d, int rows_a, int n, int k, int row_shift,
                              void* stream) {
    begin_call(stream);
    CFP_REQUIRE(a && b && d, "null pointer");
    return umma_selftest(a, b, d, rows_a, n, k, row_shift, (cudaStream_t)stream);
}

CFP_API int64_t cfp_launch_count(void) { return pstate().launches.load(); }

CFP_API int cfp_set_pdl(int on) {
    const int prev = pdl_enabled() ? 1 : 0;
    tl_pdl = on < 0 ? -1 : (on ? 1 : 0);
    return prev;
}

CFP_API int cfp_profile_start(void) {
    ProfileState& t = pstate();
    std::lock_guard<std::mutex> lk(t.mu);
    for (auto& e : t.events) cudaEventDestroy(e.second);
    t.events.clear();
    if (t.first) cudaEventDestroy(t.first);
    t.first = nullptr;
    t.profiling = true;
    return 0;
}

CFP_API int cfp_profile_stop(char* out, size_t cap) {
    ProfileState& t = pstate();
    t.profiling = false;
    std::lock_guard<std::mutex> lk(t.mu);
    CFP_REQUIRE(out && cap > 2, "null output buffer");
    struct Acc { const char* name; int count; double ms; };
    std::vector<Acc> acc;
    cudaEvent_t prev = t.first;
    for (auto& e : t.events) {
        cudaEventSynchronize(e.second);
        if (!e.first) { prev = e.second; continue; }  // start of an API call
        float ms = 0.f;
        if (prev) cudaEventElapsedTime(&ms, prev, e.second);
        prev = e.second;
        bool found = false;
        for (auto& a : acc)
            if (std::strcmp(a.name, e.first) == 0) { a.count++; a.ms += ms; found = true; break; }
        if (!found) acc.push_back({e.first, 1, (double)ms});
    }
    std::string js = "{";
    for (size_t i = 0; i < acc.size(); ++i) {
        char buf[256];
        snprintf(buf, sizeof(buf), "%s\"%s\": [%d, %.6f]", i ? ", " : "", acc[i].name, acc[i].count, acc[i].ms);
        js += buf;
    }
    js += "}";
    for (auto& e : t.events) cudaEventDestroy(e.second);
    t.events.clear();
    if (t.first) cudaEventDestroy(t.first);
    t.first = nullptr;
    CFP_REQUIRE(js.size() + 1 <= cap, "profile buffer too small (%zu needed)", js.size() + 1);
    std::memcpy(out, js.c_str(), js.size() + 1);
    return 0;
}

}  // extern "C"
