// lk_level.cu -- host-side entry of the fused per-level LK kernel: tensor maps, argument checks and
// the dispatch on the window size.  The kernels themselves are instantiated one window per
// translation unit (lk_win.cu, compiled once per -DLK_WIN=n) so that the build runs in parallel.
#include "lk_level.cuh"

#include <cstdlib>
#include <mutex>

namespace ofb {

bool pdl_enabled()
{
    static const bool on = [] {
        const char *e = getenv("OFB_PDL"); // off by default: measured on B200 it does not pay (ofb_common.cuh)
        return e && e[0] == '1';
    }();
    return on;
}

PFN_encodeTiled get_encode_tiled()
{
    static PFN_encodeTiled fn = nullptr;
    static std::once_flag once;
    std::call_once(once, [] {
        void *sym = nullptr;
        cudaDriverEntryPointQueryResult qres;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &qres) == cudaSuccess &&
            qres == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<PFN_encodeTiled>(sym);
    });
    return fn;
}

// Encoded tensor maps are kept per host thread in a small round-robin cache keyed by everything that goes into them: a
// frame loop or a replayed batch meets the same few (pointer, shape, box) combinations over and over, and an encode
// costs about a microsecond of host time (three per level launch).
namespace {
struct MapKey {
    const void *base;
    int type, w, h, n, box_w, box_rows;
    size_t s0, s1;
    bool operator==(const MapKey &o) const
    {
        return base == o.base && type == o.type && w == o.w && h == o.h && n == o.n && box_w == o.box_w && box_rows == o.box_rows &&
               s0 == o.s0 && s1 == o.s1;
    }
};
struct MapCache {
    static constexpr int N = 32;
    MapKey key[N];
    CUtensorMap map[N];
    int used = 0, next = 0;
    const CUtensorMap *find(const MapKey &k) const
    {
        for (int i = 0; i < used; i++)
            if (key[i] == k) return &map[i];
        return nullptr;
    }
    void put(const MapKey &k, const CUtensorMap &m)
    {
        key[next] = k;
        map[next] = m;
        next = (next + 1) % N;
        if (used < N) used++;
    }
};
thread_local MapCache g_maps;
} // namespace

// u8 image batch as a 3-D tensor (x, y, image); box = box_w x box_rows x 1; OOB reads give 0.
int lk_make_image_map(CUtensorMap *tm, const uint8_t *base, int w, int h, int n, size_t pitch, size_t stride, int box_w,
                      int box_rows)
{
    PFN_encodeTiled enc = get_encode_tiled();
    if (!enc) {
        set_error("cuTensorMapEncodeTiled is not available from this driver");
        return OFB_ERR_CUDA;
    }
    if ((reinterpret_cast<uintptr_t>(base) & 15) || (pitch & 15) || (stride & 15)) {
        set_error("device images must be 16-byte aligned with pitch and image stride multiples of 16 "
                  "(base %p pitch %zu stride %zu)", (const void *)base, pitch, stride);
        return OFB_ERR_INVALID;
    }
    cuuint64_t dims[3] = {(cuuint64_t)w, (cuuint64_t)h, (cuuint64_t)n};
    cuuint64_t strides[2] = {(cuuint64_t)pitch, (cuuint64_t)(n > 1 ? stride : pitch * (size_t)h)};
    if (strides[1] & 15) strides[1] = (strides[1] + 15) & ~(cuuint64_t)15;
    const MapKey key{base, 0, w, h, n, box_w, box_rows, (size_t)strides[0], (size_t)strides[1]};
    if (const CUtensorMap *hit = g_maps.find(key)) {
        *tm = *hit;
        return OFB_OK;
    }
    cuuint32_t box[3] = {(cuuint32_t)box_w, (cuuint32_t)box_rows, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, const_cast<uint8_t *>(base), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeTiled failed with CUresult %d (w %d h %d n %d pitch %zu)", (int)r, w, h, n, pitch);
        return OFB_ERR_CUDA;
    }
    g_maps.put(key, *tm);
    return OFB_OK;
}

// float2 flow field batch as a 3-D tensor of floats (2*w, h, pair); box = 2*box_w x box_rows x 1; OOB reads give 0.
// Returns OFB_OK with *usable = 0 when the layout cannot have a tensor map (base, row or pair stride not a
// multiple of 16 bytes: odd widths); the kernel then copies its tiles itself.
int lk_make_flow_map(CUtensorMap *tm, const float *base, int w, int h, int n, size_t pair_stride_vec, int box_w, int box_rows,
                     int *usable)
{
    *usable = 0;
    PFN_encodeTiled enc = get_encode_tiled();
    if (!enc) {
        set_error("cuTensorMapEncodeTiled is not available from this driver");
        return OFB_ERR_CUDA;
    }
    const size_t row_bytes = (size_t)w * 8, pair_bytes = pair_stride_vec * 8;
    if ((reinterpret_cast<uintptr_t>(base) & 15) || (row_bytes & 15) || (n > 1 && (pair_bytes & 15))) return OFB_OK;
    cuuint64_t dims[3] = {(cuuint64_t)(2 * w), (cuuint64_t)h, (cuuint64_t)n};
    cuuint64_t strides[2] = {(cuuint64_t)row_bytes, (cuuint64_t)(n > 1 ? pair_bytes : row_bytes * (size_t)h)};
    const MapKey key{base, 1, w, h, n, box_w, box_rows, (size_t)strides[0], (size_t)strides[1]};
    if (const CUtensorMap *hit = g_maps.find(key)) {
        *tm = *hit;
        *usable = 1;
        return OFB_OK;
    }
    cuuint32_t box[3] = {(cuuint32_t)(2 * box_w), (cuuint32_t)box_rows, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float *>(base), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeTiled (flow) failed with CUresult %d (w %d h %d n %d)", (int)r, w, h, n);
        return OFB_ERR_CUDA;
    }
    g_maps.put(key, *tm);
    *usable = 1;
    return OFB_OK;
}

template <int WIN> int launch_lk_win(const LkLevelArgs &a, cudaStream_t stream, unsigned long long *launches); // lk_win.cu

int launch_lk_level(const LkLevelArgs &a, cudaStream_t stream, unsigned long long *launches)
{
    if (a.w < 1 || a.h_local < 1 || a.n_pairs < 1 || a.out_y0 < 0 || a.out_y1 > a.h_local || a.out_y0 >= a.out_y1) {
        set_error("lk_level: bad geometry (w %d h_local %d pairs %d out rows [%d,%d))", a.w, a.h_local, a.n_pairs,
                  a.out_y0, a.out_y1);
        return OFB_ERR_INVALID;
    }
    if (a.pitch * (size_t)a.h_local > 0x7fffffffull || (size_t)a.w * a.h_local > 0x3fffffffull) {
        set_error("lk_level: one image is limited to 2^31 bytes (pitch %zu x %d rows)", a.pitch, a.h_local);
        return OFB_ERR_INVALID;
    }
    if (a.n_pairs > 65535) {
        set_error("lk_level: at most 65535 pairs per launch (got %d)", a.n_pairs);
        return OFB_ERR_INVALID;
    }
    if (a.cum_in && (a.w > 32768 || a.h_global > 32768)) {
        set_error("lk_level: warped levels are limited to 32768 x 32768 pixels (got %d x %d)", a.w, a.h_global);
        return OFB_ERR_INVALID;
    }
    if (a.warp_mode < OFB_WARP_AS_WRITTEN || a.warp_mode > OFB_WARP_BILINEAR) {
        set_error("lk_level: unknown warp mode %d", a.warp_mode);
        return OFB_ERR_INVALID;
    }
    // (the kernel picks 256-bit, 128-bit or scalar stores per row segment from the actual addresses; the cumulative
    // flow of a row strip lands inside the next level's buffer at a row offset, which for odd widths is 8-byte aligned)
    if ((reinterpret_cast<uintptr_t>(a.flow_out) & 15) || (a.cum_out && (reinterpret_cast<uintptr_t>(a.cum_out) & 7))) {
        set_error("lk_level: the flow buffer must be 16-byte aligned, the cumulative flow 8-byte aligned");
        return OFB_ERR_INVALID;
    }
    switch (a.win) {
    case 3: return launch_lk_win<3>(a, stream, launches);
    case 5: return launch_lk_win<5>(a, stream, launches);
    case 7: return launch_lk_win<7>(a, stream, launches);
    case 9: return launch_lk_win<9>(a, stream, launches);
    case 11: return launch_lk_win<11>(a, stream, launches);
    case 13: return launch_lk_win<13>(a, stream, launches);
    case 15: return launch_lk_win<15>(a, stream, launches);
    case 17: return launch_lk_win<17>(a, stream, launches);
    case 19: return launch_lk_win<19>(a, stream, launches);
    default:
        set_error("lk_level: window %d not supported (odd 3..19)", a.win);
        return OFB_ERR_UNSUPPORTED;
    }
}

LkLevelArgs lk_args_frame(const uint8_t *prev, const uint8_t *next, size_t pitch, size_t image_stride, int w, int h, int n_pairs,
                          int win, int warp_mode, float flow_scale, float *flow_out, int sm_count, int solve_fast)
{
    LkLevelArgs a{};
    a.prev = prev;
    a.next = next;
    a.pitch = pitch;
    a.image_stride = image_stride;
    a.w = w;
    a.h_local = a.h_global = h;
    a.y_off = 0;
    a.out_y0 = 0;
    a.out_y1 = h;
    a.n_pairs = n_pairs;
    a.win = win;
    a.warp_mode = warp_mode;
    a.flow_scale = flow_scale;
    a.flow_out = flow_out;
    a.flow_pair_stride = (size_t)w * h;
    a.sm_count = sm_count;
    a.solve_fast = solve_fast;
    return a;
}

LkLevelArgs lk_args_strip(const uint8_t *prev, const uint8_t *next, size_t pitch, int w, int h_local, int y_off, int h_global,
                          int out_y0, int out_y1, int win, int warp_mode, float flow_scale, float *flow_out, int sm_count,
                          int solve_fast)
{
    LkLevelArgs a{};
    a.prev = prev;
    a.next = next;
    a.pitch = pitch;
    a.image_stride = pitch * (size_t)h_local;
    a.w = w;
    a.h_local = h_local;
    a.y_off = y_off;
    a.h_global = h_global;
    a.out_y0 = out_y0;
    a.out_y1 = out_y1;
    a.n_pairs = 1;
    a.win = win;
    a.warp_mode = warp_mode;
    a.flow_scale = flow_scale;
    a.flow_out = flow_out;
    a.sm_count = sm_count;
    a.solve_fast = solve_fast;
    return a;
}

template <int WIN> int preload_lk_win(); // lk_win.cu
int preload_lk_level(int win)
{
    switch (win) {
    case 3: return preload_lk_win<3>();
    case 5: return preload_lk_win<5>();
    case 7: return preload_lk_win<7>();
    case 9: return preload_lk_win<9>();
    case 11: return preload_lk_win<11>();
    case 13: return preload_lk_win<13>();
    case 15: return preload_lk_win<15>();
    case 17: return preload_lk_win<17>();
    case 19: return preload_lk_win<19>();
    default: set_error("lk_level: window %d not supported (odd 3..19)", win); return OFB_ERR_UNSUPPORTED;
    }
}

} // namespace ofb
