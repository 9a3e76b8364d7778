// pnpb200_tile.cuh -- shared-memory row tiles filled by TMA (cp.async.bulk[.tensor] + mbarrier).
//
// Used by every one-problem-per-thread kernel: a CTA is ONE warp that owns 32 consecutive
// problems.  RowTile (multi-pass solvers): lane l copies problem l's whole [n_total, 2] pixel row from
// HBM into a padded shared-memory row with a single bulk copy.  RowStream (single-pass kernels): the
// rows go through two small buffers chunk by chunk, one 2-D tensor copy per chunk of all 32 rows.
// The row pitch is an odd multiple of 16 bytes, so the per-lane 16-byte reads that follow are
// bank-conflict free.
#pragma once
#include <stdint.h>
#include <stdlib.h>
#include "pnpb200_math.cuh"

namespace pnpb200 {

template <typename T> struct Vec2;
template <> struct Vec2<double> { typedef double2 type; };
template <> struct Vec2<float> { typedef float2 type; };

// normalised correspondences of one problem: that problem's row in shared memory (thread mapping)
template <typename T>
struct PtsRow {
    const T* row;          // [n_total][2], already multiplied by K^-1
    const int32_t* idx;    // shared-memory copy of the landmark selection, or nullptr
    PNP_DEV void get(int i, T& bx, T& by) const
    {
        const int j = idx ? idx[i] : i;
        const typename Vec2<T>::type p = reinterpret_cast<const typename Vec2<T>::type*>(row)[j];
        bx = p.x;
        by = p.y;
    }
    // every selected landmark takes part (the masked accessor below overrides these two)
    PNP_DEV bool vis(int) const { return true; }
    PNP_DEV int count(int n) const { return n; }
};

// bit j % 32 of word j / 32: landmark j of the caller's 0..n_total-1 numbering is visible (per-problem mask)
PNP_DEV bool mask_bit(const uint32_t* words, int j) { return (__ldg(words + (j >> 5)) >> (j & 31)) & 1u; }

// A point accessor restricted to the visible landmarks of one problem: the solvers skip i where vis(i) is false, so
// hidden pixels are never read, and count() is the number of visible selected landmarks.
template <typename Base>
struct PtsMasked : Base {
    const uint32_t* words;   // this problem's visibility words
    int nvis;
    PNP_DEV bool vis(int i) const { return mask_bit(words, this->idx ? this->idx[i] : i); }
    PNP_DEV int count(int) const { return nvis; }
};

// fewer visible landmarks than this: a problem is not solved (NaN pose), its report and check statistics are NaN
constexpr int kMinVisible = 4;

// visible landmarks among the n selected ones (idx = nullptr: landmarks 0..n-1)
PNP_DEV int count_visible(const uint32_t* words, const int32_t* idx, int n)
{
    if (idx) {
        int c = 0;
        for (int i = 0; i < n; ++i) c += mask_bit(words, idx[i]) ? 1 : 0;
        return c;
    }
    int c = 0;
    for (int w = 0; w < (n >> 5); ++w) c += __popc(__ldg(words + w));
    if (n & 31) c += __popc(__ldg(words + (n >> 5)) & ((1u << (n & 31)) - 1u));
    return c;
}

// ---- TMA bulk copy + mbarrier (sm_90+ PTX; SASS: UBLKCP / SYNCS)
PNP_DEV uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
PNP_DEV void mbar_init(uint64_t* bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // the initialised barrier, as the async proxy (TMA) sees it
}
PNP_DEV void mbar_expect_tx(uint64_t* bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
PNP_DEV void mbar_wait(uint64_t* bar, uint32_t parity)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
PNP_DEV void bulk_copy_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
// one TMA tensor copy of a (box_x x box_y) tile at element coordinates (x, y) of a 2-D tensor map (SASS: UTMALDG)
PNP_DEV void tensor_copy_2d_g2s(void* dst_smem, const void* tmap, int x, int y, uint64_t* bar)
{
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
                     smem_u32(dst_smem)),
                 "l"(reinterpret_cast<uint64_t>(tmap)), "r"(x), "r"(y), "r"(smem_u32(bar))
                 : "memory");
}
PNP_DEV void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ------------------------------------------------------------------------------------------
// Row tile: 32 consecutive problems' pixel rows staged in shared memory by one warp.
// Lane l issues one TMA bulk copy of row l (completion on an mbarrier), waits, and multiplies its
// row by K^-1 in place (f2_get_B_xy :3291-3312).  Row pitch = odd multiple of 16 B.
// ------------------------------------------------------------------------------------------
constexpr int kTileProblems = 32;

template <typename T>
struct RowTile {
    T* rows;
    uint64_t* bar;
    const T* uv;
    long long B;
    int n_total, row_pitch, use_tma;
    uint32_t phase, row_bytes;
    T k00, k01, k02, k10, k11, k12;

    bool normalise;

    PNP_DEV void init(T* rows_, uint64_t* bar_, const T* uv_, long long B_, int n_total_, int row_pitch_, int use_tma_,
                      const double* kinv, int lane, bool normalise_ = true)
    {
        rows = rows_; bar = bar_; uv = uv_; B = B_; n_total = n_total_; row_pitch = row_pitch_; use_tma = use_tma_;
        normalise = normalise_;
        phase = 0; row_bytes = (uint32_t)n_total * 2u * (uint32_t)sizeof(T);
        k00 = (T)kinv[0]; k01 = (T)kinv[1]; k02 = (T)kinv[2]; k10 = (T)kinv[3]; k11 = (T)kinv[4]; k12 = (T)kinv[5];
        if (use_tma) {
            if (lane == 0) mbar_init(bar, 1);
            __syncwarp();
        }
    }
    // start filling the tile; returns the number of valid problems in it
    PNP_DEV int issue(long long tile, int lane)
    {
        const long long b0 = tile * kTileProblems;
        const int valid = (int)((B - b0 < kTileProblems) ? (B - b0) : kTileProblems);
        if (use_tma) {
            if (lane == 0) mbar_expect_tx(bar, row_bytes * (uint32_t)valid);
            __syncwarp();
            if (lane < valid) bulk_copy_g2s(rows + (size_t)lane * row_pitch, uv + (size_t)(b0 + lane) * n_total * 2, row_bytes, bar);
        } else {
            // rows not 16-byte granular (FP32 with odd n_total): coalesced element loads instead
            const int per_row = n_total * 2;
            for (int e = lane; e < valid * per_row; e += 32) {
                const int p = e / per_row, c = e - p * per_row;
                rows[(size_t)p * row_pitch + c] = __ldg(uv + (size_t)b0 * per_row + e);
            }
        }
        return valid;
    }
    // wait for the fill, normalise, return this lane's row (spare lanes of a ragged tile shadow
    // the last valid problem so that the whole warp stays converged)
    PNP_DEV const T* acquire(int lane, int valid)
    {
        typedef typename Vec2<T>::type V2;
        if (use_tma) { mbar_wait(bar, phase); phase ^= 1u; }
        else         { __syncwarp(); }
        const int my = (lane < valid) ? lane : (valid - 1);
        T* row = rows + (size_t)my * row_pitch;
        if (normalise && lane < valid) {                  // nu = K^-1 [u, v, 1]^T (:3305)
            V2* r2 = reinterpret_cast<V2*>(row);
#pragma unroll 4
            for (int i = 0; i < n_total; ++i) {
                const V2 px = r2[i];
                V2 o;
                normalise_px<T>(px.x, px.y, k00, k01, k02, k10, k11, k12, o.x, o.y);
                r2[i] = o;
            }
        }
        __syncwarp();
        return row;
    }
    // generic-proxy accesses to the tile are done; the next async-proxy fill may start
    PNP_DEV void release()
    {
        __syncwarp();
        fence_proxy_async();
    }
};

template <typename T>
PNP_DEV uint64_t* carve_bar(unsigned char* smem_raw, const void* after)
{
    return reinterpret_cast<uint64_t*>(smem_raw + (((size_t)((const unsigned char*)after - smem_raw) + 7) & ~(size_t)7));
}


struct RowGeom { int row_pitch, use_tma; size_t tile_bytes; };

template <typename T>
inline RowGeom row_geometry(int n_total)
{
    // row pitch = odd multiple of 16 bytes (conflict-free 16-byte per-lane reads, TMA-aligned)
    RowGeom g;
    const size_t row_bytes = (size_t)n_total * 2 * sizeof(T);
    size_t units = (row_bytes + 15) / 16;
    if ((units & 1) == 0) ++units;
    g.row_pitch = (int)(units * 16 / sizeof(T));
    g.use_tma = (row_bytes % 16 == 0) ? 1 : 0;
    g.tile_bytes = (size_t)kTileProblems * g.row_pitch * sizeof(T);
    return g;
}

// ------------------------------------------------------------------------------------------
// Row stream: the same 32 problems per warp, but for kernels that read every pixel ONCE
// (moments, residual, error report).  Rows are streamed in chunks of `chunk` points through two
// small shared-memory buffers (one mbarrier per buffer), so a warp holds ~17 KB instead of a whole
// 35 KB tile and twice as many warps fit per SM, and the copy of chunk c+1 overlaps the arithmetic
// on chunk c.  A chunk of all 32 rows is ONE TMA tensor copy (2-D tensor map over uv[B][2 n], box =
// chunk x 32 rows, issued by lane 0; rows and columns past the end are zero-filled and counted) when
// the buffer rows are dense (pitch = chunk, the normal case); otherwise lane l bulk-copies its own row
// chunk, which the compiler serialises into 32 UBLKCP issues with a broadcast each.
// ------------------------------------------------------------------------------------------
struct StreamGeom { int chunk, pitch, use_stream; size_t buf_bytes; };
constexpr int kStreamChunkUnits = 17;                     // 272-byte chunks

// Points per chunk, in units of 16 bytes.  Odd, so that the row pitch is an odd multiple of 16 B.
// Smaller chunks = smaller buffers = more resident warps (shared memory is what limits them), but
// more mbarrier round trips per row.  PNPB200_STREAM_CHUNK overrides the default (tuning only).
inline int stream_chunk_units()
{
    static const int units = []() {
        const char* e = getenv("PNPB200_STREAM_CHUNK");
        int u = e ? atoi(e) : 0;
        if (u < 1 || u > 127) u = kStreamChunkUnits;
        return u | 1;
    }();
    return units;
}

template <typename T>
inline StreamGeom stream_geometry(int n_total)
{
    StreamGeom g;
    const int per16 = 16 / (2 * (int)sizeof(T));             // points per 16 bytes: 1 (double), 2 (float)
    g.use_stream = (n_total % per16 == 0) ? 1 : 0;
    int c = stream_chunk_units() * per16;
    if (c > n_total) c = n_total;
    g.chunk = c;
    size_t units = ((size_t)c * 2 * sizeof(T) + 15) / 16;
    if ((units & 1) == 0) ++units;                            // odd multiple of 16 B: conflict-free lanes
    g.pitch = (int)(units * 16 / sizeof(T));
    g.buf_bytes = (size_t)kTileProblems * g.pitch * sizeof(T);
    return g;
}

template <typename T>
struct RowStream {
    typedef typename Vec2<T>::type V2;
    T* buf0;            // two buffers of kTileProblems * pitch elements
    uint64_t* bar;      // two mbarriers
    const T* uv;
    long long B, b0;
    int n_total, chunk, pitch, n_chunks, valid;
    uint32_t phase;     // bit s = parity to wait for on buffer s
    const void* tmap;   // tensor map of uv (kernel parameter space), or nullptr

    PNP_DEV T* buf(int s) const { return buf0 + (size_t)s * kTileProblems * pitch; }

    PNP_DEV void init(T* smem, uint64_t* bars, const T* uv_, long long B_, int n_total_, int chunk_, int pitch_, int lane,
                      const void* tmap_ = nullptr)
    {
        buf0 = smem;
        tmap = (pitch_ == chunk_ * 2) ? tmap_ : nullptr;
        bar = bars; uv = uv_; B = B_; n_total = n_total_; chunk = chunk_; pitch = pitch_;
        n_chunks = (n_total + chunk - 1) / chunk;
        phase = 0;
        if (lane == 0) { mbar_init(bar, 1); mbar_init(bar + 1, 1); }
        __syncwarp();
    }
    PNP_DEV int count(int c) const { const int rem = n_total - c * chunk; return rem < chunk ? rem : chunk; }
    PNP_DEV void issue(int c, int lane)
    {
        const int s = c & 1;
        if (tmap) {
            if (lane == 0) {
                mbar_expect_tx(bar + s, (uint32_t)kTileProblems * (uint32_t)pitch * (uint32_t)sizeof(T));   // the full box
                tensor_copy_2d_g2s(buf(s), tmap, c * chunk * 2, (int)b0, bar + s);
            }
            return;
        }
        const uint32_t bytes = (uint32_t)count(c) * 2u * (uint32_t)sizeof(T);
        if (lane == 0) mbar_expect_tx(bar + s, bytes * (uint32_t)valid);
        __syncwarp();
        if (lane < valid)
            bulk_copy_g2s(buf(s) + (size_t)lane * pitch, uv + ((size_t)(b0 + lane) * n_total + (size_t)c * chunk) * 2, bytes, bar + s);
    }
    PNP_DEV void begin_tile(long long tile, int lane)
    {
        b0 = tile * kTileProblems;
        valid = (int)((B - b0 < kTileProblems) ? (B - b0) : kTileProblems);
        issue(0, lane);
        if (n_chunks > 1) issue(1, lane);
    }
    // this lane's row chunk c (spare lanes of a ragged tile shadow the last valid problem)
    PNP_DEV const V2* wait(int c, int lane)
    {
        const int s = c & 1;
        mbar_wait(bar + s, (phase >> s) & 1u);
        phase ^= (1u << s);
        const int my = (lane < valid) ? lane : (valid - 1);
        return reinterpret_cast<const V2*>(buf(s) + (size_t)my * pitch);
    }
    // chunk c has been consumed by every lane: its buffer may be refilled with chunk c + 2
    PNP_DEV void done(int c, int lane)
    {
        __syncwarp();
        if (c + 2 < n_chunks) {
            fence_proxy_async();
            issue(c + 2, lane);
        }
    }
};

}  // namespace pnpb200
