// Host <-> device movement of whole batches of tiles for the tile loops, and the evaluation
// sums of a decoded batch.
//
// The reference rechunks the slide into patch_size^2 tiles with dask and hands them to the
// codec one at a time (src/compress.py:101-128); decompress.py:72-96 does the reverse.  Here a
// batch of tiles moves between the row-major H x W x c slide in (page-locked) host memory and a
// tile-major device buffer as strided DMA copies -- no host-side gather, no staging copy -- on
// the caller's stream, so uploads, kernels and downloads of neighbouring batches overlap.
#include "cae_common.cuh"

#include <vector>

// dst[k] (device, ps x ps x c, tile-major) = tile (tile_yx[2k], tile_yx[2k+1]) of the host image;
// the part of an edge tile beyond the image is zero (zarr's chunk padding, fill_value 0).
extern "C" int cae_tiles_upload_u8(const uint8_t *src, int64_t H, int64_t W, int c, int ps,
                                   const int32_t *tile_yx, int n, uint8_t *dst, void *stream) {
  CAE_CHECK(src && dst && tile_yx && H > 0 && W > 0 && c > 0 && ps > 0 && n >= 0, 2,
            "cae_tiles_upload_u8: bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  const size_t row = (size_t)ps * c, tile = row * ps;
  for (int k = 0; k < n; ++k) {
    const int64_t y0 = (int64_t)tile_yx[2 * k] * ps, x0 = (int64_t)tile_yx[2 * k + 1] * ps;
    CAE_CHECK(y0 >= 0 && x0 >= 0 && y0 < H && x0 < W, 2, "cae_tiles_upload_u8: tile %d outside the image", k);
    const int64_t h_in = y0 + ps <= H ? ps : H - y0, w_in = x0 + ps <= W ? ps : W - x0;
    uint8_t *d = dst + (size_t)k * tile;
    if (h_in < ps || w_in < ps) CAE_CUDA(cudaMemsetAsync(d, 0, tile, st));
    CAE_CUDA(cudaMemcpy2DAsync(d, row, src + ((size_t)y0 * W + x0) * c, (size_t)W * c,
                               (size_t)w_in * c, (size_t)h_in, cudaMemcpyHostToDevice, st));
  }
  return 0;
}

// The inverse: tile k of the device buffer -> its place in the host image (edge tiles cropped).
extern "C" int cae_tiles_download_u8(const uint8_t *src, int n, int ps, int c,
                                     const int32_t *tile_yx, uint8_t *dst, int64_t H, int64_t W,
                                     void *stream) {
  CAE_CHECK(src && dst && tile_yx && H > 0 && W > 0 && c > 0 && ps > 0 && n >= 0, 2,
            "cae_tiles_download_u8: bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  const size_t row = (size_t)ps * c, tile = row * ps;
  for (int k = 0; k < n; ++k) {
    const int64_t y0 = (int64_t)tile_yx[2 * k] * ps, x0 = (int64_t)tile_yx[2 * k + 1] * ps;
    CAE_CHECK(y0 >= 0 && x0 >= 0 && y0 < H && x0 < W, 2, "cae_tiles_download_u8: tile %d outside the image", k);
    const int64_t h_in = y0 + ps <= H ? ps : H - y0, w_in = x0 + ps <= W ? ps : W - x0;
    CAE_CUDA(cudaMemcpy2DAsync(dst + ((size_t)y0 * W + x0) * c, (size_t)W * c, src + (size_t)k * tile,
                               row, (size_t)w_in * c, (size_t)h_in, cudaMemcpyDeviceToHost, st));
  }
  return 0;
}

// ---------------------------------------------------------------------------------------------
// Banded variants.  The per-tile copies above move rows of ps * c bytes (1.5 KB for 512^2 RGB
// tiles): 38-42 GB/s on a link that does 56 GB/s with long rows (tools/micro/iobench.py).  Tiles
// that sit side by side in one tile row of the slide (the order the tile loops walk them) are
// therefore exchanged as ONE two-dimensional copy of the whole band segment -- rows of r * ps * c
// bytes -- with a device kernel re-tiling between the tile-major buffer and a band-major scratch
// buffer of the same size (16-byte units, HBM bound, ~1 % of the copy's time).
namespace {
// tiles [r][ps][row16] <-> band [ps][r][row16], 16-byte units
__global__ void __launch_bounds__(256) retile_kernel(const uint4 *__restrict__ src, uint4 *__restrict__ dst,
                                                     int r, int ps, int row16, int to_band) {
  const size_t total = (size_t)r * ps * row16;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (size_t)gridDim.x * blockDim.x) {
    const int u = (int)(i % row16);
    const size_t q = i / row16;
    // i indexes the band: (y, k, u)
    const int k = (int)(q % r), y = (int)(q / r);
    const size_t t = ((size_t)k * ps + y) * row16 + u;
    if (to_band) dst[i] = src[t]; else dst[t] = src[i];
  }
}

// length of the run of full-size tiles starting at k that continue tile k's row to the right
inline int band_run(const int32_t *tile_yx, int k, int n, int ps, int64_t H, int64_t W) {
  const int64_t y0 = (int64_t)tile_yx[2 * k] * ps;
  if (y0 + ps > H) return 0;
  int r = 0;
  while (k + r < n && tile_yx[2 * (k + r)] == tile_yx[2 * k] &&
         tile_yx[2 * (k + r) + 1] == tile_yx[2 * k + 1] + r &&
         ((int64_t)tile_yx[2 * (k + r) + 1] + 1) * ps <= W)
    ++r;
  return r;
}
}  // namespace

extern "C" int cae_tiles_download_u8_banded(const uint8_t *src, int n, int ps, int c,
                                            const int32_t *tile_yx, uint8_t *dst, int64_t H,
                                            int64_t W, uint8_t *scratch, void *stream) {
  CAE_CHECK(src && dst && tile_yx && scratch && H > 0 && W > 0 && c > 0 && ps > 0 && n >= 0, 2,
            "cae_tiles_download_u8_banded: bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  const size_t row = (size_t)ps * c, tile = row * ps;
  const bool units = row % 16 == 0 && ((uintptr_t)src % 16 == 0) && ((uintptr_t)scratch % 16 == 0);
  for (int k = 0; k < n;) {
    const int r = units ? band_run(tile_yx, k, n, ps, H, W) : 0;
    if (r < 2) {
      if (int rc = cae_tiles_download_u8(src + (size_t)k * tile, 1, ps, c, tile_yx + 2 * k, dst, H, W, stream))
        return rc;
      ++k;
      continue;
    }
    const int64_t y0 = (int64_t)tile_yx[2 * k] * ps, x0 = (int64_t)tile_yx[2 * k + 1] * ps;
    uint8_t *band = scratch + (size_t)k * tile;
    const size_t total = (size_t)r * ps * (row / 16);
    const int blocks = (int)((total + 255) / 256 < (size_t)(8 * cae_sm_count()) ? (total + 255) / 256 : 8 * cae_sm_count());
    retile_kernel<<<blocks, 256, 0, st>>>(reinterpret_cast<const uint4 *>(src + (size_t)k * tile),
                                          reinterpret_cast<uint4 *>(band), r, ps, (int)(row / 16), 1);
    cae_count_launch();
    CAE_CUDA(cudaGetLastError());
    CAE_CUDA(cudaMemcpy2DAsync(dst + ((size_t)y0 * W + x0) * c, (size_t)W * c, band, (size_t)r * row,
                               (size_t)r * row, (size_t)ps, cudaMemcpyDeviceToHost, st));
    k += r;
  }
  return 0;
}

extern "C" int cae_tiles_upload_u8_banded(const uint8_t *src, int64_t H, int64_t W, int c, int ps,
                                          const int32_t *tile_yx, int n, uint8_t *dst,
                                          uint8_t *scratch, void *stream) {
  CAE_CHECK(src && dst && tile_yx && scratch && H > 0 && W > 0 && c > 0 && ps > 0 && n >= 0, 2,
            "cae_tiles_upload_u8_banded: bad argument");
  cudaStream_t st = (cudaStream_t)stream;
  const size_t row = (size_t)ps * c, tile = row * ps;
  const bool units = row % 16 == 0 && ((uintptr_t)dst % 16 == 0) && ((uintptr_t)scratch % 16 == 0);
  for (int k = 0; k < n;) {
    const int r = units ? band_run(tile_yx, k, n, ps, H, W) : 0;
    if (r < 2) {
      if (int rc = cae_tiles_upload_u8(src, H, W, c, ps, tile_yx + 2 * k, 1, dst + (size_t)k * tile, stream))
        return rc;
      ++k;
      continue;
    }
    const int64_t y0 = (int64_t)tile_yx[2 * k] * ps, x0 = (int64_t)tile_yx[2 * k + 1] * ps;
    uint8_t *band = scratch + (size_t)k * tile;
    CAE_CUDA(cudaMemcpy2DAsync(band, (size_t)r * row, src + ((size_t)y0 * W + x0) * c, (size_t)W * c,
                               (size_t)r * row, (size_t)ps, cudaMemcpyHostToDevice, st));
    const size_t total = (size_t)r * ps * (row / 16);
    const int blocks = (int)((total + 255) / 256 < (size_t)(8 * cae_sm_count()) ? (total + 255) / 256 : 8 * cae_sm_count());
    retile_kernel<<<blocks, 256, 0, st>>>(reinterpret_cast<const uint4 *>(band),
                                          reinterpret_cast<uint4 *>(dst + (size_t)k * tile), r, ps,
                                          (int)(row / 16), 0);
    cae_count_launch();
    CAE_CUDA(cudaGetLastError());
    k += r;
  }
  return 0;
}

// ---------------------------------------------------------------------------------------------
// Region reads and writes (region.py).  A piece {k, b, sy, sx, dy, dx, h, w} pairs rows
// [sy, sy + h) x columns [sx, sx + w) of tile k with rows [dy, dy + h) x columns [dx, dx + w) of
// box b.  cae_tiles_crop_u8 copies tile -> box (k = -1 writes zeros: zarr's fill value for a chunk
// whose file is missing); cae_tiles_paste_u8 copies box -> tile (b = -1 writes zeros: the padding
// of edge chunks).  HBM bound.  Block (p, q) copies rows [q * rows, (q + 1) * rows) of piece p in
// the widest unit that the piece's source rows, destination rows and row length all allow (16, 4
// or 1 bytes): with c = 3 and windows at arbitrary offsets the byte loop is the common case.
namespace {
constexpr int kCropThreads = 256;

template <typename T>
__device__ __forceinline__ void crop_rows(const uint8_t *src, size_t src_pitch, uint8_t *dst,
                                          size_t dst_pitch, int rows, int row_bytes) {
  const int units = row_bytes / (int)sizeof(T);
  const int total = rows * units;
  for (int i = threadIdx.x; i < total; i += kCropThreads) {
    const int r = i / units, u = i - r * units;
    T *d = reinterpret_cast<T *>(dst + r * dst_pitch) + u;
    if (src) *d = __ldg(reinterpret_cast<const T *>(src + r * src_pitch) + u);
    else *d = T{};
  }
}

// `rows` rows of `row_bytes` from src (nullptr: zeros) to dst in the widest unit that fits
__device__ __forceinline__ void copy_rows(const uint8_t *src, size_t src_pitch, uint8_t *dst,
                                          size_t dst_pitch, int rows, int row_bytes) {
  const uintptr_t bits = reinterpret_cast<uintptr_t>(dst) | dst_pitch | (uintptr_t)row_bytes |
                         (src ? reinterpret_cast<uintptr_t>(src) | src_pitch : 0);
  if ((bits & 15) == 0) crop_rows<uint4>(src, src_pitch, dst, dst_pitch, rows, row_bytes);
  else if ((bits & 3) == 0) crop_rows<uint32_t>(src, src_pitch, dst, dst_pitch, rows, row_bytes);
  else crop_rows<uint8_t>(src, src_pitch, dst, dst_pitch, rows, row_bytes);
}

__global__ void __launch_bounds__(kCropThreads) tiles_crop_u8_kernel(
    const uint8_t *__restrict__ tiles, int ps, int c, const int4 *__restrict__ pieces,
    uint8_t *__restrict__ out, int box_h, int box_w, int rows_per_block) {
  const int4 p0 = pieces[2 * blockIdx.x], p1 = pieces[2 * blockIdx.x + 1];
  const int k = p0.x, b = p0.y, sy = p0.z, sx = p0.w, dy = p1.x, dx = p1.y, h = p1.z, w = p1.w;
  const int r0 = blockIdx.y * rows_per_block;
  if (r0 >= h) return;
  const uint8_t *src = k < 0 ? nullptr
                             : tiles + (((size_t)k * ps + sy + r0) * ps + sx) * c;
  uint8_t *dst = out + (((size_t)b * box_h + dy + r0) * box_w + dx) * c;
  copy_rows(src, (size_t)ps * c, dst, (size_t)box_w * c, min(rows_per_block, h - r0), w * c);
}

__global__ void __launch_bounds__(kCropThreads) tiles_paste_u8_kernel(
    uint8_t *__restrict__ tiles, int ps, int c, const int4 *__restrict__ pieces,
    const uint8_t *__restrict__ boxes, int box_h, int box_w, int rows_per_block) {
  const int4 p0 = pieces[2 * blockIdx.x], p1 = pieces[2 * blockIdx.x + 1];
  const int k = p0.x, b = p0.y, sy = p0.z, sx = p0.w, dy = p1.x, dx = p1.y, h = p1.z, w = p1.w;
  const int r0 = blockIdx.y * rows_per_block;
  if (r0 >= h) return;
  const uint8_t *src = b < 0 ? nullptr
                             : boxes + (((size_t)b * box_h + dy + r0) * box_w + dx) * c;
  uint8_t *dst = tiles + (((size_t)k * ps + sy + r0) * ps + sx) * c;
  copy_rows(src, (size_t)box_w * c, dst, (size_t)ps * c, min(rows_per_block, h - r0), w * c);
}

// Host side of both: every piece is checked before anything is copied or launched (k >= tile_min,
// b >= box_min; a piece lies inside its tile, and inside its box unless b = -1), then the table
// goes up to pieces_dev on the stream and the grid is sized.
int check_pieces(const char *fn, const int32_t *pieces, int m, int n_tiles, int tile_min,
                 int n_boxes, int box_min, int ps, int c, int box_h, int box_w, dim3 *grid,
                 int *rows_per_block) {
  CAE_CHECK((int64_t)ps * ps * c <= INT32_MAX && (int64_t)box_w * c <= INT32_MAX, 2,
            "%s: tile or box row too large", fn);
  int max_h = 0, max_row = 0;
  for (int i = 0; i < m; ++i) {
    const int32_t *p = pieces + 8 * (size_t)i;
    const int k = p[0], b = p[1], sy = p[2], sx = p[3], dy = p[4], dx = p[5], h = p[6], w = p[7];
    CAE_CHECK(k >= tile_min && k < n_tiles, 2, "%s: piece %d names tile %d of %d", fn, i, k,
              n_tiles);
    CAE_CHECK(b >= box_min && b < n_boxes, 2, "%s: piece %d names box %d of %d", fn, i, b,
              n_boxes);
    CAE_CHECK(h > 0 && w > 0 && sy >= 0 && sx >= 0 && sy <= ps - h && sx <= ps - w, 2,
              "%s: piece %d (rows %d+%d, columns %d+%d) lies outside its %d^2 tile",
              fn, i, sy, h, sx, w, ps);
    CAE_CHECK(b < 0 || (dy >= 0 && dx >= 0 && dy <= box_h - h && dx <= box_w - w), 2,
              "%s: piece %d (rows %d+%d, columns %d+%d) lies outside its %d x %d box",
              fn, i, dy, h, dx, w, box_h, box_w);
    max_h = h > max_h ? h : max_h;
    max_row = w * c > max_row ? w * c : max_row;
  }
  // ~8 KB per block: enough work to hide the piece lookup, enough blocks for small requests
  int rows = 8192 / max_row;
  rows = rows < 1 ? 1 : rows > 64 ? 64 : rows;
  const int grid_y = (max_h + rows - 1) / rows;
  CAE_CHECK(grid_y <= 65535, 2, "%s: pieces of %d rows are too tall", fn, max_h);
  *grid = dim3((unsigned)m, (unsigned)grid_y);
  *rows_per_block = rows;
  return 0;
}
}  // namespace

extern "C" int cae_tiles_crop_u8(const uint8_t *tiles, int n_tiles, int ps, int c,
                                 const int32_t *pieces, int m, int32_t *pieces_dev, uint8_t *out,
                                 int n_boxes, int box_h, int box_w, void *stream) {
  CAE_CHECK(n_tiles >= 0 && ps > 0 && c > 0 && m >= 0 && n_boxes > 0 && box_h > 0 && box_w > 0, 2,
            "cae_tiles_crop_u8: bad argument");
  if (m == 0) return 0;
  CAE_CHECK(pieces && pieces_dev && out && (tiles || n_tiles == 0), 2,
            "cae_tiles_crop_u8: null pointer");
  CAE_CHECK((uintptr_t)pieces_dev % 16 == 0, 2, "cae_tiles_crop_u8: pieces_dev is not 16-byte aligned");
  dim3 grid;
  int rows;
  if (int rc = check_pieces("cae_tiles_crop_u8", pieces, m, n_tiles, -1, n_boxes, 0, ps, c, box_h,
                            box_w, &grid, &rows))
    return rc;
  cudaStream_t st = (cudaStream_t)stream;
  CAE_CUDA(cudaMemcpyAsync(pieces_dev, pieces, sizeof(int32_t) * 8 * (size_t)m,
                           cudaMemcpyHostToDevice, st));
  tiles_crop_u8_kernel<<<grid, kCropThreads, 0, st>>>(
      tiles, ps, c, reinterpret_cast<const int4 *>(pieces_dev), out, box_h, box_w, rows);
  cae_count_launch();
  CAE_CUDA(cudaGetLastError());
  return 0;
}

extern "C" int cae_tiles_paste_u8(uint8_t *tiles, int n_tiles, int ps, int c,
                                  const int32_t *pieces, int m, int32_t *pieces_dev,
                                  const uint8_t *boxes, int n_boxes, int box_h, int box_w,
                                  void *stream) {
  CAE_CHECK(n_tiles >= 0 && ps > 0 && c > 0 && m >= 0 && n_boxes >= 0 && box_h > 0 && box_w > 0, 2,
            "cae_tiles_paste_u8: bad argument");
  if (m == 0) return 0;
  CAE_CHECK(pieces && pieces_dev && tiles && (boxes || n_boxes == 0), 2,
            "cae_tiles_paste_u8: null pointer");
  CAE_CHECK((uintptr_t)pieces_dev % 16 == 0, 2, "cae_tiles_paste_u8: pieces_dev is not 16-byte aligned");
  dim3 grid;
  int rows;
  if (int rc = check_pieces("cae_tiles_paste_u8", pieces, m, n_tiles, 0, n_boxes, -1, ps, c, box_h,
                            box_w, &grid, &rows))
    return rc;
  cudaStream_t st = (cudaStream_t)stream;
  CAE_CUDA(cudaMemcpyAsync(pieces_dev, pieces, sizeof(int32_t) * 8 * (size_t)m,
                           cudaMemcpyHostToDevice, st));
  tiles_paste_u8_kernel<<<grid, kCropThreads, 0, st>>>(
      tiles, ps, c, reinterpret_cast<const int4 *>(pieces_dev), boxes, box_h, box_w, rows);
  cae_count_launch();
  CAE_CUDA(cudaGetLastError());
  return 0;
}

// ---------------------------------------------------------------------------------------------
// Reduced-resolution region reads (region.SlideLevel).  A piece is the crop's record in level-f
// pixels followed by the in-array extent of tile k in level-0 pixels: {k, b, sy, sx, dy, dx, h, w,
// vh, vw, 0, 0}.  Level pixel (i, j) of tile k, channel ch, is the mean, rounded half up, of
// level-0 rows [i f, min((i + 1) f, vh)) x columns [j f, min((j + 1) f, vw)) of the tile: the
// decoded padding of an edge tile never enters a mean.  k = -1 writes zeros.
//
// Bound by the source bytes it reads (a batch of decoded tiles, just written by the synthesis and
// L2-resident); the output is 1/f^2 of them.  Block (p, q, r) covers nb output rows x wb output
// columns of piece p, sized to read ~32 KB.  Its threads own VEC-byte units of the source rows
// (16 where the tiles allow) and split the f source rows of each output row among `split` thread
// groups: each thread sums its rows of its unit in registers and adds the sums into the block's
// column sums in shared memory.  Then groups of g lanes each add part of one output element's f
// columns (stride c in shared memory: no bank conflicts for odd c) and finish with shuffles.
namespace {
constexpr int kReduceThreads = 256;
constexpr int kReduceSource = 32768;   // source bytes per block
constexpr int kReduceSpan = 4096;      // source bytes per row of a block, unless one pixel is wider
constexpr int kReduceSmem = 40960;     // column sums per block, bytes

template <int VEC>
__device__ __forceinline__ void add_unit(const uint8_t *p, uint32_t (&acc)[VEC]) {
  if constexpr (VEC == 16) {
    const uint4 v = __ldg(reinterpret_cast<const uint4 *>(p));
    const uint32_t wd[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
    for (int i = 0; i < 16; ++i) acc[i] += (wd[i >> 2] >> (8 * (i & 3))) & 255u;
  } else if constexpr (VEC == 4) {
    const uint32_t v = __ldg(reinterpret_cast<const uint32_t *>(p));
#pragma unroll
    for (int i = 0; i < 4; ++i) acc[i] += (v >> (8 * i)) & 255u;
  } else {
    acc[0] += __ldg(p);
  }
}

// n / d as a multiply-high by m = magic(d) = ceil(2^32 / d): exact while n * d < 2^32
__device__ __forceinline__ uint32_t magic(uint32_t d) { return d == 1 ? 0u : 0xFFFFFFFFu / d + 1; }
__device__ __forceinline__ uint32_t div_by(uint32_t n, uint32_t d, uint32_t m) {
  return d == 1 ? n : __umulhi(n, m);
}

template <int VEC>
__global__ void __launch_bounds__(kReduceThreads, 4) tiles_crop_reduce_u8_kernel(
    const uint8_t *__restrict__ tiles, int ps, int c, int lf, const int4 *__restrict__ pieces,
    uint8_t *__restrict__ out, int box_h, int box_w, int nb, int wb, int g) {
  extern __shared__ uint32_t colsum[];
  const int4 p0 = pieces[3 * blockIdx.x], p1 = pieces[3 * blockIdx.x + 1],
             p2 = pieces[3 * blockIdx.x + 2];
  const int k = p0.x, b = p0.y, sy = p0.z, sx = p0.w, dy = p1.x, dx = p1.y, h = p1.z, w = p1.w;
  const int vh = p2.x, vw = p2.y;
  const int o0 = blockIdx.y * nb, j0 = blockIdx.z * wb;
  if (o0 >= h || j0 >= w) return;
  const int f = 1 << lf, rows = min(nb, h - o0), cols = min(wb, w - j0);
  const int row_out = cols * c, n_out = rows * row_out;
  uint8_t *dst = out + (((size_t)b * box_h + dy + o0) * box_w + dx + j0) * c;
  const size_t dst_pitch = (size_t)box_w * c;
  if (k < 0) {
    for (int e = threadIdx.x; e < n_out; e += kReduceThreads) {
      const int o = e / row_out;
      dst[o * dst_pitch + e - o * row_out] = 0;
    }
    return;
  }
  // bytes [a0, end) of every source row: the block's columns, from a VEC-aligned start
  const int a0 = (((sx + j0) << lf) * c) & ~(VEC - 1);
  const int end = min((sx + j0 + cols) << lf, vw) * c;
  const int units = (end - a0 + VEC - 1) / VEC, stride = units * VEC;
  // vertical: item (rg, o, u) sums rows rg, rg + split, ... < f of output row o, unit u.  Threads
  // share an (o, u) only when there are too few of them to fill the block (large f); then the
  // sums meet through shared-memory atomics, else each (o, u) has one writer.
  const int pairs = rows * units;
  int split = 1;
  while (split < f && 2 * split * pairs <= kReduceThreads) split *= 2;
  if (split > 1) {
    for (int i = threadIdx.x; i < rows * stride; i += kReduceThreads) colsum[i] = 0;
    __syncthreads();
  }
  const int row0 = (sy + o0) << lf;
  const int src_rows = min(rows << lf, vh - row0);           // the band's rows inside the array
  const size_t pitch = (size_t)ps * c;
  const uint8_t *src = tiles + ((size_t)k * ps + row0) * pitch + a0;
  const uint32_t m_units = magic(units), m_rows = magic(rows);
  for (int i = threadIdx.x; i < pairs * split; i += kReduceThreads) {
    const int q = (int)div_by(i, units, m_units), u = i - q * units;
    const int rg = (int)div_by(q, rows, m_rows), o = q - rg * rows;
    const int t_end = min(f, src_rows - (o << lf));
    uint32_t acc[VEC] = {};
#pragma unroll 2
    for (int t = rg; t < t_end; t += split)
      add_unit<VEC>(src + (size_t)((o << lf) + t) * pitch + u * VEC, acc);
    uint32_t *cs = colsum + o * stride + u * VEC;
    if (split == 1) {
#pragma unroll
      for (int v = 0; v < VEC; ++v) cs[v] = acc[v];
    } else if (rg < t_end) {
#pragma unroll
      for (int v = 0; v < VEC; ++v) atomicAdd(cs + v, acc[v]);
    }
  }
  __syncthreads();
  // horizontal: g lanes per output element, each adding every g-th of its columns
  const int lane = threadIdx.x & (g - 1), per_pass = kReduceThreads / g;
  const uint32_t m_row = magic(row_out), m_c = magic(c);
  for (int e0 = 0; e0 < n_out; e0 += per_pass) {
    const int e = e0 + threadIdx.x / g;
    uint32_t s = 0;
    int o = 0, r = 0, nc = f, nr = f;
    if (e < n_out) {
      o = (int)div_by(e, row_out, m_row);
      r = e - o * row_out;
      const int jj = (int)div_by(r, c, m_c), ch = r - jj * c;
      const int col0 = (sx + j0 + jj) << lf;
      nc = min(f, vw - col0);
      nr = min(f, vh - row0 - (o << lf));
      const uint32_t *cs = colsum + o * stride + col0 * c + ch - a0;
      for (int t = lane; t < nc; t += g) s += cs[t * c];
    }
    for (int off = g >> 1; off > 0; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
    if (e < n_out && lane == 0) {
      const uint32_t n = (uint32_t)nc * (uint32_t)nr;      // f^2 except in edge blocks
      dst[o * dst_pitch + r] = (uint8_t)(n == (1u << 2 * lf) ? (s + n / 2) >> 2 * lf : (s + n / 2) / n);
    }
  }
}
}  // namespace

extern "C" int cae_tiles_crop_reduce_u8(const uint8_t *tiles, int n_tiles, int ps, int c, int f,
                                        const int32_t *pieces, int m, int32_t *pieces_dev,
                                        uint8_t *out, int n_boxes, int box_h, int box_w,
                                        void *stream) {
  const char *fn = "cae_tiles_crop_reduce_u8";
  CAE_CHECK(n_tiles >= 0 && ps > 0 && c > 0 && m >= 0 && n_boxes > 0 && box_h > 0 && box_w > 0, 2,
            "%s: bad argument", fn);
  CAE_CHECK(f >= 1 && f <= 512 && (f & (f - 1)) == 0 && ps % f == 0, 2,
            "%s: the factor %d is not a power of two in [1, 512] that divides the tile size %d", fn,
            f, ps);
  CAE_CHECK((int64_t)ps * ps * c <= INT32_MAX && (int64_t)box_w * c <= INT32_MAX, 2,
            "%s: tile or box row too large", fn);
  CAE_CHECK(((int64_t)f * c + 32) * 4 <= kReduceSmem, 2, "%s: %d x %d bytes per pixel is too wide",
            fn, f, c);
  if (m == 0) return 0;
  CAE_CHECK(pieces && pieces_dev && out && (tiles || n_tiles == 0), 2, "%s: null pointer", fn);
  CAE_CHECK((uintptr_t)pieces_dev % 16 == 0, 2, "%s: pieces_dev is not 16-byte aligned", fn);
  const int lps = ps / f;
  int max_h = 0, max_w = 0;
  for (int i = 0; i < m; ++i) {
    const int32_t *p = pieces + 12 * (size_t)i;
    const int k = p[0], b = p[1], sy = p[2], sx = p[3], dy = p[4], dx = p[5], h = p[6], w = p[7];
    const int vh = p[8], vw = p[9];
    CAE_CHECK(k >= -1 && k < n_tiles, 2, "%s: piece %d names tile %d of %d", fn, i, k, n_tiles);
    CAE_CHECK(b >= 0 && b < n_boxes, 2, "%s: piece %d names box %d of %d", fn, i, b, n_boxes);
    CAE_CHECK(h > 0 && w > 0 && sy >= 0 && sx >= 0 && sy <= lps - h && sx <= lps - w, 2,
              "%s: piece %d (rows %d+%d, columns %d+%d) lies outside its %d^2 level tile", fn, i,
              sy, h, sx, w, lps);
    CAE_CHECK(vh > 0 && vw > 0 && vh <= ps && vw <= ps, 2,
              "%s: piece %d: in-array extent %d x %d of a %d^2 tile", fn, i, vh, vw, ps);
    CAE_CHECK((int64_t)(sy + h - 1) * f < vh && (int64_t)(sx + w - 1) * f < vw, 2,
              "%s: piece %d (rows %d+%d, columns %d+%d) starts past the in-array part %d x %d",
              fn, i, sy, h, sx, w, vh, vw);
    CAE_CHECK(dy >= 0 && dx >= 0 && dy <= box_h - h && dx <= box_w - w, 2,
              "%s: piece %d (rows %d+%d, columns %d+%d) lies outside its %d x %d box", fn, i, dy,
              h, dx, w, box_h, box_w);
    max_h = h > max_h ? h : max_h;
    max_w = w > max_w ? w : max_w;
  }
  if (f == 1) {   // the level image is the slide itself: the crop kernel copies in wide units
    std::vector<int32_t> p8(8 * (size_t)m);
    for (int i = 0; i < m; ++i)
      for (int j = 0; j < 8; ++j) p8[8 * (size_t)i + j] = pieces[12 * (size_t)i + j];
    return cae_tiles_crop_u8(tiles, n_tiles, ps, c, p8.data(), m, pieces_dev, out, n_boxes, box_h,
                             box_w, stream);
  }
  const int vec = tiles == nullptr ? 16
                  : ((uintptr_t)tiles | (uintptr_t)ps * c) % 16 == 0 ? 16
                  : ((uintptr_t)tiles | (uintptr_t)ps * c) % 4 == 0  ? 4 : 1;
  // a block: ~kReduceSource source bytes, rows of at most kReduceSpan bytes (or one pixel)
  const int fc = f * c;
  int span = kReduceSource / f < kReduceSpan ? kReduceSource / f : kReduceSpan;
  int wb = (span > fc ? span : fc) / fc;
  wb = wb < max_w ? wb : max_w;
  const int row_smem = (wb * fc + 2 * vec) * 4;
  int nb = kReduceSource / (f * wb * fc);
  nb = nb < kReduceSmem / row_smem ? nb : kReduceSmem / row_smem;
  nb = nb < max_h ? nb : max_h;
  nb = nb < 1 ? 1 : nb;
  const int gy = (max_h + nb - 1) / nb, gz = (max_w + wb - 1) / wb;
  CAE_CHECK(gy <= 65535 && gz <= 65535, 2, "%s: pieces of %d x %d are too large", fn, max_h, max_w);
  int lf = 0;
  while ((1 << lf) < f) ++lf;
  const int g = f / 4 < 1 ? 1 : f / 4 > 32 ? 32 : f / 4;
  cudaStream_t st = (cudaStream_t)stream;
  CAE_CUDA(cudaMemcpyAsync(pieces_dev, pieces, sizeof(int32_t) * 12 * (size_t)m,
                           cudaMemcpyHostToDevice, st));
  const dim3 grid((unsigned)m, (unsigned)gy, (unsigned)gz);
  const size_t smem = (size_t)nb * row_smem;
  const int4 *pd = reinterpret_cast<const int4 *>(pieces_dev);
  if (vec == 16)
    tiles_crop_reduce_u8_kernel<16><<<grid, kReduceThreads, smem, st>>>(tiles, ps, c, lf, pd, out,
                                                                        box_h, box_w, nb, wb, g);
  else if (vec == 4)
    tiles_crop_reduce_u8_kernel<4><<<grid, kReduceThreads, smem, st>>>(tiles, ps, c, lf, pd, out,
                                                                       box_h, box_w, nb, wb, g);
  else
    tiles_crop_reduce_u8_kernel<1><<<grid, kReduceThreads, smem, st>>>(tiles, ps, c, lf, pd, out,
                                                                       box_h, box_w, nb, wb, g);
  cae_count_launch();
  CAE_CUDA(cudaGetLastError());
  return 0;
}

// ---------------------------------------------------------------------------------------------
// Resolution pyramid (region.CompressedSlide.build_pyramid): levels 1..K of a batch of decoded
// tiles in one launch, each tile read once.  Record t = {i, j, vh, vw}: tile t is level-0 chunk
// (i, j) with in-array extent vh x vw; the chunks of one call lie in one level-1 chunk row (equal
// i >> 1, hence equal i >> k at every level), since `out` holds one chunk row per level.  Its level-k pixels, the same means as
// cae_tiles_crop_reduce_u8 at f = 2^k, land in tile j >> k of level k's chunk-row buffer at
// ((i mod 2^k) ps/2^k, (j mod 2^k) ps/2^k); only the ceil(vh/2^k) x ceil(vw/2^k) pixels inside
// the array are written.
//
// Block (q, t) covers a Q x Q square of tile t, Q = max(2^K, S): every level pixel of the square
// lies in it, so no sum crosses blocks.  The block stages S x S level-0 squares (S = 64 or the
// largest power of two dividing ps, if smaller) in shared memory one at a time, zeroing the
// pixels outside the array, and builds the 2 x 2 sums level by level in shared memory (integer
// sums of level-0 pixels at every level, never means of means), storing each level's means as it
// goes.  The S x S totals then feed the levels above log2 S the same way.
namespace {
constexpr int kPyrThreads = 256;
constexpr int kPyrMaxLevels = 9;
constexpr int kPyrSmem = 48 * 1024;

struct PyrLevels {
  int off[kPyrMaxLevels + 1];   // off[k]: first tile of level k's chunk-row buffer in `out`
};

// Level-l pixel (py, px) of the tile (level-l pixels, tile-local), channel ch, from its sum s.
__device__ __forceinline__ void pyr_store(uint8_t *__restrict__ out, const int *off, int ps,
                                          int c, int l, int i, int j, int vh, int vw, int py,
                                          int px, int ch, uint32_t s) {
  const int y0 = py << l, x0 = px << l;
  if (y0 >= vh || x0 >= vw) return;
  const uint32_t n = (uint32_t)min(1 << l, vh - y0) * (uint32_t)min(1 << l, vw - x0);
  const int lps = ps >> l, mask = (1 << l) - 1;
  const size_t row = (size_t)(i & mask) * lps + py, col = (size_t)(j & mask) * lps + px;
  uint8_t *t = out + (size_t)(off[l] + (j >> l)) * ps * ps * c;
  t[(row * ps + col) * c + ch] =
      (uint8_t)(n == (1u << 2 * l) ? (s + n / 2) >> 2 * l : (s + n / 2) / n);
}

// dst (n/2 x n/2 x c) = the 2 x 2 sums of src (n x n x c): level l, whose pixel (y, x) is level-l
// pixel (py0 + y, px0 + x) of the tile.
template <typename T>
__device__ __forceinline__ void pyr_level(const T *src, uint32_t *dst, int n, int c,
                                          uint8_t *__restrict__ out, const int *off, int ps,
                                          int l, int i, int j, int vh, int vw, int py0, int px0) {
  const int h = n >> 1, lh = 31 - __clz(h), m = (h * h) * c;
  for (int e = threadIdx.x; e < m; e += kPyrThreads) {
    const int q = e / c, ch = e - q * c, y = q >> lh, x = q & (h - 1);
    const T *s0 = src + ((size_t)(2 * y) * n + 2 * x) * c + ch;
    const uint32_t s = (uint32_t)s0[0] + (uint32_t)s0[c] + (uint32_t)s0[n * c] +
                       (uint32_t)s0[n * c + c];
    dst[e] = s;
    pyr_store(out, off, ps, c, l, i, j, vh, vw, py0 + y, px0 + x, ch, s);
  }
  __syncthreads();
}

template <int VEC>
__global__ void __launch_bounds__(kPyrThreads) tiles_pyramid_u8_kernel(
    const uint8_t *__restrict__ tiles, int ps, int c, int levels, int ls, int lq,
    const int4 *__restrict__ recs, uint8_t *__restrict__ out, PyrLevels lv) {
  extern __shared__ __align__(16) uint8_t pyr_smem[];
  __shared__ int off[kPyrMaxLevels + 1];
  if (threadIdx.x <= kPyrMaxLevels) off[threadIdx.x] = lv.off[threadIdx.x];
  const int4 r = recs[blockIdx.y];
  const int i = r.x, j = r.y, vh = r.z, vw = r.w;
  const int S = 1 << ls, Q = 1 << lq, per_row = ps >> lq;
  const int Y0 = (blockIdx.x / per_row) << lq, X0 = (blockIdx.x % per_row) << lq;
  if (Y0 >= vh || X0 >= vw) return;          // no pixel of the square is inside the array
  const int row_b = S * c;
  uint8_t *px = pyr_smem;                                                   // S x S x c bytes
  uint32_t *a = reinterpret_cast<uint32_t *>(pyr_smem + ((S * row_b + 15) & ~15));
  uint32_t *b = a + (S / 2) * (S / 2) * c;                                  // (S/4)^2 x c
  uint32_t *top = b + (S / 4) * (S / 4) * c;                                // (Q/S)^2 x c
  uint32_t *top2 = top + (Q / S) * (Q / S) * c;                             // (Q/2S)^2 x c
  const int nsub = Q >> ls, l_in = min(levels, ls);
  const uint8_t *tile = tiles + (size_t)blockIdx.y * ps * ps * c;
  const int units = row_b / VEC;
  for (int s = 0; s < nsub * nsub; ++s) {
    const int y0 = Y0 + (s / nsub) * S, x0 = X0 + (s % nsub) * S;
    const int v_rows = vh - y0, v_bytes = (vw - x0) * c;     // inside the array (may be <= 0)
    for (int u = threadIdx.x; u < S * units; u += kPyrThreads) {
      const int rr = u / units, b0 = (u - rr * units) * VEC;
      const uint8_t *g = tile + ((size_t)(y0 + rr) * ps + x0) * c + b0;
      uint8_t *d = px + rr * row_b + b0;
      if (VEC == 16 && rr < v_rows && b0 + 16 <= v_bytes) {
        *reinterpret_cast<uint4 *>(d) = __ldg(reinterpret_cast<const uint4 *>(g));
      } else {
#pragma unroll
        for (int v = 0; v < VEC; ++v) d[v] = rr < v_rows && b0 + v < v_bytes ? __ldg(g + v) : 0;
      }
    }
    __syncthreads();
    pyr_level<uint8_t>(px, a, S, c, out, off, ps, 1, i, j, vh, vw, y0 >> 1, x0 >> 1);
    uint32_t *src = a, *dst = b;
    for (int l = 2; l <= l_in; ++l) {
      pyr_level<uint32_t>(src, dst, S >> (l - 1), c, out, off, ps, l, i, j, vh, vw, y0 >> l,
                          x0 >> l);
      uint32_t *t = src; src = dst; dst = t;
    }
    // the square's totals (src is 1 x 1 x c when levels > ls); the next square's staging
    // barrier orders this read before `a` and `b` are written again
    if (levels > ls && threadIdx.x < c) top[s * c + threadIdx.x] = src[threadIdx.x];
  }
  if (levels > ls) {
    __syncthreads();
    uint32_t *src = top, *dst = top2;
    for (int l = ls + 1; l <= levels; ++l) {
      pyr_level<uint32_t>(src, dst, nsub >> (l - ls - 1), c, out, off, ps, l, i, j, vh, vw,
                          Y0 >> l, X0 >> l);
      uint32_t *t = src; src = dst; dst = t;
    }
  }
}
}  // namespace

extern "C" int cae_tiles_pyramid_u8(const uint8_t *tiles, int n_tiles, int ps, int c, int levels,
                                    const int32_t *recs, int32_t *recs_dev, int gy, int gx,
                                    uint8_t *out, void *stream) {
  const char *fn = "cae_tiles_pyramid_u8";
  CAE_CHECK(n_tiles >= 0 && n_tiles <= 65535 && ps > 0 && c > 0 && gy > 0 && gx > 0, 2,
            "%s: bad argument", fn);
  CAE_CHECK(levels >= 1 && levels <= kPyrMaxLevels && ps % (1 << levels) == 0, 2,
            "%s: %d levels: K must be in [1, %d] with 2^K dividing the tile size %d", fn, levels,
            kPyrMaxLevels, ps);
  CAE_CHECK((int64_t)ps * ps * c <= INT32_MAX, 2, "%s: tile too large", fn);
  int ls = 0;                 // S = 2^ls: min(64, the largest power of two dividing ps)
  while (ls < 6 && ps % (2 << ls) == 0) ++ls;
  const int lq = levels > ls ? levels : ls;
  const int64_t S = 1 << ls, nsub = 1 << (lq - ls);
  const int64_t smem = ((S * S * c + 15) & ~15) +
                       4 * c * (S * S / 4 + S * S / 16 + nsub * nsub + nsub * nsub / 4);
  CAE_CHECK(smem <= kPyrSmem, 2, "%s: %d channels need %lld bytes of shared memory", fn, c,
            (long long)smem);
  if (n_tiles == 0) return 0;
  CAE_CHECK(tiles && recs && recs_dev && out, 2, "%s: null pointer", fn);
  CAE_CHECK((uintptr_t)recs_dev % 16 == 0, 2, "%s: recs_dev is not 16-byte aligned", fn);
  for (int t = 0; t < n_tiles; ++t) {
    const int32_t *p = recs + 4 * (size_t)t;
    CAE_CHECK(p[0] >= 0 && p[0] < gy && p[1] >= 0 && p[1] < gx, 2,
              "%s: record %d names chunk (%d, %d) of a %d x %d grid", fn, t, p[0], p[1], gy, gx);
    CAE_CHECK(p[2] > 0 && p[2] <= ps && p[3] > 0 && p[3] <= ps, 2,
              "%s: record %d: in-array extent %d x %d of a %d^2 tile", fn, t, p[2], p[3], ps);
    CAE_CHECK(p[0] >> 1 == recs[0] >> 1, 2,
              "%s: record %d (chunk row %d) and record 0 (chunk row %d) are in different level-1 "
              "chunk rows", fn, t, p[0], recs[0]);
  }
  PyrLevels lv = {};
  for (int l = 1; l < levels; ++l) lv.off[l + 1] = lv.off[l] + (gx + (1 << l) - 1) / (1 << l);
  cudaStream_t st = (cudaStream_t)stream;
  CAE_CUDA(cudaMemcpyAsync(recs_dev, recs, sizeof(int32_t) * 4 * (size_t)n_tiles,
                           cudaMemcpyHostToDevice, st));
  const dim3 grid((unsigned)((ps >> lq) * (ps >> lq)), (unsigned)n_tiles);
  const int4 *rd = reinterpret_cast<const int4 *>(recs_dev);
  if (((uintptr_t)tiles | (uintptr_t)(S * c)) % 16 == 0)
    tiles_pyramid_u8_kernel<16><<<grid, kPyrThreads, (size_t)smem, st>>>(tiles, ps, c, levels, ls,
                                                                         lq, rd, out, lv);
  else
    tiles_pyramid_u8_kernel<1><<<grid, kPyrThreads, (size_t)smem, st>>>(tiles, ps, c, levels, ls,
                                                                        lq, rd, out, lv);
  cae_count_launch();
  CAE_CUDA(cudaGetLastError());
  return 0;
}

// ---------------------------------------------------------------------------------------------
// Evaluation sums on the device (SURVEY.md 8f-4; src/test_cae.py:60-63 PSNR, :57-58 RMSE and the
// distortion term of src/models/criteria/_ratedist.py:57-63 in uint8 units): per image
//   sse[i] += sum (a - b)^2   over the `per_image` uint8 values of image i.
// HBM-bound: two 16-byte loads per thread per step, warp-shuffle + one atomic per block.
namespace {
__global__ void __launch_bounds__(256) sse_u8_kernel(const uint8_t *__restrict__ a,
                                                     const uint8_t *__restrict__ b,
                                                     size_t per_image, unsigned long long *sse) {
  const int img = blockIdx.y;
  const uint8_t *pa = a + (size_t)img * per_image, *pb = b + (size_t)img * per_image;
  unsigned long long acc = 0;
  const size_t n16 = ((reinterpret_cast<uintptr_t>(pa) | reinterpret_cast<uintptr_t>(pb)) & 15) ? 0 : per_image / 16;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += (size_t)gridDim.x * blockDim.x) {
    const uint4 va = __ldg(reinterpret_cast<const uint4 *>(pa) + i);
    const uint4 vb = __ldg(reinterpret_cast<const uint4 *>(pb) + i);
    const uint32_t wa[4] = {va.x, va.y, va.z, va.w}, wb[4] = {vb.x, vb.y, vb.z, vb.w};
    uint32_t s = 0;
#pragma unroll
    for (int w = 0; w < 4; ++w) {
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const int d = (int)((wa[w] >> (8 * k)) & 255u) - (int)((wb[w] >> (8 * k)) & 255u);
        s += (uint32_t)(d * d);
      }
    }
    acc += s;
  }
  for (size_t i = n16 * 16 + (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < per_image;
       i += (size_t)gridDim.x * blockDim.x) {
    const int d = (int)pa[i] - (int)pb[i];
    acc += (unsigned long long)(d * d);
  }
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  __shared__ unsigned long long part[8];
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned long long t = 0;
    for (int w = 0; w < 8; ++w) t += part[w];
    if (t) atomicAdd(sse + img, t);
  }
}
}  // namespace

extern "C" int cae_sse_u8(const uint8_t *a, const uint8_t *b, int n_images, int64_t per_image,
                          uint64_t *sse, void *stream) {
  CAE_CHECK(a && b && sse && n_images > 0 && per_image > 0, 2, "cae_sse_u8: bad argument");
  CAE_CHECK(n_images <= 65535, 2, "cae_sse_u8: more than 65535 images per call");
  int bx = (int)((per_image / 16 + 255) / 256);
  const int want = (4 * cae_sm_count() + n_images - 1) / n_images;   // ~4 blocks per SM in total
  if (bx > want) bx = want;
  if (bx < 1) bx = 1;
  sse_u8_kernel<<<dim3((unsigned)bx, (unsigned)n_images), 256, 0, (cudaStream_t)stream>>>(
      a, b, (size_t)per_image, reinterpret_cast<unsigned long long *>(sse));
  cae_count_launch();
  CAE_CUDA(cudaGetLastError());
  return 0;
}
