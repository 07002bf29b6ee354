// Host <-> device movement of whole batches of tiles for the tile loops, and the evaluation
// sums of a decoded batch.
//
// The reference rechunks the slide into patch_size^2 tiles with dask and hands them to the
// codec one at a time (src/compress.py:101-128); decompress.py:72-96 does the reverse.  Here a
// batch of tiles moves between the row-major H x W x c slide in (page-locked) host memory and a
// tile-major device buffer as strided DMA copies -- no host-side gather, no staging copy -- on
// the caller's stream, so uploads, kernels and downloads of neighbouring batches overlap.
#include "cae_common.cuh"

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
