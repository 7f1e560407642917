// visible_cells / count_visible: per-environment line of sight over top-down maps from many viewpoints
// (include/dungeon_maps_b200.h: dm_line_of_sight_u8).  Target t = o + (dx, dz) is visible from origin o with radius r
// when dx^2 + dz^2 <= r^2, t is inside the map, no cell strictly between o and t on the integer line from o to t is
// blocking, and no diagonal step of that line passes between two blocking side cells (no corner leak).  The line is
// Bresenham with halves rounded away from the origin: with ax = |dx|, az = |dz|, m = max(ax, az) and ax >= az, cell i is
// (ox + sx * i, oz + sz * floor((2 * i * az + m) / (2 * m))), the axes swapped when az > ax.  Integer only: exact.
//
// One kernel on the caller's stream, no host sync.  One CTA per (environment, origin, band of window rows):
//   1. stage the blocking cells of the (2r+1)^2 window as a bit array in dynamic shared memory, only the rows between
//      the origin's row and the band (no line to a band target leaves them); map rows are read coalesced and packed
//      with ballots, cells outside the map are 0;
//   2. a warp takes 32 consecutive targets of a band row and walks each line with an incremental error term that
//      reproduces the floor formula's cells, reading only shared memory, and stops at the first blocker;
//   3. mask mode stores the 32 visibility bytes coalesced; count mode keeps the band's visibility words in shared
//      memory, then reads each target plane's band rows coalesced where a bit is set, sums with warp reductions and
//      adds one integer per (CTA, plane) into counts, zeroed on the stream first.  Integer adds: the counts do not
//      depend on their order.
#include "dm_common.cuh"

namespace dm {
namespace {

constexpr int kLosThreads = 256;
constexpr int kLosWarps = kLosThreads / 32;
constexpr int kMaxBandRows = 64;                          // bounds count mode's band words in shared memory
constexpr int kMaxRadius = 512;                           // (2r+1)^2 bits = 131 KB of shared memory at r = 512

struct LosArgs {
  const uint8_t* blocking;    // (b, H, W)
  const long long* origins;   // (b, n, 2) [x, z]
  const uint8_t* targets;     // (b, C, H, W) or nullptr
  uint8_t* visible;           // (b, n, 2r+1, 2r+1) or nullptr
  int32_t* counts;            // (b, C, n) or nullptr
  int b, H, W, n, C, r;
  int side, words;            // 2r+1, and 32-bit words per staged row
  int band_rows, bands;
  long long n_blocks;         // b * n * bands
};

__device__ __forceinline__ bool blocked(const uint32_t* s, int words, int x, int z) {
  return (s[z * words + (x >> 5)] >> (x & 31)) & 1u;
}

// Visibility of window cell (r + dx, r + dz) from the window centre (r, r) over the staged bits.
__device__ __forceinline__ bool line_clear(const uint32_t* s, int words, int r, int dx, int dz) {
  const int ax = abs(dx), az = abs(dz);
  const int sx = dx < 0 ? -1 : 1, sz = dz < 0 ? -1 : 1;
  const bool xmajor = ax >= az;
  const int m = xmajor ? ax : az, mn = xmajor ? az : ax;
  const int jx = xmajor ? sx : 0, jz = xmajor ? 0 : sz;   // the major step
  const int kx = xmajor ? 0 : sx, kz = xmajor ? sz : 0;   // the minor step
  // e = 2 * i * mn + m - 2 * m * q_i in [0, 2m), q_i the minor offset of cell i; q grows by 1 when e reaches 2m
  int e = m, x = r, z = r;
  for (int i = 1; i <= m; ++i) {
    e += 2 * mn;
    const bool diag = e >= 2 * m;
    e -= diag ? 2 * m : 0;
    const int nx = x + jx + (diag ? kx : 0), nz = z + jz + (diag ? kz : 0);
    if (diag && blocked(s, words, nx, z) && blocked(s, words, x, nz)) return false;
    if (i < m && blocked(s, words, nx, nz)) return false;
    x = nx;
    z = nz;
  }
  return true;
}

__global__ void __launch_bounds__(kLosThreads) line_of_sight_kernel(const LosArgs a) {
  extern __shared__ uint32_t smem[];
  __shared__ int warp_acc[kLosWarps];
  uint32_t* stage = smem;                                 // side x words
  uint32_t* band_bits = smem + a.side * a.words;          // band_rows x words (count mode)
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int r = a.r, side = a.side, words = a.words;
  const long long HW = (long long)a.H * a.W;
  for (long long bid = blockIdx.x; bid < a.n_blocks; bid += gridDim.x) {
    const int band = (int)(bid % a.bands);
    const long long ik = bid / a.bands;                   // environment * n + origin
    const long long env = ik / a.n;
    const long long ox = a.origins[2 * ik], oz = a.origins[2 * ik + 1];
    const bool inside = ox >= 0 && ox < a.W && oz >= 0 && oz < a.H;
    const int row0 = band * a.band_rows, row1 = min(row0 + a.band_rows, side);   // window rows [row0, row1)
    const int tasks = (row1 - row0) * words;
    if (!inside) {                                        // uniform in the CTA: sees nothing, counts stay 0
      if (a.visible)
        for (int t = warp; t < tasks; t += kLosWarps) {
          const int row = row0 + t / words, col = (t % words) * 32 + lane;
          if (col < side) a.visible[(ik * side + row) * side + col] = 0;
        }
      continue;
    }
    const uint8_t* blk = a.blocking + env * HW;
    const int s0 = min(row0, r), s1 = max(row1, r + 1);  // staged window rows [s0, s1)
    for (int t = warp; t < (s1 - s0) * words; t += kLosWarps) {
      const int row = s0 + t / words, col = (t % words) * 32 + lane;
      const long long mz = oz - r + row, mx = ox - r + col;
      const bool on = col < side && mz >= 0 && mz < a.H && mx >= 0 && mx < a.W && blk[mz * a.W + mx] != 0;
      const uint32_t bits = __ballot_sync(0xffffffffu, on);
      if (lane == 0) stage[row * words + (t % words)] = bits;
    }
    __syncthreads();
    for (int t = warp; t < tasks; t += kLosWarps) {
      const int row = row0 + t / words, col = (t % words) * 32 + lane;
      const int dx = col - r, dz = row - r;
      const long long tx = ox + dx, tz = oz + dz;
      const bool cand = col < side && dx * dx + dz * dz <= r * r && tx >= 0 && tx < a.W && tz >= 0 && tz < a.H;
      const bool vis = cand && line_clear(stage, words, r, dx, dz);
      if (a.visible) {
        if (col < side) a.visible[(ik * side + row) * side + col] = vis ? 1 : 0;
      } else {
        const uint32_t bits = __ballot_sync(0xffffffffu, vis);
        if (lane == 0) band_bits[t] = bits;
      }
    }
    if (a.counts) {
      __syncthreads();                                    // band_bits complete
      for (int c = 0; c < a.C; ++c) {
        const uint8_t* plane = a.targets + (env * a.C + c) * HW;
        int hits = 0;
        for (int t = warp; t < tasks; t += kLosWarps) {
          const uint32_t bits = band_bits[t];
          if (!bits) continue;                            // uniform in the warp
          const int row = row0 + t / words, col = (t % words) * 32 + lane;
          const long long tx = ox + col - r, tz = oz + row - r;   // inside the map wherever a bit is set
          hits += (bits >> lane & 1u) ? (int)(plane[tz * a.W + tx] != 0) : 0;
        }
        hits = __reduce_add_sync(0xffffffffu, hits);
        if (lane == 0) warp_acc[warp] = hits;
        __syncthreads();
        if (threadIdx.x == 0) {
          int sum = 0;
#pragma unroll
          for (int w = 0; w < kLosWarps; ++w) sum += warp_acc[w];
          if (sum) atomicAdd(a.counts + (env * a.C + c) * a.n + ik % a.n, sum);
        }
        __syncthreads();                                  // warp_acc is rewritten for the next plane
      }
    }
    __syncthreads();                                      // stage and band_bits are rewritten next
  }
}

}  // namespace
}  // namespace dm

using namespace dm;

extern "C" int dm_line_of_sight_u8(const uint8_t* blocking, int32_t b, int32_t H, int32_t W, const int64_t* origins,
                                   int32_t n, int32_t radius, uint8_t* visible, const uint8_t* targets, int32_t C,
                                   int32_t* counts, void* stream_) {
  DM_TRACE();
  if (!blocking || !origins) return DM_EINVAL;
  if (!visible == !counts) return DM_EINVAL;                        // exactly one output
  if (counts ? (!targets || C < 1) : (targets || C != 0)) return DM_EINVAL;
  if (b <= 0 || H <= 0 || W <= 0 || n <= 0 || radius < 0 || radius > kMaxRadius) return DM_EINVAL;
  if ((long long)b * n >= (1ll << 31) || (long long)H * W >= (1ll << 31) ||
      (long long)b * C * H * W >= (1ll << 31))
    return DM_EINVAL;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  LosArgs a;
  a.blocking = blocking;
  a.origins = reinterpret_cast<const long long*>(origins);
  a.targets = targets;
  a.visible = visible;
  a.counts = counts;
  a.b = b;
  a.H = H;
  a.W = W;
  a.n = n;
  a.C = C;
  a.r = radius;
  a.side = 2 * radius + 1;
  a.words = (a.side + 31) / 32;
  // enough bands that even a few origins fill every SM several times over; the result does not depend on the split
  const long long origins_total = (long long)b * n;
  const long long want = (8ll * sm_count() + origins_total - 1) / origins_total;
  const int bands = (int)min(max(want, 1ll), (long long)a.side);
  a.band_rows = min((a.side + bands - 1) / bands, kMaxBandRows);
  a.bands = (a.side + a.band_rows - 1) / a.band_rows;
  a.n_blocks = origins_total * a.bands;
  const size_t smem = (size_t)(a.side + (counts ? a.band_rows : 0)) * a.words * sizeof(uint32_t);
  if (smem > 48 * 1024)
    DM_CUDA_OK(cudaFuncSetAttribute(line_of_sight_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  if (counts) DM_CUDA_OK(cudaMemsetAsync(counts, 0, (size_t)b * C * n * sizeof(int32_t), stream));
  const long long cap = 1ll << 20;                                  // larger problems loop inside the kernel
  line_of_sight_kernel<<<(unsigned)min(a.n_blocks, cap), kLosThreads, smem, stream>>>(a);
  DM_LAUNCHED();
  return DM_OK;
}
