// mrs_neighbors.cu -- neighbour lists of the COMM_RANGE graph (mrs_neighbors, include/mrs_b200.h): the graph of the
// dense A of MRS.calc_A (MRS.py:117-124) as per-agent lists of ascending neighbour indices, padded with -1, plus the
// true degree.  A graph learner reads 4 (M + 1) bytes per agent-step instead of 4 N (C4: 260 B instead of 16 KB).
//
// The hit test is the one of the dense kernels -- adjacency_pair() against Derived::s_max, every pair a hit when
// COMM_RANGE = +inf, never the diagonal -- so the lists are bit-exact with A (NaN positions, +-1 ulp around the
// range, R = 0 / inf).  Order comes from warp ballots and prefix popcounts, not atomics: every row is written in
// ascending j, and two calls write identical bytes.  Two shapes (DESIGN.md §4d):
//   N <= 32  neighbors_group_kernel: a group of G = pow2ceil(N) lanes per row, 32 / G rows per warp; lane l of a
//            group holds column l, so one segmented ballot answers the whole row.
//   N > 32   neighbors_warp_kernel: one warp per row, one ballot per 32-column tile; the columns' positions are
//            read straight from the state planes (L2-resident; the 8 rows of a CTA share them through L1).
#include "mrs_common.cuh"

namespace mrs {

namespace {

constexpr int kNbrBlock = 256;
constexpr int kNbrTiles = 4;          // column tiles whose positions are in flight at once (N > 32)

__device__ __forceinline__ bool nbr_hit(float xi, float yi, float zi, float xj, float yj, float zj, bool self, float s_max,
                                        int comm_inf) {
    return !self && (comm_inf || adjacency_pair(xi, yi, zi, xj, yj, zj, s_max) != 0.f);
}

// one row truncated: sticky status bit + stats counter, aggregated per warp (at most one atomic pair per warp)
__device__ __forceinline__ void nbr_overflow(bool over, unsigned* status, unsigned long long* stats) {
    const unsigned m = __ballot_sync(kFull32, over);
    if (m && (threadIdx.x & 31u) == 0u) {
        if (status) atomicOr(status, (unsigned)MRS_STATUS_NEIGHBOR_OVERFLOW);
        if (stats) atomicAdd(stats + MRS_STAT_NEIGHBOR_OVERFLOW, (unsigned long long)__popc(m));
    }
}

}  // namespace

// N <= 32.  Row r = e * N + i is group g of warp w (r = w * (32 / G) + g); lane l of the group loads the position of
// agent l of env e (the row's own position arrives by shuffle from lane i), so the whole row is one ballot.  The
// rows of a warp are contiguous in idx: its stores cover (32 / G) * M consecutive ints.
__global__ void __launch_bounds__(kNbrBlock)
neighbors_group_kernel(const float* __restrict__ state, unsigned S, int N, int G, int M, float s_max, int comm_inf,
                       int* __restrict__ idx, int* __restrict__ cnt, unsigned* status, unsigned long long* stats) {
    const unsigned t = blockIdx.x * kNbrBlock + threadIdx.x;
    const unsigned lane = threadIdx.x & 31u;
    const unsigned l = lane & (unsigned)(G - 1);
    const unsigned base = lane - l;                                   // first lane of the group
    const unsigned row = t / (unsigned)G;
    const bool row_ok = row < S;
    const unsigned i = row % (unsigned)N;
    const unsigned e0 = row - i;                                      // slot of agent 0 of the row's env
    const bool col_ok = row_ok && l < (unsigned)N;
    float xj = 0.f, yj = 0.f, zj = 0.f;
    if (col_ok) {
        xj = __ldg(state + e0 + l); yj = __ldg(state + S + e0 + l); zj = __ldg(state + 2 * (size_t)S + e0 + l);
    }
    const float xi = __shfl_sync(kFull32, xj, (int)(base + i));
    const float yi = __shfl_sync(kFull32, yj, (int)(base + i));
    const float zi = __shfl_sync(kFull32, zj, (int)(base + i));
    const bool hit = col_ok && nbr_hit(xi, yi, zi, xj, yj, zj, l == i, s_max, comm_inf);
    const unsigned gmask = (G == 32) ? kFull32 : ((1u << G) - 1u);
    const unsigned seg = (__ballot_sync(kFull32, hit) >> base) & gmask;
    const int deg = __popc(seg);
    if (row_ok && M > 0) {
        int* out = idx + (size_t)row * (unsigned)M;
        const int pos = __popc(seg & ((1u << l) - 1u));
        if (hit && pos < M) out[pos] = (int)l;
        for (int k = (deg < M ? deg : M) + (int)l; k < M; k += G) out[k] = -1;
    }
    if (row_ok && l == 0) cnt[row] = deg;
    nbr_overflow(row_ok && l == 0 && M > 0 && deg > M, status, stats);
}

// N > 32.  Warp w of the grid owns row r = w; lane l tests column 32 t + l of tile t.  kNbrTiles tiles of column
// positions are loaded before their ballots so that the loads of a warp overlap; hit lanes store their neighbour at
// (hits of the earlier tiles + prefix popcount), which is ascending j and one coalesced store per tile.
__global__ void __launch_bounds__(kNbrBlock)
neighbors_warp_kernel(const float* __restrict__ state, unsigned S, int N, int M, float s_max, int comm_inf,
                      int* __restrict__ idx, int* __restrict__ cnt, unsigned* status, unsigned long long* stats) {
    const unsigned row = (blockIdx.x * kNbrBlock + threadIdx.x) >> 5;
    const unsigned lane = threadIdx.x & 31u;
    if (row >= S) return;                                             // whole warps: S rows, 32 lanes each
    const unsigned i = row % (unsigned)N;
    const unsigned e0 = row - i;
    const float xi = __ldg(state + row), yi = __ldg(state + S + row), zi = __ldg(state + 2 * (size_t)S + row);
    int* out = idx + (size_t)row * (unsigned)M;
    const unsigned below = (1u << lane) - 1u;
    int deg = 0;
    for (int j0 = 0; j0 < N; j0 += 32 * kNbrTiles) {
        float xj[kNbrTiles], yj[kNbrTiles], zj[kNbrTiles];
#pragma unroll
        for (int u = 0; u < kNbrTiles; ++u) {
            const unsigned j = (unsigned)(j0 + 32 * u) + lane;
            xj[u] = yj[u] = zj[u] = 0.f;
            if (j < (unsigned)N) {
                xj[u] = __ldg(state + e0 + j); yj[u] = __ldg(state + S + e0 + j); zj[u] = __ldg(state + 2 * (size_t)S + e0 + j);
            }
        }
#pragma unroll
        for (int u = 0; u < kNbrTiles; ++u) {
            const unsigned j = (unsigned)(j0 + 32 * u) + lane;
            const bool hit = j < (unsigned)N && nbr_hit(xi, yi, zi, xj[u], yj[u], zj[u], j == i, s_max, comm_inf);
            const unsigned m = __ballot_sync(kFull32, hit);
            const int pos = deg + __popc(m & below);
            if (hit && pos < M) out[pos] = (int)j;
            deg += __popc(m);
        }
    }
    if (M > 0)
        for (int k = (deg < M ? deg : M) + (int)lane; k < M; k += 32) out[k] = -1;
    if (lane == 0) cnt[row] = deg;
    nbr_overflow(lane == 0 && M > 0 && deg > M, status, stats);
}

}  // namespace mrs

using namespace mrs;

extern "C" int mrs_neighbors(const MrsConfig* cfg, const MrsBuffers* bufs, int max_nbr, int* idx, int* cnt, void* stream) {
    int rc = check_cfg(cfg);
    if (rc) return rc;
    if (!bufs || !bufs->state || !cnt || max_nbr < 0 || (max_nbr > 0 && !idx)) return MRS_ERR_ARG;
    const unsigned long long S = (unsigned long long)cfg->E * (unsigned long long)cfg->N;
    // thread index (32 lanes per row at most) and state offsets run in 32 bits; idx offsets (< 2^27 rows x max_nbr
    // < 2^31) in size_t
    if (S * 32ull > 0xffffffffull) return MRS_ERR_UNSUPPORTED;
    const Derived d = make_derived(*cfg);         // s_max / comm_inf exactly as the step kernels derive them
    cudaStream_t st = (cudaStream_t)stream;
    const int N = cfg->N;
    if (N <= 32) {
        int G = 1;
        while (G < N) G <<= 1;
        const unsigned long long threads = S * (unsigned long long)G;
        neighbors_group_kernel<<<(unsigned)((threads + kNbrBlock - 1) / kNbrBlock), kNbrBlock, 0, st>>>(
            bufs->state, (unsigned)S, N, G, max_nbr, d.s_max, d.comm_inf, idx, cnt, bufs->status, bufs->stats);
    } else {
        const unsigned long long threads = S * 32ull;
        neighbors_warp_kernel<<<(unsigned)((threads + kNbrBlock - 1) / kNbrBlock), kNbrBlock, 0, st>>>(
            bufs->state, (unsigned)S, N, max_nbr, d.s_max, d.comm_inf, idx, cnt, bufs->status, bufs->stats);
    }
    return last_error();
}
