// Nearest-neighbour search over a device-resident fp32 matrix -- the target / token / path table or a caller's code
// vectors: gensim's KeyedVectors.most_similar (what the reference README's `--save_t2v` / `--save_w2v` workflow runs
// on the exported text files, README.md:236-251) without leaving the GPU.
//
//   compose_kernel : the query vector of a word query, unitvec(mean_t(w_t . B_t / |B_t|)), as gensim forms it.
//   nearest_kernel : cosine top-k of a chunk of queries against a contiguous row range of the bank (one CTA per
//                    (query chunk, row slice)).  Row tiles stream into shared memory with 1-D bulk copies
//                    (cp.async.bulk, completion on an mbarrier per stage), STAGES deep.  TPR threads share a row, each
//                    a strided quarter of its float4s, and keep a register block of 2 rows x QB queries plus the row's
//                    sum of squares: the norm comes from the same pass as the dots, so nothing cached can go stale
//                    after a train step, a load or a lazy-Adam replay.  fp32 FFMA throughout.  A score is tested
//                    against the running k-th best of its (CTA, query) before it is queued, so once the list has
//                    filled most rows cost one comparison; queued candidates are merged into the sorted list by rank
//                    (one warp per query) after each tile.
//   merge_kernel   : k-way merge of the per-slice lists into the final k.
// Order: score descending, ties to the lower row (better(), kernels.cuh) at every level, and the per-slice lists are
// exact, so the result depends neither on the number of slices nor on how the queries are chunked.
#pragma once
#include "ctx_fused.cuh"
#include "kernels.cuh"

namespace c2v {
namespace sim {

constexpr int kThreads = 256;
constexpr int kRowsPerThread = 2;       // rows in a thread's register block
constexpr int kMaxK = 64;               // the same cap as c2v_dims.top_k
constexpr int kMaxExclude = 16;
constexpr int kMaxTerms = 16;
constexpr int kSlices = 148;            // CTAs along the rows of the bank: one per B200 SM
constexpr int kMaxStages = 4;
constexpr int kQueryBytes = 32768;      // shared memory for one chunk's query vectors
constexpr int kSmemBudget = 227 * 1024 - 256;

// threads per row: each thread then owns >= 4 float4s of a row at the java14m widths (128, 384), and a quarter warp
// always reads 128 contiguous bytes of one row (conflict-free LDS.128 without padding)
__host__ __device__ inline int tpr_for(int dim) { return dim <= 256 ? 8 : (dim <= 512 ? 16 : 32); }
__host__ __device__ inline int tile_rows(int dim) { return kThreads / tpr_for(dim) * kRowsPerThread; }   // 64, 32, 16
inline int query_capacity(int dim) {                     // queries per chunk: a multiple of 8, 8 .. 64
  const int q = (kQueryBytes / (dim * 4)) / 8 * 8;
  return q < 8 ? 8 : (q > 64 ? 64 : q);
}
inline int slices_for(int64_t rows) { return rows < kSlices ? (int)rows : kSlices; }

// shared-memory carve-up of nearest_kernel (byte offsets), computed on the host
struct Layout {
  int tr, qc, stages;
  int off_q, off_qn, off_ex, off_list, off_cand, off_thr, off_cnt, off_len, off_bar, total;
};

inline Layout make_layout(int dim, int k) {
  Layout L{};
  L.tr = tile_rows(dim);
  L.qc = query_capacity(dim);
  const int stage = L.tr * dim * 4;
  int off = 0;
  auto take = [&](int bytes, int align) { off = (off + align - 1) / align * align; const int o = off; off += bytes; return o; };
  L.off_q = take(L.qc * dim * 4, 16);
  L.off_qn = take(L.qc * 4, 16);
  L.off_ex = take(L.qc * kMaxExclude * 4, 16);
  L.off_list = take(L.qc * k * 8, 16);
  L.off_cand = take(L.qc * L.tr * 8, 16);
  L.off_thr = take(L.qc * 8, 16);
  L.off_cnt = take(L.qc * 4, 16);
  L.off_len = take(L.qc * 4, 16);
  L.off_bar = take(kMaxStages * 8, 16);
  const int fixed = (off + 127) / 128 * 128;
  int stages = (kSmemBudget - fixed) / stage;
  L.stages = stages > kMaxStages ? kMaxStages : stages;      // >= 2 at every dim <= 1024, k <= 64
  // stages first (bulk-copy destinations, 128-byte aligned), then the fixed part
  const int shift = L.stages * stage;
  L.off_q += shift; L.off_qn += shift; L.off_ex += shift; L.off_list += shift; L.off_cand += shift;
  L.off_thr += shift; L.off_cnt += shift; L.off_len += shift; L.off_bar += shift;
  L.total = shift + fixed;
  return L;
}

__device__ __forceinline__ float block_sum256(float v, float* red) {      // fixed order: lanes, then warps 0..7
  v = warp_sum(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  float s = 0.f;
#pragma unroll
  for (int w = 0; w < kThreads / 32; ++w) s += red[w];
  return s;
}

// One block per query.  term_rows[q, t]: bank row (unit-normalised, then weighted), -2: the caller's vector
// term_vecs[q, t, :] weighted as given (gensim uses array terms unnormalised), -1 or a row outside the bank: no term.
__global__ void __launch_bounds__(kThreads)
compose_kernel(const float* __restrict__ bank, int64_t rows, int dim, const int32_t* __restrict__ term_rows,
               const float* __restrict__ term_w, const float* __restrict__ term_vecs, int max_terms, float* __restrict__ out) {
  __shared__ float red[kThreads / 32];
  const int q = blockIdx.x, i = threadIdx.x, D4 = dim >> 2;
  const bool active = i < D4;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  int cnt = 0;
  for (int t = 0; t < max_terms; ++t) {
    const int r = term_rows[(size_t)q * max_terms + t];
    const float w = term_w[(size_t)q * max_terms + t];
    const float* src;
    if (r >= 0 && r < rows) src = bank + (size_t)r * dim;
    else if (r == -2) src = term_vecs + ((size_t)q * max_terms + t) * dim;
    else continue;
    const float4 x = active ? reinterpret_cast<const float4*>(src)[i] : make_float4(0.f, 0.f, 0.f, 0.f);
    ++cnt;
    if (r >= 0) {
      const float nrm = sqrtf(block_sum256(x.x * x.x + x.y * x.y + x.z * x.z + x.w * x.w, red));
      if (!(nrm > 0.f)) continue;                       // a zero row adds nothing (and still counts towards the mean)
      acc.x += w * (x.x / nrm); acc.y += w * (x.y / nrm); acc.z += w * (x.z / nrm); acc.w += w * (x.w / nrm);
    } else {
      acc.x += w * x.x; acc.y += w * x.y; acc.z += w * x.z; acc.w += w * x.w;
    }
  }
  if (cnt) {
    const float c = (float)cnt;
    acc.x /= c; acc.y /= c; acc.z /= c; acc.w /= c;
  }
  const float nrm = sqrtf(block_sum256(acc.x * acc.x + acc.y * acc.y + acc.z * acc.z + acc.w * acc.w, red));
  if (nrm > 0.f) { acc.x /= nrm; acc.y /= nrm; acc.z /= nrm; acc.w /= nrm; }
  if (active) reinterpret_cast<float4*>(out + (size_t)q * dim)[i] = acc;
}

// grid (query chunks, row slices).  cand_out[(query * slices + slice) * k + p]: the slice's exact top k, sorted,
// padded with (-inf, -1).
template <int QB>
__global__ void __launch_bounds__(kThreads, 1)
nearest_kernel(const float* __restrict__ bank, int rows, int dim, const float* __restrict__ queries, int n, int k,
               const int32_t* __restrict__ exclude, int n_exclude, const Layout L, ValIdx* __restrict__ cand_out) {
  extern __shared__ __align__(128) uint8_t smem[];
  float* sq = reinterpret_cast<float*>(smem + L.off_q);
  float* sqn = reinterpret_cast<float*>(smem + L.off_qn);
  int* sex = reinterpret_cast<int*>(smem + L.off_ex);
  ValIdx* slist = reinterpret_cast<ValIdx*>(smem + L.off_list);
  ValIdx* scand = reinterpret_cast<ValIdx*>(smem + L.off_cand);
  ValIdx* sthr = reinterpret_cast<ValIdx*>(smem + L.off_thr);
  int* scnt = reinterpret_cast<int*>(smem + L.off_cnt);
  int* slen = reinterpret_cast<int*>(smem + L.off_len);
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + L.off_bar);

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int tr = L.tr, qc = L.qc, stages = L.stages, D4 = dim >> 2;
  const int q0 = blockIdx.x * qc, nq = min(qc, n - q0);
  const int slice = blockIdx.y, nslices = gridDim.y;
  const int r_begin = (int)((int64_t)rows * slice / nslices), r_end = (int)((int64_t)rows * (slice + 1) / nslices);
  const int ntiles = (r_end - r_begin + tr - 1) / tr;

  if (tid == 0) {
    for (int s = 0; s < stages; ++s) umma::mbar_init(&full[s], 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  for (int e = tid; e < qc * D4; e += kThreads) {       // this chunk's queries, zero-padded to qc
    const int q = e / D4, j = e - q * D4;
    reinterpret_cast<float4*>(sq)[e] = (q < nq) ? reinterpret_cast<const float4*>(queries + (size_t)(q0 + q) * dim)[j]
                                                : make_float4(0.f, 0.f, 0.f, 0.f);
  }
  for (int e = tid; e < qc * kMaxExclude; e += kThreads) {
    const int q = e / kMaxExclude, j = e - q * kMaxExclude;
    sex[e] = (q < nq && j < n_exclude) ? exclude[(size_t)(q0 + q) * n_exclude + j] : -1;
  }
  for (int q = tid; q < qc; q += kThreads) {
    scnt[q] = 0; slen[q] = 0;
    sthr[q].v = -INFINITY; sthr[q].i = INT_MAX;
  }
  __syncthreads();
  for (int q = warp; q < qc; q += kThreads / 32) {     // query norms, one fixed order per dim
    float s = 0.f;
    for (int j = lane; j < dim; j += 32) s = fmaf(sq[q * dim + j], sq[q * dim + j], s);
    s = warp_sum(s);
    if (lane == 0) sqn[q] = sqrtf(s);
  }

  auto issue = [&](int t) {                               // thread 0: bulk copy of row tile t into its stage
    const int r0 = r_begin + t * tr;
    const int nr = min(tr, r_end - r0);
    const uint32_t bytes = (uint32_t)nr * (uint32_t)dim * 4u;
    const int s = t % stages;
    umma::mbar_expect_tx(&full[s], bytes);
    umma::bulk_copy_g2s(smem + (size_t)s * tr * dim * 4, bank + (size_t)r0 * dim, bytes, &full[s]);
  };
  if (tid == 0)
    for (int t = 0; t < stages && t < ntiles; ++t) issue(t);
  __syncthreads();

  const int TPR = tpr_for(dim), G = kThreads / TPR;
  const int g = tid / TPR, sl = tid - g * TPR;
  for (int t = 0; t < ntiles; ++t) {
    const int s = t % stages;
    umma::mbar_wait(&full[s], (uint32_t)((t / stages) & 1));
    const float* tile = reinterpret_cast<const float*>(smem + (size_t)s * tr * dim * 4);
    const int r0 = r_begin + t * tr, nr = min(tr, r_end - r0);
    const float4* rowp[kRowsPerThread];
#pragma unroll
    for (int b = 0; b < kRowsPerThread; ++b) rowp[b] = reinterpret_cast<const float4*>(tile + (size_t)(g + b * G) * dim);
    float ss[kRowsPerThread];
#pragma unroll
    for (int b = 0; b < kRowsPerThread; ++b) ss[b] = 0.f;
    for (int qb = 0; qb < nq; qb += QB) {
      float acc[kRowsPerThread][QB];
#pragma unroll
      for (int b = 0; b < kRowsPerThread; ++b)
#pragma unroll
        for (int c = 0; c < QB; ++c) acc[b][c] = 0.f;
      const float4* qp = reinterpret_cast<const float4*>(sq + (size_t)qb * dim);
      for (int i = sl; i < D4; i += TPR) {
        float4 x[kRowsPerThread];
#pragma unroll
        for (int b = 0; b < kRowsPerThread; ++b) x[b] = rowp[b][i];
        if (qb == 0) {
#pragma unroll
          for (int b = 0; b < kRowsPerThread; ++b) {
            ss[b] = fmaf(x[b].x, x[b].x, ss[b]); ss[b] = fmaf(x[b].y, x[b].y, ss[b]);
            ss[b] = fmaf(x[b].z, x[b].z, ss[b]); ss[b] = fmaf(x[b].w, x[b].w, ss[b]);
          }
        }
#pragma unroll
        for (int c = 0; c < QB; ++c) {
          const float4 y = qp[(size_t)c * D4 + i];
#pragma unroll
          for (int b = 0; b < kRowsPerThread; ++b) {
            acc[b][c] = fmaf(x[b].x, y.x, acc[b][c]); acc[b][c] = fmaf(x[b].y, y.y, acc[b][c]);
            acc[b][c] = fmaf(x[b].z, y.z, acc[b][c]); acc[b][c] = fmaf(x[b].w, y.w, acc[b][c]);
          }
        }
      }
      // the TPR partial sums of a row: butterfly over the row's lanes (TPR divides 32, groups are lane-aligned)
      for (int o = TPR >> 1; o > 0; o >>= 1) {
#pragma unroll
        for (int b = 0; b < kRowsPerThread; ++b) {
          if (qb == 0) ss[b] += __shfl_xor_sync(0xffffffffu, ss[b], o);
#pragma unroll
          for (int c = 0; c < QB; ++c) acc[b][c] += __shfl_xor_sync(0xffffffffu, acc[b][c], o);
        }
      }
      if (sl == 0) {
#pragma unroll
        for (int b = 0; b < kRowsPerThread; ++b) {
          const int rr = g + b * G;
          const float nb = sqrtf(ss[b]);
          if (rr >= nr || !(nb > 0.f)) continue;         // rows past the tile, zero (or NaN) rows: never returned
          const int row = r0 + rr;
#pragma unroll
          for (int c = 0; c < QB; ++c) {
            const int q = qb + c;
            const float qn = sqn[q];
            if (q >= nq || !(qn > 0.f)) continue;        // padding queries, zero queries: no results
            const float sc = acc[b][c] / (nb * qn);
            if (sc != sc) continue;                      // NaN score
            const ValIdx th = sthr[q];
            if (!better(sc, row, th.v, th.i)) continue;
            bool skip = false;
#pragma unroll
            for (int j = 0; j < kMaxExclude; ++j) skip |= (sex[q * kMaxExclude + j] == row);
            if (skip) continue;
            const int pos = atomicAdd(&scnt[q], 1);
            scand[q * tr + pos].v = sc;
            scand[q * tr + pos].i = row;
          }
        }
      }
    }
    __syncthreads();                                     // every thread is done with stage s and has queued its candidates
    if (tid == 0 && t + stages < ntiles) issue(t + stages);
    for (int q = warp; q < nq; q += kThreads / 32) {     // merge the queued candidates into the sorted list by rank
      const int m = scnt[q];
      if (m == 0) continue;
      const int cur = slen[q], tot = cur + m;            // <= k + tr <= 128
      ValIdx* Lq = slist + q * k;
      const ValIdx* Cq = scand + q * tr;
      ValIdx ev[4];
      int rk[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int e = lane + 32 * u;
        rk[u] = INT_MAX;
        if (e >= tot) continue;
        ev[u] = e < cur ? Lq[e] : Cq[e - cur];
        int r = 0;
        if (e < cur) r = e;                              // the list is sorted: e list entries come before it
        else for (int j = 0; j < cur; ++j) r += better(Lq[j].v, Lq[j].i, ev[u].v, ev[u].i) ? 1 : 0;
        for (int j = 0; j < m; ++j) r += better(Cq[j].v, Cq[j].i, ev[u].v, ev[u].i) ? 1 : 0;
        rk[u] = r;
      }
      __syncwarp();
#pragma unroll
      for (int u = 0; u < 4; ++u)
        if (rk[u] < k) Lq[rk[u]] = ev[u];
      __syncwarp();
      if (lane == 0) {
        const int nl = min(k, tot);
        slen[q] = nl;
        if (nl == k) sthr[q] = Lq[k - 1];
        scnt[q] = 0;
      }
    }
    __syncthreads();
  }
  for (int e = tid; e < nq * k; e += kThreads) {
    const int q = e / k, p = e - q * k;
    ValIdx o;
    if (p < slen[q]) o = slist[q * k + p];
    else { o.v = -INFINITY; o.i = -1; }
    cand_out[((size_t)(q0 + q) * nslices + slice) * k + p] = o;
  }
}

// One block per query: k rounds of block arg-best over the heads of the per-slice sorted lists (nslices <= 256).
__global__ void __launch_bounds__(kTopkThreads)
merge_kernel(const ValIdx* __restrict__ cand, int nslices, int k, int32_t* __restrict__ idx_out, float* __restrict__ val_out) {
  __shared__ ValIdx red[32];
  const int q = blockIdx.x, tid = threadIdx.x;
  const ValIdx* mine = cand + ((size_t)q * nslices + tid) * k;
  int head = 0;
  for (int r = 0; r < k; ++r) {
    float hv = -INFINITY;
    int hi = INT_MAX;
    if (tid < nslices && head < k) {
      const ValIdx c = mine[head];
      if (c.i >= 0) { hv = c.v; hi = c.i; }
    }
    const ValIdx w = block_argbest(hv, hi, red);
    if (hi != INT_MAX && w.i == hi) ++head;
    if (tid == 0) {
      const bool none = (w.i == INT_MAX);
      idx_out[(size_t)q * k + r] = none ? -1 : w.i;
      val_out[(size_t)q * k + r] = none ? -INFINITY : w.v;
    }
  }
}

}  // namespace sim
}  // namespace c2v
