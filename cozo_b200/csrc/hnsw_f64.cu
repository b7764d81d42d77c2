// hnsw_f64.cu — batched k-NN search on an F64 vector index (manifest.dtype == VecElementType::F64).
//
// The reference computes distances of F64 vectors in f64 throughout (runtime/hnsw.rs:73-76, 86-93, 102-107) and
// casts the query to the index dtype first (hnsw.rs:879-884).  This is a second, self-contained instantiation of
// hnsw_search_level / hnsw_knn (hnsw.rs:539-587, 869-1012) on `double`: one warp per query, the query and the
// sorted found/candidate array (f64 keys) in shared memory, rows read with coalesced 8-byte loads.  It shares the
// graph layout, the visited bitmaps and the workspace pool with the f32 path and leaves that path's register and
// shared-memory budget untouched.  F64 indexes are search-only on the device (maintenance re-stages).
#include <algorithm>
#include <cstring>
#include <vector>

#include "hnsw_host.hpp"

namespace cozo {

struct Search64Params {
  const double* queries;
  const double* vec64;  // [n x ld64]
  uint32_t ld64;
  uint32_t B, k, ef;
  int has_radius;
  double radius;
  uint32_t* out_ids;
  double* out_dist;
  uint32_t* out_count;
  uint32_t* qstats;
  uint32_t* counter;
  uint32_t* vis;
  uint32_t nwords;
  uint32_t* vlog;
  uint32_t logcap;
  uint32_t warp_smem, off_fi, off_pend, off_q;
  const uint32_t* filter_mask;
};

__device__ __forceinline__ double warp_sum_f64(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// VectorCache::dist for (F64, F64) operands
template <int METRIC>
__device__ __forceinline__ double dist64(const double* q, const double* __restrict__ row, uint32_t dim, int lane,
                                         double qnorm) {
  double a = 0.0, b = 0.0;
#pragma unroll 4
  for (uint32_t i = lane; i < dim; i += 32) {
    const double x = q[i], y = __ldg(row + i);
    if (METRIC == COZO_GPU_L2) {
      const double d = x - y;
      a = fma(d, d, a);
    } else {
      a = fma(x, y, a);
      if (METRIC == COZO_GPU_COSINE) b = fma(y, y, b);
    }
  }
  a = warp_sum_f64(a);
  if (METRIC == COZO_GPU_L2) return a;
  if (METRIC == COZO_GPU_IP) return 1.0 - a;
  b = warp_sum_f64(b);
  return 1.0 - a / sqrt(qnorm * b);
}

// found_nn.push + pop-if-over-ef (hnsw.rs:577-580) on the sorted array; equal keys keep arrival order, NaN sorts last
__device__ __forceinline__ void sorted_insert64(WarpCtx& w, double* fd, uint32_t ef, double d, uint32_t id, int lane) {
  uint32_t pos = 0;
  for (uint32_t base = 0; base < w.len; base += 32) {
    uint32_t i = base + lane;
    bool le = (i < w.len) && !precedes(d, fd[i]);
    uint32_t bal = __ballot_sync(0xffffffffu, le);
    pos += __popc(bal);
    if (bal != 0xffffffffu) break;
  }
  uint32_t newlen = w.len < ef ? w.len + 1 : ef;
  for (int top = (int)newlen - 1; top > (int)pos; top -= 32) {
    int i = top - 1 - lane;
    bool act = i >= (int)pos;
    double td = 0.0;
    uint32_t ti = 0;
    if (act) {
      td = fd[i];
      ti = w.fi[i];
    }
    __syncwarp();
    if (act) {
      fd[i + 1] = td;
      w.fi[i + 1] = ti;
    }
    __syncwarp();
  }
  __syncwarp();
  if (lane == 0) {
    fd[pos] = d;
    w.fi[pos] = id;
  }
  __syncwarp();
  w.len = newlen;
  if (pos < w.cursor) w.cursor = pos;
}

template <int METRIC>
__device__ __forceinline__ void search_level64(const HnswDev& g, const Search64Params& p, WarpCtx& w, double* fd,
                                               const double* q, double qnorm, uint32_t ef, uint32_t level, int lane) {
  for (uint32_t base = 0; base < w.len; base += 32) {  // visited <- keys(found) (hnsw.rs:554-557)
    uint32_t i = base + lane;
    uint32_t id = NONE;
    if (i < w.len) {
      id = w.fi[i] & IDMASK;
      w.fi[i] = id;
    }
    uint32_t nm;
    visit_mark(w, id, lane, nm);
  }
  __syncwarp();
  w.cursor = 0;
  const uint32_t stride = level == 0 ? g.s0 : g.su;
  for (;;) {
    uint32_t ci = NONE;  // candidates.pop(): nearest not-yet-expanded entry (hnsw.rs:559)
    for (uint32_t base = w.cursor & ~31u; base < w.len; base += 32) {
      uint32_t i = base + lane;
      bool un = (i < w.len) && (i >= w.cursor) && !(w.fi[i] & EXPANDED);
      uint32_t bal = __ballot_sync(0xffffffffu, un);
      if (bal) {
        ci = base + __ffs(bal) - 1;
        break;
      }
    }
    if (ci == NONE) break;  // == `candidate_dist > furthest_dist` (hnsw.rs:562)
    uint32_t cand = w.fi[ci];
    __syncwarp();
    if (lane == 0) w.fi[ci] = cand | EXPANDED;
    w.cursor = ci + 1;
    w.nodes_expanded++;
    const uint32_t* row = level == 0 ? g.adj0 + (size_t)cand * g.s0
                                     : g.adj_up + (size_t)(g.upper_off[cand] + level - 1) * g.su;
    for (uint32_t nb = 0; nb < stride; nb += 32) {  // hnsw_get_neighbours: one padded row
      uint32_t id = __ldg(row + nb + lane);
      uint32_t validmask = __ballot_sync(0xffffffffu, id != NONE);
      if (!validmask) break;
      w.nbr_reads += __popc(validmask);
      uint32_t newmask;
      bool isnew = visit_mark(w, id, lane, newmask);  // hnsw.rs:569-571,582
      uint32_t cnt = __popc(newmask);
      if (isnew) w.pend[__popc(newmask & ((1u << lane) - 1))] = id;
      __syncwarp();
      w.dist_evals += cnt;
      for (uint32_t c = 0; c < cnt; ++c) {
        const uint32_t nid = w.pend[c];
        const double d = dist64<METRIC>(q, p.vec64 + (size_t)nid * p.ld64, g.dim, lane, qnorm);
        __syncwarp();
        if (w.len < ef || d < fd[w.len - 1]) sorted_insert64(w, fd, ef, d, nid, lane);  // hnsw.rs:575-581
      }
      __syncwarp();
    }
  }
  visit_clear(w, lane);
}

template <int METRIC>
__global__ void __launch_bounds__(128) hnsw_search_f64_kernel(HnswDev g, Search64Params p) {
  extern __shared__ __align__(16) uint8_t smem64[];
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int wpc = blockDim.x >> 5;
  uint8_t* base = smem64 + (size_t)warp * p.warp_smem;
  double* fd = reinterpret_cast<double*>(base);
  double* q = reinterpret_cast<double*>(base + p.off_q);
  WarpCtx w;
  w.fd = nullptr;
  w.fi = reinterpret_cast<uint32_t*>(base + p.off_fi);
  w.pend = reinterpret_cast<uint32_t*>(base + p.off_pend);
  w.bars = nullptr;
  w.ring = nullptr;
  const size_t slot = (size_t)blockIdx.x * wpc + warp;
  w.vis = p.vis + slot * p.nwords;
  w.nwords = p.nwords;
  w.vlog = p.vlog + slot * p.logcap;
  w.logcap = p.logcap;
  w.ns = 0;
  w.nlog = 0;
  w.head = 0;
  w.phase = 0;
  for (;;) {
    uint32_t qi = 0;
    if (lane == 0) qi = atomicAdd(p.counter, 1u);
    qi = __shfl_sync(0xffffffffu, qi, 0);
    if (qi >= p.B) break;
    double qn = 0.0;
    for (uint32_t i = lane; i < g.dim; i += 32) {
      const double x = p.queries[(size_t)qi * g.dim + i];
      q[i] = x;
      qn = fma(x, x, qn);
    }
    qn = warp_sum_f64(qn);
    __syncwarp();
    w.len = 0;
    w.cursor = 0;
    w.dist_evals = w.nodes_expanded = w.nbr_reads = 0;
    uint32_t found = 0;
    if (g.entry != NONE) {  // empty index => no rows (hnsw.rs:903-909)
      const double d = dist64<METRIC>(q, p.vec64 + (size_t)g.entry * p.ld64, g.dim, lane, qn);
      w.dist_evals = 1;
      if (lane == 0) {
        fd[0] = d;
        w.fi[0] = g.entry;
      }
      w.len = 1;
      __syncwarp();
      for (uint32_t lvl = g.top_level; lvl >= 1; --lvl) search_level64<METRIC>(g, p, w, fd, q, qn, 1, lvl, lane);
      search_level64<METRIC>(g, p, w, fd, q, qn, p.ef, 0, lane);
      // hnsw.rs:943-956, 997-1006: radius, filter verdicts, then the first k
      for (uint32_t base_i = 0; base_i < w.len && found < p.k; base_i += 32) {
        const uint32_t i = base_i + lane;
        bool ok = i < w.len;
        uint32_t id = 0;
        double d2 = 0.0;
        if (ok) {
          id = w.fi[i] & IDMASK;
          d2 = fd[i];
          ok = !(p.has_radius && d2 > p.radius) && (!p.filter_mask || ((p.filter_mask[id >> 5] >> (id & 31)) & 1u));
        }
        const uint32_t bal = __ballot_sync(0xffffffffu, ok);
        const uint32_t pos = found + __popc(bal & ((1u << lane) - 1));
        if (ok && pos < p.k) {
          p.out_ids[(size_t)qi * p.k + pos] = id;
          p.out_dist[(size_t)qi * p.k + pos] = d2;
        }
        found += __popc(bal);
      }
      if (found > p.k) found = p.k;
    }
    for (uint32_t i = found + lane; i < p.k; i += 32) {
      p.out_ids[(size_t)qi * p.k + i] = NONE;
      p.out_dist[(size_t)qi * p.k + i] = INFINITY;
    }
    if (lane == 0) {
      if (p.out_count) p.out_count[qi] = found;
      if (p.qstats) reinterpret_cast<uint4*>(p.qstats)[qi] = make_uint4(w.dist_evals, w.nodes_expanded, w.nbr_reads, 0);
    }
    __syncwarp();
  }
}

}  // namespace cozo

using namespace cozo;

extern "C" int cozo_gpu_hnsw_search_f64(cozo_gpu_hnsw_t* h, const double* queries, uint32_t B, uint32_t k, uint32_t ef,
                                        double radius, const uint32_t* row_mask, uint32_t* out_ids, double* out_dist,
                                        uint32_t* out_count, CozoGpuSearchStats* stats) {
  if (!h) return set_error(COZO_GPU_EINVAL, "null index handle");
  if (!h->f64) return set_error(COZO_GPU_EINVAL, "not an F64 index: use cozo_gpu_hnsw_search");
  if (k == 0) return set_error(COZO_GPU_EINVAL, "k must be positive");
  if (ef == 0) return set_error(COZO_GPU_EINVAL, "ef must be positive");
  if (B && (!queries || !out_ids || !out_dist)) return set_error(COZO_GPU_EINVAL, "null buffer");
  int rc = ensure_init();
  if (rc) return rc;
  if (stats) memset(stats, 0, sizeof(*stats));
  if (B == 0) return 0;
  const DeviceInfo& di = device_info();
  const HnswDev& g = h->dev;
  HnswWorkspace* ws = hnsw_acquire_ws(h);
  if (!ws) return COZO_GPU_ECUDA;
  struct Bufs {
    cozo_gpu_hnsw* h;
    HnswWorkspace* ws;
    void* p[6] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    ~Bufs() {
      for (void* q : p)
        if (q) cudaFree(q);
      hnsw_release_ws(h, ws);
    }
  } bf{h, ws};
  cudaStream_t st = ws->stream;
  Search64Params p{};
  const uint32_t efcap = round_up(ef, 32);
  p.off_fi = efcap * 8;
  p.off_pend = p.off_fi + efcap * 4;
  p.off_q = round_up(p.off_pend + 128, 16);
  p.warp_smem = round_up(p.off_q + g.dim * 8, 16);
  uint32_t wpc = 4;
  size_t smem = (size_t)p.warp_smem * wpc;
  while (smem > di.smem_optin && wpc > 1) {
    wpc >>= 1;
    smem = (size_t)p.warp_smem * wpc;
  }
  if (smem > di.smem_optin)
    return set_error(COZO_GPU_EUNSUP, "ef=%u / dim=%u need %zu B of shared memory per warp (limit %zu)", ef, g.dim, smem,
                     di.smem_optin);
  using K64 = void (*)(HnswDev, Search64Params);
  K64 fn = g.metric == COZO_GPU_L2       ? (K64)hnsw_search_f64_kernel<COZO_GPU_L2>
           : g.metric == COZO_GPU_COSINE ? (K64)hnsw_search_f64_kernel<COZO_GPU_COSINE>
                                         : (K64)hnsw_search_f64_kernel<COZO_GPU_IP>;
  COZO_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)di.smem_optin));
  int cps = 0;
  COZO_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&cps, fn, wpc * 32, smem));
  if (cps < 1) return set_error(COZO_GPU_ECUDA, "F64 search kernel does not fit on an SM");
  uint32_t grid = std::min<uint32_t>((uint32_t)di.sm_count * (uint32_t)cps, (B + wpc - 1) / wpc);
  const uint32_t nwords = round_up((g.n + 31) / 32, 4);
  const uint32_t logcap = std::min<uint32_t>(65536u, std::max<uint32_t>(4096u, 64u * ef));
  const size_t slots = (size_t)grid * wpc;
  rc = hnsw_ws_reserve(ws, slots * nwords, slots * logcap, st);
  if (rc) return rc;
  const size_t qb = (size_t)B * g.dim * 8;
  COZO_CUDA(cudaMalloc(&bf.p[0], qb));
  COZO_CUDA(cudaMalloc(&bf.p[1], (size_t)B * k * 4));
  COZO_CUDA(cudaMalloc(&bf.p[2], (size_t)B * k * 8));
  COZO_CUDA(cudaMalloc(&bf.p[3], (size_t)B * 4));
  COZO_CUDA(cudaMalloc(&bf.p[4], (size_t)B * 16));
  if (row_mask) {
    const size_t words = ((size_t)g.n + 31) / 32;
    COZO_CUDA(cudaMalloc(&bf.p[5], std::max<size_t>(words, 1) * 4));
    COZO_CUDA(cudaMemcpyAsync(bf.p[5], row_mask, words * 4, cudaMemcpyHostToDevice, st));
  }
  COZO_CUDA(cudaMemcpyAsync(bf.p[0], queries, qb, cudaMemcpyHostToDevice, st));
  p.queries = static_cast<const double*>(bf.p[0]);
  p.vec64 = h->d_vec64;
  p.ld64 = h->ld64;
  p.B = B;
  p.k = k;
  p.ef = ef;
  p.has_radius = radius >= 0.0;
  p.radius = radius;
  p.out_ids = static_cast<uint32_t*>(bf.p[1]);
  p.out_dist = static_cast<double*>(bf.p[2]);
  p.out_count = static_cast<uint32_t*>(bf.p[3]);
  p.qstats = static_cast<uint32_t*>(bf.p[4]);
  p.counter = ws->counter;
  p.vis = ws->vis;
  p.nwords = nwords;
  p.vlog = ws->vlog;
  p.logcap = logcap;
  p.filter_mask = row_mask ? static_cast<const uint32_t*>(bf.p[5]) : nullptr;
  COZO_CUDA(cudaMemsetAsync(ws->counter, 0, 4, st));
  COZO_CUDA(cudaEventRecord(ws->e0, st));
  fn<<<grid, wpc * 32, smem, st>>>(g, p);
  COZO_CUDA(cudaGetLastError());
  COZO_CUDA(cudaEventRecord(ws->e1, st));
  COZO_CUDA(cudaMemcpyAsync(out_ids, bf.p[1], (size_t)B * k * 4, cudaMemcpyDeviceToHost, st));
  COZO_CUDA(cudaMemcpyAsync(out_dist, bf.p[2], (size_t)B * k * 8, cudaMemcpyDeviceToHost, st));
  if (out_count) COZO_CUDA(cudaMemcpyAsync(out_count, bf.p[3], (size_t)B * 4, cudaMemcpyDeviceToHost, st));
  std::vector<uint32_t> qs;
  if (stats) {
    qs.resize((size_t)B * 4);
    COZO_CUDA(cudaMemcpyAsync(qs.data(), bf.p[4], (size_t)B * 16, cudaMemcpyDeviceToHost, st));
  }
  COZO_CUDA(cudaStreamSynchronize(st));
  if (stats) {
    float ms = 0;
    cudaEventElapsedTime(&ms, ws->e0, ws->e1);
    stats->n_queries = B;
    stats->kernel_ms = ms;
    for (uint32_t i = 0; i < B; ++i) {
      stats->dist_evals += qs[(size_t)i * 4 + 0];
      stats->nodes_expanded += qs[(size_t)i * 4 + 1];
      stats->nbr_reads += qs[(size_t)i * 4 + 2];
    }
  }
  return 0;
}
