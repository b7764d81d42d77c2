// hnsw_build_kernels.cuh — device code of the index builder (hnsw_build.cu): batch search (K1), heuristic selection
// with optional candidate extension (K2), link / shrink (K4), edge distances, removal.  A header so that the same source
// is compiled by nvcc into libcozo_gpu.so and by tests/emu (CPU SIMT emulator, test infrastructure) into a host program.
#pragma once
#include "hnsw_device.cuh"

namespace cozo {

struct SmemLayout {
  uint32_t off_fi, off_pend, off_bars, off_ring, warp_bytes;
};
inline SmemLayout make_layout(uint32_t ef, uint32_t ns, uint32_t ld) {
  SmemLayout l;
  uint32_t efcap = round_up(ef, 32);
  l.off_fi = efcap * 4;
  l.off_pend = l.off_fi + efcap * 4;
  l.off_bars = l.off_pend + 32 * 4;
  l.off_ring = round_up(l.off_bars + ns * 8, 128);
  l.warp_bytes = round_up(l.off_ring + ns * ld * 4, 128);
  return l;
}

struct BuildDev {
  uint32_t* adj0;
  float* adj0_d;
  uint32_t* deg0;
  uint32_t* adj_up;
  float* adj_up_d;
  uint32_t* deg_up;
  const uint8_t* node_level;
  uint32_t m_max0, m_max;
  int keep_pruned;
  // extend_candidates (hnsw.rs:499-511): per-task scratch of `ext_cap` (a power of two) entries each
  int extend;
  const uint32_t* upper_off;
  unsigned long long* ext_keys;
  float* ext_d;
  uint32_t* ext_id;
  uint32_t ext_cap;
};

struct BatchParams {
  uint32_t begin, count;  // node ids [begin, begin+count)
  uint32_t top;           // top layer before the batch
  uint32_t ef_c;
  const uint32_t* coff;        // [count+1] first candidate list of node i
  const uint32_t* list_node;   // [T]
  const uint32_t* list_level;  // [T]
  uint32_t T;
  float* cand_d;       // [T x ef_c] ascending
  uint32_t* cand_id;   // [T x ef_c]
  uint32_t* cand_cnt;  // [T]
  // in-edge queue
  unsigned long long* req_key;  // (layer << 32) | target
  uint32_t* req_src;
  float* req_d;
  uint32_t* req_count;
  // workspace
  uint32_t* counter;
  uint32_t* vis;
  uint32_t nwords;
  uint32_t* vlog;
  uint32_t logcap;
  uint32_t ns;
  SmemLayout lay;
};

// K1 ------------------------------------------------------------------------
template <int NV, int METRIC>
__device__ __forceinline__ void build_search_body(const HnswDev& g, const BuildDev& b, const BatchParams& p, uint8_t* smem) {
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int wpc = blockDim.x >> 5;
  uint8_t* base = smem + (size_t)warp * p.lay.warp_bytes;
  WarpCtx w;
  w.fd = reinterpret_cast<float*>(base);
  w.fi = reinterpret_cast<uint32_t*>(base + p.lay.off_fi);
  w.pend = reinterpret_cast<uint32_t*>(base + p.lay.off_pend);
  w.bars = reinterpret_cast<uint64_t*>(base + p.lay.off_bars);
  w.ring = reinterpret_cast<float*>(base + p.lay.off_ring);
  const size_t slot = (size_t)blockIdx.x * wpc + warp;
  w.vis = p.vis + slot * p.nwords;
  w.nwords = p.nwords;
  w.vlog = p.vlog + slot * p.logcap;
  w.logcap = p.logcap;
  w.ns = p.ns;
  w.nlog = 0;
  w.head = 0;
  w.phase = 0;
  if (lane == 0) {
    for (uint32_t s = 0; s < p.ns; ++s) mbar_init(&w.bars[s], 1);
    mbar_fence_init();
  }
  __syncwarp();
  const int nvec4 = g.ld >> 2;
  for (;;) {
    uint32_t i = 0;
    if (lane == 0) i = atomicAdd(p.counter, 1u);
    i = __shfl_sync(0xffffffffu, i, 0);
    if (i >= p.count) break;
    const uint32_t id = p.begin + i;
    const uint32_t lq = b.node_level[id];
    float4 q[NV];
    float qnorm;
    load_query<NV>(g.vec + (size_t)id * g.ld, g.ld, lane, q, qnorm);
    float d = dist_ldg1<NV, METRIC>(q, reinterpret_cast<const float4*>(g.vec + (size_t)g.entry * g.ld), lane, nvec4,
                                    qnorm);
    if (lane == 0) {
      w.fd[0] = d;
      w.fi[0] = g.entry;
    }
    w.len = 1;
    w.cursor = 0;
    w.dist_evals = w.nodes_expanded = w.nbr_reads = 0;
    __syncwarp();
    for (uint32_t L = p.top; L > lq; --L) search_level<NV, METRIC, true>(g, w, q, qnorm, 1, L, lane);
    uint32_t L = lq < p.top ? lq : p.top;
    const uint32_t l0 = p.coff[i];
    for (;; --L) {
      search_level<NV, METRIC, true>(g, w, q, qnorm, p.ef_c, L, lane);
      const size_t list = (size_t)(l0 + L) * p.ef_c;
      for (uint32_t j = lane; j < w.len; j += 32) {
        p.cand_d[list + j] = w.fd[j];
        p.cand_id[list + j] = w.fi[j] & IDMASK;
      }
      if (lane == 0) p.cand_cnt[l0 + L] = w.len;
      __syncwarp();
      if (L == 0) break;
    }
  }
}

// hnsw_select_neighbours_heuristic (hnsw.rs:470-538) over candidates sorted by
// ascending distance to the base vector.  `cd/cid` may live in global or shared
// memory; bit31 of cid is set on selected entries.  Returns |ret|.
template <int NV, int METRIC>
__device__ __forceinline__ uint32_t heuristic_select(const HnswDev& g, const float* cd, uint32_t* cid, uint32_t cnt,
                                                     uint32_t mm, bool keep_pruned, uint32_t* sel_id, float* sel_d,
                                                     int lane) {
  const int nvec4 = g.ld >> 2;
  uint32_t ns = 0;
  uint32_t c = 0;
  for (; c < cnt && ns < mm; ++c) {  // hnsw.rs:512
    const uint32_t id = cid[c] & IDMASK;
    const float dq = cd[c];
    float4 cv[NV];
    float cnorm;
    load_query<NV>(g.vec + (size_t)id * g.ld, g.ld, lane, cv, cnorm);
    bool add = true;
    for (uint32_t e = 0; e < ns; ++e) {  // hnsw.rs:515-523
      float de = dist_ldg1<NV, METRIC>(cv, reinterpret_cast<const float4*>(g.vec + (size_t)sel_id[e] * g.ld), lane,
                                       nvec4, cnorm);
      if (de < dq) {
        add = false;
        break;
      }
    }
    if (add) {
      __syncwarp();  // all lanes have read cid[c] / sel_id[..] before lane 0 updates them
      if (lane == 0) {
        sel_id[ns] = id;
        sel_d[ns] = dq;
        cid[c] = id | EXPANDED;
      }
      ++ns;
      __syncwarp();
    }
  }
  if (keep_pruned && c == cnt) {  // discarded back-fill, nearest first (hnsw.rs:530-536)
    for (uint32_t j = 0; j < cnt && ns < mm; ++j) {
      uint32_t v = cid[j];
      if (v & EXPANDED) continue;
      if (lane == 0) {
        sel_id[ns] = v;
        sel_d[ns] = cd[j];
      }
      ++ns;
    }
    __syncwarp();
  }
  return ns;
}

// ---- extend_candidates (hnsw.rs:499-511) ----------------------------------------------------------------------
// candidates = found ∪ neighbours(found) at the layer, every distance to the base vector (re)computed, popped nearest
// first.  A fidelity mode for small indexes: it multiplies the distance evaluations of selection by the degree
// (the reference pays the same), so the builder restricts it to small batches.  The base vector's own key is skipped:
// the reference's shrink path would admit it (and overwrite its self-loop row, hnsw.rs:413-432), which the oracle
// treats as a defect too.
__device__ __forceinline__ uint32_t f32_order_key(float f) {
  const uint32_t b = __float_as_uint(f);
  return b ^ ((b >> 31) ? 0xFFFFFFFFu : 0x80000000u);
}
__device__ __forceinline__ float f32_from_order_key(uint32_t k) {
  return __uint_as_float((k & 0x80000000u) ? (k ^ 0x80000000u) : ~k);
}
// bitonic sort of n (a power of two) u64 keys by one warp
__device__ __forceinline__ void warp_bitonic_sort(unsigned long long* a, uint32_t n, int lane) {
  for (uint32_t k = 2; k <= n; k <<= 1)
    for (uint32_t j = k >> 1; j > 0; j >>= 1) {
      for (uint32_t i = lane; i < n; i += 32) {
        const uint32_t ixj = i ^ j;
        if (ixj > i) {
          const unsigned long long x = a[i], y = a[ixj];
          const bool up = (i & k) == 0;
          if ((x > y) == up) {
            a[i] = y;
            a[ixj] = x;
          }
        }
      }
      __syncwarp();
    }
}
// Builds the extended, distance-sorted candidate list of `task` in its scratch slice; returns its length.
// base_d / base_id: the found list (ascending); q: the base vector; self: its id.
template <int NV, int METRIC>
__device__ __forceinline__ uint32_t extend_candidate_list(const HnswDev& g, const BuildDev& b, const float4 (&q)[NV],
                                                          float qnorm, uint32_t self, uint32_t level, const float* base_d,
                                                          const uint32_t* base_id, uint32_t cnt, size_t task, int lane) {
  unsigned long long* keys = b.ext_keys + task * b.ext_cap;
  float* cd = b.ext_d + task * b.ext_cap;
  uint32_t* cid = b.ext_id + task * b.ext_cap;
  const uint32_t cap = b.ext_cap;
  const int nvec4 = g.ld >> 2;
  // A. raw ids: the found items (they carry their distance) and every neighbour of a found item
  for (uint32_t i = lane; i < cnt && i < cap; i += 32) keys[i] = ((unsigned long long)(base_id[i] & IDMASK) << 32) | i;
  uint32_t nraw = cnt < cap ? cnt : cap;
  const uint32_t stride = level == 0 ? g.s0 : g.su;
  for (uint32_t f = 0; f < cnt; ++f) {
    const uint32_t fid = base_id[f] & IDMASK;
    const uint32_t* row = level == 0 ? b.adj0 + (size_t)fid * g.s0 : b.adj_up + (size_t)(b.upper_off[fid] + level - 1) * g.su;
    for (uint32_t nb = 0; nb < stride; nb += 32) {
      const uint32_t id = row[nb + lane];
      if (!__ballot_sync(0xffffffffu, id != NONE)) break;
      const bool ok = id != NONE && id != self;
      const uint32_t bal = __ballot_sync(0xffffffffu, ok);
      const uint32_t pos = nraw + __popc(bal & ((1u << lane) - 1));
      if (ok && pos < cap) keys[pos] = ((unsigned long long)id << 32) | 0xFFFFFFFFull;
      nraw += __popc(bal);
    }
  }
  if (nraw > cap) nraw = cap;
  uint32_t n2 = 32;
  while (n2 < nraw) n2 <<= 1;
  for (uint32_t i = nraw + lane; i < n2; i += 32) keys[i] = ~0ull;
  __syncwarp();
  warp_bitonic_sort(keys, n2, lane);  // by (id, origin): a found item precedes the neighbour copies of the same id
  // B. unique ids; distances: known for found items, computed for the rest
  uint32_t nu = 0;
  for (uint32_t base = 0; base < nraw; base += 32) {
    const uint32_t i = base + lane;
    const unsigned long long k = i < nraw ? keys[i] : ~0ull;
    const uint32_t id = (uint32_t)(k >> 32);
    const uint32_t prev = (i > 0 && i < nraw) ? (uint32_t)(keys[i - 1] >> 32) : NONE;
    const bool keep = i < nraw && id != prev;
    const uint32_t bal = __ballot_sync(0xffffffffu, keep);
    const uint32_t pos = nu + __popc(bal & ((1u << lane) - 1));
    if (keep) {
      cid[pos] = id;
      const uint32_t origin = (uint32_t)k;
      cd[pos] = origin != 0xFFFFFFFFu ? base_d[origin] : __int_as_float(0x7FC00000);
    }
    nu += __popc(bal);
  }
  __syncwarp();
  for (uint32_t i = 0; i < nu; ++i) {
    float d = cd[i];
    if (d != d) {  // not yet known (warp-uniform: every lane reads the same slot)
      d = dist_ldg1<NV, METRIC>(q, reinterpret_cast<const float4*>(g.vec + (size_t)cid[i] * g.ld), lane, nvec4, qnorm);
      __syncwarp();
      if (lane == 0) cd[i] = d;
    }
  }
  __syncwarp();
  // C. nearest first (ties by id)
  n2 = 32;
  while (n2 < nu) n2 <<= 1;
  for (uint32_t i = lane; i < n2; i += 32)
    keys[i] = i < nu ? (((unsigned long long)f32_order_key(cd[i]) << 32) | cid[i]) : ~0ull;
  __syncwarp();
  warp_bitonic_sort(keys, n2, lane);
  for (uint32_t i = lane; i < nu; i += 32) {
    const unsigned long long k = keys[i];
    cd[i] = f32_from_order_key((uint32_t)(k >> 32));
    cid[i] = (uint32_t)k;
  }
  __syncwarp();
  return nu;
}

__device__ __forceinline__ void adj_row(const HnswDev& g, const BuildDev& b, uint32_t node, uint32_t level,
                                        uint32_t*& ids, float*& ds, uint32_t*& deg, uint32_t& stride, uint32_t& mm) {
  if (level == 0) {
    ids = b.adj0 + (size_t)node * g.s0;
    ds = b.adj0_d + (size_t)node * g.s0;
    deg = b.deg0 + node;
    stride = g.s0;
    mm = b.m_max0;
  } else {
    size_t row = (size_t)g.upper_off[node] + level - 1;
    ids = b.adj_up + row * g.su;
    ds = b.adj_up_d + row * g.su;
    deg = b.deg_up + row;
    stride = g.su;
    mm = b.m_max;
  }
}

// K2 ------------------------------------------------------------------------
template <int NV, int METRIC>
__device__ __forceinline__ void build_select_body(const HnswDev& g, const BuildDev& b, const BatchParams& p, uint8_t* smem) {
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const uint32_t mcap = b.m_max0 > b.m_max ? b.m_max0 : b.m_max;
  uint32_t* sel_id = reinterpret_cast<uint32_t*>(smem) + (size_t)warp * 2 * mcap;
  float* sel_d = reinterpret_cast<float*>(sel_id + mcap);
  const uint32_t t = blockIdx.x * (blockDim.x >> 5) + warp;
  if (t >= p.T) return;
  const uint32_t node = p.list_node[t], level = p.list_level[t];
  uint32_t *ids, *deg;
  float* ds;
  uint32_t stride, mm;
  adj_row(g, b, node, level, ids, ds, deg, stride, mm);
  const size_t list = (size_t)t * p.ef_c;
  const float* cd = p.cand_d + list;
  uint32_t* cid = p.cand_id + list;
  uint32_t ccnt = p.cand_cnt[t];
  if (b.extend) {  // hnsw.rs:499-511
    float4 q[NV];
    float qn;
    load_query<NV>(g.vec + (size_t)node * g.ld, g.ld, lane, q, qn);
    ccnt = extend_candidate_list<NV, METRIC>(g, b, q, qn, node, level, cd, cid, ccnt, t, lane);
    cd = b.ext_d + (size_t)t * b.ext_cap;
    cid = b.ext_id + (size_t)t * b.ext_cap;
  }
  uint32_t ns = heuristic_select<NV, METRIC>(g, cd, cid, ccnt, mm, b.keep_pruned != 0, sel_id, sel_d, lane);
  __syncwarp();
  uint32_t rbase = 0;
  // The reference writes a neighbour's out edge, its in edge and the shrink of that neighbour one neighbour at a time
  // (hnsw.rs:279-357).  With extend_candidates a shrink reads the rows of the target's neighbours — the new node among
  // them — so it sees only the out edges written SO FAR.  In that mode the row starts empty here and the sequential link
  // step appends out edge r right before it links in edge r.  Without extension nothing reads the new node's row while
  // its neighbours are linked, and the whole row is written at once.
  const bool incremental = b.extend != 0;
  if (lane == 0) {
    *deg = incremental ? 0u : ns;
    rbase = atomicAdd(p.req_count, ns);
  }
  rbase = __shfl_sync(0xffffffffu, rbase, 0);
  if (incremental)
    for (uint32_t j = lane; j < stride; j += 32) ids[j] = NONE;
  for (uint32_t j = lane; j < ns; j += 32) {
    if (!incremental) {
      ids[j] = sel_id[j];  // out edge (hnsw.rs:281-298)
      ds[j] = sel_d[j];
    }
    p.req_key[rbase + j] = ((unsigned long long)level << 32) | sel_id[j];  // in edge (hnsw.rs:300-318)
    p.req_src[rbase + j] = node;
    p.req_d[rbase + j] = sel_d[j];
  }
}

// segment heads of the sorted in-edge queue
__global__ void build_heads_kernel(const unsigned long long* keys, uint32_t n, uint32_t* heads, uint32_t* nheads) {
  uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n) return;
  if (r == 0 || keys[r] != keys[r - 1]) heads[atomicAdd(nheads, 1u)] = r;
}

// K4 ------------------------------------------------------------------------
template <int NV, int METRIC>
__device__ __forceinline__ void build_link_body(const HnswDev& g, const BuildDev& b, const unsigned long long* keys,
                                                         const uint32_t* perm, const uint32_t* req_src,
                                                         const float* req_d, uint32_t nreq, const uint32_t* heads,
                                                         uint32_t nheads, uint8_t* smem) {
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const uint32_t mcap = b.m_max0 > b.m_max ? b.m_max0 : b.m_max;
  const uint32_t ucap = mcap + 32;
  // per warp: u_id,u_d,s_id,s_d [ucap] ; sel_id, sel_d [mcap]
  uint32_t* wbase = reinterpret_cast<uint32_t*>(smem) + (size_t)warp * (4 * ucap + 2 * mcap);
  uint32_t* u_id = wbase;
  float* u_d = reinterpret_cast<float*>(wbase + ucap);
  uint32_t* s_id = wbase + 2 * ucap;
  float* s_d = reinterpret_cast<float*>(wbase + 3 * ucap);
  uint32_t* sel_id = wbase + 4 * ucap;
  float* sel_d = reinterpret_cast<float*>(wbase + 4 * ucap + mcap);
  const uint32_t h = blockIdx.x * (blockDim.x >> 5) + warp;
  if (h >= nheads) return;
  const uint32_t start = heads[h];
  const unsigned long long key = keys[start];
  const uint32_t level = (uint32_t)(key >> 32), node = (uint32_t)(key & 0xFFFFFFFFull);
  uint32_t end = start + 1;
  while (end < nreq && keys[end] == key) ++end;
  uint32_t *ids, *degp;
  float* ds;
  uint32_t stride, mm;
  if (b.extend) {  // sequential mode, one request per launch: the source's out edge first (hnsw.rs:281-298) ...
    end = start + 1;
    const uint32_t r = perm[start];
    const uint32_t src = req_src[r];
    uint32_t *sids, *sdeg, sstride, smm;
    float* sds;
    adj_row(g, b, src, level, sids, sds, sdeg, sstride, smm);
    if (lane == 0) {
      const uint32_t d = *sdeg;
      sids[d] = node;
      sds[d] = req_d[r];
      *sdeg = d + 1;
    }
    __syncwarp();
  }
  adj_row(g, b, node, level, ids, ds, degp, stride, mm);  // ... then the in edge (hnsw.rs:300-318)
  uint32_t deg = *degp;
  for (uint32_t a0 = start; a0 < end; a0 += 32) {
    const uint32_t na = min(32u, end - a0);
    uint32_t asrc = NONE;
    float ad = 0.f;
    if ((uint32_t)lane < na) {
      uint32_t r = perm[a0 + lane];
      asrc = req_src[r];
      ad = req_d[r];
    }
    if (deg + na <= mm) {  // plain append (hnsw.rs:338-339 not exceeded)
      if ((uint32_t)lane < na) {
        ids[deg + lane] = asrc;
        ds[deg + lane] = ad;
      }
      deg += na;
      __syncwarp();
      continue;
    }
    // shrink (hnsw.rs:376-469): candidates = stored out-neighbours + arrivals
    const uint32_t nc = deg + na;
    for (uint32_t j = lane; j < deg; j += 32) {
      u_id[j] = ids[j];
      u_d[j] = ds[j];
    }
    if ((uint32_t)lane < na) {
      u_id[deg + lane] = asrc;
      u_d[deg + lane] = ad;
    }
    __syncwarp();
    // rank sort by (distance, position).  The order must be total for the ranks to be a permutation: with raw
    // compares every NaN distance (a zero-norm Cosine row) got rank 0 and slots of s_id were left unwritten.
    for (uint32_t j = lane; j < nc; j += 32) {
      float dj = u_d[j];
      uint32_t rank = 0;
      for (uint32_t x = 0; x < nc; ++x) {
        float dx = u_d[x];
        rank += precedes(dx, dj) || (!precedes(dj, dx) && x < j);
      }
      s_id[rank] = u_id[j];
      s_d[rank] = dj;
    }
    __syncwarp();
    uint32_t ns;
    if (b.extend) {  // hnsw_shrink_neighbour selects through the same routine, extension included (hnsw.rs:394-409)
      float4 q[NV];
      float qn;
      load_query<NV>(g.vec + (size_t)node * g.ld, g.ld, lane, q, qn);
      const uint32_t ne = extend_candidate_list<NV, METRIC>(g, b, q, qn, node, level, s_d, s_id, nc, h, lane);
      ns = heuristic_select<NV, METRIC>(g, b.ext_d + (size_t)h * b.ext_cap, b.ext_id + (size_t)h * b.ext_cap, ne, mm,
                                        b.keep_pruned != 0, sel_id, sel_d, lane);
    } else {
      ns = heuristic_select<NV, METRIC>(g, s_d, s_id, nc, mm, b.keep_pruned != 0, sel_id, sel_d, lane);
    }
    __syncwarp();
    for (uint32_t j = lane; j < stride; j += 32) {
      bool in = j < ns;
      if (in || j < nc) {
        ids[j] = in ? sel_id[j] : NONE;
        ds[j] = in ? sel_d[j] : 0.f;
      }
    }
    deg = ns;
    __syncwarp();
  }
  if (lane == 0) *degp = deg;
}

// distances of the stored edges of an index that was staged from the host (the index relation
// keeps them in its `dist` column, runtime/relation.rs:1064-1126; the staged layout does not)
template <int NV, int METRIC>
__global__ void __launch_bounds__(128) build_edge_dist_kernel(HnswDev g, BuildDev b, const uint32_t* row_owner,
                                                              uint32_t n_rows, int upper) {
  const int lane = threadIdx.x & 31;
  const uint32_t r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (r >= n_rows) return;
  const uint32_t owner = upper ? row_owner[r] : r;
  const uint32_t stride = upper ? g.su : g.s0;
  uint32_t* ids = (upper ? b.adj_up : b.adj0) + (size_t)r * stride;
  float* ds = (upper ? b.adj_up_d : b.adj0_d) + (size_t)r * stride;
  uint32_t* deg = (upper ? b.deg_up : b.deg0) + r;
  if (owner == NONE) {
    if (lane == 0) *deg = 0;
    return;
  }
  const int nvec4 = g.ld >> 2;
  float4 q[NV];
  float qn;
  load_query<NV>(g.vec + (size_t)owner * g.ld, g.ld, lane, q, qn);
  uint32_t cnt = 0;
  for (uint32_t j = 0; j < stride; ++j) {
    const uint32_t t = ids[j];
    if (t == NONE) break;
    float d = dist_ldg1<NV, METRIC>(q, reinterpret_cast<const float4*>(g.vec + (size_t)t * g.ld), lane, nvec4, qn);
    if (lane == 0) ds[j] = d;
    ++cnt;
  }
  if (lane == 0) *deg = cnt;
}

// hnsw_remove_vec (hnsw.rs:754-868): the node's rows are deleted on every layer and every edge
// that points at it goes away.  One warp per adjacency row drops dead targets and repacks.
__global__ void __launch_bounds__(128) remove_compact_kernel(uint32_t* adj, float* adj_d, uint32_t* deg, uint32_t stride,
                                                             uint32_t n_rows, const uint32_t* row_owner,
                                                             const uint8_t* dead) {
  const int lane = threadIdx.x & 31;
  const uint32_t r = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (r >= n_rows) return;
  uint32_t* ids = adj + (size_t)r * stride;
  float* ds = adj_d ? adj_d + (size_t)r * stride : nullptr;
  const uint32_t owner = row_owner ? row_owner[r] : r;
  const bool owner_dead = owner == NONE || dead[owner];
  uint32_t out = 0;
  for (uint32_t base = 0; base < stride; base += 32) {
    const uint32_t t = ids[base + lane];
    const float d = ds ? ds[base + lane] : 0.f;
    const bool keep = !owner_dead && t != NONE && !dead[t];
    const uint32_t m = __ballot_sync(0xffffffffu, keep);
    const bool any_valid = __ballot_sync(0xffffffffu, t != NONE) != 0;
    __syncwarp();
    if (keep) {
      const uint32_t pos = out + __popc(m & ((1u << lane) - 1));
      ids[pos] = t;  // pos <= base + lane: never overtakes an unread slot of a later chunk
      if (ds) ds[pos] = d;
    }
    out += __popc(m);
    __syncwarp();
    if (!any_valid) break;
  }
  for (uint32_t j = out + lane; j < stride; j += 32) ids[j] = NONE;
  if (deg && lane == 0) deg[r] = out;
}

__global__ void mark_dead_kernel(const uint32_t* ids, uint32_t count, uint8_t* dead) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < count) dead[ids[i]] = 1;
}

}  // namespace cozo
