// hnsw_device.cuh — device-side HNSW layer search shared by the batched k-NN
// kernel and the batched index builder.
//
// Semantics follow SessionTx::hnsw_search_level (runtime/hnsw.rs:539-587) with
// one warp per query:
//   * `found_nn` (max-queue bounded by ef) and `candidates` (min-queue) are ONE
//     sorted array in shared memory: found = the array, candidates = its not yet
//     expanded entries.  An admitted neighbour that was later evicted from
//     found_nn has dist >= furthest, so the reference pops it only to `break`
//     (hnsw.rs:562); dropping it changes nothing except on exact distance ties.
//   * the neighbours of one candidate are evaluated together; admission
//     (hnsw.rs:575-581) is applied in neighbour order with the live bound, so the
//     traversal, dist_evals and nodes_expanded equal the reference's.
//   * `visited` (hnsw.rs:549) is a per-warp bitmap in HBM, set with atomicOr and
//     cleared at the end of every layer through a log of the ids that were set.
#pragma once
#include "common.cuh"

namespace cozo {

struct HnswDev {
  const float* vec;  // [n x ld] row-major f32, rows zero-padded to ld (multiple of 4)
  uint32_t n, dim, ld;
  int metric;
  const uint32_t* adj0;       // layer 0: [n x s0], ids packed at the front, NONE padded
  uint32_t s0;                // multiple of 32
  const uint32_t* upper_off;  // [n] first row in adj_up of the node's layer -1 list, NONE if layer 0 only
  const uint32_t* adj_up;     // [rows x su]; node on layers 1..t owns rows upper_off .. upper_off+t-1
  uint32_t su;                // multiple of 32
  uint32_t entry;             // NONE = empty index
  uint32_t top_level;         // entry lives on layer -top_level
};

struct WarpCtx {
  float* fd;       // smem: sorted distances (ascending)
  uint32_t* fi;    // smem: ids, bit31 = expanded
  uint32_t* pend;  // smem [32]: compacted unvisited neighbour ids of the current hop
  float* ring;     // smem: NS row buffers (bulk mode)
  uint64_t* bars;  // smem: NS mbarriers (bulk mode)
  uint32_t* vis;   // HBM: this warp's visited bitmap, all zero between layers
  uint32_t nwords;
  uint32_t* vlog;  // HBM: ids whose bit was set on this layer
  uint32_t logcap;
  uint32_t ns;     // ring stages
  // registers, warp-uniform
  uint32_t len, cursor, nlog;
  uint32_t head, phase;  // ring position / per-stage parity bits
  uint32_t dist_evals, nodes_expanded, nbr_reads;
};

constexpr uint32_t EXPANDED = 0x80000000u;
constexpr uint32_t IDMASK = 0x7FFFFFFFu;

template <int METRIC>
__device__ __forceinline__ void accum(const float4& q, const float4& v, float& a, float& b) {
  if (METRIC == COZO_GPU_L2) {
    float dx = q.x - v.x, dy = q.y - v.y, dz = q.z - v.z, dw = q.w - v.w;
    a = fmaf(dx, dx, a);
    a = fmaf(dy, dy, a);
    a = fmaf(dz, dz, a);
    a = fmaf(dw, dw, a);
  } else {
    a = fmaf(q.x, v.x, a);
    a = fmaf(q.y, v.y, a);
    a = fmaf(q.z, v.z, a);
    a = fmaf(q.w, v.w, a);
    if (METRIC == COZO_GPU_COSINE) {
      b = fmaf(v.x, v.x, b);
      b = fmaf(v.y, v.y, b);
      b = fmaf(v.z, v.z, b);
      b = fmaf(v.w, v.w, b);
    }
  }
}

// VectorCache::dist (hnsw.rs:66-109): reduce the per-lane partials and apply the
// metric's final scalar step in f64, then round to the f32 ordering key.
template <int METRIC>
__device__ __forceinline__ float finish(float a, float b, float qnorm) {
  a = warp_sum(a);
  if (METRIC == COZO_GPU_L2) return a;
  if (METRIC == COZO_GPU_IP) return (float)(1.0 - (double)a);
  b = warp_sum(b);
  return (float)(1.0 - (double)a / sqrt((double)qnorm * (double)b));
}

template <int NV, int METRIC>
__device__ __forceinline__ float dist_smem(const float4 (&q)[NV], const float4* row, int lane, int nvec4,
                                           float qnorm) {
  float a = 0.f, b = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    int idx = lane + 32 * i;
    if (idx < nvec4) accum<METRIC>(q[i], row[idx], a, b);
  }
  return finish<METRIC>(a, b, qnorm);
}

// two rows at once straight from HBM: all 2*NV 128-bit loads are issued before
// the first use so one warp keeps 2 rows in flight.
template <int NV, int METRIC>
__device__ __forceinline__ void dist_ldg2(const float4 (&q)[NV], const float4* r0, const float4* r1, int lane,
                                          int nvec4, float qnorm, float& d0, float& d1) {
  float4 v0[NV], v1[NV];
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    int idx = lane + 32 * i;
    if (idx < nvec4) {
      v0[i] = ldg_nc_f4(r0 + idx);
      v1[i] = ldg_nc_f4(r1 + idx);
    }
  }
  float a0 = 0.f, b0 = 0.f, a1 = 0.f, b1 = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    int idx = lane + 32 * i;
    if (idx < nvec4) {
      accum<METRIC>(q[i], v0[i], a0, b0);
      accum<METRIC>(q[i], v1[i], a1, b1);
    }
  }
  d0 = finish<METRIC>(a0, b0, qnorm);
  d1 = finish<METRIC>(a1, b1, qnorm);
}

template <int NV, int METRIC>
__device__ __forceinline__ float dist_ldg1(const float4 (&q)[NV], const float4* r0, int lane, int nvec4,
                                           float qnorm) {
  float4 v0[NV];
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    int idx = lane + 32 * i;
    if (idx < nvec4) v0[i] = ldg_nc_f4(r0 + idx);
  }
  float a0 = 0.f, b0 = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    int idx = lane + 32 * i;
    if (idx < nvec4) accum<METRIC>(q[i], v0[i], a0, b0);
  }
  return finish<METRIC>(a0, b0, qnorm);
}

// found_nn.push + pop-if-over-ef (hnsw.rs:577-580) on the sorted array.
// Precondition: len < ef || d < fd[len-1].  Equal keys keep arrival order; NaN keys sort last (`precedes`).
__device__ __forceinline__ void sorted_insert(WarpCtx& w, uint32_t ef, float d, uint32_t id, int lane) {
  uint32_t pos = 0;
  for (uint32_t base = 0; base < w.len; base += 32) {
    uint32_t i = base + lane;
    bool le = (i < w.len) && !precedes(d, w.fd[i]);
    uint32_t bal = __ballot_sync(0xffffffffu, le);
    pos += __popc(bal);
    if (bal != 0xffffffffu) break;
  }
  uint32_t newlen = w.len < ef ? w.len + 1 : ef;
  for (int top = (int)newlen - 1; top > (int)pos; top -= 32) {
    int i = top - 1 - lane;
    bool act = i >= (int)pos;
    float td = 0.f;
    uint32_t ti = 0;
    if (act) {
      td = w.fd[i];
      ti = w.fi[i];
    }
    __syncwarp();
    if (act) {
      w.fd[i + 1] = td;
      w.fi[i + 1] = ti;
    }
    __syncwarp();
  }
  __syncwarp();  // every lane has finished reading fd[len-1] / the shifted slots (vote ops do not order memory)
  if (lane == 0) {
    w.fd[pos] = d;
    w.fi[pos] = id;
  }
  __syncwarp();
  w.len = newlen;
  if (pos < w.cursor) w.cursor = pos;
}

// visited.insert for the ids in `id` (one per lane, NONE = idle); returns whether
// this lane's id was newly inserted.  Newly set ids are logged for the clear.
__device__ __forceinline__ bool visit_mark(WarpCtx& w, uint32_t id, int lane, uint32_t& newmask) {
  bool isnew = false;
  if (id != NONE) {
    uint32_t bit = 1u << (id & 31);
    uint32_t old = atomicOr(&w.vis[id >> 5], bit);
    isnew = !(old & bit);
  }
  newmask = __ballot_sync(0xffffffffu, isnew);
  if (isnew) {
    uint32_t p = w.nlog + __popc(newmask & ((1u << lane) - 1));
    if (p < w.logcap) w.vlog[p] = id;
  }
  w.nlog += __popc(newmask);
  return isnew;
}

__device__ __forceinline__ void visit_clear(WarpCtx& w, int lane) {
  __syncwarp();
  if (w.nlog <= w.logcap && w.nlog * 4 <= w.nwords) {
    for (uint32_t i = lane; i < w.nlog; i += 32) atomicAnd(&w.vis[w.vlog[i] >> 5], 0u);
  } else {
    uint4 z = make_uint4(0, 0, 0, 0);
    uint4* p = reinterpret_cast<uint4*>(w.vis);
    for (uint32_t i = lane; i < w.nwords / 4; i += 32) p[i] = z;
    __threadfence();
  }
  w.nlog = 0;
  __syncwarp();
}

// hnsw_search_level (hnsw.rs:539-587) for one query held in registers.
// `level` 0 is the bottom layer.  On entry the sorted array holds found_nn.
template <int NV, int METRIC, bool BULK>
__device__ __forceinline__ void search_level(const HnswDev& g, WarpCtx& w, const float4 (&q)[NV], float qnorm,
                                             uint32_t ef, uint32_t level, int lane) {
  const int nvec4 = g.ld >> 2;
  const uint32_t row_bytes = g.ld * 4;
  // visited <- keys(found); candidates <- found (hnsw.rs:554-557)
  for (uint32_t base = 0; base < w.len; base += 32) {
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
    // candidates.pop(): nearest not-yet-expanded entry (hnsw.rs:559)
    uint32_t ci = NONE;
    for (uint32_t base = w.cursor & ~31u; base < w.len; base += 32) {
      uint32_t i = base + lane;
      bool un = (i < w.len) && (i >= w.cursor) && !(w.fi[i] & EXPANDED);
      uint32_t bal = __ballot_sync(0xffffffffu, un);
      if (bal) {
        ci = base + __ffs(bal) - 1;
        break;
      }
    }
    if (ci == NONE) break;  // == `candidate_dist > furthest_dist` break (hnsw.rs:562)
    uint32_t cand = w.fi[ci];
    __syncwarp();
    if (lane == 0) w.fi[ci] = cand | EXPANDED;
    w.cursor = ci + 1;
    w.nodes_expanded++;
    if (level == 0 && ci + 1 + lane < w.len && lane < 2) {
      // the next pop is most likely one of the following entries: pull their adjacency rows into L2
      uint32_t nxt = w.fi[ci + 1 + lane];
      if (!(nxt & EXPANDED))
        prefetch_l2(g.adj0 + (size_t)nxt * g.s0);
    }
    // hnsw_get_neighbours (hnsw.rs:588-629): one padded row
    const uint32_t* row;
    if (level == 0) {
      row = g.adj0 + (size_t)cand * g.s0;
    } else {
      uint32_t off = g.upper_off[cand];
      row = g.adj_up + (size_t)(off + level - 1) * g.su;
    }
    for (uint32_t nb = 0; nb < stride; nb += 32) {
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
      if (BULK) {
        // ring indices advance by compare-and-wrap (a runtime `% ns` costs ~20 instructions)
        uint32_t issued = 0, si = w.head, sc = w.head;
        for (uint32_t c = 0; c < cnt; ++c) {
          if (lane == 0) {
            fence_proxy_async_smem();
            while (issued < cnt && issued - c < w.ns) {
              mbar_expect_tx(&w.bars[si], row_bytes);
              bulk_g2s(w.ring + (size_t)si * g.ld, g.vec + (size_t)w.pend[issued] * g.ld, row_bytes, &w.bars[si]);
              ++issued;
              if (++si == w.ns) si = 0;
            }
          }
          mbar_wait(&w.bars[sc], (w.phase >> sc) & 1u);
          w.phase ^= (1u << sc);
          float d = dist_smem<NV, METRIC>(q, reinterpret_cast<const float4*>(w.ring + (size_t)sc * g.ld), lane, nvec4,
                                          qnorm);
          if (++sc == w.ns) sc = 0;
          uint32_t nid = w.pend[c];
          __syncwarp();
          if (w.len < ef || d < w.fd[w.len - 1]) sorted_insert(w, ef, d, nid, lane);  // hnsw.rs:575-581
        }
        w.head = sc;
      } else {
        for (uint32_t c = 0; c < cnt; c += 2) {
          uint32_t id0 = w.pend[c];
          bool two = c + 1 < cnt;
          uint32_t id1 = two ? w.pend[c + 1] : id0;
          float d0, d1;
          if (two) {
            dist_ldg2<NV, METRIC>(q, reinterpret_cast<const float4*>(g.vec + (size_t)id0 * g.ld),
                                  reinterpret_cast<const float4*>(g.vec + (size_t)id1 * g.ld), lane, nvec4, qnorm, d0,
                                  d1);
          } else {
            d0 = dist_ldg1<NV, METRIC>(q, reinterpret_cast<const float4*>(g.vec + (size_t)id0 * g.ld), lane, nvec4,
                                       qnorm);
            d1 = 0.f;
          }
          if (w.len < ef || d0 < w.fd[w.len - 1]) sorted_insert(w, ef, d0, id0, lane);
          if (two && (w.len < ef || d1 < w.fd[w.len - 1])) sorted_insert(w, ef, d1, id1, lane);
        }
      }
      __syncwarp();
    }
  }
  visit_clear(w, lane);
}

// ---------------------------------------------------------------------------------------------
// Cooperative form: ONE CTA (4 warps) per query.  Warp 0 owns the sorted found/candidate array, the
// visited bitmap and the admission order — exactly the routine above — but the rows of a hop are
// dealt round-robin to all warps, each with its own bulk-copy ring, and their distances meet in
// shared memory before warp 0 applies the admissions IN NEIGHBOUR ORDER.  Same traversal, same
// counters, same results; a query advances ~4x faster, which is what small batches (and the tail of
// a large one) need: there are not enough queries to fill the SMs with one warp each.
struct CoopShared {
  uint32_t* pend;    // [32] unvisited neighbour ids of the current round
  float* pdist;      // [32] their distances
  uint32_t* ctrl;    // [0] = number of rows of this round, COOP_DONE = layer finished
};
constexpr uint32_t COOP_DONE = 0xFFFFFFFFu;
constexpr uint32_t COOP_WARPS = 4;

template <int NV, int METRIC>
__device__ __forceinline__ void coop_search_level(const HnswDev& g, WarpCtx& w, const CoopShared& cs,
                                                  const float4 (&q)[NV], float qnorm, uint32_t ef, uint32_t level,
                                                  int lane, int warp) {
  const int nvec4 = g.ld >> 2;
  const uint32_t row_bytes = g.ld * 4;
  const uint32_t stride = level == 0 ? g.s0 : g.su;
  // warp-0 state of the current expansion
  const uint32_t* row = nullptr;
  uint32_t nb = stride;  // chunk offset inside the candidate's adjacency row; stride = need a new candidate
  if (warp == 0) {
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
  }
  for (;;) {
    if (warp == 0) {
      uint32_t cnt = 0;
      while (cnt == 0) {
        if (nb >= stride) {  // candidates.pop() (hnsw.rs:559)
          uint32_t ci = NONE;
          for (uint32_t base = w.cursor & ~31u; base < w.len; base += 32) {
            uint32_t i = base + lane;
            bool un = (i < w.len) && (i >= w.cursor) && !(w.fi[i] & EXPANDED);
            uint32_t bal = __ballot_sync(0xffffffffu, un);
            if (bal) {
              ci = base + __ffs(bal) - 1;
              break;
            }
          }
          if (ci == NONE) {
            cnt = COOP_DONE;
            break;
          }
          uint32_t cand = w.fi[ci];
          __syncwarp();
          if (lane == 0) w.fi[ci] = cand | EXPANDED;
          w.cursor = ci + 1;
          w.nodes_expanded++;
          if (level == 0 && ci + 1 + lane < w.len && lane < 2) {
            uint32_t nxt = w.fi[ci + 1 + lane];
            if (!(nxt & EXPANDED)) prefetch_l2(g.adj0 + (size_t)nxt * g.s0);
          }
          row = level == 0 ? g.adj0 + (size_t)cand * g.s0
                           : g.adj_up + (size_t)(g.upper_off[cand] + level - 1) * g.su;
          nb = 0;
        }
        uint32_t id = __ldg(row + nb + lane);
        uint32_t validmask = __ballot_sync(0xffffffffu, id != NONE);
        nb = validmask ? nb + 32 : stride;  // rows are packed: an empty chunk ends the row
        if (!validmask) continue;
        w.nbr_reads += __popc(validmask);
        uint32_t newmask;
        bool isnew = visit_mark(w, id, lane, newmask);
        cnt = __popc(newmask);
        if (isnew) cs.pend[__popc(newmask & ((1u << lane) - 1))] = id;
        w.dist_evals += cnt;
      }
      if (lane == 0) cs.ctrl[0] = cnt;
    }
    __syncthreads();  // the round's ids are published
    const uint32_t cnt = cs.ctrl[0];
    if (cnt == COOP_DONE) break;
    {  // every warp: rows warp, warp+4, ... through its own ring
      uint32_t issued = warp, si = w.head, sc = w.head;
      for (uint32_t c = warp; c < cnt; c += COOP_WARPS) {
        if (lane == 0) {
          fence_proxy_async_smem();
          while (issued < cnt && (issued - c) / COOP_WARPS < w.ns) {
            mbar_expect_tx(&w.bars[si], row_bytes);
            bulk_g2s(w.ring + (size_t)si * g.ld, g.vec + (size_t)cs.pend[issued] * g.ld, row_bytes, &w.bars[si]);
            issued += COOP_WARPS;
            if (++si == w.ns) si = 0;
          }
        }
        mbar_wait(&w.bars[sc], (w.phase >> sc) & 1u);
        w.phase ^= (1u << sc);
        float d = dist_smem<NV, METRIC>(q, reinterpret_cast<const float4*>(w.ring + (size_t)sc * g.ld), lane, nvec4,
                                        qnorm);
        if (++sc == w.ns) sc = 0;
        if (lane == 0) cs.pdist[c] = d;
        __syncwarp();
      }
      w.head = sc;
    }
    __syncthreads();  // all distances of the round are in shared memory
    if (warp == 0) {
      for (uint32_t c = 0; c < cnt; ++c) {  // hnsw.rs:575-581, in neighbour order with the live bound
        const float d = cs.pdist[c];
        const uint32_t nid = cs.pend[c];
        __syncwarp();
        if (w.len < ef || d < w.fd[w.len - 1]) sorted_insert(w, ef, d, nid, lane);
      }
    }
  }
  if (warp == 0) visit_clear(w, lane);
  __syncthreads();
}

// load one query into registers (zero padded), optionally its squared norm
template <int NV>
__device__ __forceinline__ void load_query(const float* qp, uint32_t dim, int lane, float4 (&q)[NV], float& qnorm) {
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    uint32_t e = (uint32_t)(lane + 32 * i) * 4;
    float4 v;
    v.x = e + 0 < dim ? qp[e + 0] : 0.f;
    v.y = e + 1 < dim ? qp[e + 1] : 0.f;
    v.z = e + 2 < dim ? qp[e + 2] : 0.f;
    v.w = e + 3 < dim ? qp[e + 3] : 0.f;
    q[i] = v;
    s = fmaf(v.x, v.x, s);
    s = fmaf(v.y, v.y, s);
    s = fmaf(v.z, v.z, s);
    s = fmaf(v.w, v.w, s);
  }
  qnorm = warp_sum(s);
}

}  // namespace cozo
