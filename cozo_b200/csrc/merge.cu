// merge.cu — global top-k over the per-shard top-k lists of a row-sharded corpus
// (SURVEY.md §8e).  Each shard ran the same hnsw_knn over its own index; the lists
// arrive nearest-first, so the merge is a k-way merge: one warp per query, lane s
// owns the head of shard s' list for s' = s, s+32, ...
#include "common.cuh"

namespace cozo {

__global__ void __launch_bounds__(128) topk_merge_kernel(const float* __restrict__ dist,
                                                         const uint32_t* __restrict__ ids, uint32_t n_shards,
                                                         uint32_t B, uint32_t k,
                                                         const unsigned long long* __restrict__ shard_offsets,
                                                         unsigned long long* __restrict__ out_ids,
                                                         float* __restrict__ out_dist) {
  const int lane = threadIdx.x & 31;
  const uint32_t q = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (q >= B) return;
  // this lane's current head among the shards it owns
  uint32_t my_shard = NONE, my_pos = 0;
  float my_d = INFINITY;
  uint32_t pos[8];  // heads of up to 8 owned shards (n_shards <= 256)
#pragma unroll
  for (int j = 0; j < 8; ++j) pos[j] = 0;
  auto refresh = [&]() {
    my_d = INFINITY;
    my_shard = NONE;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      uint32_t s = lane + 32 * j;
      if (s < n_shards && pos[j] < k) {
        size_t at = ((size_t)s * B + q) * k + pos[j];
        float d = dist[at];
        uint32_t id = ids[at];
        // (dist, shard) order with NaN last: a NaN head is taken once every finite head is out
        if (id != NONE && (my_shard == NONE || precedes(d, my_d) || (!precedes(my_d, d) && s < my_shard))) {
          my_d = d;
          my_shard = s;
          my_pos = pos[j];
        }
      }
    }
  };
  refresh();
  for (uint32_t r = 0; r < k; ++r) {
    // warp argmin on (dist, shard); NONE = this lane's shards are exhausted
    float bd = my_d;
    uint32_t bs = my_shard;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      float od = __shfl_xor_sync(0xffffffffu, bd, o);
      uint32_t os = __shfl_xor_sync(0xffffffffu, bs, o);
      if (os != NONE && (bs == NONE || precedes(od, bd) || (!precedes(bd, od) && os < bs))) {
        bd = od;
        bs = os;
      }
    }
    if (bs == NONE) {  // every list exhausted: pad
      if (lane == 0) {
        out_ids[(size_t)q * k + r] = ~0ull;
        out_dist[(size_t)q * k + r] = INFINITY;
      }
      continue;
    }
    if (my_shard == bs && (bs & 31) == (uint32_t)lane) {
      size_t at = ((size_t)bs * B + q) * k + my_pos;
      out_ids[(size_t)q * k + r] = shard_offsets[bs] + ids[at];
      out_dist[(size_t)q * k + r] = bd;
      pos[bs >> 5]++;
      refresh();
    }
    __syncwarp();
  }
}

}  // namespace cozo

using namespace cozo;

extern "C" int cozo_gpu_topk_merge_dev(const float* dist_dev, const uint32_t* ids_dev, uint32_t n_shards, uint32_t B,
                                       uint32_t k, const uint64_t* shard_offsets_dev, uint64_t* out_ids_dev,
                                       float* out_dist_dev, void* stream) {
  if (!dist_dev || !ids_dev || !shard_offsets_dev || !out_ids_dev || !out_dist_dev)
    return set_error(COZO_GPU_EINVAL, "null buffer");
  if (n_shards == 0 || n_shards > 256) return set_error(COZO_GPU_EINVAL, "n_shards must be in [1,256]");
  if (k == 0) return set_error(COZO_GPU_EINVAL, "k must be positive");
  int rc = ensure_init();
  if (rc) return rc;
  if (B == 0) return 0;
  topk_merge_kernel<<<(B + 3) / 4, 128, 0, (cudaStream_t)stream>>>(
      dist_dev, ids_dev, n_shards, B, k, reinterpret_cast<const unsigned long long*>(shard_offsets_dev),
      reinterpret_cast<unsigned long long*>(out_ids_dev), out_dist_dev);
  COZO_CUDA(cudaGetLastError());
  return 0;
}
