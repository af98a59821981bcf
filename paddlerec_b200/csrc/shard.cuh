// K5 helpers: row-cyclic table sharding (owner = id mod world, local row = id div world).
//
// Behavioural spec: the PSGPU/HeterPS pull/push of the reference's GPUBox trainer
// (tools/static_gpubox_trainer.py:152-159,244-259): keys are sharded over the GPUs of one box,
// each batch exchanges keys -> owners and rows -> requesters.  The exchange itself is an NCCL
// all-to-all issued by the host (torch.distributed); this file produces the bucket order.
#pragma once

#include <cub/device/device_radix_sort.cuh>

#include "common.cuh"

namespace b200rec {

__global__ void shard_keys_kernel(const int64_t* __restrict__ ids, int64_t n, int world, int64_t V,
                                  uint32_t* __restrict__ owner, int32_t* __restrict__ pos,
                                  unsigned long long* __restrict__ counts) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int64_t id = ids[i];
  const bool in_range = (uint64_t)id < (uint64_t)V;
  const uint32_t o = in_range ? (uint32_t)(id % world) : 0u;
  owner[i] = o;
  pos[i] = (int32_t)i;
  // warp-aggregated histogram (integer atomics: order-independent result)
  const unsigned active = __activemask();
  const unsigned peers = __match_any_sync(active, o);
  if ((int)(__ffs(peers) - 1) == (int)(threadIdx.x & 31))
    atomicAdd(counts + o, (unsigned long long)__popc(peers));
}

__global__ void shard_emit_kernel(const int64_t* __restrict__ ids,
                                  const int32_t* __restrict__ sorted_pos, int64_t n, int world,
                                  int64_t V, int64_t* __restrict__ send_ids,
                                  int64_t* __restrict__ perm, int32_t* __restrict__ inv_perm) {
  const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const int32_t p = sorted_pos[k];
  const int64_t id = ids[p];
  const bool in_range = (uint64_t)id < (uint64_t)V;
  send_ids[k] = in_range ? id / world : (int64_t)-1;
  perm[p] = k;
  inv_perm[k] = p;
}

struct ShardPlan {
  size_t off_owner_in, off_owner_out, off_pos_in, off_pos_out, off_cub, cub_bytes, total;
  int bits;
};

static int make_shard_plan(int64_t n, int world, ShardPlan* p) {
  B200_REQUIRE(n >= 0 && n < (int64_t)INT32_MAX, "shard_bucketize: n must fit int32");
  B200_REQUIRE(world >= 1 && world <= 65536, "shard_bucketize: bad world=%d", world);
  int bits = 1;
  while ((1 << bits) < world) ++bits;
  p->bits = bits;
  size_t cub_bytes = 0;
  B200_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, cub_bytes, (const uint32_t*)nullptr,
                                            (uint32_t*)nullptr, (const int32_t*)nullptr,
                                            (int32_t*)nullptr, (int)n, 0, bits));
  p->cub_bytes = cub_bytes;
  size_t off = 0;
  p->off_owner_in = off;  off += align_up((size_t)n * 4, 256);
  p->off_owner_out = off; off += align_up((size_t)n * 4, 256);
  p->off_pos_in = off;    off += align_up((size_t)n * 4, 256);
  p->off_pos_out = off;   off += align_up((size_t)n * 4, 256);
  p->off_cub = off;       off += align_up(cub_bytes, 256);
  p->total = off + 256;
  return B200REC_OK;
}

static int launch_shard_bucketize(const int64_t* ids, int64_t n, int world, int64_t V,
                                  int64_t* send_ids, int64_t* perm, int32_t* inv_perm,
                                  int64_t* counts, void* ws, size_t ws_bytes, cudaStream_t st) {
  ShardPlan p;
  int rc = make_shard_plan(n, world, &p);
  if (rc != B200REC_OK) return rc;
  B200_CUDA(cudaMemsetAsync(counts, 0, (size_t)world * sizeof(int64_t), st));
  if (n == 0) return B200REC_OK;
  if (ws_bytes < p.total) {
    set_error("shard_bucketize: workspace %zu < %zu bytes", ws_bytes, p.total);
    return B200REC_ERR_WORKSPACE;
  }
  unsigned char* base =
      reinterpret_cast<unsigned char*>(align_up((size_t)(uintptr_t)ws, 256));
  uint32_t* owner_in = reinterpret_cast<uint32_t*>(base + p.off_owner_in);
  uint32_t* owner_out = reinterpret_cast<uint32_t*>(base + p.off_owner_out);
  int32_t* pos_in = reinterpret_cast<int32_t*>(base + p.off_pos_in);
  int32_t* pos_out = reinterpret_cast<int32_t*>(base + p.off_pos_out);
  const unsigned grid = (unsigned)((n + 255) / 256);
  shard_keys_kernel<<<grid, 256, 0, st>>>(ids, n, world, V, owner_in, pos_in,
                                          reinterpret_cast<unsigned long long*>(counts));
  B200_LAUNCH_CHECK();
  size_t cub_bytes = p.cub_bytes;
  B200_CUDA(cub::DeviceRadixSort::SortPairs(base + p.off_cub, cub_bytes, owner_in, owner_out,
                                            pos_in, pos_out, (int)n, 0, p.bits, st));
  shard_emit_kernel<<<grid, 256, 0, st>>>(ids, pos_out, n, world, V, send_ids, perm, inv_perm);
  B200_LAUNCH_CHECK();
  return B200REC_OK;
}

// ------------------------------------------------------------------------------------------------
// The exchange itself over NVLink PEER MEMORY (no NCCL call on the data path): every GPU maps the
// receive buffers of its peers (symmetric memory) and the kernels below store straight into them.
//
//   gather_push : owner side of the pull.  The random gather of the rows that peer r asked for and
//                 their transfer are ONE kernel: each row is read from the local shard once and
//                 written once — into r's receive buffer, at the position r's fused K1 expects
//                 (bucket order).  The transfer of a tile overlaps the gather of the next.
//   push_rows   : requester side of the push.  The per-slot gradient rows (bucket order) go into
//                 the owners' receive buffers, aligned with the ids each owner received.
// Segment tables (who asked for what, where it goes) live on the device: they are the outputs of
// the count exchange, so the data path needs no host round trip.  A device-side barrier over the
// same symmetric memory (host: torch's _SymmetricMemory.barrier) publishes the rows.
// Reference behaviour: pull_sparse / push_sparse of tools/static_gpubox_trainer.py:244-259.
constexpr int kPushThreads = 256;
constexpr int kPushRowsPerGroup = 4;
constexpr int kMaxPeers = 16;

struct PeerTable {
  float* base[kMaxPeers];     // receive buffer of every rank, mapped in this process
};

// segment tables on the device: seg_dev [world+1] = rows [seg[r], seg[r+1]) of the local list belong
// to peer r; dst_dev [world] = first row inside peer r's buffer (int64)
__device__ __forceinline__ int peer_of(const int64_t* seg, int world, int64_t i) {
  int r = 0;
#pragma unroll 1
  for (int k = 1; k < world; ++k) r += (i >= seg[k]) ? 1 : 0;
  return r;
}

// Thread mapping: CHUNK-linear.  A row is D/VEC chunks of VEC floats; thread t of a pass handles
// chunk (pass base + t), so consecutive lanes write consecutive 16-byte pieces of the destination
// (rows of one peer are contiguous there: a warp store is one 512-byte run over NVLink) while the
// D/VEC lanes that share a row read its bytes from the shard together.  kPushRowsPerGroup passes are
// in flight per thread.
template <int VEC>
__global__ void __launch_bounds__(kPushThreads)
shard_gather_push_kernel(const float* __restrict__ W, const int64_t* __restrict__ ids,
                         const int64_t* __restrict__ seg_dev, const int64_t* __restrict__ dst_dev,
                         PeerTable peers, int world, int64_t n, int D, int64_t V, int64_t pad,
                         int64_t ldw, int64_t ld_dst) {
  __shared__ int64_t s_seg[kMaxPeers + 1];
  __shared__ int64_t s_dst[kMaxPeers];
  if (threadIdx.x <= world) s_seg[threadIdx.x] = seg_dev[threadIdx.x];
  if (threadIdx.x < world) s_dst[threadIdx.x] = dst_dev[threadIdx.x];
  __syncthreads();
  const int cpr = D / VEC;                                   // chunks per row
  const int64_t m = s_seg[world] < n ? s_seg[world] : n;     // rows actually requested
  const int64_t total = m * cpr;
  const int64_t base = (int64_t)blockIdx.x * kPushThreads * kPushRowsPerGroup + threadIdx.x;
  Vec<VEC> e[kPushRowsPerGroup];
  int64_t row[kPushRowsPerGroup];
  int part[kPushRowsPerGroup];
#pragma unroll
  for (int j = 0; j < kPushRowsPerGroup; ++j) {
    e[j] = vzero<VEC>();
    const int64_t c = base + (int64_t)j * kPushThreads;
    row[j] = c / cpr;
    part[j] = (int)(c - row[j] * cpr);
    if (c < total) {
      const int64_t id = __ldg(ids + row[j]);
      const bool in_range = (uint64_t)id < (uint64_t)V;
      if (in_range && id != pad) e[j] = ld_row<VEC>(W + (size_t)id * ldw + part[j] * VEC);
    }
  }
#pragma unroll
  for (int j = 0; j < kPushRowsPerGroup; ++j) {
    const int64_t c = base + (int64_t)j * kPushThreads;
    if (c < total) {
      const int p = peer_of(s_seg, world, row[j]);
      float* out = peers.base[p] + (size_t)(s_dst[p] + (row[j] - s_seg[p])) * ld_dst + part[j] * VEC;
      st_plain<VEC>(out, e[j]);      // NVLink store (or a local store for p == this rank)
    }
  }
}

template <int VEC>
__global__ void __launch_bounds__(kPushThreads)
shard_push_rows_kernel(const float* __restrict__ rows, int64_t ld,
                       const int64_t* __restrict__ seg_dev, const int64_t* __restrict__ dst_dev,
                       PeerTable peers, int world, int64_t n, int D, int64_t ld_dst) {
  __shared__ int64_t s_seg[kMaxPeers + 1];
  __shared__ int64_t s_dst[kMaxPeers];
  if (threadIdx.x <= world) s_seg[threadIdx.x] = seg_dev[threadIdx.x];
  if (threadIdx.x < world) s_dst[threadIdx.x] = dst_dev[threadIdx.x];
  __syncthreads();
  const int cpr = D / VEC;
  const int64_t m = s_seg[world] < n ? s_seg[world] : n;
  const int64_t total = m * cpr;
  const int64_t base = (int64_t)blockIdx.x * kPushThreads * kPushRowsPerGroup + threadIdx.x;
  Vec<VEC> e[kPushRowsPerGroup];
  int64_t row[kPushRowsPerGroup];
  int part[kPushRowsPerGroup];
#pragma unroll
  for (int j = 0; j < kPushRowsPerGroup; ++j) {
    e[j] = vzero<VEC>();
    const int64_t c = base + (int64_t)j * kPushThreads;
    row[j] = c / cpr;
    part[j] = (int)(c - row[j] * cpr);
    if (c < total) e[j] = ld_row<VEC>(rows + (size_t)row[j] * ld + part[j] * VEC);
  }
#pragma unroll
  for (int j = 0; j < kPushRowsPerGroup; ++j) {
    const int64_t c = base + (int64_t)j * kPushThreads;
    if (c < total) {
      const int p = peer_of(s_seg, world, row[j]);
      float* out = peers.base[p] + (size_t)(s_dst[p] + (row[j] - s_seg[p])) * ld_dst + part[j] * VEC;
      st_plain<VEC>(out, e[j]);
    }
  }
}

// K2 (sparse part) of DeepFM fused with the gradient push of the sharded path.  In the sharded
// backward every position is its own segment (the owner merges duplicates), so the per-slot
// gradient row  [ g2*(S - feat) + dfeat_dnn | g1 | 0.. ]  (models/rank/deepfm/net.py:123-137
// differentiated) is computed here and stored DIRECTLY into the owner's receive buffer over NVLink —
// the [n,G] staging buffer, its write and its re-read by a separate push kernel disappear.
//   feat [B,N,D], S [B,D], dfeat_dnn [B,N,D] or null, gy1/gy2 [B], inv_perm [B*F] = position held by
//   every bucket slot; the row of slot k goes to peer o = owner segment of k, row dst[o] + k - seg[o].
//   Chunk-linear in the DESTINATION (like shard_push_rows): remote stores are contiguous per peer,
//   the scattered side is the local 64-byte reads of feat, which L2 absorbs.
__global__ void __launch_bounds__(kPushThreads)
shard_fm_grads_push_kernel(const float* __restrict__ feat, const float* __restrict__ S,
                           const float* __restrict__ dfeat, const float* __restrict__ gy1,
                           const float* __restrict__ gy2, const int32_t* __restrict__ inv_perm,
                           const int64_t* __restrict__ seg_dev, const int64_t* __restrict__ dst_dev,
                           PeerTable peers, int world, int64_t n, int F, int N, int D, int G,
                           int64_t ld_dst) {
  __shared__ int64_t s_seg[kMaxPeers + 1];
  __shared__ int64_t s_dst[kMaxPeers];
  if (threadIdx.x <= world) s_seg[threadIdx.x] = seg_dev[threadIdx.x];
  if (threadIdx.x < world) s_dst[threadIdx.x] = dst_dev[threadIdx.x];
  __syncthreads();
  const int cpr = G / 4;                 // chunks per gradient row: D/4 embedding chunks, then [g1,0,0,0], zeros
  const int ce = D / 4;
  const int64_t total = n * cpr;
  for (int64_t c = (int64_t)blockIdx.x * kPushThreads + threadIdx.x; c < total;
       c += (int64_t)gridDim.x * kPushThreads) {
    const int64_t k = c / cpr;
    const int part = (int)(c - k * cpr);
    const int64_t p = __ldg(inv_perm + k);
    const int64_t b = p / F;
    const int f = (int)(p - b * F);
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (part < ce) {
      const size_t off = ((size_t)b * N + f) * D + part * 4;
      const float4 e = __ldg(reinterpret_cast<const float4*>(feat + off));
      const float4 s = __ldg(reinterpret_cast<const float4*>(S + (size_t)b * D + part * 4));
      const float g2 = __ldg(gy2 + b);
      float4 d = make_float4(0.f, 0.f, 0.f, 0.f);
      if (dfeat != nullptr) d = __ldg(reinterpret_cast<const float4*>(dfeat + off));
      // same rounding as FmRowContrib::add (embed_fm.cuh): one fma per element
      v = make_float4(fmaf(g2, s.x - e.x, d.x), fmaf(g2, s.y - e.y, d.y), fmaf(g2, s.z - e.z, d.z),
                      fmaf(g2, s.w - e.w, d.w));
    } else if (part == ce) {
      v.x = __ldg(gy1 + b);
    }
    const int o = peer_of(s_seg, world, k);
    float* out = peers.base[o] + (size_t)(s_dst[o] + (k - s_seg[o])) * ld_dst + part * 4;
    *reinterpret_cast<float4*>(out) = v;
  }
}

static int launch_shard_fm_grads_push(const float* feat, const float* S, const float* dfeat,
                                      const float* gy1, const float* gy2, const int32_t* inv_perm,
                                      const int64_t* seg_dev, const int64_t* dst_dev,
                                      const uint64_t* peer_ptrs_host, int64_t ld_dst, int world,
                                      int64_t B, int F, int Dn, int D, int G, cudaStream_t st);

// `align`: bytes of the widest store the kernel issues through the pointers (float4 / float2).
static int fill_peer_table(PeerTable* t, const uint64_t* peer_ptrs_host, int world, int align) {
  B200_REQUIRE(world >= 1 && world <= kMaxPeers, "shard push: world=%d (max %d)", world, kMaxPeers);
  for (int r = 0; r < kMaxPeers; ++r) {
    const uint64_t p = r < world ? peer_ptrs_host[r] : 0;
    B200_REQUIRE(r >= world || p != 0, "shard push: receive buffer of rank %d is NULL", r);
    B200_REQUIRE(p % (uint64_t)align == 0,
                 "shard push: receive buffer of rank %d is not %d-byte aligned", r, align);
    t->base[r] = reinterpret_cast<float*>((uintptr_t)p);
  }
  return B200REC_OK;
}

static int launch_shard_gather_push(const float* W, int64_t ldw, int D, int64_t V, int64_t pad,
                                    const int64_t* ids, const int64_t* seg_dev,
                                    const int64_t* dst_dev, const uint64_t* peer_ptrs_host,
                                    int64_t ld_dst, int world, int64_t n, cudaStream_t st) {
  RowShape rs;
  B200_REQUIRE(pick_row_shape(D, &rs), "shard_gather_push: unsupported D=%d", D);
  PeerTable t;
  int rc = fill_peer_table(&t, peer_ptrs_host, world, rs.vec * 4);
  if (rc != B200REC_OK) return rc;
  B200_REQUIRE(ldw >= D && ld_dst >= D && ldw % rs.vec == 0 && ld_dst % rs.vec == 0,
               "shard_gather_push: bad row strides");
  B200_REQUIRE(reinterpret_cast<uintptr_t>(W) % (rs.vec * 4) == 0,
               "shard_gather_push: shard must be %d-byte aligned", rs.vec * 4);
  if (n == 0) return B200REC_OK;
  const int64_t chunks = n * (D / rs.vec);
  const int64_t per_block = (int64_t)kPushThreads * kPushRowsPerGroup;
  const unsigned grid = (unsigned)((chunks + per_block - 1) / per_block);
  if (rs.vec == 4)
    shard_gather_push_kernel<4><<<grid, kPushThreads, 0, st>>>(W, ids, seg_dev, dst_dev, t, world, n, D,
                                                              V, pad, ldw, ld_dst);
  else if (rs.vec == 2)
    shard_gather_push_kernel<2><<<grid, kPushThreads, 0, st>>>(W, ids, seg_dev, dst_dev, t, world, n, D,
                                                              V, pad, ldw, ld_dst);
  else
    shard_gather_push_kernel<1><<<grid, kPushThreads, 0, st>>>(W, ids, seg_dev, dst_dev, t, world, n, D,
                                                              V, pad, ldw, ld_dst);
  B200_LAUNCH_CHECK();
  return B200REC_OK;
}

static int launch_shard_push_rows(const float* rows, int64_t ld, int D, const int64_t* seg_dev,
                                  const int64_t* dst_dev, const uint64_t* peer_ptrs_host,
                                  int64_t ld_dst, int world, int64_t n, cudaStream_t st) {
  RowShape rs;
  B200_REQUIRE(pick_row_shape(D, &rs), "shard_push_rows: unsupported D=%d", D);
  PeerTable t;
  int rc = fill_peer_table(&t, peer_ptrs_host, world, rs.vec * 4);
  if (rc != B200REC_OK) return rc;
  B200_REQUIRE(ld >= D && ld_dst >= D && ld % rs.vec == 0 && ld_dst % rs.vec == 0,
               "shard_push_rows: bad row strides");
  B200_REQUIRE(reinterpret_cast<uintptr_t>(rows) % (rs.vec * 4) == 0,
               "shard_push_rows: rows must be %d-byte aligned", rs.vec * 4);
  if (n == 0) return B200REC_OK;
  const int64_t chunks = n * (D / rs.vec);
  const int64_t per_block = (int64_t)kPushThreads * kPushRowsPerGroup;
  const unsigned grid = (unsigned)((chunks + per_block - 1) / per_block);
  if (rs.vec == 4)
    shard_push_rows_kernel<4><<<grid, kPushThreads, 0, st>>>(rows, ld, seg_dev, dst_dev, t, world, n, D,
                                                            ld_dst);
  else if (rs.vec == 2)
    shard_push_rows_kernel<2><<<grid, kPushThreads, 0, st>>>(rows, ld, seg_dev, dst_dev, t, world, n, D,
                                                            ld_dst);
  else
    shard_push_rows_kernel<1><<<grid, kPushThreads, 0, st>>>(rows, ld, seg_dev, dst_dev, t, world, n, D,
                                                            ld_dst);
  B200_LAUNCH_CHECK();
  return B200REC_OK;
}

static int launch_shard_fm_grads_push(const float* feat, const float* S, const float* dfeat,
                                      const float* gy1, const float* gy2, const int32_t* inv_perm,
                                      const int64_t* seg_dev, const int64_t* dst_dev,
                                      const uint64_t* peer_ptrs_host, int64_t ld_dst, int world,
                                      int64_t B, int F, int Dn, int D, int G, cudaStream_t st) {
  PeerTable t;
  int rc = fill_peer_table(&t, peer_ptrs_host, world, 16);
  if (rc != B200REC_OK) return rc;
  B200_REQUIRE(D > 0 && D % 4 == 0 && G % 4 == 0 && G >= D + 1 && ld_dst >= G && ld_dst % 4 == 0,
               "shard_fm_grads_push: needs D %% 4 == 0 and G %% 4 == 0, G >= D+1 (D=%d G=%d)", D, G);
  B200_REQUIRE(aligned16(feat) && aligned16(S) && (dfeat == nullptr || aligned16(dfeat)),
               "shard_fm_grads_push: feat / S / dfeat must be 16-byte aligned");
  const int64_t n = B * F;
  if (n == 0) return B200REC_OK;
  const int64_t chunks = n * (G / 4);
  const int64_t want = (chunks + kPushThreads - 1) / kPushThreads;
  const unsigned grid = (unsigned)min(want, (int64_t)sm_count() * 32);
  shard_fm_grads_push_kernel<<<grid, kPushThreads, 0, st>>>(feat, S, dfeat, gy1, gy2, inv_perm, seg_dev,
                                                          dst_dev, t, world, n, F, F + Dn, D, G,
                                                          ld_dst);
  B200_LAUNCH_CHECK();
  return B200REC_OK;
}

}  // namespace b200rec
