// Raw item bytes -> database, fused: lib/server/src/db/loading.rs:317-359 update_item_raw (convert_pt_to_poly :278-299,
// pack_ntt_poly :34-41, db.upsert) for a whole group of items in one launch, with no intermediate polynomial buffer.
//
// One CTA (512 threads, 256 per CRT modulus) = one (item, slice) chunk: chunk c of an item is the bytes_per_chunk bytes at
// offset c * bytes_per_chunk of the item's data, zero beyond its length (the zero padding of update_item_raw); byte i is
// plaintext coefficient i, recentred mod q_n, then forward-transformed.  The packed words lo | hi << 32 are placed by the
// layout's store (`Store`, defined next to its layout: mul_kernels.cu, imma_kernels.cu, tc5_kernels.cu), the same helper the
// single-polynomial upsert kernels use.  Items of one launch must be distinct: two CTAs writing one item would race.
#pragma once
#include "kernels.h"

namespace b200pir {
namespace item_write {

struct TwGlobal {            // both halves of the forward table straight from global memory (through L1)
  const Twiddle* p;
  __device__ __forceinline__ Twiddle operator()(int i) const {
    uint2 v = __ldg(reinterpret_cast<const uint2*>(p + i));
    return Twiddle{v.x, v.y};
  }
  __device__ __forceinline__ void load2(int i, Twiddle (&t)[2]) const {
    uint4 v = __ldg(reinterpret_cast<const uint4*>(p + i));
    t[0] = Twiddle{v.x, v.y}; t[1] = Twiddle{v.z, v.w};
  }
  __device__ __forceinline__ void load4(int i, Twiddle (&t)[4]) const {
    uint4 v = __ldg(reinterpret_cast<const uint4*>(p + i)), w = __ldg(reinterpret_cast<const uint4*>(p + i) + 1);
    t[0] = Twiddle{v.x, v.y}; t[1] = Twiddle{v.z, v.w}; t[2] = Twiddle{w.x, w.y}; t[3] = Twiddle{w.z, w.w};
  }
};

// grid = (items, slices), 512 threads
template <typename Store>
__global__ void __launch_bounds__(512)
k_write_items(DevParams P, Store st, const ItemWrite* __restrict__ items, const uint8_t* __restrict__ data, int bpc, uint64_t pt) {
  __shared__ __align__(16) uint32_t smem[2 * NTT_SMEM_WORDS];
  const int n = threadIdx.x >> 8, tid = threadIdx.x & 255;
  const int slice = blockIdx.y;
  const ItemWrite it = items[blockIdx.x];
  const uint32_t q = n ? P.q[1] : P.q[0];
  const Twiddle* fwd = n ? P.fwd[1] : P.fwd[0];
  const int begin = slice * bpc;
  const int have = it.len > (uint32_t)begin ? min((int)(it.len - begin), bpc) : 0;
  const uint8_t* src = data + it.off + begin;
  struct S { __device__ __forceinline__ void operator()() const { __syncthreads(); } };
  uint32_t x[8];
#pragma unroll
  for (int a = 0; a < 8; a++) {
    const int i = a * 256 + tid;
    const uint64_t v = i < have ? (uint64_t)src[i] : 0;
    x[a] = (v > pt / 2) ? (uint32_t)(q - (uint32_t)(pt - v)) : (uint32_t)v;       // recenter_mod, then mod q_n
  }
  uint32_t* mine = smem + n * NTT_SMEM_WORDS;
  ntt_forward_group_lz<NTT_OUT_CANON>(tid, x, mine, TwGlobal{fwd}, TwGlobal{fwd}, q, S());   // inputs canonical
  __syncthreads();                                  // the transform's scratch becomes the [n][z] exchange buffer
#pragma unroll
  for (int k = 0; k < 8; k++) mine[tid * 8 + k] = x[k];
  __syncthreads();
  for (int z = threadIdx.x; z < POLY; z += 512)
    st(slice, (int)it.il, (int)it.j, z, (uint64_t)smem[z] | ((uint64_t)smem[NTT_SMEM_WORDS + z] << 32));
}

template <typename Store>
void launch(const DevParams& P, const Store& st, const ItemWrite* items, int count, int slices, const uint8_t* data, int bpc,
            uint64_t pt, cudaStream_t s) {
  if (count <= 0) return;
  ++g_kernel_launches;
  k_write_items<Store><<<dim3((unsigned)count, (unsigned)slices), 512, 0, s>>>(P, st, items, data, bpc, pt);
}

}  // namespace item_write
}  // namespace b200pir
