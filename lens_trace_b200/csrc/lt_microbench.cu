// lt_microbench.cu -- measured ceilings for the node-fetch side of the roofline (SURVEY.md 8(d): "use measured
// L2/L1 bandwidth, micro-benchmark to add").
//
// A BVH traversal step is a per-lane GATHER: every lane of a warp reads its own 32-byte record with one
// ld.global.nc.v8.f32 (LDG.E.ENL2.256.CONSTANT), at an address that depends on the ray.  The rate the memory
// system sustains for that access pattern is what bounds k_wf_trace / k_flat, not the 128 B/clk/SM a coalesced
// request stream can reach.  This kernel measures it: persistent blocks, every lane issues `ILP` independent
// 32-byte gathers per iteration at pseudo-random records of a table of a given size (21 KB: the Cornell tree's
// copies, L1-resident; 112 MB: the 1 M-triangle traversal set, L2-resident; 0.9 GB: the 5 M-triangle set, HBM).
// `dependent` = the next record index comes out of the record just loaded (a pointer chase per lane, which is what
// one ray does): that is the latency-bound form, reported beside the independent one.
#include "lens_trace_b200.h"
#include "lt_internal.h"

#include <string>

struct LtGatherRec {
  float4 a, b;  // b.w carries the bits of a random "next" record index (dependent mode)
};

__device__ __forceinline__ void mb_ldg256(const void* p, float4& a, float4& b) {
  asm volatile("ld.global.nc.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=f"(a.x), "=f"(a.y), "=f"(a.z), "=f"(a.w), "=f"(b.x), "=f"(b.y), "=f"(b.z), "=f"(b.w)
               : "l"(p));
}

__device__ __forceinline__ unsigned mb_xorshift(unsigned s) {
  s ^= s << 13;
  s ^= s >> 17;
  s ^= s << 5;
  return s;
}

__global__ void k_mb_fill(LtGatherRec* t, unsigned records) {
  unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= records) return;
  unsigned s = mb_xorshift(mb_xorshift(i * 2654435761u + 12345u) + 0x9e3779b9u);
  LtGatherRec r;
  r.a = make_float4(1.0f, 2.0f, 3.0f, 4.0f);
  r.b = make_float4(5.0f, 6.0f, 7.0f, __uint_as_float(__umulhi(s, records)));
  t[i] = r;
}

template <int ILP, bool DEPENDENT>
__global__ void __launch_bounds__(128) k_mb_gather(const LtGatherRec* __restrict__ table, unsigned records, int iters,
                                                   unsigned* __restrict__ sink) {
  unsigned s[ILP], idx[ILP];
  unsigned acc = 0u;
#pragma unroll
  for (int k = 0; k < ILP; k++) {
    s[k] = mb_xorshift((blockIdx.x * blockDim.x + threadIdx.x) * 747796405u + 2891336453u * (unsigned)(k + 1));
    idx[k] = __umulhi(s[k], records);
  }
  for (int it = 0; it < iters; it++) {
#pragma unroll
    for (int k = 0; k < ILP; k++) {
      float4 a, b;
      mb_ldg256(table + idx[k], a, b);
      acc += __float_as_uint(a.x) ^ __float_as_uint(b.z);
      if (DEPENDENT) {  // next record from the loaded word, salted per lane so that chains never merge
        s[k] += 0x9e3779b9u;
        idx[k] = __umulhi(mb_xorshift(__float_as_uint(b.w) ^ s[k]), records);
      } else {
        s[k] = mb_xorshift(s[k]);
        idx[k] = __umulhi(s[k], records);
      }
    }
  }
  if (acc == 0x12345679u) sink[0] = acc;  // keeps the loads alive
}

extern "C" int lt_debug_gather_peak(lt_ctx* ctx, uint64_t table_bytes, int dependent, int ilp, int blocks_per_sm,
                                    int iters, double* out_gbs, double* out_ns_per_load) {
  if (!ctx || ctx->group || table_bytes < sizeof(LtGatherRec) || iters < 1 || blocks_per_sm < 1 || blocks_per_sm > 16)
    return LT_ERR_INVALID;
  if (table_bytes / sizeof(LtGatherRec) > 0xffffffffull) return LT_ERR_INVALID;
  lt_stats st;
  lt_last_stats(ctx, &st);
  if (cudaSetDevice(lt_internal_ctx_device(ctx)) != cudaSuccess) return LT_ERR_CUDA;
  LtStream owned;
  if (owned.create() != cudaSuccess) return LT_ERR_CUDA;
  const cudaStream_t stream = owned.get();
  const unsigned records = (unsigned)(table_bytes / sizeof(LtGatherRec));
  LtBuf<LtGatherRec> tableBuf;
  LtBuf<unsigned> sinkBuf;
  LtEvents ev;
  int rc = LT_OK;
  float best = 0.0f;
  const int blocks = st.sm_count * blocks_per_sm;
  auto launch = [&](int n) {
    const LtGatherRec* table = tableBuf.get();
    unsigned* sink = sinkBuf.get();
    if (dependent) {
      if (ilp >= 4) k_mb_gather<4, true><<<blocks, 128, 0, stream>>>(table, records, n, sink);
      else if (ilp >= 2) k_mb_gather<2, true><<<blocks, 128, 0, stream>>>(table, records, n, sink);
      else k_mb_gather<1, true><<<blocks, 128, 0, stream>>>(table, records, n, sink);
    } else {
      if (ilp >= 4) k_mb_gather<4, false><<<blocks, 128, 0, stream>>>(table, records, n, sink);
      else if (ilp >= 2) k_mb_gather<2, false><<<blocks, 128, 0, stream>>>(table, records, n, sink);
      else k_mb_gather<1, false><<<blocks, 128, 0, stream>>>(table, records, n, sink);
    }
  };
  if (tableBuf.grow(records) != cudaSuccess || sinkBuf.grow(64) != cudaSuccess ||
      ev.grow(2, cudaEventDefault) != cudaSuccess) {
    rc = LT_ERR_CUDA;
  } else {
    k_mb_fill<<<(records + 255) / 256, 256, 0, stream>>>(tableBuf.get(), records);
    launch(iters / 4 > 0 ? iters / 4 : 1);  // warm-up: caches, clocks
    for (int rep = 0; rep < 3 && rc == LT_OK; rep++) {
      cudaEventRecord(ev[0], stream);
      launch(iters);
      cudaEventRecord(ev[1], stream);
      if (cudaStreamSynchronize(stream) != cudaSuccess) {
        rc = LT_ERR_CUDA;
        break;
      }
      float ms = 0.0f;
      cudaEventElapsedTime(&ms, ev[0], ev[1]);
      if (best == 0.0f || ms < best) best = ms;
    }
  }
  const int effIlp = ilp >= 4 ? 4 : (ilp >= 2 ? 2 : 1);
  const double loads = (double)blocks * 128.0 * (double)iters * effIlp;
  if (rc == LT_OK && best > 0.0f) {
    if (out_gbs) *out_gbs = loads * 32.0 / (best * 1e-3) / 1e9;
    if (out_ns_per_load) *out_ns_per_load = best * 1e6 / ((double)iters * effIlp);  // per lane, serial view
  }
  cudaGetLastError();
  return rc;
}
