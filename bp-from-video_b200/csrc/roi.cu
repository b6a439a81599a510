// F1 — ROI sampling: uint8 HWC-BGR frames -> exact per-ROI (sumB, sumG, sumR, N) and the float64
// sample the reference's np.mean produces (signal_processor.py:176-189).
//
// HBM-bound byte work (no tensor cores).  One thread group (32 / 128 / 256 threads) per ROI.  The
// ROI is walked as a flat list of 16-byte-aligned vectors (rows x vectors-per-row); every thread
// keeps UNROLL independent 128-bit streaming loads in flight.  A vector holds 16 interleaved BGR
// bytes whose channel phase depends on its offset from the row's first pixel; the three channel
// sums come from 12 dp4a against constant 0/1 byte selectors and are rotated by the phase.
// Head/tail vectors are byte-masked.  Integer partials are reduced with warp shuffles (uint64).
#include "common.cuh"

namespace bpv {

struct RoiArgs {
  const uint8_t* frames;
  const uint8_t* const* frame_ptrs;
  long long frame_stride, row_stride;
  int H, W, R, mode;
  long long num_rois;
  const int32_t* boxes;
  unsigned long long* out_sums;
  double* out_value;
};

// Python seq[a:b] normalisation on an axis of length L -> [s, e), e >= s.
__device__ __forceinline__ void py_slice(int a, int b, int L, int& s, int& e) {
  long long aa = a, bb = b;
  if (aa < 0) { aa += L; if (aa < 0) aa = 0; } else if (aa > L) aa = L;
  if (bb < 0) { bb += L; if (bb < 0) bb = 0; } else if (bb > L) bb = L;
  if (bb < aa) bb = aa;
  s = (int)aa; e = (int)bb;
}

__device__ __forceinline__ uint4 ld_stream_v4(const void* p) {
  uint4 v;
  asm volatile("ld.global.nc.L1::no_allocate.L2::64B.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
  return v;
}

// HOST: frames in pinned host memory, read with plain ld.global (see launch_rows); else ld_stream_v4
template <bool HOST>
__device__ __forceinline__ uint4 ld_row_v4(const void* p) {
  if (!HOST) return ld_stream_v4(p);
  uint4 v;
  asm volatile("ld.global.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p));
  return v;
}

// bytes [l, h) of a 32-bit word (l, h may lie outside 0..4)
__device__ __forceinline__ uint32_t byte_mask(int l, int h) {
  uint32_t lo = l <= 0 ? 0xffffffffu : (l >= 4 ? 0u : 0xffffffffu << (8 * l));
  uint32_t hi = h >= 4 ? 0xffffffffu : (h <= 0 ? 0u : 0xffffffffu >> (8 * (4 - h)));
  return lo & hi;
}

// selector q keeps byte b of the vector iff (q + b) % 3 == 0
__device__ __forceinline__ void channel_sums(const uint4& v, uint32_t& s0, uint32_t& s1, uint32_t& s2) {
  s0 = __dp4a(v.x, 0x01000001u, __dp4a(v.y, 0x00010000u, __dp4a(v.z, 0x00000100u, __dp4a(v.w, 0x01000001u, 0u))));
  s1 = __dp4a(v.x, 0x00010000u, __dp4a(v.y, 0x00000100u, __dp4a(v.z, 0x01000001u, __dp4a(v.w, 0x00010000u, 0u))));
  s2 = __dp4a(v.x, 0x00000100u, __dp4a(v.y, 0x01000001u, __dp4a(v.z, 0x00010000u, __dp4a(v.w, 0x00000100u, 0u))));
}

template <int GROUP, int UNROLL>
__global__ void __launch_bounds__(256) roi_sample_kernel(const RoiArgs a) {
  constexpr int GROUPS_PER_BLOCK = 256 / GROUP;
  constexpr int WARPS_PER_GROUP = GROUP / 32;
  const int grp = threadIdx.x / GROUP, gt = threadIdx.x % GROUP;
  const long long roi = (long long)blockIdx.x * GROUPS_PER_BLOCK + grp;
  const bool live = roi < a.num_rois;

  int xs = 0, xe = 0, ys = 0, ye = 0;
  bool has_box = false;
  const uint8_t* base = nullptr;
  if (live) {
    const int4 b = __ldg(reinterpret_cast<const int4*>(a.boxes) + roi);
    has_box = b.x != BPV_NO_BOX;
    if (has_box) {
      py_slice(b.x, b.z, a.W, xs, xe);
      py_slice(b.y, b.w, a.H, ys, ye);
      const long long f = roi / a.R;
      const uint8_t* fp = a.frame_ptrs ? a.frame_ptrs[f] : a.frames + f * a.frame_stride;
      base = fp + (long long)ys * a.row_stride + (long long)xs * 3;
    }
  }
  const int nrows = ye - ys, row_bytes = (xe - xs) * 3;
  uint32_t sB = 0, sG = 0, sR = 0;
  if (nrows > 0 && row_bytes > 0) {
    const uint32_t vpr = (uint32_t)(row_bytes + 14) / 16u + 1u;  // most aligned vectors a row can touch
    const uint32_t total = (uint32_t)nrows * vpr;
    uint32_t row = (uint32_t)gt / vpr, v = (uint32_t)gt % vpr;
    const uint32_t dq = (uint32_t)GROUP / vpr, dr = (uint32_t)GROUP % vpr;
    for (uint32_t idx = gt; idx < total; idx += GROUP * UNROLL) {
      uint4 d[UNROLL];
      int lo[UNROLL], hi[UNROLL], ph[UNROLL];
#pragma unroll
      for (int u = 0; u < UNROLL; ++u) {
        hi[u] = 0;
        if (idx + u * GROUP < total) {
          const uintptr_t a0 = reinterpret_cast<uintptr_t>(base) + (uintptr_t)row * (uintptr_t)a.row_stride;
          const int off = (int)(a0 & 15);
          const int rel = 16 * (int)v - off;  // vector byte 0 relative to the row's first pixel byte
          const int e = row_bytes - rel;      // bytes of the row at/after vector byte 0
          if (e > 0) {
            lo[u] = rel < 0 ? -rel : 0;
            hi[u] = e < 16 ? e : 16;
            ph[u] = (rel + 15) % 3;
            d[u] = ld_stream_v4(reinterpret_cast<const void*>(a0 + rel));
          }
        }
        row += dq; v += dr;
        if (v >= vpr) { v -= vpr; ++row; }
      }
#pragma unroll
      for (int u = 0; u < UNROLL; ++u) {
        if (hi[u] > 0) {
          uint4 w = d[u];
          if (lo[u] > 0 || hi[u] < 16) {
            w.x &= byte_mask(lo[u], hi[u]);
            w.y &= byte_mask(lo[u] - 4, hi[u] - 4);
            w.z &= byte_mask(lo[u] - 8, hi[u] - 8);
            w.w &= byte_mask(lo[u] - 12, hi[u] - 12);
          }
          uint32_t s0, s1, s2;
          channel_sums(w, s0, s1, s2);
          const int p = ph[u];
          sB += p == 0 ? s0 : (p == 1 ? s1 : s2);
          sG += p == 0 ? s2 : (p == 1 ? s0 : s1);
          sR += p == 0 ? s1 : (p == 1 ? s2 : s0);
        }
      }
    }
  }

  unsigned long long tB = warp_sum_u64(sB), tG = warp_sum_u64(sG), tR = warp_sum_u64(sR);
  if (WARPS_PER_GROUP > 1) {
    __shared__ unsigned long long part[8][3];
    const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) { part[wid][0] = tB; part[wid][1] = tG; part[wid][2] = tR; }
    __syncthreads();
    if (gt == 0) {
      tB = tG = tR = 0;
      const int w0 = grp * WARPS_PER_GROUP;
#pragma unroll
      for (int w = 0; w < WARPS_PER_GROUP; ++w) { tB += part[w0 + w][0]; tG += part[w0 + w][1]; tR += part[w0 + w][2]; }
    }
  }
  if (live && gt == 0) {
    const unsigned long long N = (unsigned long long)(nrows > 0 ? nrows : 0) * (unsigned long long)(xe - xs);
    if (a.out_sums) {
      ulonglong4 o; o.x = tB; o.y = tG; o.z = tR; o.w = N;
      *reinterpret_cast<ulonglong4*>(a.out_sums + 4 * roi) = o;
    }
    double val;
    if (!has_box || N == 0) val = nan_f64();
    else if (a.mode == BPV_GREEN) val = (double)tG / (double)N;
    else val = (double)(2 * (long long)tG - (long long)tB - (long long)tR + 2 * (long long)N) / (double)(4 * N);
    a.out_value[roi] = val;
  }
}


// ---------------------------------------------------------------------------------------------
// Fast path (row_stride % 16 == 0, i.e. every standard frame width): the 16-byte alignment offset
// of a ROI row is the same for all rows, so a thread that always visits the same vector column
// has a loop-invariant channel phase and head/tail mask.  Both are folded into per-thread dp4a
// selector registers before the row loop; the loop body is pointer bump + LDG.128 + 8 (12) dp4a.
// Threads are laid out (rows_per_step x vectors_per_row) over the group.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t sel_word(int q, int j) {  // selector q, word j (see channel_sums)
  const int k = (q + j) % 3;
  return k == 0 ? 0x01000001u : (k == 1 ? 0x00010000u : 0x00000100u);
}

template <int GROUP, bool WANT_SUMS, bool HOST>
__global__ void __launch_bounds__(256, 4) roi_rows_kernel(const RoiArgs a) {
  constexpr int UNROLL = 4;
  constexpr int GROUPS_PER_BLOCK = 256 / GROUP;
  constexpr int WARPS_PER_GROUP = GROUP / 32;
  const int grp = threadIdx.x / GROUP, gt = threadIdx.x % GROUP;
  const long long roi = (long long)blockIdx.x * GROUPS_PER_BLOCK + grp;
  const bool live = roi < a.num_rois;

  int xs = 0, xe = 0, ys = 0, ye = 0;
  bool has_box = false;
  uintptr_t base = 0;
  if (live) {
    const int4 b = __ldg(reinterpret_cast<const int4*>(a.boxes) + roi);
    has_box = b.x != BPV_NO_BOX;
    if (has_box) {
      py_slice(b.x, b.z, a.W, xs, xe);
      py_slice(b.y, b.w, a.H, ys, ye);
      const long long f = roi / a.R;
      const uint8_t* fp = a.frame_ptrs ? a.frame_ptrs[f] : a.frames + f * a.frame_stride;
      base = reinterpret_cast<uintptr_t>(fp) + (uintptr_t)((long long)ys * a.row_stride + (long long)xs * 3);
    }
  }
  const int nrows = ye - ys, row_bytes = (xe - xs) * 3;
  uint32_t sG = 0, sT = 0, sB = 0;  // per-thread partial sums: green, all bytes, blue
  if (nrows > 0 && row_bytes > 0) {
    const int off = (int)(base & 15);
    const int vpr = (off + row_bytes + 15) >> 4;  // aligned vectors per row (same for every row)
    int rps, r0, v0;
    if (vpr >= GROUP) { rps = 1; r0 = 0; v0 = gt; }
    else { rps = GROUP / vpr; r0 = gt / vpr; v0 = gt - r0 * vpr; if (r0 >= rps) v0 = vpr; }
    const long long step = (long long)rps * a.row_stride;
    for (int v = v0; v < vpr; v += GROUP) {
      const int rel = 16 * v - off;
      const int lo = rel < 0 ? -rel : 0;
      const int e = row_bytes - rel;
      const int hi = e < 16 ? e : 16;
      const int ph = (rel + 15) % 3;
      uint32_t cT[4], cG[4], cB[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const uint32_t m = byte_mask(lo - 4 * j, hi - 4 * j);
        cT[j] = m & 0x01010101u;
        cG[j] = m & sel_word((ph + 2) % 3, j);
        cB[j] = m & sel_word(ph, j);
      }
      const uint8_t* p = reinterpret_cast<const uint8_t*>(base - off) + (long long)r0 * a.row_stride + 16 * v;
      for (int r = r0; r < nrows; r += rps * UNROLL) {
        uint4 d[UNROLL];
#pragma unroll
        for (int u = 0; u < UNROLL; ++u)
          if (r + u * rps < nrows) d[u] = ld_row_v4<HOST>(p + u * step);
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) {
          if (r + u * rps < nrows) {
            sT = __dp4a(d[u].x, cT[0], __dp4a(d[u].y, cT[1], __dp4a(d[u].z, cT[2], __dp4a(d[u].w, cT[3], sT))));
            sG = __dp4a(d[u].x, cG[0], __dp4a(d[u].y, cG[1], __dp4a(d[u].z, cG[2], __dp4a(d[u].w, cG[3], sG))));
            if (WANT_SUMS)
              sB = __dp4a(d[u].x, cB[0], __dp4a(d[u].y, cB[1], __dp4a(d[u].z, cB[2], __dp4a(d[u].w, cB[3], sB))));
          }
        }
        p += UNROLL * step;
      }
    }
  }

  const unsigned long long N = (unsigned long long)(nrows > 0 ? nrows : 0) * (unsigned long long)(xe - xs);
  unsigned long long tG, tT, tB = 0;
  // 32-bit shuffles are enough while 3*255*N fits (group-uniform choice: N is per ROI; a warp never
  // straddles ROIs with GROUP >= 32)
  if (N < 5600000ull) {
    tG = warp_sum<uint32_t>(sG); tT = warp_sum<uint32_t>(sT);
    if (WANT_SUMS) tB = warp_sum<uint32_t>(sB);
  } else {
    tG = warp_sum_u64(sG); tT = warp_sum_u64(sT);
    if (WANT_SUMS) tB = warp_sum_u64(sB);
  }
  if (WARPS_PER_GROUP > 1) {
    __shared__ unsigned long long part[8][3];
    const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) { part[wid][0] = tG; part[wid][1] = tT; part[wid][2] = tB; }
    __syncthreads();
    if (gt == 0) {
      tG = tT = tB = 0;
      const int w0 = grp * WARPS_PER_GROUP;
#pragma unroll
      for (int w = 0; w < WARPS_PER_GROUP; ++w) { tG += part[w0 + w][0]; tT += part[w0 + w][1]; tB += part[w0 + w][2]; }
    }
  }
  if (live && gt == 0) {
    if (WANT_SUMS) {
      ulonglong4 o; o.x = tB; o.y = tG; o.z = tT - tG - tB; o.w = N;
      *reinterpret_cast<ulonglong4*>(a.out_sums + 4 * roi) = o;
    }
    double val;
    if (!has_box || N == 0) val = nan_f64();
    else if (a.mode == BPV_GREEN) val = (double)tG / (double)N;
    // 2G - B - R + 2N = 3G - (B+G+R) + 2N
    else val = (double)(3 * (long long)tG - (long long)tT + 2 * (long long)N) / (double)(4 * N);
    a.out_value[roi] = val;
  }
}

// ---------------------------------------------------------------------------------------------
// Shared-memory staged fast path: one ROI per CTA.  The register path above can keep at most
// UNROLL x 16 B per thread in flight (64 KB per SM at 4 CTAs); staging decouples the bytes in flight
// from the register file, so a CTA has its whole ROI tile (or a K-row-step batch of it) outstanding.
// Every thread issues up to K 16-byte cp.async (LDGSTS, L2::64B fill) into its OWN slots and reads
// the same slots back -> no CTA barrier at all, only cp.async.wait_all.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// 16-byte LDGSTS with a 64-byte L2 fill granule and an evict-first L2 policy: ROI bytes are read exactly once, so they
// must not push the window pipeline's L2-resident scratch (proc_x / proc_y, ~80 MB, rewritten every step) out to DRAM.
__device__ __forceinline__ unsigned long long l2_evict_first_policy() {
  unsigned long long pol;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ void cp_async16_64B(uint32_t dst, const void* src, unsigned long long pol) {
  asm volatile("cp.async.cg.shared.global.L2::cache_hint.L2::64B [%0], [%1], 16, %2;" :: "r"(dst), "l"(src), "l"(pol) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() {
  asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;" ::: "memory");
}
__device__ __forceinline__ uint4 lds128(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr) : "memory");
  return v;
}

template <int THREADS, int K, bool WANT_SUMS>
__global__ void __launch_bounds__(THREADS) roi_staged_kernel(const RoiArgs a) {
  extern __shared__ __align__(128) uint8_t stage[];
  constexpr int WARPS = THREADS / 32;
  const int gt = threadIdx.x;
  const long long roi = blockIdx.x;

  int xs = 0, xe = 0, ys = 0, ye = 0;
  bool has_box = false;
  uintptr_t base = 0;
  {
    const int4 b = __ldg(reinterpret_cast<const int4*>(a.boxes) + roi);
    has_box = b.x != BPV_NO_BOX;
    if (has_box) {
      py_slice(b.x, b.z, a.W, xs, xe);
      py_slice(b.y, b.w, a.H, ys, ye);
      const long long f = roi / a.R;
      const uint8_t* fp = a.frame_ptrs ? a.frame_ptrs[f] : a.frames + f * a.frame_stride;
      base = reinterpret_cast<uintptr_t>(fp) + (uintptr_t)((long long)ys * a.row_stride + (long long)xs * 3);
    }
  }
  const int nrows = ye - ys, row_bytes = (xe - xs) * 3;
  uint32_t sG = 0, sT = 0, sB = 0;
  if (nrows > 0 && row_bytes > 0) {
    const int off = (int)(base & 15);
    const int vpr = (off + row_bytes + 15) >> 4;
    int rps, r0, v0;
    if (vpr >= THREADS) { rps = 1; r0 = 0; v0 = gt; }
    else { rps = THREADS / vpr; r0 = gt / vpr; v0 = gt - r0 * vpr; if (r0 >= rps) v0 = vpr; }
    const long long step = (long long)rps * a.row_stride;
    const uint32_t slot0 = smem_u32(stage) + 16u * (uint32_t)gt;
    const unsigned long long pol = l2_evict_first_policy();
    for (int v = v0; v < vpr; v += THREADS) {
      const int rel = 16 * v - off;
      const int lo = rel < 0 ? -rel : 0;
      const int e = row_bytes - rel;
      const int hi = e < 16 ? e : 16;
      const int ph = (rel + 15) % 3;
      uint32_t cT[4], cG[4], cB[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const uint32_t m = byte_mask(lo - 4 * j, hi - 4 * j);
        cT[j] = m & 0x01010101u;
        cG[j] = m & sel_word((ph + 2) % 3, j);
        cB[j] = m & sel_word(ph, j);
      }
      const uint8_t* p = reinterpret_cast<const uint8_t*>(base - off) + (long long)r0 * a.row_stride + 16 * v;
      for (int r = r0; r < nrows; r += rps * K) {
#pragma unroll
        for (int u = 0; u < K; ++u)
          if (r + u * rps < nrows) cp_async16_64B(slot0 + (uint32_t)(u * THREADS * 16), p + u * step, pol);
        cp_async_wait_all();
#pragma unroll
        for (int u = 0; u < K; ++u) {
          if (r + u * rps < nrows) {
            const uint4 d = lds128(slot0 + (uint32_t)(u * THREADS * 16));
            sT = __dp4a(d.x, cT[0], __dp4a(d.y, cT[1], __dp4a(d.z, cT[2], __dp4a(d.w, cT[3], sT))));
            sG = __dp4a(d.x, cG[0], __dp4a(d.y, cG[1], __dp4a(d.z, cG[2], __dp4a(d.w, cG[3], sG))));
            if (WANT_SUMS)
              sB = __dp4a(d.x, cB[0], __dp4a(d.y, cB[1], __dp4a(d.z, cB[2], __dp4a(d.w, cB[3], sB))));
          }
        }
        p += K * step;
      }
    }
  }

  const unsigned long long N = (unsigned long long)(nrows > 0 ? nrows : 0) * (unsigned long long)(xe - xs);
  unsigned long long tG, tT, tB = 0;
  if (N < 5600000ull) {
    tG = warp_sum<uint32_t>(sG); tT = warp_sum<uint32_t>(sT);
    if (WANT_SUMS) tB = warp_sum<uint32_t>(sB);
  } else {
    tG = warp_sum_u64(sG); tT = warp_sum_u64(sT);
    if (WANT_SUMS) tB = warp_sum_u64(sB);
  }
  if (WARPS > 1) {
    __shared__ unsigned long long part[WARPS][3];
    const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) { part[wid][0] = tG; part[wid][1] = tT; part[wid][2] = tB; }
    __syncthreads();
    if (gt == 0) {
      tG = tT = tB = 0;
#pragma unroll
      for (int w = 0; w < WARPS; ++w) { tG += part[w][0]; tT += part[w][1]; tB += part[w][2]; }
    }
  }
  if (gt == 0) {
    if (WANT_SUMS) {
      ulonglong4 o; o.x = tB; o.y = tG; o.z = tT - tG - tB; o.w = N;
      *reinterpret_cast<ulonglong4*>(a.out_sums + 4 * roi) = o;
    }
    double val;
    if (!has_box || N == 0) val = nan_f64();
    else if (a.mode == BPV_GREEN) val = (double)tG / (double)N;
    else val = (double)(3 * (long long)tG - (long long)tT + 2 * (long long)N) / (double)(4 * N);
    a.out_value[roi] = val;
  }
}

template <int THREADS, int K>
static void launch_staged(const RoiArgs& a, cudaStream_t st) {
  const int smem = THREADS * K * 16;
  auto k1 = roi_staged_kernel<THREADS, K, true>;
  auto k0 = roi_staged_kernel<THREADS, K, false>;
  // a failed opt-in is not fatal here: the launch below then fails and check_launch() reports it
  (void)ensure_dyn_smem((const void*)k1, 200 * 1024, true);
  (void)ensure_dyn_smem((const void*)k0, 200 * 1024, true);
  if (a.out_sums) k1<<<(unsigned)a.num_rois, THREADS, smem, st>>>(a);
  else k0<<<(unsigned)a.num_rois, THREADS, smem, st>>>(a);
}

template <int GROUP, bool HOST>
static void launch_rows(const RoiArgs& a, unsigned grid, cudaStream_t st) {
  // Device frames: ld.global.nc.L1::no_allocate.L2::64B: the default L2 fill granule on B200 is the whole
  // 128-byte line; asking for 64 B cuts the DRAM over-fetch around short unaligned ROI rows from 1.50x
  // to 1.17x of the algorithmic bytes (ncu dram__bytes_read, profiles/r1a_roi_l2_fill_probe.txt).
  // HOST: plain ld.global, for frames in pinned host memory: over PCIe the 128-byte requests move
  // 32.8 GB/s of ROI bytes (49 GB/s on the wire) against 19.9 GB/s with 64-byte requests
  // (profiles/r1e_roi_host_variants.txt).
  // Host frames are PCIe-bound (one 256-thread CTA per SM already keeps 2.4 MB of reads in flight): an unused dynamic
  // shared-memory request caps the kernel at one CTA per SM, so the window pipeline of the previous batch can run
  // beside it on another stream instead of queueing behind a machine-filling F1 grid.
  size_t smem = 0;
  if (HOST) {
    smem = 120 * 1024;
    (void)ensure_dyn_smem((const void*)roi_rows_kernel<GROUP, true, HOST>, smem);
    (void)ensure_dyn_smem((const void*)roi_rows_kernel<GROUP, false, HOST>, smem);
  }
  if (a.out_sums) roi_rows_kernel<GROUP, true, HOST><<<grid, 256, smem, st>>>(a);
  else roi_rows_kernel<GROUP, false, HOST><<<grid, 256, smem, st>>>(a);
}

// ---------------------------------------------------------------------------------------------
// F1 on NV12 frames (SURVEY.md 8f row 2): decoders (NVDEC, V4L2) hand out NV12 — a full-resolution Y plane followed
// by a half-resolution interleaved UV plane — and the reference only ever sees the BGR frame cv2.VideoCapture makes
// of it (video_reader.py:93).  Sampling the ROI straight from the NV12 planes reads 1.5 bytes per pixel instead of 3
// and never materialises the BGR frame; the per-pixel conversion is OpenCV's integer BT.601 (cvtColor
// COLOR_YUV2BGR_NV12, imgproc/src/color_yuv.simd.hpp: 20-bit fixed point, limited-range Y), so the sums are those of
// the BGR frame the reference would have sampled, bit for bit.
// One 128-thread CTA per ROI, threads laid out rows x 16-pixel vector columns as in the BGR kernels.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ int sat_u8(int v) {
  int r;
  asm("cvt.sat.u8.s32 %0, %1;" : "=r"(r) : "r"(v));           // one instruction instead of a min / max pair
  return r;
}

// Byte loads, for planes that are not 16-byte aligned (aligned ones go to roi_nv12_vec_kernel below); ALL = false (GREEN
// without sums): only the green channel is converted.  Thread layout as the BGR kernels: rows x 16-pixel vector columns, so
// a thread's column — and with it the mask of its pixels that lie inside [xs, xe) — is loop invariant.
template <bool WANT_SUMS, bool ALL>
__global__ void __launch_bounds__(128) roi_nv12_kernel(const uint8_t* __restrict__ frames, long long frame_stride, long long pitch,
                                                       int H, int W, int R, int mode, long long num_rois,
                                                       const int32_t* __restrict__ boxes,
                                                       unsigned long long* __restrict__ out_sums, double* __restrict__ out_value) {
  constexpr int THREADS = 128, WARPS = THREADS / 32;
  const int gt = threadIdx.x;
  const long long roi = blockIdx.x;
  int xs = 0, xe = 0, ys = 0, ye = 0;
  bool has_box = false;
  const int4 b = __ldg(reinterpret_cast<const int4*>(boxes) + roi);
  has_box = b.x != BPV_NO_BOX;
  if (has_box) { py_slice(b.x, b.z, W, xs, xe); py_slice(b.y, b.w, H, ys, ye); }
  const uint8_t* yp = frames + (roi / R) * frame_stride;
  const uint8_t* uvp = yp + (long long)H * pitch;
  const int nrows = ye - ys, ncols = xe - xs;
  uint32_t sB = 0, sG = 0, sR = 0;
  if (nrows > 0 && ncols > 0) {
    const int x0 = xs & ~15;                                  // 16-pixel aligned vector columns (x0 even: UV pairs intact)
    const int vpr = (xe - x0 + 15) >> 4;
    // the row unit is a CHROMA row: the two luma rows 2c and 2c + 1 share its UV samples, so their chroma terms are
    // computed once and the two Y vectors are independent loads in flight together
    const int c_lo = ys >> 1, c_hi = (ye - 1) >> 1, ncr = c_hi - c_lo + 1;
    int rps, r0, v0;
    if (vpr >= THREADS) { rps = 1; r0 = 0; v0 = gt; }
    else { rps = THREADS / vpr; r0 = gt / vpr; v0 = gt - r0 * vpr; if (r0 >= rps) v0 = vpr; }
    for (int v = v0; v < vpr; v += THREADS) {
      const int xv = x0 + 16 * v;
      unsigned inm = 0;                                       // pixels of the group inside [xs, xe)
#pragma unroll
      for (int e = 0; e < 16; ++e) inm |= (xv + e >= xs && xv + e < xe) ? 1u << e : 0u;
      for (int r = r0; r < ncr; r += rps) {
        const int cy = c_lo + r;
        const bool row_on[2] = {2 * cy >= ys, 2 * cy + 1 < ye};
        const uint8_t* yrow = yp + (long long)(2 * cy) * pitch + xv;
        const uint8_t* uvrow = uvp + (long long)cy * pitch + xv;
        uint32_t yw[2][4], cw[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          yw[0][j] = yw[1][j] = cw[j] = 0;
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const int e = 4 * j + k;
            if (inm >> e & 1) {
              if (row_on[0]) yw[0][j] |= (uint32_t)yrow[e] << (8 * k);
              if (row_on[1]) yw[1][j] |= (uint32_t)yrow[pitch + e] << (8 * k);
            }
            if (inm >> (e & ~1) & 3) cw[j] |= (uint32_t)uvrow[e] << (8 * k);   // a pair's U and V when either pixel is in range
          }
        }
        // (a predicate-free copy of this body for interior vectors was measured: 217 us against 144 us per 8192 frames —
        // the doubled code costs more than the skipped tests save; profiles/r2h_ingest.txt)
#pragma unroll
        for (int pr = 0; pr < 8; ++pr) {
          if (!(inm >> (2 * pr) & 3u)) continue;
          const uint32_t c2 = cw[pr >> 1] >> (16 * (pr & 1));
          const int uu = (int)(c2 & 0xffu) - 128, vv = (int)(c2 >> 8 & 0xffu) - 128;
          const int guv = (1 << 19) - 852492 * vv - 409993 * uu;
          const int ruv = (1 << 19) + 1673527 * vv;
          const int buv = (1 << 19) + 2116026 * uu;
#pragma unroll
          for (int ro = 0; ro < 2; ++ro) {
            if (!row_on[ro]) continue;
#pragma unroll
            for (int e = 0; e < 2; ++e) {
              const int px = 2 * pr + e;
              if (!(inm >> px & 1u)) continue;
              const int yy = (int)(yw[ro][px >> 2] >> (8 * (px & 3)) & 0xffu) - 16;
              const int yc = (yy > 0 ? yy : 0) * 1220542;
              sG += (uint32_t)sat_u8((yc + guv) >> 20);
              if (ALL) {
                sR += (uint32_t)sat_u8((yc + ruv) >> 20);
                sB += (uint32_t)sat_u8((yc + buv) >> 20);
              }
            }
          }
        }
      }
    }
  }
  const unsigned long long N = (unsigned long long)(nrows > 0 ? nrows : 0) * (unsigned long long)(ncols > 0 ? ncols : 0);
  unsigned long long tB = warp_sum_u64(sB), tG = warp_sum_u64(sG), tR = warp_sum_u64(sR);
  __shared__ unsigned long long part[WARPS][3];
  const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) { part[wid][0] = tB; part[wid][1] = tG; part[wid][2] = tR; }
  __syncthreads();
  if (gt == 0) {
    tB = tG = tR = 0;
#pragma unroll
    for (int w = 0; w < WARPS; ++w) { tB += part[w][0]; tG += part[w][1]; tR += part[w][2]; }
    if (WANT_SUMS) {
      ulonglong4 o; o.x = tB; o.y = tG; o.z = tR; o.w = N;
      *reinterpret_cast<ulonglong4*>(out_sums + 4 * roi) = o;
    }
    double val;
    if (!has_box || N == 0) val = nan_f64();
    else if (mode == BPV_GREEN) val = (double)tG / (double)N;
    else val = (double)(2 * (long long)tG - (long long)tB - (long long)tR + 2 * (long long)N) / (double)(4 * N);
    out_value[roi] = val;
  }
}

// Branch-free body for aligned planes (frame base, frame stride and pitch multiples of 16: every decoder surface).  The
// kernel above tests the ROI's edges per pixel (914 instructions per 32 pixels, ~120 of them branches and predicates); here
//   * the column mask of a thread's 16-pixel group is loop invariant and is folded into the accumulation as a 0 / 1
//     multiplier (sum = value * m + sum is one IMAD, the same cost as the plain add),
//   * the two luma rows of a chroma row accumulate into row-local partial sums that enter the totals with a 0 / 1 row weight
//     (only the first / last chroma row of a ROI can have a luma row outside it), so nothing in the loop branches,
//   * the constant offsets (Y - 16, U - 128, V - 128) are folded into the per-pair chroma terms:
//       c = max(Y, 16) * CY + [2^19 - 16 CY + k_u (U - 128) + k_v (V - 128)]        (one IMAD per channel and pixel)
// Same integer arithmetic as OpenCV's (20-bit fixed point, >> 20, saturate), bit for bit.
// d = { c[15:0], sat_u8(a), sat_u8(b) }: two saturating conversions and the packing in ONE instruction (I2IP.U8.S32.SAT)
__device__ __forceinline__ uint32_t pack_sat_u8(int a, int b, uint32_t c) {
  uint32_t d;
  asm("cvt.pack.sat.u8.s32.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
  return d;
}

template <bool WANT_SUMS, bool ALL>
__global__ void __launch_bounds__(128) roi_nv12_vec_kernel(const uint8_t* __restrict__ frames, long long frame_stride, long long pitch,
                                                           int H, int W, int R, int mode, long long num_rois,
                                                           const int32_t* __restrict__ boxes,
                                                           unsigned long long* __restrict__ out_sums, double* __restrict__ out_value) {
  constexpr int THREADS = 128, WARPS = THREADS / 32;
  constexpr int CY = 1220542, CVR = 1673527, CVG = -852492, CUG = -409993, CUB = 2116026;
  const int gt = threadIdx.x;
  const long long roi = blockIdx.x;
  int xs = 0, xe = 0, ys = 0, ye = 0;
  bool has_box = false;
  const int4 b = __ldg(reinterpret_cast<const int4*>(boxes) + roi);
  has_box = b.x != BPV_NO_BOX;
  if (has_box) { py_slice(b.x, b.z, W, xs, xe); py_slice(b.y, b.w, H, ys, ye); }
  const uint8_t* yp = frames + (roi / R) * frame_stride;
  const uint8_t* uvp = yp + (long long)H * pitch;
  const int nrows = ye - ys, ncols = xe - xs;
  uint32_t sB = 0, sG = 0, sR = 0;                           // !WANT_SUMS: sB carries B + R (all the chrominance formula needs)
  if (nrows > 0 && ncols > 0) {
    const int x0 = xs & ~15;
    const int vpr = (xe - x0 + 15) >> 4;
    const int c_lo = ys >> 1, c_hi = (ye - 1) >> 1, ncr = c_hi - c_lo + 1;
    int rps, r0, v0;
    if (vpr >= THREADS) { rps = 1; r0 = 0; v0 = gt; }
    else { rps = THREADS / vpr; r0 = gt / vpr; v0 = gt - r0 * vpr; if (r0 >= rps) v0 = vpr; }
    for (int v = v0; v < vpr; v += THREADS) {
      const int xv = x0 + 16 * v;
      // per pixel PAIR (2 pr, 2 pr + 1): byte selectors for the packed saturated values — the values of a pair are summed by
      // one dp4a against the pair's 0 / 1 byte mask, so the ROI's left / right edge costs nothing in the loop
      uint32_t m2[8], m4[8];                                   // {e0, e1} in bytes {1, 0} / {e0, e0, e1, e1} in bytes {3, 2, 1, 0}
#pragma unroll
      for (int pr = 0; pr < 8; ++pr) {
        const uint32_t a0 = (xv + 2 * pr >= xs && xv + 2 * pr < xe) ? 1u : 0u, a1 = (xv + 2 * pr + 1 >= xs && xv + 2 * pr + 1 < xe) ? 1u : 0u;
        m2[pr] = a0 << 8 | a1;
        m4[pr] = a0 * 0x01010000u | a1 * 0x00000101u;
        asm volatile("" : "+r"(m2[pr]), "+r"(m4[pr]));         // opaque registers: the compiler must not re-derive them per row
      }
      for (int r = r0; r < ncr; r += rps) {
        const int cy = c_lo + r;
        uint32_t w0 = 2 * cy >= ys ? 1u : 0u, w1 = 2 * cy + 1 < ye ? 1u : 0u;
        asm volatile("" : "+r"(w0), "+r"(w1));
        const uint8_t* yrow = yp + (long long)(2 * cy) * pitch + xv;
        // both luma rows of a chroma row exist in the frame (H even), bytes beyond the row's last pixel lie inside the pitch.
        // (Requesting the thread's next chroma row before converting the current one was measured: 92.2 us again for the
        // chrominance mode, 70.2 instead of 61.4 us for green only — 80 registers cost more occupancy than the overlap gains.)
        const uint4 c4 = ld_stream_v4(uvp + (long long)cy * pitch + xv);
        const uint4 a4 = ld_stream_v4(yrow), b4 = ld_stream_v4(yrow + pitch);
        const uint32_t cw[4] = {c4.x, c4.y, c4.z, c4.w};
        const uint32_t yw[2][4] = {{a4.x, a4.y, a4.z, a4.w}, {b4.x, b4.y, b4.z, b4.w}};
        uint32_t pG[2] = {0, 0}, pR[2] = {0, 0}, pB[2] = {0, 0};
#pragma unroll
        for (int pr = 0; pr < 8; ++pr) {
          const int uu = (int)__byte_perm(cw[pr >> 1], 0, 0x4440 + 2 * (pr & 1));
          const int vv = (int)__byte_perm(cw[pr >> 1], 0, 0x4441 + 2 * (pr & 1));
          const int guv = ((1 << 19) - 16 * CY - 128 * (CVG + CUG)) + CVG * vv + CUG * uu;
          const int ruv = ((1 << 19) - 16 * CY - 128 * CVR) + CVR * vv;
          const int buv = ((1 << 19) - 16 * CY - 128 * CUB) + CUB * uu;
#pragma unroll
          for (int ro = 0; ro < 2; ++ro) {
            const int y0 = max((int)__byte_perm(yw[ro][pr >> 1], 0, 0x4440 + 2 * (pr & 1)), 16);
            const int y1 = max((int)__byte_perm(yw[ro][pr >> 1], 0, 0x4441 + 2 * (pr & 1)), 16);
            pG[ro] = __dp4a(pack_sat_u8((y0 * CY + guv) >> 20, (y1 * CY + guv) >> 20, 0u), m2[pr], pG[ro]);
            if (ALL) {
              if (WANT_SUMS) {
                pR[ro] = __dp4a(pack_sat_u8((y0 * CY + ruv) >> 20, (y1 * CY + ruv) >> 20, 0u), m2[pr], pR[ro]);
                pB[ro] = __dp4a(pack_sat_u8((y0 * CY + buv) >> 20, (y1 * CY + buv) >> 20, 0u), m2[pr], pB[ro]);
              } else {                                        // {R0, B0, R1, B1}: both channels of both pixels in one dp4a
                const uint32_t q0 = pack_sat_u8((y0 * CY + ruv) >> 20, (y0 * CY + buv) >> 20, 0u);
                pB[ro] = __dp4a(pack_sat_u8((y1 * CY + ruv) >> 20, (y1 * CY + buv) >> 20, q0), m4[pr], pB[ro]);
              }
            }
          }
        }
        sG += pG[0] * w0 + pG[1] * w1;
        if (ALL) { sB += pB[0] * w0 + pB[1] * w1; if (WANT_SUMS) sR += pR[0] * w0 + pR[1] * w1; }
      }
    }
  }
  const unsigned long long N = (unsigned long long)(nrows > 0 ? nrows : 0) * (unsigned long long)(ncols > 0 ? ncols : 0);
  unsigned long long tB = warp_sum_u64(sB), tG = warp_sum_u64(sG), tR = warp_sum_u64(sR);
  __shared__ unsigned long long part[WARPS][3];
  const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) { part[wid][0] = tB; part[wid][1] = tG; part[wid][2] = tR; }
  __syncthreads();
  if (gt == 0) {
    tB = tG = tR = 0;
#pragma unroll
    for (int w = 0; w < WARPS; ++w) { tB += part[w][0]; tG += part[w][1]; tR += part[w][2]; }
    if (WANT_SUMS) {
      ulonglong4 o; o.x = tB; o.y = tG; o.z = tR; o.w = N;
      *reinterpret_cast<ulonglong4*>(out_sums + 4 * roi) = o;
    }
    double val;
    if (!has_box || N == 0) val = nan_f64();
    else if (mode == BPV_GREEN) val = (double)tG / (double)N;
    else val = (double)(2 * (long long)tG - (long long)tB - (long long)tR + 2 * (long long)N) / (double)(4 * N);   // tR = 0 when tB carries B + R
    out_value[roi] = val;
  }
}

// ---------------------------------------------------------------------------------------------
// F1 on a frame the reference would first have resized (SURVEY.md 8f row 2): VideoReader runs
// cv2.resize(frame, target_res[::-1]) on file input (video_reader.py:95-96) and the ROI boxes live in the resized
// frame.  The resized frame is never materialised: every ROI pixel is produced on the fly with OpenCV's own integer
// bilinear arithmetic (imgproc/src/resize.cpp: 11-bit coefficients from float32 fractions, horizontal pass in 2048ths,
// vertical pass ((b0 * (h0 >> 4)) >> 16) + ((b1 * (h1 >> 4)) >> 16) + 2) >> 2; exact 2x decimation = INTER_AREA fast
// path), so the sums equal those of the frame cv2.resize would have produced, bit for bit.
// One 128-thread CTA per ROI; the ROI's column / row taps (source index + 11-bit weights) are tabulated in shared memory.
// ---------------------------------------------------------------------------------------------
struct ResizeTap { int i0, i1; short w0, w1; };

__device__ __forceinline__ ResizeTap resize_tap(int d, double scale, int sn, bool clamp_fraction) {
  // fx = (float)((dx + 0.5) * scale - 0.5); sx = cvFloor(fx); fx -= sx;  (resize.cpp)
  float f = (float)__dadd_rn(__dmul_rn((double)d + 0.5, scale), -0.5);   // no FMA contraction: OpenCV rounds the product
  int s0 = (int)floorf(f);
  float fr = f - (float)s0;
  ResizeTap t;
  if (clamp_fraction) {                       // columns: fraction dropped at the borders
    if (s0 < 0) { fr = 0.f; s0 = 0; }
    if (s0 >= sn - 1) { fr = 0.f; s0 = sn - 1; }
    t.i0 = s0; t.i1 = s0 + 1 < sn ? s0 + 1 : sn - 1;
  } else {                                    // rows: weights kept, indices clipped
    t.i0 = s0 < 0 ? 0 : (s0 > sn - 1 ? sn - 1 : s0);
    t.i1 = s0 + 1 < 0 ? 0 : (s0 + 1 > sn - 1 ? sn - 1 : s0 + 1);
  }
  t.w0 = (short)__float2int_rn((1.f - fr) * 2048.f);
  t.w1 = (short)__float2int_rn(fr * 2048.f);
  return t;
}

// ALL = false (GREEN without sums): only the green channel goes through the bilinear arithmetic.  The four source pixels
// of an output pixel are read with byte loads (L1 serves them: neighbouring threads share lines); U = 4 row steps per
// iteration keep 4 x 12 of them in flight.  Measured per 8192 frames of 1080p -> 720p boxes (profiles/r2h_ingest.txt):
// byte loads + 4 row steps 289 us (green only 139 us), one row step 315 us, aligned 32-bit loads + funnel shifts 391-507 us.
template <bool WANT_SUMS, bool ALL, int U>
__global__ void __launch_bounds__(128) roi_resized_kernel(const uint8_t* __restrict__ frames, long long frame_stride, long long row_stride,
                                                          int sh, int sw, int dh, int dw, int R, int mode, long long num_rois,
                                                          const int32_t* __restrict__ boxes,
                                                          unsigned long long* __restrict__ out_sums, double* __restrict__ out_value) {
  extern __shared__ __align__(16) unsigned char rsm[];
  constexpr int THREADS = 128, WARPS = THREADS / 32;
  const int gt = threadIdx.x;
  const long long roi = blockIdx.x;
  int xs = 0, xe = 0, ys = 0, ye = 0;
  const int4 b = __ldg(reinterpret_cast<const int4*>(boxes) + roi);
  const bool has_box = b.x != BPV_NO_BOX;
  if (has_box) { py_slice(b.x, b.z, dw, xs, xe); py_slice(b.y, b.w, dh, ys, ye); }   // box lives in the RESIZED frame
  const int nrows = ye - ys, ncols = xe - xs;
  ResizeTap* ctap = reinterpret_cast<ResizeTap*>(rsm);          // [ncols]
  ResizeTap* rtap = ctap + (ncols > 0 ? ncols : 0);             // [nrows]
  const uint8_t* fp = frames + (roi / R) * frame_stride;
  const bool area2 = sw == 2 * dw && sh == 2 * dh;
  uint32_t sB = 0, sG = 0, sR = 0;
  if (nrows > 0 && ncols > 0) {
    if (!area2) {
      const double scale_x = 1.0 / ((double)dw / (double)sw), scale_y = 1.0 / ((double)dh / (double)sh);
      for (int c = gt; c < ncols; c += THREADS) ctap[c] = resize_tap(xs + c, scale_x, sw, true);
      for (int r = gt; r < nrows; r += THREADS) rtap[r] = resize_tap(ys + r, scale_y, sh, false);
    }
    __syncthreads();
    // threads laid out rows x columns (no per-pixel division): a thread keeps its column taps in registers
    int rps, r0, c0;
    if (ncols >= THREADS) { rps = 1; r0 = 0; c0 = gt; }
    else { rps = THREADS / ncols; r0 = gt / ncols; c0 = gt - r0 * ncols; if (r0 >= rps) c0 = ncols; }
    // U row steps per iteration: their 4 x U source loads are all in flight together.  ALL = false (GREEN without sums):
    // only the green channel goes through the bilinear arithmetic.
    for (int c = c0; c < ncols; c += THREADS) {
      ResizeTap tc;
      if (!area2) tc = ctap[c];
      for (int rb = r0; rb < nrows; rb += rps * U) {
        uint32_t a0[U], a1[U], b0[U], b1[U];          // (source row 0 | 1) x (column tap 0 | 1), packed B | G << 8 | R << 16
        int wr0[U], wr1[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int r = rb + u * rps;
          a0[u] = a1[u] = b0[u] = b1[u] = 0; wr0[u] = wr1[u] = 0;
          if (r >= nrows) continue;
          if (area2) {
            const uint8_t* p0 = fp + (long long)(2 * (ys + r)) * row_stride;
            const uint8_t* p1 = p0 + row_stride;
            const int off = 6 * (xs + c);
            a0[u] = p0[off] | p0[off + 1] << 8 | p0[off + 2] << 16; a1[u] = p0[off + 3] | p0[off + 4] << 8 | p0[off + 5] << 16;
            b0[u] = p1[off] | p1[off + 1] << 8 | p1[off + 2] << 16; b1[u] = p1[off + 3] | p1[off + 4] << 8 | p1[off + 5] << 16;
          } else {
            const ResizeTap tr = rtap[r];
            wr0[u] = tr.w0; wr1[u] = tr.w1;
            const uint8_t* q0 = fp + (long long)tr.i0 * row_stride;
            const uint8_t* q1 = fp + (long long)tr.i1 * row_stride;
            a0[u] = q0[3 * tc.i0] | q0[3 * tc.i0 + 1] << 8 | q0[3 * tc.i0 + 2] << 16; a1[u] = q0[3 * tc.i1] | q0[3 * tc.i1 + 1] << 8 | q0[3 * tc.i1 + 2] << 16;
            b0[u] = q1[3 * tc.i0] | q1[3 * tc.i0 + 1] << 8 | q1[3 * tc.i0 + 2] << 16; b1[u] = q1[3 * tc.i1] | q1[3 * tc.i1 + 1] << 8 | q1[3 * tc.i1 + 2] << 16;
          }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
          if (rb + u * rps >= nrows) continue;
          int px[3] = {0, 0, 0};
#pragma unroll
          for (int ch = 0; ch < 3; ++ch) {
            if (!ALL && ch != 1) continue;
            const int A0 = (int)(a0[u] >> (8 * ch) & 255), A1 = (int)(a1[u] >> (8 * ch) & 255);
            const int B0 = (int)(b0[u] >> (8 * ch) & 255), B1 = (int)(b1[u] >> (8 * ch) & 255);
            if (area2) px[ch] = (A0 + A1 + B0 + B1 + 2) >> 2;
            else {
              const int h0 = A0 * tc.w0 + A1 * tc.w1, h1 = B0 * tc.w0 + B1 * tc.w1;
              const int v = (((wr0[u] * (h0 >> 4)) >> 16) + ((wr1[u] * (h1 >> 4)) >> 16) + 2) >> 2;
              px[ch] = v < 0 ? 0 : (v > 255 ? 255 : v);
            }
          }
          sB += (uint32_t)px[0]; sG += (uint32_t)px[1]; sR += (uint32_t)px[2];
        }
      }
    }
  }
  const unsigned long long N = (unsigned long long)(nrows > 0 ? nrows : 0) * (unsigned long long)(ncols > 0 ? ncols : 0);
  unsigned long long tB = warp_sum_u64(sB), tG = warp_sum_u64(sG), tR = warp_sum_u64(sR);
  __shared__ unsigned long long part[WARPS][3];
  const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
  __syncthreads();
  if (lane == 0) { part[wid][0] = tB; part[wid][1] = tG; part[wid][2] = tR; }
  __syncthreads();
  if (gt == 0) {
    tB = tG = tR = 0;
#pragma unroll
    for (int w = 0; w < WARPS; ++w) { tB += part[w][0]; tG += part[w][1]; tR += part[w][2]; }
    if (WANT_SUMS) {
      ulonglong4 o; o.x = tB; o.y = tG; o.z = tR; o.w = N;
      *reinterpret_cast<ulonglong4*>(out_sums + 4 * roi) = o;
    }
    double val;
    if (!has_box || N == 0) val = nan_f64();
    else if (mode == BPV_GREEN) val = (double)tG / (double)N;
    else val = (double)(2 * (long long)tG - (long long)tB - (long long)tR + 2 * (long long)N) / (double)(4 * N);
    out_value[roi] = val;
  }
}

// ---------------------------------------------------------------------------------------------
// Fused resize, staged variant (aligned frames, bilinear case): the ROI's SOURCE footprint is staged in shared memory with
// 16-byte cp.async vectors exactly as the BGR kernel stages its tile (the byte-load kernel above issues 12 byte loads and ~90
// instructions per output pixel), and the bilinear arithmetic is regrouped without changing a single intermediate value:
//   * a thread owns one output column and a contiguous run of output rows; its column's two source pixels are 6 adjacent
//     bytes at a loop-invariant offset, so two PRMTs with per-thread selectors turn four aligned 32-bit shared-memory loads
//     into {B0 B1 G0 G1} and {R0 R1 . .}, and the horizontal pass  h = s0 * a0 + s1 * a1  is ONE dp2a per channel against the
//     packed 11-bit weights (a0 | a1 << 16);
//   * consecutive output rows share source rows (scale 1.5: every other one), so the horizontal result of the previous
//     row's lower source row is kept in registers;
//   * the vertical pass ((b0 * (h0 >> 4)) >> 16) + ((b1 * (h1 >> 4)) >> 16) + 2 is two IMAD.HI with the weights pre-shifted
//     by 16 (all operands are non-negative), >> 2 and the saturation come from one packed convert.
// Output rows are processed in bands whose source rows fit the stage.
// ---------------------------------------------------------------------------------------------
struct RowTap4 { int i0, i1; uint32_t w0s, w1s; };          // source rows + 11-bit weights << 16
struct ColTap2 { int i0; uint32_t wpair; };                 // left source column + (a0 | a1 << 16); the right one is i0 + 1 (a1 = 0 at the border)

template <bool WANT_SUMS, bool ALL>
__global__ void __launch_bounds__(128) roi_resized_staged_kernel(const uint8_t* __restrict__ frames, long long frame_stride, long long row_stride,
                                                                 int sh, int sw, int dh, int dw, int R, int mode, long long num_rois,
                                                                 const int32_t* __restrict__ boxes,
                                                                 unsigned long long* __restrict__ out_sums, double* __restrict__ out_value,
                                                                 int smem_total, double scale_x, double scale_y) {
  extern __shared__ __align__(16) unsigned char rsm[];
  constexpr int THREADS = 128, WARPS = THREADS / 32;
  const int gt = threadIdx.x;
  const long long roi = blockIdx.x;
  int xs = 0, xe = 0, ys = 0, ye = 0;
  const int4 b = __ldg(reinterpret_cast<const int4*>(boxes) + roi);
  const bool has_box = b.x != BPV_NO_BOX;
  if (has_box) { py_slice(b.x, b.z, dw, xs, xe); py_slice(b.y, b.w, dh, ys, ye); }   // box lives in the RESIZED frame
  const int nrows = ye - ys, ncols = xe - xs;
  // dynamic shared memory (smem_total bytes): stage from the front, the ROI's row taps [nrows] at the back; the column tap is
  // per thread (loop invariant), so the tables do not grow with the frame width
  unsigned char* stage = rsm;
  RowTap4* rtap = reinterpret_cast<RowTap4*>(rsm + smem_total) - (nrows > 0 ? nrows : 0);
  const int stage_bytes = smem_total - (nrows > 0 ? nrows : 0) * (int)sizeof(RowTap4);
  const uint8_t* fp = frames + (roi / R) * frame_stride;
  uint32_t sB = 0, sG = 0, sR = 0;                           // !WANT_SUMS: sB carries B + R
  __shared__ int s_xrange[2];
  if (nrows > 0 && ncols > 0) {
    // scale_x / scale_y = 1 / (dst / src) as cv::resize computes them: IEEE double divisions, done once on the host
    for (int r = gt; r < nrows; r += THREADS) {
      const ResizeTap t = resize_tap(ys + r, scale_y, sh, false);
      rtap[r].i0 = t.i0; rtap[r].i1 = t.i1; rtap[r].w0s = (uint32_t)(unsigned short)t.w0 << 16; rtap[r].w1s = (uint32_t)(unsigned short)t.w1 << 16;
    }
    if (gt >= THREADS - 2) s_xrange[gt - (THREADS - 2)] = resize_tap(gt == THREADS - 2 ? xs : xe - 1, scale_x, sw, true).i0;
    __syncthreads();
    const int xmin = s_xrange[0], xlast = s_xrange[1];
    const int xmax = xlast + 1 < sw ? xlast + 1 : sw - 1;
    const int tile_x0 = (3 * xmin) & ~15;                     // staged bytes [tile_x0, tile_x0 + rowb) of every source row
    const int rowb = (3 * xmax + 3 - tile_x0 + 15) & ~15;
    const int rowb_s = rowb + 16;                             // row slot: the border column's don't-care bytes stay inside it
    const int vpr = rowb >> 4;
    const uint32_t sbase = smem_u32(stage);
    const unsigned long long pol = l2_evict_first_policy();
    // this thread's column(s) and row run inside a band
    int rps, r0, c0;
    if (ncols >= THREADS) { rps = 1; r0 = 0; c0 = gt; }
    else { rps = THREADS / ncols; r0 = gt / ncols; c0 = gt - r0 * ncols; if (r0 >= rps) c0 = ncols; }
    int rb = 0;
    while (rb < nrows) {
      const int src0 = rtap[rb].i0;
      int re = nrows;                                         // the usual case: the whole footprint fits the stage
      if ((rtap[nrows - 1].i1 - src0 + 1) * rowb_s > stage_bytes) {
        re = rb + 1;
        while (re < nrows && (rtap[re].i1 - src0 + 1) * rowb_s <= stage_bytes) ++re;   // rtap is monotone: uniform scan
      }
      const int nsrc = rtap[re - 1].i1 - src0 + 1;
      {                                                       // (row, vector) walked without a division per vector
        const int dr = THREADS / vpr, dv = THREADS - dr * vpr;
        int rr = gt / vpr, v = gt - rr * vpr;
        const uint8_t* g = fp + (long long)(src0 + rr) * row_stride + tile_x0 + 16 * v;
        uint32_t d = sbase + (uint32_t)(rr * rowb_s + 16 * v);
        const long long gstep = (long long)dr * row_stride + 16 * dv;
        const uint32_t dstep = (uint32_t)(dr * rowb_s + 16 * dv);
        const long long gwrap = row_stride - 16ll * vpr;
        const uint32_t dwrap = (uint32_t)(rowb_s - 16 * vpr);
        while (rr < nsrc) {
          cp_async16_64B(d, g, pol);
          rr += dr; v += dv; g += gstep; d += dstep;
          if (v >= vpr) { v -= vpr; ++rr; g += gwrap; d += dwrap; }
        }
      }
      cp_async_wait_all();
      __syncthreads();
      const int band = re - rb, run = (band + rps - 1) / rps;
      const int my0 = rb + r0 * run, my1 = my0 + run < re ? my0 + run : re;
      for (int c = c0; c < ncols; c += THREADS) {
        ColTap2 ct;
        {
          const ResizeTap t = resize_tap(xs + c, scale_x, sw, true);
          ct.i0 = t.i0; ct.wpair = (uint32_t)(unsigned short)t.w0 | (uint32_t)(unsigned short)t.w1 << 16;
        }
        const int off = 3 * ct.i0 - tile_x0, shb = off & 3;
        const uint32_t a1 = (uint32_t)(off & ~3), a2 = a1 + (shb == 3 ? 4u : 0u);
        const int s2 = shb == 3 ? 1 : shb + 2;
        const uint32_t sel1 = (uint32_t)(shb | (shb + 3) << 4 | (shb + 1) << 8 | (shb + 4) << 12);   // {B0 B1 G0 G1}
        const uint32_t sel2 = (uint32_t)(s2 | (s2 + 3) << 4);                                       // {R0 R1 . .}
        // branch-free row loop: both source rows of every output row go through the horizontal pass (keeping the previous
        // row's result for the rows that share a source row — every other one at scale 1.5 — was measured slower: the two
        // tests and the divergent copies cost more issue slots than the 12-instruction pass they save)
        auto hpass = [&](int srow, uint32_t& hB, uint32_t& hG, uint32_t& hR) {
          const uint32_t base = sbase + (uint32_t)((srow - src0) * rowb_s);
          uint32_t w0, w1, w2, w3;
          asm volatile("ld.shared.u32 %0, [%1];" : "=r"(w0) : "r"(base + a1));
          asm volatile("ld.shared.u32 %0, [%1];" : "=r"(w1) : "r"(base + a1 + 4u));
          const uint32_t p1 = __byte_perm(w0, w1, sel1);
          hG = __dp2a_hi(ct.wpair, p1, 0u) >> 4;
          if (ALL) {
            asm volatile("ld.shared.u32 %0, [%1];" : "=r"(w2) : "r"(base + a2));
            asm volatile("ld.shared.u32 %0, [%1];" : "=r"(w3) : "r"(base + a2 + 4u));
            const uint32_t p2 = __byte_perm(w2, w3, sel2);
            hB = __dp2a_lo(ct.wpair, p1, 0u) >> 4;
            hR = __dp2a_lo(ct.wpair, p2, 0u) >> 4;
          }
        };
#pragma unroll 2
        for (int r = my0; r < my1; ++r) {
          const RowTap4 tr = rtap[r];
          uint32_t hB0 = 0, hG0 = 0, hR0 = 0, hB1 = 0, hG1 = 0, hR1 = 0;
          hpass(tr.i0, hB0, hG0, hR0);
          hpass(tr.i1, hB1, hG1, hR1);
          const uint32_t g = (__umulhi(hG0, tr.w0s) + __umulhi(hG1, tr.w1s) + 2u) >> 2;
          sG += g < 255u ? g : 255u;
          if (ALL) {
            const uint32_t bb = (__umulhi(hB0, tr.w0s) + __umulhi(hB1, tr.w1s) + 2u) >> 2;
            const uint32_t rr = (__umulhi(hR0, tr.w0s) + __umulhi(hR1, tr.w1s) + 2u) >> 2;
            if (WANT_SUMS) { sB += bb < 255u ? bb : 255u; sR += rr < 255u ? rr : 255u; }
            else sB = __dp4a(pack_sat_u8((int)bb, (int)rr, 0u), 0x00000101u, sB);
          }
        }
      }
      rb = re;
      if (rb < nrows) __syncthreads();                        // band consumed before the next one overwrites the stage
    }
  }
  const unsigned long long N = (unsigned long long)(nrows > 0 ? nrows : 0) * (unsigned long long)(ncols > 0 ? ncols : 0);
  unsigned long long tB = warp_sum_u64(sB), tG = warp_sum_u64(sG), tR = warp_sum_u64(sR);
  __shared__ unsigned long long part[WARPS][3];
  const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
  __syncthreads();
  if (lane == 0) { part[wid][0] = tB; part[wid][1] = tG; part[wid][2] = tR; }
  __syncthreads();
  if (gt == 0) {
    tB = tG = tR = 0;
#pragma unroll
    for (int w = 0; w < WARPS; ++w) { tB += part[w][0]; tG += part[w][1]; tR += part[w][2]; }
    if (WANT_SUMS) {
      ulonglong4 o; o.x = tB; o.y = tG; o.z = tR; o.w = N;
      *reinterpret_cast<ulonglong4*>(out_sums + 4 * roi) = o;
    }
    double val;
    if (!has_box || N == 0) val = nan_f64();
    else if (mode == BPV_GREEN) val = (double)tG / (double)N;
    else val = (double)(2 * (long long)tG - (long long)tB - (long long)tR + 2 * (long long)N) / (double)(4 * N);   // tR = 0 when tB carries B + R
    out_value[roi] = val;
  }
}

}  // namespace bpv

extern "C" int bpv_roi_sample_nv12(const uint8_t* frames, int64_t frame_stride_bytes, int64_t pitch_bytes,
                                   int32_t H, int32_t W, int64_t num_frames, const int32_t* boxes, int32_t R, int32_t mode,
                                   uint64_t* out_sums, double* out_value, void* stream) {
  using namespace bpv;
  BPV_REQUIRE(frames && boxes && out_value, BPV_E_INVALID, "bpv_roi_sample_nv12: NULL pointer");
  BPV_REQUIRE(H > 0 && W > 0 && (H % 2) == 0 && (W % 2) == 0 && R > 0 && num_frames >= 0, BPV_E_INVALID,
              "bpv_roi_sample_nv12: H and W must be positive and even");
  BPV_REQUIRE(pitch_bytes >= W && frame_stride_bytes >= pitch_bytes * (H + H / 2), BPV_E_INVALID,
              "bpv_roi_sample_nv12: pitch < W or frame stride < pitch * 3H/2");
  BPV_REQUIRE(mode == BPV_GREEN || mode == BPV_CHROM_GREEN, BPV_E_UNSUPPORTED,
              "bpv_roi_sample_nv12: unknown color channel %d (NotImplementedError, signal_processor.py:185)", mode);
  BPV_REQUIRE(num_frames * (int64_t)R <= INT32_MAX, BPV_E_TOO_LARGE, "bpv_roi_sample_nv12: more than 2^31-1 ROIs in one call");
  if (num_frames == 0) return 0;
  const long long n = num_frames * R;
  cudaStream_t st = (cudaStream_t)stream;
  // 128-bit loads need aligned rows; the Y plane of frame f starts at f * frame_stride and the UV plane H * pitch later
  const bool vec = (((uintptr_t)frames | (uintptr_t)frame_stride_bytes | (uintptr_t)pitch_bytes) & 15) == 0;
  const bool all = mode != BPV_GREEN;
#define BPV_NV12(S, A) roi_nv12_kernel<S, A><<<(unsigned)n, 128, 0, st>>>(frames, frame_stride_bytes, pitch_bytes, H, W, R, mode, n, boxes, \
                                                                        (unsigned long long*)out_sums, out_value)
#define BPV_NV12V(S, A) roi_nv12_vec_kernel<S, A><<<(unsigned)n, 128, 0, st>>>(frames, frame_stride_bytes, pitch_bytes, H, W, R, mode, n, boxes, \
                                                                             (unsigned long long*)out_sums, out_value)
  if (vec) {
    if (out_sums) BPV_NV12V(true, true);
    else if (all) BPV_NV12V(false, true);
    else BPV_NV12V(false, false);
  }
  else if (out_sums) BPV_NV12(true, true);
  else if (all) BPV_NV12(false, true);
  else BPV_NV12(false, false);
#undef BPV_NV12
#undef BPV_NV12V
  return check_launch("bpv_roi_sample_nv12");
}

extern "C" int bpv_roi_sample_resized_u8(const uint8_t* frames, int64_t frame_stride_bytes, int64_t row_stride_bytes,
                                         int32_t src_h, int32_t src_w, int32_t dst_h, int32_t dst_w, int64_t num_frames,
                                         const int32_t* boxes, int32_t R, int32_t mode,
                                         uint64_t* out_sums, double* out_value, void* stream) {
  using namespace bpv;
  BPV_REQUIRE(frames && boxes && out_value, BPV_E_INVALID, "bpv_roi_sample_resized_u8: NULL pointer");
  BPV_REQUIRE(src_h > 0 && src_w > 0 && dst_h > 0 && dst_w > 0 && R > 0 && num_frames >= 0, BPV_E_INVALID,
              "bpv_roi_sample_resized_u8: bad sizes");
  BPV_REQUIRE(row_stride_bytes >= 3ll * src_w, BPV_E_INVALID, "bpv_roi_sample_resized_u8: row_stride_bytes < 3*src_w");
  BPV_REQUIRE(mode == BPV_GREEN || mode == BPV_CHROM_GREEN, BPV_E_UNSUPPORTED,
              "bpv_roi_sample_resized_u8: unknown color channel %d (NotImplementedError, signal_processor.py:185)", mode);
  BPV_REQUIRE((int64_t)(dst_h + dst_w) * (int64_t)sizeof(ResizeTap) <= 200 * 1024, BPV_E_TOO_LARGE,
              "bpv_roi_sample_resized_u8: target size too large for the tap tables");
  BPV_REQUIRE(num_frames * (int64_t)R <= INT32_MAX, BPV_E_TOO_LARGE, "bpv_roi_sample_resized_u8: more than 2^31-1 ROIs in one call");
  if (num_frames == 0) return 0;
  const long long n = num_frames * R;
  const int smem = (dst_h + dst_w) * (int)sizeof(ResizeTap);        // worst case: a ROI spanning the whole resized frame
  cudaStream_t st = (cudaStream_t)stream;
#define BPV_RSZ(S, A)                                                                                                       \
  do {                                                                                                                      \
    if (int rc = ensure_dyn_smem((const void*)roi_resized_kernel<S, A, 4>, smem)) return rc;                                 \
    roi_resized_kernel<S, A, 4><<<(unsigned)n, 128, smem, st>>>(frames, frame_stride_bytes, row_stride_bytes, src_h, src_w,   \
                                                                dst_h, dst_w, R, mode, n, boxes,                             \
                                                                (unsigned long long*)out_sums, out_value);                   \
  } while (0)
  // staged variant: aligned frames, bilinear case (the exact 2x decimation keeps the byte-load kernel), and a stage that holds
  // the two source rows of one output row at the frame's full width
  const bool aligned = (((uintptr_t)frames | (uintptr_t)frame_stride_bytes | (uintptr_t)row_stride_bytes) & 15) == 0;
  const bool area2 = src_w == 2 * dst_w && src_h == 2 * dst_h;
  const int smem2 = 26 * 1024;                                        // 8 CTAs per SM
  const long long rowslot = ((3ll * src_w + 15) & ~15ll) + 32;
  if (aligned && !area2 && 2 * rowslot + (long long)dst_h * (long long)sizeof(RowTap4) <= smem2) {
#define BPV_RSZ2(S, A)                                                                                                      \
  do {                                                                                                                      \
    if (int rc = ensure_dyn_smem((const void*)roi_resized_staged_kernel<S, A>, smem2)) return rc;                            \
    roi_resized_staged_kernel<S, A><<<(unsigned)n, 128, smem2, st>>>(frames, frame_stride_bytes, row_stride_bytes, src_h,    \
                                                                     src_w, dst_h, dst_w, R, mode, n, boxes,                 \
                                                                     (unsigned long long*)out_sums, out_value, smem2,        \
                                                                     1.0 / ((double)dst_w / (double)src_w),                  \
                                                                     1.0 / ((double)dst_h / (double)src_h));                 \
  } while (0)
    if (out_sums) BPV_RSZ2(true, true);
    else if (mode != BPV_GREEN) BPV_RSZ2(false, true);
    else BPV_RSZ2(false, false);
#undef BPV_RSZ2
    return check_launch("bpv_roi_sample_resized_u8");
  }
  if (out_sums) BPV_RSZ(true, true);
  else if (mode != BPV_GREEN) BPV_RSZ(false, true);
  else BPV_RSZ(false, false);
#undef BPV_RSZ
  return check_launch("bpv_roi_sample_resized_u8");
}

extern "C" int bpv_roi_sample_u8(const uint8_t* frames, const uint8_t* const* frame_ptrs,
                                 int64_t frame_stride_bytes, int64_t row_stride_bytes,
                                 int32_t H, int32_t W, int64_t num_frames,
                                 const int32_t* boxes, int32_t R, int32_t mode,
                                 uint64_t* out_sums, double* out_value,
                                 int64_t roi_pixels_hint, void* stream) {
  using namespace bpv;
  BPV_REQUIRE(frames || frame_ptrs, BPV_E_INVALID, "bpv_roi_sample_u8: frames and frame_ptrs are both NULL");
  BPV_REQUIRE(boxes && out_value, BPV_E_INVALID, "bpv_roi_sample_u8: NULL boxes/out_value");
  BPV_REQUIRE(H > 0 && W > 0 && R > 0 && num_frames >= 0, BPV_E_INVALID, "bpv_roi_sample_u8: bad H/W/R/num_frames");
  BPV_REQUIRE((int64_t)H * W * 3 < (1ll << 31), BPV_E_TOO_LARGE, "bpv_roi_sample_u8: frame larger than 2 GiB");
  BPV_REQUIRE(row_stride_bytes >= 3ll * W, BPV_E_INVALID, "bpv_roi_sample_u8: row_stride_bytes < 3*W");
  BPV_REQUIRE(frame_stride_bytes >= 0, BPV_E_INVALID, "bpv_roi_sample_u8: negative frame_stride_bytes");   // 0 = one frame, many box sets
  BPV_REQUIRE(num_frames * (int64_t)R <= INT32_MAX, BPV_E_TOO_LARGE, "bpv_roi_sample_u8: more than 2^31-1 ROIs in one call");
  BPV_REQUIRE(mode == BPV_GREEN || mode == BPV_CHROM_GREEN, BPV_E_UNSUPPORTED,
              "bpv_roi_sample_u8: unknown color channel %d (NotImplementedError, signal_processor.py:185)", mode);
  if (num_frames == 0) return 0;
  RoiArgs a{frames, frame_ptrs, frame_stride_bytes, row_stride_bytes, H, W, R, mode,
            num_frames * R, boxes, (unsigned long long*)out_sums, out_value};
  cudaStream_t st = (cudaStream_t)stream;
  const long long n = a.num_rois;
  bool host_frames = false;
  if (frames) {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, frames) == cudaSuccess) host_frames = at.type == cudaMemoryTypeHost;
    else cudaGetLastError();
  }
  // threads per ROI: ~>= 4 vectors per thread before widening the group
  const long long px = roi_pixels_hint > 0 ? roi_pixels_hint : 4096;
  const int g = px * 3 <= 32 * 16 * 8 ? 32 : (px * 3 <= 128 * 16 * 16 ? 128 : 256);
  const unsigned grid = (unsigned)((n + 256 / g - 1) / (256 / g));
  if (row_stride_bytes % 16 == 0) {  // fast path: loop-invariant alignment per ROI
    // small ROIs: a warp per ROI, loads held in registers; everything else: one ROI per CTA, tile staged in
    // shared memory by cp.async (whole ROI in flight; measured 64.5 us vs 76.3 us for the register path on the
    // config-2 boxes, 6.2 TB/s on 320x160 boxes; profiles/r1e_roi_variants.txt).  Frames in pinned host memory
    // (zero-copy e2e path) are PCIe-bound and want full-line requests: register path with plain loads.
    if (host_frames) {
      if (g == 32) launch_rows<32, true>(a, grid, st);
      else launch_rows<128, true>(a, (unsigned)((n + 1) / 2), st);
    }
    else if (g == 32) launch_rows<32, false>(a, grid, st);
    else launch_staged<128, 12>(a, st);
  } else {                           // generic path: alignment changes row by row
    if (g == 32) roi_sample_kernel<32, 4><<<grid, 256, 0, st>>>(a);
    else if (g == 128) roi_sample_kernel<128, 4><<<grid, 256, 0, st>>>(a);
    else roi_sample_kernel<256, 4><<<grid, 256, 0, st>>>(a);
  }
  return check_launch("bpv_roi_sample_u8");
}
