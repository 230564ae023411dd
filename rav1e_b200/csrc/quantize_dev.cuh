// quantize_dev.cuh — the quantize chain's device code and host-side setup, shared by quantize.cu (batched
// chain) and encode_tx.cu (the chain fused between the forward and the inverse transform).
#pragma once
#include <cuda_runtime.h>

#include <algorithm>
#include <limits>
#include <vector>

#include "common.cuh"

namespace {

// transform/mod.rs:101-123 order
const int kQtxW[19] = {4, 8, 16, 32, 64, 4, 8, 8, 16, 16, 32, 32, 64, 4, 16, 8, 32, 16, 64};
const int kQtxH[19] = {4, 8, 16, 32, 64, 8, 4, 16, 8, 32, 16, 64, 32, 16, 4, 32, 8, 64, 16};

struct QuantArgs {
  const void *coeffs;
  void *qcoeffs, *rcoeffs;
  uint16_t *eob;
  unsigned long long *tx_dist;
  const uint16_t *scan, *iscan;
  size_t n;
  int area, coded, log_tx_scale;
  int deadzone;  // already cast to the coefficient type
  uint32_t dc_quant, ac_quant, dc_offset, ac_offset0, ac_offset1;
  uint32_t dc_mul[3], ac_mul[3];
};

// quantize/mod.rs:148-157
__device__ __forceinline__ uint32_t divu_pair(uint32_t x, const uint32_t (&d)[3]) {
  return (uint32_t)((((unsigned long long)d[0] * x + d[1]) >> 32) >> d[2]);
}

// (c * c) as u64 with c: i32 (wrapping multiply, then sign extension), encoder.rs:1622-1624
__device__ __forceinline__ unsigned long long sq_i32(int c) {
  return (unsigned long long)(long long)(int)((uint32_t)c * (uint32_t)c);
}

// quantize/mod.rs:384-390
__device__ __forceinline__ int dequant1(int c, uint32_t quant, int log_tx_scale) {
  const int offset = (1 << log_tx_scale) - 1;
  return (int)((uint32_t)c * quant + (uint32_t)((c >> 31) & offset)) >> log_tx_scale;
}

// `c.abs() >= deadzone` with c: T, quantize/mod.rs:296.  The reference's release build negates with
// wrapping, so T::MIN.abs() is T::MIN and never reaches the deadzone.  Evaluated in 32 bits with T::MIN
// singled out: a 16-bit abs of -32768 on the device yields +32768, which counted a -32768 coefficient
// towards the end of block.
template <typename T>
__device__ __forceinline__ bool reaches_deadzone(T v, int deadzone) {
  const int iv = (int)v;
  return iv != (int)std::numeric_limits<T>::min() && (iv < 0 ? -iv : iv) >= deadzone;
}

// h(x) = after(before(x)) for functions {0,1} -> {0,1} stored as bit x = f(x)
__device__ __forceinline__ uint32_t compose(uint32_t after, uint32_t before) {
  return ((after >> (before & 1)) & 1) | (((after >> ((before >> 1) & 1)) & 1) << 1);
}

// QuantizationContext::quantize + dequantize + raw tx-domain distortion of ONE block by one warp
// (quantize/mod.rs:269-392, encoder.rs:1611-1640).  c: the block's coefficients (any address space),
// q: quantized coefficients out, r: dequantized ones out (may be NULL); both `coded` long.
template <typename T>
__device__ __forceinline__ void quantize_block_warp(const QuantArgs &a, const T *c, T *q, T *r, uint16_t *eob_out,
                                                    unsigned long long *dist_out, int lane) {
    // ---- pass 1: sum of squares of every coefficient, end of block (quantize/mod.rs:292-305),
    // zero fill of the outputs ("assume that qcoeffs is pre-filled with zeros", :343-344)
    unsigned long long ss = 0;
    uint32_t em1 = 0;
    for (int i = lane; i < a.area; i += 32) {
      const T v = c[i];
      ss += sq_i32((int)v);
      if (i < a.coded) {
        if (reaches_deadzone(v, a.deadzone)) em1 = max(em1, (uint32_t)a.iscan[i]);
        q[i] = 0;
        if (r) r[i] = 0;
      }
    }
    em1 = __reduce_max_sync(0xffffffffu, em1);
    __syncwarp();  // the zero fill is ordered before the scattered stores below
    // ---- DC (its own step size and offset), :272-279
    const int c0 = (int)c[0];
    const int coeff0 = (int)((uint32_t)c0 << a.log_tx_scale);
    const uint32_t abs0 = coeff0 < 0 ? 0u - (uint32_t)coeff0 : (uint32_t)coeff0;
    const uint32_t aq0 = divu_pair(abs0 + a.dc_offset, a.dc_mul);
    const T q0 = (T)(coeff0 < 0 ? -(int)aq0 : (int)aq0);
    const T r0 = (T)dequant1((int)q0, a.dc_quant, a.log_tx_scale);
    unsigned long long adj = 0;  // sum over touched positions of (c - r)^2 - c^2 (mod 2^64)
    if (lane == 0) {
      q[0] = q0;
      if (r) r[0] = r0;
      adj = sq_i32(c0 - (int)r0) - sq_i32(c0);
    }
    const uint32_t eob = em1 > 0 ? em1 + 1 : (uint32_t)(q0 != 0);
    // ---- the scan-order loop, :318-341, 32 positions per step
    uint32_t carry = 1;  // level_mode
    for (uint32_t base = 1; base < eob; base += 32) {
      const uint32_t j = base + lane;
      const bool on = j < eob;
      int pos = 0, coeff = 0, cv = 0;
      uint32_t aq_lm1 = 0, aq_lm0 = 0, f = 2u;  // identity: f(0) = 0, f(1) = 1
      if (on) {
        pos = a.scan[j];
        cv = (int)c[pos];
        coeff = (int)((uint32_t)cv << a.log_tx_scale);
        const uint32_t ab = coeff < 0 ? 0u - (uint32_t)coeff : (uint32_t)coeff;
        const uint32_t level0 = divu_pair(ab, a.ac_mul);
        const uint32_t lim = (level0 + 1) * a.ac_quant;
        // level0 > 1 - level_mode: level_mode 1 -> level0 > 0, level_mode 0 -> level0 > 1
        aq_lm1 = level0 + (uint32_t)(ab + (level0 > 0 ? a.ac_offset1 : a.ac_offset0) >= lim);
        aq_lm0 = level0 + (uint32_t)(ab + (level0 > 1 ? a.ac_offset1 : a.ac_offset0) >= lim);
        // next level_mode: from 1: 0 iff abs_qcoeff == 0; from 0: 1 iff abs_qcoeff > 1
        f = (uint32_t)(aq_lm0 > 1) | ((uint32_t)(aq_lm1 != 0) << 1);
      }
      uint32_t incl = f;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const uint32_t before = __shfl_up_sync(0xffffffffu, incl, d);
        if (lane >= d) incl = compose(incl, before);
      }
      const uint32_t excl = __shfl_up_sync(0xffffffffu, incl, 1);
      const uint32_t lm_in = lane == 0 ? carry : ((excl >> carry) & 1);
      carry = (__shfl_sync(0xffffffffu, incl, 31) >> carry) & 1;
      if (on) {
        const uint32_t aq = lm_in ? aq_lm1 : aq_lm0;
        const T qv = (T)(coeff < 0 ? -(int)aq : (int)aq);
        const T rv = (T)dequant1((int)qv, a.ac_quant, a.log_tx_scale);
        q[pos] = qv;
        if (r) r[pos] = rv;
        adj += sq_i32(cv - (int)rv) - sq_i32(cv);
      }
    }
    if (dist_out) {
      unsigned long long tot = ss + adj;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) tot += __shfl_xor_sync(0xffffffffu, tot, o);
      const int bits = 2 * (3 - a.log_tx_scale);  // encoder.rs:1627-1631
      if (lane == 0) *dist_out = (tot + (1ull << (bits - 1))) >> bits;
    }
    if (lane == 0 && eob_out) *eob_out = (uint16_t)eob;
}

template <typename T>
__global__ void __launch_bounds__(256) quantize_chain_kernel(const __grid_constant__ QuantArgs a) {
  const int lane = threadIdx.x & 31;
  const size_t warp0 = (size_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const size_t nwarps = (size_t)gridDim.x * (blockDim.x >> 5);
  for (size_t blk = warp0; blk < a.n; blk += nwarps) {
    quantize_block_warp<T>(a, (const T *)a.coeffs + blk * (size_t)a.area, (T *)a.qcoeffs + blk * (size_t)a.coded,
                           a.rcoeffs ? (T *)a.rcoeffs + blk * (size_t)a.coded : nullptr, a.eob ? a.eob + blk : nullptr,
                           a.tx_dist ? a.tx_dist + blk : nullptr, lane);
    __syncwarp();
  }
}

// quantize/mod.rs:129-146
void divu_gen(uint32_t d, uint32_t out[3]) {
  const unsigned long long nbits = 32;
  const unsigned long long m = nbits - (unsigned long long)__builtin_clz(d) - 1;
  if ((d & (d - 1)) == 0) {
    out[0] = out[1] = 0xFFFFFFFFu;
  } else {
    const unsigned long long t = (1ull << (m + nbits)) / d;
    const unsigned long long rr = (t * d + d) & ((1ull << nbits) - 1);
    if (rr <= 1ull << m) {
      out[0] = (uint32_t)t + 1;
      out[1] = 0;
    } else {
      out[0] = out[1] = (uint32_t)t;
    }
  }
  out[2] = (uint32_t)m;
}

// av1_scan_orders[tx_size][tx_type] (scan_order.rs:949-1321) regenerated from the rule the tables
// follow in rav1e's transposed coefficient layout (index = col * H + row): types 0..9 walk
// anti-diagonals (bottom-up for wide blocks, top-down for tall ones, alternating for square ones),
// V_* types walk rows, H_* types are the identity.  64-point dimensions code 32.
void make_scan(int tx_size, int kind, std::vector<uint16_t> *scan, std::vector<uint16_t> *iscan) {
  const int W = std::min(kQtxW[tx_size], 32), H = std::min(kQtxH[tx_size], 32);
  scan->clear();
  if (kind == 2) {
    for (int i = 0; i < W * H; i++) scan->push_back((uint16_t)i);
  } else if (kind == 1) {
    for (int r = 0; r < H; r++)
      for (int c = 0; c < W; c++) scan->push_back((uint16_t)(c * H + r));
  } else {
    for (int d = 0; d < W + H - 1; d++) {
      const int r_lo = std::max(d - (W - 1), 0), r_hi = std::min(d, H - 1);
      const bool down = W < H || (W == H && (d & 1));
      for (int k = 0; k <= r_hi - r_lo; k++) {
        const int r = down ? r_lo + k : r_hi - k;
        scan->push_back((uint16_t)((d - r) * H + r));
      }
    }
  }
  iscan->assign(scan->size(), 0);
  for (size_t i = 0; i < scan->size(); i++) (*iscan)[(*scan)[i]] = (uint16_t)i;
}

// device copies of the scan tables, one per (ctx, tx_size, kind), created on first use and owned by
// the context (b200_ctx_destroy frees them); uploaded on the ctx's stream, so the kernel that
// follows on the same stream is ordered behind the copy
int scan_tables(b200_ctx *ctx, int tx_size, int kind, const uint16_t **d_scan, const uint16_t **d_iscan) {
  const int key = tx_size * 4 + kind;
  const size_t n = (size_t)std::min(kQtxW[tx_size], 32) * std::min(kQtxH[tx_size], 32);
  auto it = ctx->scan_dev.find(key);
  if (it == ctx->scan_dev.end()) {
    std::vector<uint16_t> scan, iscan;
    make_scan(tx_size, kind, &scan, &iscan);
    std::vector<uint16_t> &img = ctx->scan_host[key];
    img = scan;
    img.insert(img.end(), iscan.begin(), iscan.end());
    uint16_t *d = nullptr;
    B200_CUDA(ctx, cudaMalloc(&d, 2 * n * sizeof(uint16_t)));
    const cudaError_t e = cudaMemcpyAsync(d, img.data(), 2 * n * sizeof(uint16_t), cudaMemcpyHostToDevice, ctx->stream);
    if (e != cudaSuccess) {
      cudaFree(d);
      ctx->scan_host.erase(key);
      B200_CUDA(ctx, e);
    }
    it = ctx->scan_dev.emplace(key, d).first;
  }
  *d_scan = it->second;
  *d_iscan = it->second + n;
  return B200_OK;
}

// QuantizationContext::update (quantize/mod.rs:219-267) + the per-call geometry: everything the device
// code reads except the buffers.
inline int quant_setup(b200_ctx *ctx, int tx_size, int tx_type, uint32_t dc_quant, uint32_t ac_quant, int is_intra,
                       int coeff_is_i32, QuantArgs *out) {
  QuantArgs a{};
  const int kind = tx_type < 10 ? 0 : ((tx_type & 1) ? 2 : 1);
  if (int st = scan_tables(ctx, tx_size, kind, &a.scan, &a.iscan)) return st;
  a.area = kQtxW[tx_size] * kQtxH[tx_size];
  a.coded = std::min(kQtxW[tx_size], 32) * std::min(kQtxH[tx_size], 32);
  a.log_tx_scale = (a.area > 256) + (a.area > 1024);  // quantize/mod.rs:29-34
  a.dc_quant = dc_quant;
  a.ac_quant = ac_quant;
  divu_gen(dc_quant, a.dc_mul);
  divu_gen(ac_quant, a.ac_mul);
  a.dc_offset = dc_quant * (is_intra ? 109u : 108u) / 256;
  a.ac_offset0 = ac_quant * (is_intra ? 98u : 97u) / 256;
  a.ac_offset1 = ac_quant * (is_intra ? 109u : 108u) / 256;
  const uint32_t ac_offset_eob = ac_quant * (is_intra ? 88u : 44u) / 256;
  // deadzone, :287-291: (ac_quant - ac_offset_eob).align_power_of_two_and_shift(log_tx_scale) cast to T
  const size_t dz = ((size_t)ac_quant - ac_offset_eob + ((size_t)1 << a.log_tx_scale) - 1) >> a.log_tx_scale;
  a.deadzone = coeff_is_i32 ? (int)(int32_t)dz : (int)(int16_t)dz;
  *out = a;
  return B200_OK;
}

}  // namespace
