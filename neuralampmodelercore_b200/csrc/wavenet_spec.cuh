// wavenet_spec.cuh -- the MODEL-SPECIALISED fused WaveNet kernel for sm_100a.
//
// This file is compiled once per model (NVRTC at load time, jit_spec.cpp; or nvcc for tools/spec_proto.cu) together
// with a generated header that defines namespace `spec`: the layer table as constexpr data and the weights as
// `__device__ const unsigned Wb[]` bit patterns read through spec::w(i).  Every loop below has compile-time bounds and is fully unrolled, so every weight
// becomes the 32-bit IMMEDIATE of an FFMA (`FFMA R, Rx, 0.1234, R`): no weight loads, no weight registers, no
// shared-memory copy of the weights.  Why: the generic fused kernel (wavenet_fused.cuh) broadcasts weights from shared
// memory, and at two frames per thread one uniform LDS.128 (2 wavefronts) feeds only 4 FFMA2 -- the shared-memory pipe
// runs at 67 % while the FMA pipe reaches 59 % (profiles/r01g_*): the two saturate together.  With immediates the FMA
// pipe is fed by the instruction stream alone; shared memory carries only the activations.
//
// What it computes (reference file:line, all under NAM/): the same path as wavenet_fused.cuh --
//   wavenet/model.cpp:822-910 WaveNet::process, :463-549 LayerArray::Process, :183-393 Layer::Process (non-gated, no
//   FiLM, no head1x1), conv1d.cpp:666-683 Conv1D::Process, ring_buffer.cpp:7-109 RingBuffer, dsp.cpp:436-836 Conv1x1,
//   activations.h:59-133 -- in the same summation order (bias + mixin first, taps oldest to newest, input channels
//   ascending), so its results are bit-identical to the generic fused kernel's.
//
// Mapping: one persistent CTA owns one stream at a time and walks its call in tiles of T = S * NT frames; thread t owns
// frames {t, t + NT, ..} for the whole depth of the network (see wavenet_fused.cuh).  What is new here:
//   * TMA-engine staging of the history (cp.async.bulk, SASS UBLKCP): before a layer runs, the last `lookback` columns of
//     its input ring are copied global -> shared by bulk-async copies that complete on an mbarrier, into the columns
//     directly in front of the tile: buf[plane][LS - lookback .. LS) | tile columns [LS .. LS + T).  Every dilated tap
//     of every layer is then ONE shared-memory load at a compile-time offset from the thread's own column: no ring
//     addressing, no branch, no per-thread global load in the compute path.  The copy of layer l+1's history is issued
//     right after layer l's last tap read (barrier B1) and lands under layer l's 1x1 phase.
//   * the tile's newest columns go back to the ring with bulk-async stores shared -> global, issued by the same lanes
//     (so the async-proxy store -> load order on a ring is per-thread program order + wait_group).
// Ring layout and semantics are those of wavenet_fused.cuh ([C/4][R][4] floats, R a power of two >= lookback, indexed
// by absolute frame number), so calls served by this kernel and by the generic kernels can be mixed on one handle.
#pragma once

#ifndef NAMB200_SPEC_HEADER_INCLUDED
#error "include the generated model header (namespace spec) before wavenet_spec.cuh"
#endif

namespace namb200_spec
{
typedef unsigned long long u64;
typedef unsigned int u32;

// Activation codes == namb200::KACT_* (wavenet_desc.h)
enum : int
{
  ACT_TANH = 0,
  ACT_HARDTANH = 1,
  ACT_FASTTANH = 2,
  ACT_RELU = 3,
  ACT_LEAKYRELU = 4,
  ACT_PRELU = 5,
  ACT_SIGMOID = 6,
  ACT_SILU = 7,
  ACT_HARDSWISH = 8,
  ACT_LEAKYHARDTANH = 9,
  ACT_SOFTSIGN = 10
};

struct SpecParams
{
  float* state; // [batch][state_stride]: the rings of wavenet_fused.cuh
  long state_stride; // floats
  const float* in; // [batch][in_stride]
  float* out;
  long in_stride, out_stride;
  int batch, n_frames;
  u32 t_base; // absolute frame index of in[:, 0] (mod 2^32)
  float* scratch; // S = 2: [grid][scratch_stride] floats, a CTA's stream pair in the interleaved layout
  long scratch_stride; // 2 * state_stride
};

// ---- scalar helpers (same arithmetic as wavenet_fused.cuh) ------------------------------------------------------
__device__ __forceinline__ float rcp_approx(float x)
{
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ u64 pack2(const float lo, const float hi)
{
  u64 r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void unpack2(const u64 v, float& lo, float& hi)
{
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ u64 fma2(u64 a, u64 b, u64 c)
{
  u64 d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
__device__ __forceinline__ u64 mul2(u64 a, u64 b)
{
  u64 d;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
__device__ __forceinline__ u64 add2(u64 a, u64 b)
{
  u64 d;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
__device__ __forceinline__ u64 dup2(float v)
{
  return pack2(v, v);
}
// the reference's rational fast_tanh (activations.h:91-98) on a packed pair.  The denominator's |x + c x |x|| is
// evaluated as |x| + c x^2 (the same number: c > 0, so the factor 1 + c |x| is positive; one rounding differs, < 1e-7
// relative): one packed multiply and one 64-bit AND fewer per pair than the literal form in wavenet_fused.cuh.
__device__ __forceinline__ u64 fast_tanh2(u64 x)
{
  constexpr u64 kAbs = 0x7FFFFFFF7FFFFFFFull;
  const u64 ax = x & kAbs;
  const u64 x2 = mul2(x, x);
  const u64 c0 = dup2(2.45550750702956f);
  const u64 t1 = fma2(dup2(0.821226666969744f), ax, dup2(0.893229853513558f));
  const u64 t0 = fma2(c0, ax, c0);
  const u64 num = mul2(x, fma2(t1, x2, t0));
  const u64 s = fma2(dup2(0.814642734961073f), x2, ax);
  const u64 d0 = dup2(2.44506634652299f);
  const u64 den = fma2(add2(x2, d0), s, d0);
  float dl, dh;
  unpack2(den, dl, dh);
  return mul2(num, pack2(rcp_approx(dl), rcp_approx(dh)));
}
__device__ __forceinline__ float act_sigmoid(float x)
{
  return rcp_approx(1.0f + expf(-x));
}

// ---- frame vectors -------------------------------------------------------------------------------------------------------
// S = 1: a thread owns frame `tid` of ONE stream, V = float.
// S = 2: a thread owns frame `tid` of a PAIR of streams (2q, 2q + 1), V = a packed f32x2 pair (low half = the even
// stream).  Everything a layer does is written once over V.  For S = 2 one instruction serves both streams:
// `FFMA2 Racc, Rx.F32x2, <imm32>, Racc` -- the packed FMA takes the weight as a BROADCAST IMMEDIATE, so the weight stream
// costs one issue slot and 16 instruction bytes per weight for two frames, and the kernel is bound by the FMA pipe itself
// instead of by instruction issue / fetch (profiles/r02a_*: S = 1 issues 16,800 instructions per warp-frame, 79 % FFMA,
// top stall no_instruction).  The pair must sit in an aligned register pair, so the activations of the two streams are
// interleaved element-wise wherever they are stored: a column of a "sub-plane" is 16 bytes = (c A, c B, c' A, c' B) for
// two channels c, c' -- one LDS.128 yields two ready pairs, conflict-free.  The rings of the library keep one stream
// per ring ([C/4][R][4 floats]), so the kernel converts a pair's rings into a per-CTA scratch in the interleaved layout
// when it picks the pair up, runs all tiles of the call on the scratch (bulk copies move interleaved columns), and
// converts back at the end: other kernels never see the interleaved layout.
template <int S>
struct FrameVec;
template <>
struct FrameVec<1>
{
  typedef float type;
};
template <>
struct FrameVec<2>
{
  typedef u64 type;
};

__device__ __forceinline__ float vfma(const float x, const float w, const float a)
{
  return fmaf(w, x, a);
}
__device__ __forceinline__ u64 vfma(const u64 x, const float w, const u64 a)
{
  return fma2(x, dup2(w), a);
}
__device__ __forceinline__ float vadd(const float a, const float b)
{
  return a + b;
}
__device__ __forceinline__ u64 vadd(const u64 a, const u64 b)
{
  return add2(a, b);
}
__device__ __forceinline__ float vaddc(const float a, const float c)
{
  return a + c;
}
__device__ __forceinline__ u64 vaddc(const u64 a, const float c)
{
  return add2(a, dup2(c));
}
__device__ __forceinline__ void vsplat(float& v, const float c)
{
  v = c;
}
__device__ __forceinline__ void vsplat(u64& v, const float c)
{
  v = dup2(c);
}
// The 4 channels of plane `pl` at column offset `off` behind this thread's own column.  `col0` = the thread's column in
// (sub-)plane 0, W = columns per (sub-)plane.  S = 1: one 16-byte column of a 4-channel plane.  S = 2: two 16-byte
// columns of two 2-channel sub-planes, each (c A, c B, c' A, c' B).
template <int W>
__device__ __forceinline__ void load_plane(const float4* col0, const int pl, const int off, float (&x)[4])
{
  const float4 q = col0[pl * W - off];
  x[0] = q.x, x[1] = q.y, x[2] = q.z, x[3] = q.w;
}
template <int W>
__device__ __forceinline__ void load_plane(const float4* col0, const int pl, const int off, u64 (&x)[4])
{
  const float4 q0 = col0[(2 * pl) * W - off], q1 = col0[(2 * pl + 1) * W - off];
  x[0] = pack2(q0.x, q0.y), x[1] = pack2(q0.z, q0.w), x[2] = pack2(q1.x, q1.y), x[3] = pack2(q1.z, q1.w);
}
template <int W>
__device__ __forceinline__ void store_plane(float4* col0, const int pl, const float (&x)[4])
{
  col0[pl * W] = make_float4(x[0], x[1], x[2], x[3]);
}
template <int W>
__device__ __forceinline__ void store_plane(float4* col0, const int pl, const u64 (&x)[4])
{
  float4 q0, q1;
  unpack2(x[0], q0.x, q0.y), unpack2(x[1], q0.z, q0.w), unpack2(x[2], q1.x, q1.y), unpack2(x[3], q1.z, q1.w);
  col0[(2 * pl) * W] = q0, col0[(2 * pl + 1) * W] = q1;
}

// one element of layer LI's activation, channel i (activations.h:59-133)
template <int LI, int C>
__device__ __forceinline__ float act_scalar(const float x, const int i)
{
  constexpr spec::Layer Ld = spec::L[LI];
  if constexpr (Ld.act == ACT_TANH)
    return tanhf(x);
  else if constexpr (Ld.act == ACT_HARDTANH)
    return fminf(fmaxf(x, -1.0f), 1.0f);
  else if constexpr (Ld.act == ACT_RELU)
    return x > 0.0f ? x : 0.0f;
  else if constexpr (Ld.act == ACT_LEAKYRELU)
    return x > 0.0f ? x : Ld.ap0 * x;
  else if constexpr (Ld.act == ACT_PRELU)
    return x > 0.0f ? x : spec::w(Ld.w_off + Ld.K * C * C + C + C + C * C + C + i) * x;
  else if constexpr (Ld.act == ACT_SIGMOID)
    return act_sigmoid(x);
  else if constexpr (Ld.act == ACT_SILU)
    return x * act_sigmoid(x);
  else if constexpr (Ld.act == ACT_HARDSWISH)
  {
    const float t = x + 3.0f;
    const float cl = t < 0.0f ? 0.0f : (t > 6.0f ? 6.0f : t);
    return x * cl * (1.0f / 6.0f);
  }
  else if constexpr (Ld.act == ACT_LEAKYHARDTANH)
    return x < Ld.ap0 ? (x - Ld.ap0) * Ld.ap2 + Ld.ap0 : (x > Ld.ap1 ? (x - Ld.ap1) * Ld.ap3 + Ld.ap1 : x);
  else if constexpr (Ld.act == ACT_SOFTSIGN)
    return x * rcp_approx(1.0f + fabsf(x));
  else
    return x;
}

template <int LI, int C>
__device__ __forceinline__ void apply_activation(float (&v)[C])
{
  if constexpr (spec::L[LI].act == ACT_FASTTANH)
  {
#pragma unroll
    for (int q = 0; q < C / 2; q++) // two channels of the frame per packed operation
      unpack2(fast_tanh2(pack2(v[2 * q], v[2 * q + 1])), v[2 * q], v[2 * q + 1]);
  }
  else
  {
#pragma unroll
    for (int i = 0; i < C; i++)
      v[i] = act_scalar<LI, C>(v[i], i);
  }
}
template <int LI, int C>
__device__ __forceinline__ void apply_activation(u64 (&v)[C])
{
#pragma unroll
  for (int i = 0; i < C; i++)
  {
    if constexpr (spec::L[LI].act == ACT_FASTTANH)
      v[i] = fast_tanh2(v[i]); // the two frames of the channel per packed operation
    else
    {
      float a, b;
      unpack2(v[i], a, b);
      v[i] = pack2(act_scalar<LI, C>(a, i), act_scalar<LI, C>(b, i));
    }
  }
}

// ---- mbarrier / bulk-async copy primitives ------------------------------------------------------------------------
__device__ __forceinline__ u32 smem_addr(const void* p)
{
  return (u32)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(u64* bar, int count)
{
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(u64* bar, u32 bytes)
{
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(u64* bar, u32 parity)
{
  asm volatile(
    "{\n"
    ".reg .pred p;\n"
    "WAIT_%=:\n"
    "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
    "@p bra DONE_%=;\n"
    "bra WAIT_%=;\n"
    "DONE_%=:\n"
    "}\n" ::"r"(smem_addr(bar)),
    "r"(parity)
    : "memory");
}
// global -> shared, completes `bytes` on the mbarrier (SASS: UBLKCP)
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, u32 bytes, u64* bar)
{
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                 smem_addr(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(smem_addr(bar))
               : "memory");
}
// shared -> global, tracked by the issuing thread's bulk async-group
__device__ __forceinline__ void bulk_s2g(void* dst_gmem, const void* src_smem, u32 bytes)
{
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst_gmem), "r"(smem_addr(src_smem)),
               "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void bulk_commit()
{
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
__device__ __forceinline__ void bulk_wait_all()
{
  asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}
// generic-proxy writes to shared memory -> visible to the async proxy (the bulk stores that read the tile)
__device__ __forceinline__ void fence_async_smem()
{
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// ---- one ring <-> the staging buffer --------------------------------------------------------------------------------
// A "history unit" = one ring of P planes: a layer's input ring or an array's head-accumulator ring.
// Lane `pl` (< P) of warp 0 moves plane pl: at most two contiguous pieces when the range wraps around the ring.
//   load : ring columns [tabs0 - L, tabs0)            -> buf[pl][LS - L, LS)
//   store: tile columns [tv - n, tv), n = min(L, tv)  -> ring columns [tabs0 + tv - n, tabs0 + tv)
template <int P, int L, int RMASK, int W>
__device__ __forceinline__ void hist_load(float4* buf, float* ring_f, const u32 tabs0, u64* bar, const int lane)
{
  constexpr int R = RMASK + 1;
  static_assert(L <= R && L <= spec::LS, "ring / staging geometry");
  if (lane == 0)
    mbar_expect_tx(bar, (u32)(P * L * 16)); // (a kernel-size-1 layer has no history: the phase completes at once)
  __syncwarp();
  if (L > 0 && lane < P)
  {
    const float4* ring = reinterpret_cast<const float4*>(ring_f) + lane * R;
    float4* dst = buf + lane * W + (spec::LS - L);
    const int start = (int)((tabs0 - (u32)L) & (u32)RMASK);
    const int n1 = min(L, R - start);
    bulk_g2s(dst, ring + start, (u32)n1 * 16u, bar);
    if (n1 < L)
      bulk_g2s(dst + n1, ring, (u32)(L - n1) * 16u, bar);
  }
}
template <int P, int L, int RMASK, int W>
__device__ __forceinline__ void hist_store(const float4* buf, float* ring_f, const u32 tabs0, const int tv, const int lane)
{
  constexpr int R = RMASK + 1;
  if (L > 0 && lane < P)
  {
    float4* ring = reinterpret_cast<float4*>(ring_f) + lane * R;
    const int n = min(L, tv);
    const float4* src = buf + lane * W + spec::LS + (tv - n);
    const int start = (int)((tabs0 + (u32)(tv - n)) & (u32)RMASK);
    const int n1 = min(n, R - start);
    bulk_s2g(ring + start, src, (u32)n1 * 16u);
    if (n1 < n)
      bulk_s2g(ring, src + n1, (u32)(n - n1) * 16u);
    bulk_commit();
  }
}

// compile-time loop over the layers of an array
template <int V>
struct IntC
{
  static constexpr int value = V;
};
template <int I, int N, typename F>
__device__ __forceinline__ void static_for(F&& f)
{
  if constexpr (I < N)
  {
    f(IntC<I>{});
    static_for<I + 1, N>(f);
  }
}

struct TileCtx
{
  float4* buf; // staging buffer: [plane][W] columns
  u64* bar; // the history mbarrier
  u32 phase; // its parity
  float* state; // this stream's rings
  u32 tabs0; // absolute frame number of the tile's first frame
  int tv; // valid frames in this tile
  int warp, lane;
};

// history of the unit that follows (AI, LI) in program order is requested right after the current unit's last read.
// The last warp issues these loads and warp 0 the ring stores: each costs its warp ~75 instructions per layer, and
// with both on warp 0 that warp reached every barrier last (4096 x 4096 a1_standard: 10.3 -> 9.5 ms per launch).  A
// ring's stores complete (wait_group 0 before B1) and a barrier passes before any load of the same columns is issued.
template <int AI, int NT, int S, int LI>
__device__ __forceinline__ void request_layer_history(TileCtx& c, IntC<LI>)
{
  constexpr spec::Layer Ld = spec::L[LI];
  constexpr int C = spec::A[AI].C;
  constexpr int W = spec::LS + NT;
  // S = 2: C/2 sub-planes of 16-byte columns; the interleaved ring of a pair is twice the size of one stream's ring
  if (c.warp == NT / 32 - 1)
    hist_load<(S == 1 ? C / 4 : C / 2), (Ld.K - 1) * Ld.dil, Ld.ring_mask, W>(c.buf, c.state + S * Ld.ring_off, c.tabs0, c.bar,
                                                                              c.lane);
}

// One layer array for the S frames a thread owns (cf. namb200::array_forward), V = FrameVec<S>.
//   hin[CIN]: the array's input (the raw sample for the first array, the previous array's last layer output after)
//   head[C]: the head accumulator, initialised by the caller (zeros, or the previous array's head output)
//   headout[HOUT]: this array's head output
//   NEXT_AI: the array that follows (-1: none) -- its first layer's history is requested after this array's last tap read
template <int AI, int NEXT_AI, int NT, int S, typename V>
__device__ __forceinline__ void array_forward(TileCtx& c, const V (&hin)[spec::A[AI].CIN], const V cond, V (&head)[spec::A[AI].C],
                                              V (&hout)[spec::A[AI].C], V (&headout)[spec::A[AI].HOUT])
{
  constexpr spec::Array A = spec::A[AI];
  constexpr int C = A.C, CIN = A.CIN, HOUT = A.HOUT, P = C / 4;
  constexpr int W = spec::LS + NT;
  constexpr int HP = (S == 1) ? C / 4 : C / 2; // (sub-)planes the history copies move
  constexpr int HEADK = A.head_kernel, HRMASK = A.head_ring_mask, HROFF = A.head_ring_off;
  constexpr int HL = (A.head_kernel - 1) * A.head_dilation; // look-back of a convolutional head (0: kernel size 1)
  float4* const col0 = c.buf + spec::LS + threadIdx.x; // this thread's column of (sub-)plane 0

  // ---- rechannel (Conv1x1, no bias; model.cpp:492) -> this thread's columns of the tile
  {
    V h[C];
#pragma unroll
    for (int o = 0; o < C; o++)
      vsplat(h[o], 0.0f);
#pragma unroll
    for (int i = 0; i < CIN; i++)
#pragma unroll
      for (int o = 0; o < C; o++)
        h[o] = vfma(hin[i], spec::w(A.rech_off + i * C + o), h[o]);
#pragma unroll
    for (int pl = 0; pl < P; pl++)
    {
      const V q[4] = {h[4 * pl], h[4 * pl + 1], h[4 * pl + 2], h[4 * pl + 3]};
      store_plane<W>(col0, pl, q);
    }
  }

  static_for<0, A.n_layers>([&](auto li_c) {
    constexpr int LI = A.layer0 + decltype(li_c)::value;
    constexpr bool last = (decltype(li_c)::value + 1 == A.n_layers);
    constexpr spec::Layer Ld = spec::L[LI];
    constexpr int K = Ld.K, dil = Ld.dil, L = (K - 1) * dil;
    constexpr int w_conv = Ld.w_off, w_bias = w_conv + K * C * C, w_mix = w_bias + C, w_p = w_mix + C,
                  w_pb = w_p + C * C;

    fence_async_smem(); // my tile columns (generic stores) -> the bulk store below
    __syncthreads(); // B0: the layer input is complete in the tile
    mbar_wait(c.bar, c.phase); // .. and its history has landed in front of it
    c.phase ^= 1u;
    if (c.warp == 0) // newest columns -> ring (reads the tile until B1)
      hist_store<HP, L, Ld.ring_mask, W>(c.buf, c.state + S * Ld.ring_off, c.tabs0, c.tv, c.lane);

    // ---- phase 1: z = b + M c + sum_k W_k h[t - (K-1-k) d];  a = act(z);  head += a
    V acc[C];
#pragma unroll
    for (int o = 0; o < C; o++)
    {
      V b;
      vsplat(b, spec::w(w_bias + o));
      acc[o] = vfma(cond, spec::w(w_mix + o), b);
    }
#pragma unroll
    for (int k = 0; k < K; k++)
    {
      const int off = (K - 1 - k) * dil;
#pragma unroll
      for (int pl = 0; pl < P; pl++)
      {
        V x[4];
        load_plane<W>(col0, pl, off, x);
#pragma unroll
        for (int i = 0; i < 4; i++)
#pragma unroll
          for (int o = 0; o < C; o++)
            acc[o] = vfma(x[i], spec::w(w_conv + (k * C + 4 * pl + i) * C + o), acc[o]);
      }
    }
    apply_activation<LI, C>(acc);
    if constexpr (S == 1)
    {
#pragma unroll
      for (int q = 0; q < C / 2; q++) // model.cpp:530 (packed add over channel pairs: half the issue slots)
        unpack2(add2(pack2(head[2 * q], head[2 * q + 1]), pack2(acc[2 * q], acc[2 * q + 1])), head[2 * q], head[2 * q + 1]);
    }
    else
    {
#pragma unroll
      for (int o = 0; o < C; o++)
        head[o] = vadd(head[o], acc[o]); // model.cpp:530
    }
    if (c.warp == 0 && c.lane < HP)
      bulk_wait_all(); // my ring stores are done: the tile may be rewritten, the rings may be re-read
    __syncthreads(); // B1: every tap read of this layer's input is done
    // the next unit's history lands under this layer's 1x1 phase
    if constexpr (!last)
      request_layer_history<AI, NT, S>(c, IntC<LI + 1>{});
    else if constexpr (HEADK > 1)
    {
      if (c.warp == NT / 32 - 1) // the head accumulator's own ring (A2 family: head{kernel_size: 16}, model.cpp:397-400)
        hist_load<HP, HL, HRMASK, W>(c.buf, c.state + S * HROFF, c.tabs0, c.bar, c.lane);
    }
    else if constexpr (NEXT_AI >= 0)
      request_layer_history<NEXT_AI, NT, S>(c, IntC<spec::A[NEXT_AI < 0 ? 0 : NEXT_AI].layer0>{});

    // ---- phase 2: h_{l+1} = h_l + p + P a  (model.cpp:243,376)
    V hn[C];
#pragma unroll
    for (int pl = 0; pl < P; pl++)
    {
      V own[4];
      load_plane<W>(col0, pl, 0, own);
#pragma unroll
      for (int i = 0; i < 4; i++)
        hn[4 * pl + i] = vaddc(own[i], spec::w(w_pb + 4 * pl + i));
    }
#pragma unroll
    for (int i = 0; i < C; i++)
#pragma unroll
      for (int o = 0; o < C; o++)
        hn[o] = vfma(acc[i], spec::w(w_p + i * C + o), hn[o]);
    if constexpr (!last)
    {
#pragma unroll
      for (int pl = 0; pl < P; pl++)
      {
        const V q[4] = {hn[4 * pl], hn[4 * pl + 1], hn[4 * pl + 2], hn[4 * pl + 3]};
        store_plane<W>(col0, pl, q);
      }
    }
    else
    {
#pragma unroll
      for (int o = 0; o < C; o++)
        hout[o] = hn[o];
    }
  });

  if constexpr (A.head_kernel > 1)
  {
    // ---- head rechannel as a causal convolution over the head accumulator (model.cpp:397-400,548): one more history
    //      unit -- the accumulator columns go through the tile, their last (HK-1)*dilation columns live in the head ring
    constexpr int HK = A.head_kernel, hd = A.head_dilation;
#pragma unroll
    for (int pl = 0; pl < P; pl++)
    {
      const V q[4] = {head[4 * pl], head[4 * pl + 1], head[4 * pl + 2], head[4 * pl + 3]};
      store_plane<W>(col0, pl, q);
    }
    fence_async_smem();
    __syncthreads(); // the accumulator columns are complete in the tile
    mbar_wait(c.bar, c.phase);
    c.phase ^= 1u;
    if (c.warp == 0)
      hist_store<HP, HL, A.head_ring_mask, W>(c.buf, c.state + S * A.head_ring_off, c.tabs0, c.tv, c.lane);
#pragma unroll
    for (int ho = 0; ho < HOUT; ho++)
      vsplat(headout[ho], spec::w(A.head_off + HK * C * HOUT + ho)); // bias first, like the fused kernel
#pragma unroll
    for (int k = 0; k < HK; k++)
    {
      const int off = (HK - 1 - k) * hd;
#pragma unroll
      for (int pl = 0; pl < P; pl++)
      {
        V x[4];
        load_plane<W>(col0, pl, off, x);
#pragma unroll
        for (int i = 0; i < 4; i++)
#pragma unroll
          for (int ho = 0; ho < HOUT; ho++)
            headout[ho] = vfma(x[i], spec::w(A.head_off + (k * C + 4 * pl + i) * HOUT + ho), headout[ho]);
      }
    }
    if (c.warp == 0 && c.lane < HP)
      bulk_wait_all();
    __syncthreads(); // every read of the accumulator columns is done
    if constexpr (NEXT_AI >= 0)
      request_layer_history<NEXT_AI, NT, S>(c, IntC<spec::A[NEXT_AI < 0 ? 0 : NEXT_AI].layer0>{});
    return;
  }

  // ---- head rechannel (kernel size 1; model.cpp:548): headout = H head (+ g)
#pragma unroll
  for (int ho = 0; ho < HOUT; ho++)
    vsplat(headout[ho], 0.0f);
#pragma unroll
  for (int i = 0; i < C; i++)
#pragma unroll
    for (int ho = 0; ho < HOUT; ho++)
      headout[ho] = vfma(head[i], spec::w(A.head_off + i * HOUT + ho), headout[ho]);
#pragma unroll
  for (int ho = 0; ho < HOUT; ho++)
    headout[ho] = vaddc(headout[ho], spec::w(A.head_off + C * HOUT + ho)); // bias (zero when the head has none)
}

template <int NT>
__device__ __forceinline__ void pair_rings_to_scratch(const float* ra, const float* rb, float* sc)
{
  static_for<0, spec::NL>([&](auto li_c) {
    constexpr int LI = decltype(li_c)::value;
    constexpr spec::Layer Ld = spec::L[LI];
    constexpr int R = Ld.ring_mask + 1;
    constexpr int C = spec::layer_channels(LI);
    const float4* a4 = reinterpret_cast<const float4*>(ra + Ld.ring_off);
    const float4* b4 = reinterpret_cast<const float4*>(rb + Ld.ring_off);
    float4* s4 = reinterpret_cast<float4*>(sc + 2 * Ld.ring_off);
    for (int idx = threadIdx.x; idx < (C / 4) * R; idx += NT)
    {
      const int pl = idx / R, col = idx - pl * R;
      const float4 a = __ldcg(a4 + idx), b = __ldcg(b4 + idx);
      __stcg(s4 + (2 * pl) * R + col, make_float4(a.x, b.x, a.y, b.y));
      __stcg(s4 + (2 * pl + 1) * R + col, make_float4(a.z, b.z, a.w, b.w));
    }
  });
}
template <int NT>
__device__ __forceinline__ void pair_scratch_to_rings(const float* sc, float* ra, float* rb, const bool live_b)
{
  static_for<0, spec::NL>([&](auto li_c) {
    constexpr int LI = decltype(li_c)::value;
    constexpr spec::Layer Ld = spec::L[LI];
    constexpr int R = Ld.ring_mask + 1;
    constexpr int C = spec::layer_channels(LI);
    float4* a4 = reinterpret_cast<float4*>(ra + Ld.ring_off);
    float4* b4 = reinterpret_cast<float4*>(rb + Ld.ring_off);
    const float4* s4 = reinterpret_cast<const float4*>(sc + 2 * Ld.ring_off);
    for (int idx = threadIdx.x; idx < (C / 4) * R; idx += NT)
    {
      const int pl = idx / R, col = idx - pl * R;
      const float4 q0 = __ldcg(s4 + (2 * pl) * R + col), q1 = __ldcg(s4 + (2 * pl + 1) * R + col);
      __stcg(a4 + idx, make_float4(q0.x, q0.z, q1.x, q1.z));
      if (live_b)
        __stcg(b4 + idx, make_float4(q0.y, q0.w, q1.y, q1.w));
    }
  });
}
// generic-proxy global accesses <-> the bulk (async-proxy) copies on the scratch
__device__ __forceinline__ void fence_async_all()
{
  asm volatile("fence.proxy.async;" ::: "memory");
}

template <int NT, int S, int MINB>
__device__ __forceinline__ void wavenet_spec_body(const SpecParams& p)
{
  static_assert(S == 1 || (spec::A[0].head_kernel == 1 && spec::A[spec::NA - 1].head_kernel == 1),
                "the stream-pair variant does not convert head rings");
  constexpr int T = NT; // one frame per thread (of one stream, or of a pair of streams)
  static_assert(spec::NA == 1 || spec::NA == 2, "one or two layer arrays");
  static_assert(S == 1 || S == 2, "one stream per thread, or a packed pair of streams");
  extern __shared__ float4 spec_smem[]; // [(sub-)planes][W] float4
  __shared__ u64 bar;
  const int tid = threadIdx.x;
  TileCtx c;
  c.buf = spec_smem;
  c.bar = &bar;
  c.phase = 0u;
  c.warp = tid >> 5;
  c.lane = tid & 31;
  if (tid == 0)
  {
    mbar_init(&bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();

  typedef typename FrameVec<S>::type V;
  const int n_units = (S == 1) ? p.batch : (p.batch + 1) / 2; // streams, or pairs of streams
  for (int unit = blockIdx.x; unit < n_units; unit += gridDim.x)
  {
    const int sa = S * unit, sb = min(sa + 1, p.batch - 1);
    const bool live_b = (S == 2) && (sa + 1 < p.batch); // an odd batch leaves the last pair's second half idle
    float* const state_a = p.state + (size_t)sa * p.state_stride;
    float* const state_b = p.state + (size_t)sb * p.state_stride;
    const float* xin_a = p.in + (size_t)sa * p.in_stride;
    const float* xin_b = p.in + (size_t)sb * p.in_stride;
    float* yout_a = p.out + (size_t)sa * p.out_stride;
    float* yout_b = p.out + (size_t)sb * p.out_stride;
    if constexpr (S == 1)
      c.state = state_a;
    else
    {
      c.state = p.scratch + (size_t)blockIdx.x * p.scratch_stride;
      pair_rings_to_scratch<NT>(state_a, state_b, c.state);
      fence_async_all(); // my scratch stores (generic proxy) -> the bulk loads below
      __syncthreads();
    }
    for (int t0 = 0; t0 < p.n_frames; t0 += T)
    {
      c.tv = min(T, p.n_frames - t0);
      c.tabs0 = p.t_base + (u32)t0;
      request_layer_history<0, NT, S>(c, IntC<spec::A[0].layer0>{});
      V x[1];
      {
        const float xa = (tid < c.tv) ? __ldg(xin_a + t0 + tid) : 0.0f;
        if constexpr (S == 1)
          x[0] = xa;
        else
          x[0] = pack2(xa, (live_b && tid < c.tv) ? __ldg(xin_b + t0 + tid) : 0.0f);
      }
      const V cond = x[0]; // no condition_dsp: condition == input (model.cpp:781)
      V y;
      constexpr int C0 = spec::A[0].C;
      V head0[C0], hout0[C0], ho0[spec::A[0].HOUT];
#pragma unroll
      for (int o = 0; o < C0; o++)
        vsplat(head0[o], 0.0f); // model.cpp:469
      if constexpr (spec::NA == 1)
      {
        array_forward<0, -1, NT, S, V>(c, x, cond, head0, hout0, ho0);
        y = ho0[0];
      }
      else
      {
        array_forward<0, spec::NA - 1, NT, S, V>(c, x, cond, head0, hout0, ho0);
        // second array: layer input = the previous array's layer output, head accumulator starts from the previous
        // array's head output (model.cpp:846-848, :473-486)
        constexpr int AI1 = spec::NA - 1;
        constexpr int C1 = spec::A[AI1].C;
        V head1[C1], hout1[C1], ho1[spec::A[AI1].HOUT];
#pragma unroll
        for (int o = 0; o < C1; o++)
          head1[o] = ho0[o];
        array_forward<AI1, -1, NT, S, V>(c, hout0, cond, head1, hout1, ho1);
        y = ho1[0];
      }
      // model.cpp:888-897
      if constexpr (S == 1)
      {
        if (tid < c.tv)
          yout_a[t0 + tid] = spec::head_scale * y;
      }
      else
      {
        float ya, yb;
        unpack2(y, ya, yb);
        if (tid < c.tv)
        {
          yout_a[t0 + tid] = spec::head_scale * ya;
          if (live_b)
            yout_b[t0 + tid] = spec::head_scale * yb;
        }
      }
      // (no barrier here: the last layer's B1 already fenced every tap read before anything of the next tile is written)
    }
    if constexpr (S == 2)
    {
      // every bulk store of the call has completed (each issuing lane waited before the last B1); make them visible to
      // the generic loads of the conversion, then hand the rings back in the library's layout
      fence_async_all();
      __syncthreads();
      pair_scratch_to_rings<NT>(c.state, state_a, state_b, live_b);
      __syncthreads(); // the scratch is rewritten for the next pair
    }
  }
}

// ==== short calls on many streams: Q streams x FQ frames per CTA ==========================================================
// The reference's hosts call process() with 64-frame blocks.  With thousands of streams such a step is not latency-bound
// per stream but occupancy-bound: every stream-call must pull ~61 KB of ring columns (a1_standard, 64 frames) through L2 /
// HBM, and the precompiled short-call geometry (4 streams per 128-thread CTA, 55 KB of weights in shared memory per CTA)
// runs 8 warps per SM -- profiles/r02i_short_call_*: long-scoreboard stalls, issue-active 32 %.  Here the weights are
// immediates, so a CTA is NT / FQ streams side by side (8 x 64 frames at 512 threads), shared memory holds only the
// tile (32 KB) and 32 warps per SM hide the ring loads.  History is NOT staged: a tap that reaches before the call reads
// its ring column directly (16 bytes per thread, consecutive frames = consecutive addresses), one that stays inside the
// call reads the tile.  Same rings as every other kernel.
//
// Two things decide this kernel (profiles/r02t_*: a launch is only two passes through ~260 KB of straight-line code, and
// the 0.5 GB of ring traffic between two launches had pushed that code out of L2, so one pass in two fetched its
// instructions from HBM -- `no_instruction` 7.3 cycles per issued instruction against 2.1 in the long-call kernel):
//  * ring loads / stores carry an L2 evict-first policy, so the code (and nothing else is reused) stays L2-resident;
//  * each warp prefetches the NEXT layer's ring windows into L2 (one `prefetch.global.L2` per lane) while it computes
//    this one, so the tap loads meet L2 latency instead of HBM latency.
#ifndef NAMB200_SHORT_HINT
#define NAMB200_SHORT_HINT 1
#endif
#ifndef NAMB200_SHORT_PREFETCH
#define NAMB200_SHORT_PREFETCH 0
#endif

__device__ __forceinline__ unsigned long long l2_evict_first_policy()
{
  unsigned long long pol;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}

__device__ __forceinline__ float4 ring_load(const float4* a, const unsigned long long pol)
{
#if NAMB200_SHORT_HINT
  float4 v;
  asm volatile("ld.global.cg.L2::cache_hint.v4.f32 {%0, %1, %2, %3}, [%4], %5;"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
               : "l"(a), "l"(pol));
  return v;
#else
  return __ldcg(a);
#endif
}

__device__ __forceinline__ void ring_store(float4* a, const float4 v, const unsigned long long pol)
{
#if NAMB200_SHORT_HINT
  asm volatile("st.global.cg.L2::cache_hint.v4.f32 [%0], {%1, %2, %3, %4}, %5;" ::"l"(a), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w),
               "l"(pol)
               : "memory");
#else
  __stcg(a, v);
#endif
}

// L2 prefetch of the ring windows layer LJ will read for this warp's 32 frames: (K - 1) history taps x P planes x 4 lines
// of 8 columns; one line per lane (two rounds when there are more).  Lines are taken from the 8-column-aligned start, which
// is exact whenever call start and dilation are multiples of 8 (the usual case); otherwise the last partial line is left out.
template <int LJ, int FQ>
__device__ __forceinline__ void prefetch_ring_windows(const float* state, const unsigned long long pol, const u32 tabs0, const int f)
{
#if NAMB200_SHORT_PREFETCH == 2
  // bulk form: one lane per (tap, plane), up to 512 contiguous bytes (two pieces where the window wraps), evict-first like
  // the loads that follow
  constexpr spec::Layer Ld = spec::L[LJ];
  constexpr int K = Ld.K, dil = Ld.dil, R = Ld.ring_mask + 1;
  constexpr int C = spec::layer_channels(LJ), P = C / 4;
  if constexpr (K > 1 && R >= 32)
  {
    const int lane = f & 31, fw = f & ~31;
    const int tap = lane / P, pl = lane % P;
    const int off = (K - 1 - tap) * dil;
    if (lane < (K - 1) * P && fw < off)
    {
      const float4* const ring = reinterpret_cast<const float4*>(state + Ld.ring_off) + pl * R;
      const int n_cols = min(32, off - fw);
      const int s0 = (int)((tabs0 + (u32)fw - (u32)off) & (u32)Ld.ring_mask);
      const int first = min(n_cols, R - s0);
      asm volatile("cp.async.bulk.prefetch.L2.global.L2::cache_hint [%0], %1, %2;" ::"l"(ring + s0), "r"(first * 16), "l"(pol)
                   : "memory");
      if (first < n_cols)
        asm volatile("cp.async.bulk.prefetch.L2.global.L2::cache_hint [%0], %1, %2;" ::"l"(ring), "r"((n_cols - first) * 16),
                     "l"(pol)
                     : "memory");
    }
  }
#elif NAMB200_SHORT_PREFETCH == 1
  constexpr spec::Layer Ld = spec::L[LJ];
  constexpr int K = Ld.K, dil = Ld.dil, R = Ld.ring_mask + 1;
  constexpr int C = spec::layer_channels(LJ), P = C / 4;
  if constexpr (K > 1 && R >= 32)
  {
    constexpr int TOTAL = (K - 1) * P * 4;
    const int lane = f & 31, fw = f & ~31;
    const float4* const ring = reinterpret_cast<const float4*>(state + Ld.ring_off);
#pragma unroll
    for (int base = 0; base < TOTAL; base += 32)
    {
      const int idx = base + lane;
      const int tap = idx / (P * 4), pl = (idx >> 2) % P, qtr = idx & 3;
      const int off = (K - 1 - tap) * dil;
      if (idx < TOTAL && fw < off)
      {
        const u32 col = ((tabs0 + (u32)(fw + 8 * qtr) - (u32)off) & (u32)Ld.ring_mask) & ~7u;
        asm volatile("prefetch.global.L2 [%0];" ::"l"(ring + pl * R + col));
      }
    }
  }
#endif
}

template <int AI, int NEXT_AI, int NT, int FQ>
__device__ __forceinline__ void array_forward_short(float4* tile, float* state, const unsigned long long pol, const u32 tabs0,
                                                    const int n, const int f, const bool live, const float (&hin)[spec::A[AI].CIN], const float cond,
                                                    float (&head)[spec::A[AI].C], float (&hout)[spec::A[AI].C],
                                                    float (&headout)[spec::A[AI].HOUT])
{
  constexpr spec::Array A = spec::A[AI];
  constexpr int C = A.C, CIN = A.CIN, HOUT = A.HOUT, P = C / 4;
  constexpr int W = NT; // tile columns per plane: Q streams x FQ frames, thread t owns column t
  static_assert(A.head_kernel == 1, "convolutional heads take the precompiled short-call geometry");
  float4* const col0 = tile + threadIdx.x;

  if constexpr (AI == 0)
    prefetch_ring_windows<A.layer0, FQ>(state, pol, tabs0, f);
  {
    float h[C];
#pragma unroll
    for (int o = 0; o < C; o++)
      h[o] = 0.0f;
#pragma unroll
    for (int i = 0; i < CIN; i++)
#pragma unroll
      for (int o = 0; o < C; o++)
        h[o] = fmaf(spec::w(A.rech_off + i * C + o), hin[i], h[o]);
#pragma unroll
    for (int pl = 0; pl < P; pl++)
      col0[pl * W] = make_float4(h[4 * pl], h[4 * pl + 1], h[4 * pl + 2], h[4 * pl + 3]);
  }

  static_for<0, A.n_layers>([&](auto li_c) {
    constexpr int LI = A.layer0 + decltype(li_c)::value;
    constexpr bool last = (decltype(li_c)::value + 1 == A.n_layers);
    constexpr spec::Layer Ld = spec::L[LI];
    constexpr int K = Ld.K, dil = Ld.dil, L = (K - 1) * dil, R = Ld.ring_mask + 1;
    constexpr int w_conv = Ld.w_off, w_bias = w_conv + K * C * C, w_mix = w_bias + C, w_p = w_mix + C,
                  w_pb = w_p + C * C;
    const float4* const ring = reinterpret_cast<const float4*>(state + Ld.ring_off);

    __syncthreads(); // B0: the layer input is complete in the tile
    if constexpr (!last)
      prefetch_ring_windows<LI + 1, FQ>(state, pol, tabs0, f);
    else if constexpr (NEXT_AI >= 0)
      prefetch_ring_windows<spec::A[NEXT_AI >= 0 ? NEXT_AI : 0].layer0, FQ>(state, pol, tabs0, f);
    float acc[C];
#pragma unroll
    for (int o = 0; o < C; o++)
      acc[o] = fmaf(spec::w(w_mix + o), cond, spec::w(w_bias + o));
    static_for<0, K>([&](auto k_c) {
      constexpr int k = decltype(k_c)::value;
      constexpr int off = (K - 1 - k) * dil;
      const bool from_ring = (off > 0) && (off >= FQ || f < off); // (warp-uniform for off >= FQ and for off a multiple of 32)
      const u32 rcol = (tabs0 + (u32)f - (u32)off) & (u32)Ld.ring_mask;
#pragma unroll
      for (int pl = 0; pl < P; pl++)
      {
        float4 q;
        if (from_ring)
          q = ring_load(ring + pl * R + rcol, pol);
        else
          q = col0[pl * W - off];
        const float x[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
        for (int i = 0; i < 4; i++)
#pragma unroll
          for (int o = 0; o < C; o++)
            acc[o] = fmaf(spec::w(w_conv + (k * C + 4 * pl + i) * C + o), x[i], acc[o]);
      }
    });
    apply_activation<LI, C>(acc);
#pragma unroll
    for (int q = 0; q < C / 2; q++) // model.cpp:530
      unpack2(add2(pack2(head[2 * q], head[2 * q + 1]), pack2(acc[2 * q], acc[2 * q + 1])), head[2 * q], head[2 * q + 1]);
    __syncthreads(); // B1: every tap read of the tile is done

    float hn[C];
#pragma unroll
    for (int pl = 0; pl < P; pl++)
    {
      const float4 own = col0[pl * W];
      // RingBuffer::Write: the call's last `look-back` columns of the layer input (ring loads of this layer are done:
      // they fed the FMAs above, and the barrier ordered every thread's loads before anybody's stores)
      if (live && f < n && f >= n - L)
        ring_store(reinterpret_cast<float4*>(state + Ld.ring_off) + pl * R + ((tabs0 + (u32)f) & (u32)Ld.ring_mask), own, pol);
      hn[4 * pl] = own.x + spec::w(w_pb + 4 * pl);
      hn[4 * pl + 1] = own.y + spec::w(w_pb + 4 * pl + 1);
      hn[4 * pl + 2] = own.z + spec::w(w_pb + 4 * pl + 2);
      hn[4 * pl + 3] = own.w + spec::w(w_pb + 4 * pl + 3);
    }
#pragma unroll
    for (int i = 0; i < C; i++)
#pragma unroll
      for (int o = 0; o < C; o++)
        hn[o] = fmaf(spec::w(w_p + i * C + o), acc[i], hn[o]);
    if constexpr (!last)
    {
#pragma unroll
      for (int pl = 0; pl < P; pl++)
        col0[pl * W] = make_float4(hn[4 * pl], hn[4 * pl + 1], hn[4 * pl + 2], hn[4 * pl + 3]);
    }
    else
    {
#pragma unroll
      for (int o = 0; o < C; o++)
        hout[o] = hn[o];
    }
  });

#pragma unroll
  for (int ho = 0; ho < HOUT; ho++)
    headout[ho] = 0.0f;
#pragma unroll
  for (int i = 0; i < C; i++)
#pragma unroll
    for (int ho = 0; ho < HOUT; ho++)
      headout[ho] = fmaf(spec::w(A.head_off + i * HOUT + ho), head[i], headout[ho]);
#pragma unroll
  for (int ho = 0; ho < HOUT; ho++)
    headout[ho] += spec::w(A.head_off + C * HOUT + ho);
}

template <int NT, int FQ>
__device__ __forceinline__ void wavenet_spec_short_body(const SpecParams& p)
{
  constexpr int Q = NT / FQ; // streams per CTA
  static_assert(Q * FQ == NT && (FQ % 32) == 0, "whole warps per stream");
  extern __shared__ float4 spec_smem[]; // [planes][NT]
  const int tid = threadIdx.x;
  const int f = tid % FQ, q = tid / FQ;
  const unsigned long long pol = l2_evict_first_policy();
  for (int slot = blockIdx.x; slot * Q < p.batch; slot += gridDim.x)
  {
    const int stream = slot * Q + q;
    const bool live = stream < p.batch;
    const int sc = min(stream, p.batch - 1);
    float* state = p.state + (size_t)sc * p.state_stride;
    const float xv = (live && f < p.n_frames) ? __ldg(p.in + (size_t)sc * p.in_stride + f) : 0.0f;
    const float x[1] = {xv};
    constexpr int C0 = spec::A[0].C;
    float head0[C0], hout0[C0], ho0[spec::A[0].HOUT];
#pragma unroll
    for (int o = 0; o < C0; o++)
      head0[o] = 0.0f;
    float y;
    array_forward_short<0, spec::NA - 1, NT, FQ>(spec_smem, state, pol, p.t_base, p.n_frames, f, live, x, xv, head0, hout0, ho0);
    if constexpr (spec::NA == 1)
      y = ho0[0];
    else
    {
      constexpr int AI1 = spec::NA - 1;
      constexpr int C1 = spec::A[AI1].C;
      float head1[C1], hout1[C1], ho1[spec::A[AI1].HOUT];
#pragma unroll
      for (int o = 0; o < C1; o++)
        head1[o] = ho0[o];
      __syncthreads(); // (the last layer's tap reads are fenced by its B1; this orders the rechannel's tile stores too)
      array_forward_short<AI1, -1, NT, FQ>(spec_smem, state, pol, p.t_base, p.n_frames, f, live, hout0, xv, head1, hout1, ho1);
      y = ho1[0];
    }
    if (live && f < p.n_frames)
      p.out[(size_t)sc * p.out_stride + f] = spec::head_scale * y;
    __syncthreads(); // the next slot rewrites the tile
  }
}

} // namespace namb200_spec

#ifndef NAMB200_SPEC_NO_KERNEL // (wavenet_lat.cuh includes this file for its helpers only)
#ifndef NAMB200_SPEC_NT
#define NAMB200_SPEC_NT 512
#endif
#ifndef NAMB200_SPEC_S
#define NAMB200_SPEC_S 1
#endif
#ifndef NAMB200_SPEC_MINB
#define NAMB200_SPEC_MINB 2
#endif

// (the entry points are compiled as two NVRTC programs side by side -- jit_spec.cpp: this one and the 64-frame short-call
// variant in the first, the 128- / 256-frame variants in the second, NAMB200_SPEC_ONLY_EXTRA_SHORT)
#ifndef NAMB200_SPEC_ONLY_EXTRA_SHORT
extern "C" __global__ void __launch_bounds__(NAMB200_SPEC_NT, NAMB200_SPEC_MINB)
  wavenet_spec_kernel(const __grid_constant__ namb200_spec::SpecParams p)
{
  namb200_spec::wavenet_spec_body<NAMB200_SPEC_NT, NAMB200_SPEC_S, NAMB200_SPEC_MINB>(p);
}
#endif
#if defined(NAMB200_SPEC_SHORT_FQ) && !defined(NAMB200_SPEC_ONLY_EXTRA_SHORT)
// short-call variant: NAMB200_SPEC_SHORT_NT / NAMB200_SPEC_SHORT_FQ streams per CTA, calls of up to NAMB200_SPEC_SHORT_FQ frames
#ifndef NAMB200_SPEC_SHORT_NT
#define NAMB200_SPEC_SHORT_NT NAMB200_SPEC_NT
#endif
extern "C" __global__ void __launch_bounds__(NAMB200_SPEC_SHORT_NT, 2)
  wavenet_spec_short_kernel(const __grid_constant__ namb200_spec::SpecParams p)
{
  namb200_spec::wavenet_spec_short_body<NAMB200_SPEC_SHORT_NT, NAMB200_SPEC_SHORT_FQ>(p);
}
#endif
// the same for calls of up to 128 / 256 frames (hosts with larger audio buffers): NT / 128 and NT / 256 streams per CTA
#ifdef NAMB200_SPEC_SHORT128_NT
extern "C" __global__ void __launch_bounds__(NAMB200_SPEC_SHORT128_NT, 2)
  wavenet_spec_short128_kernel(const __grid_constant__ namb200_spec::SpecParams p)
{
  namb200_spec::wavenet_spec_short_body<NAMB200_SPEC_SHORT128_NT, 128>(p);
}
#endif
#ifdef NAMB200_SPEC_SHORT256_NT
extern "C" __global__ void __launch_bounds__(NAMB200_SPEC_SHORT256_NT, 2)
  wavenet_spec_short256_kernel(const __grid_constant__ namb200_spec::SpecParams p)
{
  namb200_spec::wavenet_spec_short_body<NAMB200_SPEC_SHORT256_NT, 256>(p);
}
#endif
#endif // NAMB200_SPEC_NO_KERNEL
