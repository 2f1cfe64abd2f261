// k-NN graph, second-generation tensor-core path (sm_100a): TMA-staged fp16 hi/lo planes ->
// tcgen05.mma kind::f16 (three MMAs per k-step: lo.hi + hi.lo + hi.hi, fp32 accumulate in TMEM) ->
// fused per-row top-K epilogue.  Replaces DenseDilatedKnnGraph.forward's pairwise_distance +
// topk + dilation (reference torch_edge.py:7-18, 70-103, 245-255, 270-284) for K = k*d <= 8.
//
// Why fp16 planes: the normalised features are in [-1, 1]; scaled by 2^12 they split exactly into
// hi = fp16(x) and lo = fp16(x - hi) with a residual below 2^-24 |x| (better than the 3xTF32 split,
// whose truncated planes leave 2^-20), every product is exact in the fp32 accumulator, kind::f16
// issues at twice the kind::tf32 rate and the planes are half the bytes in HBM, L2 and shared memory.
//
// Two kernels, one data layout.  A "block" is 128 node rows x 64 channels, hi plane then lo plane
// (2 x 16 KB, each row one 128-byte swizzle line, loaded by one TMA box each).
//
//  * knn_stream_kernel<NH, BN, KREG>: a CTA owns 128*NH query rows of one segment.  Their blocks stay
//    RESIDENT in shared memory for the whole kernel; key blocks (BN keys) stream through a TMA ring.
//    Per key tile the MMA thread fills NH accumulators (one per 128-row query block) of a
//    double-buffered TMEM set (2 * NH * BN columns), so the top-K selection of tile t (4*NH epilogue
//    warps, one accumulator row per thread, no block-level barrier anywhere in the loop) overlaps
//    the MMAs of tile t+1.  NH = 4 / BN = 64 (C <= 64): 512 queries, 16 epilogue warps, L2->smem key
//    traffic 1/6 of the first-generation kernel, which re-streamed the query chunk with every key
//    chunk; NH = 2 / BN = 128 while 2 * C * 256 B of queries fit; NH = 1 for C <= 320.
//  * knn_self_kernel<NH, KREG>: self-graphs (keys == queries) with N <= 128*NH.  One CTA owns the
//    whole segment; every K-chunk is loaded ONCE and used as both MMA operands, all NH*NH
//    accumulators stay live in TMEM (512 columns at NH = 2) and are selected from once at the end.
//    Used where the channel count is too large for resident queries (C = 256 / 512 stages).
#include "tc_ptx.cuh"

#include <cuda_fp16.h>

#include <algorithm>
#include <climits>
#include <cstdlib>
#include <cstring>

namespace grafp {
namespace tc2 {
using namespace tcptx;

constexpr int BM = 128;                       // rows per MMA = UMMA_M = key-tile width = UMMA_N
constexpr int BK = 64;                        // fp16 per K-chunk = one 128-byte swizzle row
constexpr int UMMA_K = 16;                    // kind::f16
constexpr uint32_t kPlaneBytes = BM * BK * 2; // 16 KB
constexpr uint32_t kBlockBytes = 2 * kPlaneBytes;
constexpr int kMaxStages = 8;
constexpr uint32_t kSmemLimit = 232448;       // 227 KB opt-in maximum per CTA
constexpr float kPlaneScale = 4096.f;         // planes hold x_hat * 2^12 (see knn_normalize, mode 3)

// instruction descriptor: D = f32, A = B = f16, both K-major, M = 128, N = BN
template <int BN>
__device__ __forceinline__ constexpr uint32_t make_idesc_f16() {
  return (1u << 4) | (0u << 7) | (0u << 10) | (static_cast<uint32_t>(BN >> 3) << 17) | (static_cast<uint32_t>(BM >> 4) << 24);
}

__device__ __forceinline__ float lds_f32(uint32_t addr) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
  return v;
}

// Per-row running top-K, one accumulator row per thread.  The epilogue is issue-slot bound (one
// row x 128 columns per thread and tile), so the common case must cost as little as possible:
// a key can only enter the list if its raw accumulator exceeds a conservative per-row threshold
// `thr` (one FSETP); the warp votes, and only columns where some lane has a candidate run the
// exact distance D = (|x|^2 + (-2 s)) + |y|^2 (reference association order, torch_edge.py:16-18)
// and the branch-free insertion network (ties keep the earlier = lower key id).
template <int KREG>
struct TopK {
  float d[KREG];
  int id[KREG];
  float sq_i;  // |x_i|^2
  float lo_d;  // K > 16 runs in rounds of 16 ranks: only keys with (dist, id) > (lo_d, lo_id), the last entry of the
  int lo_id;   // previous round, may enter the list (-inf / -1: no bound)
  float base;  // (sq_i + a lower bound of |y_j|^2 over the current key tile - slack) * 2^23
  float thr;   // candidate iff acc > thr
  static constexpr float kHalfScale2 = 0.5f * kPlaneScale * kPlaneScale;
  static constexpr float kM2 = -2.f / (kPlaneScale * kPlaneScale);  // power of two: kM2 * acc is exact
  __device__ __forceinline__ void init(float sq) {
#pragma unroll
    for (int p = 0; p < KREG; ++p) { d[p] = INFINITY; id[p] = 0; }
    sq_i = sq; base = 0.f; thr = -INFINITY; lo_d = -INFINITY; lo_id = -1;
  }
  // dist < d[K-1] implies sq_i + kM2*acc + ymin < d[K-1] + 1e-6 (fp32 evaluation error of dist is < 5e-7 for
  // normalised features); 4e-6 also covers the rounding of this expression itself.
  __device__ __forceinline__ void update_thr() { thr = fmaf(-kHalfScale2, d[KREG - 1], base); }
  __device__ __forceinline__ void set_tile(float ymin) { base = (sq_i + ymin - 4e-6f) * kHalfScale2; update_thr(); }
  __device__ __forceinline__ void insert(float v, int key) {  // select network; no-op unless v < d[K-1]
    bool c[KREG];
#pragma unroll
    for (int p = 0; p < KREG; ++p) c[p] = v < d[p];
#pragma unroll
    for (int p = KREG - 1; p > 0; --p) {  // c[p-1] implies c[p]: shift down, or drop v in, or keep
      d[p] = c[p - 1] ? d[p - 1] : (c[p] ? v : d[p]);
      id[p] = c[p - 1] ? id[p - 1] : (c[p] ? key : id[p]);
    }
    d[0] = c[0] ? v : d[0];
    id[0] = c[0] ? key : id[0];
  }
  // 8 accumulator columns (acc = s * 2^24); |y|^2 of column 0 is at shared address ys_addr (YS_SHARED) or at
  // ys_glob (read through L1 only on the rare candidate path: no staging, no per-tile barrier).
  // The votes of a group of kVoteGroup columns are taken up front against the threshold as of the group
  // start (a stale threshold is only looser, the exact test is redone in `insert`), so the
  // FSETP -> VOTE -> BRA latency chain is paid once per group instead of once per column.  The
  // callers keep this in a rolled loop (8 columns per tcgen05.ld): the unrolled 32-column form was
  // 13 KB of code per tile pass and starved the instruction cache.
  static constexpr int kVoteGroup = 4;
  template <bool YS_SHARED>
  __device__ __forceinline__ void scan8(const uint32_t (&v)[8], uint32_t ys_addr, const float* ys_glob, int nvalid,
                                        int key0) {
#pragma unroll
    for (int j0 = 0; j0 < 8; j0 += kVoteGroup) {
      bool cand[kVoteGroup];
      const float t = thr;
#pragma unroll
      for (int g = 0; g < kVoteGroup; ++g) cand[g] = __any_sync(0xffffffffu, __uint_as_float(v[j0 + g]) > t);
#pragma unroll
      for (int g = 0; g < kVoteGroup; ++g) {
        if (cand[g]) {
          const int j = j0 + g;
          // warp-uniform address; columns past the last key (TMA zero fill) are pushed to +inf
          const float yj = YS_SHARED ? lds_f32(ys_addr + 4 * j) : (j < nvalid ? __ldg(ys_glob + j) : INFINITY);
          const float dist = __fadd_rn(fmaf(kM2, __uint_as_float(v[j]), sq_i), yj);
          insert(dist, key0 + j);  // (the round bounds lo_d / lo_id only exist for K > 16: queue path)
          update_thr();
        }
      }
    }
  }

  // ---- decoupled selection: per-lane candidate queue in shared memory ------------------------------------
  // The vote-gated scan above makes the whole warp pay the insertion path whenever ANY of its 32 rows has a
  // candidate, which is most columns (a row's list changes ~K ln(M/K) times, times 32 rows).  Here the scan is
  // branch-free: per quad of columns, max3/max + one FSETP against the row's (slightly stale) threshold and three
  // predicated instructions that park the four raw accumulators in the lane's own queue (slot s of lane l at
  // q0 + 512 s, q0 = warp base + 16 l: 128-bit accesses of a warp never conflict, whatever the lanes' fill
  // levels) and mark the quad in a per-tile bit mask.  The queue is drained lane-parallel - every lane walks its
  // own entries in push order, so ties still keep the lower key id - at the end of a tile, or earlier when
  // some lane is 4 slots from full.  With thr = -inf at the start everything is pushed, the first 16 columns
  // trigger a drain, and the thresholds tighten from there on their own.
  uint32_t q0, qa, qlim, qmask;
  static constexpr uint32_t kSlotStride = 512;
  __device__ __forceinline__ void queue_init(uint32_t warp_queue, int lane, int slots) {
    q0 = warp_queue + 16u * lane;
    qa = q0;
    qlim = q0 + (uint32_t)(slots - 4) * kSlotStride;
    qmask = 0u;
  }
  __device__ __forceinline__ void push4(uint32_t a, uint32_t b, uint32_t c, uint32_t d, uint32_t bit) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        ".reg .f32 m;\n\t"
        "max.f32 m, %2, %3, %4;\n\t"
        "max.f32 m, m, %5;\n\t"
        "setp.gt.f32 p, m, %6;\n\t"
        "@p st.shared.v4.f32 [%0], {%2, %3, %4, %5};\n\t"
        "@p add.u32 %0, %0, 512;\n\t"
        "@p or.b32 %1, %1, %7;\n\t"
        "}"
        : "+r"(qa), "+r"(qmask)
        : "f"(__uint_as_float(a)), "f"(__uint_as_float(b)), "f"(__uint_as_float(c)), "f"(__uint_as_float(d)), "f"(thr),
          "r"(bit)
        : "memory");
  }
  // key0 = key id of the tile's column 0; keys >= M (TMA zero fill) are skipped.  YS_VEC: the four key norms of a
  // quad are fetched with one 128-bit load next to the queue entry (the key set's norms are 16-byte aligned,
  // M % 4 == 0), so the per-element path has no dependent global load.
  template <bool YS_SHARED, bool YS_VEC>
  __device__ __forceinline__ void drain(int key0, uint32_t ys_addr, const float* ys_glob, int M) {
    uint32_t rd = q0;
    while (__any_sync(0xffffffffu, rd < qa)) {
      if (rd < qa) {
        float v0, v1, v2, v3;
        asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v0), "=f"(v1), "=f"(v2), "=f"(v3) : "r"(rd));
        rd += kSlotStride;
        const int quad = __ffs(qmask) - 1;  // lowest marked quad = oldest entry
        qmask &= qmask - 1u;
        const int key = key0 + 4 * quad;
        float y0 = 0.f, y1 = 0.f, y2 = 0.f, y3 = 0.f;
        if constexpr (YS_SHARED) {
          asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(y0), "=f"(y1), "=f"(y2), "=f"(y3) : "r"(ys_addr + 4u * key));
        } else if constexpr (YS_VEC) {  // key % 4 == 0 and M % 4 == 0: key < M implies key + 3 < M; clamped past the end
          const float4 yv = __ldg(reinterpret_cast<const float4*>(ys_glob + min(key, M - 4)));
          y0 = yv.x; y1 = yv.y; y2 = yv.z; y3 = yv.w;
        }
        if constexpr (YS_SHARED || YS_VEC) {
          // exact distances of the whole quad up front (2 instructions each) and the exact, strict test against the
          // current K-th entry: keys that only TIE with it (duplicate nodes - frequent in real point clouds, where
          // they made this path slower than the vote-gated one) are dropped here instead of walking the insertion
          // path one by one.  An insertion inside the quad only tightens d[K-1]; `insert` re-tests exactly.
          const float e0 = __fadd_rn(fmaf(kM2, v0, sq_i), y0), e1 = __fadd_rn(fmaf(kM2, v1, sq_i), y1);
          const float e2 = __fadd_rn(fmaf(kM2, v2, sq_i), y2), e3 = __fadd_rn(fmaf(kM2, v3, sq_i), y3);
          const float dk = d[KREG - 1];
          uint32_t em = (e0 < dk ? 1u : 0u) | (e1 < dk ? 2u : 0u) | (e2 < dk ? 4u : 0u) | (e3 < dk ? 8u : 0u);
          while (em != 0u) {  // lane-local, in column order; usually one element
            const int e = __ffs(em) - 1;
            em &= em - 1u;
            const float lo2 = (e & 1) ? e1 : e0, hi2 = (e & 1) ? e3 : e2;
            const float dist = (e & 2) ? hi2 : lo2;
            const int kj = key + e;
            if (kj < M && (dist > lo_d || (dist == lo_d && kj > lo_id))) {
              insert(dist, kj);
              update_thr();
            }
          }
        } else {
          uint32_t em = (v0 > thr ? 1u : 0u) | (v1 > thr ? 2u : 0u) | (v2 > thr ? 4u : 0u) | (v3 > thr ? 8u : 0u);
          while (em != 0u) {
            const int e = __ffs(em) - 1;
            em &= em - 1u;
            const float lo2 = (e & 1) ? v1 : v0, hi2 = (e & 1) ? v3 : v2;
            const float s = (e & 2) ? hi2 : lo2;
            const int kj = key + e;
            if (kj < M) {
              const float dist = __fadd_rn(fmaf(kM2, s, sq_i), __ldg(ys_glob + kj));
              if (dist > lo_d || (dist == lo_d && kj > lo_id)) {
                insert(dist, kj);
                update_thr();
              }
            }
          }
        }
      }
    }
    qa = q0;
  }
};

// ---- group-maxima selection (K <= 3, unit-norm keys) ------------------------------------------------------
// The two forms above pay for SIMT divergence: a row's list changes ~K ln(M/K) times over M keys, at different
// columns for each of the 32 rows of a warp, so either the whole warp walks the insertion path for most columns
// (vote) or the lanes queue their candidates and drain them at the pace of the fullest lane (queues): 13 / 9.6
// issued instructions per accumulator entry, against ~10 that a tensor-bound kernel could afford at C = 64.
// Here the scan is branch-free and identical for every lane.  Keys are handled in groups of 8 consecutive columns;
// per group: its maximum raw accumulator (3 FMNMX3 + 1 FMNMX), a K-entry insertion of (maximum, group id) into the
// row's list of the K best GROUP maxima, and - predicated on the group entering that list - a 32-byte spill of the
// group's 8 accumulators into one of K per-row slots in shared memory (the slot of the entry that drops out).
// After the last tile the K best keys of a row lie inside its K listed groups: if key e is among the K best, its
// group's maximum is >= acc_e, so fewer than K groups can precede it.  The 8 K spilled accumulators are then ranked
// exactly - D = (|x_i|^2 + (-2 s)) + |y_j|^2 in the reference's association order, ties to the lower key id - in
// ascending key order.  Ranking groups by the raw accumulator is ranking by distance only while all |y_j|^2 are
// equal, i.e. for unit-norm keys (what DenseDilatedKnnGraph's F.normalize gives); the kernel checks the segment's
// min / max |y|^2 and takes the vote-gated scan for segments with all-zero (or un-normalised) nodes.  Among
// near-ties, picks can differ from the fp32 reference by the spread of the computed |y|^2 around 1 (2.4e-7), well
// inside the documented tie band.  A warp skips a chunk of 32 columns when none of its rows has a group entering
// its list (neighbouring spectrogram peaks find their candidates in the same few columns).
template <int KG>
struct GroupTop {
  static constexpr int kInvalid = 0x00ffffff;
  float gv[KG];    // the KG largest group maxima, descending; ties keep the earlier (lower-id) group in front
  int gm[KG];      // (group id << 3) | spill slot
  uint32_t spill;  // shared address of this thread's slot 0: warp base + 16 * lane; slot s at +1024 s, second half +512
  __device__ __forceinline__ void init(uint32_t warp_spill, int lane) {
#pragma unroll
    for (int p = 0; p < KG; ++p) { gv[p] = -INFINITY; gm[p] = (kInvalid << 3) | p; }
    spill = warp_spill + 16u * lane;
  }
  __device__ __forceinline__ static float max8(const uint32_t* v) {
    float a, b;
    asm("max.f32 %0, %1, %2, %3;" : "=f"(a) : "f"(__uint_as_float(v[0])), "f"(__uint_as_float(v[1])), "f"(__uint_as_float(v[2])));
    asm("max.f32 %0, %1, %2, %3;" : "=f"(b) : "f"(__uint_as_float(v[3])), "f"(__uint_as_float(v[4])), "f"(__uint_as_float(v[5])));
    asm("max.f32 %0, %1, %2, %3;" : "=f"(a) : "f"(a), "f"(__uint_as_float(v[6])), "f"(__uint_as_float(v[7])));
    return fmaxf(a, b);
  }
  // group `gid` with maximum m and accumulators v[0..7]
  __device__ __forceinline__ void offer(float m, int gid, const uint32_t* v) {
    bool c[KG];
#pragma unroll
    for (int p = 0; p < KG; ++p) c[p] = m > gv[p];
    const int slot = gm[KG - 1] & 7;
    if (c[KG - 1]) {
      const uint32_t a = spill + (uint32_t)slot * 1024u;
      asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]) : "memory");
      asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a + 512u), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]) : "memory");
    }
    const int meta = (gid << 3) | slot;
#pragma unroll
    for (int p = KG - 1; p > 0; --p) {
      gv[p] = c[p - 1] ? gv[p - 1] : (c[p] ? m : gv[p]);
      gm[p] = c[p - 1] ? gm[p - 1] : (c[p] ? meta : gm[p]);
    }
    gv[0] = c[0] ? m : gv[0];
    gm[0] = c[0] ? meta : gm[0];
  }
  // one 32-column chunk of this thread's accumulator row; key0 = key id of column 0 (a multiple of 8)
  __device__ __forceinline__ void scan32(const uint32_t (&v)[32], int key0) {
    float m[4];
#pragma unroll
    for (int g = 0; g < 4; ++g) m[g] = max8(&v[8 * g]);
    float mm;
    asm("max.f32 %0, %1, %2, %3;" : "=f"(mm) : "f"(m[0]), "f"(m[1]), "f"(m[2]));
    mm = fmaxf(mm, m[3]);
    if (__any_sync(0xffffffffu, mm > gv[KG - 1])) {
#pragma unroll
      for (int g = 0; g < 4; ++g) offer(m[g], (key0 >> 3) + g, &v[8 * g]);
    }
  }
  // exact ranking of the listed groups' keys into `top` (ascending key order, so ties keep the lower id).
  // RAGGED: the key count `nkeys` need not be a multiple of 32; columns past it were masked to -inf before `scan32`
  // (so their distance is +inf) and their |y|^2 is not read.
  template <int KREG, bool YS_SHARED, bool RAGGED = false>
  __device__ __forceinline__ void finish(TopK<KREG>& top, uint32_t ys_addr, const float* ys_glob, int nkeys = 0) {
#pragma unroll
    for (int i = 0; i < KG - 1; ++i) {  // sort by group id (the slot bits cannot reorder distinct ids)
#pragma unroll
      for (int p = 0; p < KG - 1 - i; ++p) {
        const int lo = min(gm[p], gm[p + 1]), hi = max(gm[p], gm[p + 1]);
        gm[p] = lo; gm[p + 1] = hi;
      }
    }
#pragma unroll
    for (int p = 0; p < KG; ++p) {
      const int gid = gm[p] >> 3;
      if (gid == kInvalid) continue;
      const uint32_t a = spill + (uint32_t)(gm[p] & 7) * 1024u;
      float acc[8], y[8];
      asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(acc[0]), "=f"(acc[1]), "=f"(acc[2]), "=f"(acc[3]) : "r"(a));
      asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(acc[4]), "=f"(acc[5]), "=f"(acc[6]), "=f"(acc[7]) : "r"(a + 512u));
      if constexpr (YS_SHARED) {
        asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(y[0]), "=f"(y[1]), "=f"(y[2]), "=f"(y[3]) : "r"(ys_addr + 32u * gid));
        asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(y[4]), "=f"(y[5]), "=f"(y[6]), "=f"(y[7]) : "r"(ys_addr + 32u * gid + 16u));
      } else if (RAGGED && 8 * gid + 8 > nkeys) {
#pragma unroll
        for (int e = 0; e < 8; ++e) y[e] = (8 * gid + e < nkeys) ? __ldg(ys_glob + 8 * gid + e) : 0.f;
      } else {
        const float4 y0 = __ldg(reinterpret_cast<const float4*>(ys_glob + 8 * gid));
        const float4 y1 = __ldg(reinterpret_cast<const float4*>(ys_glob + 8 * gid) + 1);
        y[0] = y0.x; y[1] = y0.y; y[2] = y0.z; y[3] = y0.w; y[4] = y1.x; y[5] = y1.y; y[6] = y1.z; y[7] = y1.w;
      }
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const float dist = __fadd_rn(fmaf(TopK<KREG>::kM2, acc[e], top.sq_i), y[e]);
        top.insert(dist, 8 * gid + e);
      }
    }
  }
};

// bytes of per-warp epilogue scratch: candidate queues (QS > 0), group spill slots (QS < 0), none (vote-gated scan)
template <int QS, int KREG>
__host__ __device__ constexpr uint32_t epi_warp_bytes() {
  return QS > 0 ? (uint32_t)QS * 512u : (QS < 0 ? (uint32_t)KREG * 1024u : 0u);
}
constexpr float kUnitNormTol = 1e-4f;  // group-maxima selection needs | |y|^2 - 1 | below this for every key of the segment
// The flat search also bounds the spread of |y|^2 over the slice: ranking groups by the raw accumulator misorders two keys
// by at most that spread, and 1e-6 keeps it below the fp32 tie band 4 sqrt(d) 2^-23 (3.8e-6 at d = 64) that exact search
// is held to.  Normalised fp32 rows spread by a few 1e-7.
constexpr float kSearchUnitSpread = 1e-6f;

__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&v)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
               : "r"(taddr));
}

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
      : "r"(taddr));
}

// One tile (<= 128 accumulator columns, ncols of them backed by keys) of this thread's row through the
// candidate queue: 16 columns per tcgen05.ld, four predicated quad pushes, one vote for the early drain.
// (Software-pipelining the loads over two register sets was measured: 378 -> 390 us at stage 0, the extra 16
// registers cost more than the exposed TMEM latency.)
template <int KREG, bool YS_SHARED, bool YS_VEC>
__device__ __forceinline__ void scan_tile_queued(TopK<KREG>& top, uint32_t trow, int key0, int ncols, uint32_t ys_addr,
                                                 const float* ys_glob, int M) {
  uint32_t bq = 1u;
#pragma unroll 1
  for (int c0 = 0; c0 < ncols; c0 += 16) {
    uint32_t v[16];
    tmem_ld16(trow + c0, v);
    tmem_ld_wait();
    top.push4(v[0], v[1], v[2], v[3], bq);
    top.push4(v[4], v[5], v[6], v[7], bq << 1);
    top.push4(v[8], v[9], v[10], v[11], bq << 2);
    top.push4(v[12], v[13], v[14], v[15], bq << 3);
    bq <<= 4;
    if (c0 + 16 >= ncols || __any_sync(0xffffffffu, top.qa >= top.qlim)) top.template drain<YS_SHARED, YS_VEC>(key0, ys_addr, ys_glob, M);
  }
}

// ranks rank0 .. rank0 + KREG - 1 of the row's list; every `stride`-th global rank is written (dilation fused)
template <int KREG>
__device__ __forceinline__ void emit(const TopK<KREG>& top, long long* nn_idx, int* nn_idx32, long long o, int k_out, int stride,
                                     int rank0) {
#pragma unroll
  for (int p = 0; p < KREG; ++p) {
    const int g = rank0 + p;
    const int slot = g / stride;
    if (g - slot * stride == 0 && slot < k_out) {
      nn_idx[o + slot] = top.id[p];
      if (nn_idx32 != nullptr) nn_idx32[o + slot] = top.id[p];
    }
  }
}

// round hand-over: the last list entry of round r is the exclusive lower bound of round r + 1
template <int KREG>
__device__ __forceinline__ void load_bound(TopK<KREG>& top, const float2* bounds, long long row, int rank0) {
  if (bounds != nullptr && rank0 > 0) {
    const float2 v = bounds[row];
    top.lo_d = v.x;
    top.lo_id = __float_as_int(v.y);
  }
}
template <int KREG>
__device__ __forceinline__ void store_bound(const TopK<KREG>& top, float2* bounds, long long row, int more_rounds) {
  if (bounds != nullptr && more_rounds) bounds[row] = make_float2(top.d[KREG - 1], __int_as_float(top.id[KREG - 1]));
}

// One thread of the warp, chosen by elect.sync.  Unlike `lane == 0`, ptxas knows the branch it guards holds a single
// thread, so the uniform-datapath instructions inside (UTCHMMA, UTMALDG) need no per-instruction "which threads are
// active" loop: the MMA-issuing thread went from ~12 to ~4 issued instructions per tcgen05.mma - it was pacing the
// tensor pipe (48 MMAs of 32 cycles per key tile against ~580 dependent single-thread instructions).
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t"
      "}"
      : "=r"(pred));
  return pred != 0;
}

// Shared-memory matrix descriptors differ only in their 14-bit start-address field (low word, 16-byte units): the
// loops carry the low word and add offsets to it instead of rebuilding the 64-bit descriptor per MMA.
__device__ __forceinline__ uint32_t desc_lo(uint32_t addr) { return ((addr & 0x3FFFFu) >> 4) | (1u << 16); }
__device__ __forceinline__ uint64_t desc_of(uint32_t lo) {
  // high word: stride byte offset 1024 >> 4 (bits 32-45), descriptor version 1 (bit 46), SWIZZLE_128B (bits 61-63)
  return (static_cast<uint64_t>((1024u >> 4) | (1u << 14) | (2u << 29)) << 32) | lo;
}

// three MMAs per 16-channel step over one 64-channel block pair (A block: 128 rows, B block: BN rows);
// a_lo0 / b_lo0: descriptor low words of the blocks' hi planes
template <int BN>
__device__ __forceinline__ void mma_block(uint32_t acc, uint32_t a_lo0, uint32_t b_lo0, bool first) {
  constexpr uint32_t idesc = make_idesc_f16<BN>();
  constexpr uint32_t kAPlane16 = kPlaneBytes >> 4, kBPlane16 = (BN * BK * 2) >> 4, kStep16 = (UMMA_K * 2) >> 4;
#pragma unroll
  for (int kk = 0; kk < BK / UMMA_K; ++kk) {
    const uint64_t a_hi = desc_of(a_lo0 + kk * kStep16), a_lo = desc_of(a_lo0 + kAPlane16 + kk * kStep16);
    const uint64_t b_hi = desc_of(b_lo0 + kk * kStep16), b_lo = desc_of(b_lo0 + kBPlane16 + kk * kStep16);
    umma_f16(acc, a_lo, b_hi, idesc, (first && kk == 0) ? 0u : 1u);
    umma_f16(acc, a_hi, b_lo, idesc, 1u);
    umma_f16(acc, a_hi, b_hi, idesc, 1u);
  }
}

__device__ __forceinline__ void tmem_alloc(uint32_t* slot, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(slot)), "r"(cols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t base, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(base), "r"(cols) : "memory");
}

// ---------------------------------------------------------------------------------------------
// resident queries, streamed keys
// ---------------------------------------------------------------------------------------------
// SPLIT (the flat search, B = 1): blockIdx.y selects the key slice [s0, s0 + slice_len) of the database.  Key ids, the
// |y|^2 range test and the round bounds (per slice and query) are slice-local, and instead of `emit` the epilogue
// writes the row's best (distance, slice-local id) pairs of ranks rank0 .. to part[(slice * N + q) * k_out + rank]
// for the merge kernel.
template <int NH, int BN, int KREG, int QS, bool SPLIT = false>
__global__ void __launch_bounds__((4 * NH + 2) * 32, 1)
knn_stream_kernel(const __grid_constant__ CUtensorMap tm_x_hi, const __grid_constant__ CUtensorMap tm_x_lo,
                  const __grid_constant__ CUtensorMap tm_y_hi, const __grid_constant__ CUtensorMap tm_y_lo,
                  const float* __restrict__ xsq, const float* __restrict__ ysq, long long* __restrict__ nn_idx,
                  int* __restrict__ nn_idx32, int N, int M, int C, int k_out, int stride, int stages,
                  float2* bounds, int rank0, int more_rounds, int slice_len, float2* __restrict__ part) {
  constexpr int kProducerWarp = 4 * NH, kMmaWarp = 4 * NH + 1;
  constexpr uint32_t kTmemCols = 2 * NH * BN;  // two accumulator sets of NH tiles, BN keys wide
  constexpr uint32_t kKeyBlockBytes = 2 * BN * BK * 2;  // hi + lo plane of BN keys x 64 channels
  extern __shared__ unsigned char smem_raw[];
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int num_kc = (C + BK - 1) / BK;
  int s0 = 0;  // first key of this CTA's slice; M becomes the slice's key count
  if constexpr (SPLIT) {
    s0 = blockIdx.y * slice_len;
    M = min(slice_len, M - s0);
    ysq += s0;
  }
  const int num_tiles = (M + BN - 1) / BN;
  unsigned char* q_base = smem;                                    // [NH][num_kc] blocks
  unsigned char* ring = q_base + (size_t)NH * num_kc * kBlockBytes; // [stages] blocks
  unsigned char* queue = ring + (size_t)stages * kKeyBlockBytes;      // per-warp epilogue scratch (queues / spill slots)
  uint64_t* bars = reinterpret_cast<uint64_t*>(queue + (size_t)(4 * NH) * epi_warp_bytes<QS, KREG>());
  const uint32_t bar_full = smem_u32(bars);
  const uint32_t bar_empty = bar_full + 8 * kMaxStages;
  const uint32_t bar_tfull = bar_empty + 8 * kMaxStages;
  const uint32_t bar_tempty = bar_tfull + 16;
  const uint32_t bar_q = bar_tempty + 16;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kMaxStages + 5);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int b = SPLIT ? 0 : blockIdx.y;
  const int m0 = blockIdx.x * (BM * NH);

  if (threadIdx.x == 0) {
    for (int s = 0; s < stages; ++s) { mbar_init(bar_full + 8 * s, 1); mbar_init(bar_empty + 8 * s, 1); }
    for (int a = 0; a < 2; ++a) { mbar_init(bar_tfull + 8 * a, 1); mbar_init(bar_tempty + 8 * a, 4 * NH); }
    mbar_init(bar_q, 1);
    fence_barrier_init();
  }
  if (warp == kMmaWarp) tmem_alloc(tmem_slot, kTmemCols);
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == kProducerWarp) {
    if (elect_one()) {
      // resident query blocks: one barrier, NH * num_kc * 2 boxes
      mbar_arrive_expect_tx(bar_q, (uint32_t)(NH * num_kc) * kBlockBytes);
      for (int h = 0; h < NH; ++h) {
        for (int c = 0; c < num_kc; ++c) {
          const uint32_t dst = smem_u32(q_base + (size_t)(h * num_kc + c) * kBlockBytes);
          tma_load_3d(dst, &tm_x_hi, bar_q, c * BK, m0 + h * BM, b);
          tma_load_3d(dst + kPlaneBytes, &tm_x_lo, bar_q, c * BK, m0 + h * BM, b);
        }
      }
      int s = 0;
      uint32_t ph = 0;
      for (int t = 0; t < num_tiles; ++t) {
        for (int c = 0; c < num_kc; ++c) {
          mbar_wait(bar_empty + 8 * s, ph ^ 1);
          const uint32_t full = bar_full + 8 * s;
          mbar_arrive_expect_tx(full, kKeyBlockBytes);
          const uint32_t dst = smem_u32(ring + (size_t)s * kKeyBlockBytes);
          tma_load_3d(dst, &tm_y_hi, full, c * BK, s0 + t * BN, b);
          tma_load_3d(dst + kKeyBlockBytes / 2, &tm_y_lo, full, c * BK, s0 + t * BN, b);
          if (++s == stages) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == kMmaWarp) {
    if (elect_one()) {
      mbar_wait(bar_q, 0);
      tcgen05_fence_after();
      int s = 0;
      uint32_t ph = 0;
      const uint32_t q_lo0 = desc_lo(smem_u32(q_base)), ring_lo0 = desc_lo(smem_u32(ring));
      for (int t = 0; t < num_tiles; ++t) {
        const int as = t & 1;
        mbar_wait(bar_tempty + 8 * as, ((t >> 1) & 1) ^ 1);  // the epilogue has drained this accumulator set
        tcgen05_fence_after();
        for (int c = 0; c < num_kc; ++c) {
          mbar_wait(bar_full + 8 * s, ph);
          tcgen05_fence_after();
          const uint32_t b_lo0 = ring_lo0 + (uint32_t)s * (kKeyBlockBytes >> 4);
#pragma unroll
          for (int h = 0; h < NH; ++h) {
            const uint32_t a_lo0 = q_lo0 + (uint32_t)(h * num_kc + c) * (kBlockBytes >> 4);
            mma_block<BN>(tmem_base + (as * NH + h) * BN, a_lo0, b_lo0, c == 0);
          }
          tcgen05_commit(bar_empty + 8 * s);  // frees the ring slot when these MMAs retire
          if (++s == stages) { s = 0; ph ^= 1; }
        }
        tcgen05_commit(bar_tfull + 8 * as);
      }
    }
  } else {
    // ===== epilogue: warp w reads TMEM lanes 32*(w%4).., accumulator tile h = w/4 =====
    const int h = warp >> 2;
    const int quarter = warp & 3;
    const int r = quarter * 32 + lane;
    const int q = m0 + h * BM + r;
    // SPLIT: n_q need not fill the query block.  A padding row (TMA zero fill: acc = 0) with |x|^2 = 0 would have a
    // negative threshold once its list is full and take every key as a candidate, pacing its warp and, through the
    // TMEM release, the CTA; |x|^2 = +inf makes its threshold NaN, so it never has one.
    const float sq_i = (q < N) ? xsq[(long long)b * N + q] : (SPLIT ? INFINITY : 0.f);
    const float* ysq_b = ysq + (long long)b * M;
    const bool ys_vec = (M & 3) == 0 && (reinterpret_cast<uintptr_t>(ysq) & 15) == 0;
    TopK<KREG> top;
    top.init(sq_i);
    if constexpr (SPLIT) {
      if (q < N) load_bound<KREG>(top, bounds, (long long)blockIdx.y * N + q, rank0);  // round bounds per (slice, query)
    } else {
      if (q < N) load_bound<KREG>(top, bounds, (long long)b * N + q, rank0);
    }
    if constexpr (QS > 0) top.queue_init(smem_u32(queue) + (uint32_t)warp * (QS * 512), lane, QS);
    GroupTop<(QS < 0) ? KREG : 1> gt;
    if constexpr (QS < 0) gt.init(smem_u32(queue) + (uint32_t)warp * epi_warp_bytes<QS, KREG>(), lane);
    // one threshold base per segment: min over all keys of |y|^2 (1 for normalised rows, 0 for all-zero rows)
    bool unit_keys = false;
    {
      float mn = INFINITY, mx = -INFINITY;
      for (int i = lane; i < M; i += 32) { const float yv = __ldg(ysq_b + i); mn = fminf(mn, yv); mx = fmaxf(mx, yv); }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
        mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
      }
      top.set_tile(mn);
      unit_keys = mn >= 1.f - kUnitNormTol && mx <= 1.f + kUnitNormTol;  // warp- and CTA-uniform (same keys for all)
      if constexpr (SPLIT) unit_keys = unit_keys && mx - mn <= kSearchUnitSpread;
    }
    for (int t = 0; t < num_tiles; ++t) {
      const int as = t & 1;
      mbar_wait(bar_tfull + 8 * as, (t >> 1) & 1);
      tcgen05_fence_after();
      const uint32_t trow = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + (as * NH + h) * BN;
      // keys past M were zero-filled by TMA (acc = 0) and would read |y|^2 out of bounds: stop at M
      const int ncols = min(BN, M - t * BN);
      if constexpr (QS > 0) {
        if (ys_vec) scan_tile_queued<KREG, false, true>(top, trow, t * BN, ncols, 0u, ysq_b, M);
        else scan_tile_queued<KREG, false, false>(top, trow, t * BN, ncols, 0u, ysq_b, M);
      } else {
        if (QS < 0 && unit_keys) {  // group maxima (the host guarantees M % 32 == 0 for this form)
#pragma unroll 1
          for (int c0 = 0; c0 < ncols; c0 += 32) {
            uint32_t v[32];
            tmem_ld32(trow + c0, v);
            tmem_ld_wait();
            if constexpr (SPLIT) {  // the ragged last slice: TMA zero-filled columns (acc = 0) must not rank as groups
              if (c0 + 32 > ncols) {
#pragma unroll
                for (int j = 0; j < 32; ++j) v[j] = (c0 + j < ncols) ? v[j] : 0xff800000u;
              }
            }
            gt.scan32(v, t * BN + c0);
          }
        } else {
#pragma unroll 1
          for (int cc = 0; cc * 8 < ncols; ++cc) {
            uint32_t v[8];
            tmem_ld8(trow + cc * 8, v);
            tmem_ld_wait();
            top.template scan8<false>(v, 0u, ysq_b + t * BN + cc * 8, ncols - cc * 8, t * BN + cc * 8);
          }
        }
      }
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_tempty + 8 * as);
    }
    if constexpr (QS < 0) {
      if (unit_keys) gt.template finish<KREG, false, SPLIT>(top, 0u, ysq_b, M);
    }
    if (q < N) {
      if constexpr (SPLIT) {
        const long long row = (long long)blockIdx.y * N + q;
        float2* out = part + row * k_out;
#pragma unroll
        for (int p = 0; p < KREG; ++p)
          if (rank0 + p < k_out) out[rank0 + p] = make_float2(top.d[p], __int_as_float(top.id[p]));
        store_bound<KREG>(top, bounds, row, more_rounds);
      } else {
        emit<KREG>(top, nn_idx, nn_idx32, ((long long)b * N + q) * k_out, k_out, stride, rank0);
        store_bound<KREG>(top, bounds, (long long)b * N + q, more_rounds);
      }
    }
  }

  tcgen05_fence_before();
  __syncthreads();
  if (warp == kMmaWarp) {
    tcgen05_fence_after();
    tmem_dealloc(tmem_base, kTmemCols);
  }
}

// ---------------------------------------------------------------------------------------------
// self-graph of a whole segment per CTA: every chunk loaded once, used as both operands
// ---------------------------------------------------------------------------------------------
template <int NH, int KREG, int QS>
__global__ void __launch_bounds__((4 * NH + 2) * 32, (NH == 1) ? 2 : 1)
knn_self_kernel(const __grid_constant__ CUtensorMap tm_x_hi, const __grid_constant__ CUtensorMap tm_x_lo,
                const float* __restrict__ xsq, long long* __restrict__ nn_idx, int* __restrict__ nn_idx32, int B, int N, int C,
                int k_out, int stride, int stages, float2* bounds, int rank0, int more_rounds) {
  // PERSISTENT over segments b = blockIdx.x, blockIdx.x + gridDim.x, ...: the producer keeps the TMA ring full across
  // segment boundaries, so the 256 KB load of segment i + 1 overlaps the MMAs and the selection of segment i (with one
  // CTA per segment the load, the MMAs and the selection of a segment ran back to back and nothing overlapped them:
  // 512 TMEM columns at NH = 2 allow one CTA per SM).  The accumulators are single-buffered: the MMA thread waits for
  // the epilogue's "TMEM drained" arrival before the first MMA of the next segment.
  constexpr int kEpilogueThreads = 128 * NH;
  constexpr int kProducerWarp = 4 * NH, kMmaWarp = 4 * NH + 1;
  constexpr uint32_t kTmemCols = NH * NH * BM;
  constexpr uint32_t kStageBytes = NH * kBlockBytes;
  extern __shared__ unsigned char smem_raw[];
  unsigned char* smem = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int num_kc = (C + BK - 1) / BK;
  unsigned char* ring = smem;
  unsigned char* queue = ring + (size_t)stages * kStageBytes;                     // per-warp epilogue scratch
  float* ysq_s = reinterpret_cast<float*>(queue + (size_t)(4 * NH) * epi_warp_bytes<QS, KREG>());  // [NH * BM]
  float* ymin_s = ysq_s + NH * BM;                                               // [4 * NH] minima, [4 * NH] maxima
  uint64_t* bars = reinterpret_cast<uint64_t*>(ymin_s + 16);
  const uint32_t bar_full = smem_u32(bars);
  const uint32_t bar_empty = bar_full + 8 * kMaxStages;
  const uint32_t bar_tfull = bar_empty + 8 * kMaxStages;
  const uint32_t bar_tempty = bar_tfull + 8;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kMaxStages + 2);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (threadIdx.x == 0) {
    for (int s = 0; s < stages; ++s) { mbar_init(bar_full + 8 * s, 1); mbar_init(bar_empty + 8 * s, 1); }
    mbar_init(bar_tfull, 1);
    mbar_init(bar_tempty, 4 * NH);
    fence_barrier_init();
  }
  if (warp == kMmaWarp) tmem_alloc(tmem_slot, kTmemCols);
  tcgen05_fence_before();
  __syncthreads();
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == kProducerWarp) {
    if (elect_one()) {
      int s = 0;
      uint32_t ph = 0;
      for (int b = blockIdx.x; b < B; b += gridDim.x) {
        for (int c = 0; c < num_kc; ++c) {
          mbar_wait(bar_empty + 8 * s, ph ^ 1);
          const uint32_t full = bar_full + 8 * s;
          mbar_arrive_expect_tx(full, kStageBytes);
#pragma unroll
          for (int h = 0; h < NH; ++h) {
            const uint32_t dst = smem_u32(ring + (size_t)s * kStageBytes + h * kBlockBytes);
            tma_load_3d(dst, &tm_x_hi, full, c * BK, h * BM, b);
            tma_load_3d(dst + kPlaneBytes, &tm_x_lo, full, c * BK, h * BM, b);
          }
          if (++s == stages) { s = 0; ph ^= 1; }
        }
      }
    }
  } else if (warp == kMmaWarp) {
    if (elect_one()) {
      int s = 0;
      uint32_t ph = 0, it = 0;
      const uint32_t ring_lo0 = desc_lo(smem_u32(ring));
      for (int b = blockIdx.x; b < B; b += gridDim.x, ++it) {
        mbar_wait(bar_tempty, (it & 1) ^ 1);  // the previous segment's accumulators are drained (first trip: passes)
        tcgen05_fence_after();
        for (int c = 0; c < num_kc; ++c) {
          mbar_wait(bar_full + 8 * s, ph);
          tcgen05_fence_after();
          const uint32_t stage = ring_lo0 + (uint32_t)s * (kStageBytes >> 4);
#pragma unroll
          for (int h = 0; h < NH; ++h) {
#pragma unroll
            for (int t = 0; t < NH; ++t) {
              mma_block<BM>(tmem_base + (h * NH + t) * BM, stage + h * (kBlockBytes >> 4), stage + t * (kBlockBytes >> 4), c == 0);
            }
          }
          tcgen05_commit(bar_empty + 8 * s);
          if (++s == stages) { s = 0; ph ^= 1; }
        }
        tcgen05_commit(bar_tfull);
      }
    }
  } else {
    const int h = warp >> 2;
    const int quarter = warp & 3;
    const int r = quarter * 32 + lane;
    const int q = h * BM + r;
    const uint32_t trow = tmem_base + (static_cast<uint32_t>(quarter * 32) << 16) + (h * NH) * BM;
    const uint32_t ys_addr = smem_u32(ysq_s);
    uint32_t it = 0;
    for (int b = blockIdx.x; b < B; b += gridDim.x, ++it) {
      const float* xsq_b = xsq + (long long)b * N;
      const float sq_i = (q < N) ? xsq_b[q] : 0.f;
      {  // kEpilogueThreads == NH * BM: one key norm per thread, per-warp minima / maxima for the candidate threshold
        const bool real = threadIdx.x < N;
        const float yv = real ? xsq_b[threadIdx.x] : INFINITY;
        float mn = yv, mx = real ? yv : -INFINITY;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
          mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        }
        asm volatile("bar.sync 1, %0;" ::"n"(kEpilogueThreads) : "memory");  // the previous segment's readers are done
        ysq_s[threadIdx.x] = yv;
        if (lane == 0) { ymin_s[warp] = mn; ymin_s[8 + warp] = mx; }
      }
      asm volatile("bar.sync 1, %0;" ::"n"(kEpilogueThreads) : "memory");
      TopK<KREG> top;
      top.init(sq_i);
      if (q < N) load_bound<KREG>(top, bounds, (long long)b * N + q, rank0);
      bool unit_keys = false;
      {
        float mn = ymin_s[0], mx = ymin_s[8];
#pragma unroll
        for (int w = 1; w < 4 * NH; ++w) { mn = fminf(mn, ymin_s[w]); mx = fmaxf(mx, ymin_s[8 + w]); }
        top.set_tile(mn);
        unit_keys = mn >= 1.f - kUnitNormTol && mx <= 1.f + kUnitNormTol;
      }
      mbar_wait(bar_tfull, it & 1);
      tcgen05_fence_after();
      if constexpr (QS > 0) {
        top.queue_init(smem_u32(queue) + (uint32_t)warp * (QS * 512), lane, QS);
#pragma unroll 1
        for (int t = 0; t < NH; ++t) {
          const int ncols = min(BM, N - t * BM);
          if (ncols > 0) scan_tile_queued<KREG, true, false>(top, trow + t * BM, t * BM, ncols, ys_addr, nullptr, N);
        }
      } else if (QS < 0 && unit_keys) {  // group maxima (the host guarantees N % 32 == 0 for this form)
        GroupTop<(QS < 0) ? KREG : 1> gt;
        gt.init(smem_u32(queue) + (uint32_t)warp * epi_warp_bytes<QS, KREG>(), lane);
#pragma unroll 1
        for (int c0 = 0; c0 < N; c0 += 32) {
          uint32_t v[32];
          tmem_ld32(trow + c0, v);
          tmem_ld_wait();
          gt.scan32(v, c0);
        }
        // every accumulator this thread needs is in registers / its spill slots: release TMEM before the exact ranking
        tcgen05_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar_tempty);
        gt.template finish<KREG, true>(top, ys_addr, nullptr);
      } else {
#pragma unroll 1
        for (int cc = 0; cc < NH * BM / 8; ++cc) {
          uint32_t v[8];
          tmem_ld8(trow + cc * 8, v);
          tmem_ld_wait();
          top.template scan8<true>(v, ys_addr + cc * 32, nullptr, 8, cc * 8);
        }
      }
      if (!(QS < 0 && unit_keys)) {
        tcgen05_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar_tempty);
      }
      if (q < N) {
        emit<KREG>(top, nn_idx, nn_idx32, ((long long)b * N + q) * k_out, k_out, stride, rank0);
        store_bound<KREG>(top, bounds, (long long)b * N + q, more_rounds);
      }
    }
  }

  tcgen05_fence_before();
  __syncthreads();
  if (warp == kMmaWarp) {
    tcgen05_fence_after();
    tmem_dealloc(tmem_base, kTmemCols);
  }
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
// (rows x C) fp16 matrix per segment, box = 128 rows x 64 channels, 128B swizzle, zero fill out of bounds
static bool make_map_f16(CUtensorMap* map, const void* base, int B, int rows, int C, int box_rows = BM) {
  EncodeTiledFn fn = encode_tiled_fn();
  if (fn == nullptr) return false;
  const cuuint64_t dims[3] = {(cuuint64_t)C, (cuuint64_t)rows, (cuuint64_t)B};
  const cuuint64_t strides[2] = {(cuuint64_t)C * 2, (cuuint64_t)rows * C * 2};
  const cuuint32_t box[3] = {(cuuint32_t)BK, (cuuint32_t)box_rows, 1};
  const cuuint32_t estr[3] = {1, 1, 1};
  const CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, const_cast<void*>(base), dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS;
}

constexpr uint32_t kMiscBytes = 2 * BM * 4 + 64 + (2 * kMaxStages + 8) * 8 + 1024;  // ysq, barriers + TMEM slot, alignment slack

template <typename Kernel>
static int set_smem(Kernel kernel, DeviceOnce* once, const char* what) {
  if (!once->pending()) return GRAFP_OK;
  cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemLimit);
  if (e != cudaSuccess) { set_error("cudaFuncSetAttribute(%s): %s", what, cudaGetErrorString(e)); return (int)e; }
  once->mark();
  return GRAFP_OK;
}

constexpr int kQueueSlots = 6;  // candidate-queue depth per epilogue thread (16-byte quads); 0 selects the vote-gated scan
constexpr bool kGroupMaxDefault = true;  // option knn_epilogue = 0 (auto): take the group-maxima selection where it applies

struct Round {
  float2* bounds;
  int rank0, more;
};

// key slices of the flat search (SPLIT kernels): `count` slices of `len` keys, the last one ragged
struct Slices {
  int count = 0, len = 0;
  float2* part = nullptr;
};

template <int NH, int BN, int KREG, int QS, bool SPLIT>
static int launch_stream(const CUtensorMap& xh, const CUtensorMap& xl, const CUtensorMap& yh, const CUtensorMap& yl,
                         const float* xsq, const float* ysq, long long* nn_idx, int* nn_idx32, int B, int N, int M, int C,
                         int k_out, int stride, int stages, Round r, Slices sl, cudaStream_t s) {
  static DeviceOnce once;
  if (int rc = set_smem(knn_stream_kernel<NH, BN, KREG, QS, SPLIT>, &once, "knn_stream")) return rc;
  const int num_kc = (C + BK - 1) / BK;
  const size_t smem = (size_t)(NH * num_kc) * kBlockBytes + (size_t)stages * (2 * BN * BK * 2) +
                      (size_t)(4 * NH) * epi_warp_bytes<QS, KREG>() + kMiscBytes;
  // query blocks along x (the fastest launch index): the CTAs that share a key slice run in the same wave
  dim3 grid((N + BM * NH - 1) / (BM * NH), SPLIT ? sl.count : B);
  knn_stream_kernel<NH, BN, KREG, QS, SPLIT><<<grid, (4 * NH + 2) * 32, smem, s>>>(
      xh, xl, yh, yl, xsq, ysq, nn_idx, nn_idx32, N, M, C, k_out, stride, stages, r.bounds, r.rank0, r.more, sl.len, sl.part);
  return check_launch(SPLIT ? "knn_search" : "knn_stream");
}

template <int NH, int KREG, int QS>
static int launch_self(const CUtensorMap& xh, const CUtensorMap& xl, const float* xsq, long long* nn_idx, int* nn_idx32,
                       int B, int N, int C, int k_out, int stride, int stages, Round r, cudaStream_t s) {
  static DeviceOnce once;
  if (int rc = set_smem(knn_self_kernel<NH, KREG, QS>, &once, "knn_self")) return rc;
  const size_t smem = (size_t)stages * NH * kBlockBytes + (size_t)(4 * NH) * epi_warp_bytes<QS, KREG>() + kMiscBytes;
  // persistent: one CTA (NH = 2; 512 TMEM columns) or two (NH = 1) per SM, each walking segments blockIdx.x, + gridDim.x, ...
  int grid = num_sms() * (NH == 1 ? 2 : 1);
  if (grid > B) grid = B;
  knn_self_kernel<NH, KREG, QS><<<grid, (4 * NH + 2) * 32, smem, s>>>(xh, xl, xsq, nn_idx, nn_idx32, B, N, C, k_out, stride, stages,
                                                                  r.bounds, r.rank0, r.more);
  return check_launch("knn_self");
}

// Kernel configuration for one shape.  kind: 0 unsupported, 1 self, 2 stream.
struct Plan {
  int kind = 0, nh = 0, bn = 0, stages = 0, qs = 0;
};

static Plan plan_with(int N, int C, bool self, int qs);

static Plan plan(int N, int M, int C, int K, int dtype, bool self) {
  // (dtype: the planes are fp16 whatever the input was - the normalise kernel reads fp32 or bf16 rows)
  if ((dtype != GRAFP_F32 && dtype != GRAFP_BF16) || C % 8 != 0 || C < BK || N < BM || M < BM || K < 1 || K > GRAFP_KNN_MAX_K) return Plan{};
  // Which selection epilogue.  K > 8 (16-entry lists, rounds) exists in the candidate-queue form only.  For K <= 8 both
  // exist and neither dominates: on features with independent rows (random point clouds: scripts/bench_ops.py, the
  // configs[3] stress) the queue form is faster (stage 0: 385 vs 429 us) because some lane of a warp has a candidate
  // in most column groups and the vote-gated form then pays its insertion path for the whole warp; inside the
  // training step - where, as far as we can tell, the 32 consecutive rows of a warp are neighbouring spectrogram peaks
  // whose candidates sit in the SAME few key columns, so the vote-gated form skips almost everything - it wins (k-NN 5.1-5.5 vs 5.6-5.9 ms per
  // step, A/B on the same box).  The default follows the headline workload; option OPT_KNN_EPILOGUE = 2 forces the queues.
  // K <= 3 with a key count that is a multiple of 32 (every encoder stage): the group-maxima selection (qs = -1).
  const int epi = option(OPT_KNN_EPILOGUE);
  const bool force_queue = epi == 2;
  const bool group_max = K <= 3 && M % 32 == 0 && (epi == 3 || (epi == 0 && kGroupMaxDefault));
  const int qs = (K <= 8 && !force_queue) ? 0 : kQueueSlots;
  // the group-maxima selection needs 3 KB of spill slots per epilogue warp next to the resident queries; where that does
  // not fit (wide separate key sets) the vote-gated form of the same kernels is used
  Plan p = plan_with(N, C, self, group_max ? -1 : qs);
  if (p.kind == 0 && group_max) p = plan_with(N, C, self, qs);
  return p;
}

// kernel, query block, key tile and ring depth for N queries of C channels with the selection form qs
static Plan plan_with(int N, int C, bool self, int qs) {
  Plan p;
  const bool no_nh4 = false, bn128 = false;
  p.qs = qs;
  const int num_kc = (C + BK - 1) / BK;
  const uint32_t budget = kSmemLimit - kMiscBytes;
  auto queue_bytes = [&](int nh) { return (uint32_t)(4 * nh) * (p.qs > 0 ? (uint32_t)p.qs * 512u : (p.qs < 0 ? 3u * 1024u : 0u)); };
  if (self && N <= 2 * BM) {
    const int nh = (N > BM) ? 2 : 1;
    // NH = 1: two CTAs per SM (<= 113 KB each); NH = 2: one CTA owns the SM
    const uint32_t cap = ((nh == 1) ? (113u * 1024 - kMiscBytes) : budget) - queue_bytes(nh);
    int st = (int)(cap / (nh * kBlockBytes));
    if (st > num_kc) st = num_kc;
    if (st > kMaxStages) st = kMaxStages;
    if (st < 1) return p;
    p.kind = 1; p.nh = nh; p.bn = BM; p.stages = st;
    return p;
  }
  // 512 resident queries, 64-key tiles (TMEM: 2 sets x 4 tiles x 64 columns), 16 epilogue warps.  Needs the 4 query
  // blocks per channel chunk to fit next to the queue and >= 3 key stages: C <= 64.
  if (!no_nh4 && N >= 4 * BM) {
    const uint32_t resident = (uint32_t)(4 * num_kc) * kBlockBytes + queue_bytes(4);
    if (resident + 3 * (kBlockBytes / 2) <= budget) {
      int st = (int)((budget - resident) / (kBlockBytes / 2));
      p.kind = 2; p.nh = 4; p.bn = 64; p.stages = st > 4 ? 4 : st;
      return p;
    }
  }
  for (int nh = (N > BM ? 2 : 1); nh >= 1; --nh) {
    const uint32_t resident = (uint32_t)(nh * num_kc) * kBlockBytes + queue_bytes(nh);
    // 64-key tiles (16 KB stages) where fewer than three 128-key stages would fit next to the queue
    if (!bn128 && p.qs > 0 && resident + 2 * (kBlockBytes / 2) <= budget && resident + 3 * kBlockBytes > budget) {
      int st = (int)((budget - resident) / (kBlockBytes / 2));
      p.kind = 2; p.nh = nh; p.bn = 64; p.stages = st > 6 ? 6 : st;
      return p;
    }
    if (resident + 2 * kBlockBytes > budget) continue;
    int st = (int)((budget - resident) / kBlockBytes);
    p.kind = 2; p.nh = nh; p.bn = BM; p.stages = st > 4 ? 4 : st;
    return p;
  }
  return p;
}

}  // namespace tc2

bool knn_tc2_supported(int N, int M, int C, int K, int dtype, bool self) { return tc2::plan(N, M, C, K, dtype, self).kind != 0; }

namespace tc2 {

struct Args {
  const CUtensorMap *xh, *xl, *yh, *yl;
  const float *xsq, *ysq;
  long long* nn_idx;
  int* nn_idx32;
  int B, N, M, C, k_out, stride;
  cudaStream_t s;
  Slices sl;
};

template <int KR, int QS, bool SPLIT = false>
static int launch_planned(const Plan& p, const Args& a, Round r) {
#define GRAFP_SELF(NH_) launch_self<NH_, KR, QS>(*a.xh, *a.xl, a.xsq, a.nn_idx, a.nn_idx32, a.B, a.N, a.C, a.k_out, a.stride, p.stages, r, a.s)
#define GRAFP_STREAM(NH_, BN_)                                                                                          \
  launch_stream<NH_, BN_, KR, QS, SPLIT>(*a.xh, *a.xl, *a.yh, *a.yl, a.xsq, a.ysq, a.nn_idx, a.nn_idx32, a.B, a.N, a.M, a.C, \
                                         a.k_out, a.stride, p.stages, r, a.sl, a.s)
  if constexpr (!SPLIT) {
    if (p.kind == 1) return p.nh == 1 ? GRAFP_SELF(1) : GRAFP_SELF(2);
  }
  if (p.nh == 4) return GRAFP_STREAM(4, 64);
  if (p.bn == 64) return p.nh == 2 ? GRAFP_STREAM(2, 64) : GRAFP_STREAM(1, 64);
  return p.nh == 2 ? GRAFP_STREAM(2, 128) : GRAFP_STREAM(1, 128);
#undef GRAFP_STREAM
#undef GRAFP_SELF
}

}  // namespace tc2

// `bounds`: B * N float2 of scratch, used when K > 16 (rounds of 16 ranks hand their last entry to the next round)
int launch_knn_tc2(const void* xhi, const void* xlo, const float* xsq, const void* yhi, const void* ylo,
                   const float* ysq, long long* nn_idx, int* nn_idx32, int B, int N, int M, int C, int K, int k_out,
                   int stride, int dtype, bool self, void* bounds, cudaStream_t s) {
  using namespace tc2;
  const Plan p = plan(N, M, C, K, dtype, self);
  if (p.kind == 0) {
    set_error("knn_tc2: unsupported configuration");
    return GRAFP_EUNSUPPORTED;
  }
  CUtensorMap xh, xl, yh, yl;
  if (!make_map_f16(&xh, xhi, B, N, C) || !make_map_f16(&xl, xlo, B, N, C) || !make_map_f16(&yh, yhi, B, M, C, p.bn) ||
      !make_map_f16(&yl, ylo, B, M, C, p.bn)) {
    set_error("knn_tc2: cuTensorMapEncodeTiled failed (driver entry point unavailable or bad shape)");
    return GRAFP_EUNSUPPORTED;
  }
  const Args a = {&xh, &xl, &yh, &yl, xsq, ysq, nn_idx, nn_idx32, B, N, M, C, k_out, stride, s, Slices{}};
  const Round one = {nullptr, 0, 0};
  if (K <= 3) {
    if (p.qs < 0) return launch_planned<3, -1>(p, a, one);
    return p.qs > 0 ? launch_planned<3, kQueueSlots>(p, a, one) : launch_planned<3, 0>(p, a, one);
  }
  if (K <= 8) return p.qs > 0 ? launch_planned<8, kQueueSlots>(p, a, one) : launch_planned<8, 0>(p, a, one);
  // 16-entry register lists; K = 17..64 takes ceil(K / 16) passes over the keys (the Gram tiles are recomputed: the
  // tensor pipe is far from busy, the selection is what costs), each pass bounded below by the previous one's last entry
  const int rounds = (K + 15) / 16;
  if (rounds > 1 && bounds == nullptr) {
    set_error("knn_tc2: K > 16 needs the bounds scratch");
    return GRAFP_EWORKSPACE;
  }
  for (int r = 0; r < rounds; ++r) {
    const Round rd = {static_cast<float2*>(bounds), 16 * r, r + 1 < rounds ? 1 : 0};
    if (int rc = launch_planned<16, kQueueSlots>(p, a, rd)) return rc;
  }
  return GRAFP_OK;
}

}  // namespace grafp

// ---------------------------------------------------------------------------------------------
// exact flat search: the key-sliced stream kernel + a merge of the per-slice lists
// ---------------------------------------------------------------------------------------------
namespace grafp {
namespace tc2 {

constexpr int kMaxSlices = 1024;          // merge cursors per query (one byte each, k <= 128)
constexpr int kMaxSliceLen = 1 << 26;     // group ids (slice-local key / 8) stay below GroupTop::kInvalid
constexpr int kMergeWarps = 4;

struct SearchPlan {
  Plan p;
  int slices = 0, slice_len = 0;
};

// Selection form from k alone.  Database rows are independent, the case where K1 measured the candidate queue ahead of
// the vote-gated scan; k <= 3 takes the group maxima, on slices whose keys are unit-norm (the vote-gated scan elsewhere).
// Slices: (query blocks x slices) >= 2 CTAs per SM, each slice a whole number of key tiles (64 or 128 keys, so also of
// the 32-key chunks of the group maxima) and at least two of them.
static SearchPlan search_plan(int n_q, int n_db, int d, int k) {
  SearchPlan sp;
  sp.p = plan_with(n_q, d, false, k <= 3 ? -1 : kQueueSlots);
  if (sp.p.kind != 2) return SearchPlan{};
  const long long qblocks = (n_q + BM * sp.p.nh - 1) / (BM * sp.p.nh);
  const long long want = (2LL * num_sms() + qblocks - 1) / qblocks;
  const long long tile = sp.p.bn;
  long long len = ((long long)n_db + want - 1) / want;
  len = (len + tile - 1) / tile * tile;
  len = std::max(len, 2 * tile);
  len = std::min(len, (long long)kMaxSliceLen);
  sp.slice_len = (int)len;
  sp.slices = (int)(((long long)n_db + len - 1) / len);
  if (sp.slices > kMaxSlices) return SearchPlan{};
  return sp;
}

struct SearchLayout {
  size_t plane, qsq, bounds, part, total;
};
static size_t align1k(size_t v) { return (v + 1023) / 1024 * 1024; }
static SearchLayout search_layout(int n_q, int d, int k, int slices) {
  SearchLayout l;
  l.plane = align1k((size_t)n_q * d * 2);                              // query hi / lo planes (fp16)
  l.qsq = align1k((size_t)n_q * 4);                                    // |q|^2
  l.bounds = k > 16 ? align1k((size_t)slices * n_q * 8) : 0;           // round hand-over per (slice, query)
  l.part = align1k((size_t)slices * n_q * k * 8);                      // per-slice lists (dist, slice-local id)
  l.total = 2 * l.plane + l.qsq + l.bounds + l.part + 1024;            // + base alignment
  return l;
}

// One warp per query: k steps of a lexicographic (dist, global id) minimum over the heads of the slices' sorted lists.
// Slices are disjoint ascending id ranges and each list is exact, so the result is the single-pass top-k bit for bit
// (for the group maxima: up to keys closer than the slice's |y|^2 spread, see kSearchUnitSpread).
__global__ void __launch_bounds__(kMergeWarps * 32)
search_merge_kernel(const float2* __restrict__ part, int slices, int slice_len, int N, int k, long long* __restrict__ ids,
                    float* __restrict__ dist) {
  __shared__ unsigned char cursor[kMergeWarps][kMaxSlices];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int q = blockIdx.x * kMergeWarps + warp;
  if (q >= N) return;  // warp-uniform; the warps share no data
  unsigned char* cur = cursor[warp];
  for (int s = lane; s < slices; s += 32) cur[s] = 0;
  __syncwarp();
  float bd;
  int bid, bs;
  auto rescan = [&]() {  // this lane's best head over its slices lane, lane + 32, ...
    bd = INFINITY; bid = INT_MAX; bs = -1;
    for (int s = lane; s < slices; s += 32) {
      if (cur[s] >= k) continue;
      const float2 v = part[((long long)s * N + q) * k + cur[s]];
      const int gid = s * slice_len + __float_as_int(v.y);
      if (bs < 0 || v.x < bd || (v.x == bd && gid < bid)) { bd = v.x; bid = gid; bs = s; }
    }
  };
  rescan();
  for (int r = 0; r < k; ++r) {
    float md = bd;
    int mid = bid;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float od = __shfl_xor_sync(0xffffffffu, md, o);
      const int oid = __shfl_xor_sync(0xffffffffu, mid, o);
      if (od < md || (od == md && oid < mid)) { md = od; mid = oid; }
    }
    if (lane == 0) { ids[(long long)q * k + r] = mid; dist[(long long)q * k + r] = md; }
    if (bs >= 0 && bid == mid && bd == md) {  // the one lane holding the winner advances that slice
      ++cur[bs];
      rescan();
    }
    __syncwarp();
  }
}

}  // namespace tc2

size_t search_workspace_bytes(int n_q, int n_db, int d, int k) {
  using namespace tc2;
  const SearchPlan sp = search_plan(n_q, n_db, d, k);
  return sp.p.kind == 2 ? search_layout(n_q, d, k, sp.slices).total : 0;
}

int launch_search(const float* q, int n_q, const void* hi, const void* lo, const float* sq, int n_db, int d, int k,
                  long long* ids, float* dist, void* workspace, size_t workspace_bytes, cudaStream_t s) {
  using namespace tc2;
  const SearchPlan sp = search_plan(n_q, n_db, d, k);
  if (sp.p.kind != 2) {
    set_error("grafp_search_fwd: no kernel plan for n_q=%d n_db=%d d=%d k=%d", n_q, n_db, d, k);
    return GRAFP_EUNSUPPORTED;
  }
  const SearchLayout l = search_layout(n_q, d, k, sp.slices);
  if (workspace_bytes < l.total) {
    set_error("grafp_search_fwd: workspace of %zu bytes is smaller than grafp_search_workspace_bytes() = %zu", workspace_bytes, l.total);
    return GRAFP_EWORKSPACE;
  }
  char* base = reinterpret_cast<char*>((reinterpret_cast<uintptr_t>(workspace) + 1023) & ~uintptr_t(1023));
  float* q_hi = reinterpret_cast<float*>(base);
  float* q_lo = reinterpret_cast<float*>(base + l.plane);
  float* q_sq = reinterpret_cast<float*>(base + 2 * l.plane);
  float2* bounds = l.bounds ? reinterpret_cast<float2*>(base + 2 * l.plane + l.qsq) : nullptr;
  float2* part = reinterpret_cast<float2*>(base + 2 * l.plane + l.qsq + l.bounds);
  if (int rc = launch_knn_normalize<float>(q, q_hi, q_lo, q_sq, n_q, d, 3, false, s)) return rc;
  CUtensorMap xh, xl, yh, yl;
  if (!make_map_f16(&xh, q_hi, 1, n_q, d) || !make_map_f16(&xl, q_lo, 1, n_q, d) || !make_map_f16(&yh, hi, 1, n_db, d, sp.p.bn) ||
      !make_map_f16(&yl, lo, 1, n_db, d, sp.p.bn)) {
    set_error("grafp_search_fwd: cuTensorMapEncodeTiled failed (driver entry point unavailable or bad shape)");
    return GRAFP_EUNSUPPORTED;
  }
  const Args a = {&xh, &xl, &yh, &yl, q_sq, sq, nullptr, nullptr, 1, n_q, n_db, d, k, 1, s, Slices{sp.slices, sp.slice_len, part}};
  const Round one = {nullptr, 0, 0};
  int rc = GRAFP_OK;
  if (k <= 3) {
    rc = launch_planned<3, -1, true>(sp.p, a, one);
  } else if (k <= 8) {
    rc = launch_planned<8, kQueueSlots, true>(sp.p, a, one);
  } else {
    const int rounds = (k + 15) / 16;
    for (int r = 0; r < rounds && rc == GRAFP_OK; ++r) rc = launch_planned<16, kQueueSlots, true>(sp.p, a, {bounds, 16 * r, r + 1 < rounds ? 1 : 0});
  }
  if (rc != GRAFP_OK) return rc;
  search_merge_kernel<<<(n_q + kMergeWarps - 1) / kMergeWarps, kMergeWarps * 32, 0, s>>>(part, sp.slices, sp.slice_len, n_q, k,
                                                                                     ids, dist);
  return check_launch("search_merge");
}

}  // namespace grafp
