// rnn_tc.cu -- the GRU network (src/rnn.rs:251-379) on the 5th-generation tensor cores: tcgen05.mma with the
// accumulators in TMEM, the weights resident in shared memory (brought in once per CTA by the TMA bulk-copy engine),
// the activations of 128 streams living in TMEM as the A operand.
//
// One persistent CTA per SM advances tiles of M = 128 streams.  Every layer is D[128 x N] += A[128 x K] * W[K x N]:
//   * W: int8 weights are exact in f16; the host packs each layer phase as an [N][K] K-major, no-swizzle UMMA operand
//     (16-byte core-matrix rows: ((8,n),2):((1,SBO),LBO) in 16-byte units); all nine phases (185 KB) stay in shared
//     memory for the life of the CTA;
//   * A: activations are f32; each is split x = hi + lo (two f16, ~22 significant bits) and both halves are multiplied
//     (products exact in f32).  The halves live in TMEM, two f16 per 32-bit column, row = TMEM lane = stream: the
//     epilogue thread that owns a stream writes its row with tcgen05.st and the next layer reads it as the A operand
//     of tcgen05.mma (A-from-TMEM form) -- activations never touch shared memory.  Only the 42 input features, which
//     every GRU re-reads, sit in shared memory (24 KB) because TMEM is full: 288 columns of A + 192 of accumulators;
//   * D: f32 accumulators in TMEM, read back with tcgen05.ld (32 lanes x 32 bit: thread = stream) for the epilogue:
//     bias, 1/256 scale, table tanh / sigmoid (src/util.rs:29-53), the GRU update in f32 against the f32 state in HBM.
//   One elected thread issues the MMAs of a phase and commits them to an mbarrier; the 256 epilogue threads (two per
//   stream, even / odd groups of 8 neurons) wait on it.  GRU semantics: src/rnn.rs:292-327 (reset gate applied to the
//   state BEFORE the recurrent product).
// Models whose layers do not fit this budget fall back to the mma.sync kernel (rnn_mma.cu).
// tools/probes/tcgen05_probe.cu is the stand-alone check of the descriptor / TMEM layouts used here.
#include <cuda_fp16.h>

#include <algorithm>
#include <atomic>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "common.cuh"
#include "model.hpp"

namespace nnb {

extern const float kTansigTable[201];  // host.cu (src/util.rs:3-27)

namespace {

constexpr int TM = 128;           // streams per tile = MMA M
constexpr int NT = 512;           // threads: 16 warps, four per TMEM lane quarter (a warp reaches only lanes 32 (w % 4) ..)
constexpr int NCH = NT / 128;     // column slices: which groups of 8 neurons a thread takes
constexpr int A_HI = 0, A_LO = 144, D_OFF = 288;  // TMEM columns
constexpr int A_MAX_HALVES = 288; // 18 K-chunks of 16
constexpr int D_COLS = 192;
constexpr int FEAT_CHUNKS = 3;    // 48 feature columns (42 used)
constexpr int FEAT_GROUP_BYTES = TM * 16;  // one 8-column group of the shared-memory feature operand
constexpr float WEIGHTS_SCALE = 1.0f / 256.0f;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// src/util.rs:3-27, branch-free: same arithmetic on |x| clamped to 8, the saturations (NaN -> 1 like the reference's
// `!(x < 8)`) applied as selects at the end.
__device__ __forceinline__ float tansig_approx(float x, const float* __restrict__ table) {
    const float sign = (x < 0.0f) ? -1.0f : 1.0f;
    float ax = fminf(fabsf(x), 8.0f);
    const float fi = floorf(0.5f + 25.0f * ax);
    ax -= 0.04f * fi;
    float y = table[(int)fi];
    const float dy = 1.0f - y * y;
    y = y + ax * dy * (1.0f - y * ax);
    y = sign * y;
    y = !(x > -8.0f) ? -1.0f : y;
    return !(x < 8.0f) ? 1.0f : y;
}
__device__ __forceinline__ float sigmoid_approx(float x, const float* __restrict__ table) { return 0.5f + 0.5f * tansig_approx(0.5f * x, table); }
__device__ __forceinline__ float activate(int act, float x, const float* __restrict__ table) {
    if (act == 0) return tansig_approx(x, table);
    if (act == 1) return sigmoid_approx(x, table);
    return fmaxf(x, 0.0f);
}

// ---- UMMA descriptors (cute/arch/mma_sm100_desc.hpp): K-major, no swizzle ----
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr >> 4) & 0x3fff);            // start address, bits [0,14)
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3fff) << 16;  // leading byte offset (between the two 8-element K halves)
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3fff) << 32;  // stride byte offset (between 8-row groups)
    d |= (uint64_t)1 << 46;                            // descriptor version 1 (Blackwell)
    return d;
}
__device__ __forceinline__ uint32_t make_idesc(int n) {
    return (1u << 4) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(TM >> 4) << 24);  // f32 accumulate, f16 x f16, K-major A and B
}
__device__ __forceinline__ void mma_ss(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(acc)
        : "memory");
}
__device__ __forceinline__ void mma_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc, uint32_t acc) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}\n" ::"r"(d_tmem), "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(acc)
        : "memory");
}
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tWAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra DONE;\n\tbra WAIT_LOOP;\n\tDONE:\n\t}\n" ::"r"(smem_u32(bar)), "r"(parity)
        : "memory");
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float (&v)[8]) {
    uint32_t r[8];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];\n"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr));
#pragma unroll
    for (int i = 0; i < 8; i++) v[i] = __uint_as_float(r[i]);
}
// tcgen05.ld is asynchronous: registers are valid only after this wait (several loads may share one).  The empty
// volatile asm statements with "+" operands pin every use of the loaded registers behind the wait.
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory"); }
__device__ __forceinline__ void after_wait(float (&v)[8]) {
    asm volatile("" : "+f"(v[0]), "+f"(v[1]), "+f"(v[2]), "+f"(v[3]), "+f"(v[4]), "+f"(v[5]), "+f"(v[6]), "+f"(v[7])::"memory");
}
__device__ __forceinline__ void after_wait(uint32_t (&v)[4]) { asm volatile("" : "+r"(v[0]), "+r"(v[1]), "+r"(v[2]), "+r"(v[3])::"memory"); }
__device__ __forceinline__ void tmem_ld4(uint32_t taddr, uint32_t (&r)[4]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0,%1,%2,%3}, [%4];\n" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(taddr));
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const float (&v)[8]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};\n" ::"r"(taddr), "r"(__float_as_uint(v[0])),
                 "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3])), "r"(__float_as_uint(v[4])),
                 "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7]))
                 : "memory");
}
__device__ __forceinline__ void tmem_st4(uint32_t taddr, const uint32_t (&r)[4]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x4.b32 [%0], {%1,%2,%3,%4};\n" ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]) : "memory");
}

// x = hi + lo with hi, lo in f16; eight values -> four packed registers each (value 2i in the low half).  No clamp: NaN
// stays NaN and |x| > 65504 (an unbounded ReLU layer of a custom model) becomes +-inf / NaN downstream: loud, not silent.
__device__ __forceinline__ void split8(const float (&v)[8], uint32_t (&hi)[4], uint32_t (&lo)[4]) {
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const __half h0 = __float2half_rn(v[2 * i]), h1 = __float2half_rn(v[2 * i + 1]);
        const __half l0 = __float2half_rn(v[2 * i] - __half2float(h0)), l1 = __float2half_rn(v[2 * i + 1] - __half2float(h1));
        hi[i] = (uint32_t)__half_as_ushort(h0) | ((uint32_t)__half_as_ushort(h1) << 16);
        lo[i] = (uint32_t)__half_as_ushort(l0) | ((uint32_t)__half_as_ushort(l1) << 16);
    }
}

}  // namespace

namespace {

// epilogue helpers: this thread's TMEM row
struct Row {
    uint32_t tm;       // tmem base | lane offset
    int ch;            // column half (0 / 1): which groups of 8 neurons this thread takes
    __device__ __forceinline__ uint32_t d(int col) const { return tm + D_OFF + col; }
    __device__ __forceinline__ uint32_t ahi(int half_off) const { return tm + A_HI + (half_off >> 1); }
    __device__ __forceinline__ uint32_t alo(int half_off) const { return tm + A_LO + (half_off >> 1); }
    // read eight activations back as hi + lo (what the tensor core multiplies: ~22 significant bits of the f32 value):
    // issue the two loads, and after tmem_wait_ld() combine them
    __device__ __forceinline__ void get_act_issue(int half_off, uint32_t (&hi)[4], uint32_t (&lo)[4]) const {
        tmem_ld4(ahi(half_off), hi);
        tmem_ld4(alo(half_off), lo);
    }
    __device__ __forceinline__ static void get_act_finish(uint32_t (&hi)[4], uint32_t (&lo)[4], float (&v)[8]) {
        after_wait(hi);
        after_wait(lo);
#pragma unroll
        for (int i = 0; i < 4; i++) {
            v[2 * i] = __half2float(__ushort_as_half((unsigned short)(hi[i] & 0xffffu))) + __half2float(__ushort_as_half((unsigned short)(lo[i] & 0xffffu)));
            v[2 * i + 1] = __half2float(__ushort_as_half((unsigned short)(hi[i] >> 16))) + __half2float(__ushort_as_half((unsigned short)(lo[i] >> 16)));
        }
    }
    // write eight activations (columns half_off .. half_off + 7 of the A operand) as hi / lo halves
    __device__ __forceinline__ void put_act(int half_off, const float (&v)[8]) const {
        uint32_t hi[4], lo[4];
        split8(v, hi, lo);
        tmem_st4(ahi(half_off), hi);
        tmem_st4(alo(half_off), lo);
    }
};

__global__ void __launch_bounds__(NT, 1) rnn_tc_kernel(BatchBuffers bb, DeviceModelTc m, int n_tiles) {
    extern __shared__ __align__(1024) unsigned char smraw[];
    unsigned char* wblob = smraw;                                                  // weights | biases | table
    const uint32_t feat_off = (m.blob_bytes + 1023u) & ~1023u;
    unsigned char* featA = smraw + feat_off;                                       // [hi | lo][6 groups][128 rows][8 halves]
    uint64_t* bars = reinterpret_cast<uint64_t*>(featA + 2 * 2 * FEAT_CHUNKS * FEAT_GROUP_BYTES);  // [0] MMA, [1] weights
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2);
    const float* table = reinterpret_cast<const float*>(wblob + m.table_off);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int q = warp & 3, ch = warp >> 2;  // lane quarter, column slice
    const int row = 32 * q + lane;

    if (tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;\n" ::"r"(smem_u32(&bars[0])));
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;\n" ::"r"(smem_u32(&bars[1])));
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;\n" ::"r"(smem_u32(tmem_slot)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
    }
    __syncthreads();
    if (tid == 0) {
        // the whole model image in one go: TMA bulk copies (<= 64 KB each) completing on bars[1]
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(smem_u32(&bars[1])), "r"(m.blob_bytes) : "memory");
        for (uint32_t off = 0; off < m.blob_bytes; off += 65536u) {
            const uint32_t nb = min(65536u, m.blob_bytes - off);
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n" ::"r"(smem_u32(wblob + off)),
                         "l"(m.blob + off), "r"(nb), "r"(smem_u32(&bars[1]))
                         : "memory");
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
    const uint32_t tmem = *tmem_slot;
    Row R{tmem + ((uint32_t)(32 * q) << 16), ch};
    {
        // the A operand starts as zeros: a K chunk may span columns that no epilogue writes (the padding before the
        // r * h segment, its tail beyond this layer's width), where the weights are 0 -- but fresh TMEM holds anything,
        // and 0 * NaN is NaN
        const float zero8[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        for (int g = ch; g < A_MAX_HALVES / 8; g += NCH) R.put_act(8 * g, zero8);
    }
    asm volatile("tcgen05.wait::st.sync.aligned;\n" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
    mbar_wait(&bars[1], 0);  // weights, biases and the tanh table have landed
    uint32_t par = 0;  // parity of bars[0]
    const int SS = m.state_size;
    const int so_n = m.nv, so_d = m.nv + m.nn;  // state offsets in HBM (vad | noise | denoise)
    const bool vec_ok = ((m.nv | m.nn | m.ndn) & 3) == 0;

    // one phase: elected thread issues the MMAs (hi and lo halves of every K chunk against the same weights) and
    // commits them; everybody waits for the accumulators
    auto run_phase = [&](int p0, int p1) {
        asm volatile("tcgen05.wait::st.sync.aligned;\n" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
        asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
        __syncthreads();
        if (tid == 0) {
            asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
            for (int pi = 0; pi < (p1 != p0 ? 2 : 1); pi++) {  // one phase, or two that share a commit
                const int p = pi == 0 ? p0 : p1;
                const TcPhase& ph = m.ph[p];
                const uint32_t idesc = make_idesc(ph.n);
                const uint32_t d_tm = tmem + D_OFF + ph.d_col;
                const uint32_t wb = smem_u32(wblob + ph.w_off);
                uint32_t acc = 0;
                for (int kc = 0; kc < ph.nk; kc++) {
                    const uint64_t bd = make_desc(wb + kc * 2 * (ph.n * 16), ph.n * 16, 128);
                    const int c = ph.chunk[kc];
#pragma unroll
                    for (int hl = 0; hl < 2; hl++) {
                        if (c >= 0) {
                            mma_ts(d_tm, tmem + (hl ? A_LO : A_HI) + 8 * c, bd, idesc, acc);
                        } else {
                            const int f = -c - 1;
                            const uint32_t fa = smem_u32(featA + (hl * 2 * FEAT_CHUNKS + 2 * f) * FEAT_GROUP_BYTES);
                            mma_ss(d_tm, make_desc(fa, FEAT_GROUP_BYTES, 128), bd, idesc, acc);
                        }
                        acc = 1;
                    }
                }
            }
            mma_commit(&bars[0]);
        }
        mbar_wait(&bars[0], par);
        par ^= 1;
        asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
    };

    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int s = tile * TM + row;
        const bool live = s < bb.n_streams;
        const bool upd = live && !bb.silence[live ? s : 0];  // silent frames leave the RNN state and outputs untouched
        const float* fsrc = bb.features + (size_t)(live ? s : 0) * NB_FEATURES;
        float* hsrc = bb.gru_state + (size_t)(live ? s : 0) * SS;

        // ---- features -> shared-memory A operand (6 groups of 8 columns; this thread takes 3), states -> TMEM ----
        for (int g = ch; g < 2 * FEAT_CHUNKS; g += NCH) {
            float v[8];
#pragma unroll
            for (int i = 0; i < 8; i += 2) {
                const int j = 8 * g + i;
                float2 t = make_float2(0.f, 0.f);
                if (live && j < NB_FEATURES) t = __ldg(reinterpret_cast<const float2*>(fsrc + j));  // 42 is even: pairs never straddle
                v[i] = t.x;
                v[i + 1] = t.y;
            }
            uint32_t hi[4], lo[4];
            split8(v, hi, lo);
            *reinterpret_cast<uint4*>(featA + g * FEAT_GROUP_BYTES + row * 16) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
            *reinterpret_cast<uint4*>(featA + (2 * FEAT_CHUNKS + g) * FEAT_GROUP_BYTES + row * 16) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
        }
        auto load_state = [&](int nn_, int p8, int s_off, int a_off) {
            for (int g = ch; g < p8 / 8; g += NCH) {
                float v[8];
                if (live && 8 * g + 8 <= nn_ && vec_ok) {  // rows are 16-byte aligned when every layer width is a multiple of 4
                    const float4 t0 = __ldg(reinterpret_cast<const float4*>(hsrc + s_off + 8 * g));
                    const float4 t1 = __ldg(reinterpret_cast<const float4*>(hsrc + s_off + 8 * g + 4));
                    v[0] = t0.x; v[1] = t0.y; v[2] = t0.z; v[3] = t0.w; v[4] = t1.x; v[5] = t1.y; v[6] = t1.z; v[7] = t1.w;
                } else {
#pragma unroll
                    for (int i = 0; i < 8; i++) v[i] = (live && 8 * g + i < nn_) ? __ldg(hsrc + s_off + 8 * g + i) : 0.0f;
                }
                R.put_act(a_off + 8 * g, v);
            }
        };
        load_state(m.nv, m.p_v, 0, m.o_vad);
        load_state(m.nn, m.p_n, so_n, m.o_noise);
        load_state(m.ndn, m.p_dn, so_d, m.o_den);

        // ---- input_dense (src/rnn.rs:353-355) ----
        run_phase(PH_DENSE, PH_DENSE);
        {
            const float* bias = reinterpret_cast<const float*>(wblob + m.ph[PH_DENSE].b_off);
            for (int g = ch; g < m.p_d / 8; g += NCH) {
                float a[8];
                tmem_ld8(R.d(m.ph[PH_DENSE].d_col + 8 * g), a);
                tmem_wait_ld();
                after_wait(a);
#pragma unroll
                for (int i = 0; i < 8; i++) a[i] = (8 * g + i < m.nd) ? activate(m.act_dense, WEIGHTS_SCALE * (a[i] + bias[8 * g + i]), table) : 0.0f;
                R.put_act(m.o_dense + 8 * g, a);
            }
        }

        // ---- one GRU layer: z | r phase then candidate phase (src/rnn.rs:292-327) ----
        auto gru = [&](int pzr, int phh, int extra, int act, int nn_, int p8, int s_off, int a_off) {
            run_phase(pzr, extra >= 0 ? extra : pzr);
            {
                const float* bias = reinterpret_cast<const float*>(wblob + m.ph[pzr].b_off);
                const int dz = m.ph[pzr].d_col;
                for (int g = ch; g < p8 / 8; g += NCH) {
                    float z[8], r[8], hpv[8];
                    uint32_t thi[4], tlo[4];
                    tmem_ld8(R.d(dz + 8 * g), z);
                    tmem_ld8(R.d(dz + p8 + 8 * g), r);
                    R.get_act_issue(a_off + 8 * g, thi, tlo);  // previous state as the tensor core sees it (hi + lo)
                    tmem_wait_ld();
                    after_wait(z);
                    after_wait(r);
                    Row::get_act_finish(thi, tlo, hpv);
#pragma unroll
                    for (int i = 0; i < 8; i++) {
                        const int o = 8 * g + i;
                        const float hp = hpv[i];
                        z[i] = sigmoid_approx(WEIGHTS_SCALE * (z[i] + bias[o]), table);
                        r[i] = (o < nn_) ? sigmoid_approx(WEIGHTS_SCALE * (r[i] + bias[p8 + o]), table) * hp : 0.0f;  // reset gate scales the previous state
                    }
                    tmem_st8(R.d(dz + 8 * g), z);          // the update gate waits in its accumulator columns
                    R.put_act(m.o_rh + 8 * g, r);
                }
            }
            run_phase(phh, phh);
            {
                const float* bias = reinterpret_cast<const float*>(wblob + m.ph[phh].b_off);
                const int dz = m.ph[pzr].d_col, dh = m.ph[phh].d_col;
                for (int g = ch; g < p8 / 8; g += NCH) {
                    float z[8], hh[8], hpv[8];
                    uint32_t thi[4], tlo[4];
                    tmem_ld8(R.d(dz + 8 * g), z);
                    tmem_ld8(R.d(dh + 8 * g), hh);
                    R.get_act_issue(a_off + 8 * g, thi, tlo);
                    tmem_wait_ld();
                    after_wait(z);
                    after_wait(hh);
                    Row::get_act_finish(thi, tlo, hpv);
#pragma unroll
                    for (int i = 0; i < 8; i++) {
                        const int o = 8 * g + i;
                        const float c = activate(act, WEIGHTS_SCALE * (hh[i] + bias[o]), table);
                        hh[i] = (o < nn_) ? z[i] * hpv[i] + (1.0f - z[i]) * c : 0.0f;
                    }
                    if (upd) {
                        if (8 * g + 8 <= nn_ && vec_ok) {
                            *reinterpret_cast<float4*>(hsrc + s_off + 8 * g) = make_float4(hh[0], hh[1], hh[2], hh[3]);
                            *reinterpret_cast<float4*>(hsrc + s_off + 8 * g + 4) = make_float4(hh[4], hh[5], hh[6], hh[7]);
                        } else {
#pragma unroll
                            for (int i = 0; i < 8; i++)
                                if (8 * g + i < nn_) hsrc[s_off + 8 * g + i] = hh[i];
                        }
                    }
                    R.put_act(a_off + 8 * g, hh);
                }
            }
        };
        // vad_gru (src/rnn.rs:356-358)
        gru(PH_VAD_ZR, PH_VAD_H, -1, m.act_vad, m.nv, m.p_v, 0, m.o_vad);
        // noise_gru (:361-369); vad_output (:359) only reads the new vad state: its MMA rides in the same commit
        gru(PH_NOISE_ZR, PH_NOISE_H, PH_VAD_OUT, m.act_noise, m.nn, m.p_n, so_n, m.o_noise);
        if (ch == 0) {
            float a[8];
            tmem_ld8(R.d(m.ph[PH_VAD_OUT].d_col), a);
            tmem_wait_ld();
            after_wait(a);
            const float* bias = reinterpret_cast<const float*>(wblob + m.ph[PH_VAD_OUT].b_off);
            if (upd) bb.vad[s] = activate(m.act_vadout, WEIGHTS_SCALE * (a[0] + bias[0]), table);
        }
        // denoise_gru (:370-377)
        gru(PH_DEN_ZR, PH_DEN_H, -1, m.act_den, m.ndn, m.p_dn, so_d, m.o_den);
        // denoise_output (:378): 22 band gains
        run_phase(PH_OUT, PH_OUT);
        {
            const float* bias = reinterpret_cast<const float*>(wblob + m.ph[PH_OUT].b_off);
            for (int g = ch; g < (NB_BANDS + 7) / 8; g += NCH) {
                float a[8];
                tmem_ld8(R.d(m.ph[PH_OUT].d_col + 8 * g), a);
                tmem_wait_ld();
                after_wait(a);
                if (upd) {
#pragma unroll
                    for (int i = 0; i < 8; i++) {
                        const int o = 8 * g + i;
                        if (o < NB_BANDS) bb.gains[(size_t)s * NB_BANDS + o] = activate(m.act_out, WEIGHTS_SCALE * (a[i] + bias[o]), table);
                    }
                }
            }
        }
        // the next tile's loads overwrite the A operand and the feature buffer: every MMA of this tile has completed
        // (each phase was waited for), and the tcgen05.ld above are complete (wait::ld) -- one barrier suffices
        asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
        __syncthreads();
        asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
    }

    asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;\n" ::"r"(tmem) : "memory");
}

inline int pad8(int n) { return (n + 7) & ~7; }
inline int pad16(int n) { return (n + 15) & ~15; }
// dynamic shared memory of rnn_tc_kernel: model image, the feature operand at the next 1 KB boundary, two mbarriers and
// the TMEM address (the layout at the top of the kernel)
inline size_t tc_smem_bytes(const DeviceModelTc& d) {
    return (((size_t)d.blob_bytes + 1023) & ~(size_t)1023) + 2 * 2 * FEAT_CHUNKS * FEAT_GROUP_BYTES + 64;
}

}  // namespace

// ---- host: pack the model image for the kernel (weights, biases, tanh table).  Returns false if the model does not fit
// the TMEM / shared-memory budget. ----
bool build_model_tc(const HostModel& hm, DeviceModelTc* d, std::vector<unsigned char>* blob) {
    const int nd = hm.input_dense.nn, nv = hm.vad_gru.nn, nn = hm.noise_gru.nn, ndn = hm.denoise_gru.nn;
    d->nd = nd; d->nv = nv; d->nn = nn; d->ndn = ndn;
    d->p_d = pad8(nd); d->p_v = pad8(nv); d->p_n = pad8(nn); d->p_dn = pad8(ndn);
    d->o_dense = 0;
    d->o_vad = d->o_dense + d->p_d;
    d->o_noise = d->o_vad + d->p_v;
    d->o_den = d->o_noise + d->p_n;
    d->o_rh = pad16(d->o_den + d->p_dn);
    const int rh = std::max(d->p_v, std::max(d->p_n, d->p_dn));
    if (d->o_rh + rh > A_MAX_HALVES) return false;
    if (2 * d->p_dn > D_COLS || 2 * d->p_n > D_COLS) return false;
    d->act_dense = hm.input_dense.act; d->act_vad = hm.vad_gru.act; d->act_noise = hm.noise_gru.act; d->act_den = hm.denoise_gru.act;
    d->act_out = hm.denoise_output.act; d->act_vadout = hm.vad_output.act;
    d->state_size = nv + nn + ndn;
    const int8_t* B = hm.bytes.data();

    // which source does activation column a (in halves) of the TMEM operand hold?  seg: 0 dense, 1 vad, 2 noise, 3 den, 4 rh
    auto col_src = [&](int a, int* seg, int* j) {
        *seg = -1;
        if (a >= d->o_rh) { *seg = 4; *j = a - d->o_rh; }
        else if (a >= d->o_den) { *seg = 3; *j = a - d->o_den; }
        else if (a >= d->o_noise) { *seg = 2; *j = a - d->o_noise; }
        else if (a >= d->o_vad) { *seg = 1; *j = a - d->o_vad; }
        else { *seg = 0; *j = a; }
    };
    const int seg_size[5] = {nd, nv, nn, ndn, rh};
    const int seg_off[5] = {d->o_dense, d->o_vad, d->o_noise, d->o_den, d->o_rh};
    // chunks (of 16 halves) covering segment `seg` restricted to its first `len` columns
    auto chunks_of = [&](int seg, int len, std::vector<int>* out) {
        const int a0 = seg_off[seg], a1 = seg_off[seg] + len;
        for (int c = a0 / 16; c * 16 < a1; c++)
            if (std::find(out->begin(), out->end(), c) == out->end()) out->push_back(c);
    };

    // weight(seg, j, gate, o): int8 weight of input (seg, j) for output neuron o of `gate`, or 0 if that input is not wired
    struct Wire { int seg; int len; int row0; bool recurrent; };  // rows of W (or R) that segment seg feeds
    auto add_phase = [&](int pi, const std::vector<Wire>& wires, bool use_feat, int feat_row0, int nout, int ngates, int gate0, int p8,
                         size_t w_off, size_t r_off, size_t b_off, int row_stride, int d_col) -> bool {
        TcPhase& ph = d->ph[pi];
        std::vector<int> chunks;
        for (const Wire& w : wires) chunks_of(w.seg, w.len, &chunks);
        std::sort(chunks.begin(), chunks.end());
        std::vector<int> entries(chunks.begin(), chunks.end());
        if (use_feat)
            for (int f = 0; f < FEAT_CHUNKS; f++) entries.push_back(-(f + 1));
        const int np = ngates * p8;
        if (np == 0) {
            entries.clear();  // a zero-width layer has no accumulators: issue no MMA (N = 0 is not an MMA shape)
        } else if (entries.empty()) {
            // accumulators that are read but that no input feeds (a zero-width input layer): one zero-weight chunk of
            // the feature operand, which always holds finite values, makes them 0 instead of leaving stale TMEM
            entries.push_back(-1);
        }
        if ((int)entries.size() > 16) return false;
        ph.nk = (int)entries.size();
        for (int i = 0; i < ph.nk; i++) ph.chunk[i] = (short)entries[i];
        ph.n = pad16(np);
        if (ph.n > 256 || d_col + ph.n > D_COLS) return false;
        ph.d_col = d_col;
        while (blob->size() % 128) blob->push_back(0);
        ph.w_off = (uint32_t)blob->size();
        const int K = 16 * ph.nk;
        blob->resize(blob->size() + (size_t)ph.n * K * 2, 0);
        __half* wb = reinterpret_cast<__half*>(blob->data() + ph.w_off);
        for (int kc = 0; kc < ph.nk; kc++)
            for (int kk = 0; kk < 16; kk++) {
                // source row of this K column
                const int8_t* src = nullptr;  // start of the weight row (all gates), or null = not wired
                if (entries[kc] >= 0) {
                    int seg, j;
                    col_src(entries[kc] * 16 + kk, &seg, &j);
                    for (const Wire& w : wires)
                        if (w.seg == seg && j < w.len) src = B + (w.recurrent ? r_off : w_off) + (size_t)(w.row0 + j) * row_stride;
                } else {
                    const int j = (-entries[kc] - 1) * 16 + kk;
                    if (use_feat && j < NB_FEATURES) src = B + w_off + (size_t)(feat_row0 + j) * row_stride;
                }
                const int k = kc * 16 + kk;
                for (int n = 0; n < ph.n; n++) {
                    const int gate = n / p8, o = n % p8;
                    int val = 0;
                    if (src && gate < ngates && o < nout) val = src[(gate0 + gate) * nout + o];
                    // canonical K-major operand: element (n, k) at (k / 8) * (N * 16 B) + n * 16 B + (k % 8) * 2 B
                    wb[(size_t)(k / 8) * (ph.n * 8) + (size_t)n * 8 + (k % 8)] = __float2half((float)val);
                }
            }
        while (blob->size() % 16) blob->push_back(0);
        ph.b_off = (uint32_t)blob->size();
        blob->resize(blob->size() + (size_t)ph.n * 4, 0);
        float* bf = reinterpret_cast<float*>(blob->data() + ph.b_off);
        for (int n = 0; n < ph.n; n++) {
            const int gate = n / p8, o = n % p8;
            bf[n] = (gate < ngates && o < nout) ? (float)B[b_off + (size_t)(gate0 + gate) * nout + o] : 0.0f;
        }
        return true;
    };

    bool ok = true;
    const HostDense& L0 = hm.input_dense;
    const HostGru &G1 = hm.vad_gru, &G2 = hm.noise_gru, &G3 = hm.denoise_gru;
    const HostDense &LO = hm.denoise_output, &LV = hm.vad_output;
    // dense: features only
    ok = ok && add_phase(PH_DENSE, {}, true, 0, nd, 1, 0, d->p_d, L0.w_off, 0, L0.b_off, nd, 0);
    // vad_gru: input = dense_out
    ok = ok && add_phase(PH_VAD_ZR, {{0, nd, 0, false}, {1, nv, 0, true}}, false, 0, nv, 2, 0, d->p_v, G1.w_off, G1.r_off, G1.b_off, 3 * nv, 0);
    ok = ok && add_phase(PH_VAD_H, {{0, nd, 0, false}, {4, nv, 0, true}}, false, 0, nv, 1, 2, d->p_v, G1.w_off, G1.r_off, G1.b_off, 3 * nv, 2 * d->p_v > 64 ? 2 * d->p_v : 64);
    // vad_output: one neuron from the vad state; accumulators at the top of the D region
    ok = ok && add_phase(PH_VAD_OUT, {{1, nv, 0, false}}, false, 0, 1, 1, 0, 8, LV.w_off, 0, LV.b_off, 1, D_COLS - 16);
    // noise_gru: input = [dense_out | vad_state | features]; the candidate's accumulators reuse the reset gate's columns
    // (the z | r epilogue has moved r into the A operand before the candidate phase is issued)
    ok = ok && add_phase(PH_NOISE_ZR, {{0, nd, 0, false}, {1, nv, nd, false}, {2, nn, 0, true}}, true, nd + nv, nn, 2, 0, d->p_n, G2.w_off, G2.r_off,
                         G2.b_off, 3 * nn, 0);
    ok = ok && add_phase(PH_NOISE_H, {{0, nd, 0, false}, {1, nv, nd, false}, {4, nn, 0, true}}, true, nd + nv, nn, 1, 2, d->p_n, G2.w_off, G2.r_off,
                         G2.b_off, 3 * nn, d->p_n);
    // denoise_gru: input = [vad_state | noise_state | features]; the candidate's accumulators reuse the reset gate's columns
    ok = ok && add_phase(PH_DEN_ZR, {{1, nv, 0, false}, {2, nn, nv, false}, {3, ndn, 0, true}}, true, nv + nn, ndn, 2, 0, d->p_dn, G3.w_off, G3.r_off,
                         G3.b_off, 3 * ndn, 0);
    ok = ok && add_phase(PH_DEN_H, {{1, nv, 0, false}, {2, nn, nv, false}, {4, ndn, 0, true}}, true, nv + nn, ndn, 1, 2, d->p_dn, G3.w_off, G3.r_off,
                         G3.b_off, 3 * ndn, d->p_dn);
    // denoise_output
    ok = ok && add_phase(PH_OUT, {{3, ndn, 0, false}}, false, 0, NB_BANDS, 1, 0, pad8(NB_BANDS), LO.w_off, 0, LO.b_off, NB_BANDS, 0);
    if (!ok) return false;
    // neither noise GRU phase may overlap vad_output's accumulators (columns D_COLS - 16 ..), which are read after the
    // noise GRU's candidate phase
    if (d->ph[PH_NOISE_ZR].n > D_COLS - 16 || d->ph[PH_NOISE_H].d_col + d->ph[PH_NOISE_H].n > D_COLS - 16) return false;
    (void)seg_size;
    // the tanh table closes the image; image + feature operand + barriers must fit one CTA's shared memory
    while (blob->size() % 16) blob->push_back(0);
    d->table_off = (uint32_t)blob->size();
    blob->resize(blob->size() + 208 * 4, 0);
    std::memcpy(blob->data() + d->table_off, kTansigTable, 201 * 4);
    while (blob->size() % 16) blob->push_back(0);
    d->blob_bytes = (uint32_t)blob->size();
    return tc_smem_bytes(*d) <= 227 * 1024;
}

int upload_model_tc(const HostModel& hm, UploadedTc* u, cudaStream_t st) {
    u->ok = false;
    std::vector<unsigned char> blob;
    if (!build_model_tc(hm, &u->dm, &blob)) return 0;  // not an error: the caller uses the mma.sync kernel
    u->smem_bytes = tc_smem_bytes(u->dm);
    if (cudaMalloc(&u->d_blob, blob.size()) != cudaSuccess) return -1;
    if (cudaMemcpyAsync(u->d_blob, blob.data(), blob.size(), cudaMemcpyHostToDevice, st) != cudaSuccess) return -1;
    if (cudaStreamSynchronize(st) != cudaSuccess) return -1;
    u->dm.blob = u->d_blob;
    u->ok = true;
    return 0;
}

cudaError_t launch_rnn_tc(const BatchBuffers& b, const UploadedTc& u, cudaStream_t st) {
    static std::atomic<size_t> attr_smem[64];
    static std::atomic<int> sm_count[64];
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev >= 64 || u.smem_bytes > attr_smem[dev].load(std::memory_order_acquire)) {
        e = cudaFuncSetAttribute(rnn_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)u.smem_bytes);
        if (e != cudaSuccess) return e;
        if (dev < 64) {
            size_t cur = attr_smem[dev].load(std::memory_order_relaxed);
            while (cur < u.smem_bytes && !attr_smem[dev].compare_exchange_weak(cur, u.smem_bytes, std::memory_order_release)) {}
        }
    }
    int nsm = dev < 64 ? sm_count[dev].load(std::memory_order_relaxed) : 0;
    if (nsm == 0) {
        e = cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev);
        if (e != cudaSuccess) return e;
        if (dev < 64) sm_count[dev].store(nsm, std::memory_order_relaxed);
    }
    const int n_tiles = (b.n_streams + TM - 1) / TM;
    const int grid = std::min(n_tiles, nsm);
    rnn_tc_kernel<<<grid, NT, u.smem_bytes, st>>>(b, u.dm, n_tiles);
    return cudaGetLastError();
}

void free_model_tc(UploadedTc* u) {
    if (u->d_blob) cudaFree(u->d_blob);
    u->d_blob = nullptr;
    u->ok = false;
}

}  // namespace nnb

// ---- host-side self test of the PACKING (no GPU): replays the kernel's phase structure in plain f32 from the packed
// blob and compares with a direct evaluation of src/rnn.rs:343-379 from the model bytes.  Returns the largest absolute
// difference over gains, vad and the new GRU states (+inf if any is NaN); -1: model rejected, -2: model does not fit the
// tcgen05 budget of TMEM columns or shared memory (the mma.sync kernel runs it), -3: a phase whose accumulators the
// kernel reads has no K chunk (no MMA would write them), or a phase without accumulators has one (an MMA with N = 0).  Like TMEM, the replay's accumulators start as NaN and a phase only
// writes its own columns, so an epilogue that reads columns another phase has overwritten, or that no phase wrote, shows. ----
namespace nnb {
namespace {
float h_tansig(float x) {
    if (!(x < 8.0f)) return 1.0f;
    if (!(x > -8.0f)) return -1.0f;
    float sign = 1.0f;
    if (x < 0.0f) { x = -x; sign = -1.0f; }
    const int i = (int)std::floor(0.5f + 25.0f * x);
    x -= 0.04f * (float)i;
    const float y = kTansigTable[i], dy = 1.0f - y * y;
    return sign * (y + x * dy * (1.0f - y * x));
}
float h_act(int act, float x) { return act == 0 ? h_tansig(x) : (act == 1 ? 0.5f + 0.5f * h_tansig(0.5f * x) : std::max(x, 0.0f)); }
}  // namespace
}  // namespace nnb

extern "C" double nnb_tc_pack_selftest(const unsigned char* bytes, size_t len, int seed) {
    using namespace nnb;
    HostModel hm;
    if (!HostModel::parse(bytes, len, &hm)) return -1.0;
    DeviceModelTc d{};
    std::vector<unsigned char> blob;
    if (!build_model_tc(hm, &d, &blob)) return -2.0;
    for (int p = 0; p < TC_PHASES; p++)
        if ((d.ph[p].n > 0) != (d.ph[p].nk > 0)) return -3.0;
    const int8_t* B = hm.bytes.data();
    const int nd = d.nd, nv = d.nv, nn = d.nn, ndn = d.ndn;
    srand(seed);
    auto rnd = [](float a) { return a * ((float)(rand() % 20001) / 10000.0f - 1.0f); };
    std::vector<float> feat(NB_FEATURES), sv(nv), sn(nn), sd(ndn);
    for (auto& v : feat) v = rnd(3.0f);
    for (auto& v : sv) v = rnd(1.0f);
    for (auto& v : sn) v = rnd(1.0f);
    for (auto& v : sd) v = rnd(1.0f);

    // ---- direct evaluation (src/rnn.rs:251-379) ----
    auto dense = [&](const HostDense& L, const std::vector<float>& in) {
        std::vector<float> out(L.nn);
        for (int o = 0; o < L.nn; o++) {
            float acc = (float)B[L.b_off + o];
            for (int j = 0; j < L.ni; j++) acc += (float)B[L.w_off + (size_t)j * L.nn + o] * in[j];
            out[o] = h_act(L.act, acc * (1.0f / 256.0f));
        }
        return out;
    };
    auto grul = [&](const HostGru& L, const std::vector<float>& in, std::vector<float>& st) {
        const int n = L.nn, st3 = 3 * n;
        std::vector<float> z(n), r(n), h(n);
        for (int o = 0; o < n; o++) {
            float az = (float)B[L.b_off + o], ar = (float)B[L.b_off + n + o];
            for (int j = 0; j < L.ni; j++) { az += (float)B[L.w_off + (size_t)j * st3 + o] * in[j]; ar += (float)B[L.w_off + (size_t)j * st3 + n + o] * in[j]; }
            for (int j = 0; j < n; j++) { az += (float)B[L.r_off + (size_t)j * st3 + o] * st[j]; ar += (float)B[L.r_off + (size_t)j * st3 + n + o] * st[j]; }
            z[o] = h_act(1, az * (1.0f / 256.0f));
            r[o] = h_act(1, ar * (1.0f / 256.0f)) * st[o];
        }
        for (int o = 0; o < n; o++) {
            float ah = (float)B[L.b_off + 2 * n + o];
            for (int j = 0; j < L.ni; j++) ah += (float)B[L.w_off + (size_t)j * st3 + 2 * n + o] * in[j];
            for (int j = 0; j < n; j++) ah += (float)B[L.r_off + (size_t)j * st3 + 2 * n + o] * r[j];
            h[o] = z[o] * st[o] + (1.0f - z[o]) * h_act(L.act, ah * (1.0f / 256.0f));
        }
        st = h;
    };
    std::vector<float> rv = sv, rn = sn, rd = sd;
    std::vector<float> dout = dense(hm.input_dense, feat);
    grul(hm.vad_gru, dout, rv);
    const float rvad = dense(hm.vad_output, rv)[0];
    std::vector<float> nin(dout);
    nin.insert(nin.end(), rv.begin(), rv.end());
    nin.insert(nin.end(), feat.begin(), feat.end());
    grul(hm.noise_gru, nin, rn);
    std::vector<float> din(rv);
    din.insert(din.end(), rn.begin(), rn.end());
    din.insert(din.end(), feat.begin(), feat.end());
    grul(hm.denoise_gru, din, rd);
    std::vector<float> rg = dense(hm.denoise_output, rd);

    // ---- replay of the kernel's phases from the blob ----
    // the kernel zeroes its A operand once; a chunk past it would read other TMEM columns
    std::vector<float> A(A_MAX_HALVES + 16, 0.0f), F(16 * FEAT_CHUNKS, 0.0f), D(D_COLS, std::nanf(""));
    for (int j = A_MAX_HALVES; j < A_MAX_HALVES + 16; j++) A[j] = std::nanf("");
    for (int j = 0; j < NB_FEATURES; j++) F[j] = feat[j];
    for (int j = 0; j < nv; j++) A[d.o_vad + j] = sv[j];
    for (int j = 0; j < nn; j++) A[d.o_noise + j] = sn[j];
    for (int j = 0; j < ndn; j++) A[d.o_den + j] = sd[j];
    auto run = [&](int p) {
        const TcPhase& ph = d.ph[p];
        const __half* wb = reinterpret_cast<const __half*>(blob.data() + ph.w_off);
        if (ph.nk == 0) return;  // no MMA is issued: the columns keep what they held
        for (int n = 0; n < ph.n; n++) {
            float acc = 0.0f;
            for (int kc = 0; kc < ph.nk; kc++)
                for (int kk = 0; kk < 16; kk++) {
                    const int k = kc * 16 + kk;
                    const float a = ph.chunk[kc] >= 0 ? A[ph.chunk[kc] * 16 + kk] : F[(-ph.chunk[kc] - 1) * 16 + kk];
                    acc += a * __half2float(wb[(size_t)(k / 8) * (ph.n * 8) + (size_t)n * 8 + (k % 8)]);
                }
            D[ph.d_col + n] = acc;
        }
    };
    auto bias = [&](int p) { return reinterpret_cast<const float*>(blob.data() + d.ph[p].b_off); };
    run(PH_DENSE);
    for (int o = 0; o < d.p_d; o++) A[d.o_dense + o] = o < nd ? h_act(d.act_dense, (D[d.ph[PH_DENSE].d_col + o] + bias(PH_DENSE)[o]) / 256.0f) : 0.0f;
    std::vector<float> ev = sv, en = sn, ed = sd;
    float evad = 0.0f;
    auto gru = [&](int pzr, int phh, int extra, int act, int n_, int p8, std::vector<float>& st, int a_off) {
        run(pzr);
        if (extra >= 0) run(extra);
        const int dz = d.ph[pzr].d_col;
        for (int o = 0; o < p8; o++) {
            const float hp = o < n_ ? st[o] : 0.0f;
            const float z = h_act(1, (D[dz + o] + bias(pzr)[o]) / 256.0f);
            const float r = o < n_ ? h_act(1, (D[dz + p8 + o] + bias(pzr)[p8 + o]) / 256.0f) * hp : 0.0f;
            D[dz + o] = z;
            A[d.o_rh + o] = r;
        }
        run(phh);
        for (int o = 0; o < p8; o++) {
            const float hp = o < n_ ? st[o] : 0.0f;
            const float c = h_act(act, (D[d.ph[phh].d_col + o] + bias(phh)[o]) / 256.0f);
            const float hn = o < n_ ? D[dz + o] * hp + (1.0f - D[dz + o]) * c : 0.0f;
            if (o < n_) st[o] = hn;
            A[a_off + o] = hn;
        }
    };
    gru(PH_VAD_ZR, PH_VAD_H, -1, d.act_vad, nv, d.p_v, ev, d.o_vad);
    gru(PH_NOISE_ZR, PH_NOISE_H, PH_VAD_OUT, d.act_noise, nn, d.p_n, en, d.o_noise);
    evad = h_act(d.act_vadout, (D[d.ph[PH_VAD_OUT].d_col] + bias(PH_VAD_OUT)[0]) / 256.0f);
    gru(PH_DEN_ZR, PH_DEN_H, -1, d.act_den, ndn, d.p_dn, ed, d.o_den);
    run(PH_OUT);
    double worst = 0.0;
    auto diff = [&](float a, float b) {
        const double e = std::fabs((double)a - (double)b);
        worst = std::isnan(e) ? INFINITY : std::max(worst, e);
    };
    diff(evad, rvad);
    for (int o = 0; o < NB_BANDS; o++) diff(h_act(d.act_out, (D[d.ph[PH_OUT].d_col + o] + bias(PH_OUT)[o]) / 256.0f), rg[o]);
    for (int o = 0; o < nv; o++) diff(ev[o], rv[o]);
    for (int o = 0; o < nn; o++) diff(en[o], rn[o]);
    for (int o = 0; o < ndn; o++) diff(ed[o], rd[o]);
    return worst;
}
