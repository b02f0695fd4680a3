// Fused point-voxel correlation lookup (index + reduce part) -- the HBM-bound headline kernel.
//
// Replaces CorrBlock.get_voxel_feature up to out_conv (reference model/corr.py:47-71) and
// CorrBlock.get_knn_feature up to knn_conv (model/corr.py:75-91) with ONE pass over the K
// candidates of every point.  Data movement:
//   * per-iteration HBM stream = 8 B per candidate (fp32 correlation + int32 candidate id); the
//     reference's materialised [B,N,K,3] xyz tensor is replaced by a per-sample table of 16-byte (x,y,z,0) rows
//     (pvraft_xyz_pad_fwd, once per forward) that a CTA brings into shared memory with bulk copies (TMA) and gathers
//     from with ONE 128-bit load per candidate; pvraft_corr_reorder arranges every row once per forward so that the
//     lanes of a gather hit (nearly) distinct banks;
//   * a warp owns a point; its K*4-byte candidate-id row is brought into the warp's shared-memory stage by
//     the TMA engine (cp.async.bulk + mbarrier complete_tx) -- the row of the NEXT point is requested as soon as the
//     streaming pass of the current one has consumed the stage; the correlation row is prefetched to L2 and read sparsely.
// Per point the warp produces
//   * the 27-cell x `levels` voxel means: candidates inside the coarsest cube (one compare against a host-derived
//     threshold, exact) are compacted in ascending candidate order into a small list; in chunks of 32 entries, lane i
//     derives the cell of entry i at every level, entries of one cell find each other with a warp match and add their
//     correlations to the cell's shared-memory accumulator one rank at a time -> the sums equal a sequential
//     scatter_add over the stored row bit for bit, at a cost that grows with the fullest cell, not with the list;
//   * the 32 nearest candidates: exact threshold on the fp32 distance bits -- a 128-bin shared-memory histogram
//     brackets it, a short bisection with warp-wide population counts finishes (no sort), ties -> lowest slot;
//   * double-precision first/second moments of the kNN 4-vectors, from which the consumer derives the
//     GroupNorm statistics of knn_conv's output without materialising its [B,64,N,32] tensor.
// Index-deciding arithmetic is bit-faithful to the reference's fp32 op sequence: separate rn
// subtract / multiply / add (no FMA contraction), true IEEE division, round-half-even.
#include <math.h>

#include "common.cuh"

namespace pvraft {

constexpr int kLookupThreads = 640;   // 20 warps: bounded by registers (<= 102/thread) and by shared memory
constexpr int kAccCells = 128;        // >= 4 levels * 27 cells

// per-warp shared memory: staged id row (K*4) + valid-slot list (K*2, >= 1 KB: the 128-bin distance histogram of the
// kNN select and its 32 sink bins reuse it) + one 32-entry chunk (256) + kNN slots (128) + per-cell sums and counts (2 * 512) + mbarrier (16);
// rounded to 128 B so that every warp's stage stays 128-byte aligned for the bulk copies
__host__ __device__ constexpr size_t lookup_warp_bytes(int K) {
    return (((size_t)(K < 512 ? 512 : K) * 2 + (size_t)K * 4 + 256 + 128 + 2 * kAccCells * 4 + 16) + 127) & ~(size_t)127;
}

struct LookupParams {
    const void* corr_val;   // [B,N,K] f32, or bf16 bit patterns (uint16) in the reduced-precision state mode
    const void* corr_idx;   // [B,N,K] int32, or uint16 in the reduced-precision state mode
    const float4* tab;   // [B,N] (x,y,z,0) rows of xyz2
    const float* coords; // [B,N,3]
    float* vox;          // [B,N,levels*27]
    float4* knn_sel;     // [B,N,32]
    int32_t* knn_slot;   // [B,N,32] or null
    double* moments;     // [B,16] or null
    int8_t* dbg_cube;    // [B,N,K,levels] or null: the cell id (-1 = outside) this kernel derived for every candidate
    int B, N, K, levels;
    int vox_ld;          // floats per vox row (>= levels*27; the pad is zero-filled)
    float r[4];          // cell edge per level
    float inv_r[4];      // exact reciprocal when r is a power of two
    float thr_c;         // max|d| < thr_c  <=>  |round(d / r_coarsest)| <= 1 on every axis (cube_threshold())
    int warps;           // warps per block actually carved in shared memory
    int chunk;           // points per dynamic work claim
};

template <bool POW2>
__device__ __forceinline__ float div_r(float d, float r, float inv_r) {
    return POW2 ? __fmul_rn(d, inv_r) : __fdiv_rn(d, r);
}

// cell id in [0,27) of offset (dx,dy,dz) at cell edge r, or 0xFF when outside the 3x3x3 cube
// (model/corr.py:54-57: round((xyz - coords) / r), |.| <= 1 on all axes, (qx+1)*9+(qy+1)*3+(qz+1); the cell number is
// formed in fp32 -- small integers, exact -- and converted once)
template <bool POW2>
__device__ __forceinline__ unsigned cell_code(float dx, float dy, float dz, float r, float inv_r) {
    const float qx = rintf(div_r<POW2>(dx, r, inv_r));
    const float qy = rintf(div_r<POW2>(dy, r, inv_r));
    const float qz = rintf(div_r<POW2>(dz, r, inv_r));
    const bool ok = fmaxf(fmaxf(fabsf(qx), fabsf(qy)), fabsf(qz)) <= 1.f;
    const int cell = (int)fmaf(qx, 9.f, fmaf(qy, 3.f, qz + 13.f));
    return ok ? (unsigned)cell : 0xFFu;
}

// ---- mbarrier / bulk-copy (TMA) primitives ----------------------------------------------------------
__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(void* bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(void* bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(void* bar, unsigned parity) {
    asm volatile(
        "{\n\t.reg .pred P1;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n\t"
        "@P1 bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, unsigned bytes, void* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// bring a row of `bytes` bytes into L2 (64 B per lane per step); it is read sparsely (valid + kNN slots) afterwards
__device__ __forceinline__ void prefetch_row(const void* row, int bytes, int lane) {
    const char* r = reinterpret_cast<const char*>(row);
    if (bytes <= 2048) {   // one 64-byte piece per lane covers the row
        if (lane * 64 < bytes) asm volatile("prefetch.global.L2 [%0];" ::"l"(r + lane * 64));
    } else {
        for (int o = lane * 64; o < bytes; o += 32 * 64) asm volatile("prefetch.global.L2 [%0];" ::"l"(r + o));
    }
}

// element types of the per-iteration state: fp32 + int32 (8 B per candidate), or bf16 + uint16 (4 B per candidate, N <= 65536)
template <bool HALF> struct StateT { using val = float; using idx = int32_t; };
template <> struct StateT<true> { using val = uint16_t; using idx = uint16_t; };
__device__ __forceinline__ float load_val(const float* p) { return __ldg(p); }
__device__ __forceinline__ float load_val(const uint16_t* p) { return __uint_as_float((unsigned)__ldg(p) << 16); }   // bf16 -> fp32, exact

// inclusive warp scan of a word of packed 8-bit counters (no field may exceed 255)
__device__ __forceinline__ unsigned warp_scan_packed(unsigned w, int lane) {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned a = __shfl_up_sync(kFull, w, o);
        if (lane >= o) w += a;
    }
    return w;
}

template <int KPL, bool POW2, bool SMEM_TAB, bool HALF>
__global__ void __launch_bounds__(kLookupThreads, 1) k_corr_lookup(const LookupParams p) {
    using val_t = typename StateT<HALF>::val;
    using idx_t = typename StateT<HALF>::idx;
    const val_t* g_val = reinterpret_cast<const val_t*>(p.corr_val);
    const idx_t* g_idx = reinterpret_cast<const idx_t*>(p.corr_idx);
    constexpr int VEC = KPL >= 4 ? 4 : KPL;   // consecutive candidates per lane per block
    constexpr int NJ = KPL / VEC;             // blocks of 32*VEC candidates
    constexpr int K = KPL * 32;
    constexpr unsigned NIB = (1u << VEC) - 1u;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const size_t tab_bytes = SMEM_TAB ? (((size_t)p.N * 16 + 127) & ~(size_t)127) : 0;
    const float4* s_tab = reinterpret_cast<const float4*>(smem_raw);   // [N] (x,y,z,0), a verbatim copy of the sample's table
    const int w = warp_id();
    int lane;   // pinned: left to itself the compiler re-derives threadIdx.x & 31 (S2R + LOP) ~9 times per point
    asm volatile("mov.u32 %0, %%laneid;" : "=r"(lane));
    unsigned char* wbase = smem_raw + tab_bytes + (size_t)w * lookup_warp_bytes(K);
    int* s_stage = reinterpret_cast<int*>(wbase);                        // [K] candidate ids of the point being streamed
    constexpr int VL = (K < 512 ? 512 : K) * 2;   // >= 640 B: 128 histogram bins + 32 per-lane sinks
    unsigned short* s_vlist = reinterpret_cast<unsigned short*>(wbase + K * 4);   // [K] slots inside the coarsest cube
    int* s_hist = reinterpret_cast<int*>(wbase + K * 4);                 // [128 + 32] kNN distance histogram (after the list is dead)
    int* s_slots = reinterpret_cast<int*>(wbase + K * 4 + VL + 256);     // [32]  kNN slots
    float* s_acc = reinterpret_cast<float*>(wbase + K * 4 + VL + 384);   // [128] per-cell correlation sums, index level*27 + cell
    int* s_cnt = reinterpret_cast<int*>(wbase + K * 4 + VL + 384 + kAccCells * 4);                      // [128] per-cell counts
    unsigned long long* s_bar = reinterpret_cast<unsigned long long*>(wbase + K * 4 + VL + 384 + 2 * kAccCells * 4);
    pdl_trigger();   // the next kernel may be staged while this one drains
    const bool active_warp = w < p.warps;
    __shared__ int s_next;   // next unclaimed point of the current segment (static mode: warps take points dynamically)
    __shared__ unsigned long long s_tabbar;
    // 1/c in double for c = 0..K: (float)(double(sum) * rcp[c]) is the correctly rounded fp32 quotient sum/c for
    // every integer c <= 2^20 (x/c is never within 2^-34 relative of a rounding boundary), without a division
    double* s_rcp = reinterpret_cast<double*>(smem_raw + tab_bytes + (size_t)p.warps * lookup_warp_bytes(K));
    for (int i = threadIdx.x; i <= K; i += blockDim.x) s_rcp[i] = i > 0 ? 1.0 / (double)i : 1.0;

    if (active_warp && lane == 0) mbar_init(s_bar, 1);
    if (threadIdx.x == 0) mbar_init(&s_tabbar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    __syncthreads();

    // Work distribution.  With a moment buffer (zeroed by the caller) and at least one CTA per sample, the CTAs of a sample
    // share its points dynamically: warps claim chunks of 4 consecutive points from a counter kept in the unused 16th moment
    // slot (the per-point cost varies ~2x with the local density, and a cloud's points are usually stored region by region,
    // so equal contiguous shares left ~20 % of the SM time idle).  Otherwise: equal contiguous shares of B*N.
    const bool dyn = p.moments != nullptr && (int)gridDim.x >= p.B;
    const long long total = (long long)p.B * p.N;
    long long pt_begin, pt_end;
    if (dyn) {
        const int b = (int)((long long)blockIdx.x * p.B / gridDim.x);
        pt_begin = (long long)b * p.N;
        pt_end = pt_begin + p.N;
    } else {
        split_range(total, gridDim.x, blockIdx.x, pt_begin, pt_end);
    }
    const int L = p.levels;
    const int nvox = L * 27;
    const unsigned lt_mask = (1u << lane) - 1u;
    unsigned phase = 0, tab_phase = 0;
    bool waited = false;
    const int kChunk = p.chunk;
    const unsigned one = (unsigned)min(p.chunk, 1);   // == 1, but not to the compiler (see the histogram below)

    // (Letting a CTA that has finished its sample adopt points of other samples -- one more 128 KB table load each -- was
    //  measured: 104 us instead of 102.8, the kernel's tail is not a per-sample imbalance.)
    long long seg = pt_begin;
    while (seg < pt_end) {
        const int b = (int)(seg / p.N);
        long long seg_end = (long long)(b + 1) * p.N;
        if (seg_end > pt_end) seg_end = pt_end;
        const float4* tab_g = p.tab + (size_t)b * p.N;
        int* counter = dyn ? reinterpret_cast<int*>(p.moments + (size_t)b * PVRAFT_MOMENTS + 15) : nullptr;
        auto claim_chunk = [&]() -> long long {   // first point of the next unclaimed chunk of this sample
            int c = 0;
            if (lane == 0) c = atomicAdd(counter, kChunk);
            return seg + __shfl_sync(kFull, c, 0);
        };
        __syncthreads();   // previous segment's readers are done (table and point counter)
        if (SMEM_TAB && threadIdx.x == 0) {
            // the sample's table: N*16 bytes by the TMA engine (written once per forward, long before this launch, so the
            // request may precede griddepcontrol.wait and overlap the previous kernel's tail)
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            const unsigned bytes = (unsigned)p.N * 16u;
            mbar_expect_tx(&s_tabbar, bytes);
            for (unsigned off = 0; off < bytes; off += 32768u)
                bulk_g2s(smem_raw + off, reinterpret_cast<const unsigned char*>(tab_g) + off, min(32768u, bytes - off), &s_tabbar);
        }
        if (threadIdx.x == 0) s_next = 2 * p.warps;   // static mode: warp w starts with points w and w + warps
        // Launched with PDL: only the set-up above overlaps the previous kernel's tail.  Everything below reads what
        // earlier kernels of the stream wrote -- the zeroed per-sample work counter (griddepcontrol.wait is what makes
        // the predecessor's stores visible), the query coordinates -- or writes buffers they may still read.
        if (!waited) { pdl_wait(); waited = true; }
        // this warp's first two points
        long long pt0 = seg + w, nxt0 = seg + w + p.warps;
        int left0 = 0;   // points after nxt0 that remain in nxt0's chunk (dynamic mode)
        if (dyn && active_warp) { pt0 = claim_chunk(); nxt0 = pt0 + 1; left0 = kChunk - 2; }
        if (active_warp && pt0 < seg_end) {   // kick off this warp's first row
            if (lane == 0) {
                mbar_expect_tx(s_bar, K * sizeof(idx_t));
                bulk_g2s(s_stage, g_idx + pt0 * K, K * sizeof(idx_t), s_bar);
            }
            prefetch_row(g_val + pt0 * K, K * sizeof(val_t), lane);
        }
        if (SMEM_TAB) { mbar_wait(&s_tabbar, tab_phase); tab_phase ^= 1u; }
        __syncthreads();   // s_next
        double mom[14];
#pragma unroll
        for (int i = 0; i < 14; ++i) mom[i] = 0.0;

        if (active_warp) {
            int left = left0, done = 0;
            long long nxt = nxt0;
            for (long long pt = pt0; pt < seg_end; ++done) {
                const float cx = __ldg(p.coords + pt * 3 + 0);
                const float cy = __ldg(p.coords + pt * 3 + 1);
                const float cz = __ldg(p.coords + pt * 3 + 2);
                const val_t* rv = g_val + pt * K;
                const idx_t* ri = g_idx + pt * K;
                if (p.dbg_cube) {
                    for (int i = lane; i < K * L; i += 32) p.dbg_cube[pt * K * L + i] = (int8_t)-1;
                }
                // per-cell accumulators of this point
                *reinterpret_cast<float4*>(s_acc + lane * 4) = make_float4(0.f, 0.f, 0.f, 0.f);
                *reinterpret_cast<int4*>(s_cnt + lane * 4) = make_int4(0, 0, 0, 0);
                mbar_wait(s_bar, phase);
                phase ^= 1u;

                // ---- stream the staged row: slot(j,s) = j*32*VEC + lane*VEC + s -------------------------
                unsigned dist[KPL];       // fp32 bits of the (non-negative) squared distance
                unsigned valid_bits = 0;  // bit e: candidate e of this lane lies inside the coarsest 3x3x3 cube
                const float thr = p.thr_c;
                unsigned long long cxy;
                asm("mov.b64 %0, {%1, %2};" : "=l"(cxy) : "f"(cx), "f"(cy));
#pragma unroll
                for (int j = 0; j < NJ; ++j) {
                    int ci[VEC];
                    if (VEC == 4 && HALF) {
                        const uint2 c = reinterpret_cast<const uint2*>(s_stage)[j * 32 + lane];   // four uint16 ids
                        ci[0] = (int)(c.x & 0xFFFFu); ci[1 % VEC] = (int)(c.x >> 16); ci[2 % VEC] = (int)(c.y & 0xFFFFu); ci[3 % VEC] = (int)(c.y >> 16);
                    } else if (VEC == 4) {
                        const int4 c = reinterpret_cast<const int4*>(s_stage)[j * 32 + lane];
                        ci[0] = c.x; ci[1 % VEC] = c.y; ci[2 % VEC] = c.z; ci[3 % VEC] = c.w;
                    } else {
#pragma unroll
                        for (int s = 0; s < VEC; ++s) ci[s] = (int)reinterpret_cast<const idx_t*>(s_stage)[j * 32 * VEC + lane * VEC + s];
                    }
#pragma unroll
                    for (int s = 0; s < VEC; ++s) {
                        const float4 q = SMEM_TAB ? s_tab[ci[s]] : __ldg(tab_g + ci[s]);
                        // (dx,dy) and their squares as packed fp32x2 operations (one issue slot each; every component is an
                        // IEEE round-to-nearest subtract / multiply, exactly the scalar sequence of model/corr.py:78-79)
                        float dx, dy, sx, sy;
                        {
                            unsigned long long qxy, dxy, sxy;
                            asm("mov.b64 %0, {%1, %2};" : "=l"(qxy) : "f"(q.x), "f"(q.y));
                            asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(dxy) : "l"(qxy), "l"(cxy));
                            asm("mul.rn.f32x2 %0, %1, %1;" : "=l"(sxy) : "l"(dxy));
                            asm("mov.b64 {%0, %1}, %2;" : "=f"(dx), "=f"(dy) : "l"(dxy));
                            asm("mov.b64 {%0, %1}, %2;" : "=f"(sx), "=f"(sy) : "l"(sxy));
                        }
                        const float dz = __fsub_rn(q.z, cz);
                        const float d2 = __fadd_rn(__fadd_rn(sx, sy), __fmul_rn(dz, dz));
                        dist[j * VEC + s] = __float_as_uint(d2);
                        // |round(d/r)| <= 1 on every axis  <=>  fl(max|d| / r) < 1.5 (round-half-even sends 1.5 to 2;
                        // x -> fl(x/r) is monotone)  <=>  max|d| < thr, thr = the smallest float whose quotient reaches 1.5
                        const float amax = fmaxf(fmaxf(fabsf(dx), fabsf(dy)), fabsf(dz));
                        valid_bits |= (amax < thr ? 1u : 0u) << (j * VEC + s);
                    }
                }
                __syncwarp();
                // the stage is consumed (later id reads go to the L2-resident row): request the next point's row now
                if (nxt < seg_end) {
                    if (lane == 0) {
                        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                        mbar_expect_tx(s_bar, K * sizeof(idx_t));
                        bulk_g2s(s_stage, g_idx + nxt * K, K * sizeof(idx_t), s_bar);
                    }
                    prefetch_row(g_val + nxt * K, K * sizeof(val_t), lane);   // correlation row -> L2; read sparsely below
                }

                // ---- voxel means -----------------------------------------------------------------------
                // (1) ordered compaction of the valid slots: one packed warp scan gives every lane its offset in
                //     every block j, so the list is in ascending slot order (the order of a sequential scatter_add)
                if (__any_sync(kFull, valid_bits != 0u)) {
                    int list_n = 0;
                    unsigned w0 = 0, w1 = 0;
#pragma unroll
                    for (int j = 0; j < NJ; ++j) {
                        const unsigned c = __popc((valid_bits >> (j * VEC)) & NIB);
                        if (j < 4) w0 |= c << (8 * j); else w1 |= c << (8 * (j - 4));
                    }
                    const unsigned i0 = warp_scan_packed(w0, lane);
                    const unsigned t0 = __shfl_sync(kFull, i0, 31);
                    unsigned i1 = 0, t1 = 0;
                    if (NJ > 4) { i1 = warp_scan_packed(w1, lane); t1 = __shfl_sync(kFull, i1, 31); }
                    const unsigned e0 = i0 - w0, e1 = i1 - w1;
#pragma unroll
                    for (int j = 0; j < NJ; ++j) {
                        const unsigned ex = j < 4 ? (e0 >> (8 * j)) & 0xFFu : (e1 >> (8 * (j - 4))) & 0xFFu;
                        const unsigned tt = j < 4 ? (t0 >> (8 * j)) & 0xFFu : (t1 >> (8 * (j - 4))) & 0xFFu;
                        unsigned nib = (valid_bits >> (j * VEC)) & NIB;
                        int pos = list_n + (int)ex;
                        while (nib) {
                            const int s = __ffs(nib) - 1;
                            nib &= nib - 1;
                            s_vlist[pos++] = (unsigned short)(j * 32 * VEC + lane * VEC + s);
                        }
                        list_n += (int)tt;
                    }
                    __syncwarp();
                    // (2) chunks of 32 entries: lane i derives the cells of entry i at every level; (3) the entries of one
                    //     cell (warp match) add to its accumulator one rank at a time, lowest slot first
                    for (int c0 = 0; c0 < list_n; c0 += 32) {
                        const int n = min(32, list_n - c0);
                        unsigned code = 0xFFFFFFFFu;
                        float val = 0.f;
                        if (lane < n) {
                            const int slot = s_vlist[c0 + lane];
                            const int id = (int)__ldg(ri + slot);
                            val = load_val(rv + slot);
                            const float4 q = SMEM_TAB ? s_tab[id] : __ldg(tab_g + id);
                            const float dx = __fsub_rn(q.x, cx), dy = __fsub_rn(q.y, cy), dz = __fsub_rn(q.z, cz);
#pragma unroll
                            for (int l = 0; l < 4; ++l) {
                                if (l < L) {
                                    const unsigned c = cell_code<POW2>(dx, dy, dz, p.r[l], p.inv_r[l]);
                                    code = (code & ~(0xFFu << (8 * l))) | (c << (8 * l));
                                    if (p.dbg_cube) p.dbg_cube[(pt * K + slot) * L + l] = (int8_t)c;
                                }
                            }
                        }
#pragma unroll
                        for (int l = 0; l < 4; ++l) {
                            if (l < L) {
                                const unsigned c = (code >> (8 * l)) & 0xFFu;
                                const bool act = c != 0xFFu;
                                if (__any_sync(kFull, act)) {
                                    const unsigned m = __match_any_sync(kFull, c);
                                    const unsigned rank = __popc(m & lt_mask), gsize = __popc(m);
                                    const unsigned maxg = __reduce_max_sync(kFull, act ? gsize : 0u);
                                    const int cell = act ? l * 27 + (int)c : 0;
                                    if (act && rank == 0u) s_cnt[cell] += (int)gsize;
                                    for (unsigned r = 0; r < maxg; ++r) {
                                        if (act && rank == r) s_acc[cell] = __fadd_rn(s_acc[cell], val);
                                        __syncwarp();
                                    }
                                }
                            }
                        }
                    }
                }
                __syncwarp();
                {   // sum / clamp(count, 1, N) (corr.py:65-66; rcp[0] = 1) of every cell, and zeros in the row padding
                    float* vo = p.vox + pt * p.vox_ld;
#pragma unroll
                    for (int i = 0; i < 3; ++i) {   // columns 0..95 (3 levels: 81 cells + the padding of the 96-wide layout)
                        const int o = lane + 32 * i;
                        const float v = (float)((double)s_acc[o] * s_rcp[s_cnt[o]]);   // cells >= nvox were never touched: 0 * 1
                        if (o < p.vox_ld) vo[o] = v;
                    }
                    for (int o = lane + 96; o < p.vox_ld; o += 32) vo[o] = o < nvox ? (float)((double)s_acc[o] * s_rcp[s_cnt[o]]) : 0.f;
                }
                __syncwarp();

                // ---- kNN: a threshold T with count(d <= T) >= 32 > count(d < T) ---------------------------
                unsigned lmin = dist[0];
#pragma unroll
                for (int e = 1; e < KPL; ++e) lmin = min(lmin, dist[e]);
                unsigned hi = __reduce_max_sync(kFull, lmin);   // 32 distinct candidates are <= hi
                unsigned lo;
                int c_lo, c_hi;
                {
                    // 128-bucket histogram over the top 4 octaves below `hi` (bucket edges are exact in the bit
                    // pattern): one pass brackets the 32nd smallest distance inside a single bucket
                    const unsigned base = hi > 0x01FFFFFFu ? hi - 0x01FFFFFFu : 0u;
                    *reinterpret_cast<int4*>(s_hist + lane * 4) = make_int4(0, 0, 0, 0);
                    __syncwarp();
                    unsigned char* hist_b = reinterpret_cast<unsigned char*>(s_hist);
                    const unsigned dummy = 512u + 4u * (unsigned)lane;   // bins 128..159: one private sink per lane
#pragma unroll
                    for (int e = 0; e < KPL; ++e) {
                        // bucket = (max(d, base) - base) >> 18, as a byte offset: ((.) >> 16) & ~3.  Candidates beyond `hi`
                        // add to the lane's sink instead of being skipped: an `if` (or a predicated red) around a shared-memory
                        // atomic compiles to a branch + reconvergence per candidate, 10 instructions instead of 7
                        const unsigned off = ((max(dist[e], base) - base) >> 16) & 0x1FCu;
                        atomicAdd(reinterpret_cast<unsigned*>(hist_b + (dist[e] <= hi ? off : dummy)), one);
                    }
                    __syncwarp();
                    const int4 h = *reinterpret_cast<const int4*>(s_hist + lane * 4);
                    const int mine = h.x + h.y + h.z + h.w;
                    int incl = mine;
#pragma unroll
                    for (int o = 1; o < 32; o <<= 1) {
                        const int a = __shfl_up_sync(kFull, incl, o);
                        if (lane >= o) incl += a;
                    }
                    const int src = __ffs(__ballot_sync(kFull, incl >= PVRAFT_KNN)) - 1;   // exists: count(d <= hi) >= 32
                    int c = incl - mine, bq = 0, cl = c, ch = c + h.x;
                    if (ch < PVRAFT_KNN) { cl = ch; ch += h.y; bq = 1; }
                    if (ch < PVRAFT_KNN) { cl = ch; ch += h.z; bq = 2; }
                    if (ch < PVRAFT_KNN) { cl = ch; ch += h.w; bq = 3; }
                    const int B = __shfl_sync(kFull, lane * 4 + bq, src);
                    c_lo = __shfl_sync(kFull, cl, src);
                    c_hi = __shfl_sync(kFull, ch, src);
                    lo = B == 0 ? 0u : base + ((unsigned)B << 18);
                    hi = base + ((unsigned)(B + 1) << 18) - 1u;
                }
                // invariant: count(d <= hi) = c_hi >= 32, count(d < lo) = c_lo < 32; finish inside the bucket
                while (c_hi != PVRAFT_KNN && lo < hi) {
                    const unsigned mid = lo + ((hi - lo) >> 1);
                    int c = 0;
#pragma unroll
                    for (int e = 0; e < KPL; ++e) c += dist[e] <= mid ? 1 : 0;
                    c = __reduce_add_sync(kFull, c);
                    if (c >= PVRAFT_KNN) { hi = mid; c_hi = c; } else { lo = mid + 1; c_lo = c; }
                }
                const unsigned T = hi;
                if (c_hi == PVRAFT_KNN) {
                    // common case: exactly 32 candidates are <= T
                    unsigned m_le = 0;
#pragma unroll
                    for (int e = 0; e < KPL; ++e) m_le |= (dist[e] <= T ? 1u : 0u) << e;
                    int off = __popc(m_le);
                    const int n_le = off;
#pragma unroll
                    for (int o = 1; o < 32; o <<= 1) {
                        const int a = __shfl_up_sync(kFull, off, o);
                        if (lane >= o) off += a;
                    }
                    off -= n_le;
                    while (m_le) {
                        const int e = __ffs(m_le) - 1;
                        m_le &= m_le - 1;
                        s_slots[off++] = (e / VEC) * 32 * VEC + lane * VEC + (e % VEC);
                    }
                } else {
                    // exact-distance ties at the 32nd place: everything strictly closer, then ties in (lane, e) order
                    unsigned m_lt = 0, m_eq = 0;
#pragma unroll
                    for (int e = 0; e < KPL; ++e) {
                        m_lt |= (dist[e] < T ? 1u : 0u) << e;
                        m_eq |= (dist[e] == T ? 1u : 0u) << e;
                    }
                    const int n_lt = __popc(m_lt), n_eq = __popc(m_eq);
                    int off_lt = n_lt, off_eq = n_eq;   // inclusive scans over lanes
#pragma unroll
                    for (int o = 1; o < 32; o <<= 1) {
                        const int a = __shfl_up_sync(kFull, off_lt, o), c = __shfl_up_sync(kFull, off_eq, o);
                        if (lane >= o) { off_lt += a; off_eq += c; }
                    }
                    const int tot_lt = __shfl_sync(kFull, off_lt, 31);
                    off_lt -= n_lt;
                    off_eq += tot_lt - n_eq;
                    while (m_lt) {
                        const int e = __ffs(m_lt) - 1;
                        m_lt &= m_lt - 1;
                        s_slots[off_lt++] = (e / VEC) * 32 * VEC + lane * VEC + (e % VEC);
                    }
                    while (m_eq) {
                        const int e = __ffs(m_eq) - 1;
                        m_eq &= m_eq - 1;
                        if (off_eq < PVRAFT_KNN) s_slots[off_eq] = (e / VEC) * 32 * VEC + lane * VEC + (e % VEC);
                        ++off_eq;
                    }
                }
                __syncwarp();
                {
                    const int slot = s_slots[lane];
                    const float c = load_val(rv + slot);
                    const int id = (int)__ldg(ri + slot);
                    const float4 q = SMEM_TAB ? s_tab[id] : __ldg(tab_g + id);
                    const float dx = __fsub_rn(q.x, cx), dy = __fsub_rn(q.y, cy), dz = __fsub_rn(q.z, cz);
                    p.knn_sel[pt * 32 + lane] = make_float4(c, dx, dy, dz);
                    if (p.knn_slot) p.knn_slot[pt * 32 + lane] = slot;
                    const double f0 = c, f1 = dx, f2 = dy, f3 = dz;
                    mom[0] += f0; mom[1] += f1; mom[2] += f2; mom[3] += f3;
                    mom[4] += f0 * f0; mom[5] += f0 * f1; mom[6] += f0 * f2; mom[7] += f0 * f3;
                    mom[8] += f1 * f1; mom[9] += f1 * f2; mom[10] += f1 * f3;
                    mom[11] += f2 * f2; mom[12] += f2 * f3; mom[13] += f3 * f3;
                }
                __syncwarp();
                // the point after next (its row is requested once `nxt` has been streamed)
                pt = nxt;
                if (dyn) {
                    if (left > 0) { ++nxt; --left; } else { nxt = claim_chunk(); left = kChunk - 1; }
                } else {
                    int claim = 0;
                    if (lane == 0) claim = atomicAdd(&s_next, 1);
                    nxt = seg + __shfl_sync(kFull, claim, 0);
                }
            }
            if (p.moments) {
                // 16 per-lane partial sums -> one total per lane pair with a reduce-scatter butterfly (15 + 1 double shuffles
                // instead of 14 x 5): after the step with partner lane ^ d a lane keeps the half of its values selected by that
                // bit of its id, so lane l ends up with the total of value ((l >> 1) & 15)
                double v[16];
#pragma unroll
                for (int i = 0; i < 14; ++i) v[i] = mom[i];
                v[14] = (double)done;   // x 32 lanes = the number of kNN edges this warp produced
                v[15] = 0.0;
#pragma unroll
                for (int d = 16, h = 8; d >= 2; d >>= 1, h >>= 1) {
                    const bool up = (lane & d) != 0;
#pragma unroll
                    for (int i = 0; i < h; ++i) {
                        const double send = up ? v[i] : v[i + h];
                        const double keep = up ? v[i + h] : v[i];
                        v[i] = keep + __shfl_xor_sync(kFull, send, d);
                    }
                }
                v[0] += __shfl_xor_sync(kFull, v[0], 1);
                const int which = (lane >> 1) & 15;
                if ((lane & 1) == 0 && which < 15 && v[0] != 0.0) atomicAdd(p.moments + (size_t)b * PVRAFT_MOMENTS + which, v[0]);
            }
        }
        seg = seg_end;
    }
}

// (x,y,z) -> (x,y,z,0): the 16-byte rows the lookup kernel gathers with one 128-bit load
__global__ void k_xyz_pad(const float* __restrict__ xyz, long long rows, float4* __restrict__ out) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < rows) out[i] = make_float4(__ldg(xyz + 3 * i), __ldg(xyz + 3 * i + 1), __ldg(xyz + 3 * i + 2), 0.f);
}

// Bank-aware arrangement of one row's candidates (once per forward).  The lookup gathers the 16-byte table rows of 32
// candidates per instruction (slots {j*32*VEC + lane*VEC + s} for a fixed (j,s)); a 128-bit shared-memory load is served one
// quarter-warp (8 lanes x 16 B = all 32 banks) at a time, so it is conflict-free when the 8 ids of every aligned group of 8
// lanes are distinct modulo 8.  Candidates are ranked inside their class (id mod 8) in stable order; the k-th member of class c
// goes to lane c + 8*(k mod 4) of gather group k/4.  A class holds K/8 such places; members beyond that (a random row is a few
// per class over) fill the places the smaller classes leave free, in order.  One warp per row; deterministic (ranks come
// from warp match, not from atomics).
template <int KPL>
__global__ void __launch_bounds__(256) k_corr_reorder(const float* __restrict__ val_in, const int32_t* __restrict__ idx_in,
                                                       long long rows, float* __restrict__ val_out, int32_t* __restrict__ idx_out) {
    constexpr int VEC = KPL >= 4 ? 4 : KPL;
    constexpr int K = KPL * 32;
    constexpr int CAP = 4 * KPL;   // places per class
    __shared__ int s_cur[8][32];   // per warp: [0..7] class counts, [8..15] free places before class c, [16..23] overflow before class c
    const int lane = lane_id(), w = warp_id();
    const long long row = (long long)blockIdx.x * 8 + w;
    if (row >= rows) return;
    const unsigned lt_mask = (1u << lane) - 1u;
    float v[KPL];
    int id[KPL];
    int rank[KPL];
    s_cur[w][lane] = 0;
    __syncwarp();
#pragma unroll
    for (int e = 0; e < KPL; ++e) {
        v[e] = __ldg(val_in + row * K + e * 32 + lane);
        id[e] = __ldg(idx_in + row * K + e * 32 + lane);
        const int c = id[e] & 7;
        const unsigned m = __match_any_sync(kFull, c);
        rank[e] = s_cur[w][c] + __popc(m & lt_mask);   // stable: input order e*32 + lane
        __syncwarp();
        if (lane == __ffs(m) - 1) s_cur[w][c] += __popc(m);
        __syncwarp();
    }
    {
        const int n = lane < 8 ? s_cur[w][lane] : 0;
        const int fr = lane < 8 ? max(0, CAP - n) : 0, ov = lane < 8 ? max(0, n - CAP) : 0;
        int f = fr, o = ov;
#pragma unroll
        for (int d = 1; d < 8; d <<= 1) {
            const int a = __shfl_up_sync(kFull, f, d), c = __shfl_up_sync(kFull, o, d);
            if (lane >= d) { f += a; o += c; }
        }
        if (lane < 8) { s_cur[w][8 + lane] = f - fr; s_cur[w][16 + lane] = o - ov; }
    }
    __syncwarp();
#pragma unroll
    for (int e = 0; e < KPL; ++e) {
        int c = id[e] & 7, k = rank[e];
        if (k >= CAP) {   // overflow member number oi of the row takes the oi-th free place
            const int oi = s_cur[w][16 + c] + (k - CAP);
            int cc = 0;
#pragma unroll
            for (int q = 1; q < 8; ++q) cc = s_cur[w][8 + q] <= oi && s_cur[w][q] < CAP ? q : cc;   // last class whose free run starts at or before oi
            c = cc;
            k = s_cur[w][cc] + (oi - s_cur[w][8 + cc]);
        }
        const int g = k >> 2, ln = c + 8 * (k & 3);
        const int slot = (g / VEC) * 32 * VEC + ln * VEC + (g % VEC);
        val_out[row * K + slot] = v[e];
        idx_out[row * K + slot] = id[e];
    }
}

static bool is_pow2f(float r) {
    int e;
    return r > 0.f && frexpf(r, &e) == 0.5f;
}

// The smallest float t with fl(t / r) >= 1.5 in IEEE fp32 division: since x -> fl(x / r) is monotone,
// fl(x / r) < 1.5  <=>  x < t, and |round-half-even(fl(x / r))| <= 1  <=>  fl(|x| / r) < 1.5.  For a power-of-two r this is
// 1.5 * r exactly; in general the search below walks at most a few ulps from that product.
static float cube_threshold(float r) {
    volatile float t = 1.5f * r;
    auto q = [&](float x) { volatile float v = x / r; return (float)v; };
    while (q(t) >= 1.5f) t = nextafterf(t, 0.f);
    while (q(t) < 1.5f) t = nextafterf(t, INFINITY);
    return t;
}

template <int KPL, bool POW2, bool HALF>
static int launch_lookup(LookupParams& p, cudaStream_t st) {
    const int K = KPL * 32;
    const size_t per_warp = lookup_warp_bytes(K);
    const size_t tab = (((size_t)p.N * 16 + 127) & ~(size_t)127);
    const size_t rcp_bytes = (size_t)(K + 1) * sizeof(double) + 8;
    const bool smem_tab = tab + 8 * per_warp + rcp_bytes <= (size_t)kSmemBudget;
    const size_t avail = (size_t)kSmemBudget - (smem_tab ? tab : 0) - rcp_bytes;
    int warps = (int)(avail / per_warp);
    if (warps > kLookupThreads / 32) warps = kLookupThreads / 32;
    if (warps < 1) return fail(PVRAFT_ERR_SMEM, "corr_lookup: K=%d does not fit shared memory", K);
    p.warps = warps;
    p.chunk = 2;   // in-situ sweep at B=8, N=8192 (v8 kernel): 1 -> 108.4 us, 2 -> 102.6, 3 -> 103.3, 4 -> 103.8, 6 -> 105.0, 8 -> 105.3
    if (const char* e = getenv("PVRAFT_LOOKUP_CHUNK")) { const int v = atoi(e); if (v >= 1 && v <= 64) p.chunk = v; }
    const size_t rcp = (size_t)(K + 1) * sizeof(double) + 8;
    const size_t smem = (smem_tab ? tab : 0) + warps * per_warp + rcp;
    const long long total = (long long)p.B * p.N;
    int grid = sm_count();
    if ((long long)grid * warps > total) grid = (int)((total + warps - 1) / warps);
    if (grid < 1) grid = 1;
    int rc;
    if (smem_tab) {
        auto k = k_corr_lookup<KPL, POW2, true, HALF>;
        if ((rc = opt_in_smem(k, smem))) return rc;
        launch_pdl(k, grid, kLookupThreads, smem, st, p);
    } else {
        auto k = k_corr_lookup<KPL, POW2, false, HALF>;
        if ((rc = opt_in_smem(k, smem))) return rc;
        launch_pdl(k, grid, kLookupThreads, smem, st, p);
    }
    return check_launch("corr_lookup");
}

}  // namespace pvraft

using namespace pvraft;

extern "C" int pvraft_corr_reorder(const float* val_in, const int32_t* idx_in, int64_t rows, int K, float* val_out,
                                   int32_t* idx_out, void* stream) {
    if (!val_in || !idx_in || !val_out || !idx_out || rows <= 0) return fail(PVRAFT_ERR_BAD_ARG, "corr_reorder: bad argument");
    if (val_in == val_out || idx_in == idx_out) return fail(PVRAFT_ERR_BAD_ARG, "corr_reorder: in-place operation is not supported");
    const unsigned blocks = (unsigned)((rows + 7) / 8);
    cudaStream_t st = (cudaStream_t)stream;
    switch (K) {
        case 32: k_corr_reorder<1><<<blocks, 256, 0, st>>>(val_in, idx_in, rows, val_out, idx_out); break;
        case 64: k_corr_reorder<2><<<blocks, 256, 0, st>>>(val_in, idx_in, rows, val_out, idx_out); break;
        case 128: k_corr_reorder<4><<<blocks, 256, 0, st>>>(val_in, idx_in, rows, val_out, idx_out); break;
        case 256: k_corr_reorder<8><<<blocks, 256, 0, st>>>(val_in, idx_in, rows, val_out, idx_out); break;
        case 512: k_corr_reorder<16><<<blocks, 256, 0, st>>>(val_in, idx_in, rows, val_out, idx_out); break;
        case 1024: k_corr_reorder<32><<<blocks, 256, 0, st>>>(val_in, idx_in, rows, val_out, idx_out); break;
        default: return fail(PVRAFT_ERR_UNSUPPORTED, "corr_reorder: truncate_k=%d (supported: 32,64,128,256,512,1024)", K);
    }
    return check_launch("corr_reorder");
}

extern "C" int pvraft_xyz_pad_fwd(const float* xyz, int64_t rows, float* out, void* stream) {
    if (!xyz || !out || rows <= 0) return fail(PVRAFT_ERR_BAD_ARG, "xyz_pad: bad argument");
    k_xyz_pad<<<(unsigned)((rows + 255) / 256), 256, 0, (cudaStream_t)stream>>>(xyz, rows, reinterpret_cast<float4*>(out));
    return check_launch("xyz_pad");
}

static int corr_lookup_any(const void* corr_val, const void* corr_idx, bool half, const float* xyz2_pad, const float* coords, int B, int N,
                           int K, int levels, float base_scale, float* vox, int vox_ld, float* knn_sel, int32_t* knn_slot, double* moments,
                           int8_t* dbg_cube, void* stream) {
    if (!corr_val || !corr_idx || !xyz2_pad || !coords || !vox || !knn_sel) return fail(PVRAFT_ERR_BAD_ARG, "corr_lookup: null pointer");
    if (B <= 0 || N <= 0) return fail(PVRAFT_ERR_BAD_ARG, "corr_lookup: B=%d N=%d", B, N);
    if (levels < 1 || levels > 4) return fail(PVRAFT_ERR_UNSUPPORTED, "corr_lookup: levels=%d (1..4 supported)", levels);
    if (!(base_scale > 0.f)) return fail(PVRAFT_ERR_BAD_ARG, "corr_lookup: base_scale must be > 0");
    if ((reinterpret_cast<uintptr_t>(xyz2_pad) & 15u) || (reinterpret_cast<uintptr_t>(corr_idx) & 15u))
        return fail(PVRAFT_ERR_BAD_ARG, "corr_lookup: xyz2_pad and corr_idx must be 16-byte aligned (bulk copies)");
    if (half && N > 65536) return fail(PVRAFT_ERR_UNSUPPORTED, "corr_lookup: uint16 candidate ids need N <= 65536 (N=%d)", N);
    LookupParams p{};
    p.corr_val = corr_val; p.corr_idx = corr_idx; p.tab = reinterpret_cast<const float4*>(xyz2_pad); p.coords = coords;
    p.vox = vox; p.knn_sel = reinterpret_cast<float4*>(knn_sel); p.knn_slot = knn_slot; p.moments = moments;
    p.dbg_cube = dbg_cube;
    p.B = B; p.N = N; p.K = K; p.levels = levels;
    p.vox_ld = vox_ld > 0 ? vox_ld : levels * 27;
    if (p.vox_ld < levels * 27 || p.vox_ld > levels * 27 + 32) return fail(PVRAFT_ERR_BAD_ARG, "corr_lookup: vox_ld=%d", vox_ld);
    bool pow2 = true;
    for (int l = 0; l < 4; ++l) {
        // model/corr.py:53: r = base_scale * 2**i evaluated in double, then used as an fp32 divisor
        const float r = (float)((double)base_scale * (double)(1 << l));
        p.r[l] = r;
        p.inv_r[l] = 1.0f / r;
        if (l < levels && !is_pow2f(r)) pow2 = false;
    }
    p.thr_c = cube_threshold(p.r[levels - 1]);
    cudaStream_t st = (cudaStream_t)stream;
#define PVRAFT_LOOKUP_CASE(KPL_)                                                            \
    case KPL_ * 32:                                                                         \
        return pow2 ? launch_lookup<KPL_, true, false>(p, st) : launch_lookup<KPL_, false, false>(p, st);
#define PVRAFT_LOOKUP_CASE_H(KPL_)                                                          \
    case KPL_ * 32:                                                                         \
        return pow2 ? launch_lookup<KPL_, true, true>(p, st) : launch_lookup<KPL_, false, true>(p, st);
    if (half) {
        switch (K) {
            PVRAFT_LOOKUP_CASE_H(4)
            PVRAFT_LOOKUP_CASE_H(8)
            PVRAFT_LOOKUP_CASE_H(16)
            PVRAFT_LOOKUP_CASE_H(32)
            default:
                return fail(PVRAFT_ERR_UNSUPPORTED, "corr_lookup (bf16 state): truncate_k=%d (supported: 128,256,512,1024)", K);
        }
    }
    switch (K) {
        PVRAFT_LOOKUP_CASE(1)
        PVRAFT_LOOKUP_CASE(2)
        PVRAFT_LOOKUP_CASE(4)
        PVRAFT_LOOKUP_CASE(8)
        PVRAFT_LOOKUP_CASE(16)
        PVRAFT_LOOKUP_CASE(32)
        default:
            return fail(PVRAFT_ERR_UNSUPPORTED, "corr_lookup: truncate_k=%d (supported: 32,64,128,256,512,1024)", K);
    }
#undef PVRAFT_LOOKUP_CASE
#undef PVRAFT_LOOKUP_CASE_H
}

extern "C" int pvraft_corr_lookup_fwd(const float* corr_val, const int32_t* corr_idx, const float* xyz2_pad,
                                      const float* coords, int B, int N, int K, int levels, float base_scale,
                                      float* vox, int vox_ld, float* knn_sel, int32_t* knn_slot, double* moments,
                                      int8_t* dbg_cube, void* stream) {
    return corr_lookup_any(corr_val, corr_idx, false, xyz2_pad, coords, B, N, K, levels, base_scale, vox, vox_ld, knn_sel, knn_slot, moments,
                           dbg_cube, stream);
}

extern "C" int pvraft_corr_lookup_bf16_fwd(const uint16_t* corr_val_bf16, const uint16_t* corr_idx_u16, const float* xyz2_pad,
                                           const float* coords, int B, int N, int K, int levels, float base_scale,
                                           float* vox, int vox_ld, float* knn_sel, int32_t* knn_slot, double* moments,
                                           int8_t* dbg_cube, void* stream) {
    return corr_lookup_any(corr_val_bf16, corr_idx_u16, true, xyz2_pad, coords, B, N, K, levels, base_scale, vox, vox_ld, knn_sel, knn_slot,
                           moments, dbg_cube, stream);
}

// fp32 correlation values -> bf16 (round to nearest even), int32 candidate ids -> uint16: the 4-byte-per-candidate state
__global__ void k_state_pack_bf16(const float* __restrict__ val, const int32_t* __restrict__ idx, long long n, uint16_t* __restrict__ val_out,
                                  uint16_t* __restrict__ idx_out) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const unsigned u = __float_as_uint(__ldg(val + i));
    const unsigned r = u + 0x7FFFu + ((u >> 16) & 1u);            // round to nearest even on the dropped 16 bits
    // inf passes through; a NaN becomes a quiet NaN with its sign kept (truncating a NaN whose payload sits in the low 16 bits
    // would give inf)
    const unsigned special = (u & 0x007FFFFFu) ? ((u >> 16) | 0x0040u) : (u >> 16);
    val_out[i] = (u & 0x7F800000u) == 0x7F800000u ? (uint16_t)special : (uint16_t)(r >> 16);
    idx_out[i] = (uint16_t)__ldg(idx + i);
}

extern "C" int pvraft_corr_state_pack_bf16(const float* val, const int32_t* idx, int64_t n, uint16_t* val_out, uint16_t* idx_out, void* stream) {
    if (!val || !idx || !val_out || !idx_out || n <= 0) return fail(PVRAFT_ERR_BAD_ARG, "corr_state_pack_bf16: bad argument");
    k_state_pack_bf16<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(val, idx, n, val_out, idx_out);
    return check_launch("corr_state_pack_bf16");
}
