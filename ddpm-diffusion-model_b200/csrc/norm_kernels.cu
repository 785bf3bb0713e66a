// GroupNorm (+SiLU, +dropout) forward/backward, nearest-x2 up-sampling and its adjoint, channel-slice
// add and per-channel pixel reductions -- the HBM-bound glue between the implicit-GEMM convolutions.
// Replaces attention.py:38-39 / unet_backbone.py:20-21,29-31,63,98-99 (native_group_norm, silu,
// dropout, upsample_nearest2d; SURVEY.md §2.2 rows 4,5,6,9).
//
// Layout: NHWC with pitch (channel slices of concat buffers) and an optional zero halo that these
// kernels never write.  Thread mapping for every kernel here: a thread owns one 16-byte channel
// vector position `cv` and walks pixels, so global accesses are 16 B per lane and contiguous along C.
//
// HBM roofline (bf16 activations): gn_stats 2 B/elem, gn_apply 4 B/elem, gn_bwd 2x(4)+2 = 10 B/elem.
#include "common.cuh"

#include <cooperative_groups.h>
#include <unordered_map>
namespace cg = cooperative_groups;

#define NT 256
#ifndef GN_FWD_OCC
#define GN_FWD_OCC 4              // 64 registers, no spills: 83 vs 91 us at 96@64 (B=128) against 3 CTAs/SM
#endif
#ifndef GN_BWD_OCC
#define GN_BWD_OCC 3              // 80 registers: with the PixWalk state the 64-register build spilled (96@64: 186 vs 134 us)
#endif

struct PixMap {
    int cvs;    // channel vectors per pixel
    int ppi;    // pixels processed per block iteration
    int cv;     // this thread's channel vector
    int prow;   // this thread's pixel lane
    bool active;
};
template <int VEC> __device__ __forceinline__ PixMap make_map(int C) {
    PixMap m;
    m.cvs = C / VEC;
    m.ppi = NT / m.cvs; if (m.ppi < 1) m.ppi = 1;
    m.cv = threadIdx.x % m.cvs;
    m.prow = threadIdx.x / m.cvs;
    m.active = m.prow < m.ppi;
    return m;
}

template <typename T, int VEC> __device__ __forceinline__ void ldv(const T* p, float* v) {
    if (VEC == 1) v[0] = ldf<T>(p);
    else { Vec16<T> t; t.load(p);
#pragma unroll
        for (int i = 0; i < VEC; ++i) v[i] = t.v[i]; }
}
template <typename T, int VEC> __device__ __forceinline__ void stv(T* p, const float* v) {
    if (VEC == 1) stf<T>(p, v[0]);
    else { Vec16<T> t;
#pragma unroll
        for (int i = 0; i < VEC; ++i) t.v[i] = v[i];
        t.store(p); }
}
// raw 16-byte (or scalar) packet: loads are issued back to back and converted later, so a thread keeps
// U independent requests in flight at 4 registers each
template <typename T, int VEC> struct Raw { uint4 q; };
template <typename T> struct Raw<T, 1> { T q; };
template <typename T, int VEC> __device__ __forceinline__ void ldraw(const T* p, Raw<T, VEC>& r) {
    if constexpr (VEC == 1) r.q = *p; else r.q = *reinterpret_cast<const uint4*>(p);
}
template <typename T, int VEC> __device__ __forceinline__ void unraw(const Raw<T, VEC>& r, float* v) {
    if constexpr (VEC == 1) { v[0] = ldf<T>(&r.q); }
    else if constexpr (sizeof(T) == 4) {
        v[0] = __uint_as_float(r.q.x); v[1] = __uint_as_float(r.q.y); v[2] = __uint_as_float(r.q.z); v[3] = __uint_as_float(r.q.w);
    } else {
        // bf16: low half shift, high half mask -- one integer instruction per element (__bfloat1622float2 costs 1.5: PRMT + shift)
        const uint32_t w[4] = {r.q.x, r.q.y, r.q.z, r.q.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) Fmt16<T>::unpack(w[i], v[2 * i], v[2 * i + 1]);
    }
}

static inline bool vec_ok(const ddpm_tensor* t, int vec, int esz) {
    return (t->C % vec) == 0 && (t->pitch % vec) == 0 && ((((uintptr_t)t->ptr) % (vec * esz)) == 0);
}
static inline int blocks_per_image(int N, int HW, int ppi) {
    int want = (148 * 16 + N - 1) / N;
    int maxb = (HW + ppi - 1) / ppi;
    if (want < 1) want = 1;
    return want < maxb ? want : maxb;
}

// ---- per-thread cp.async pipeline ---------------------------------------------------------------------------
// ncu on the register-staged version: 48-60 % issue utilisation with `long_scoreboard` as the top stall and ~30 %
// achieved occupancy -- each warp alternated "U loads, wait a DRAM round trip, ~150 instructions per packet", so
// the bytes in flight per SM were far below what HBM latency x bandwidth needs.  Here every thread streams the
// 16-byte packets it will consume GN_PIPE_D-1 iterations later into its OWN shared-memory slots (LDGSTS, L2 only):
// no registers are held by loads in flight, no barriers (a thread only reads what it copied itself; completion
// through cp.async.wait_group), and 1024 threads x 3 iterations x 16-48 B stay in flight per SM.
#ifndef GN_PIPE_D
#define GN_PIPE_D 4               // backward (2-3 tensors per iteration); power of two
#endif
#ifndef GN_PIPE_D_FWD
#define GN_PIPE_D_FWD 8           // forward streams ONE tensor: 3 x 16 B per thread was only ~48 KB in flight per SM, at the
#endif                            // latency x bandwidth threshold (43 KB) -- the statistics pass ran at 3.4 TB/s
__device__ __forceinline__ uint32_t sm_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ uint4 lds128(uint32_t a) {
    uint4 v;
    asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a) : "memory");
    return v;
}
template <int VEC, int NTEN, int D = GN_PIPE_D> constexpr int gn_ring_bytes() {
    // the ring doubles as the [2*VEC][NT] float scratch of cta_channel_reduce (used only between streaming loops)
    return VEC == 1 ? 2 * NT * 4 : (D * NTEN * NT * 16 > 2 * VEC * NT * 4 ? D * NTEN * NT * 16 : 2 * VEC * NT * 4);
}
// Pixel p = first + j*step of an image of width W, tracked as (p, y = p / W) with adds only: the per-packet address
// arithmetic of these kernels (a division or shift/mask pair plus 64-bit multiplies per tensor and per packet, twice --
// once for the prefetch, once for the consumer) was ~50 of the ~80-240 instructions a packet costs (SASS count, round 2),
// and the kernels are issue-bound.
struct PixWalk {
    int p, y, x, W, sy, sx, step;
    __device__ __forceinline__ PixWalk(int first, int step_, int W_, int wshift) : p(first), W(W_), step(step_) {
        if (wshift >= 0) { y = first >> wshift; x = first & (W_ - 1); sy = step_ >> wshift; sx = step_ & (W_ - 1); }
        else { y = first / W_; x = first - y * W_; sy = step_ / W_; sx = step_ - sy * W_; }
    }
    __device__ __forceinline__ void next() {
        p += step; x += sx; y += sy;
        if (x >= W) { x -= W; ++y; }
    }
};
// Calls body(p, y, r) for p = first, first+step, ... < end with r[t] = the 16-byte packet of tensor t (t < nten <= NTEN)
// at pixel p (image row y), addr(t, p, y) giving its global address.  VEC == 1 (unaligned fallbacks) loads directly.
template <typename T, int VEC, int NTEN, int D = GN_PIPE_D, typename AddrF, typename BodyF>
__device__ __forceinline__ void stream_packets(unsigned char* ring, int nten, int first, int end, int step, int W, int wshift,
                                               AddrF addr, BodyF body) {
    PixWalk wc(first, step, W, wshift);                           // consumer position
    if constexpr (VEC == 1) {
        for (; wc.p < end; wc.next()) {
            Raw<T, VEC> r[NTEN];
#pragma unroll
            for (int t = 0; t < NTEN; ++t) if (t < nten) ldraw<T, VEC>(addr(t, wc.p, wc.y), r[t]);
            body(wc.p, wc.y, r);
        }
    } else {
        const uint32_t base = sm_u32(ring) + threadIdx.x * 16u;
        PixWalk wp(first, step, W, wshift);                       // prefetch position (D-1 iterations ahead)
#pragma unroll
        for (int d = 0; d < D - 1; ++d) {
            if (wp.p < end) {
#pragma unroll
                for (int t = 0; t < NTEN; ++t) if (t < nten) cp_async16(base + (uint32_t)((d * NTEN + t) * NT * 16), addr(t, wp.p, wp.y));
            }
            cp_async_commit(); wp.next();
        }
        int st = 0;
        for (; wc.p < end; wc.next()) {
            const int sf = (st + D - 1) & (D - 1);               // the slot the previous iteration consumed
            if (wp.p < end) {
#pragma unroll
                for (int t = 0; t < NTEN; ++t) if (t < nten) cp_async16(base + (uint32_t)((sf * NTEN + t) * NT * 16), addr(t, wp.p, wp.y));
            }
            cp_async_commit(); wp.next();
            cp_async_wait<D - 1>();                              // this iteration's group has landed
            Raw<T, VEC> r[NTEN];
#pragma unroll
            for (int t = 0; t < NTEN; ++t) if (t < nten) r[t].q = lds128(base + (uint32_t)((st * NTEN + t) * NT * 16));
            body(wc.p, wc.y, r);
            st = (st + 1) & (D - 1);
        }
        cp_async_wait<0>();
    }
}

__device__ __forceinline__ void cluster_arrive() { asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory"); }
__device__ __forceinline__ void cluster_wait() { asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory"); }

// ================================================================================================
// GroupNorm, one thread-block CLUSTER per image.
//
// The reference's chain cast -> native_group_norm(fp32) -> SiLU -> dropout -> cast moves 20-37 B per
// element (SURVEY.md §8a a10).  Here an image is owned by a cluster of CS CTAs:
//   phase 1  every CTA streams its share of the image's pixels from HBM and reduces per-channel
//            moments (registers -> shared memory), the CTAs exchange per-group (forward) or
//            per-channel (backward) partials through distributed shared memory,
//   phase 2  the same CTA re-reads the same pixels -- now L2 hits, the image was touched microseconds
//            ago and at most ~50 clusters are in flight -- and writes the result.
// HBM traffic: forward 2 (read) + 2 (write) = 4 B/elem bf16, backward 4 + 2 = 6 B/elem (+2 when
// accumulating into dx), instead of 6 and 10 for separate stats / apply launches.
// Thread mapping: a thread owns one 16-byte channel vector position `cv` and walks pixels; its packets stream through a
// private cp.async ring in shared memory (below).  Halo pixels are never read or written.
// ================================================================================================
struct GnP {
    TV x, dy, o;                 // forward: x -> o;  backward: x, dy -> o (= dx)
    int G; float eps; int act; float p_drop; float keep_scale; uint32_t thr16;
    const uint64_t* rng; uint32_t layer;
    const float* gamma; const float* beta;
    double* stats;               // [N][G][2] (sum, sum of squares)
    float* dgamma; float* dbeta; // backward: accumulated with atomics (may be NULL)
    float* cs_nc; float* cs_c;   // backward: per-image / total channel sums of the final dx (conv bias and time-bias gradients)
    int accumulate;              // backward: dx += ...
    int stash;                   // backward: dy may be overwritten -> phase 1 leaves dz there, phase 2 skips mask / act'

    int wshift;                  // log2(W) when W is a power of two, else -1
};

// interior pixel index p = y*W + x  ->  padded-linear pixel index of a view (3 integer instructions when W is
// a power of two); the element offset from the image's padded origin is q * pitch
struct PixAddr {
    int ws, W, Wp, h2, q0, pitch;
    __device__ __forceinline__ PixAddr(const TV& t, int wshift)
        : ws(wshift), W(t.W), Wp(t.Wp), h2(2 * t.halo), q0(t.halo * t.Wp + t.halo), pitch(t.pitch) {}
    __device__ __forceinline__ int q(int p) const {
        if (ws >= 0) return p + h2 * (p >> ws) + q0;
        const int y = p / W;
        return y * Wp + (p - y * W) + q0;
    }
    template <typename T> __device__ __forceinline__ T* at(T* img, int p) const { return img + (int64_t)q(p) * pitch; }
    // same, with the image row y = p / W supplied by a PixWalk: q = p + 2*halo*y + q0
    template <typename T> __device__ __forceinline__ T* at(T* img, int p, int y) const { return img + (int64_t)(p + h2 * y + q0) * pitch; }
};
template <typename T> __device__ __forceinline__ T* img_origin(const TV& t, int n, int c0) {
    return reinterpret_cast<T*>(t.ptr) + (int64_t)n * t.Hp * t.Wp * t.pitch + c0;
}

__device__ __forceinline__ void split_pix(int p, int W, int wshift, int& y, int& x) {
    if (wshift >= 0) { y = p >> wshift; x = p & (W - 1); }
    else { y = p / W; x = p - y * W; }
}

// CTA-wide reduction of NV per-thread partial sums per channel-vector element:
// part[k][tid] -> chan[k / VEC][c], c = cv*VEC + (k % VEC), summed over the threads that share `cv`.
template <int VEC, int NSTAT>
__device__ __forceinline__ void cta_channel_reduce(float (*part)[NT], const float* vals, double* chan, int C, const PixMap& m) {
#pragma unroll
    for (int k = 0; k < NSTAT * VEC; ++k) part[k][threadIdx.x] = vals[k];
    __syncthreads();
    for (int o = threadIdx.x; o < NSTAT * C; o += NT) {
        const int st = o / C, c = o - st * C;
        const int cv = c / VEC, k = c - cv * VEC;
        double a = 0.0;
        for (int r = 0; r < m.ppi; ++r) a += (double)part[st * VEC + k][r * m.cvs + cv];
        chan[o] = a;
    }
    __syncthreads();
}

// MODE 0: fused stats + apply; 1: stats only; 2: apply only (stats given)
template <typename T, int VEC, int MODE>
__global__ void __launch_bounds__(NT, GN_FWD_OCC) gn_fwd_kernel(GnP a) {
    extern __shared__ __align__(16) unsigned char gsm[];
    const int C = a.x.C, G = a.G, cpg = C / G, HW = a.x.H * a.x.W;
    constexpr bool FAST_ACT = std::is_same<T, bf16>::value;  // bf16 tensors: tanh-based SiLU; fp16 keeps the exact form (common.cuh)
    constexpr int RING = gn_ring_bytes<VEC, 1, GN_PIPE_D_FWD>();
    unsigned char* ring = gsm;
    float (*part)[NT] = reinterpret_cast<float (*)[NT]>(gsm);    // aliases the ring (see gn_ring_bytes)
    double* chan = reinterpret_cast<double*>(gsm + RING);     // [2][C]
    double* gpart = chan + 2 * C;                            // [2][G]  (read by the other CTAs of the cluster)
    float* gm = reinterpret_cast<float*>(gpart + 2 * G);     // [G] mean
    float* gr = gm + G;                                      // [G] rstd
    cg::cluster_group cl = cg::this_cluster();
    const int CS = (int)cl.num_blocks(), rank = (int)cl.block_rank();
    const int n = blockIdx.x / CS;
    const PixMap m = make_map<VEC>(C);
    const int per = (HW + CS - 1) / CS;
    const int p0 = rank * per, p1 = min(HW, p0 + per);
    const int c0 = m.cv * VEC;
    const uint32_t dkey = a.thr16 ? dropout_key(a.rng, a.layer) : 0u;
    const uint32_t ebase = (uint32_t)n * (uint32_t)HW * (uint32_t)C + (uint32_t)c0;   // wrapping element index (mask hash input)
    const PixAddr ax(a.x, a.wshift), ao(a.o, a.wshift);
    const T* xb = img_origin<T>(a.x, n, c0);
    T* ob = img_origin<T>(a.o, n, c0);
    const int pend = m.active ? p1 : 0;
    auto xaddr = [&](int, int p, int y) { return ax.at(xb, p, y); };

    if (MODE != 2) {
        float acc[2 * VEC];
#pragma unroll
        for (int i = 0; i < 2 * VEC; ++i) acc[i] = 0.f;
        stream_packets<T, VEC, 1, GN_PIPE_D_FWD>(ring, 1, p0 + m.prow, pend, m.ppi, a.x.W, a.wshift, xaddr, [&](int, int, Raw<T, VEC>* r) {
            float v[VEC];
            unraw<T, VEC>(r[0], v);
#pragma unroll
            for (int i = 0; i < VEC; ++i) { acc[i] += v[i]; acc[VEC + i] = fmaf(v[i], v[i], acc[VEC + i]); }
        });
        __syncthreads();                                     // every thread is done with its ring slots (part aliases them)
        cta_channel_reduce<VEC, 2>(part, acc, chan, C, m);
        for (int o = threadIdx.x; o < 2 * G; o += NT) {
            const int st = o / G, g = o - st * G;
            double s = 0.0;
            for (int j = 0; j < cpg; ++j) s += chan[st * C + g * cpg + j];
            gpart[o] = s;
        }
        cluster_arrive(); cluster_wait();                    // every CTA's gpart is complete
        for (int g = threadIdx.x; g < G; g += NT) {
            double s = 0.0, q = 0.0;
            for (int r = 0; r < CS; ++r) {
                const double* rp = cl.map_shared_rank(gpart, r);
                s += rp[g]; q += rp[G + g];
            }
            if (rank == 0 && a.stats) { a.stats[((size_t)n * G + g) * 2] = s; a.stats[((size_t)n * G + g) * 2 + 1] = q; }
            const double cnt = (double)cpg * HW, mu = s / cnt;
            double var = q / cnt - mu * mu; if (var < 0.0) var = 0.0;
            gm[g] = (float)mu; gr[g] = (float)(1.0 / sqrt(var + (double)a.eps));
        }
        cluster_arrive();                                    // remote reads done; waited for before exit
        __syncthreads();
    } else {
        for (int g = threadIdx.x; g < G; g += NT) {
            const double s = a.stats[((size_t)n * G + g) * 2], q = a.stats[((size_t)n * G + g) * 2 + 1];
            const double cnt = (double)cpg * HW, mu = s / cnt;
            double var = q / cnt - mu * mu; if (var < 0.0) var = 0.0;
            gm[g] = (float)mu; gr[g] = (float)(1.0 / sqrt(var + (double)a.eps));
        }
        __syncthreads();
    }

    if ((MODE == 0 || MODE == 2) && m.active) {
        float sc[VEC], sh[VEC];
#pragma unroll
        for (int i = 0; i < VEC; ++i) {
            const int c = c0 + i, g = c / cpg;
            sc[i] = gr[g] * __ldg(a.gamma + c);
            sh[i] = __ldg(a.beta + c) - gm[g] * sc[i];
            if (FAST_ACT && a.act) { sc[i] *= 0.5f; sh[i] *= 0.5f; }     // the affine produces z/2 directly (silu_half)
        }
        stream_packets<T, VEC, 1, GN_PIPE_D_FWD>(ring, 1, p0 + m.prow, p1, m.ppi, a.x.W, a.wshift, xaddr, [&](int p, int y, Raw<T, VEC>* r) {
            float v[VEC];
            unraw<T, VEC>(r[0], v);
#pragma unroll
            for (int i = 0; i < VEC; ++i) {
                const float z = fmaf(v[i], sc[i], sh[i]);
                v[i] = a.act ? (FAST_ACT ? silu_half(z) : silu_f(z)) : z;
            }
            if (a.thr16) dropout_apply<VEC>(v, dkey, ebase + (uint32_t)p * (uint32_t)C, a.thr16, a.keep_scale);
            stv<T, VEC>(ao.at(ob, p, y), v);
        });
    }
    if (MODE != 2) cluster_wait();                           // do not exit while peers may still read gpart
}

// backward: z = x*sc+sh, y = drop(act(z)); dz = dy * mask/(1-p) * act'(z)
//   S1[c] = sum_p dz, S2[c] = sum_p dz*xhat;  A_g = mean_g(gamma*S1), B_g = mean_g(gamma*S2)
//   dx = rstd * (dz*gamma - A_g - xhat*B_g);  dbeta += S1, dgamma += S2
template <typename T, int VEC, bool STASH>
__global__ void __launch_bounds__(NT, STASH ? GN_BWD_OCC : 2) gn_bwd_kernel(GnP a) {
    extern __shared__ __align__(16) unsigned char gsm[];
    const int C = a.x.C, G = a.G, cpg = C / G, HW = a.x.H * a.x.W;
    constexpr bool FAST_ACT = std::is_same<T, bf16>::value;  // bf16 tensors: tanh-based SiLU; fp16 keeps the exact form (common.cuh)
    constexpr int RING = gn_ring_bytes<VEC, 3>();
    unsigned char* ring = gsm;
    float (*part)[NT] = reinterpret_cast<float (*)[NT]>(gsm);    // aliases the ring (see gn_ring_bytes)
    double* chan = reinterpret_cast<double*>(gsm + RING);    // [2][C] this CTA's per-channel partials (read by peers)
    float* tot = reinterpret_cast<float*>(chan + 2 * C);     // [2][C] cluster totals
    float* gA = tot + 2 * C;                                 // [G]
    float* gB = gA + G;                                      // [G]
    float* gm = gB + G;                                      // [G] mean
    float* gr = gm + G;                                      // [G] rstd
    cg::cluster_group cl = cg::this_cluster();
    const int CS = (int)cl.num_blocks(), rank = (int)cl.block_rank();
    const int n = blockIdx.x / CS;
    const PixMap m = make_map<VEC>(C);
    const int per = (HW + CS - 1) / CS;
    const int p0 = rank * per, p1 = min(HW, p0 + per);
    const int c0 = m.cv * VEC;
    const uint32_t dkey = a.thr16 ? dropout_key(a.rng, a.layer) : 0u;
    const uint32_t ebase = (uint32_t)n * (uint32_t)HW * (uint32_t)C + (uint32_t)c0;
    const PixAddr ax(a.x, a.wshift), ad(a.dy, a.wshift), ao(a.o, a.wshift);
    const T* xb = img_origin<T>(a.x, n, c0);
    T* db = img_origin<T>(a.dy, n, c0);
    T* ob = img_origin<T>(a.o, n, c0);
    const int pend = m.active ? p1 : 0;
    auto addr = [&](int t, int p, int y) -> const T* { return t == 0 ? ax.at(xb, p, y) : (t == 1 ? ad.at(db, p, y) : ao.at(ob, p, y)); };

    for (int g = threadIdx.x; g < G; g += NT) {
        const double s = a.stats[((size_t)n * G + g) * 2], q = a.stats[((size_t)n * G + g) * 2 + 1];
        const double cnt = (double)cpg * HW, mu = s / cnt;
        double var = q / cnt - mu * mu; if (var < 0.0) var = 0.0;
        gm[g] = (float)mu; gr[g] = (float)(1.0 / sqrt(var + (double)a.eps));
    }
    __syncthreads();

    // ---- phase 1: per-channel sums S1 = sum dz, S2 = sum dz*xhat (dz = dy * mask/(1-p) * act'(z))
    {
        // z = x*sc + sh.  The second moment is accumulated against x, not xhat (two fewer constants and one fewer
        // FMA per element); S2 = rstd * sum(dz*x) - mean*rstd * sum(dz) is formed from the double-precision totals.
        float sc[VEC], sh[VEC];
#pragma unroll
        for (int i = 0; i < VEC; ++i) {
            const int c = min(c0 + i, C - 1), g = c / cpg;
            sc[i] = gr[g] * __ldg(a.gamma + c); sh[i] = __ldg(a.beta + c) - gm[g] * sc[i];
            if (FAST_ACT) { sc[i] *= 0.5f; sh[i] *= 0.5f; }          // z/2 for dsilu_half (z itself is only needed there)
        }
        float acc[2 * VEC];
#pragma unroll
        for (int i = 0; i < 2 * VEC; ++i) acc[i] = 0.f;
        // dropout's 1/(1-p) rides on the constants of the SiLU derivative (one multiply per element less)
        const bool fold = FAST_ACT && a.act && a.thr16;
        const float hs = fold ? 0.5f * a.keep_scale : 0.5f, dscale = fold ? 1.0f : a.keep_scale;
        stream_packets<T, VEC, 2>(ring, 2, p0 + m.prow, pend, m.ppi, a.x.W, a.wshift, addr, [&](int p, int y, Raw<T, VEC>* r) {
            float v[VEC], d[VEC];
            unraw<T, VEC>(r[0], v); unraw<T, VEC>(r[1], d);
            if (a.thr16) dropout_apply<VEC>(d, dkey, ebase + (uint32_t)p * (uint32_t)C, a.thr16, dscale);
#pragma unroll
            for (int i = 0; i < VEC; ++i) {
                float dz = d[i];
                if (a.act) dz *= FAST_ACT ? dsilu_half_scaled(fmaf(v[i], sc[i], sh[i]), hs) : dsilu_f(fmaf(v[i], sc[i], sh[i]));
                acc[i] += dz; acc[VEC + i] = fmaf(dz, v[i], acc[VEC + i]);
                d[i] = dz;
            }
            if (STASH) stv<T, VEC>(ad.at(db, p, y), d);
        });
        __syncthreads();                                     // every thread is done with its ring slots (part aliases them)
        cta_channel_reduce<VEC, 2>(part, acc, chan, C, m);
    }
    cluster_arrive(); cluster_wait();                        // every CTA's chan[] is complete
    for (int c = threadIdx.x; c < C; c += NT) {
        double s1 = 0.0, sx = 0.0;
        for (int r = 0; r < CS; ++r) { const double* rp = cl.map_shared_rank(chan, r); s1 += rp[c]; sx += rp[C + c]; }
        const int g = c / cpg;
        const double s2 = (double)gr[g] * (sx - (double)gm[g] * s1);       // sum dz*xhat
        tot[c] = (float)s1; tot[C + c] = (float)s2;
        if (rank == 0) {
            if (a.dbeta) atomicAdd(a.dbeta + c, (float)s1);
            if (a.dgamma) atomicAdd(a.dgamma + c, (float)s2);
        }
    }
    cluster_arrive();                                        // remote reads done; waited for before exit
    __syncthreads();
    for (int g = threadIdx.x; g < G; g += NT) {
        float sa = 0.f, sb = 0.f;
        for (int j = 0; j < cpg; ++j) {
            const int c = g * cpg + j;
            const float gmm = __ldg(a.gamma + c);
            sa = fmaf(gmm, tot[c], sa); sb = fmaf(gmm, tot[C + c], sb);
        }
        const float inv = 1.0f / ((float)cpg * (float)HW);
        gA[g] = sa * inv; gB[g] = sb * inv;
    }
    __syncthreads();

    // ---- phase 2: dx = rs*(dz*ga - A_g - xhat*B_g) = k0*dz - k1*x + k2   (x and dy/dz are L2 hits now)
    float csum[VEC];
#pragma unroll
    for (int i = 0; i < VEC; ++i) csum[i] = 0.f;
    if (m.active) {
        float k0[VEC], k1[VEC], k2[VEC], rs[VEC], mr[VEC], ga[VEC], be[VEC];
#pragma unroll
        for (int i = 0; i < VEC; ++i) {
            const int c = min(c0 + i, C - 1), g = c / cpg;
            const float r_ = gr[g], m_ = gm[g] * gr[g], g_ = __ldg(a.gamma + c);
            k0[i] = r_ * g_; k1[i] = r_ * r_ * gB[g]; k2[i] = m_ * r_ * gB[g] - r_ * gA[g];
            rs[i] = r_; mr[i] = m_; ga[i] = g_; be[i] = __ldg(a.beta + c);      // only used when !STASH
        }
        stream_packets<T, VEC, 3>(ring, a.accumulate ? 3 : 2, p0 + m.prow, p1, m.ppi, a.x.W, a.wshift, addr, [&](int p, int y, Raw<T, VEC>* rw) {
            float v[VEC], d[VEC], r[VEC];
            unraw<T, VEC>(rw[0], v); unraw<T, VEC>(rw[1], d);
            if (a.accumulate) unraw<T, VEC>(rw[2], r);
            if (!STASH) {                                          // recompute dz (phase 1 could not leave it in dy)
                if (a.thr16) dropout_apply<VEC>(d, dkey, ebase + (uint32_t)p * (uint32_t)C, a.thr16, a.keep_scale);
                if (a.act) {
#pragma unroll
                    for (int i = 0; i < VEC; ++i) {
                        const float z = fmaf(fmaf(v[i], rs[i], -mr[i]), ga[i], be[i]);
                        d[i] *= FAST_ACT ? dsilu_half(0.5f * z) : dsilu_f(z);
                    }
                }
            }
#pragma unroll
            for (int i = 0; i < VEC; ++i) {
                const float g = fmaf(-v[i], k1[i], fmaf(d[i], k0[i], k2[i]));
                r[i] = a.accumulate ? r[i] + g : g;
                csum[i] += r[i];
            }
            stv<T, VEC>(ao.at(ob, p, y), r);
        });
    }
    cluster_wait();                                          // peers are done with chan[] -> it can be reused
    if (a.cs_nc || a.cs_c) {
        // fused column sums of dx: the bias gradient of the convolution that produced x and the
        // per-image time-bias gradient (replaces a separate pass over dx, ddpm_colsum)
        __syncthreads();                                     // ring slots are dead before part[] is written
        cta_channel_reduce<VEC, 1>(part, csum, chan, C, m);
        for (int c = threadIdx.x; c < C; c += NT) {
            const float v = (float)chan[c];
            if (a.cs_nc) atomicAdd(a.cs_nc + (size_t)n * C + c, v);
            if (a.cs_c) atomicAdd(a.cs_c + c, v);
        }
    }
}

// cluster size: enough CTAs per image that a thread sees ~16 packets per phase, at most 8 (portable limit)
static int gn_cluster_size(int HW, int cvs, int N = 1 << 30) {
    const int64_t packets = (int64_t)HW * cvs;
    int cs = 1;
    // Round 2 measured smaller clusters for the mid-size shapes (>= 48 packets per thread instead of >= 12): alone, 192@32
    // backward 82.8 -> 70.7 us, forward 47.3 -> 40.4, 384@16 backward 46.6 -> 40.1 (profiles/r2_gn_cluster_granularity.txt)
    // -- but in the train step and in DDIM-100 the same-box A/B showed no change (11.96 vs 12.04 ms; 6.69 vs 6.63 ms per
    // evaluation, inside the noise), so the rule stays as it was.
    while (cs < 8 && packets / (cs * NT) >= 24) cs <<= 1;
    // Very few large images (fewer CTAs than SMs with clusters of 8): clusters of 16 (non-portable size) double the number of
    // CTAs per image -- 256-px sampling at B = 16: 12.3 -> 11.5 ms per evaluation; at B = 32 (256 CTAs already) it measured
    // 1.4 % SLOWER, hence the N * 8 <= 148 bound.
    if (cs == 8 && (int64_t)N * 8 <= 148 && packets / (16 * NT) >= 24) cs = 16;
    return cs;
}
static int log2_exact(int v) { int s = 0; while ((1 << s) < v) ++s; return (1 << s) == v ? s : -1; }

template <typename K>
static int launch_cluster(K kernel, int grid, int cs, size_t smem, cudaStream_t st, GnP& p) {
    if (smem > 48 * 1024) {                                  // once per kernel instantiation (all share the type K)
        static std::unordered_map<const void*, size_t> configured;
        size_t& have = configured[(const void*)kernel];
        if (smem > have) {
            cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) return (int)e;
            have = smem;
        }
    }
    if (cs > 8) {
        static std::unordered_map<const void*, int> np;
        int& have = np[(const void*)kernel];
        if (!have) {
            cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
            if (e != cudaSuccess) return (int)e;
            have = 1;
        }
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(grid); cfg.blockDim = dim3(NT); cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = cs; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    cudaError_t e = cudaLaunchKernelEx(&cfg, kernel, p);
    if (e != cudaSuccess) return (int)e;
    LAUNCH_OK();
    return 0;
}

static int gn_fill(GnP& p, const ddpm_tensor* x, int groups, const double* stats, const float* gamma, const float* beta,
                   float eps, int act, float p_drop, const uint64_t* rng, uint32_t layer) {
    if (p_drop > 0.f && !rng) return DDPM_E_ARG;
    if (p_drop < 0.f || p_drop >= 1.f) return DDPM_E_ARG;
    p.x = TV(*x); p.G = groups; p.eps = eps; p.act = act; p.p_drop = p_drop;
    p.thr16 = p_drop > 0.f ? (uint32_t)(p_drop * 65536.0f + 0.5f) : 0u;
    p.keep_scale = p_drop > 0.f ? 1.0f / (1.0f - p_drop) : 1.0f;
    p.rng = rng; p.layer = layer; p.gamma = gamma; p.beta = beta; p.stats = const_cast<double*>(stats);
    p.dgamma = p.dbeta = nullptr; p.cs_nc = p.cs_c = nullptr; p.accumulate = 0; p.stash = 0; p.wshift = log2_exact(x->W);
    return 0;
}

template <int MODE>
static int gn_fwd_dispatch(GnP& p, const ddpm_tensor* x, const ddpm_tensor* out, int dtype, cudaStream_t st) {
    const int HW = x->H * x->W, C = x->C, G = p.G;
    const size_t sm0 = sizeof(double) * (2 * C + 2 * G) + sizeof(float) * 2 * G;
#define GO(T, VEC) { int cvs = C / VEC; if (cvs > NT) return DDPM_E_ARG; \
        int cs = MODE == 2 ? 1 : gn_cluster_size(HW, cvs, x->N); \
        if (MODE == 2) { cs = 1; int want = (HW * cvs) / (NT * 16); while (cs < 8 && cs < want) cs <<= 1; } \
        return launch_cluster(gn_fwd_kernel<T, VEC, MODE>, x->N * cs, cs, sm0 + gn_ring_bytes<VEC, 1, GN_PIPE_D_FWD>(), st, p); }
    const bool v8 = vec_ok(x, 8, 2) && (MODE == 1 || vec_ok(out, 8, 2));
    const bool v4 = vec_ok(x, 4, 4) && (MODE == 1 || vec_ok(out, 4, 4));
    if (dtype == DDPM_BF16) { if (v8) GO(bf16, 8) else GO(bf16, 1) }
    else if (dtype == DDPM_F16) { if (v8) GO(f16, 8) else GO(f16, 1) }
    else if (dtype == DDPM_F32) { if (v4) GO(float, 4) else GO(float, 1) }
#undef GO
    return DDPM_E_ARG;
}

extern "C" int ddpm_gn_stats(const ddpm_tensor* x, int dtype, int groups, double* stats, void* stream) {
    if (!tensor_ok(x) || !stats || groups <= 0 || x->C % groups) return DDPM_E_ARG;
    GnP p; int rc = gn_fill(p, x, groups, stats, nullptr, nullptr, 0.f, 0, 0.f, nullptr, 0); if (rc) return rc;
    p.o = p.x; p.dy = p.x;
    return gn_fwd_dispatch<1>(p, x, x, dtype, (cudaStream_t)stream);
}

extern "C" int ddpm_gn_apply(const ddpm_tensor* x, int dtype, int groups, const double* stats, const float* gamma,
                             const float* beta, float eps, int act, float p_drop, const uint64_t* rng,
                             uint32_t layer_id, const ddpm_tensor* out, void* stream) {
    if (!tensor_ok(x) || !tensor_ok(out) || !stats || !gamma || !beta || groups <= 0 || x->C % groups) return DDPM_E_ARG;
    if (out->N != x->N || out->H != x->H || out->W != x->W || out->C != x->C) return DDPM_E_ARG;
    GnP p; int rc = gn_fill(p, x, groups, stats, gamma, beta, eps, act, p_drop, rng, layer_id); if (rc) return rc;
    p.o = TV(*out); p.dy = p.x;
    return gn_fwd_dispatch<2>(p, x, out, dtype, (cudaStream_t)stream);
}

extern "C" int ddpm_gn_fwd(const ddpm_tensor* x, int dtype, int groups, double* stats, const float* gamma,
                           const float* beta, float eps, int act, float p_drop, const uint64_t* rng,
                           uint32_t layer_id, const ddpm_tensor* out, void* stream) {
    if (!tensor_ok(x) || !tensor_ok(out) || !stats || !gamma || !beta || groups <= 0 || x->C % groups) return DDPM_E_ARG;
    if (out->N != x->N || out->H != x->H || out->W != x->W || out->C != x->C) return DDPM_E_ARG;
    GnP p; int rc = gn_fill(p, x, groups, stats, gamma, beta, eps, act, p_drop, rng, layer_id); if (rc) return rc;
    p.o = TV(*out); p.dy = p.x;
    return gn_fwd_dispatch<0>(p, x, out, dtype, (cudaStream_t)stream);
}

static int gn_bwd_impl(const ddpm_tensor* x, int dtype, int groups, const double* stats, const float* gamma,
                       const float* beta, float eps, int act, float p_drop, const uint64_t* rng,
                       uint32_t layer_id, const ddpm_tensor* dy, const ddpm_tensor* dx, int accumulate,
                       float* dgamma, float* dbeta, float* cs_nc, float* cs_c, int dy_scratch, void* stream) {
    if (!tensor_ok(x) || !tensor_ok(dy) || !tensor_ok(dx) || !stats || !gamma || !beta) return DDPM_E_ARG;
    if (groups <= 0 || x->C % groups || dy->C != x->C || dx->C != x->C) return DDPM_E_ARG;
    if (dy->N != x->N || dy->H != x->H || dy->W != x->W || dx->N != x->N || dx->H != x->H || dx->W != x->W) return DDPM_E_ARG;
    GnP p; int rc = gn_fill(p, x, groups, stats, gamma, beta, eps, act, p_drop, rng, layer_id); if (rc) return rc;
    p.dy = TV(*dy); p.o = TV(*dx); p.accumulate = accumulate; p.dgamma = dgamma; p.dbeta = dbeta;
    p.cs_nc = cs_nc; p.cs_c = cs_c; p.stash = dy_scratch ? 1 : 0;
    cudaStream_t st = (cudaStream_t)stream;
    const int HW = x->H * x->W, C = x->C;
    const size_t sm0 = sizeof(double) * 2 * C + sizeof(float) * (2 * C + 4 * groups);
    // colsum_nc is zeroed only once the shape is accepted: a rejected call writes nothing
#define GO(T, VEC) { int cvs = C / VEC; if (cvs > NT) return DDPM_E_ARG; int cs = gn_cluster_size(HW, cvs, x->N); \
        const size_t sm = sm0 + gn_ring_bytes<VEC, 3>(); \
        if (cs_nc) CUDA_TRY(cudaMemsetAsync(cs_nc, 0, sizeof(float) * x->N * x->C, st)); \
        if (p.stash) return launch_cluster(gn_bwd_kernel<T, VEC, true>, x->N * cs, cs, sm, st, p); \
        return launch_cluster(gn_bwd_kernel<T, VEC, false>, x->N * cs, cs, sm, st, p); }
    if (dtype == DDPM_BF16) { if (vec_ok(x, 8, 2) && vec_ok(dy, 8, 2) && vec_ok(dx, 8, 2)) GO(bf16, 8) else GO(bf16, 1) }
    else if (dtype == DDPM_F16) { if (vec_ok(x, 8, 2) && vec_ok(dy, 8, 2) && vec_ok(dx, 8, 2)) GO(f16, 8) else GO(f16, 1) }
    else if (dtype == DDPM_F32) { if (vec_ok(x, 4, 4) && vec_ok(dy, 4, 4) && vec_ok(dx, 4, 4)) GO(float, 4) else GO(float, 1) }
#undef GO
    return DDPM_E_ARG;
}

extern "C" int ddpm_gn_bwd(const ddpm_tensor* x, int dtype, int groups, const double* stats, const float* gamma,
                           const float* beta, float eps, int act, float p_drop, const uint64_t* rng,
                           uint32_t layer_id, const ddpm_tensor* dy, const ddpm_tensor* dx, int accumulate,
                           float* dgamma, float* dbeta, float* ws, void* stream) {
    (void)ws;                                  // kept in the signature for ABI stability; no longer needed
    return gn_bwd_impl(x, dtype, groups, stats, gamma, beta, eps, act, p_drop, rng, layer_id, dy, dx, accumulate,
                       dgamma, dbeta, nullptr, nullptr, 0, stream);
}

extern "C" int ddpm_gn_bwd_colsum(const ddpm_tensor* x, int dtype, int groups, const double* stats, const float* gamma,
                                  const float* beta, float eps, int act, float p_drop, const uint64_t* rng,
                                  uint32_t layer_id, const ddpm_tensor* dy, const ddpm_tensor* dx, int accumulate,
                                  float* dgamma, float* dbeta, float* colsum_nc, float* colsum_c, int dy_scratch, void* stream) {
    return gn_bwd_impl(x, dtype, groups, stats, gamma, beta, eps, act, p_drop, rng, layer_id, dy, dx, accumulate,
                       dgamma, dbeta, colsum_nc, colsum_c, dy_scratch, stream);
}

// ------------------------------------------------------------------------------------ pixel maps
// generic walker over (n, y, x, cv) of the OUTPUT view
template <typename T, int VEC, typename F>
__global__ void __launch_bounds__(NT) pix_kernel(int N, int H, int W, int C, F f) {
    const int cvs = C / VEC;
    const int64_t total = (int64_t)N * H * W * cvs;
    for (int64_t i = (int64_t)blockIdx.x * NT + threadIdx.x; i < total; i += (int64_t)gridDim.x * NT) {
        int cv = (int)(i % cvs); int64_t r = i / cvs;
        int x = (int)(r % W); r /= W;
        int y = (int)(r % H); int n = (int)(r / H);
        f(n, y, x, cv * VEC);
    }
}
static inline int pix_grid(int64_t total) {
    int64_t g = (total + NT - 1) / NT;
    return (int)(g < 148 * 8 ? (g < 1 ? 1 : g) : 148 * 8);
}

template <typename T, int VEC> struct UpFwd {
    TV in, out;
    __device__ void operator()(int n, int y, int x, int c) const {
        float v[VEC];
        ldv<T, VEC>(in.at<T>(n, y >> 1, x >> 1, c), v);
        stv<T, VEC>(out.at<T>(n, y, x, c), v);
    }
};
extern "C" int ddpm_upsample2x(const ddpm_tensor* x, const ddpm_tensor* out, int dtype, void* stream) {
    if (!tensor_ok(x) || !tensor_ok(out) || out->H != 2 * x->H || out->W != 2 * x->W || out->C != x->C || out->N != x->N) return DDPM_E_ARG;
    cudaStream_t st = (cudaStream_t)stream;
#define GO(T, VEC) { UpFwd<T, VEC> f{TV(*x), TV(*out)}; int64_t tot = (int64_t)out->N * out->H * out->W * (out->C / VEC); \
        if (launch_kernel(pix_kernel<T, VEC, decltype(f)>, dim3(pix_grid(tot)), dim3(NT), 0, st, out->N, out->H, out->W, out->C, f) != cudaSuccess) return (int)cudaGetLastError(); }
    if (dtype == DDPM_BF16) { if (vec_ok(x, 8, 2) && vec_ok(out, 8, 2)) GO(bf16, 8) else GO(bf16, 1) }
    else if (dtype == DDPM_F16) { if (vec_ok(x, 8, 2) && vec_ok(out, 8, 2)) GO(f16, 8) else GO(f16, 1) }
    else if (dtype == DDPM_F32) { if (vec_ok(x, 4, 4) && vec_ok(out, 4, 4)) GO(float, 4) else GO(float, 1) }
    else return DDPM_E_ARG;
#undef GO
    LAUNCH_OK();
    return 0;
}

template <typename T, int VEC> struct UpBwd {
    TV dy, dx; int acc;
    __device__ void operator()(int n, int y, int x, int c) const {
        float s[VEC], v[VEC];
#pragma unroll
        for (int i = 0; i < VEC; ++i) s[i] = 0.f;
        if (acc) ldv<T, VEC>(dx.at<T>(n, y, x, c), s);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            ldv<T, VEC>(dy.at<T>(n, 2 * y + (j >> 1), 2 * x + (j & 1), c), v);
#pragma unroll
            for (int i = 0; i < VEC; ++i) s[i] += v[i];
        }
        stv<T, VEC>(dx.at<T>(n, y, x, c), s);
    }
};
extern "C" int ddpm_upsample2x_bwd(const ddpm_tensor* dy, const ddpm_tensor* dx, int dtype, int accumulate, void* stream) {
    if (!tensor_ok(dy) || !tensor_ok(dx) || dy->H != 2 * dx->H || dy->W != 2 * dx->W || dy->C != dx->C || dy->N != dx->N) return DDPM_E_ARG;
    cudaStream_t st = (cudaStream_t)stream;
#define GO(T, VEC) { UpBwd<T, VEC> f{TV(*dy), TV(*dx), accumulate}; int64_t tot = (int64_t)dx->N * dx->H * dx->W * (dx->C / VEC); \
        if (launch_kernel(pix_kernel<T, VEC, decltype(f)>, dim3(pix_grid(tot)), dim3(NT), 0, st, dx->N, dx->H, dx->W, dx->C, f) != cudaSuccess) return (int)cudaGetLastError(); }
    if (dtype == DDPM_BF16) { if (vec_ok(dy, 8, 2) && vec_ok(dx, 8, 2)) GO(bf16, 8) else GO(bf16, 1) }
    else if (dtype == DDPM_F16) { if (vec_ok(dy, 8, 2) && vec_ok(dx, 8, 2)) GO(f16, 8) else GO(f16, 1) }
    else if (dtype == DDPM_F32) { if (vec_ok(dy, 4, 4) && vec_ok(dx, 4, 4)) GO(float, 4) else GO(float, 1) }
    else return DDPM_E_ARG;
#undef GO
    LAUNCH_OK();
    return 0;
}

template <typename T, int VEC> struct ZeroUp {
    TV in, out;
    __device__ void operator()(int n, int y, int x, int c) const {
        float v[VEC];
        if (((y | x) & 1) == 0) ldv<T, VEC>(in.at<T>(n, y >> 1, x >> 1, c), v);
        else {
#pragma unroll
            for (int i = 0; i < VEC; ++i) v[i] = 0.f;
        }
        stv<T, VEC>(out.at<T>(n, y, x, c), v);
    }
};
extern "C" int ddpm_zero_upsample2x(const ddpm_tensor* x, const ddpm_tensor* out, int dtype, void* stream) {
    if (!tensor_ok(x) || !tensor_ok(out) || out->H != 2 * x->H || out->W != 2 * x->W || out->C != x->C || out->N != x->N) return DDPM_E_ARG;
    cudaStream_t st = (cudaStream_t)stream;
#define GO(T, VEC) { ZeroUp<T, VEC> f{TV(*x), TV(*out)}; int64_t tot = (int64_t)out->N * out->H * out->W * (out->C / VEC); \
        if (launch_kernel(pix_kernel<T, VEC, decltype(f)>, dim3(pix_grid(tot)), dim3(NT), 0, st, out->N, out->H, out->W, out->C, f) != cudaSuccess) return (int)cudaGetLastError(); }
    if (dtype == DDPM_BF16) { if (vec_ok(x, 8, 2) && vec_ok(out, 8, 2)) GO(bf16, 8) else GO(bf16, 1) }
    else if (dtype == DDPM_F16) { if (vec_ok(x, 8, 2) && vec_ok(out, 8, 2)) GO(f16, 8) else GO(f16, 1) }
    else if (dtype == DDPM_F32) { if (vec_ok(x, 4, 4) && vec_ok(out, 4, 4)) GO(float, 4) else GO(float, 1) }
    else return DDPM_E_ARG;
#undef GO
    LAUNCH_OK();
    return 0;
}

template <typename T, int VEC> struct AddOp {
    TV a, b, o;
    __device__ void operator()(int n, int y, int x, int c) const {
        float u[VEC], v[VEC];
        ldv<T, VEC>(a.at<T>(n, y, x, c), u);
        ldv<T, VEC>(b.at<T>(n, y, x, c), v);
#pragma unroll
        for (int i = 0; i < VEC; ++i) u[i] += v[i];
        stv<T, VEC>(o.at<T>(n, y, x, c), u);
    }
};
extern "C" int ddpm_add(const ddpm_tensor* a, const ddpm_tensor* b, const ddpm_tensor* out, int dtype, void* stream) {
    if (!tensor_ok(a) || !tensor_ok(b) || !tensor_ok(out)) return DDPM_E_ARG;
    if (a->N != out->N || a->H != out->H || a->W != out->W || a->C != out->C) return DDPM_E_ARG;
    if (b->N != out->N || b->H != out->H || b->W != out->W || b->C != out->C) return DDPM_E_ARG;
    cudaStream_t st = (cudaStream_t)stream;
#define GO(T, VEC) { AddOp<T, VEC> f{TV(*a), TV(*b), TV(*out)}; int64_t tot = (int64_t)out->N * out->H * out->W * (out->C / VEC); \
        if (launch_kernel(pix_kernel<T, VEC, decltype(f)>, dim3(pix_grid(tot)), dim3(NT), 0, st, out->N, out->H, out->W, out->C, f) != cudaSuccess) return (int)cudaGetLastError(); }
    if (dtype == DDPM_BF16) { if (vec_ok(a, 8, 2) && vec_ok(b, 8, 2) && vec_ok(out, 8, 2)) GO(bf16, 8) else GO(bf16, 1) }
    else if (dtype == DDPM_F16) { if (vec_ok(a, 8, 2) && vec_ok(b, 8, 2) && vec_ok(out, 8, 2)) GO(f16, 8) else GO(f16, 1) }
    else if (dtype == DDPM_F32) { if (vec_ok(a, 4, 4) && vec_ok(b, 4, 4) && vec_ok(out, 4, 4)) GO(float, 4) else GO(float, 1) }
    else return DDPM_E_ARG;
#undef GO
    LAUNCH_OK();
    return 0;
}

// ------------------------------------------------------------------------------------ colsum
template <typename T, int VEC>
__global__ void __launch_bounds__(NT) colsum_kernel(TV dy, float* out_nc, float* dbias) {
    extern __shared__ float acc[];           // [C]
    const int n = blockIdx.y, C = dy.C, HW = dy.H * dy.W;
    for (int c = threadIdx.x; c < C; c += NT) acc[c] = 0.f;
    __syncthreads();
    PixMap m = make_map<VEC>(C);
    if (m.active) {
        float s[VEC];
#pragma unroll
        for (int i = 0; i < VEC; ++i) s[i] = 0.f;
        const int per = (HW + gridDim.x - 1) / gridDim.x;
        const int p0 = blockIdx.x * per, p1 = min(HW, p0 + per);
        for (int p = p0 + m.prow; p < p1; p += m.ppi) {
            int y = p / dy.W, xx = p - y * dy.W;
            float v[VEC];
            ldv<T, VEC>(dy.at<T>(n, y, xx, m.cv * VEC), v);
#pragma unroll
            for (int i = 0; i < VEC; ++i) s[i] += v[i];
        }
#pragma unroll
        for (int i = 0; i < VEC; ++i) atomicAdd(&acc[m.cv * VEC + i], s[i]);
    }
    __syncthreads();
    for (int c = threadIdx.x; c < C; c += NT) {
        if (out_nc) atomicAdd(&out_nc[(size_t)n * C + c], acc[c]);
        if (dbias) atomicAdd(&dbias[c], acc[c]);
    }
}
extern "C" int ddpm_colsum(const ddpm_tensor* dy, int dtype, float* out_nc, float* dbias, void* stream) {
    if (!tensor_ok(dy) || (!out_nc && !dbias)) return DDPM_E_ARG;
    cudaStream_t st = (cudaStream_t)stream;
    if (out_nc) CUDA_TRY(cudaMemsetAsync(out_nc, 0, sizeof(float) * dy->N * dy->C, st));
    TV v(*dy);
    int HW = dy->H * dy->W;
#define GO(T, VEC) { int cvs = dy->C / VEC; if (cvs > NT) return DDPM_E_ARG; int ppi = NT / cvs; \
        dim3 grid(blocks_per_image(dy->N, HW, ppi * 8), dy->N); \
        if (launch_kernel(colsum_kernel<T, VEC>, grid, dim3(NT), sizeof(float) * dy->C, st, v, out_nc, dbias) != cudaSuccess) return (int)cudaGetLastError(); }
    if (dtype == DDPM_BF16) { if (vec_ok(dy, 8, 2)) GO(bf16, 8) else GO(bf16, 1) }
    else if (dtype == DDPM_F16) { if (vec_ok(dy, 8, 2)) GO(f16, 8) else GO(f16, 1) }
    else if (dtype == DDPM_F32) { if (vec_ok(dy, 4, 4)) GO(float, 4) else GO(float, 1) }
    else return DDPM_E_ARG;
#undef GO
    LAUNCH_OK();
    return 0;
}
