#include "kernels.cuh"

// resident CTAs per SM the register allocator must allow, per block-size specialisation
#ifndef RS_MIN_BLOCKS_288
#define RS_MIN_BLOCKS_288 3  // ranges up to 1152 hands: 288 threads, <= 75 registers
#endif
#ifndef RS_MIN_BLOCKS_352
#define RS_MIN_BLOCKS_352 2  // up to 1326 hands: 352 threads, <= 93 registers
#endif

#ifndef RS_POLL_SLEEP_NS
#define RS_POLL_SLEEP_NS 64  // pause between two rounds of flag polls of the dispatcher
#endif

namespace rs {

namespace {

// ------------------------------------------------------------------------------------------------
// small helpers
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t ld_acquire_u32(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
// system scope: flags that live in a peer GPU's memory
__device__ __forceinline__ uint32_t ld_acquire_sys_u32(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_sys_u32(uint32_t* p, uint32_t v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ void st_release_u32(uint32_t* p, uint32_t v) {
    asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
// bulk L2 prefetch (TMA unit, no destination): bytes must be a multiple of 16, p 16-byte aligned
__device__ __forceinline__ void prefetch_l2_bulk(const void* p, uint32_t bytes) {
    if (bytes) asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(p), "r"(bytes) : "memory");
}
__device__ __forceinline__ float4 ldcg4(const float* p) { return __ldcg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ void stcg4(float* p, float4 v) { __stcg(reinterpret_cast<float4*>(p), v); }
__device__ __forceinline__ float4 f4zero() { return make_float4(0.f, 0.f, 0.f, 0.f); }
__device__ __forceinline__ float4 f4add(float4 a, float4 b) { return make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w); }
__device__ __forceinline__ float f4get(const float4& v, int i) { return i == 0 ? v.x : (i == 1 ? v.y : (i == 2 ? v.z : v.w)); }
__device__ __forceinline__ void f4set(float4& v, int i, float x) {
    if (i == 0) v.x = x;
    else if (i == 1) v.y = x;
    else if (i == 2) v.z = x;
    else v.w = x;
}
__device__ __forceinline__ void unpack4(uint2 u, uint32_t (&o)[4]) {
    o[0] = u.x & 0xffffu;
    o[1] = u.x >> 16;
    o[2] = u.y & 0xffffu;
    o[3] = u.y >> 16;
}

// barrier among the compute warps only (the dispatcher warp never joins it)
__device__ __forceinline__ void csync(int n_compute) { asm volatile("bar.sync 2, %0;" ::"r"(n_compute) : "memory"); }
// barrier between the compute warps and the dispatcher warp: one per task
__device__ __forceinline__ void hsync(int n_all) { asm volatile("bar.sync 1, %0;" ::"r"(n_all) : "memory"); }

// shared-memory mbarrier: the compute warps arrive when a task's body is finished, the dispatcher tests it
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(uint32_t(__cvta_generic_to_shared(bar))), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.release.cta.shared::cta.b64 _, [%0];" ::"r"(uint32_t(__cvta_generic_to_shared(bar))) : "memory");
}
__device__ __forceinline__ bool mbar_test(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\tmbarrier.test_wait.parity.acquire.cta.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(uint32_t(__cvta_generic_to_shared(bar))), "r"(parity)
        : "memory");
    return ok != 0;
}

// Called once per round of a spin loop.  Cheap on most rounds; every 256th looks at the device abort word and the
// clock, every 4096th at the host's abort word (a read over PCIe).  Returns true when the kernel has to give up.
__device__ __forceinline__ bool wait_gives_up(const TaskArgs& A, unsigned long long t_start, uint32_t& spins) {
    if ((++spins & 255u) != 0) return false;
    if (*reinterpret_cast<const volatile unsigned int*>(&A.ctl->abort)) return true;
    bool trip = false;
    if ((spins & 4095u) == 0 && A.host_abort && *A.host_abort) trip = true;
    if (A.wait_timeout_ns) {
        unsigned long long now;
        asm volatile("mov.u64 %0, %globaltimer;" : "=l"(now));
        if (now - t_start > A.wait_timeout_ns) trip = true;
    }
    if (trip) atomicExch(&A.ctl->abort, 1u);
    return trip;
}
__device__ __forceinline__ unsigned long long global_ns() {
    unsigned long long now;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(now));
    return now;
}

struct Ctx {
    int nc;  // compute threads
    int tid, lane, warp, nwarps;
    int pos4;  // first of the four hands this thread owns
    int p, o, Hp, Ho, HpP, HoP, Hx;
};

// Shared memory of a CTA at COMPILE-TIME offsets: the arrays need no pointer registers and every access is base +
// immediate.  The capacity HC = 4 * MAXT is what the build's threads cover (1152 positions in the 288-thread build, 1408 =
// 1326 hands padded in the wide one): every function that touches these arrays is a template on HC.  A smaller
// footprint leaves more of the SM's combined L1 / shared-memory array to L1 (spills, table loads).
//   SM_RS  [HC]          opponent reach being scanned
//   SM_P   [HC + 4]      exclusive prefix of reach by position (strength order on the river)
//   SM_GB  [2*HC + 8]    exclusive prefix of reach over the opponent's per-card lists
//   SM_WSA / SM_WSB [32] warp totals of the two scans
//   SM_B   [64]          boundaries of the opponent's non-empty card lists: B[j] = GB at the start of list j, B[J] = the
//                        total; B[54] = B[55] = 0 for a card the opponent does not hold (tasks.h: HandRec)
//   SM_WSC / SM_WSD [32] warp totals of the two scans of a fold reach scanned alongside (scan_reach<true>)
//   SM_BF  [64]          the boundaries B of that fold reach
//   SM_REC [4][HC]       the traverser's per-hand records of the board, staged by cp.async at the start of a task
//   SM_CL  [HC] words    the opponent's per-card lists of the board (u16 pairs), staged the same way
//   SM_X   [slots][Hx]   scratch vectors (terminal-child reach, bucketed rows), Hx known at run time
extern __shared__ __align__(16) float smem_raw[];
#define SM_RS (smem_raw)
#define SM_P (smem_raw + HC)
#define SM_GB (smem_raw + 2 * HC + 4)
#define SM_WSA (smem_raw + 4 * HC + 12)
#define SM_WSB (smem_raw + 4 * HC + 44)
#define SM_B (smem_raw + 4 * HC + 76)
#define SM_WSC (smem_raw + 4 * HC + 140)
#define SM_WSD (smem_raw + 4 * HC + 172)
#define SM_BF (smem_raw + 4 * HC + 204)
#define SM_REC (reinterpret_cast<uint32_t*>(smem_raw + 4 * HC + 268))
#define SM_CL (reinterpret_cast<uint32_t*>(smem_raw + 8 * HC + 268))
#define SM_X (smem_raw + 9 * HC + 268)
constexpr int smem_fixed_floats(int HC) { return 9 * HC + 268; }

// Copy the thread's eight entries of the opponent's per-card lists (cl_pos of the board, u16) into shared memory with
// cp.async; scan_reach reads them back.  Like the hand records (stage_recs) this is issued when a task starts, so the
// L2 round trip overlaps the reach load instead of following it, and costs no registers.
template <int HC>
__device__ __forceinline__ void stage_lists_raw(int tid, int HoP, const uint16_t* __restrict__ cl_pos_b) {
    if (8 * tid < 2 * HoP)
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(uint32_t(__cvta_generic_to_shared(SM_CL + 4 * tid))), "l"(cl_pos_b + 8 * tid)
                     : "memory");
    asm volatile("cp.async.commit_group;" ::: "memory");
}

// Exclusive prefix sums of opponent reach r (shared memory, HoP floats, zero past the live hands):
//   P[i]  = reach of the i weakest hands           (position order)
//   GB[e] = reach of the first e entries of the opponent's concatenated per-card lists
// One pass: every thread scans its 4 positions and its 8 list entries; warp shuffles + one cross-warp step.
// Returns the total reach (all threads).  Positions from 4 * nc on are not scanned (a round launched with fewer threads
// holds no live hand there), so in the 288-thread build, whose arrays end at 4 * 288 positions, the totals go to
// P[min(HoP, 4 * nc)] and GB[2 * min(HoP, 4 * nc)].
//
// FOLD: the same pass also scans a second reach vector rf for what a fold value needs (hand_mass): its total, returned
// in *total_f, and its list boundaries in SM_BF; it writes no P or GB.  An opponent node with a fold and a showdown child
// values both after one pass (three barriers) instead of two.  Every sum of rf is formed exactly as a scan of rf alone
// would form it, so the values are bit-identical either way.
template <int HC, bool FOLD>
__device__ __forceinline__ float scan_reach(const Ctx& c, const float* r, const float* rf = nullptr, float* total_f = nullptr) {
    csync(c.nc);  // r (and rf) are complete; previous readers of P / GB / B are done
    const int hend = HC >= 4 * MAX_TASK_THREADS ? c.HoP : min(c.HoP, 4 * c.nc);  // the wide build holds every HoP
    float4 x = f4zero();
    float lc = 0.f;  // FOLD: the thread's four positions of rf, summed as they are loaded
    if (c.pos4 < c.HoP) {
        x = *reinterpret_cast<const float4*>(r + c.pos4);
        if (FOLD) {
            const float4 xf = *reinterpret_cast<const float4*>(rf + c.pos4);
            lc = (xf.x + xf.y) + (xf.z + xf.w);
        }
    }
    float y[8], yf[8];
    uint32_t w[4];
    {
        // the thread's eight list entries were staged by stage_lists when the task started
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        uint4 u = make_uint4(0x07ff07ffu, 0x07ff07ffu, 0x07ff07ffu, 0x07ff07ffu);
        if (8 * c.tid < 2 * c.HoP) u = *reinterpret_cast<const uint4*>(SM_CL + 4 * c.tid);
        w[0] = u.x;
        w[1] = u.y;
        w[2] = u.z;
        w[3] = u.w;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const uint32_t a = w[i] & CL_POS_MASK, b = (w[i] >> 16) & CL_POS_MASK;
            y[2 * i] = a != CL_POS_NONE ? r[a] : 0.f;
            y[2 * i + 1] = b != CL_POS_NONE ? r[b] : 0.f;
            if (FOLD) {
                yf[2 * i] = a != CL_POS_NONE ? rf[a] : 0.f;
                yf[2 * i + 1] = b != CL_POS_NONE ? rf[b] : 0.f;
            }
        }
    }
    const float la = (x.x + x.y) + (x.z + x.w);
    float lb = 0.f, ld = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        lb += y[i];
        if (FOLD) ld += yf[i];
    }
    float ia = la, ib = lb, ic = lc, id = ld;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const float ta = __shfl_up_sync(0xffffffffu, ia, d);
        const float tb = __shfl_up_sync(0xffffffffu, ib, d);
        float tc = 0.f, td = 0.f;
        if (FOLD) {
            tc = __shfl_up_sync(0xffffffffu, ic, d);
            td = __shfl_up_sync(0xffffffffu, id, d);
        }
        if (c.lane >= d) {
            ia += ta;
            ib += tb;
            if (FOLD) {
                ic += tc;
                id += td;
            }
        }
    }
    if (c.lane == 31) {
        SM_WSA[c.warp] = ia;
        SM_WSB[c.warp] = ib;
        if (FOLD) {
            SM_WSC[c.warp] = ic;
            SM_WSD[c.warp] = id;
        }
    }
    csync(c.nc);
    // every warp scans the (<= 11) warp totals itself
    float wa = c.lane < c.nwarps ? SM_WSA[c.lane] : 0.f;
    float wb = c.lane < c.nwarps ? SM_WSB[c.lane] : 0.f;
    float wc = 0.f, wd = 0.f;
    if (FOLD) {
        wc = c.lane < c.nwarps ? SM_WSC[c.lane] : 0.f;
        wd = c.lane < c.nwarps ? SM_WSD[c.lane] : 0.f;
    }
#pragma unroll
    for (int d = 1; d < 16; d <<= 1) {
        const float ta = __shfl_up_sync(0xffffffffu, wa, d);
        const float tb = __shfl_up_sync(0xffffffffu, wb, d);
        float tc = 0.f, td = 0.f;
        if (FOLD) {
            tc = __shfl_up_sync(0xffffffffu, wc, d);
            td = __shfl_up_sync(0xffffffffu, wd, d);
        }
        if (c.lane >= d) {
            wa += ta;
            wb += tb;
            if (FOLD) {
                wc += tc;
                wd += td;
            }
        }
    }
    const float total = __shfl_sync(0xffffffffu, wa, c.nwarps - 1);
    const float total_b = __shfl_sync(0xffffffffu, wb, c.nwarps - 1);
    const float base_a = c.warp > 0 ? __shfl_sync(0xffffffffu, wa, c.warp - 1) : 0.f;
    const float base_b = c.warp > 0 ? __shfl_sync(0xffffffffu, wb, c.warp - 1) : 0.f;
    float ea = base_a + ia - la, eb = base_b + ib - lb;
    float total_d = 0.f, ed = 0.f;
    if (FOLD) {
        *total_f = __shfl_sync(0xffffffffu, wc, c.nwarps - 1);
        total_d = __shfl_sync(0xffffffffu, wd, c.nwarps - 1);
        const float base_d = c.warp > 0 ? __shfl_sync(0xffffffffu, wd, c.warp - 1) : 0.f;
        ed = base_d + id - ld;
    }
    if (c.pos4 < c.HoP) {
        float4 o;
        o.x = ea;
        o.y = ea + x.x;
        o.z = o.y + x.y;
        o.w = o.z + x.z;
        *reinterpret_cast<float4*>(SM_P + c.pos4) = o;
    }
    if (8 * c.tid < 2 * c.HoP) {
        float4 o0, o1;
        o0.x = eb;
        o0.y = o0.x + y[0];
        o0.z = o0.y + y[1];
        o0.w = o0.z + y[2];
        o1.x = o0.w + y[3];
        o1.y = o1.x + y[4];
        o1.z = o1.y + y[5];
        o1.w = o1.z + y[6];
        *reinterpret_cast<float4*>(SM_GB + 8 * c.tid) = o0;
        *reinterpret_cast<float4*>(SM_GB + 8 * c.tid + 4) = o1;
        // boundaries of the card lists: an entry flagged CL_FIRST stores its exclusive prefix as B[ordinal]; the thread's
        // first ordinal rides in the spare bits of its first two entries (thread 0 carries the number of lists there)
        const uint32_t ord0 = ((w[0] >> 11) & 7u) | (((w[0] >> 27) & 7u) << 3);
        const uint32_t b0 = c.tid == 0 ? 0u : ord0;
        float* bp = SM_B + b0;
        const float ex[8] = {o0.x, o0.y, o0.z, o0.w, o1.x, o1.y, o1.z, o1.w};
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const bool first = ((w[i >> 1] >> ((i & 1) * 16)) & CL_FIRST) != 0;
            if (first) *bp++ = ex[i];
        }
        if (c.tid == 0) SM_B[ord0] = total_b;  // ord0 of thread 0 = J, the number of non-empty lists
        if (FOLD) {  // the same exclusive prefixes of rf, kept only at the list boundaries
            float* bf = SM_BF + b0;
            float e = ed;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const bool first = ((w[i >> 1] >> ((i & 1) * 16)) & CL_FIRST) != 0;
                if (first) *bf++ = e;
                e += yf[i];
            }
            if (c.tid == 0) SM_BF[ord0] = total_d;
        }
    }
    if (c.tid == 0) {
        SM_P[hend] = total;
        SM_GB[2 * hend] = total_b;
    }
    csync(c.nc);
    return total;
}

// The per-hand records of a board are stored as four word planes [4][Hpad]: one 128-bit copy per plane gives the
// thread the same word of its four hands, fully coalesced across the warp.
// The records are needed only after the first scan of a task.  Loading them into registers up front would cost 16
// registers across the scan, loading them afterwards exposes an L2 round trip: instead every thread copies its own
// 4 x 16 bytes into shared memory with cp.async when the task starts and reads them back when it needs them (no
// barrier: a thread only ever reads what it copied itself).
template <int HC>
__device__ __forceinline__ void stage_recs(const Ctx& c, const uint32_t* __restrict__ planes) {
    if (c.pos4 < c.HpP) {
#pragma unroll
        for (int w = 0; w < 4; ++w)
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(uint32_t(__cvta_generic_to_shared(SM_REC + w * HC + c.pos4))),
                         "l"(planes + size_t(w) * c.HpP + c.pos4)
                         : "memory");
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
}
__device__ __forceinline__ void staged_recs_wait() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }
template <int HC>
__device__ __forceinline__ void staged_recs4(const Ctx& c, uint4 (&rec)[4]) {
    const uint4 w0 = *reinterpret_cast<const uint4*>(SM_REC + c.pos4);
    const uint4 w1 = *reinterpret_cast<const uint4*>(SM_REC + HC + c.pos4);
    const uint4 w2 = *reinterpret_cast<const uint4*>(SM_REC + 2 * HC + c.pos4);
    const uint4 w3 = *reinterpret_cast<const uint4*>(SM_REC + 3 * HC + c.pos4);
    rec[0] = make_uint4(w0.x, w1.x, w2.x, w3.x);
    rec[1] = make_uint4(w0.y, w1.y, w2.y, w3.y);
    rec[2] = make_uint4(w0.z, w1.z, w2.z, w3.z);
    rec[3] = make_uint4(w0.w, w1.w, w2.w, w3.w);
}

// After scan_reach: for the traverser's hand record `rec`
//   mass = opponent reach compatible with the hand (total - both cards' sums + the identical combo)
//   sd   = weaker minus stronger compatible opponent reach (showdown, cfr.rs:532-556)
__device__ __forceinline__ float ldsb(const float* base, uint32_t byte_off) {  // shared-memory load at base + byte offset
    return *reinterpret_cast<const float*>(reinterpret_cast<const char*>(base) + byte_off);
}
template <int HC>
__device__ __forceinline__ void hand_terms(const Ctx& c, const float* r, float total, const uint4& rec, float& mass, float& sd) {
    const uint32_t k0 = rec.w & 0x1ffu, k1 = (rec.w >> 9) & 0x1ffu, same4 = rec.w >> 18;
    const float g0s = ldsb(SM_B, k0), g0e = ldsb(SM_B + 1, k0), g1s = ldsb(SM_B, k1), g1e = ldsb(SM_B + 1, k1);
    mass = total - (g0e - g0s) - (g1e - g1s) + (same4 != HREC_SAME_NONE ? ldsb(r, same4) : 0.f);
    sd = ldsb(SM_P, rec.x & 0xffffu) + ldsb(SM_P, rec.x >> 16) - total - ldsb(SM_GB, rec.y & 0xffffu) - ldsb(SM_GB, rec.y >> 16) + g0s + g0e -
         ldsb(SM_GB, rec.z & 0xffffu) - ldsb(SM_GB, rec.z >> 16) + g1s + g1e;
}
// B: the boundaries of r's scan (SM_B, or SM_BF for the fold reach of scan_reach<true>)
__device__ __forceinline__ float hand_mass(const float* B, const float* r, float total, const uint4& rec) {
    const uint32_t k0 = rec.w & 0x1ffu, k1 = (rec.w >> 9) & 0x1ffu, same4 = rec.w >> 18;
    return total - (ldsb(B + 1, k0) - ldsb(B, k0)) - (ldsb(B + 1, k1) - ldsb(B, k1)) + (same4 != HREC_SAME_NONE ? ldsb(r, same4) : 0.f);
}

// Opponent reach of the thread's four positions for this task (masked by what the board removes).
__device__ __forceinline__ float4 load_reach4(const TaskArgs& A, const Ctx& c, const NodeTask& nt, const RoundArgs& Rk, int k, int b) {
    float4 r = f4zero();
    if (c.pos4 >= c.HoP) return r;
    if (nt.r_in == RIN_INITIAL) {
        const uint32_t nl = Rk.rp[c.o].n_live[b];
        uint32_t s[4];
        unpack4(__ldg(reinterpret_cast<const uint2*>(Rk.rp[c.o].slot_of_pos + size_t(b) * c.HoP + c.pos4)), s);
        const float* __restrict__ w = A.root_weights[c.o];
#pragma unroll
        for (int i = 0; i < 4; ++i) f4set(r, i, uint32_t(c.pos4 + i) < nl ? __ldg(w + s[i]) : 0.f);
    } else if (nt.rin_parent_round) {
        const RoundArgs& Rp = A.rounds[k - 1];
        const float* src = Rp.rbuf + (size_t(nt.r_in) * Rp.n_boards + Rk.parent_board[b]) * c.HoP;
        uint32_t pp[4];
        unpack4(__ldg(reinterpret_cast<const uint2*>(Rk.rp[c.o].parent_pos + size_t(b) * c.HoP + c.pos4)), pp);
#pragma unroll
        for (int i = 0; i < 4; ++i) f4set(r, i, pp[i] != 0xffffu ? __ldcg(src + pp[i]) : 0.f);  // the dealt card removes hands
    } else {
        r = ldcg4(Rk.rbuf + (size_t(nt.r_in) * Rk.n_boards + b) * c.HoP + c.pos4);
    }
    return r;
}

// Sum of the value vectors feeding one child (thread's four positions).
__device__ __forceinline__ float4 child_value4(const TaskArgs& A, const Ctx& c, const RoundArgs& Rk, const TaskChild& ch, int b) {
    float4 v = f4zero();
    if (c.pos4 >= c.HpP) return v;
    for (int s = 0; s < ch.n_src; ++s) {
        const TaskSrc sr = A.srcs[ch.src_first + s];
        const float* base = (sr.kind == SK_CBUF ? Rk.cbuf : Rk.gathered) + (size_t(sr.buf) * Rk.n_boards + b) * c.HpP;
        v = f4add(v, ldcg4(base + c.pos4));
    }
    return v;
}

// Store a node's value for the thread's four positions.  Street roots write in the parent board's hand order
// (positions the child board removes are never written and stay zero), so the chance gather is a coalesced sum.
__device__ __forceinline__ void store_value4(const Ctx& c, const NodeTask& nt, const RoundArgs& Rk, int b, float* out, float4 v) {
    if (!nt.root_scatter) {
        stcg4(out + c.pos4, v);
        return;
    }
    uint32_t pp[4];
    unpack4(__ldg(reinterpret_cast<const uint2*>(Rk.rp[c.p].parent_pos + size_t(b) * c.HpP + c.pos4)), pp);
    if (pp[0] != 0xffffu) __stcg(out + pp[0], v.x);
    if (pp[1] != 0xffffu) __stcg(out + pp[1], v.y);
    if (pp[2] != 0xffffu) __stcg(out + pp[2], v.z);
    if (pp[3] != 0xffffu) __stcg(out + pp[3], v.w);
}
__device__ __forceinline__ void store_value1(const Ctx& c, const NodeTask& nt, const RoundArgs& Rk, int b, float* out, int pos, float v) {
    if (!nt.root_scatter) {
        __stcg(out + pos, v);
        return;
    }
    const uint32_t pp = Rk.rp[c.p].parent_pos[size_t(b) * c.HpP + pos];
    if (pp != 0xffffu) __stcg(out + pp, v);
}

// Regret matching of one row held in registers (infoset.rs:83-123).
template <int NA>
__device__ __forceinline__ void sigma_row(const float (&g)[4 * NA], int i, float (&sg)[NA]) {
    float norm = 0.f;
#pragma unroll
    for (int a = 0; a < NA; ++a) {
        sg[a] = fmaxf(g[i * NA + a], 0.f);
        norm += sg[a];
    }
    const float inv = __fdividef(1.0f, norm);  // MUFU.RCP + one multiply (2 ulp), not the IEEE division sequence; only used when norm > 0
#pragma unroll
    for (int a = 0; a < NA; ++a) sg[a] = norm > 0.f ? sg[a] * inv : 1.0f / float(NA);
}

// Four table rows x NA actions into registers.  identity: rows are the thread's four positions (contiguous 4*NA
// floats, NA 128-bit loads); otherwise rows come from row_of_pos and are loaded one by one.
template <int NA>
__device__ __forceinline__ void load_rows(const float* __restrict__ slab, bool identity, int pos4, uint32_t n_rows_pad,
                                          const uint32_t (&rows)[4], float (&g)[4 * NA]) {
    if (identity) {
        if (uint32_t(pos4) < n_rows_pad) {
#pragma unroll
            for (int v = 0; v < NA; ++v) {
                const float4 t = *reinterpret_cast<const float4*>(slab + size_t(pos4) * NA + 4 * v);
                g[4 * v] = t.x;
                g[4 * v + 1] = t.y;
                g[4 * v + 2] = t.z;
                g[4 * v + 3] = t.w;
            }
        } else {
#pragma unroll
            for (int e = 0; e < 4 * NA; ++e) g[e] = 0.f;
        }
    } else {
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int a = 0; a < NA; ++a) g[i * NA + a] = rows[i] != 0xffffu ? slab[size_t(rows[i]) * NA + a] : 0.f;
    }
}

// ------------------------------------------------------------------------------------------------
// TK_DOWN: opponent node (cfr.rs:582-586) + its terminal children (cfr.rs:523-558)
// ------------------------------------------------------------------------------------------------
// one sampled action per opponent hand (cfr.rs:466-475): the first action whose cumulative probability exceeds u
template <int NA>
__device__ __forceinline__ void xs_pick(const TaskArgs& A, float u, float (&sg)[NA]) {
    int pick = NA - 1;
    bool found = false;
    float cum = 0.f;
#pragma unroll
    for (int a = 0; a + 1 < NA; ++a) {
        cum += sg[a];
        if (!found && u < cum) {
            pick = a;
            found = true;
        }
    }
#pragma unroll
    for (int a = 0; a < NA; ++a) sg[a] = (a == pick) ? (A.xs_mode == 2 ? sg[a] : 1.0f) : 0.f;
}

// The terminal children of an opponent node (cfr.rs:523-558), whose reach vectors are staged in SM_X slots 0, 1, ... in
// action order, and the hand records and per-card lists staged by cp.async.  Stores the node's terminal partial value:
// the sum of coef * term over those children, accumulated in action order.  A fold and a showdown child (most river
// opponent nodes) share one scan pass; any other set of terminal children is scanned child by child.
template <int HC>
__device__ __forceinline__ void down_terminals(const Ctx& c, const NodeTask& nt, const RoundArgs& Rk, int b, int n_act) {
    const uint32_t nl_p = Rk.rp[c.p].n_live[b];
    const float scale = Rk.chance_scale[b];
    int n_fold = 0, n_sd = 0, a_fold = 0, a_sd = 0;
    for (int a = 0; a < n_act; ++a) {
        const int ck = nt.child[a].kind;
        if (ck == CK_FOLD) {
            ++n_fold;
            a_fold = a;
        } else if (ck == CK_SHOWDOWN) {
            ++n_sd;
            a_sd = a;
        }
    }
    float4 acc = f4zero();
    if (n_fold == 1 && n_sd == 1) {
        const bool fold_first = a_fold < a_sd;
        const float* rf = SM_X + (fold_first ? 0 : c.Hx);
        const float* rs = SM_X + (fold_first ? c.Hx : 0);
        float total_f;
        const float total = scan_reach<HC, true>(c, rs, rf, &total_f);
        const float cf = nt.child[a_fold].coef * scale, cs = nt.child[a_sd].coef * scale;
        const float c0 = fold_first ? cf : cs, c1 = fold_first ? cs : cf;
        staged_recs_wait();
        if (c.pos4 < c.HpP) {
            uint4 rec[4];
            staged_recs4<HC>(c, rec);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                if (uint32_t(c.pos4 + i) < nl_p) {
                    float m_sd, sd;  // m_sd: the showdown reach's mass, not needed
                    hand_terms<HC>(c, rs, total, rec[i], m_sd, sd);
                    const float m = hand_mass(SM_BF, rf, total_f, rec[i]);
                    const float t0 = fold_first ? m : sd, t1 = fold_first ? sd : m;
                    f4set(acc, i, f4get(acc, i) + c0 * t0);
                    f4set(acc, i, f4get(acc, i) + c1 * t1);
                }
            }
        }
    } else {
        int slot = 0;
        for (int a = 0; a < n_act; ++a) {
            const int ck = nt.child[a].kind;
            if (ck != CK_FOLD && ck != CK_SHOWDOWN) continue;
            const float* r = SM_X + slot * c.Hx;
            ++slot;
            const float cf = nt.child[a].coef * scale;
            const float total = scan_reach<HC, false>(c, r);
            staged_recs_wait();
            if (c.pos4 < c.HpP) {
                uint4 rec[4];
                staged_recs4<HC>(c, rec);  // read back for every terminal child instead of held in registers across the scans
#pragma unroll
                for (int i = 0; i < 4; ++i) {
                    if (uint32_t(c.pos4 + i) < nl_p) {
                        float m, sd;
                        if (ck == CK_FOLD) {
                            m = hand_mass(SM_B, r, total, rec[i]);
                            f4set(acc, i, f4get(acc, i) + cf * m);
                        } else {
                            hand_terms<HC>(c, r, total, rec[i], m, sd);
                            f4set(acc, i, f4get(acc, i) + cf * sd);
                        }
                    }
                }
            }
        }
    }
    if (c.pos4 < c.HpP) stcg4(Rk.cbuf + (size_t(nt.out) * Rk.n_boards + b) * c.HpP + c.pos4, acc);
}

template <int HC, int MODE, int NA, bool XS>
__device__ __forceinline__ void task_down(const TaskArgs& A, const Ctx& c, const NodeTask& nt, const RoundArgs& Rk, int k, int b) {
    const DevRoundPlayer& O = Rk.rp[c.o];
    const uint32_t nrp = O.n_rows_pad[b];
    const float* __restrict__ slab = (MODE == KM_CFR ? O.regrets : O.ssum) + O.board_off[b] + size_t(nrp) * nt.cum_a;
    if (nt.out >= 0) {
        stage_lists_raw<HC>(c.tid, c.HoP, O.cl_pos + size_t(b) * 2 * c.HoP);
        stage_recs<HC>(c, reinterpret_cast<const uint32_t*>(Rk.rp[c.p].hrec) + size_t(b) * 4 * c.HpP);
    }
    const float4 r4 = load_reach4(A, c, nt, Rk, k, b);
    uint32_t rows[4] = {0xffffu, 0xffffu, 0xffffu, 0xffffu};
    if (!O.identity && c.pos4 < c.HoP) unpack4(__ldg(reinterpret_cast<const uint2*>(O.row_of_pos + size_t(b) * c.HoP + c.pos4)), rows);
    float g[4 * NA];
    load_rows<NA>(slab, O.identity != 0, c.pos4, nrp, rows, g);
    float4 v[NA];
    uint32_t xs_slot[4] = {0, 0, 0, 0};
    if (XS && c.pos4 < c.HoP) unpack4(__ldg(reinterpret_cast<const uint2*>(O.slot_of_pos + size_t(b) * c.HoP + c.pos4)), xs_slot);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        float sg[NA];
        sigma_row<NA>(g, i, sg);
        if (XS) xs_pick<NA>(A, xs_uniform(A.xs_key, nt.an_index, uint32_t(Rk.board_base + b), xs_slot[i]), sg);
        const float r = f4get(r4, i);
#pragma unroll
        for (int a = 0; a < NA; ++a) f4set(v[a], i, r * sg[a]);
    }
    int slot = 0;
#pragma unroll
    for (int a = 0; a < NA; ++a) {
        const int ck = nt.child[a].kind;
        if (c.pos4 < c.HoP) {
            if (ck == CK_FOLD || ck == CK_SHOWDOWN) *reinterpret_cast<float4*>(SM_X + slot * c.Hx + c.pos4) = v[a];
            else if (nt.child[a].buf >= 0) stcg4(Rk.rbuf + (size_t(nt.child[a].buf) * Rk.n_boards + b) * c.HoP + c.pos4, v[a]);
        }
        if (ck == CK_FOLD || ck == CK_SHOWDOWN) ++slot;
    }
    if (nt.out < 0) return;
    down_terminals<HC>(c, nt, Rk, b, NA);
}

// any number of actions, any row mapping: scalar loads, two passes over the actions
template <int HC, int MODE, bool XS>
__device__ __forceinline__ void task_down_generic(const TaskArgs& A, const Ctx& c, const NodeTask& nt, const RoundArgs& Rk, int k, int b) {
    const DevRoundPlayer& O = Rk.rp[c.o];
    const uint32_t nrp = O.n_rows_pad[b];
    const float* __restrict__ slab = (MODE == KM_CFR ? O.regrets : O.ssum) + O.board_off[b] + size_t(nrp) * nt.cum_a;
    const float4 r4 = load_reach4(A, c, nt, Rk, k, b);
    const int n_act = nt.n_act;
    const uint32_t nl_o = O.n_live[b];
    uint32_t rows[4] = {0xffffu, 0xffffu, 0xffffu, 0xffffu};
    if (c.pos4 < c.HoP) unpack4(__ldg(reinterpret_cast<const uint2*>(O.row_of_pos + size_t(b) * c.HoP + c.pos4)), rows);
    if (c.pos4 < c.HoP) {
        for (int i = 0; i < 4; ++i) {
            const bool live = uint32_t(c.pos4 + i) < nl_o && rows[i] != 0xffffu;
            const float r = live ? f4get(r4, i) : 0.f;
            float norm = 0.f;
            if (live)
                for (int a = 0; a < n_act; ++a) norm += fmaxf(slab[size_t(rows[i]) * n_act + a], 0.f);
            int pick = -1;  // sampled-opponent-action mode: the one action this hand keeps its reach on
            if (XS && live) {
                const float u = xs_uniform(A.xs_key, nt.an_index, uint32_t(Rk.board_base + b), O.slot_of_pos[size_t(b) * c.HoP + c.pos4 + i]);
                pick = n_act - 1;
                float cum = 0.f;
                for (int a = 0; a + 1 < n_act; ++a) {
                    cum += norm > 0.f ? fmaxf(slab[size_t(rows[i]) * n_act + a], 0.f) / norm : 1.0f / float(n_act);
                    if (u < cum) {
                        pick = a;
                        break;
                    }
                }
            }
            int slot = 0;
            for (int a = 0; a < n_act; ++a) {
                float v = 0.f;
                if (live) v = norm > 0.f ? r * fmaxf(slab[size_t(rows[i]) * n_act + a], 0.f) / norm : r / float(n_act);
                if (XS && live) v = (a == pick) ? (A.xs_mode == 2 ? v : r) : 0.f;
                const int ck = nt.child[a].kind;
                if (ck == CK_FOLD || ck == CK_SHOWDOWN) SM_X[(slot++) * c.Hx + c.pos4 + i] = v;
                else if (nt.child[a].buf >= 0) __stcg(Rk.rbuf + (size_t(nt.child[a].buf) * Rk.n_boards + b) * c.HoP + c.pos4 + i, v);
            }
        }
    }
    if (nt.out < 0) return;
    // generic path: staged right before the scans
    stage_lists_raw<HC>(c.tid, c.HoP, O.cl_pos + size_t(b) * 2 * c.HoP);
    stage_recs<HC>(c, reinterpret_cast<const uint32_t*>(Rk.rp[c.p].hrec) + size_t(b) * 4 * c.HpP);
    down_terminals<HC>(c, nt, Rk, b, n_act);
}

// ------------------------------------------------------------------------------------------------
// TK_UP_TRAV: traverser node (cfr.rs:588, 612-621)
// ------------------------------------------------------------------------------------------------
// common front part: stage the reach, run the scan, produce per-hand mass and showdown term
template <int HC>
__device__ __forceinline__ void trav_terms(const TaskArgs& A, const Ctx& c, const NodeTask& nt, const RoundArgs& Rk, int k, int b,
                                           bool need_sd, float4& mass, float4& sd) {
    const DevRoundPlayer& Pp = Rk.rp[c.p];
    stage_lists_raw<HC>(c.tid, c.HoP, Rk.rp[c.o].cl_pos + size_t(b) * 2 * c.HoP);
    stage_recs<HC>(c, reinterpret_cast<const uint32_t*>(Pp.hrec) + size_t(b) * 4 * c.HpP);
    const float4 r4 = load_reach4(A, c, nt, Rk, k, b);
    if (c.pos4 < c.HoP) *reinterpret_cast<float4*>(SM_RS + c.pos4) = r4;
    const float total = scan_reach<HC, false>(c, SM_RS);
    mass = f4zero();
    sd = f4zero();
    const uint32_t nl_p = Pp.n_live[b];
    staged_recs_wait();
    if (c.pos4 < c.HpP) {
        uint4 rec[4];
        staged_recs4<HC>(c, rec);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            if (uint32_t(c.pos4 + i) < nl_p) {
                float m, s = 0.f;
                if (need_sd) hand_terms<HC>(c, SM_RS, total, rec[i], m, s);
                else m = hand_mass(SM_B, SM_RS, total, rec[i]);
                f4set(mass, i, m);
                f4set(sd, i, s);
            }
        }
    }
}

// mass / showdown terms of a traverser node: computed here (scan + per-hand terms), or, on chain rounds, read from the
// two value buffers the node's TK_TRAV_TERMS task left
template <int HC>
__device__ __forceinline__ void trav_terms_or_load(const TaskArgs& A, const Ctx& c, const NodeTask& nt, const RoundArgs& Rk, int k, int b,
                                                   bool need_sd, float4& mass, float4& sd) {
    if (!nt.pre_terms) {
        trav_terms<HC>(A, c, nt, Rk, k, b, need_sd, mass, sd);
        return;
    }
    mass = f4zero();
    sd = f4zero();
    if (c.pos4 < c.HpP) {
        const float* m = Rk.cbuf + (size_t(nt.aux) * Rk.n_boards + b) * c.HpP + c.pos4;
        mass = ldcg4(m);
        if (need_sd) sd = ldcg4(m + size_t(Rk.n_boards) * c.HpP);
    }
}

// Update rule (rs_set_update_rule, DR builds only): {fp, fn, fs, floor} of this iteration, read once per task.  The regret
// update R' = max((R > 0 ? fp : fn) * R + d, floor), d already zero for a pruned action.
__device__ __forceinline__ float4 rule_factors(const TaskArgs& A) { return ldcg4(A.ctl->rule); }
__device__ __forceinline__ float rule_regret(const float4& f, float r, float d) { return fmaxf((r > 0.f ? f.x : f.y) * r + d, f.w); }

template <int HC, int MODE, int NA, bool DR>
__device__ __forceinline__ void task_trav(const TaskArgs& A, const Ctx& c, const NodeTask& nt, const RoundArgs& Rk, int k, int b) {
    const DevRoundPlayer& Pp = Rk.rp[c.p];
    const float scale = Rk.chance_scale[b];
    float4 dr;
    if (DR) dr = rule_factors(A);
    float4 v[NA];
    bool need_sd = false;
#pragma unroll
    for (int a = 0; a < NA; ++a) {
        v[a] = f4zero();
        need_sd |= (nt.child[a].kind == CK_SHOWDOWN);
    }
    float4 mass, sd;
    trav_terms_or_load<HC>(A, c, nt, Rk, k, b, need_sd, mass, sd);
    // child values that come from other tasks: loaded after the scan (held across it they cost registers the
    // 64-register build does not have: measured +2 %)
#pragma unroll
    for (int a = 0; a < NA; ++a)
        if (nt.child[a].kind == CK_VALUE) v[a] = child_value4(A, c, Rk, nt.child[a], b);
#pragma unroll
    for (int a = 0; a < NA; ++a) {
        const int ck = nt.child[a].kind;
        const float cf = nt.child[a].coef * scale;
        if (ck == CK_FOLD) v[a] = make_float4(cf * mass.x, cf * mass.y, cf * mass.z, cf * mass.w);
        else if (ck == CK_SHOWDOWN) v[a] = make_float4(cf * sd.x, cf * sd.y, cf * sd.z, cf * sd.w);
    }
    const uint32_t nrp = Pp.n_rows_pad[b];
    const uint32_t nl_p = Pp.n_live[b];
    float* out = (nt.root_scatter ? Rk.sbuf : Rk.cbuf) + (size_t(nt.out) * Rk.n_boards + b) * c.HpP;
    float* tabR = Pp.regrets + Pp.board_off[b] + size_t(nrp) * nt.cum_a;
    float* tabS = Pp.ssum + Pp.board_off[b] + size_t(nrp) * nt.cum_a;
    if (Pp.identity) {
        // rows are the thread's own four positions: everything stays in registers
        if (uint32_t(c.pos4) >= nrp) {
            if (c.pos4 < c.HpP && !nt.root_scatter) stcg4(out + c.pos4, f4zero());
            return;
        }
        const uint32_t none[4] = {0, 0, 0, 0};
        float g[4 * NA], ss[4 * NA];
        if (MODE == KM_CFR) load_rows<NA>(tabR, true, c.pos4, nrp, none, g);
        if (MODE != KM_BR) load_rows<NA>(tabS, true, c.pos4, nrp, none, ss);
        float4 vn4 = f4zero();
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            float sg[NA];
            float vn;
            if (MODE == KM_BR) {
                vn = -3.0e38f;
#pragma unroll
                for (int a = 0; a < NA; ++a) vn = fmaxf(vn, f4get(v[a], i));
            } else {
                if (MODE == KM_CFR) sigma_row<NA>(g, i, sg);
                else sigma_row<NA>(ss, i, sg);
                vn = 0.f;
#pragma unroll
                for (int a = 0; a < NA; ++a) vn += sg[a] * f4get(v[a], i);
            }
            const bool live = uint32_t(c.pos4 + i) < nl_p;
            f4set(vn4, i, live ? vn : 0.f);
            if (MODE == KM_CFR) {
                const float w = f4get(mass, i) * scale;
#pragma unroll
                for (int a = 0; a < NA; ++a) {
                    if (DR) {
                        const float r = g[i * NA + a];
                        if (live) {
                            g[i * NA + a] = rule_regret(dr, r, r > A.prune_threshold ? f4get(v[a], i) - vn : 0.f);
                            ss[i * NA + a] = dr.z * ss[i * NA + a] + sg[a] * w;
                        }
                    } else {
                        g[i * NA + a] += (live && g[i * NA + a] > A.prune_threshold) ? f4get(v[a], i) - vn : 0.f;
                        ss[i * NA + a] += live ? sg[a] * w : 0.f;
                    }
                }
            }
        }
        if (MODE == KM_CFR) {
#pragma unroll
            for (int q = 0; q < NA; ++q) {
                *reinterpret_cast<float4*>(tabR + size_t(c.pos4) * NA + 4 * q) = make_float4(g[4 * q], g[4 * q + 1], g[4 * q + 2], g[4 * q + 3]);
                *reinterpret_cast<float4*>(tabS + size_t(c.pos4) * NA + 4 * q) = make_float4(ss[4 * q], ss[4 * q + 1], ss[4 * q + 2], ss[4 * q + 3]);
            }
        }
        store_value4(c, nt, Rk, b, out, vn4);
        return;
    }
    // bucketed rows: values and masses go through shared memory, one thread per row (CSR row -> positions)
    float* M = SM_X;
    if (c.pos4 < c.HpP) {
        *reinterpret_cast<float4*>(M + c.pos4) = mass;
#pragma unroll
        for (int a = 0; a < NA; ++a) *reinterpret_cast<float4*>(SM_X + (1 + a) * c.Hx + c.pos4) = v[a];
        if (!nt.root_scatter) stcg4(out + c.pos4, f4zero());
    }
    csync(c.nc);
    const uint32_t n_rows = Pp.n_rows[b];
    const uint16_t* __restrict__ rstart = Pp.row_start + size_t(b) * (c.HpP + 4);
    const uint16_t* __restrict__ rpos = Pp.row_pos + size_t(b) * c.HpP;
    const float* V1 = SM_X + c.Hx;
    for (uint32_t row = c.tid; row < n_rows; row += c.nc) {
        float rg[NA], sr[NA], sg[NA], d[NA];
        float norm = 0.f;
#pragma unroll
        for (int a = 0; a < NA; ++a) {
            rg[a] = MODE == KM_CFR ? tabR[size_t(row) * NA + a] : 0.f;
            sr[a] = MODE != KM_BR ? tabS[size_t(row) * NA + a] : 0.f;
            sg[a] = fmaxf(MODE == KM_CFR ? rg[a] : sr[a], 0.f);
            norm += sg[a];
            d[a] = 0.f;
        }
        const float inv = norm > 0.f ? 1.0f / norm : 0.f;
#pragma unroll
        for (int a = 0; a < NA; ++a) sg[a] = norm > 0.f ? sg[a] * inv : 1.0f / float(NA);
        float msum = 0.f;
        const int hs = rstart[row], he = rstart[row + 1];
        for (int q = hs; q < he; ++q) {
            const int h = rpos[q];
            float va[NA];
            float vn = (MODE == KM_BR) ? -3.0e38f : 0.f;
#pragma unroll
            for (int a = 0; a < NA; ++a) {
                va[a] = V1[a * c.Hx + h];
                if (MODE == KM_BR) vn = fmaxf(vn, va[a]);
                else vn += sg[a] * va[a];
            }
            if (MODE == KM_CFR) {
#pragma unroll
                for (int a = 0; a < NA; ++a) d[a] += va[a] - vn;
                msum += M[h];
            }
            store_value1(c, nt, Rk, b, out, h, vn);
        }
        if (MODE == KM_CFR) {
            const float w = msum * scale;
#pragma unroll
            for (int a = 0; a < NA; ++a) {
                if (DR) {
                    tabR[size_t(row) * NA + a] = rule_regret(dr, rg[a], rg[a] > A.prune_threshold ? d[a] : 0.f);
                    tabS[size_t(row) * NA + a] = dr.z * sr[a] + sg[a] * w;
                } else {
                    tabR[size_t(row) * NA + a] = rg[a] + (rg[a] > A.prune_threshold ? d[a] : 0.f);
                    tabS[size_t(row) * NA + a] = sr[a] + sg[a] * w;
                }
            }
        }
    }
}

// wide nodes (more than FAST_ACTIONS actions): values in shared memory, dynamic loops over the actions
template <int HC, int MODE, bool DR>
__device__ __forceinline__ void task_trav_generic(const TaskArgs& A, const Ctx& c, const NodeTask& nt, const RoundArgs& Rk, int k, int b) {
    const DevRoundPlayer& Pp = Rk.rp[c.p];
    const float scale = Rk.chance_scale[b];
    float4 dr;
    if (DR) dr = rule_factors(A);
    const int n_act = nt.n_act;
    bool need_sd = false;
    for (int a = 0; a < n_act; ++a) {
        const int ck = nt.child[a].kind;
        if (ck == CK_VALUE && c.pos4 < c.HpP) *reinterpret_cast<float4*>(SM_X + (1 + a) * c.Hx + c.pos4) = child_value4(A, c, Rk, nt.child[a], b);
        need_sd |= (ck == CK_SHOWDOWN);
    }
    float4 mass, sd;
    trav_terms_or_load<HC>(A, c, nt, Rk, k, b, need_sd, mass, sd);
    float* out = (nt.root_scatter ? Rk.sbuf : Rk.cbuf) + (size_t(nt.out) * Rk.n_boards + b) * c.HpP;
    if (c.pos4 < c.HpP) {
        *reinterpret_cast<float4*>(SM_X + c.pos4) = mass;
        for (int a = 0; a < n_act; ++a) {
            const int ck = nt.child[a].kind;
            const float cf = nt.child[a].coef * scale;
            if (ck == CK_FOLD) *reinterpret_cast<float4*>(SM_X + (1 + a) * c.Hx + c.pos4) = make_float4(cf * mass.x, cf * mass.y, cf * mass.z, cf * mass.w);
            else if (ck == CK_SHOWDOWN) *reinterpret_cast<float4*>(SM_X + (1 + a) * c.Hx + c.pos4) = make_float4(cf * sd.x, cf * sd.y, cf * sd.z, cf * sd.w);
        }
        if (!nt.root_scatter) stcg4(out + c.pos4, f4zero());
    }
    csync(c.nc);
    const uint32_t nrp = Pp.n_rows_pad[b];
    const uint32_t n_rows = Pp.n_rows[b];
    float* tabR = Pp.regrets + Pp.board_off[b] + size_t(nrp) * nt.cum_a;
    float* tabS = Pp.ssum + Pp.board_off[b] + size_t(nrp) * nt.cum_a;
    const uint16_t* __restrict__ rstart = Pp.row_start + size_t(b) * (c.HpP + 4);
    const uint16_t* __restrict__ rpos = Pp.row_pos + size_t(b) * c.HpP;
    const float* M = SM_X;
    const float* V1 = SM_X + c.Hx;
    for (uint32_t row = c.tid; row < n_rows; row += c.nc) {
        const float* tsrc = (MODE == KM_EVAL ? tabS : tabR) + size_t(row) * n_act;
        float norm = 0.f;
        if (MODE != KM_BR)
            for (int a = 0; a < n_act; ++a) norm += fmaxf(tsrc[a], 0.f);
        const float inv = norm > 0.f ? 1.0f / norm : 0.f;
        const float uni = 1.0f / float(n_act);
        float msum = 0.f, vsum = 0.f;
        const int hs = rstart[row], he = rstart[row + 1];
        for (int q = hs; q < he; ++q) {
            const int h = rpos[q];
            float vn = (MODE == KM_BR) ? -3.0e38f : 0.f;
            for (int a = 0; a < n_act; ++a) {
                const float va = V1[a * c.Hx + h];
                if (MODE == KM_BR) vn = fmaxf(vn, va);
                else vn += (norm > 0.f ? fmaxf(tsrc[a], 0.f) * inv : uni) * va;
            }
            vsum += vn;
            msum += M[h];
            store_value1(c, nt, Rk, b, out, h, vn);
        }
        if (MODE == KM_CFR) {
            const float w = msum * scale;
            for (int a = 0; a < n_act; ++a) {
                float da = -vsum;
                for (int q = hs; q < he; ++q) da += V1[a * c.Hx + rpos[q]];
                const float old = tabR[size_t(row) * n_act + a];
                const float sga = norm > 0.f ? fmaxf(old, 0.f) * inv : uni;
                if (DR) {
                    tabS[size_t(row) * n_act + a] = dr.z * tabS[size_t(row) * n_act + a] + sga * w;
                    tabR[size_t(row) * n_act + a] = rule_regret(dr, old, old > A.prune_threshold ? da : 0.f);
                } else {
                    tabS[size_t(row) * n_act + a] += sga * w;
                    tabR[size_t(row) * n_act + a] = old + (old > A.prune_threshold ? da : 0.f);
                }
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// the persistent kernel
// ------------------------------------------------------------------------------------------------
// instance -> board.  Full traversal: the instance number IS the (local) board.  Sampled mode: round 0 keeps its
// boards, deeper rounds run on the sampled run-outs only.
__device__ __forceinline__ int board_of(const TaskArgs& A, int k, int inst) {
    return (k > 0 && A.sample_board[k] != nullptr) ? A.sample_board[k][inst] : inst;
}
// instance of the PARENT-round task that feeds instance `inst` of round k (flags are indexed by instance)
__device__ __forceinline__ int parent_instance(const TaskArgs& A, const RoundArgs& Rk, int k, int inst, int b) {
    if (A.sample_board[k] == nullptr) return Rk.parent_board[b];
    return k - 1 == 0 ? Rk.parent_board[b] : inst;  // path i of round k hangs off path i of round k-1
}

// pull the table slab(s) the NEXT task of this CTA will read into L2 while the current task runs
template <int MODE>
__device__ __forceinline__ void prefetch_task_tables(const TaskArgs& A, uint32_t tk, uint32_t j) {
    const NodeTask* g = A.tasks + j;
    const int kind = g->kind;
    if (kind != TK_DOWN && kind != TK_UP_TRAV) return;
    const RoundArgs& Rk = A.rounds[g->round_k];
    const int b = board_of(A, g->round_k, int(tk - g->first));
    const int q = kind == TK_DOWN ? 1 - A.trav : A.trav;
    const DevRoundPlayer& D = Rk.rp[q];
    const uint32_t nrp = D.n_rows_pad[b];
    const size_t off = D.board_off[b] + size_t(nrp) * g->cum_a;
    const uint32_t bytes = nrp * uint32_t(g->n_act) * 4u;
    if (kind == TK_DOWN) {
        prefetch_l2_bulk((MODE == KM_CFR ? D.regrets : D.ssum) + off, bytes);
    } else {
        if (MODE == KM_CFR) prefetch_l2_bulk(D.regrets + off, bytes);
        if (MODE != KM_BR) prefetch_l2_bulk(D.ssum + off, bytes);
    }
}

struct TaskSlot {
    uint32_t ticket;  // the instance slot (first slot of its node task + instance); >= t1: no more work
    uint32_t epoch;   // launch number: the value that marks flags "done" in this launch
    uint32_t xseq;    // ctl->xch_seq at launch: flag value and buffer parity of the in-kernel exchange
    uint32_t pad;
    NodeTask nt;
};

// KM: KM_CFR, KM_BR, KM_EVAL, or KM_CFR_DR (CFR with the update rule of TaskCtl::rule)
template <int KM, int MAXT, int MINB, bool XS>
__global__ void __launch_bounds__(MAXT + 32, MINB) task_kernel(const __grid_constant__ TaskArgs A) {
    constexpr bool DR = KM == KM_CFR_DR;
    constexpr int MODE = DR ? int(KM_CFR) : KM;
    constexpr int HC = 4 * MAXT;  // positions the shared-memory arrays hold
    __shared__ __align__(16) TaskSlot s_slot[2];

    __shared__ __align__(8) uint64_t s_done;  // phase i completes when every compute warp has finished task i

    const int NC = blockDim.x - 32;  // compute threads; the last warp is the dispatcher
    const int tid = threadIdx.x;
    if (tid == 0) mbar_init(&s_done, uint32_t(NC >> 5));
    if (tid < 2) SM_B[54 + tid] = SM_BF[54 + tid] = 0.f;  // boundaries of "a card the opponent does not hold" (HREC_K_NONE), never overwritten
    __syncthreads();

    if (tid >= NC) {
        // ---------------- dispatcher warp ----------------
        // Runs one task ahead of the compute warps: draws the ticket, finds the node-task, copies its descriptor to
        // shared memory, pulls its table slabs into L2 and polls the producers' flags.  While polling it keeps
        // testing the mbarrier and publishes the flag of the task the compute warps just finished the moment they
        // are done: a finished task is never held back by the look-ahead (that would deadlock across CTAs).
        const int lane = tid - NC;
        uint32_t epoch = 0, xseq = 0;
        if (lane == 0) {
            epoch = ld_acquire_u32(&A.ctl->epoch);
            xseq = *reinterpret_cast<const volatile unsigned int*>(&A.ctl->xch_seq);  // only written by the last CTA of a launch
        }
        epoch = __shfl_sync(0xffffffffu, epoch, 0);
        uint32_t prev_tk = 0xffffffffu, parity = 0;
        int buf = 0;
        // the ticket for the task prepared in iteration i was drawn in iteration i-1: its round trip is hidden
        uint32_t tk_next = 0;
        if (lane == 0) tk_next = A.t0 + uint32_t(atomicAdd(&A.ctl->ticket, 1ull));
        tk_next = __shfl_sync(0xffffffffu, tk_next, 0);
        for (;;) {
            bool published = (prev_tk == 0xffffffffu);  // meaningful on lane 0
            auto try_publish = [&]() {
                if (lane == 0 && !published && mbar_test(&s_done, parity)) {
#ifndef RS_NO_PUBLISH_FENCE
                    __threadfence();
#endif
                    st_release_u32(A.flags + prev_tk, epoch);
                    published = true;
                }
            };
            uint32_t tk = tk_next;
            uint32_t sl = A.t1;  // the instance slot this ticket stands for (flags, descriptors and instances go by slot)
            if (tk < A.t1) {
                unsigned long long pend = 0;
                if (lane == 0) pend = atomicAdd(&A.ctl->ticket, 1ull);  // consumed at the end of this iteration
                sl = A.order ? __ldg(A.order + tk) : tk;
                const uint32_t j = __ldg(A.task_of_ticket + sl);
                const NodeTask* gt = A.tasks + j;
                NodeTask& st = s_slot[buf].nt;
                for (int i = lane; i < int(sizeof(NodeTask) / 4); i += 32)
                    reinterpret_cast<uint32_t*>(&st)[i] = __ldg(reinterpret_cast<const uint32_t*>(gt) + i);
                __syncwarp();
                const int kind = st.kind;
                const int k = st.round_k;
                const int inst = int(sl - st.first);
                const int b = board_of(A, k, inst);
                const RoundArgs& Rk = A.rounds[k];
                const int nd = st.n_dep;
                const bool sampled = A.sample_board[1] != nullptr;
                int total;
                uint32_t gfirst = 0;
                if (kind == TK_GATHER) {
                    if (sampled) {  // children = the sampled paths: all of them below the root board, else this path's own
                        gfirst = uint32_t(st.dep[0]) + uint32_t(k == 0 ? 0 : inst);
                        total = k == 0 ? A.n_paths : 1;
                    } else {
                        gfirst = uint32_t(st.dep[0]) + uint32_t(Rk.per_parent > 0 ? b * Rk.per_parent : 0);
                        total = Rk.per_parent > 0 ? Rk.per_parent : Rk.n_boards_next;
                    }
                } else {
                    total = nd + st.n_src_all;
                }
                // each lane resolves the flag index of its first producer now (loads overlap the prefetch setup)
                auto flag_index = [&](int i, bool& has) -> uint32_t {
                    has = true;
                    if (kind == TK_GATHER) return gfirst + uint32_t(i);
                    int dfirst, dk = DK_SAME_BOARD;
                    if (i < nd) {
                        dfirst = st.dep[i];
                        dk = st.dep_kind[i];
                    } else {
                        dfirst = __ldg(&A.srcs[st.src_all_first + (i - nd)].dep);
                    }
                    has = dfirst >= 0;
                    return uint32_t(dfirst) + uint32_t(dk == DK_PARENT_BOARD ? parent_instance(A, Rk, k, inst, b) : inst);
                };
                int i = lane;
                bool has = false;
                uint32_t idx = 0;
                if (i < total) idx = flag_index(i, has);
                if (lane == 0) prefetch_task_tables<MODE>(A, sl, j);
                // the vectors the task will read (value sources, same-round reach), when a large round pushed them out of L2
                // (config 4: +2 %; streaming cache hints on the table traffic instead measured -7 %)
                if (kind == TK_UP_TRAV || kind == TK_UP_OPP)
                    for (int q = lane; q < int(st.n_src_all); q += 32) {
                        const TaskSrc sr = A.srcs[st.src_all_first + q];
                        prefetch_l2_bulk((sr.kind == SK_CBUF ? Rk.cbuf : Rk.gathered) + (size_t(sr.buf) * Rk.n_boards + b) * A.HpP, uint32_t(A.HpP) * 4u);
                    }
                if (lane == 1 && st.r_in != RIN_INITIAL && !st.rin_parent_round && (kind == TK_DOWN || kind == TK_TRAV_TERMS || (kind == TK_UP_TRAV && !st.pre_terms)))
                    prefetch_l2_bulk(Rk.rbuf + (size_t(st.r_in) * Rk.n_boards + b) * A.HoP, uint32_t(A.HoP) * 4u);
                try_publish();
                (void)b;
                const unsigned long long t_wait = global_ns();
                uint32_t spins = 0;
                bool gave_up = false;
                for (;;) {  // one flag test per lane per round
                    if (i < total) {
                        if (!has || idx < A.t0 || ld_acquire_u32(A.flags + idx) == epoch) {
                            i += 32;
                            if (i < total) idx = flag_index(i, has);
                        }
                    }
                    try_publish();
                    if (__all_sync(0xffffffffu, i >= total)) break;
                    __nanosleep(RS_POLL_SLEEP_NS);
                    if (__any_sync(0xffffffffu, lane == 0 && wait_gives_up(A, t_wait, spins))) {
                        gave_up = true;
                        break;
                    }
                }
                tk_next = A.t0 + uint32_t(__shfl_sync(0xffffffffu, pend, 0));
                if (gave_up) tk = tk_next = sl = A.t1;  // hand the compute warps the end marker: the producers will never finish
            }
            if (lane == 0) {
                s_slot[buf].ticket = sl;
                s_slot[buf].epoch = epoch;
                s_slot[buf].xseq = xseq;
            }
            __syncwarp();
            hsync(NC + 32);  // slot[buf] handed over; the compute warps are done with the previous task
            if (lane == 0 && !published) {
#ifndef RS_NO_PUBLISH_FENCE
                __threadfence();
#endif
                st_release_u32(A.flags + prev_tk, epoch);
            }
            if (prev_tk != 0xffffffffu) parity ^= 1;
            if (tk >= A.t1) break;
            prev_tk = sl;
            buf ^= 1;
        }
        // the last CTA to leave re-arms the dispatcher state for the next launch
        if (lane == 0) {
            __threadfence();
            const unsigned int e = atomicAdd(&A.ctl->exited, 1u);
            if (e == gridDim.x - 1) {
                A.ctl->ticket = 0ull;
                A.ctl->exited = 0u;
                if (A.xch_bump) A.ctl->xch_seq = xseq + 1;
                __threadfence();
                st_release_u32(&A.ctl->epoch, epoch + 1);
            }
        }
        return;
    }

    // ---------------- compute warps ----------------
    Ctx c;
    c.nc = NC;
    c.tid = tid;
    c.lane = tid & 31;
    c.warp = tid >> 5;
    c.nwarps = NC >> 5;
    c.pos4 = 4 * tid;
    c.p = A.trav;
    c.o = 1 - c.p;
    c.Hp = A.H[c.p];
    c.Ho = A.H[c.o];
    c.HpP = A.HpP;
    c.HoP = A.HoP;
    c.Hx = A.Hx;

    int buf = 0;
    for (;;) {
        hsync(NC + 32);
        const uint32_t t = s_slot[buf].ticket;
        if (t >= A.t1) break;
        const NodeTask& nt = s_slot[buf].nt;
        const int kind = nt.kind;
        const int k = nt.round_k;
        const int inst = int(t - nt.first);
        const int b = board_of(A, k, inst);
        const RoundArgs& Rk = A.rounds[k];
#ifdef RS_TASK_TIMING
        const long long tm1 = clock64();
        if (tid == 0 && A.timing) {
            unsigned long long gt0;
            asm volatile("mov.u64 %0, %globaltimer;" : "=l"(gt0));
            atomicMin(A.timing + 32 + (kind * 3 + k) * 2, gt0);
        }
#endif
        switch (kind) {
            case TK_DOWN: {
                switch (nt.n_act) {
                    case 2: task_down<HC, MODE, 2, XS>(A, c, nt, Rk, k, b); break;
                    case 3: task_down<HC, MODE, 3, XS>(A, c, nt, Rk, k, b); break;
                    case 4: task_down<HC, MODE, 4, XS>(A, c, nt, Rk, k, b); break;
                    case 5: task_down<HC, MODE, 5, XS>(A, c, nt, Rk, k, b); break;
                    default: task_down_generic<HC, MODE, XS>(A, c, nt, Rk, k, b); break;
                }
                break;
            }
            case TK_UP_TRAV: {
                switch (nt.n_act) {
                    case 2: task_trav<HC, MODE, 2, DR>(A, c, nt, Rk, k, b); break;
                    case 3: task_trav<HC, MODE, 3, DR>(A, c, nt, Rk, k, b); break;
                    case 4: task_trav<HC, MODE, 4, DR>(A, c, nt, Rk, k, b); break;
                    case 5: task_trav<HC, MODE, 5, DR>(A, c, nt, Rk, k, b); break;
                    default: task_trav_generic<HC, MODE, DR>(A, c, nt, Rk, k, b); break;
                }
                break;
            }
            case TK_UP_OPP: {  // opponent node at a street root: terminal partial + children (sigma is inside the reach)
                if (c.pos4 < c.HpP) {
                    float4 v = nt.aux >= 0 ? ldcg4(Rk.cbuf + (size_t(nt.aux) * Rk.n_boards + b) * c.HpP + c.pos4) : f4zero();
                    for (int a = 0; a < nt.n_act; ++a)
                        if (nt.child[a].kind == CK_VALUE) v = f4add(v, child_value4(A, c, Rk, nt.child[a], b));
                    store_value4(c, nt, Rk, b, (nt.root_scatter ? Rk.sbuf : Rk.cbuf) + (size_t(nt.out) * Rk.n_boards + b) * c.HpP, v);
                }
                break;
            }
            case TK_GATHER: {  // cfr.rs:502-522: sum over the dealt cards, fixed board order
                if (c.pos4 < c.HpP) {
                    const RoundArgs& Rn = A.rounds[k + 1];
                    // the child-street roots stored their values in THIS board's hand order (store_value4)
                    const float* base = Rn.sbuf + size_t(nt.aux) * Rn.n_boards * c.HpP + c.pos4;
                    float4 acc = f4zero();
                    if (A.sample_board[k + 1] != nullptr) {
                        // sampled run-outs (generate_hand, cfr.rs:100-143): uniform sampling of the next card, weight
                        // = (#possible deals) / (#sampled children)
                        const int32_t* sb = A.sample_board[k + 1];
                        const int s0 = k == 0 ? 0 : inst, ns = k == 0 ? A.n_paths : 1;
                        for (int i = 0; i < ns; ++i) acc = f4add(acc, ldcg4(base + size_t(sb[s0 + i]) * c.HpP));
                        const float w = A.gather_scale[k];
                        acc = make_float4(acc.x * w, acc.y * w, acc.z * w, acc.w * w);
                    } else {
                        const int cb0 = Rk.per_parent > 0 ? b * Rk.per_parent : 0;
                        const int ncb = Rk.per_parent > 0 ? Rk.per_parent : Rk.n_boards_next;
                        const float* src = base + size_t(cb0) * c.HpP;
                        for (int i0 = 0; i0 < ncb; i0 += 8) {  // eight loads in flight; summation order = board order
                            float4 val[8];
#pragma unroll
                            for (int u = 0; u < 8; ++u) val[u] = (i0 + u < ncb) ? ldcg4(src + size_t(i0 + u) * c.HpP) : f4zero();
#pragma unroll
                            for (int u = 0; u < 8; ++u) acc = f4add(acc, val[u]);
                        }
                    }
                    stcg4(Rk.gathered + (size_t(nt.out) * Rk.n_boards + b) * c.HpP + c.pos4, acc);
                }
                if (A.xch_world > 1 && k + 1 == A.xch_round) {
                    // Board-sharded traversal: the sum above only covers this GPU's boards.  Every rank writes its
                    // partial vector straight into the peers' exchange buffers (NVLink stores), raises one flag per
                    // peer, waits for the partials of all ranks to land in its own buffer and adds them up in rank
                    // order (bit-identical on every GPU).  This is the one exchange step of the path, inside the
                    // traversal kernel: no second launch, no NCCL call.  Buffers alternate with the parity of the exchange
                    // sequence number (TaskCtl::xch_seq, the same on every rank): a rank can be at most one traversal ahead
                    // of a peer that still reads.
                    const uint32_t ep = s_slot[buf].xseq;
                    const size_t vec = ((size_t(ep & 1u) * A.xch_leaves + nt.out) * Rk.n_boards + b) * A.xch_world;
                    if (c.pos4 < c.HpP) {
                        const float4 part = ldcg4(Rk.gathered + (size_t(nt.out) * Rk.n_boards + b) * c.HpP + c.pos4);
                        for (int peer = 0; peer < A.xch_world; ++peer)
                            *reinterpret_cast<float4*>(A.xch_peer[peer] + (vec + A.xch_rank) * c.HpP + c.pos4) = part;
                    }
                    __threadfence_system();
                    csync(c.nc);
                    if (tid < A.xch_world) {
                        st_release_sys_u32(A.xflag_peer[tid] + vec + A.xch_rank, ep);
                        const uint32_t* mine = A.xflag_peer[A.xch_rank] + vec + tid;
                        const unsigned long long t_wait = global_ns();
                        uint32_t spins = 0;
                        while (ld_acquire_sys_u32(mine) != ep) {  // a peer that never launches: bounded, see wait_gives_up
                            __nanosleep(100);
                            spins += 31;  // this loop sleeps longer than the dispatcher's: look at the clock every 8th round
                            if (wait_gives_up(A, t_wait, spins)) break;
                        }
                    }
                    csync(c.nc);
                    if (c.pos4 < c.HpP) {
                        const float* src = A.xch_peer[A.xch_rank] + vec * c.HpP + c.pos4;
                        float4 acc = f4zero();
                        for (int r = 0; r < A.xch_world; ++r) acc = f4add(acc, ldcg4(src + size_t(r) * c.HpP));
                        stcg4(Rk.gathered + (size_t(nt.out) * Rk.n_boards + b) * c.HpP + c.pos4, acc);
                    }
                }
                break;
            }
            case TK_TRAV_TERMS: {  // chain rounds: the reach-only part of a traverser node, ahead of its children
                bool need_sd = false;
                for (int a = 0; a < nt.n_act; ++a) need_sd |= (nt.child[a].kind == CK_SHOWDOWN);
                float4 mass, sd;
                trav_terms<HC>(A, c, nt, Rk, k, b, need_sd, mass, sd);
                if (c.pos4 < c.HpP) {
                    float* m = Rk.cbuf + (size_t(nt.out) * Rk.n_boards + b) * c.HpP + c.pos4;
                    stcg4(m, mass);
                    stcg4(m + size_t(Rk.n_boards) * c.HpP, sd);
                }
                break;
            }
            case TK_ROOT_SHOWDOWN: {
                float4 mass, sd;
                trav_terms<HC>(A, c, nt, Rk, k, b, true, mass, sd);
                const float cf = nt.child[0].coef * Rk.chance_scale[b];
                if (c.pos4 < c.HpP)
                    store_value4(c, nt, Rk, b, (nt.root_scatter ? Rk.sbuf : Rk.cbuf) + (size_t(nt.out) * Rk.n_boards + b) * c.HpP,
                                 make_float4(cf * sd.x, cf * sd.y, cf * sd.z, cf * sd.w));
                break;
            }
            case TK_CHANCE_DOWN: {
                const float4 r4 = load_reach4(A, c, nt, Rk, k, b);
                if (c.pos4 < c.HoP) stcg4(Rk.rbuf + (size_t(nt.aux) * Rk.n_boards + b) * c.HoP + c.pos4, r4);
                break;
            }
            case TK_CHANCE_UP: {
                if (c.pos4 < c.HpP)
                    store_value4(c, nt, Rk, b, (nt.root_scatter ? Rk.sbuf : Rk.cbuf) + (size_t(nt.out) * Rk.n_boards + b) * c.HpP,
                                 ldcg4(Rk.gathered + (size_t(nt.aux) * Rk.n_boards + b) * c.HpP + c.pos4));
                break;
            }
            default: break;
        }
#ifdef RS_TASK_TIMING
        if (tid == 0 && A.timing) {
            atomicAdd(A.timing + kind * 4 + 0, 1ull);
            atomicAdd(A.timing + kind * 4 + 2, (unsigned long long)(clock64() - tm1));  // body
            unsigned long long gt1;
            asm volatile("mov.u64 %0, %globaltimer;" : "=l"(gt1));
            atomicMax(A.timing + 32 + (kind * 3 + k) * 2 + 1, gt1);
        }
#endif
        __syncwarp();
        if (c.lane == 0) mbar_arrive(&s_done);  // this warp's part of the task is written
        buf ^= 1;
    }
}

__global__ void scale_kernel(float* __restrict__ data, size_t n, float d) {
    const size_t n4 = n / 4;
    float4* v4 = reinterpret_cast<float4*>(data);
    const size_t stride = size_t(gridDim.x) * blockDim.x;
    for (size_t i = size_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n4; i += stride) {
        float4 v = v4[i];
        v.x *= d;
        v.y *= d;
        v.z *= d;
        v.w *= d;
        v4[i] = v;
    }
    if (blockIdx.x == 0 && threadIdx.x < n - n4 * 4) data[n4 * 4 + threadIdx.x] *= d;
}

__global__ void set_rule_kernel(TaskCtl* ctl, float4 f) { *reinterpret_cast<float4*>(ctl->rule) = f; }

__global__ void normalize_kernel(const float* __restrict__ in, float* __restrict__ out, uint32_t n_rows, uint32_t A) {
    const uint32_t row = blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= n_rows) return;
    float norm = 0.f;
    for (uint32_t a = 0; a < A; ++a) norm += fmaxf(in[size_t(row) * A + a], 0.f);
    for (uint32_t a = 0; a < A; ++a)
        out[size_t(row) * A + a] = norm > 0.f ? fmaxf(in[size_t(row) * A + a], 0.f) / norm : 1.0f / float(A);
}

__global__ void unpermute_kernel(const float* __restrict__ in, const uint16_t* __restrict__ slot_of_pos, const uint32_t* __restrict__ n_live,
                                 float* __restrict__ out, uint32_t hp, uint32_t H) {
    const uint32_t b = blockIdx.y;
    const uint32_t pos = blockIdx.x * blockDim.x + threadIdx.x;
    if (pos < n_live[b]) out[size_t(b) * H + slot_of_pos[size_t(b) * hp + pos]] = in[size_t(b) * hp + pos];
}

}  // namespace

size_t task_kernel_smem_bytes(bool wide, int slots, int Hp_pad, int Ho_pad) {
    const int hx = Hp_pad > Ho_pad ? Hp_pad : Ho_pad;
    const int hc = 4 * (wide ? 352 : 288);  // HC of the build launch_task_kernel picks
    size_t floats = size_t(smem_fixed_floats(hc)) + size_t(slots) * hx;  // fixed-offset arrays (SM_*), then the scratch vectors
    return floats * sizeof(float);
}

template <int MAXT, int MINB>
static cudaError_t configure_for(size_t smem, int threads, int* blocks_per_sm) {
    cudaError_t e;
    e = cudaFuncSetAttribute(task_kernel<KM_CFR, MAXT, MINB, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(task_kernel<KM_CFR, MAXT, MINB, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(task_kernel<KM_CFR_DR, MAXT, MINB, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(task_kernel<KM_CFR_DR, MAXT, MINB, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(task_kernel<KM_BR, MAXT, MINB, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(task_kernel<KM_EVAL, MAXT, MINB, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
    if (e != cudaSuccess) return e;
    int n = 0, m = 0, x = 0;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, task_kernel<KM_CFR, MAXT, MINB, false>, threads + 32, smem);
    if (e != cudaSuccess) return e;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&m, task_kernel<KM_BR, MAXT, MINB, false>, threads + 32, smem);
    if (e != cudaSuccess) return e;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&x, task_kernel<KM_CFR, MAXT, MINB, true>, threads + 32, smem);
    if (e != cudaSuccess) return e;
    n = n < x ? n : x;
    *blocks_per_sm = n < m ? n : m;
    return cudaSuccess;
}

cudaError_t configure_task_kernels(size_t smem, int threads, bool wide, int* blocks_per_sm) {
    if (threads <= 288 && !wide) return configure_for<288, RS_MIN_BLOCKS_288>(smem, threads, blocks_per_sm);
    return configure_for<352, RS_MIN_BLOCKS_352>(smem, threads, blocks_per_sm);
}

template <int MAXT, int MINB>
static void launch_for(const TaskArgs& a, int mode, int grid, int threads, size_t smem, cudaStream_t st) {
    switch (mode) {
        // one extra warp per CTA: the dispatcher
        case KM_CFR: task_kernel<KM_CFR, MAXT, MINB, false><<<grid, threads + 32, smem, st>>>(a); break;
        case KM_CFR_XS: task_kernel<KM_CFR, MAXT, MINB, true><<<grid, threads + 32, smem, st>>>(a); break;
        case KM_CFR_DR: task_kernel<KM_CFR_DR, MAXT, MINB, false><<<grid, threads + 32, smem, st>>>(a); break;
        case KM_CFR_XS_DR: task_kernel<KM_CFR_DR, MAXT, MINB, true><<<grid, threads + 32, smem, st>>>(a); break;
        case KM_BR: task_kernel<KM_BR, MAXT, MINB, false><<<grid, threads + 32, smem, st>>>(a); break;
        default: task_kernel<KM_EVAL, MAXT, MINB, false><<<grid, threads + 32, smem, st>>>(a); break;
    }
}

cudaError_t launch_task_kernel(const TaskArgs& a, int mode, int grid, int threads, bool wide, size_t smem, cudaStream_t st) {
    if (grid <= 0 || a.t1 <= a.t0) return cudaSuccess;
    if (threads <= 288 && !wide) launch_for<288, RS_MIN_BLOCKS_288>(a, mode, grid, threads, smem, st);
    else launch_for<352, RS_MIN_BLOCKS_352>(a, mode, grid, threads, smem, st);
    return cudaGetLastError();
}

cudaError_t launch_scale(float* data, size_t n, float d, cudaStream_t st) {
    if (n == 0) return cudaSuccess;
    const int threads = 256;
    size_t blocks = (n / 4 + threads - 1) / threads;
    if (blocks < 1) blocks = 1;
    if (blocks > 148 * 16) blocks = 148 * 16;
    scale_kernel<<<unsigned(blocks), threads, 0, st>>>(data, n, d);
    return cudaGetLastError();
}

cudaError_t launch_set_rule(TaskCtl* ctl, const float f[4], cudaStream_t st) {
    set_rule_kernel<<<1, 1, 0, st>>>(ctl, make_float4(f[0], f[1], f[2], f[3]));
    return cudaGetLastError();
}

cudaError_t launch_unpermute(const float* in, const uint16_t* slot_of_pos, const uint32_t* n_live, float* out, uint32_t n_boards, uint32_t hp,
                             uint32_t H, cudaStream_t st) {
    if (n_boards == 0) return cudaSuccess;
    unpermute_kernel<<<dim3((hp + 255) / 256, n_boards), 256, 0, st>>>(in, slot_of_pos, n_live, out, hp, H);
    return cudaGetLastError();
}

cudaError_t launch_normalize(const float* in, float* out, uint32_t n_rows, uint32_t A, cudaStream_t st) {
    if (n_rows == 0) return cudaSuccess;
    normalize_kernel<<<(n_rows + 255) / 256, 256, 0, st>>>(in, out, n_rows, A);
    return cudaGetLastError();
}

}  // namespace rs
