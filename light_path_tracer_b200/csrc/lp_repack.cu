// lp_repack.cu — the fused frame kernel with LANE RE-PACKING (north star item 1: "warp-ballot /
// shuffle ray compaction, or persistent-thread re-packing, so rays that have escaped or been
// captured stop wasting lanes near the photon sphere").  Same per-ray arithmetic as
// lp_render_kernel (lp_trace.cu) — binet_init, rk4_step, binet_cross, binet_finish, remap_pixel
// are the shared device functions — so the frame is bit-identical; only the schedule differs.
// Replaces the same reference lines: metrics.py:49-145 / :661-668 behind image_lens.py:133-178,
// :296-397.
//
// Schedule.  A warp owns LP_RP_CHUNK (256) consecutive pixels of its tile and streams them
// through its 32 lanes:
//   * prepare: when the warp's in-queue is empty and a lane is idle, ALL 32 lanes compute the
//     per-ray head (pixel -> alpha(f32) -> sin -> b -> w0) of the next 32 pixels together and
//     push them to the in-queue (shared memory);
//   * loop: every lane that holds a ray runs one trip of four RK4 steps; a lane whose ray left
//     the band pushes the raw exit state (u_prev, w_prev, u, w, step) to the warp's out-queue
//     and, in the same trip, pops the next prepared ray — ballot + popc ranks, no atomics;
//   * finish: whenever 32 exit states have gathered, ALL 32 lanes run the per-ray tail together
//     (crossing interpolation, final direction, remap, source gather) and put the pixel into the
//     chunk's staging tile in shared memory;
//   * write-out: the finished chunk leaves as 16-byte vector stores (full sectors — the tile may
//     live in a peer GPU's memory, dist.PeerFrame).
// The divergent phases of the one-ray-per-thread kernel (head and tail run by whichever lanes
// happen to be there) become convergent, and the loop never runs with idle lanes except while a
// chunk drains (<= 1/8 of the rays of a chunk can be in that phase).
//
// No global state, no device-side allocation: the chunk -> warp assignment is static
// (blockIdx), CTAs are small (64 threads = 2 chunks) and back-filled by the hardware work
// distributor exactly like lp_render_kernel's.
#include "lp_trace.cuh"

#define LP_RP_CHUNK 256
#define LP_RP_BLOCK 64
#define LP_RP_WARPS (LP_RP_BLOCK / 32)
#define LP_RP_OUTQ 64

enum { RP_INVALID = 0, RP_ESCAPE = 1, RP_CAPTURE = 2, RP_RANOUT = 3 };

// per-warp queues (structure of arrays: conflict-free for lane-consecutive slots)
struct RpQueues {
    double in_w0[32];
    int in_pix[32];
    float in_a32[32];
    double out_up[LP_RP_OUTQ], out_wp[LP_RP_OUTQ], out_u[LP_RP_OUTQ], out_w[LP_RP_OUTQ];
    int out_pix[LP_RP_OUTQ];
    float out_a32[LP_RP_OUTQ];
    int out_k[LP_RP_OUTQ];       // step index of the exit step (RP_RANOUT: steps done so far)
    int out_code[LP_RP_OUTQ];
    int out_tail;                // entries in the out-queue (slots are claimed with a shared-memory atomic)
    int pad_[3];
};

// The per-ray tail for one queue entry: what binet_trace_fast does after its loop.
template <bool FUSED>
__device__ __forceinline__ void rp_finish_ray(const BinetConsts &c, const LoopRegs &L, int code, int k,
                                              double up, double wp, double u, double w, double alpha,
                                              int retrace_steps, int retrace_steps_small, float retrace_h, float retrace_off, RayResult &r)
{
    if (code == RP_INVALID) {
        r.status = 0; r.nh = 0; r.steps = 0; r.fa = __longlong_as_double(0x7ff8000000000000LL);
        return;
    }
    int status = 2;
    double phi;
    if (code == RP_RANOUT) {
        // cold path (a ray that reaches phi_max): the remaining full steps one at a time, then the
        // shortened last steps — metrics.py:72-115 as in binet_trace_fast
        const double M3 = L.M3, h = L.h, hh = L.hh, h6 = L.h6;
        bool crossed = false;
        double u1, w1;
        for (; k < L.n_full; ++k) {
            rk4_full_step<FUSED>(L, u, w, u1, w1);
            if (u1 >= band_hi<FUSED>(c)) { status = -1; crossed = true; }
            else if (u1 <= band_lo<FUSED>(c)) { status = 1; crossed = true; }
            if (crossed) { up = u; wp = w; u = u1; w = w1; break; }
            u = u1; w = w1;
        }
        if (crossed) {
            r.steps = k + 1;
            binet_cross_s<FUSED>(c, status == -1, h, binet_phi_at<FUSED>(c, k), up, wp, u, w, phi);
        } else {
            r.steps = L.n_full;
            phi = c.phi_end;
            for (int j = 0; j < c.n_tail; ++j) {
                const double hj = c.tail_h[j];
                up = u; wp = w;
                rk4_step<FUSED>(up, wp, M3, hj, mul_(0.5, hj), __ddiv_rn(hj, 6.0), u, w);
                r.steps++;
                if (u >= band_hi<FUSED>(c)) { status = -1; binet_cross_s<FUSED>(c, true, hj, c.tail_phi[j], up, wp, u, w, phi); break; }
                if (u <= band_lo<FUSED>(c)) { status = 1; binet_cross_s<FUSED>(c, false, hj, c.tail_phi[j], up, wp, u, w, phi); break; }
            }
            if (status == 2) binet_scale_out<FUSED>(c, u, w);
        }
    } else {
        const bool cap = (code == RP_CAPTURE);
        status = cap ? -1 : 1;
        r.steps = k + 1;
        binet_cross_s<FUSED>(c, cap, L.h, binet_phi_at<FUSED>(c, k), up, wp, u, w, phi);
    }
    binet_finish<FUSED>(c, status, phi, u, w, r);
    if (FUSED && hybrid_needs_retrace(r, retrace_steps, retrace_steps_small, retrace_h, retrace_off))
        binet_trace<false, true>(c, load_loop_regs<false>(c), alpha, r);     // LP_TRACE_HYBRID
}

// per-warp frame statistics (shared memory; filled by warp reductions in the finish phase so that
// no accumulator lives in registers across the RK4 loop)
struct RpStats {
    unsigned long long sum_steps, min_fa, max_fa;     // min/max as ordered bit patterns (dbl_to_ordered)
    unsigned int n_rays, escaped, captured, invalid, winding, max_steps, max_winding, trips;
};

template <bool FUSED, typename T, int MINB>
__global__ void __launch_bounds__(LP_RP_BLOCK, MINB)
lp_render_repack_kernel(const TraceArgs a, const RemapArgs ra, const BinetConsts c, const CamConsts cam,
                        const int refill_min)
{
    extern __shared__ __align__(16) unsigned char rp_smem[];
    __shared__ RpStats rp_stats[LP_RP_WARPS];
    const LoopRegs L = load_loop_regs<FUSED>(c);
    const int lane = threadIdx.x & 31, wrp = threadIdx.x >> 5;
    const unsigned full = 0xffffffffu;
    const unsigned lt_mask = (1u << lane) - 1u;
    const int C = ra.channels;
    const size_t stage_bytes = ((size_t)LP_RP_CHUNK * C * sizeof(T) + 15) & ~(size_t)15;
    RpQueues &q = *reinterpret_cast<RpQueues *>(rp_smem + (size_t)wrp * (sizeof(RpQueues) + stage_bytes));
    T *stage = reinterpret_cast<T *>(rp_smem + (size_t)wrp * (sizeof(RpQueues) + stage_bytes) + sizeof(RpQueues));
    RpStats &ws = rp_stats[wrp];
    if (lane == 0) {
        q.out_tail = 0;
        ws.sum_steps = 0ull; ws.min_fa = ~0ull; ws.max_fa = 0ull;
        ws.n_rays = ws.escaped = ws.captured = ws.invalid = ws.winding = ws.max_steps = ws.max_winding = ws.trips = 0u;
    }
    __syncwarp();

    const long long chunk0 = ((long long)blockIdx.x * LP_RP_WARPS + wrp) * LP_RP_CHUNK;   // first pixel of the chunk
    const int n_chunk = (int)min((long long)LP_RP_CHUNK, a.n - chunk0);                  // <= 0: nothing to do
    const int n_batches = n_chunk > 0 ? (n_chunk + 31) / 32 : 0;

    // lane state.  code: -2 no ray, -1 integrating
    int code = -2;
    double u = 0.0, w = 0.0;
    int k = 0, pix = 0;
    float a32 = 0.0f;
    // warp-uniform queue state (every lane derives the same values from ballots)
    int in_head = 0, in_count = 0, out_count = 0, next_batch = 0;

    const double M3 = L.M3, h = L.h, hh = L.hh, h6 = L.h6;
    const unsigned lo_hi = L.lo_hi, span = L.span;
    const int n_full = L.n_full;
    const double b_hi = band_hi<FUSED>(c), b_lo = band_lo<FUSED>(c);

    // Each phase appears ONCE in the code (the kernel is instruction-cache sensitive: the finish
    // phase with its strict re-trace is ~5 k instructions).  Capacity of the out-queue: exit
    // states are pushed (<= 32 at a time) and invalid rays prepared (<= 32) only while fewer than
    // 32 are queued -> never more than 63 of 64.
    while (true) {
        // ---- finish: 32 gathered exit states, or whatever is left when the chunk has drained ----
        const bool rays_left = in_count > 0 || next_batch < n_batches;
        const bool any_ray = __ballot_sync(full, code != -2) != 0u;
        if (out_count >= 32 || (!rays_left && !any_ray && out_count > 0)) {
            const int cnt = min(out_count, 32);
            const int e = out_count - cnt + lane;
            const bool mine = lane < cnt;
            RayResult r;
            r.status = 0; r.steps = 0; r.nh = 0; r.fa = 0.0;
            if (mine) {
                const int p = q.out_pix[e];
                const float al = q.out_a32[e];
                rp_finish_ray<FUSED>(c, L, q.out_code[e], q.out_k[e], q.out_up[e], q.out_wp[e], q.out_u[e], q.out_w[e],
                                     (double)al, a.retrace_steps, a.retrace_steps_small, a.retrace_h, a.retrace_off, r);
                const long long i = chunk0 + p;
                int row, col;
                long long oi;
                tile_pixel(a, cam.width, i, row, col, oi);
                const float fa32 = (float)((r.status == 1) ? r.fa : __longlong_as_double(0x7ff8000000000000LL));
                const long long nh = r.nh < 0 ? 0 : (r.nh > 65535 ? 65535 : r.nh);
                if (a.out_fa) ((float *)a.out_fa)[i] = fa32;
                if (a.out_w) ((unsigned short *)a.out_w)[i] = (unsigned short)nh;
                remap_pixel_xy<T, true>(ra, cam, stage + (size_t)p * C, cam_x(cam, col), cam_y(cam, row), fa32, (unsigned)nh,
                                        r.fa, r.cf, r.sf);
            }
            if (a.stats) {
                const unsigned st = mine ? (unsigned)r.steps : 0u;
                const unsigned nhc = mine ? (unsigned)(r.nh < 0 ? 0 : (r.nh > 65535 ? 65535 : r.nh)) : 0u;
                const bool esc = mine && r.status == 1;
                const unsigned s_sum = __reduce_add_sync(full, st), s_max = __reduce_max_sync(full, st);
                const unsigned w_max = __reduce_max_sync(full, nhc);
                const unsigned n_esc = __popc(__ballot_sync(full, esc));
                const unsigned n_cap = __popc(__ballot_sync(full, mine && r.status == -1));
                const unsigned n_inv = __popc(__ballot_sync(full, mine && r.status == 0));
                const unsigned n_win = __popc(__ballot_sync(full, esc && (float)r.fa > LP_HALF_PI_F32));
                unsigned long long mn = (esc && r.fa == r.fa) ? dbl_to_ordered(r.fa) : ~0ull;
                unsigned long long mx = (esc && r.fa == r.fa) ? dbl_to_ordered(r.fa) : 0ull;
                for (int off = 16; off > 0; off >>= 1) {
                    mn = min(mn, __shfl_xor_sync(full, mn, off));
                    mx = max(mx, __shfl_xor_sync(full, mx, off));
                }
                if (lane == 0) {
                    ws.sum_steps += s_sum; ws.max_steps = max(ws.max_steps, s_max);
                    ws.max_winding = max(ws.max_winding, w_max);
                    ws.n_rays += (unsigned)cnt; ws.escaped += n_esc; ws.captured += n_cap; ws.invalid += n_inv;
                    ws.winding += n_win; ws.min_fa = min(ws.min_fa, mn); ws.max_fa = max(ws.max_fa, mx);
                }
            }
            out_count -= cnt;
            if (lane == 0) q.out_tail = out_count;
            __syncwarp();
            continue;
        }
        if (!rays_left && !any_ray) break;

        // ---- refill: lanes without a ray pop prepared rays; prepare the next 32 pixels when none are left ----
        const unsigned need = __ballot_sync(full, code == -2);
        if (need && rays_left) {
            if (in_count == 0) {
                // per-ray head of batch `next_batch`, all lanes together
                const int p = next_batch * 32 + lane;
                next_batch++;
                bool valid = false;
                const bool live = p < n_chunk;
                double w0 = 0.0, uu;
                float al = 0.0f;
                if (live) {
                    int row, col;
                    long long oi;
                    tile_pixel(a, cam.width, chunk0 + p, row, col, oi);
                    al = (float)pixel_alpha64(cam, cam_x(cam, col), cam_y(cam, row));
                    valid = binet_init<FUSED>(c, (double)al, uu, w0);
                }
                const unsigned vm = __ballot_sync(full, valid);
                const unsigned im = __ballot_sync(full, live && !valid);
                if (valid) {
                    const int s = __popc(vm & lt_mask);
                    q.in_w0[s] = w0; q.in_pix[s] = p; q.in_a32[s] = al;
                }
                if (live && !valid) {                         // status 0 (metrics.py:52-63): straight to the out-queue
                    const int s = out_count + __popc(im & lt_mask);
                    q.out_pix[s] = p; q.out_a32[s] = al; q.out_code[s] = RP_INVALID; q.out_k[s] = 0;
                    q.out_up[s] = 0.0; q.out_wp[s] = 0.0; q.out_u[s] = 0.0; q.out_w[s] = 0.0;
                }
                in_head = 0;
                in_count = __popc(vm);
                out_count += __popc(im);
                if (lane == 0) q.out_tail = out_count;
                __syncwarp();
                if (in_count == 0) continue;             // nothing valid in this batch (may have to finish first)
            }
            const int rank = __popc(need & lt_mask);
            if (code == -2 && rank < in_count) {
                const int s = in_head + rank;
                w = q.in_w0[s]; pix = q.in_pix[s]; a32 = q.in_a32[s];
                u = c.u0; k = 0; code = -1;
                binet_scale_in<FUSED>(c, u, w);          // the FMA loop carries 3M u (rk4_step)
            }
            const int taken = min(__popc(need), in_count);
            in_head += taken;
            in_count -= taken;
            __syncwarp();
            // lanes may still be empty (the in-queue ran dry): go round again unless nothing is left
            if (__ballot_sync(full, code == -2) != 0u && (in_count > 0 || next_batch < n_batches)) continue;
        }

        // ---- integrate: trips of four RK4 steps (a trip of binet_trace_fast<FUSED, 4>) until enough lanes have left
        // the band to make a refill worth its bookkeeping (refill_min; everything, once no ray is left to pop) ----
        // A lane that leaves the band claims a slot of the out-queue (shared-memory atomic) and stores its raw
        // exit state there at once — nothing but (u, w, k) stays live across trips.
        const int stop_at = (in_count > 0 || next_batch < n_batches) ? refill_min : 32;
        unsigned idle;
        do {
            if (code == -1) {
                double up, wp;
                int xcode = -1;
                if (k + 4 <= n_full) {
                    double u1, w1, u2, w2, u3, w3, u4, w4;
                    rk4_full_step<FUSED>(L, u, w, u1, w1);
                    rk4_full_step<FUSED>(L, u1, w1, u2, w2);
                    rk4_full_step<FUSED>(L, u2, w2, u3, w3);
                    rk4_full_step<FUSED>(L, u3, w3, u4, w4);
                    const unsigned t1 = (unsigned)__double2hiint(u1) - lo_hi;
                    const unsigned t2 = (unsigned)__double2hiint(u2) - lo_hi;
                    const unsigned t3 = (unsigned)__double2hiint(u3) - lo_hi;
                    const unsigned t4 = (unsigned)__double2hiint(u4) - lo_hi;
                    int which = 0;
                    bool cap = false;
                    if (max(max(t1, t2), max(t3, t4)) >= span) {
                        if (u1 >= b_hi) { which = 1; cap = true; }
                        else if (u1 <= b_lo) { which = 1; }
                        else if (u2 >= b_hi) { which = 2; cap = true; }
                        else if (u2 <= b_lo) { which = 2; }
                        else if (u3 >= b_hi) { which = 3; cap = true; }
                        else if (u3 <= b_lo) { which = 3; }
                        else if (u4 >= b_hi) { which = 4; cap = true; }
                        else if (u4 <= b_lo) { which = 4; }
                    }
                    if (which == 0) { u = u4; w = w4; k += 4; }
                    else {
                        xcode = cap ? RP_CAPTURE : RP_ESCAPE;
                        k += which - 1;                     // index of the exit step
                        if (which == 1) { up = u; wp = w; u = u1; w = w1; }
                        else if (which == 2) { up = u1; wp = w1; u = u2; w = w2; }
                        else if (which == 3) { up = u2; wp = w2; u = u3; w = w3; }
                        else { up = u3; wp = w3; u = u4; w = w4; }
                    }
                } else {
                    xcode = RP_RANOUT; up = u; wp = w;      // fewer than four full steps left: finished in the tail
                }
                if (xcode >= 0) {
                    const int s = atomicAdd(&q.out_tail, 1);
                    q.out_up[s] = up; q.out_wp[s] = wp; q.out_u[s] = u; q.out_w[s] = w;
                    q.out_pix[s] = pix; q.out_a32[s] = a32; q.out_k[s] = k; q.out_code[s] = xcode;
                    code = -2;
                }
            }
            if (a.stats && lane == 0) ws.trips++;
            idle = __ballot_sync(full, code != -1);
        } while (__popc(idle) < stop_at);
        __syncwarp();
        out_count = *(volatile int *)&q.out_tail;
    }

    // ---- write-out of the chunk's pixels ----
    if (n_chunk > 0) {
        for (int b = 0; b < n_batches; ++b) {
            const int p0 = b * 32;
            const int cnt = min(32, n_chunk - p0);
            int row, col;
            long long oi;
            tile_pixel(a, cam.width, chunk0 + p0 + (lane < cnt ? lane : 0), row, col, oi);
            const int bytes = 32 * C * (int)sizeof(T);
            if (ra.vec_ok && cnt == 32) {
                // the 32 pixels are contiguous in the output and start on a 16-byte boundary
                const long long o0 = __shfl_sync(full, oi, 0);
                const uint4 *s4 = reinterpret_cast<const uint4 *>(stage + (size_t)p0 * C);
                uint4 *d4 = reinterpret_cast<uint4 *>((T *)ra.out + o0 * C);
                for (int v = lane; v < bytes / 16; v += 32) d4[v] = s4[v];
            } else if (lane < cnt) {
                const T *s = stage + (size_t)(p0 + lane) * C;
                T *d = (T *)ra.out + oi * C;
                for (int ch = 0; ch < C; ++ch) d[ch] = s[ch];
            }
        }
    }
    if (a.stats) {
        StatAcc acc;
        acc.init();
        unsigned long long n_rays = 0ull;
        if (lane == 0) {
            acc.escaped = ws.escaped; acc.captured = ws.captured; acc.invalid = ws.invalid; acc.winding = ws.winding;
            acc.max_steps = ws.max_steps; acc.max_winding = ws.max_winding; acc.sum_steps = ws.sum_steps;
            acc.warp_steps = 128ull * ws.trips;
            acc.min_fa = __longlong_as_double((long long)ws.min_fa);
            acc.max_fa = __longlong_as_double((long long)ws.max_fa);
            n_rays = ws.n_rays;
        }
        lp_stats_flush(acc, n_rays, a.stats);
    }
}

// The lane re-packing frame kernel.  vec_ok: every full 32-pixel batch of a chunk is contiguous in the output
// (contiguous rows, or frame rows a multiple of 32 wide) and 16-byte aligned (the chunks are staged by construction).
int lp_launch_render_repack(TraceArgs a, RemapArgs ra, const BinetConsts &c, const CamConsts &cam, int elem,
                            bool fused, cudaStream_t stream)
{
    ra.vec_ok = ((!a.out_frame_rows || cam.width % 32 == 0) && ((uintptr_t)ra.out % 16) == 0) ? 1 : 0;
    // 16 CTAs of 64 threads per SM at 64 registers; let the whole shared memory be used for it
    const void *const kernels[3][2] = {
        {(const void *)lp_render_repack_kernel<false, unsigned char, 16>, (const void *)lp_render_repack_kernel<true, unsigned char, 16>},
        {(const void *)lp_render_repack_kernel<false, float, 16>, (const void *)lp_render_repack_kernel<true, float, 16>},
        {(const void *)lp_render_repack_kernel<false, double, 16>, (const void *)lp_render_repack_kernel<true, double, 16>}};
    const void *fn = kernels[elem][fused];
    const size_t esz = elem == ELEM_F64 ? 8 : elem == ELEM_F32 ? 4 : 1;
    const size_t stage_bytes = ((size_t)LP_RP_CHUNK * ra.channels * esz + 15) & ~(size_t)15;
    const size_t smem = LP_RP_WARPS * (sizeof(RpQueues) + stage_bytes);
    if (cudaFuncSetAttribute(fn, cudaFuncAttributePreferredSharedMemoryCarveout, 100) != cudaSuccess) cudaGetLastError();
    if (smem > 48 * 1024 &&
        cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) {
        cudaGetLastError();
        return LP_ERR_UNSUPPORTED;
    }
    // refill: idle lanes that trigger a refill (1 = after every trip that saw an exit; larger values trade idle
    // lanes for less bookkeeping)
    int refill = lp_trace_knobs().repack_refill;
    void *args[] = {&a, &ra, (void *)&c, (void *)&cam, &refill};
    return lp_launch_ctas(fn, a.n, (long long)LP_RP_WARPS * LP_RP_CHUNK, LP_RP_BLOCK, smem, args, stream);
}
