/* vs_flow_rows.cu -- the flow-only render kernel of libvoicesynth_cuda for batches without glottal noise: a warp per
 * row, lanes along the row.  (Everything else -- the fused generator + filter, the filter alone, flow with noise -- is
 * vs_render.cu, one lane per row.) */
#include "vs_device.cuh"

/* ================================================================================================
 * Flow only, no glottal noise: LANES ALONG THE ROW (vs_flow_rows_kernel).
 *
 * Without the filter nothing is carried from one sample to the next: sample m of a voice is
 *     x[m] = max(ceil(A_p * table[m - start_p]), (short)DC)          (flowgen_shimmer.c:316-336, see gen_fast above)
 * with p the pitch period that contains m -- a function of the period table alone.  So a WARP takes a row (one
 * time-chunk of one voice) and its lanes spread along it: per step the warp writes 256 consecutive samples, lane l
 * the pairs  M + 64u + 2l, u = 0..3  -- every store instruction of the warp is one whole 128-byte line, every table
 * load 256 consecutive bytes, no tile, no TMA, nothing staged.  What the lane-per-row generator kept per lane in
 * registers (its current and next period), a warp keeps in shared memory for 32 periods at a time: their first
 * samples (a prefix sum of the lengths), amplitudes as doubles, and the value of their first sample -- the one a
 * pair that straddles two periods needs.  A lane finds its periods by counting the period starts of the step
 * (warp-uniform loop, one or two iterations for speech).
 * Rows are handed out by an atomic ticket: the grid is persistent, rows of any length balance.
 * ceil() is one FP64 add in round-up mode against 1.5*2^52 (the integer lands in the low word): the conversion
 * instruction F2I.F64 runs on the quarter-rate XU pipe, which would bind this kernel.  |A*table| < 2^31 holds for
 * every stream row_validate() accepts with T2 >= 2 (the host sends other batches to the lane-per-row kernel).
 * ============================================================================================== */
#define VS_SPAN 256            /* samples per warp step: 32 lanes x 4 pairs */

__device__ __forceinline__ int vs_ceil_magic(double p)
{
    return __double2loint(__dadd_ru(p, 6755399441055744.0));
}

/* p += (bnd <= m): one compare and one predicated add */
__device__ __forceinline__ void vs_count_le(int &p, int bnd, int m)
{
    asm("{\n\t.reg .pred q;\n\tsetp.le.s32 q, %1, %2;\n\t@q add.s32 %0, %0, 1;\n\t}" : "+r"(p) : "r"(bnd), "r"(m));
}

__global__ void __launch_bounds__(VS_FLOWROWS_WARPS * 32, 4) vs_flow_rows_kernel(const VsRenderArgs a)
{
    /* per warp, for the periods qb + j, j = 0..31: {first sample, length - 1, amplitude (double)} and the value of the
     * period's first sample; entry 32 = the end of the batch */
    __shared__ __align__(16) uint4 s_ent[VS_FLOWROWS_WARPS][34];
    __shared__ int s_first[VS_FLOWROWS_WARPS][34];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint4 *ent = s_ent[warp];
    int *first = s_first[warp];

    for (;;) {
        uint32_t row = 0;
        if (lane == 0) row = atomicAdd(a.ticket, 1u) - a.ticket_base;
        row = __shfl_sync(VS_FULL, row, 0);
        if (row >= a.n_rows) break;                         /* (every warp draws exactly one ticket beyond the last row) */
        const uint32_t chunk_id = __ldg(a.order + row);
        if (chunk_id == VS_NO_CHUNK) continue;
        const uint4 c0 = __ldg(reinterpret_cast<const uint4 *>(a.chunks + chunk_id));        /* stream, emit_lo, emit_hi, gen_target */
        const uint2 c1 = __ldg(reinterpret_cast<const uint2 *>(a.chunks + chunk_id) + 2);    /* first_period, first_start */
        const VsStream *st = a.streams + c0.x;
        const int lo = (int)c0.y, hi = (int)c0.z;
        const uint32_t np = min(__ldg(a.n_periods + c0.x), st->tab_cap);
        uint32_t qb = c1.x;
        int sb = (int)c1.y;
        if (qb >= np) {                                     /* the plan kernel did not reach this chunk: refuse to walk garbage */
            if (lane == 0) atomicExch(a.status, VS_ECUDA);
            continue;
        }
        int16_t *orow = a.pcm_out + st->out_off;
        const uint2 *ptab = reinterpret_cast<const uint2 *>(a.table) + st->tab_off;           /* VsPeriodC */
        /* the pulse table: n2 entries, two zeros, and the same again moved up by one entry (vs_batch_plan.cpp, VsTables::pulse_table) */
        const double *tab = a.costab + st->pulse_off;
        const uint32_t n2 = 2u * (uint32_t)st->T2;
        const int DCs = st->DCs;
        const double h0 = __ldg(tab);

        int blimit = 0;                                     /* samples below it can be evaluated from the batch in `ent` */
        bool more = false;                                  /* the table goes on after the batch */
        auto load_batch = [&]() {
            const uint32_t idx = qb + (uint32_t)lane;
            const bool valid = idx < np;
            uint2 e = make_uint2(0u, 0u);
            if (valid) e = __ldg(ptab + idx);
            const int T = (int)e.y;
            int incl = T;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int up = __shfl_up_sync(VS_FULL, incl, o);
                if (lane >= o) incl += up;
            }
            const int start = sb + incl - T;
            const double Ad = (double)__uint_as_float(e.x);
            const int fv = max(vs_ceil_magic(__dmul_rn(Ad, h0)), DCs);
            __syncwarp();                                   /* the previous batch has been read by every lane */
            ent[lane] = make_uint4((uint32_t)start, (uint32_t)(T - 1), (uint32_t)__double2loint(Ad), (uint32_t)__double2hiint(Ad));
            first[lane] = fv;
            if (lane == 31) { ent[32] = make_uint4((uint32_t)(start + T), 0xffffffffu, 0u, 0u); first[32] = DCs; }
            __syncwarp();
            more = qb + 32u < np;
            /* with more periods to come the batch's last one only serves as the `next` of a straddling pair */
            blimit = __shfl_sync(VS_FULL, more ? start : start + T, 31);
        };
        load_batch();

        /* steps are anchored on the 128-byte lines of the row's own address */
        const int ph64 = (int)((reinterpret_cast<uintptr_t>(orow) >> 1) & 63);
        int P = 0;                                          /* batch index of the period that contains the previous step's last sample */
        for (int M = lo - ((ph64 + lo) & 63); M < hi; M += VS_SPAN) {
            const int Mend = min(M + VS_SPAN, hi);
            if (Mend > blimit && more) {                    /* re-base the batch on the current period */
                qb += (uint32_t)P;
                sb = (int)ent[P].x;
                P = 0;
                load_batch();
            }
            if (Mend > blimit) {                            /* the period table does not cover the row */
                if (lane == 0) atomicExch(a.status, VS_ECUDA);
                break;
            }
            /* the period of each of the lane's four pairs: P + the period starts since then at or before the pair */
            const int Mlast = Mend - 1;
            const int m0 = M + 2 * lane;
            int pu[4] = {P, P, P, P};
            {
                int j = P + 1;
                int bnd = (int)ent[j].x;
                while (bnd <= Mlast) {
                    vs_count_le(pu[0], bnd, m0);
                    vs_count_le(pu[1], bnd, m0 + 64);
                    vs_count_le(pu[2], bnd, m0 + 128);
                    vs_count_le(pu[3], bnd, m0 + 192);
                    j++;
                    bnd = (int)ent[j].x;
                }
                P = j - 1;
            }
            /* all loads of the step first: four 16-byte table reads per lane in flight */
            double A[4];
            double2 f[4];
            bool str[4];
#pragma unroll
            for (int u = 0; u < 4; u++) {
                const uint4 e0 = ent[pu[u]];
                const uint32_t i0 = (uint32_t)(m0 + 64 * u) - e0.x;      /* "negative" before the row's first period */
                A[u] = __hiloint2double((int)e0.w, (int)e0.z);
                str[u] = (int)i0 >= (int)e0.y;              /* the pair's second sample opens the next period */
                const uint32_t ic = min(i0, n2);            /* beyond the open phase the table is zero */
                uint32_t off;                               /* odd: the copy moved up by one entry: ic + (ic & 1) * (n2 + 1) */
                asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(off) : "r"(ic & 1u), "r"(n2 + 1u), "r"(ic));
                f[u] = __ldg(reinterpret_cast<const double2 *>(tab + off));
            }
            int x0[4], x1[4];
#pragma unroll
            for (int u = 0; u < 4; u++) {
                x0[u] = max(vs_ceil_magic(__dmul_rn(A[u], f[u].x)), DCs);
                x1[u] = max(vs_ceil_magic(__dmul_rn(A[u], f[u].y)), DCs);
                if (str[u]) x1[u] = first[pu[u] + 1];
            }
            if (M >= lo && M + VS_SPAN <= hi) {
                uint32_t *const o32 = reinterpret_cast<uint32_t *>(orow + m0);
#pragma unroll
                for (int u = 0; u < 4; u++) o32[32 * u] = __byte_perm((uint32_t)x0[u], (uint32_t)x1[u], 0x5410);
            } else {                                        /* a stream's first or last step */
#pragma unroll
                for (int u = 0; u < 4; u++) {
                    const int m = m0 + 64 * u;
                    if (m >= lo && m < hi) orow[m] = (int16_t)x0[u];
                    if (m + 1 >= lo && m + 1 < hi) orow[m + 1] = (int16_t)x1[u];
                }
            }
        }
    }
}

/* the lanes-along-the-row flow kernel: grid CTAs of VS_FLOWROWS_WARPS warps.  The ticket counter is never reset: a
 * launch starts at a.ticket_base and leaves it at ticket_base + n_rows + (warps of the grid) */
cudaError_t vs_launch_flow_rows(const VsRenderArgs &a, cudaStream_t s)
{
    vs_flow_rows_kernel<<<a.grid, VS_FLOWROWS_WARPS * 32, 0, s>>>(a);
    return cudaGetLastError();
}

