// tc_contract.cuh -- the binomial score contraction on the tcgen05 INT8 tensor cores, exact to FP64 rounding.
//
// FullStat of the logistic solver (ElasticNetBinaryNEmainEff.c:1693-1735) needs, for every candidate c,
//     G[p][c] = sum_h x_c[h] (w[h] phi_p[h]) / s_c,   ze[c] = sum_h x_c[h] e[h],   bb[c] = sum_h x_c[h]^2 w[h]
// again after every block of actions, because the IRLS weights w change.  On genotype-coded designs x is an exact small
// integer, so only the right-hand sides carry 53-bit mantissas.  Each right-hand-side column b (w o phi_p for p < M, then
// e) is scaled by a power of two and cut into 8 balanced base-128 digit planes (b = scale * sum_s d_s 128^-(s+1), digits
// in [-64, 64], every step exact); the planes are multiplied by the int8 training matrix in exact int32 arithmetic and
// recombined in FP64 by Horner's rule.  The result is the exact dot product of x_c with b truncated 56 bits below the
// column's largest entry: an error of at most N 2^-57 max|b| max|x|, below the rounding error of an FP64 summation.
// bb is the squared matrix X o X against column 0's planes (phi_0 = 1, so column 0 is w).  |x| <= 11 keeps x^2 in int8.
// The int32 sum of one plane is at most N max|x|^2 64 in magnitude: the host takes this path only while that is below 2^31
// (N = 277,000 training rows at |x| = 11).
//
// Form (tcgen05.mma.cta_group::1.kind::i8, operands in shared memory, accumulators in tensor memory):
//   * D[128 candidates][8 planes x up to TC_COLS columns] += A[128 x 32 rows] B[8 TC_COLS x 32 rows]' per 32-row stage,
//     plus D_bb[128][16] += Asq B[rows 0..15]' in the first pass (only its first 8 columns, column 0's planes, are read).
//   * Both operands are stored in the canonical K-major layout without swizzle: 8-row x 16-byte core matrices, the two
//     16-byte halves of a 32-row stage 128 bytes apart, consecutive 8-row groups 256 bytes apart.  The operand images are
//     built in that layout in global memory (FoldData::Xtc / Xtcsq, per fold, tiled [128-candidate tile][stage]; the
//     digit planes per pass in the slab, [stage][column]), so one stage of each is one cp.async.bulk.
//   * One thread streams the stages through a two-deep shared-memory ring (mbarrier complete_tx) and issues the MMAs;
//     tcgen05.commit to a second mbarrier per slot frees a slot once the MMAs that read it are done.
//   * Epilogue: every warp reads 32 candidates (its TMEM lane quarter) of half of the columns with tcgen05.ld.
// The MMA issue order, and with it every sum, depends on the row index only: exact duplicate columns tie exactly.
#pragma once
#include "common.cuh"
#include "gauss_fit.cuh"

namespace pareben {

constexpr int TC_TILE = 128;                                   // candidates per MMA (the M of the instruction)
constexpr int TC_KS = 32;                                      // training rows per stage (the K of one kind::i8 MMA)
constexpr int TC_PLANES = 8;
constexpr int TC_COLS = 30;                                    // columns per pass: 8 x 30 accumulator columns + 16 for bb
constexpr int TC_BB_COL = 240;
constexpr int TC_TMEM_COLS = 256;                              // per block: two resident blocks share the SM's 512 columns
constexpr int TC_A_BYTES = TC_TILE * TC_KS;                    // one stage of one candidate tile
constexpr int TC_COL_BYTES = TC_PLANES * TC_KS;                // one stage of one column's planes
constexpr int TC_SLOTS = 2;                                     // stages in flight (more were measured slower: the L2 is the limit)
constexpr int TC_RING_BYTES = 40448;                           // the ring: as many slots of a pass's stage size as fit (<= TC_SLOTS)
constexpr int TC_SMEM_BYTES = TC_RING_BYTES + 8 * TC_COLS;     // the ring + the column scales
static_assert(TC_PLANES * TC_COLS + 16 <= TC_TMEM_COLS, "accumulators exceed the tensor-memory allocation");
static_assert(2 * (2 * TC_A_BYTES + TC_COLS * TC_COL_BYTES) <= TC_RING_BYTES, "the ring must hold two stages of any pass");

// Kept in static shared memory for the life of the kernel: the TMEM allocation, the ring's barriers and the parities of
// their next phases (bit s for slot s; only thread 0 issues, waits on and updates them).
struct TcState {
    unsigned long long full[TC_SLOTS], done[TC_SLOTS];
    unsigned tmem;
    unsigned fpar, cpar;                 // next phase of full[s]; next phase of done[s] (every commit has been waited for)
    unsigned ep_slot, ep_par;            // the barrier phase that ends the current tile, for the epilogue's wait
};

// byte offset of (candidate c, training row h) in an operand image with nst stages per candidate tile
__host__ __device__ inline size_t tc_image_offset(int c, int h, int nst)
{
    const int tile = c >> 7, cl = c & 127, st = h >> 5, hk = h & 31;
    return (size_t)(tile * nst + st) * TC_A_BYTES + (cl >> 3) * 256 + (hk >> 4) * 128 + (cl & 7) * 16 + (hk & 15);
}

// shared-memory matrix descriptor: K-major, no swizzle, 16-byte halves of a stage 128 B apart, 8-row groups 256 B apart
__device__ inline unsigned long long tc_desc(const void *smem)
{
    return (unsigned long long)((smem_u32(smem) & 0x3ffff) >> 4) | ((unsigned long long)(128 >> 4) << 16) |
           ((unsigned long long)(256 >> 4) << 32) | (1ull << 46);
}
// instruction descriptor: s32 accumulators, signed int8 A and B, both K-major, M = 128
__device__ inline unsigned tc_idesc(int n) { return (2u << 4) | (1u << 7) | (1u << 10) | ((unsigned)(n >> 3) << 17) | ((unsigned)(TC_TILE >> 4) << 24); }

__device__ inline void tc_mma(unsigned d, unsigned long long a, unsigned long long b, unsigned idesc, int accumulate)
{
    asm volatile("{\n.reg .pred p;\nsetp.ne.b32 p, %4, 0;\ntcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n}\n"
                 ::"r"(d), "l"(a), "l"(b), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ inline void tc_commit(unsigned long long *bar)
{
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ inline void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ inline void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }

// 16 consecutive accumulator columns of this thread's TMEM lane
__device__ inline void tc_ld16(unsigned addr, int (&r)[16])
{
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];\n"
                 "tcgen05.wait::ld.sync.aligned;"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                   "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
                 : "r"(addr) : "memory");
}

// Block-wide, once at kernel start: warp 0 allocates the block's tensor memory (and gives up the right to allocate more,
// so that the other resident block's allocation never waits), thread 0 sets up the ring's barriers.
__device__ inline void tc_open(TcState &ts)
{
    if (threadIdx.x < 32) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&ts.tmem)), "r"(TC_TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (threadIdx.x == 0) {
        for (int b = 0; b < TC_SLOTS; b++) { mbar_init(&ts.full[b], 1); mbar_init(&ts.done[b], 1); }
        ts.fpar = 0; ts.cpar = 0;
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
}

// Block-wide, once before the kernel exits (every MMA has been waited for by then).
__device__ inline void tc_close(TcState &ts)
{
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    if (threadIdx.x < 32)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(ts.tmem), "r"(TC_TMEM_COLS) : "memory");
}

// Digit extraction stages a column in chunks of TC_DIG_ROWS training rows through shared memory (the ring is idle while
// it runs): a lane issues the cp.async copies of its four consecutive rows of every 128-row group (TC_DIG_V values) at
// once, so a chunk costs one trip to L2, and the column's maximum and its digits both read the staged copy.  Element k
// of lane l sits at [32 k + l], so a warp's reads of one k are one contiguous 256-byte row.
constexpr int TC_DIG_GROUPS = 4;
constexpr int TC_DIG_V = 4 * TC_DIG_GROUPS;                   // values per lane and chunk
constexpr int TC_DIG_ROWS = 128 * TC_DIG_GROUPS;              // rows per chunk
constexpr int TC_DIG_WARPS = 8;                               // warps per block (FIT_T = 256 threads) the staging area serves
static_assert((TC_DIG_WARPS + 1) * TC_DIG_ROWS * 8 <= TC_RING_BYTES, "the digit staging area must fit the ring");

// 8-byte copy global -> shared, zero-filled when !valid (src is then not read)
__device__ inline void cp_async8(double *dst, const double *src, bool valid)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;" ::"r"(smem_u32(dst)), "l"(src), "r"(valid ? 8 : 0) : "memory");
}
__device__ inline void cp_async_wait_all() { asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;" ::: "memory"); }

// Digit planes of columns j0 .. j0 + ncols - 1 ([stage][column][16-row half][plane][16 rows]) and their scales.  Column
// j < R is wv o col(j), column R is ev.  A warp per column, a lane per four consecutive rows of every 128-row group; the
// digits are peeled off a 56-bit fixed-point integer (rounded once, every later step exact).  stage: shared memory for
// TC_DIG_WARPS + 1 chunks.  When the rows fit one chunk (N <= 512), wv is staged once for the whole block and every
// column is read once; longer columns take one pass over the chunks for the maximum and a second one for the digits
// (which begins with the chunk still staged from the first), with wv read from global memory.
template <class Col>
__device__ inline void tc_digits(int j0, int ncols, int N, int nst, int R, Col col, const double *__restrict__ wv,
                                 const double *__restrict__ ev, int8_t *__restrict__ planes, double *bscale, double *stage)
{
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
    const int nrow = nst * TC_KS, nch = (nrow + TC_DIG_ROWS - 1) / TC_DIG_ROWS;
    auto row = [&](int ch, int k) { return ch * TC_DIG_ROWS + 128 * (k >> 2) + 4 * lane + (k & 3); };
    // this lane's rows of chunk ch of a -> d[32 k + lane], 0 past row N
    auto stage_chunk = [&](double *d, const double *__restrict__ a, int ch) {
#pragma unroll
        for (int k = 0; k < TC_DIG_V; k++) { const int h = row(ch, k); cp_async8(d + 32 * k + lane, h < N ? a + h : a, h < N); }
        cp_async_wait_all();
    };
    double *ws = stage, *cs = stage + (size_t)(1 + wid) * TC_DIG_ROWS;
    if (nch == 1) {
        if (wid == 0) stage_chunk(ws, wv, 0);
        __syncthreads();
    }
    for (int jl = wid; jl < ncols; jl += nw) {
        const int j = j0 + jl;
        const bool prod = j < R;
        const double *__restrict__ src = prod ? col(j) : ev;
        auto val = [&](int ch, int k) -> double {              // the column's value at row(ch, k), staged
            const double x = cs[32 * k + lane];
            if (!prod) return x;
            if (nch == 1) return ws[32 * k + lane] * x;
            const int h = row(ch, k);
            return h < N ? wv[h] * x : 0.0;
        };
        double mx = 0.0;
        bool bad = false;
        for (int ch = 0; ch < nch; ch++) {
            stage_chunk(cs, src, ch);
#pragma unroll
            for (int k = 0; k < TC_DIG_V; k++) { const double a = fabs(val(ch, k)); if (!(a <= 1.7976931348623157e308)) bad = true; mx = fmax(mx, a); }
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        bad = __any_sync(0xffffffffu, bad);
        int ex = 0;
        (void)frexp(mx, &ex);                                   // mx = m 2^ex, m in [1/2, 1)
        const bool live = !bad && mx > 1e-290;                  // an all-zero (or denormal) column contributes zeros
        const double down = live ? scalbn(1.0, 55 - ex) : 0.0;  // |val * down| < 2^55, exact
        // the column's scale 2^(ex+1) is stored as 2^(ex-1), and Horner's last step multiplies by 2^-5 instead of 2^-7:
        // 2^(ex+1) itself overflows for a column maximum >= 2^1022 (ex = 1023, 1024).  Horner's sum is never subnormal,
        // so both forms are one exact power-of-two scaling (rounded only on overflow) and agree bit for bit below 2^1022.
        if (lane == 0) bscale[jl] = bad ? __longlong_as_double(0x7ff8000000000000LL) : (live ? scalbn(1.0, ex - 1) : 0.0);
        int8_t *colp = planes + (size_t)jl * TC_COL_BYTES;
        for (int ch = nch - 1; ch >= 0; ch--) {
            if (ch < nch - 1) stage_chunk(cs, src, ch);
#pragma unroll 1                                                // rolled: fewer spills in the fit kernel around it
            for (int g = 0; g < TC_DIG_GROUPS; g++) {
                const int p4 = row(ch, 4 * g);
                if (p4 >= nrow) break;
                unsigned wout[TC_PLANES];
#pragma unroll
                for (int s = 0; s < TC_PLANES; s++) wout[s] = 0u;
#pragma unroll
                for (int b = 0; b < 4; b++) {
                    // rows past N are staged as 0: their digits are 0
                    const long long q = live ? __double2ll_rn(val(ch, 4 * g + b) * down) : 0LL;
                    // balanced base-128 digits, least significant first, in 32-bit arithmetic: the low 28 bits give four
                    // digits and a carry into the high part, which gives the other four
                    int lo = (int)(q & 0xfffffff), hi = (int)(q >> 28);
#pragma unroll
                    for (int s = TC_PLANES - 1; s >= 0; s--) {
                        int &x = s >= 4 ? lo : hi;
                        const int d = ((x + 64) & 127) - 64;        // in [-64, 63]
                        x = (x - d) >> 7;                           // exact
                        if (s == 4) hi += lo;                       // the carry (0 or 1)
                        const int dig = s == 0 ? d + (x << 7) : d;  // the top digit takes what is left (|.| <= 64)
                        wout[s] |= ((unsigned)dig & 0xffu) << (8 * b);
                    }
                }
                int8_t *dst = colp + (size_t)(p4 >> 5) * ncols * TC_COL_BYTES + ((p4 >> 4) & 1) * 128 + (p4 & 15);
#pragma unroll
                for (int s = 0; s < TC_PLANES; s++) *reinterpret_cast<unsigned *>(dst + s * 16) = wout[s];
            }
        }
    }
}

// Columns j in [0, R]: j < R is wv o col(j) (stored to dest(j) divided by the candidate's scale), j == R is ev (stored
// to ze_out); bb_out[c] = sum_h x_c[h]^2 wv[h].  The binomial FullStat's contraction, on FoldData::Xtc.
template <class Col, class Dest>
__device__ inline void tc_contract(const FoldData &F, int Kc, int R, Col col, Dest dest, const double *__restrict__ wv,
                                   const double *__restrict__ ev, double *bb_out, double *ze_out, int8_t *planes, double *sV,
                                   TcState &ts)
{
    const int N = F.ntr, nst = (N + TC_KS - 1) / TC_KS, ntile = (Kc + TC_TILE - 1) / TC_TILE;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    char *ring = reinterpret_cast<char *>(sV);
    double *bscale = reinterpret_cast<double *>(ring + TC_RING_BYTES);
    const unsigned tmem = ts.tmem;
    __syncthreads();
    PHASE(PH_CONTRACT);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");    // the ring held generic-proxy data of other phases
    const int ncol_all = R + 1;
    for (int j0 = 0; j0 < ncol_all;) {
        const bool first = j0 == 0;                             // the first pass also streams X o X for bb
        const int ncols = min(TC_COLS, ncol_all - j0), ncp = (ncols + 1) & ~1;
        __syncthreads();                                        // the previous pass's planes are fully consumed
        tc_digits(j0, ncols, N, nst, R, col, wv, ev, planes, bscale, reinterpret_cast<double *>(ring));
        asm volatile("fence.proxy.async.global;" ::: "memory");     // the planes are read by the bulk copies
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // the digits were staged in the ring
        __syncthreads();
        // A slot holds ncp columns: with an odd column count the MMA (N = 8 ncp), and with one column the bb MMA (N = 16),
        // read one column's planes past the copied ones.  They stay inside the slot, and the accumulator columns they feed
        // are never read.
        const unsigned tx_bytes = TC_A_BYTES * (first ? 2 : 1) + ncols * TC_COL_BYTES;
        const unsigned stage_bytes = TC_A_BYTES * (first ? 2 : 1) + ncp * TC_COL_BYTES;
        const int nslot = min(TC_SLOTS, TC_RING_BYTES / (int)stage_bytes);
        const int n_item = ntile * nst;                         // (tile, stage) pairs of this pass, tile-major
        const unsigned idesc = tc_idesc(8 * ncp), idesc_bb = tc_idesc(16);
        // thread 0's view of the ring: item k sits in slot k % nslot; a slot is refilled once the MMAs that read it are done
        int issued = 0;
        auto load = [&](int k) {
            const int sl = k % nslot, t = k / nst, st = k - t * nst;
            if (k >= nslot) mbar_wait(&ts.done[sl], ((ts.cpar >> sl) & 1) ^ 1);       // the slot's last commit
            char *dst = ring + sl * stage_bytes;
            const size_t ao = ((size_t)t * nst + st) * TC_A_BYTES;
            mbar_expect_tx(&ts.full[sl], tx_bytes);
            bulk_load(dst, F.Xtc + ao, TC_A_BYTES, &ts.full[sl]);
            if (first) bulk_load(dst + TC_A_BYTES, F.Xtcsq + ao, TC_A_BYTES, &ts.full[sl]);
            bulk_load(dst + (first ? 2 : 1) * TC_A_BYTES, planes + (size_t)st * ncols * TC_COL_BYTES, ncols * TC_COL_BYTES, &ts.full[sl]);
        };
        for (int t = 0; t < ntile; t++) {
            if (threadIdx.x == 0) {
                for (int st = 0; st < nst; st++) {
                    const int k = t * nst + st;
                    while (issued < min(k + nslot, n_item)) load(issued++);
                    const int sl = k % nslot;
                    mbar_wait(&ts.full[sl], (ts.fpar >> sl) & 1);
                    ts.fpar ^= 1u << sl;
                    tc_fence_after();
                    const char *buf = ring + sl * stage_bytes;
                    const unsigned long long bd = tc_desc(buf + (first ? 2 : 1) * TC_A_BYTES);
                    tc_mma(tmem, tc_desc(buf), bd, idesc, st > 0);
                    if (first) tc_mma(tmem + TC_BB_COL, tc_desc(buf + TC_A_BYTES), bd, idesc_bb, st > 0);
                    tc_commit(&ts.done[sl]);
                    ts.cpar ^= 1u << sl;                        // bit = parity of the NEXT commit's phase on this slot
                    if (st == nst - 1) { ts.ep_slot = sl; ts.ep_par = ((ts.cpar >> sl) & 1) ^ 1; }
                }
                // the next tile's first stages travel while this tile's epilogue runs
                while (issued < min((t + 1) * nst + nslot, n_item)) load(issued++);
            }
            __syncthreads();
            mbar_wait(&ts.done[ts.ep_slot], ts.ep_par);
            tc_fence_after();
            // epilogue: warp w reads TMEM lanes 32 (w % 4) .. + 31 (one candidate each), warps 0-3 the first half of
            // the columns and warps 4-7 the rest, two columns (16 accumulator columns) per load
            const int c = t * TC_TILE + 32 * (wid & 3) + lane;
            const bool live = c < Kc;
            const unsigned lane_addr = tmem + ((unsigned)(32 * (wid & 3)) << 16);
            const int half = (((ncols + 1) >> 1) + 1) & ~1;
            const int jb = (wid >> 2) ? half : 0, je = (wid >> 2) ? ncols : min(half, ncols);
            double sc = 1.0, isc = 1.0;
            if (live) { sc = F.scale[c]; isc = 1.0 / sc; }
            for (int jl = jb; jl < je; jl += 2) {
                int acc[16];
                tc_ld16(lane_addr + 8 * jl, acc);
#pragma unroll
                for (int u = 0; u < 2; u++) {
                    const int jj = jl + u;
                    if (jj < je && live) {
                        double v = 0.0;
#pragma unroll
                        for (int s = TC_PLANES - 1; s >= 0; s--) v = (v + (double)acc[8 * u + s]) * (s ? 0.0078125 : 0.03125);   // Horner, 128^-1 exact
                        v *= bscale[jj];
                        const int j = j0 + jj;
                        if (j < R) { bool dv = false; double *row = dest(j, dv); row[c] = dv ? div_by(v, sc, isc) : v; }
                        else ze_out[c] = v;
                    }
                }
            }
            if (first && (wid >> 2) == 0) {
                int acc[16];
                tc_ld16(lane_addr + TC_BB_COL, acc);
                if (live) {
                    double v = 0.0;
#pragma unroll
                    for (int s = TC_PLANES - 1; s >= 0; s--) v = (v + (double)acc[s]) * (s ? 0.0078125 : 0.03125);
                    bb_out[c] = v * bscale[0];
                }
            }
            tc_fence_before();
            __syncthreads();                                    // the accumulators are free for the next tile
        }
        if (threadIdx.x == 0)                                   // every commit of the pass has landed: the next pass may lay
            for (int sl = 0; sl < TC_SLOTS; sl++) mbar_wait(&ts.done[sl], ((ts.cpar >> sl) & 1) ^ 1);   // the slots out anew
        j0 += ncols;
    }
    __syncthreads();
}

}  // namespace pareben
