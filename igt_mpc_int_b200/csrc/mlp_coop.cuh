// mlp_coop.cuh -- the gt_mpc value term (mpc.py:326-354, :367-369; model.py:14-67) evaluated exactly
// (the solver's own precision, fp64 on the parity path) by the whole CTA.
//
// Value + first and second forward tangents in (s_N, v_N): six rows per evaluation through every layer.  The
// per-thread version (mlp_eval_thread) streams each thread's activations through HBM and every thread reads the
// whole weight matrices.  Here the valid requests of the CTA are compacted into a list and evaluated in waves of
// (warps x COOP_E): a warp keeps the six activation rows of its COOP_E evaluations in shared memory, lane l owns
// outputs l, l + 32, l + 64, l + 96 of a layer (COOP_E x 24 independent accumulators), and the weights (stored
// transposed, [in][out]) stream through shared memory in tiles of COOP_TI inputs, double-buffered with cp.async and
// shared by all warps of the CTA -- one pass over a layer's weights per wave instead of one per evaluation (round 2's
// first version read 131 KB of weights from L1 / L2 per evaluation and layer and ran at a sixth of the FP64 rate).
// Same operation order per output as mlp_eval_thread: bit-identical results (tests/hostsim runs that one on the
// CPU).  Any network with layer widths <= MLP_COOP_W.
//
// Network bank (mlp_coop_eval_bank): every request names one of up to MAX_MLP_NETS networks.  The requests are
// compacted by network instead (a counting sort, thread order kept inside a group), and each non-empty group runs the
// same waves with its own descriptor, biases and output layer staged in shared memory.  The operation order per output
// is unchanged, so a request's result is bit-identical to the single-network evaluation of its network, whatever
// shares its wave.
//
// Request capacity (template argument CAP of both entry points and their size functions).  CAP = 0: one request slot
// per thread and COOP_E evaluations per warp and wave (the throughput kernels).  CAP > 0: slots for CAP requests only,
// one evaluation per warp and wave, and weight tiles of COOP_TI_CAP inputs -- the latency kernel, whose CTA holds one
// problem and so asks for at most n_alpha <= MAX_ALPHA = COOP_CAP values at a time (the first candidate of its line
// search, its speculative halvings, or the value at a fresh problem), next to its workspace in shared memory; a request
// takes the slot of its position in the compacted list.  The operation order per output does not depend on the tile
// size (inputs in ascending order, the one zero pad row of an odd layer last), so both capacities give the same bits.
#pragma once
#include <cstdint>

namespace igt {

constexpr int MLP_COOP_W = 128;                       // widest layer handled
constexpr int COOP_ITEM = 8, COOP_ROWS = 6;
constexpr int COOP_E = 2;                             // evaluations per warp and wave
constexpr int COOP_TI = 16;                           // inputs per weight tile
constexpr int COOP_CAP = MAX_ALPHA;                   // request capacity of the latency kernel's buffers
constexpr int COOP_TI_CAP = 8;                        // inputs per weight tile with a request capacity
template <int CAP>
struct CoopShape {
    static constexpr int E = CAP ? 1 : COOP_E;        // evaluations per warp and wave
    static constexpr int TI = CAP ? COOP_TI_CAP : COOP_TI;
    static constexpr int slots(int block) { return CAP ? CAP : block; }        // request / result slots
    static constexpr int act_warps(int block) { return CAP ? CAP : block / 32; }   // warps with activation rows
};
// [requests slots x 8] [results slots x 6] [activations act_warps x E x 6 x W] [weight tiles 2 x TI x W]
// [biases of every layer + the output layer's weights: (MAX_MLP_LAYERS + 1) x W] [list: slots + warps ints]
template <typename T, int CAP = 0>
constexpr int mlp_coop_smem_bytes(int block)
{
    using S = CoopShape<CAP>;
    return (int)sizeof(T) * (S::slots(block) * (COOP_ITEM + COOP_ROWS) + S::act_warps(block) * S::E * COOP_ROWS * MLP_COOP_W +
                             2 * S::TI * MLP_COOP_W + (MAX_MLP_LAYERS + 1) * MLP_COOP_W) + 4 * (S::slots(block) + 32);
}
// the bank variant appends the current group's descriptor and the per-warp group counts [MAX_MLP_NETS][32]
template <typename T>
constexpr int mlp_coop_desc_bytes() { return (int)((sizeof(MlpNet<T>) + 15) / 16 * 16); }
template <typename T, int CAP = 0>
constexpr int mlp_coop_bank_smem_bytes(int block)
{
    return mlp_coop_smem_bytes<T, CAP>(block) + mlp_coop_desc_bytes<T>() + 4 * MAX_MLP_NETS * 32;
}

#ifdef __CUDACC__
// rows [i0, i0 + rows) of a transposed weight matrix -> tile[ii * W + o]; every thread copies its share with cp.async.
// An odd number of rows is padded with a row of zeros (the FMA loop takes two inputs per pass, unguarded).
template <typename T>
__device__ __forceinline__ void coop_load_tile(T *tile, const T *Wt, int i0, int rows, int nout)
{
    // thread t copies column t % W of rows t / W, t / W + blockDim.x / W, ... (W = 128 divides the block: no division)
    const int o = threadIdx.x & (MLP_COOP_W - 1), step = blockDim.x >> 7;
    if (o < nout)
        for (int ii = threadIdx.x >> 7; ii < rows; ii += step) {
            const unsigned d = (unsigned)__cvta_generic_to_shared(tile + ii * MLP_COOP_W + o);
            const T *src = Wt + (long)(i0 + ii) * nout + o;
            if (sizeof(T) == 8) asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(d), "l"(src) : "memory");
            else asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(d), "l"(src) : "memory");
        }
    if ((rows & 1) && (int)threadIdx.x < MLP_COOP_W) tile[rows * MLP_COOP_W + threadIdx.x] = T(0);
}

// acc[e][j][r] += sum over the tile's inputs of weight(input, output lane + 32 j) * activation row r of evaluation e,
// inputs in ascending order per accumulator (as mlp_eval_thread); two inputs per pass, all loads unguarded
template <int NE, int E, typename T>
__device__ __forceinline__ void coop_tile_fma(T (&acc)[E][4][6], const T *tile_lane, const T *act_i0, int rows2)
{
    constexpr int W = MLP_COOP_W;
#pragma unroll 2
    for (int ii = 0; ii < rows2; ii += 2) {
        T w[2][4], h[NE][2][6];
#pragma unroll
        for (int u = 0; u < 2; u++)
#pragma unroll
            for (int j = 0; j < 4; j++) w[u][j] = tile_lane[(ii + u) * W + 32 * j];
#pragma unroll
        for (int e = 0; e < NE; e++)
#pragma unroll
            for (int u = 0; u < 2; u++)
#pragma unroll
                for (int r = 0; r < 6; r++) h[e][u][r] = act_i0[(e * COOP_ROWS + r) * W + ii + u];
#pragma unroll
        for (int e = 0; e < NE; e++)
#pragma unroll
            for (int u = 0; u < 2; u++)
#pragma unroll
                for (int j = 0; j < 4; j++)
#pragma unroll
                    for (int r = 0; r < 6; r++) acc[e][j][r] += w[u][j] * h[e][u][r];
    }
}

// biases of every layer and the output layer's weights of network P -> shared memory (NP: DevParams<T> or MlpNet<T>)
template <typename T, typename NP>
__device__ __forceinline__ void coop_stage(const NP &P, T *bias, T *wlast)
{
    constexpr int W = MLP_COOP_W;
    const int tid = threadIdx.x, nthr = blockDim.x;
    for (int idx = tid; idx < (P.n_layers + 1) * W; idx += nthr) {
        const int l = idx / W, o = idx - l * W;
        if (l < P.n_layers) { if (o < P.dims[l + 1]) bias[idx] = P.b[l][o]; }
        else if (o < P.dims[P.n_layers - 1]) wlast[o] = P.Wt[P.n_layers - 1][o];
    }
}

// the waves of the nv requests list[0 .. nv) through network P (staged by coop_stage); CTA-uniform
template <int CAP, typename T, typename NP>
__device__ __forceinline__ void coop_waves(const NP &P, const T *items, T *res, T *act, T *tiles, const T *bias, const T *wlast,
                                           const int *list, int nv)
{
    constexpr int W = MLP_COOP_W, E = CoopShape<CAP>::E, TI = CoopShape<CAP>::TI;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    for (int wave0 = 0; wave0 < nv; wave0 += nw * E) {             // CTA-uniform
        int ev[E];
#pragma unroll
        for (int e = 0; e < E; e++) { const int idx = wave0 + e * nw + warp; ev[e] = idx < nv ? list[idx] : -1; }   // a thin wave: one per warp
        const bool any = ev[0] >= 0, two = ev[E - 1] >= 0;          // warp-uniform
        if (lane < 6) {   // whitened feature x = Wn ((s_tv, v_tv, e_tv, s_N - s_tv, v_N - v_tv, e_ego - e_tv) - mu_f), mpc.py:326-337
#pragma unroll
            for (int e = 0; e < E; e++)
                if (ev[e] >= 0) {
                    const T *q = items + ev[e] * COOP_ITEM;
                    T *hi = act + e * COOP_ROWS * W;
                    const T xN[6] = { q[2], q[3], q[4], q[0] - q[2], q[1] - q[3], q[5] - q[4] };
                    T a = T(0);
                    for (int j = 0; j < 6; j++) a += P.Wn[lane * 6 + j] * (xN[j] - P.mu_f[j]);
                    hi[0 * W + lane] = a;
                    hi[1 * W + lane] = P.Wn[lane * 6 + 3];
                    hi[2 * W + lane] = P.Wn[lane * 6 + 4];
                    hi[3 * W + lane] = hi[4 * W + lane] = hi[5 * W + lane] = T(0);
                }
        }
        __syncwarp();
        for (int l = 0; l < P.n_layers; l++) {
            const int nin = P.dims[l], nout = P.dims[l + 1];
            const T *Wt = P.Wt[l], *b = bias + l * W;
            if (l < P.n_layers - 1) {
                T acc[E][4][6];
#pragma unroll
                for (int e = 0; e < E; e++)
#pragma unroll
                    for (int j = 0; j < 4; j++) {
                        const int o = lane + 32 * j;
                        acc[e][j][0] = o < nout ? b[o] : T(0);
#pragma unroll
                        for (int r = 1; r < 6; r++) acc[e][j][r] = T(0);
                    }
                const int ntile = (nin + TI - 1) / TI;
                coop_load_tile(tiles, Wt, 0, nin < TI ? nin : TI, nout);
                for (int t = 0; t < ntile; t++) {
                    asm volatile("cp.async.wait_all;" ::: "memory");
                    __syncthreads();                               // tile t has landed; everybody is done with tile t - 1
                    if (t + 1 < ntile) {
                        const int r1 = nin - (t + 1) * TI;
                        coop_load_tile(tiles + ((t + 1) & 1) * TI * W, Wt, (t + 1) * TI, r1 < TI ? r1 : TI, nout);
                    }
                    if (!any) continue;
                    const T *tile_lane = tiles + (t & 1) * TI * W + lane;
                    const int i0 = t * TI, rows = nin - i0 < TI ? nin - i0 : TI, rows2 = (rows + 1) & ~1;
                    if (E > 1 && two) coop_tile_fma<E>(acc, tile_lane, act + i0, rows2);
                    else coop_tile_fma<1>(acc, tile_lane, act + i0, rows2);
                }
                __syncthreads();                                   // the last tile's buffer is free for the next layer's first
                if (any) {
                    __syncwarp();                                  // every lane has read its inputs: the rows are replaced in place
#pragma unroll
                    for (int e = 0; e < E; e++) {
                        if (ev[e] < 0) continue;
                        T *ho = act + e * COOP_ROWS * W;
#pragma unroll
                        for (int j = 0; j < 4; j++) {
                            const int o = lane + 32 * j;
                            if (o < nout) {
                                const T y = tanh(acc[e][j][0]), d1 = T(1) - y * y, d2 = T(-2) * y * d1, ts = acc[e][j][1], tv = acc[e][j][2];
                                ho[0 * W + o] = y;
                                ho[1 * W + o] = d1 * ts;
                                ho[2 * W + o] = d1 * tv;
                                ho[3 * W + o] = d1 * acc[e][j][3] + d2 * ts * ts;
                                ho[4 * W + o] = d1 * acc[e][j][4] + d2 * ts * tv;
                                ho[5 * W + o] = d1 * acc[e][j][5] + d2 * tv * tv;
                            } else {
#pragma unroll
                                for (int r = 0; r < 6; r++) ho[r * W + o] = T(0);
                            }
                        }
                    }
                    __syncwarp();
                }
            } else {                                              // output layer (nout = 1): lane r of the e-th group of six sums row r in input order
                const int e = lane / 6, r = lane - 6 * e;
                int mine = -1;
#pragma unroll
                for (int q = 0; q < E; q++) if (e == q) mine = ev[q];
                if (mine >= 0) {
                    const T *hi = act + e * COOP_ROWS * W;
                    T a = r == 0 ? b[0] : T(0);
                    int i = 0;
                    for (; i + 16 <= nin; i += 16) {               // sixteen inputs' operands loaded ahead of their (ordered) FMAs
                        T wv[16], hv[16];
#pragma unroll
                        for (int u = 0; u < 16; u++) { wv[u] = wlast[i + u]; hv[u] = hi[r * W + i + u]; }
#pragma unroll
                        for (int u = 0; u < 16; u++) a += wv[u] * hv[u];
                    }
                    for (; i < nin; i++) a += wlast[i] * hi[r * W + i];
                    res[mine * COOP_ROWS + r] = r == 0 ? a * P.sigma_t + P.mu_t : a * P.sigma_t;
                }
                __syncwarp();
            }
        }
    }
}

// CTA-uniform call (like mlp_tc_eval): every thread passes its own request (valid = false: none) and gets
// out[6] = (V, dV/ds, dV/dv, d2V/dss, d2V/dsv, d2V/dvv), already scaled by sigma_t (+ mu_t on V).
// Shared memory: mlp_coop_smem_bytes<T, CAP>.
template <typename T, int CAP = 0>
__device__ __noinline__ void mlp_coop_eval(const DevParams<T> &P, uint8_t *smem, bool valid, T sN, T vN, const T *ctx, T *out)
{
    constexpr int W = MLP_COOP_W, E = CoopShape<CAP>::E, TI = CoopShape<CAP>::TI;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, nthr = blockDim.x, nw = nthr >> 5;
    const int ns = CAP ? CAP : nthr, na = CAP ? CAP : nw;       // request slots, warps with activation rows
    T *items = reinterpret_cast<T *>(smem);                       // [slots][8]: sN, vN, ctx[4]
    T *res = items + ns * COOP_ITEM;                              // [slots][6]
    T *act = res + ns * COOP_ROWS + warp * (E * COOP_ROWS * W);   // this warp's [E][6][W] activation rows (updated in place)
    T *tiles = res + ns * COOP_ROWS + na * (E * COOP_ROWS * W);   // [2][TI][W]
    T *bias = tiles + 2 * TI * W, *wlast = bias + MAX_MLP_LAYERS * W;   // [layers][W], [W]: staged once per call
    int *list = reinterpret_cast<int *>(wlast + W), *wcnt = list + ns;
    coop_stage(P, bias, wlast);
    if (CAP == 0 || warp < CAP)
        for (int idx = lane; idx < E * COOP_ROWS * W; idx += 32) act[idx] = T(0);
    if constexpr (CAP == 0) {                                     // slot = thread
        items[tid * COOP_ITEM + 0] = sN; items[tid * COOP_ITEM + 1] = vN;
#pragma unroll
        for (int i = 0; i < 4; i++) items[tid * COOP_ITEM + 2 + i] = ctx[i];
    }
    // the valid requests in thread order
    const unsigned vm = __ballot_sync(0xffffffffu, valid);
    if (lane == 0) wcnt[warp] = __popc(vm);
    __syncthreads();
    int base = 0, nv = 0;
    for (int i = 0; i < nw; i++) { const int c = wcnt[i]; if (i < warp) base += c; nv += c; }
    if constexpr (CAP == 0) {
        if (valid) list[base + __popc(vm & ((1u << lane) - 1u))] = tid;
        __syncthreads();
        coop_waves<CAP>(P, items, res, act, tiles, bias, wlast, list, nv);
        __syncthreads();
        if (valid) {
#pragma unroll
            for (int r = 0; r < 6; r++) out[r] = res[tid * COOP_ROWS + r];
        }
    } else {                                                      // slot = position in the list (at most CAP requests)
        if (nv > CAP) __trap();                                   // (the caller's bound, see the file comment)
        const int sl = base + __popc(vm & ((1u << lane) - 1u));
        if (valid) {
            items[sl * COOP_ITEM + 0] = sN; items[sl * COOP_ITEM + 1] = vN;
#pragma unroll
            for (int i = 0; i < 4; i++) items[sl * COOP_ITEM + 2 + i] = ctx[i];
        }
        if (tid < CAP) list[tid] = tid;
        __syncthreads();
        coop_waves<CAP>(P, items, res, act, tiles, bias, wlast, list, nv);
        __syncthreads();
        if (valid) {
#pragma unroll
            for (int r = 0; r < 6; r++) out[r] = res[sl * COOP_ROWS + r];
        }
    }
    __syncthreads();
}

// one network group of the bank evaluation: nets[g] -> desc and the staged biases, then the waves of list[0 .. n)
template <int CAP, typename T>
__device__ __forceinline__ void coop_bank_group(const MlpNet<T> *nets, int g, MlpNet<T> *desc, const T *items, T *res, T *act,
                                                T *tiles, T *bias, T *wlast, const int *list, int n)
{
    {   // descriptor -> shared memory (the previous group's waves are done with it: barrier at their end)
        const int *src = reinterpret_cast<const int *>(nets + g);
        int *dst = reinterpret_cast<int *>(desc);
        for (int i = threadIdx.x; i < (int)(sizeof(MlpNet<T>) / 4); i += blockDim.x) dst[i] = src[i];
    }
    __syncthreads();
    coop_stage(*desc, bias, wlast);
    __syncthreads();
    coop_waves<CAP>(*desc, items, res, act, tiles, bias, wlast, list, n);
    __syncthreads();
}

// The same over a network bank: request t uses nets[net] (0 <= net < MAX_MLP_NETS, a loaded slot: the callers check).
// Shared memory: mlp_coop_bank_smem_bytes<T, CAP>.
template <typename T, int CAP = 0>
__device__ __noinline__ void mlp_coop_eval_bank(const MlpNet<T> *nets, uint8_t *smem, bool valid, int net, T sN, T vN, const T *ctx, T *out)
{
    constexpr int W = MLP_COOP_W, E = CoopShape<CAP>::E, TI = CoopShape<CAP>::TI;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, nthr = blockDim.x, nw = nthr >> 5;
    const int ns = CAP ? CAP : nthr, na = CAP ? CAP : nw;
    T *items = reinterpret_cast<T *>(smem);
    T *res = items + ns * COOP_ITEM;
    T *act = res + ns * COOP_ROWS + warp * (E * COOP_ROWS * W);
    T *tiles = res + ns * COOP_ROWS + na * (E * COOP_ROWS * W);
    T *bias = tiles + 2 * TI * W, *wlast = bias + MAX_MLP_LAYERS * W;   // staged once per group
    int *list = reinterpret_cast<int *>(wlast + W);
    MlpNet<T> *desc = reinterpret_cast<MlpNet<T> *>(smem + mlp_coop_smem_bytes<T, CAP>(nthr));   // the current group's network
    int *gcnt = reinterpret_cast<int *>(reinterpret_cast<uint8_t *>(desc) + mlp_coop_desc_bytes<T>());   // [net][warp]
    if (CAP == 0 || warp < CAP)
        for (int idx = lane; idx < E * COOP_ROWS * W; idx += 32) act[idx] = T(0);
    if constexpr (CAP == 0) {
        items[tid * COOP_ITEM + 0] = sN; items[tid * COOP_ITEM + 1] = vN;
#pragma unroll
        for (int i = 0; i < 4; i++) items[tid * COOP_ITEM + 2 + i] = ctx[i];
    }
    // counting sort of the valid requests by network: group g holds its requests in thread order
    int rank = 0;
    for (int g = 0; g < MAX_MLP_NETS; g++) {
        const bool mine = valid && net == g;
        const unsigned m = __ballot_sync(0xffffffffu, mine);
        if (lane == 0) gcnt[g * nw + warp] = __popc(m);
        if (mine) rank = __popc(m & ((1u << lane) - 1u));
    }
    __syncthreads();
    if constexpr (CAP == 0) {
        if (valid && (unsigned)net < (unsigned)MAX_MLP_NETS) {
            int base = rank;
            for (int g = 0; g <= net; g++)
                for (int i = 0; i < nw; i++) if (g < net || i < warp) base += gcnt[g * nw + i];
            list[base] = tid;
        }
        __syncthreads();
        for (int g = 0, start = 0; g < MAX_MLP_NETS; g++) {       // CTA-uniform
            int n = 0;
            for (int i = 0; i < nw; i++) n += gcnt[g * nw + i];
            if (n == 0) continue;
            coop_bank_group<CAP>(nets, g, desc, items, res, act, tiles, bias, wlast, list + start, n);
            start += n;
        }
        if (valid) {
#pragma unroll
            for (int r = 0; r < 6; r++) out[r] = res[tid * COOP_ROWS + r];
        }
    } else {                                                      // slot = position in the sorted list (at most CAP requests)
        const bool listed = valid && (unsigned)net < (unsigned)MAX_MLP_NETS;
        int sl = rank;
        if (listed) {
            for (int g = 0; g <= net; g++)
                for (int i = 0; i < nw; i++) if (g < net || i < warp) sl += gcnt[g * nw + i];
            if (sl >= CAP) __trap();
            items[sl * COOP_ITEM + 0] = sN; items[sl * COOP_ITEM + 1] = vN;
#pragma unroll
            for (int i = 0; i < 4; i++) items[sl * COOP_ITEM + 2 + i] = ctx[i];
        }
        if (tid < CAP) list[tid] = tid;
        for (int g = 0, start = 0; g < MAX_MLP_NETS; g++) {       // CTA-uniform (the first group's barriers publish the items)
            int n = 0;
            for (int i = 0; i < nw; i++) n += gcnt[g * nw + i];
            if (n == 0) continue;
            coop_bank_group<CAP>(nets, g, desc, items, res, act, tiles, bias, wlast, list + start, n);
            start += n;
        }
        if (listed) {
#pragma unroll
            for (int r = 0; r < 6; r++) out[r] = res[sl * COOP_ROWS + r];
        }
    }
    __syncthreads();
}
#endif

}  // namespace igt
