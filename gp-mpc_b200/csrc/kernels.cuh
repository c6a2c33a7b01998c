// Device kernels of the GP hot path other than the DMMA GEMM family.
// Reference semantics are cited as file:line of helgeanl/GP-MPC.
#pragma once
#include <type_traits>
#include "common.cuh"

// hyper layout per output (device copy): [ell_0..ell_{Nx-1}, sf, sn]  (gp_class.py:139-142)
#define KB_TILE 64

// ---------------------------------------------------------------------------------------
// a1/a2  K = sf2 exp(-1/2 sum_d ((x_id - x_jd)/ell_d)^2) + (sn2 + jitter) I   (gp_functions.py:17-22,
//   optimize.py:303-319, :342-344), with the pairwise distances on the fp64 TENSOR pipe.
//   With u_i = sqrt(log2 e) (x_i - mu)/ell and q_i = -1/2 |u_i|^2 + 1/2 log2 sf2,
//       log2 k(x_i, x_j) = q_i + q_j + u_i . u_j            (= log2 sf2 - log2(e)/2 |xs_i - xs_j|^2)
//   so the O(N^2 Nx) part is a rank-Nx product done with DMMA m8n8k4 (tensor pipe), leaving the
//   fp64 pipe only ~12 instructions per pair (two adds, clamp, a 256-entry-table exp2 with a
//   degree-4 polynomial).  ncu on the first (direct-difference, libm exp) kernel showed the fp64 pipe 48 % busy and DRAM 41 %:
//   the two pipes now overlap and the kernel becomes write-bandwidth bound.
//   The kernel is translation invariant, so inputs are centred on the column means mu: the
//   expansion's cancellation error is eps*|u|^2 with |u| measured from the data centre
//   (<= 6e-16 relative on both reference fixtures, same as direct differences; the reference's
//   own numpy path uses the un-centred expansion, optimize.py:315-319).
//   One CTA = one 128x128 tile of the lower triangle; off-diagonal tiles also store the
//   mirrored tile (each exp2 serves two outputs).  q_i + q_j and the k-ordered dot product are
//   commutative, so K is bitwise symmetric, including inside diagonal tiles.
// ---------------------------------------------------------------------------------------
// 2^(n/256), n = 0..255, correctly rounded (generated with 40-digit arithmetic)
__constant__ double c_exp2_tab256[256] = {
    1, 1.0027112750502025, 1.0054299011128027, 1.0081558981184175,
    1.0108892860517005, 1.0136300849514894, 1.0163783149109531, 1.0191339960777379,
    1.0218971486541166, 1.0246677928971357, 1.0274459491187637, 1.030231637686041,
    1.0330248790212284, 1.0358256936019572, 1.0386341019613787, 1.0414501246883161,
    1.0442737824274138, 1.0471050958792898, 1.0499440858006872, 1.0527907730046264,
    1.0556451783605572, 1.0585073227945128, 1.0613772272892621, 1.0642549128844645,
    1.0671404006768237, 1.0700337118202419, 1.0729348675259756, 1.075843889062791,
    1.0787607977571199, 1.0816856149932152, 1.0846183622133092, 1.0875590609177697,
    1.0905077326652577, 1.0934643990728858, 1.0964290818163769, 1.0994018026302219,
    1.1023825833078409, 1.1053714457017412, 1.1083684117236787, 1.1113735033448175,
    1.1143867425958924, 1.1174081515673693, 1.1204377524096067, 1.1234755673330199,
    1.1265216186082418, 1.1295759285662881, 1.1326385195987192, 1.1357094141578055,
    1.1387886347566916, 1.1418762039695616, 1.1449721444318042, 1.1480764788401789,
    1.1511892299529827, 1.1543104205902159, 1.1574400736337511, 1.1605782120274988,
    1.1637248587775775, 1.1668800369524817, 1.1700437696832502, 1.1732160801636373,
    1.1763969916502812, 1.1795865274628758, 1.182784710984341, 1.1859915656609938,
    1.189207115002721, 1.1924313825831512, 1.1956643920398273, 1.1989061670743806,
    1.2021567314527031, 1.2054161090051239, 1.2086843236265816, 1.2119613992768012,
    1.215247359980469, 1.2185422298274085, 1.2218460329727576, 1.2251587936371455,
    1.22848053610687, 1.2318112847340759, 1.2351510639369334, 1.2384998981998165,
    1.241857812073484, 1.245224830175258, 1.2486009771892048, 1.2519862778663162,
    1.2553807570246911, 1.2587844395497165, 1.2621973503942507, 1.2656195145788063,
    1.2690509571917332, 1.2724917033894028, 1.275941778396392, 1.2794012075056693,
    1.2828700160787783, 1.2863482295460256, 1.2898358734066657, 1.2933329732290895,
    1.2968395546510096, 1.3003556433796506, 1.3038812651919358, 1.3074164459346773,
    1.3109612115247644, 1.3145155879493546, 1.318079601266064, 1.3216532776031575,
    1.3252366431597413, 1.3288297242059544, 1.3324325470831615, 1.3360451382041458,
    1.3396675240533029, 1.3432997311868353, 1.3469417862329458, 1.3505937158920345,
    1.3542555469368927, 1.3579273062129011, 1.3616090206382248, 1.3653007172040119,
    1.3690024229745905, 1.3727141650876684, 1.3764359707545302, 1.380167867260238,
    1.383909881963832, 1.3876620422985291, 1.3914243757719262, 1.3951969099662003,
    1.3989796725383112, 1.4027726912202048, 1.4065759938190154, 1.4103896082172707,
    1.4142135623730951, 1.4180478843204152, 1.4218926021691656, 1.4257477441054942,
    1.42961333839197, 1.4334894133677889, 1.4373759974489824, 1.4412731191286257,
    1.4451808069770467, 1.449099089642035, 1.4530279958490526, 1.4569675544014438,
    1.460917794180647, 1.4648787441464057, 1.4688504333369818, 1.4728328908693675,
    1.4768261459394993, 1.4808302278224719, 1.4848451658727524, 1.488870989524397,
    1.4929077282912648, 1.4969554117672355, 1.5010140696264256, 1.5050837316234065,
    1.5091644275934228, 1.5132561874526098, 1.5173590411982147, 1.5214730189088146,
    1.5255981507445384, 1.529734466947287, 1.5338819978409559, 1.5380407738316568,
    1.5422108254079407, 1.5463921831410214, 1.550584877685, 1.5547889397770887,
    1.5590044002378369, 1.5632312899713576, 1.567469639965553, 1.5717194812923414,
    1.5759808451078865, 1.5802537626528246, 1.5845382652524937, 1.588834384317164,
    1.593142151342267, 1.5974615979086271, 1.6017927556826934, 1.606135656416771,
    1.6104903319492543, 1.6148568142048607, 1.6192351351948637, 1.6236253270173289,
    1.6280274218573478, 1.632441451987275, 1.6368674497669644, 1.6413054476440063,
    1.6457554781539649, 1.6502175739206177, 1.6546917676561943, 1.6591780921616162,
    1.6636765803267364, 1.6681872651305825, 1.6727101796415966, 1.6772453570178785,
    1.681792830507429, 1.6863526334483934, 1.6909247992693053, 1.6955093614893326,
    1.7001063537185235, 1.7047158096580513, 1.7093377631004629, 1.713972247929926,
    1.7186192981224779, 1.723278947746274, 1.7279512309618377, 1.7326361820223111,
    1.7373338352737062, 1.7420442251551564, 1.746767386199169, 1.7515033530318782,
    1.7562521603732995, 1.7610138430375839, 1.7657884359332727, 1.7705759740635547,
    1.7753764925265212, 1.7801900265154245, 1.785016611318935, 1.789856282321401,
    1.7947090750031072, 1.7995750249405351, 1.8044541678066239, 1.809346539371032,
    1.8142521755003989, 1.8191711121586085, 1.8241033854070534, 1.8290490314048973,
    1.8340080864093424, 1.8389805867758937, 1.843966568958626, 1.8489660695104508,
    1.8539791250833855, 1.8590057724288205, 1.864046048397789, 1.8690999899412386,
    1.8741676341103, 1.8792490180565602, 1.8843441790323345, 1.8894531543909392,
    1.8945759815869656, 1.8997126981765553, 1.9048633418176741, 1.9100279502703899,
    1.9152065613971474, 1.9203992131630474, 1.925605943636125, 1.9308267909876271,
    1.9360617934922943, 1.9413109895286405, 1.9465744175792332, 1.9518521162309783,
    1.9571441241754002, 1.9624504802089273, 1.9677712232331759, 1.9731063922552343,
    1.9784560263879509, 1.9838201648502194, 1.9891988469672663, 1.9945921121709402};

// 2^t for -1020 <= t <= ~1000 (the CALLER clamps: rint(256 t) must fit the low word and the exponent stay normal): 256-entry table + degree-4 polynomial on
// |f| <= 1/512 (truncation 3.8e-17), ~1.7 ulp.  Per value: 2 (rint by magic constant) + 1 (f) +
// 4 (Horner) + table load + multiply + exponent insert -- the r1 kernel (16-entry table, degree 7)
// was bound by issue slots (67 % active), not by HBM.
__device__ __forceinline__ double exp2_t256(double t, const double* __restrict__ T256)
{
    const double SH = 6755399441055744.0;            // 1.5 * 2^52: rint(256 t) lands in the low word
    const double s = fma(t, 256.0, SH);
    const int n = __double2loint(s);
    const double f = fma(s - SH, -0.00390625, t);    // |f| <= 1/512, exact
    double p = 0.009618129107628477;                 // (ln 2)^k / k!, k = 4..1
    p = fma(p, f, 0.05550410866482158);
    p = fma(p, f, 0.24022650695910072);
    p = fma(p, f, 0.6931471805599453);
    p = fma(p, f, 1.0);
    p *= T256[n & 255];
    return __hiloint2double(__double2hiint(p) + ((n >> 8) << 20), __double2loint(p));
}

// same with the 16-entry table (c_exp2_tab, one entry per shared-memory bank => conflict-free) and a
// degree-7 polynomial on |f| <= 1/32
__constant__ double c_exp2_tab[16] = {
    1.0, 1.0442737824274138, 1.0905077326652577, 1.1387886347566916, 1.189207115002721,
    1.241857812073484, 1.2968395546510096, 1.3542555469368927, 1.4142135623730951,
    1.4768261459394993, 1.5422108254079407, 1.6104903319492543, 1.681792830507429,
    1.7562521603732995, 1.8340080864093424, 1.9152065613971474};
__device__ __forceinline__ double exp2_t16(double t, const double* __restrict__ T16)
{
    const double SH = 6755399441055744.0;
    const double s = fma(t, 16.0, SH);
    const int n = __double2loint(s);
    const double f = fma(s - SH, -0.0625, t);        // |f| <= 1/32, exact
    double p = 1.5252733804059838e-05;               // (ln 2)^k / k!, k = 7..1
    p = fma(p, f, 0.00015403530393381606);
    p = fma(p, f, 0.0013333558146428441);
    p = fma(p, f, 0.009618129107628477);
    p = fma(p, f, 0.055504108664821576);
    p = fma(p, f, 0.2402265069591007);
    p = fma(p, f, 0.6931471805599453);
    p = fma(p, f, 1.0);
    p *= T16[n & 15];
    return __hiloint2double(__double2hiint(p) + ((n >> 4) << 20), __double2loint(p));
}

// Two-level table: 2^t = 2^e * T1[(n >> 4) & 15] * T2[n & 15] * 2^f with n = rint(256 t), T1[k] = 2^(k/16), T2[m] = 2^(m/256),
// |f| <= 1/512 (degree-4 polynomial, truncation 3.8e-17).  Both tables have ONE entry per shared-memory bank, so the
// lookups are conflict-free whatever the lane pattern (the flat 256-entry table replays ~3x), and the polynomial needs four
// coefficients instead of seven (each costs two UMOVs in the loop on this target).  ~2.2 ulp.
__constant__ double c_exp2_tab2[16] = {
    1, 1.0027112750502025, 1.0054299011128027, 1.0081558981184175, 1.0108892860517005, 1.0136300849514894,
    1.0163783149109531, 1.0191339960777379, 1.0218971486541166, 1.0246677928971357, 1.0274459491187637,
    1.030231637686041, 1.0330248790212284, 1.0358256936019572, 1.0386341019613787, 1.0414501246883161};
__device__ __forceinline__ double exp2_t2lvl(double t, const double* __restrict__ T32)
{
    const double SH = 6755399441055744.0;            // 1.5 * 2^52: rint(256 t) lands in the low word
    const double s = fma(t, 256.0, SH);
    const int n = __double2loint(s);
    const double f = fma(s - SH, -0.00390625, t);    // |f| <= 1/512, exact
    double p = 0.009618129107628477;                 // (ln 2)^k / k!, k = 4..1
    p = fma(p, f, 0.05550410866482158);
    p = fma(p, f, 0.24022650695910072);
    p = fma(p, f, 0.6931471805599453);
    p = fma(p, f, 1.0);
    p *= T32[(n >> 4) & 15];
    p *= T32[16 + (n & 15)];
    return __hiloint2double(__double2hiint(p) + ((n >> 8) << 20), __double2loint(p));
}

struct KbTrue { __device__ constexpr operator bool() const { return true; } };
struct KbFalse { __device__ constexpr operator bool() const { return false; } };

#define KB2_TILE 128
template <bool FULL>
__global__ void __launch_bounds__(256)
kbuild_dmma_kernel(const double* __restrict__ XT, int ldx, int N, int Nx, const double* __restrict__ mu,
                   const double* __restrict__ hyp, int hyp_ld, const double* __restrict__ jitter,
                   double* __restrict__ K, int ld, long long sK)
{
    extern __shared__ double sm[];
    const int KD = (Nx + 3) & ~3;                         // k extent of the MMA, zero padded
    const int S = ((KD >> 2) & 1) ? KD : KD + 4;          // row stride: S/4 odd => conflict-free frags
    double* Ui = sm;                                      // [128][S]
    double* Uj = Ui + KB2_TILE * S;                       // [128][S]
    double* qi = Uj + KB2_TILE * S;                       // [128]
    double* qj = qi + KB2_TILE;                           // [128]
    double* T256 = qj + KB2_TILE;                         // [256]

    const int a = blockIdx.z;
    const double* hp = hyp + (long long)a * hyp_ld;
    const int tt = blockIdx.x;
    int bi = (int)((sqrt(8.0 * (double)tt + 1.0) - 1.0) * 0.5);
    while (bi * (bi + 1) / 2 > tt) --bi;
    while ((bi + 1) * (bi + 2) / 2 <= tt) ++bi;
    const int bj = tt - bi * (bi + 1) / 2;
    const int i0 = bi * KB2_TILE, j0 = bj * KB2_TILE;
    const int tid = threadIdx.x;
    const double sf2 = hp[Nx] * hp[Nx];
    const double l2sf2 = log2(sf2);

    __shared__ double sc[36], mus[36];                    // sqrt(log2 e) / ell_d and the column means: one division per dimension per CTA
    if (tid < S) {
        sc[tid] = (tid < Nx) ? 1.2011224087864498 / hp[tid] : 0.0;
        mus[tid] = (tid < Nx) ? mu[tid] : 0.0;
    }
    // two 16-entry tables (exp2_t2lvl): conflict-free lookups and a degree-4 polynomial
    if (tid < 16) T256[tid] = c_exp2_tab[tid];
    else if (tid < 32) T256[tid] = c_exp2_tab2[tid - 16];
    __syncthreads();
    {   // scaled, centred coordinates of the 128 row points (tid < 128) / column points
        const int p = (tid < KB2_TILE) ? i0 + tid : j0 + tid - KB2_TILE;
        double* U = (tid < KB2_TILE) ? Ui + tid * S : Uj + (tid - KB2_TILE) * S;
        double nrm = 0.0;
        for (int d = 0; d < S; ++d) {
            double u = 0.0;
            if (d < Nx) u = (XT[(long long)d * ldx + p] - mus[d]) * sc[d];
            U[d] = u;
            nrm = fma(u, u, nrm);
        }
        ((tid < KB2_TILE) ? qi : qj)[tid & (KB2_TILE - 1)] = fma(-0.5, nrm, 0.5 * l2sf2);
    }
    __syncthreads();

    const int warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
    const double dg = hp[Nx + 1] * hp[Nx + 1] + (jitter ? jitter[a] : 0.0);
    double* Ka = K + (long long)a * sK;
    const bool offdiag = (bi != bj);
    const bool mirror = FULL && offdiag;
    // tiles that touch the diagonal or the identity tail take the checked epilogue
    const bool special = !offdiag || (i0 + KB2_TILE > N) || (j0 + KB2_TILE > N);
    const int nk4 = KD >> 2;
    // SP = tile touches the diagonal or the identity tail (checked epilogue, upper clamp); MR = mirrored tile stored too.
    // Both are CTA-uniform.  No fmin/fmax anywhere (their NaN semantics cost ~7 instructions each on this target; a plain
    // compare-select is 3).
    auto tile_body = [&](auto sp_tag, auto mr_tag) {
        const bool SP = sp_tag, MR = mr_tag;      // KbTrue / KbFalse fold at compile time, plain bools stay run-time
#pragma unroll 1
        for (int mi = 0; mi < 2; ++mi) {
            const int rl = warp * 16 + mi * 8 + g;            // local row of this lane's accumulators
            const int row = i0 + rl;
            const double* ua = Ui + rl * S + t;
            const double qr = qi[rl];
            double* drow = Ka + (long long)row * ld + j0 + 2 * t;              // direct:  K[row][j0 + cl]
            double* mcol = Ka + (long long)(j0 + 2 * t) * ld + row;            // mirror:  K[j0 + cl][row]
#pragma unroll 1
            for (int ng = 0; ng < 4; ++ng) {
                double acc[4][2];
#pragma unroll
                for (int q = 0; q < 4; ++q) { acc[q][0] = 0.0; acc[q][1] = 0.0; }
                const double* ub = Uj + (ng * 32 + g) * S + t;
                for (int kk = 0; kk < nk4; ++kk) {
                    const double av = ua[kk * 4];
#pragma unroll
                    for (int q = 0; q < 4; ++q) dmma884(acc[q][0], acc[q][1], av, ub[q * 8 * S + kk * 4]);
                }
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const int cl0 = ng * 32 + q * 8;          // + 2t folded into the base pointers
                    const double2 qc = *reinterpret_cast<const double2*>(qj + cl0 + 2 * t);
                    // log2 k, clamped from below (far-apart points under tiny length scales: SLSQP probes them; 2^-1020 ~ 0)
                    double t0 = (qr + qc.x) + acc[q][0], t1 = (qr + qc.y) + acc[q][1];
                    t0 = (t0 < -1020.0) ? -1020.0 : t0;
                    t1 = (t1 < -1020.0) ? -1020.0 : t1;
                    if (SP) {                                 // k <= sf2 despite rounding: only where the distance can be 0
                        t0 = (t0 > l2sf2) ? l2sf2 : t0;
                        t1 = (t1 > l2sf2) ? l2sf2 : t1;
                    }
                    double v0 = exp2_t2lvl(t0, T256), v1 = exp2_t2lvl(t1, T256);
                    if (SP) {
                        const int col = j0 + cl0 + 2 * t;
                        if (row == col) v0 += dg;
                        if (row == col + 1) v1 += dg;
                        if (row >= N || col >= N) v0 = (row == col) ? 1.0 : 0.0;
                        if (row >= N || col + 1 >= N) v1 = (row == col + 1) ? 1.0 : 0.0;
                    }
                    *reinterpret_cast<double2*>(drow + cl0) = make_double2(v0, v1);
                    if (MR) {
                        double* m = mcol + (long long)cl0 * ld;        // independent address per store pair (no serial pointer chain)
                        m[0] = v0;
                        m[ld] = v1;
                    }
                }
            }
        }
    };
    if (FULL) {
        // store-bound: one body with run-time flags (four specialised copies measured 5 % slower: CTAs of different kinds
        // share an SM and the instruction working set quadruples)
        tile_body(special, mirror);
    } else if (special) {
        tile_body(KbTrue{}, KbFalse{});
    } else {
        tile_body(KbFalse{}, KbFalse{});      // instruction-bound: the hot path carries no checks at all
    }
}

// ---------------------------------------------------------------------------------------
// a3 leaf: 128x128 diagonal block  ->  L (in place, zeros above the diagonal) and L^-1.
//   np.linalg.cholesky at optimize.py:346/485; a non-positive pivot is reported LAPACK
//   style (1-based global index) so the host can apply the reference's single 1e-8
//   jitter retry (optimize.py:347-350).  One CTA per batch entry; whole block in smem.
// ---------------------------------------------------------------------------------------
#define LEAF_N 128
#define LEAF_LD 129
__global__ void __launch_bounds__(256, 1)
leaf_potrf_trtri_kernel(double* __restrict__ A, int lda, long long sA,
                        double* __restrict__ Li, int ldi, long long sLi,
                        int* __restrict__ info, int info_base)
{
    extern __shared__ double S[];           // [128][129]
    __shared__ double colbuf[LEAF_N];
    const int tid = threadIdx.x;
    double* Ab = A + (long long)blockIdx.x * sA;
    double* Lb = Li + (long long)blockIdx.x * sLi;
    for (int idx = tid; idx < LEAF_N * LEAF_N; idx += 256) {
        const int r = idx >> 7, c = idx & 127;
        S[r * LEAF_LD + c] = Ab[(long long)r * lda + c];
    }
    __syncthreads();
    const int tx = tid & 15, ty = tid >> 4;
    for (int j = 0; j < LEAF_N; ++j) {
        const double d = S[j * LEAF_LD + j];
        if (!(d > 0.0) && tid == 0) atomicCAS(info + blockIdx.x, 0, info_base + j + 1);
        const double dj = sqrt(d);
        const double inv = 1.0 / dj;
        __syncthreads();                    // everyone has read the pivot
        if (tid < LEAF_N) {
            if (tid == j) S[j * LEAF_LD + j] = dj;
            else if (tid > j) S[tid * LEAF_LD + j] *= inv;
        }
        __syncthreads();
        for (int i = j + 1 + ty; i < LEAF_N; i += 16) {
            const double lij = S[i * LEAF_LD + j];
            for (int k = j + 1 + tx; k <= i; k += 16)
                S[i * LEAF_LD + k] = fma(-lij, S[k * LEAF_LD + j], S[i * LEAF_LD + k]);
        }
        __syncthreads();
    }
    for (int idx = tid; idx < LEAF_N * LEAF_N; idx += 256) {
        const int r = idx >> 7, c = idx & 127;
        Ab[(long long)r * lda + c] = (c <= r) ? S[r * LEAF_LD + c] : 0.0;
    }
    // in-place lower-triangular inverse, last column first:
    //   Linv[j][j] = 1/L[j][j];  Linv[i][j] = -Linv[j][j] * sum_{k=j+1..i} Linv[i][k] * L[k][j]
    for (int j = LEAF_N - 1; j >= 0; --j) {
        if (tid < LEAF_N && tid > j) colbuf[tid] = S[tid * LEAF_LD + j];
        const double djj = 1.0 / S[j * LEAF_LD + j];
        __syncthreads();
        const int i = j + 1 + (tid >> 1);
        double s0 = 0.0, s1 = 0.0;
        if (i < LEAF_N) {
            int k = j + 1 + (tid & 1);
            for (; k + 2 <= i; k += 4) {
                s0 = fma(S[i * LEAF_LD + k], colbuf[k], s0);
                s1 = fma(S[i * LEAF_LD + k + 2], colbuf[k + 2], s1);
            }
            if (k <= i) s0 = fma(S[i * LEAF_LD + k], colbuf[k], s0);
        }
        double s = s0 + s1;
        s += __shfl_xor_sync(0xffffffffu, s, 1);
        __syncthreads();
        if (i < LEAF_N && (tid & 1) == 0) S[i * LEAF_LD + j] = -djj * s;
        if (tid == 0) S[j * LEAF_LD + j] = djj;
        __syncthreads();
    }
    for (int idx = tid; idx < LEAF_N * LEAF_N; idx += 256) {
        const int r = idx >> 7, c = idx & 127;
        Lb[(long long)r * ldi + c] = (c <= r) ? S[r * LEAF_LD + c] : 0.0;
    }
}

// ---------------------------------------------------------------------------------------
// a3 leaf v2: blocked (nb = 16) Cholesky + triangular inverse of a 128x128 diagonal block,
// entirely in shared memory.  Per block step: one warp factorises and inverts the 16x16
// diagonal block (smem, __syncwarp only); all threads form the panel L21 = A21 D^-T with the
// small inverse; the trailing update and the inverse assembly run on DMMA fragments read
// straight from shared memory (row stride 132 doubles: (g*32 + t*8) mod 128 conflict-free).
// Same outputs / info convention as the v1 kernel (which it replaced: 233 us -> see profiles/).
// ---------------------------------------------------------------------------------------
#define LF_LD 132
// optional phase clock stamps of CTA 0 (diagnostics: gpmpc_profile_leaf)
__device__ long long* d_leaf_prof = nullptr;
#define LEAF_STAMP(k) do { if (d_leaf_prof && blockIdx.x == 0 && threadIdx.x == 0) d_leaf_prof[k] = clock64(); } while (0)
#define LF_NB 16
#define LF_XLD 20
#define LF_SMEM_DOUBLES (LEAF_N * LF_LD + 8 * 16 * 17 + 2 * LEAF_N * LF_XLD)

__device__ __forceinline__ void warp_potrf16_trtri16(double* D, double* Dinv, int* info, int info_val0, int lane)
{
    // D: 16x16 block (lower part valid) with row stride LF_LD; Dinv: [16][17].
    // Register-resident: lane r (and its mirror r+16) holds row r; pivots / multipliers travel
    // by shuffle, so the 16 column steps need no shared-memory round trips.
    const unsigned full = 0xffffffffu;
    const int r = lane & 15;
    double a[16], ipd[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) a[k] = D[r * LF_LD + k];
#pragma unroll
    for (int j = 0; j < 16; ++j) {
        const double d = __shfl_sync(full, a[j], j);
        if (!(d > 0.0) && lane == 0) atomicCAS(info, 0, info_val0 + j + 1);
        // sqrt and reciprocal from one rsqrt + Newton corrections (shorter dependent chain than
        // DSQRT followed by a division; both results are correctly rounded to ~0.5 ulp)
        double y = rsqrt(d);
        double pv = d * y;
        pv = fma(fma(-pv, pv, d), 0.5 * y, pv);
        y = fma(fma(-pv, y, 1.0), y, y);
        if (!(d > 0.0)) { pv = sqrt(d); y = 1.0 / pv; }     // keep NaN/inf propagation of the plain formula
        ipd[j] = y;
        a[j] = (r == j) ? pv : a[j] * ipd[j];              // l_rj for r > j (LAPACK dpotf2 scales by 1/ajj too)
#pragma unroll
        for (int k = j + 1; k < 16; ++k) {
            const double lkj = __shfl_sync(full, a[j], k);
            a[k] = fma(-a[j], lkj, a[k]);                  // meaningful for r >= k; upper part is never read
        }
    }
    __syncwarp();
    if (lane < 16) {
#pragma unroll
        for (int k = 0; k < 16; ++k) if (k <= r) D[r * LF_LD + k] = a[k];
    }
    // column r of the inverse by forward substitution; L[i][k] is broadcast from lane i
    double x[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        double sacc = 0.0;
#pragma unroll
        for (int k = 0; k < i; ++k) sacc = fma(__shfl_sync(full, a[k], i), x[k], sacc);
        x[i] = (i < r) ? 0.0 : ((i == r) ? ipd[i] : -sacc * ipd[i]);
        if (lane < 16) Dinv[i * 17 + r] = x[i];
    }
    __syncwarp();
}

__global__ void __launch_bounds__(256, 1)
leaf_potrf_trtri_v2_kernel(double* __restrict__ A, int lda, long long sA,
                           double* __restrict__ Li, int ldi, long long sLi,
                           int* __restrict__ info, int info_base)
{
    extern __shared__ __align__(16) double S[];                // [128][132]
    double* DinvAll = S + LEAF_N * LF_LD;                      // [8][16][17]
    double* Xs = DinvAll + 8 * 16 * 17;                        // scratch for the inverse assembly (2 x 128 x 20 doubles)
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
    double* Ab = A + (long long)blockIdx.x * sA;
    double* Lb = Li + (long long)blockIdx.x * sLi;
    LEAF_STAMP(0);
    for (int idx = tid; idx < LEAF_N * LEAF_N; idx += 256) {
        const int r = idx >> 7, c = idx & 127;
        S[r * LF_LD + c] = Ab[(long long)r * lda + c];
    }
    __syncthreads();
    LEAF_STAMP(1);

    // ---------------- Cholesky, right-looking, nb = 16, with look-ahead ----------------
    // After the panel of step kb only the next block column is updated by everyone (C1); then warp 0
    // factorises + inverts the next diagonal block WHILE warps 1..7 finish the trailing update (C2).
    auto panel = [&](int c0, const double* Dinv) {
        // P[r][j] = sum_{k<=j} A[r][c0+k] * Dinv[j][k]; two threads per row (8 columns each)
        const int nbel = LEAF_N - c0 - LF_NB;
        const int rr = tid >> 1, half = tid & 1;
        double a[16];
        if (rr < nbel) {
            const double* src = S + (c0 + LF_NB + rr) * LF_LD + c0;
#pragma unroll
            for (int k = 0; k < 16; ++k) a[k] = src[k];
        }
        __syncwarp();
        if (rr < nbel) {
            double* dst = S + (c0 + LF_NB + rr) * LF_LD + c0;
#pragma unroll
            for (int jj = 0; jj < 8; ++jj) {
                const int j = half * 8 + jj;
                double sacc = 0.0;
#pragma unroll
                for (int k = 0; k < 16; ++k) if (k <= j) sacc = fma(a[k], Dinv[j * 17 + k], sacc);
                dst[j] = sacc;
            }
        }
    };
    auto update_tile = [&](int c0, int ti, int tj) {      // C(8x8 at tile ti,tj of the trailing block) -= P_R P_C^T
        const int R0 = c0 + LF_NB + 8 * ti, C0 = c0 + LF_NB + 8 * tj;
        double* cp = S + (R0 + g) * LF_LD + C0 + 2 * t;
        double acc0 = cp[0], acc1 = cp[1];
        const double* pa = S + (R0 + g) * LF_LD + c0 + t;
        const double* pb = S + (C0 + g) * LF_LD + c0 + t;
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) dmma884(acc0, acc1, -pa[kk * 4], pb[kk * 4]);
        cp[0] = acc0; cp[1] = acc1;
    };
    if (warp == 0) warp_potrf16_trtri16(S, DinvAll, info + blockIdx.x, info_base, lane);
    __syncthreads();
    panel(0, DinvAll);
    __syncthreads();
    LEAF_STAMP(2);
    for (int kb = 0; kb < 7; ++kb) {
        const int c0 = kb * LF_NB, b0 = c0 + LF_NB;
        const int nt8 = (LEAF_N - b0) >> 3;
        // C1: the two 8-wide tile columns of the next block column
        for (int tl = warp; tl < 2 * nt8; tl += 8) {
            const int ti = tl >> 1, tj = tl & 1;
            if (tj <= ti) update_tile(c0, ti, tj);
        }
        __syncthreads();
        if (warp == 0) {
            warp_potrf16_trtri16(S + b0 * LF_LD + b0, DinvAll + (kb + 1) * 16 * 17, info + blockIdx.x, info_base + b0, lane);
        } else {
            // C2: tiles 2 <= tj <= ti < nt8 on warps 1..7
            const int m = nt8 - 2;
            const int ntile = m > 0 ? m * (m + 1) / 2 : 0;
            for (int tl = warp - 1; tl < ntile; tl += 7) {
                int ti = (int)((sqrtf(8.0f * (float)tl + 1.0f) - 1.0f) * 0.5f);
                while (ti * (ti + 1) / 2 > tl) --ti;
                while ((ti + 1) * (ti + 2) / 2 <= tl) ++ti;
                const int tj = tl - ti * (ti + 1) / 2;
                update_tile(c0, ti + 2, tj + 2);
            }
        }
        __syncthreads();
        panel(b0, DinvAll + (kb + 1) * 16 * 17);
        __syncthreads();
        LEAF_STAMP(3 + kb);
    }
    for (int idx = tid; idx < LEAF_N * LEAF_N; idx += 256) {
        const int r = idx >> 7, c = idx & 127;
        Ab[(long long)r * lda + c] = (c <= r) ? S[r * LF_LD + c] : 0.0;
    }
    __syncthreads();
    LEAF_STAMP(10);

    // ---------------- triangular inverse by recursive doubling ----------------
    // the 16x16 diagonal inverses are known; for s = 16, 32, 64 every aligned pair of inverted
    // blocks [A^-1 (p..p+s), C^-1 (p+s..p+2s)] is completed with  X = -C^-1 (B A^-1)  written over
    // B = L[p+s.., p..] in place: 3 levels x 2 DMMA products instead of 8 sequential block columns
    {
        const int r = tid >> 4, c = tid & 15;               // 16 x 16 threads
        for (int kb = 0; kb < 8; ++kb)                      // exact zeros above the diagonal: DMMA k-ranges read them
            S[(kb * 16 + r) * LF_LD + kb * 16 + c] = (c <= r) ? DinvAll[kb * 16 * 17 + r * 17 + c] : 0.0;
    }
    __syncthreads();
    double* T1 = Xs;                                        // [pairs][s][s+4], at most 4096+ doubles (Xs and Ys are adjacent)
    for (int sz = 16; sz < LEAF_N; sz <<= 1) {
        const int npair = LEAF_N / (2 * sz), t8 = sz >> 3, ldt = sz + 4;
        const int ntile = npair * t8 * t8;
        // T1 = B * Ainv   (Ainv lower: k >= j)
        for (int tl = warp; tl < ntile; tl += 8) {
            const int pr = tl / (t8 * t8), ti = (tl / t8) % t8, tj = tl % t8;
            const int p0 = pr * 2 * sz;
            const double* pa = S + (p0 + sz + 8 * ti + g) * LF_LD + p0 + t;            // B rows
            const double* pb = S + (p0 + t) * LF_LD + p0 + 8 * tj + g;                 // Ainv[k][n]
            double a0 = 0.0, a1 = 0.0;
            for (int k0 = 8 * tj; k0 < sz; k0 += 4) dmma884(a0, a1, pa[k0], pb[k0 * LF_LD]);
            double* tp = T1 + pr * sz * ldt + (8 * ti + g) * ldt + 8 * tj + 2 * t;
            tp[0] = a0; tp[1] = a1;
        }
        __syncthreads();
        // X = -Cinv * T1  (Cinv lower: k <= i), written over B
        for (int tl = warp; tl < ntile; tl += 8) {
            const int pr = tl / (t8 * t8), ti = (tl / t8) % t8, tj = tl % t8;
            const int p0 = pr * 2 * sz;
            const double* pa = S + (p0 + sz + 8 * ti + g) * LF_LD + p0 + sz + t;       // Cinv rows
            const double* pb = T1 + pr * sz * ldt + t * ldt + 8 * tj + g;              // T1[k][n]
            double a0 = 0.0, a1 = 0.0;
            for (int k0 = 0; k0 < 8 * ti + 8; k0 += 4) dmma884(a0, a1, -pa[k0], pb[k0 * ldt]);
            double* xp = S + (p0 + sz + 8 * ti + g) * LF_LD + p0 + 8 * tj + 2 * t;
            xp[0] = a0; xp[1] = a1;
        }
        __syncthreads();
        LEAF_STAMP(sz == 16 ? 11 : (sz == 32 ? 12 : 13));
    }
    for (int idx = tid; idx < LEAF_N * LEAF_N; idx += 256) {
        const int r = idx >> 7, c = idx & 127;
        Lb[(long long)r * ldi + c] = (c <= r) ? S[r * LF_LD + c] : 0.0;
    }
    LEAF_STAMP(14);
}

// ---------------------------------------------------------------------------------------
// a3 leaf v3.  Same contract as v2; the 128-pivot dependency chain is the only thing left on
// the critical path (r2b profile of v2: 74 us = 140k cycles, of which the warp-level 16x16
// potrf+trtri 35 %, the Dinv panel products 13 %, the block load 10 %, the serial inverse
// assembly 16 %):
//   * per 16-column block step the chain is  potrf16 (warp 0, registers + shuffles, fp32-seeded
//     rsqrt: ~170 cycles per pivot)  ->  panel by FORWARD SUBSTITUTION with the 16x16 factor (one
//     thread per row, the factor is broadcast from shared memory; no 16x16 inverse needed)  ->
//     DMMA update of the next block column;
//   * everything else runs beside it: warps 2..7 finish the trailing update of the previous step
//     and warp 1 inverts the previous 16x16 diagonal block (needed only by the inverse assembly)
//     while warp 0 factorises the next one;
//   * the triangular inverse is assembled by recursive doubling with four independent DMMA
//     accumulator chains per warp (v2 ran one dependent chain per 8x8 tile);
//   * 16-byte global loads / stores.
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ double rsqrt_seeded(double d)
{
    // rsqrt.approx.f64 (SASS MUFU.RSQ64H on the high word, ~2^-22, no fp32 round trip) + two Newton steps in
    // fp64: relative error ~1e-15; tiny / huge / non-positive arguments take the library routine
    if (!(d > 1e-290 && d < 1e290)) return rsqrt(d);
    double y;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(d));
    double e = fma(-(d * y), y, 1.0);
    y = fma(0.5 * y, e, y);
    e = fma(-(d * y), y, 1.0);
    y = fma(0.5 * y, e, y);
    return y;
}

// 16x16 Cholesky in registers (lane r and r+16 hold row r); writes the factor back (lower part) and
// the reciprocal pivots to ipd[16]
__device__ __forceinline__ void warp_potrf16(double* D, double* ipd, int* info, int info_val0, int lane)
{
    const unsigned full = 0xffffffffu;
    const int r = lane & 15;
    double a[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) a[k] = D[r * LF_LD + k];
#pragma unroll
    for (int j = 0; j < 16; ++j) {
        const double d = __shfl_sync(full, a[j], j);
        if (!(d > 0.0) && lane == 0) atomicCAS(info, 0, info_val0 + j + 1);
        double y = rsqrt_seeded(d);
        double pv = d * y;
        pv = fma(fma(-pv, pv, d), 0.5 * y, pv);             // sqrt(d) to ~0.5 ulp
        if (!(d > 0.0)) { pv = sqrt(d); y = 1.0 / pv; }     // keep NaN/inf propagation of the plain formula
        a[j] = (r == j) ? pv : a[j] * y;
        if (lane == 0) ipd[j] = y;
#pragma unroll
        for (int k = j + 1; k < 16; ++k) {
            const double lkj = __shfl_sync(full, a[j], k);
            a[k] = fma(-a[j], lkj, a[k]);                  // meaningful for r >= k; upper part is never read
        }
    }
    __syncwarp();                                           // lanes 16..31 read the same rows above (ordered by the shuffles; explicit for racecheck)
    if (lane < 16) {
#pragma unroll
        for (int k = 0; k < 16; ++k) if (k <= r) D[r * LF_LD + k] = a[k];
    }
    __syncwarp();
}

// Same contract, TWO columns per step: the pivots' reciprocal square roots are the longest dependent chain
// of the whole factorisation (~9 dependent fp64 operations at ~40 cycles each per pivot).  For columns
// j, j+1 with Schur-complement entries p = S_jj, q = S_j+1,j, r = S_j+1,j+1 the second pivot is
// s = r - q^2/p = det/p with det = p r - q^2, so  1/sqrt(s) = rsqrt(det) * sqrt(p):  rsqrt(p) and rsqrt(det)
// are independent and run concurrently -- 11 dependent operations per two pivots instead of 18.  Arithmetic is
// the standard Cholesky recurrence (same stability: s inherits the relative error eps p r / det either way).
__device__ __forceinline__ void warp_potrf16x2(double* D, double* ipd, int* info, int info_val0, int lane)
{
    const unsigned full = 0xffffffffu;
    const int r = lane & 15;
    double a[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) a[k] = D[r * LF_LD + k];
#pragma unroll
    for (int j = 0; j < 16; j += 2) {
        const double p = __shfl_sync(full, a[j], j);
        const double q = __shfl_sync(full, a[j], j + 1);
        const double rr = __shfl_sync(full, a[j + 1], j + 1);
        const double det = fma(p, rr, -(q * q));
        if (lane == 0) {
            if (!(p > 0.0)) atomicCAS(info, 0, info_val0 + j + 1);
            else if (!(det > 0.0)) atomicCAS(info, 0, info_val0 + j + 2);
        }
        double yp = rsqrt_seeded(p), yd = rsqrt_seeded(det);            // independent chains
        double sp = p * yp;
        sp = fma(fma(-sp, sp, p), 0.5 * yp, sp);                         // sqrt(p)
        if (!(p > 0.0)) { sp = sqrt(p); yp = 1.0 / sp; }
        const double c21 = q * yp;                                       // L[j+1][j]
        double ys = yd * sp;                                             // 1 / sqrt(s)
        const double s2 = fma(-c21, c21, rr);                            // s by the standard formula: diagonal entry only (off the chain)
        double ss = s2 * ys;
        ss = fma(fma(-ss, ss, s2), 0.5 * ys, ss);                        // sqrt(s)
        if (!(det > 0.0) || !(p > 0.0)) { ss = sqrt(s2); ys = 1.0 / ss; }
        const double lj = (r == j) ? sp : a[j] * yp;                     // column j
        const double t = fma(-lj, c21, a[j + 1]);
        const double lj1 = (r == j + 1) ? ss : t * ys;                   // column j+1 (row j: above the diagonal, never read)
        a[j] = lj; a[j + 1] = lj1;
        if (lane == 0) { ipd[j] = yp; ipd[j + 1] = ys; }
#pragma unroll
        for (int k = j + 2; k < 16; ++k) {
            const double lkj = __shfl_sync(full, lj, k);
            const double lkj1 = __shfl_sync(full, lj1, k);
            a[k] = fma(-lj1, lkj1, fma(-lj, lkj, a[k]));               // meaningful for r >= k
        }
    }
    __syncwarp();
    if (lane < 16) {
#pragma unroll
        for (int k = 0; k < 16; ++k) if (k <= r) D[r * LF_LD + k] = a[k];
    }
    __syncwarp();
}

// inverse of a factorised 16x16 block (off the critical path): lane r computes column r by forward
// substitution; two partial sums shorten the dependent FMA chain
__device__ __forceinline__ void warp_trtri16(const double* D, const double* ipd, double* Dinv, int lane)
{
    const int r = lane & 15;
    double x[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        double s0 = 0.0, s1 = 0.0;
#pragma unroll
        for (int k = 0; k < i; ++k) {
            const double l = D[i * LF_LD + k];              // broadcast read
            if (k & 1) s1 = fma(l, x[k], s1); else s0 = fma(l, x[k], s0);
        }
        const double ip = ipd[i];
        x[i] = (i < r) ? 0.0 : ((i == r) ? ip : -(s0 + s1) * ip);
        if (lane < 16) Dinv[i * 17 + r] = x[i];
    }
}

#define LF3_SMEM_DOUBLES (LEAF_N * LF_LD + 8 * 16 * 17 + 8 * 16 + 64 * 68 + 64)
template <bool TWOCOL>
__global__ void __launch_bounds__(256, 1)
leaf_potrf_trtri_v3_kernel(double* __restrict__ A, int lda, long long sA,
                           double* __restrict__ Li, int ldi, long long sLi,
                           int* __restrict__ info, int info_base)
{
    extern __shared__ __align__(16) double S[];                // [128][132]
    double* DinvAll = S + LEAF_N * LF_LD;                      // [8][16][17]
    double* ipdAll = DinvAll + 8 * 16 * 17;                    // [8][16] reciprocal pivots
    double* T1 = ipdAll + 8 * 16;                              // inverse-assembly scratch: npair x sz x (sz+4) <= 64 x 68
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
    double* Ab = A + (long long)blockIdx.x * sA;
    double* Lb = Li + (long long)blockIdx.x * sLi;
    LEAF_STAMP(0);
    {   // 128 x 128 block -> shared memory, 16-byte loads, 16 in flight per thread
        double2 v[16];
#pragma unroll
        for (int half = 0; half < 2; ++half) {
#pragma unroll
            for (int q = 0; q < 16; ++q) {
                const int idx = tid + 256 * (q + 16 * half);       // double2 index: row = idx >> 6, col2 = idx & 63
                v[q] = *reinterpret_cast<const double2*>(Ab + (long long)(idx >> 6) * lda + 2 * (idx & 63));
            }
#pragma unroll
            for (int q = 0; q < 16; ++q) {
                const int idx = tid + 256 * (q + 16 * half);
                *reinterpret_cast<double2*>(S + (idx >> 6) * LF_LD + 2 * (idx & 63)) = v[q];
            }
        }
    }
    __syncthreads();
    LEAF_STAMP(1);

    auto panel = [&](int c0, const double* ipd) {
        // rows below the diagonal block: x = a D^-T by forward substitution (x_j = (a_j - sum_{k<j} x_k L_jk)/L_jj)
        const int rr = c0 + LF_NB + tid;
        if (rr < LEAF_N) {
            double* row = S + rr * LF_LD + c0;
            const double* Dk = S + c0 * LF_LD + c0;
            double a[16];
#pragma unroll
            for (int k = 0; k < 16; ++k) a[k] = row[k];
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                a[j] *= ipd[j];
#pragma unroll
                for (int k = j + 1; k < 16; ++k) a[k] = fma(-a[j], Dk[k * LF_LD + j], a[k]);
            }
#pragma unroll
            for (int k = 0; k < 16; ++k) row[k] = a[k];
        }
    };
    auto update_tile = [&](int c0, int ti, int tj) {      // C(8x8 at tile ti,tj of the trailing block) -= P_R P_C^T
        const int R0 = c0 + LF_NB + 8 * ti, C0 = c0 + LF_NB + 8 * tj;
        double* cp = S + (R0 + g) * LF_LD + C0 + 2 * t;
        double acc0 = cp[0], acc1 = cp[1];
        const double* pa = S + (R0 + g) * LF_LD + c0 + t;
        const double* pb = S + (C0 + g) * LF_LD + c0 + t;
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) dmma884(acc0, acc1, -pa[kk * 4], pb[kk * 4]);
        cp[0] = acc0; cp[1] = acc1;
    };
    if (warp == 0) {
        if (TWOCOL) warp_potrf16x2(S, ipdAll, info + blockIdx.x, info_base, lane);
        else warp_potrf16(S, ipdAll, info + blockIdx.x, info_base, lane);
    }
    __syncthreads();
    panel(0, ipdAll);
    __syncthreads();
    LEAF_STAMP(2);
    for (int kb = 0; kb < 7; ++kb) {
        const int c0 = kb * LF_NB, b0 = c0 + LF_NB;
        const int nt8 = (LEAF_N - b0) >> 3;
        // C1: the two 8-wide tile columns of the next block column
        for (int tl = warp; tl < 2 * nt8; tl += 8) {
            const int ti = tl >> 1, tj = tl & 1;
            if (tj <= ti) update_tile(c0, ti, tj);
        }
        __syncthreads();
        if (warp == 0) {
            if (TWOCOL) warp_potrf16x2(S + b0 * LF_LD + b0, ipdAll + (kb + 1) * 16, info + blockIdx.x, info_base + b0, lane);
            else warp_potrf16(S + b0 * LF_LD + b0, ipdAll + (kb + 1) * 16, info + blockIdx.x, info_base + b0, lane);
        } else if (warp == 1) {
            warp_trtri16(S + c0 * LF_LD + c0, ipdAll + kb * 16, DinvAll + kb * 16 * 17, lane);
        } else {
            // C2: tiles 2 <= tj <= ti < nt8 on warps 2..7
            const int m = nt8 - 2;
            const int ntile = m > 0 ? m * (m + 1) / 2 : 0;
            for (int tl = warp - 2; tl < ntile; tl += 6) {
                int ti = (int)((sqrtf(8.0f * (float)tl + 1.0f) - 1.0f) * 0.5f);
                while (ti * (ti + 1) / 2 > tl) --ti;
                while ((ti + 1) * (ti + 2) / 2 <= tl) ++ti;
                const int tj = tl - ti * (ti + 1) / 2;
                update_tile(c0, ti + 2, tj + 2);
            }
        }
        __syncthreads();
        panel(b0, ipdAll + (kb + 1) * 16);
        __syncthreads();
        LEAF_STAMP(3 + kb);
    }
    if (warp == 1) warp_trtri16(S + 112 * LF_LD + 112, ipdAll + 7 * 16, DinvAll + 7 * 16 * 17, lane);
    // L out (exact zeros above the diagonal), 16-byte stores; warp 1 joins after its last 16x16 inverse
    for (int idx = tid; idx < LEAF_N * LEAF_N / 2; idx += 256) {
        const int r = idx >> 6, c = 2 * (idx & 63);
        double2 v = *reinterpret_cast<const double2*>(S + r * LF_LD + c);
        if (c > r) v.x = 0.0;
        if (c + 1 > r) v.y = 0.0;
        *reinterpret_cast<double2*>(Ab + (long long)r * lda + c) = v;
    }
    __syncthreads();
    LEAF_STAMP(10);

    // ---------------- triangular inverse by recursive doubling ----------------
    {
        const int r = tid >> 4, c = tid & 15;               // 16 x 16 threads
        for (int kb = 0; kb < 8; ++kb)                      // exact zeros above the diagonal: DMMA k-ranges read them
            S[(kb * 16 + r) * LF_LD + kb * 16 + c] = (c <= r) ? DinvAll[kb * 16 * 17 + r * 17 + c] : 0.0;
    }
    __syncthreads();
    for (int sz = 16; sz < LEAF_N; sz <<= 1) {
        const int npair = LEAF_N / (2 * sz), t8 = sz >> 3, ldt = sz + 4;
        const int gw = (t8 < 4) ? t8 : 4;                   // tiles per group (same tile row, consecutive tile columns)
        const int ngrp = npair * t8 * (t8 / gw);
        // T1 = B * Ainv   (Ainv lower: k >= j; the group starts at its first column's k)
        for (int gi = warp; gi < ngrp; gi += 8) {
            const int per = t8 * (t8 / gw);
            const int pr = gi / per, rem = gi % per, ti = rem / (t8 / gw), tj0 = (rem % (t8 / gw)) * gw;
            const int p0 = pr * 2 * sz;
            const double* pa = S + (p0 + sz + 8 * ti + g) * LF_LD + p0 + t;            // B rows
            const double* pb = S + (p0 + t) * LF_LD + p0 + 8 * tj0 + g;                // Ainv[k][n]
            double acc[4][2];
#pragma unroll
            for (int q = 0; q < 4; ++q) { acc[q][0] = 0.0; acc[q][1] = 0.0; }
            for (int k0 = 8 * tj0; k0 < sz; k0 += 4) {
                const double av = pa[k0];
#pragma unroll
                for (int q = 0; q < 4; ++q)       // column tile tj0+q only has k >= 8 (tj0+q): above that Ainv is zero by
                    if (q < gw && k0 >= 8 * (tj0 + q))   // structure, but the storage there holds stale values
                        dmma884(acc[q][0], acc[q][1], av, pb[k0 * LF_LD + 8 * q]);
            }
#pragma unroll
            for (int q = 0; q < 4; ++q)
                if (q < gw) {
                    double* tp = T1 + pr * sz * ldt + (8 * ti + g) * ldt + 8 * (tj0 + q) + 2 * t;
                    tp[0] = acc[q][0]; tp[1] = acc[q][1];
                }
        }
        __syncthreads();
        // X = -Cinv * T1  (Cinv lower: k <= i), written over B
        for (int gi = warp; gi < ngrp; gi += 8) {
            const int per = t8 * (t8 / gw);
            const int pr = gi / per, rem = gi % per, ti = rem / (t8 / gw), tj0 = (rem % (t8 / gw)) * gw;
            const int p0 = pr * 2 * sz;
            const double* pa = S + (p0 + sz + 8 * ti + g) * LF_LD + p0 + sz + t;       // Cinv rows
            const double* pb = T1 + pr * sz * ldt + t * ldt + 8 * tj0 + g;             // T1[k][n]
            double acc[4][2];
#pragma unroll
            for (int q = 0; q < 4; ++q) { acc[q][0] = 0.0; acc[q][1] = 0.0; }
            for (int k0 = 0; k0 < 8 * ti + 8; k0 += 4) {
                const double av = -pa[k0];
#pragma unroll
                for (int q = 0; q < 4; ++q)
                    if (q < gw) dmma884(acc[q][0], acc[q][1], av, pb[k0 * ldt + 8 * q]);
            }
#pragma unroll
            for (int q = 0; q < 4; ++q)
                if (q < gw) {
                    double* xp = S + (p0 + sz + 8 * ti + g) * LF_LD + p0 + 8 * (tj0 + q) + 2 * t;
                    xp[0] = acc[q][0]; xp[1] = acc[q][1];
                }
        }
        __syncthreads();
        LEAF_STAMP(sz == 16 ? 11 : (sz == 32 ? 12 : 13));
    }
    for (int idx = tid; idx < LEAF_N * LEAF_N / 2; idx += 256) {
        const int r = idx >> 6, c = 2 * (idx & 63);
        double2 v = *reinterpret_cast<const double2*>(S + r * LF_LD + c);
        if (c > r) v.x = 0.0;
        if (c + 1 > r) v.y = 0.0;
        *reinterpret_cast<double2*>(Lb + (long long)r * ldi + c) = v;
    }
    LEAF_STAMP(14);
}

// batched 2-D copy  dst[b][r][c] = src[b][r][c]   (cols multiple of 2, 16-byte aligned)
__global__ void copy2d_kernel(const double* __restrict__ src, int lds, long long ss,
                              double* __restrict__ dst, int ldd, long long sd, int rows, int cols)
{
    const double* s = src + (long long)blockIdx.z * ss;
    double* d = dst + (long long)blockIdx.z * sd;
    const int c2 = cols >> 1;
    for (int r = blockIdx.y; r < rows; r += gridDim.y)
        for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < c2; c += gridDim.x * blockDim.x)
            reinterpret_cast<double2*>(d + (long long)r * ldd)[c] =
                reinterpret_cast<const double2*>(s + (long long)r * lds)[c];
}

// U = Linv^T for the lower tiles of Linv (32x32 smem transpose); U's strictly lower
// tiles are never written and stay zero from allocation.
__global__ void transpose_lower_kernel(const double* __restrict__ Li, double* __restrict__ U, int ld, int nt32)
{
    __shared__ double tile[32][33];
    const int bi = blockIdx.y, bj = blockIdx.x;
    if (bj > bi) return;
    const int tx = threadIdx.x, ty = threadIdx.y;   // 32 x 8
    for (int r = ty; r < 32; r += 8) tile[r][tx] = Li[(long long)(bi * 32 + r) * ld + bj * 32 + tx];
    __syncthreads();
    for (int r = ty; r < 32; r += 8) U[(long long)(bj * 32 + r) * ld + bi * 32 + tx] = tile[tx][r];
    if (bj < bi)      // keep U exactly upper-triangular (the buffer doubles as a staging area)
        for (int r = ty; r < 32; r += 8) U[(long long)(bi * 32 + r) * ld + bj * 32 + tx] = 0.0;
}

// w = T * y with T lower-triangular (one warp per row).   a5: alpha = L^-T (L^-1 y)
__global__ void trmv_lower_kernel(const double* __restrict__ T, int ld, long long sT,
                                  const double* __restrict__ y, long long sy,
                                  double* __restrict__ w, long long sw, int n)
{
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= n) return;
    const double* Tr = T + (long long)blockIdx.z * sT + (long long)row * ld;
    const double* yy = y + (long long)blockIdx.z * sy;
    double s = 0.0;
    for (int k = lane; k <= row; k += 32) s = fma(Tr[k], yy[k], s);
    s = warp_sum(s);
    if (lane == 0) w[(long long)blockIdx.z * sw + row] = s;
}

// out = T^T * w with T lower-triangular: out[k] = sum_{i>=k} T[i][k] w[i]; 32 columns per CTA
__global__ void __launch_bounds__(256)
trmv_lower_T_kernel(const double* __restrict__ T, int ld, long long sT,
                    const double* __restrict__ w, long long sw,
                    double* __restrict__ out, long long so, int n)
{
    __shared__ double red[8][33];
    const int lane = threadIdx.x & 31, wp = threadIdx.x >> 5;
    const int k = blockIdx.x * 32 + lane;
    const double* Tb = T + (long long)blockIdx.z * sT;
    const double* ww = w + (long long)blockIdx.z * sw;
    double s = 0.0;
    for (int i = blockIdx.x * 32 + wp; i < n; i += 8)
        if (i >= k) s = fma(Tb[(long long)i * ld + k], ww[i], s);
    red[wp][lane] = s;
    __syncthreads();
    if (wp == 0) {
        double r = 0.0;
#pragma unroll
        for (int q = 0; q < 8; ++q) r += red[q][lane];
        out[(long long)blockIdx.z * so + k] = r;
    }
}

// out = T^T * w in row chunks of TRT_ROWS: grid (n/32, ceil(n/TRT_ROWS), batch); block (k-block, c)
// sums rows [c*TRT_ROWS, (c+1)*TRT_ROWS) of its 32 columns into P[batch][c][k].  Chunks entirely
// above the diagonal are skipped; the consumer sums chunks c >= k/TRT_ROWS in ascending order
// (deterministic).  The one-block-per-32-columns kernel above needs N/32 >= #SMs*4 to fill the GPU
// (244 us at N=4096); this one has N^2/16384 blocks.
#define TRT_ROWS 512
__global__ void __launch_bounds__(256)
trmv_lower_T_part_kernel(const double* __restrict__ T, int ld, long long sT,
                         const double* __restrict__ w, long long sw,
                         double* __restrict__ P, long long sP, int n)
{
    __shared__ double red[8][33];
    const int lane = threadIdx.x & 31, wp = threadIdx.x >> 5;
    const int k0 = blockIdx.x * 32, c = blockIdx.y;
    const int r1 = min(n, (c + 1) * TRT_ROWS);
    if (r1 <= k0) return;
    const int r0 = max(c * TRT_ROWS, k0);
    const int k = k0 + lane;
    const double* Tb = T + (long long)blockIdx.z * sT;
    const double* ww = w + (long long)blockIdx.z * sw;
    double s = 0.0;
    for (int i = r0 + wp; i < r1; i += 8)
        if (i >= k) s = fma(Tb[(long long)i * ld + k], ww[i], s);
    red[wp][lane] = s;
    __syncthreads();
    if (wp == 0) {
        double r = 0.0;
#pragma unroll
        for (int q = 0; q < 8; ++q) r += red[q][lane];
        P[(long long)blockIdx.z * sP + (long long)c * n + k] = r;
    }
}

// alpha[k] = sum of the row-chunk partials; res[0] = 2 sum_i log L_ii (a4, optimize.py:352), res[1] = y . alpha
__global__ void __launch_bounds__(1024)
alpha_logdet_kernel(const double* __restrict__ P, long long sP, int nch,
                    const double* __restrict__ L, int ld, long long sL,
                    const double* __restrict__ y, long long sy,
                    double* __restrict__ al, long long sal, int n, double* __restrict__ res)
{
    __shared__ double r0[32], r1[32];
    const double* Lb = L + (long long)blockIdx.x * sL;
    const double* Pb = P + (long long)blockIdx.x * sP;
    double s0 = 0.0, s1 = 0.0;
    for (int i = threadIdx.x; i < n; i += 1024) {
        double a = 0.0;
        for (int c = i / TRT_ROWS; c < nch; ++c) a += Pb[(long long)c * n + i];
        al[(long long)blockIdx.x * sal + i] = a;
        s0 += log(fabs(Lb[(long long)i * ld + i]));
        s1 = fma(y[(long long)blockIdx.x * sy + i], a, s1);
    }
    s0 = warp_sum(s0); s1 = warp_sum(s1);
    if ((threadIdx.x & 31) == 0) { r0[threadIdx.x >> 5] = s0; r1[threadIdx.x >> 5] = s1; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double a = 0.0, b = 0.0;
        for (int q = 0; q < 32; ++q) { a += r0[q]; b += r1[q]; }
        res[2 * blockIdx.x] = 2.0 * a;
        res[2 * blockIdx.x + 1] = b;
    }
}

// per batch entry: res[0] = sum_i log(L_ii) * 2 (a4, optimize.py:352), res[1] = y . alpha
__global__ void __launch_bounds__(256)
logdet_dot_kernel(const double* __restrict__ L, int ld, long long sL,
                  const double* __restrict__ y, long long sy,
                  const double* __restrict__ al, long long sal, int n, double* __restrict__ res)
{
    __shared__ double r0[8], r1[8];
    const double* Lb = L + (long long)blockIdx.x * sL;
    double s0 = 0.0, s1 = 0.0;
    for (int i = threadIdx.x; i < n; i += 256) {
        s0 += log(fabs(Lb[(long long)i * ld + i]));
        s1 = fma(y[(long long)blockIdx.x * sy + i], al[(long long)blockIdx.x * sal + i], s1);
    }
    s0 = warp_sum(s0); s1 = warp_sum(s1);
    if ((threadIdx.x & 31) == 0) { r0[threadIdx.x >> 5] = s0; r1[threadIdx.x >> 5] = s1; }
    __syncthreads();
    if (threadIdx.x == 0) {
        double a = 0.0, b = 0.0;
        for (int q = 0; q < 8; ++q) { a += r0[q]; b += r1[q]; }
        res[2 * blockIdx.x] = 2.0 * a;
        res[2 * blockIdx.x + 1] = b;
    }
}

// ---------------------------------------------------------------------------------------
// a8/a9 stage 1: ks, partial mean and partial Jacobian for every (output, test point).
//   ks_i = covSE(X_i, z)               gp_functions.py:114-117,132
//   mean = ks^T alpha                  gp_functions.py:119-120,135
//   J_d  = sum_i alpha_i ks_i (X_id - z_d)/ell_d^2   (closed form of ca.jacobian, :146-147)
//   KST[a][h][i] (h-major) is the A operand of the v = Linv ks tensor-core product; rows h >= H are zero-filled.
// One CTA = 8 test points x CH training points of one output.  A thread owns ONE test point (lane / 4) and every 32nd
// training point of the chunk (subset 4 warp + lane % 4) for the whole loop, so the mean / Jacobian partial sums stay in
// its registers and are reduced across lanes and warps ONCE per CTA.  (The r2 mid-round kernel looped test points per CTA
// and ran a 13-value warp reduction per test point: ~260 instructions per covariance evaluation, 23 us at one C5 output
// and 113 us at eight; this shape needs ~70.)  The chunk of X^T is staged in shared memory pre-scaled by 1/ell
// (dimension-major: staging stores and the broadcast reads are both conflict-free), alpha next to it; a quarter-warp
// reads 4 consecutive training points, a warp stores 8 rows x 32 B of KS^T per step.
// grid (Npad/CH, BM/8, outputs); PMJ[a][h][blk][1 + Nx].
// ---------------------------------------------------------------------------------------
template <int NXP, int CH, int UNR>
__global__ void __launch_bounds__(256, (NXP <= 12 ? 2 : 1))
ks_tile_kernel(const double* __restrict__ XT, int ldx, int N, int Nx,
               const double* __restrict__ hyp, int hyp_ld,
               const double* __restrict__ alpha, long long sal,
               const double* __restrict__ Z, int H,
               double* __restrict__ KST, int ldk, long long sK,
               double* __restrict__ PMJ, int nblk)
{
    extern __shared__ double sm[];                         // xs[NXP][CH] (x / ell), als[CH]
    __shared__ double red[8][8][NXP + 1];
    __shared__ double ie[NXP], zs[8][NXP], T32s[32], l2sf2_s;
    double* xs = sm;
    double* als = sm + NXP * CH;
    // let the dependent product kernel start launching once every CTA of this grid is resident (it waits
    // for this grid's completion before reading KS^T): hides its launch latency and prologue
    asm volatile("griddepcontrol.launch_dependents;");
    const int a = blockIdx.z, rg = blockIdx.y, blk = blockIdx.x, tid = threadIdx.x;
    const int lane = tid & 31, warp = tid >> 5;
    const int i0 = blk * CH;
    const double* hp = hyp + (long long)a * hyp_ld;
    // every global load of the prologue is issued before the first dependent instruction (in-order issue: a
    // load -> scale -> store loop pays one L2 round trip per iteration, 20 iterations = 8 us at C5)
    constexpr int RP = (CH + 255) / 256;
    double xv[RP][NXP], av[RP];
#pragma unroll
    for (int q = 0; q < RP; ++q) {
        const int rr = tid + 256 * q;
        const bool in = (CH % 256 == 0 || rr < CH) && (i0 + rr < N);
#pragma unroll
        for (int d = 0; d < NXP; ++d) xv[q][d] = (in && d < Nx) ? XT[(long long)d * ldx + i0 + rr] : 0.0;
        av[q] = in ? alpha[(long long)a * sal + i0 + rr] : 0.0;
    }
    if (tid < NXP) ie[tid] = (tid < Nx) ? 1.0 / hp[tid] : 0.0;
    if (tid >= 64 && tid < 80) T32s[tid - 64] = c_exp2_tab[tid - 64];
    else if (tid >= 80 && tid < 96) T32s[tid - 64] = c_exp2_tab2[tid - 80];
    if (tid == 96) l2sf2_s = 2.0 * log2(fabs(hp[Nx]));
    for (int idx = tid; idx < 8 * NXP; idx += 256) {       // Z may live in mapped host memory: one read per CTA
        const int rr = idx / NXP, d = idx - rr * NXP, hh = rg * 8 + rr;
        zs[rr][d] = (hh < H && d < Nx) ? Z[(long long)hh * Nx + d] : 0.0;
    }
    __syncthreads();
#pragma unroll
    for (int q = 0; q < RP; ++q) {
        const int rr = tid + 256 * q;
        if (CH % 256 == 0 || rr < CH) {
#pragma unroll
            for (int d = 0; d < NXP; ++d) xs[d * CH + rr] = xv[q][d] * ie[d];
            als[rr] = av[q];
        }
    }
    const int r = lane >> 2, s = warp * 4 + (lane & 3);
    const int h = rg * 8 + r;
    const bool active = h < H;
    double z[NXP], aj[NXP], am = 0.0;
#pragma unroll
    for (int d = 0; d < NXP; ++d) {
        z[d] = zs[r][d] * ie[d];
        aj[d] = 0.0;
    }
    const double l2sf2 = l2sf2_s;
    __syncthreads();
    double* krow = KST + (long long)a * sK + (long long)h * ldk + i0;
    if (active) {
#pragma unroll UNR
        for (int il = s; il < CH; il += 32) {
            double df[NXP], d0 = 0.0, d1 = 0.0;
#pragma unroll
            for (int d = 0; d < NXP; d += 2) {
                df[d] = xs[d * CH + il] - z[d];
                df[d + 1] = xs[(d + 1) * CH + il] - z[d + 1];
                d0 = fma(df[d], df[d], d0);
                d1 = fma(df[d + 1], df[d + 1], d1);
            }
            // sf2 exp(-dist/2) = 2^(log2 sf2 - log2(e)/2 dist) with the two-level table exp2 of the K build (~2 ulp)
            double te = fma(-0.72134752044448170, d0 + d1, l2sf2);
            te = (te < -1020.0) ? -1020.0 : te;
            double ks = exp2_t2lvl(te, T32s);
            if (i0 + il >= N) ks = 0.0;
            const double w = als[il] * ks;
            am += w;
#pragma unroll
            for (int d = 0; d < NXP; ++d) aj[d] = fma(w, df[d], aj[d]);
            if (i0 + il < ldk) krow[il] = ks;
        }
    } else {
        for (int il = s; il < CH; il += 32)
            if (i0 + il < ldk) krow[il] = 0.0;               // padding rows of the A operand: zeros
    }
    // one reduction per CTA: the 4 subsets of a row inside the warp, then the 8 warps through shared memory
    am += __shfl_xor_sync(0xffffffffu, am, 1);
    am += __shfl_xor_sync(0xffffffffu, am, 2);
#pragma unroll
    for (int d = 0; d < NXP; ++d) {
        aj[d] += __shfl_xor_sync(0xffffffffu, aj[d], 1);
        aj[d] += __shfl_xor_sync(0xffffffffu, aj[d], 2);
    }
    if ((lane & 3) == 0) {
        red[warp][r][0] = am;
#pragma unroll
        for (int d = 0; d < NXP; ++d) red[warp][r][d + 1] = aj[d];
    }
    __syncthreads();
    if (tid < 8 * (Nx + 1)) {
        const int rr = tid / (Nx + 1), f = tid - rr * (Nx + 1), hh = rg * 8 + rr;
        double sacc = ((red[0][rr][f] + red[1][rr][f]) + (red[2][rr][f] + red[3][rr][f])) +
                      ((red[4][rr][f] + red[5][rr][f]) + (red[6][rr][f] + red[7][rr][f]));
        if (f > 0) sacc *= ie[f - 1];                        // df was scaled by 1/ell: one more 1/ell makes (x - z)/ell^2
        if (hh < H) PMJ[(((long long)a * H + hh) * nblk + blk) * (Nx + 1) + f] = sacc;
    }
}

// ---------------------------------------------------------------------------------------
// a6/a7 analytic NLML gradient, fused with a K rebuild so dK/dtheta is never stored:
//   dNLL/dtheta = 1/2 tr((K^-1 - alpha alpha^T) dK/dtheta)   (R&W eq. 5.9; objective of
//   optimize.py:322-356).  theta = [ell.., sf, sn] are standard deviations (q1):
//   dK/dell_d = Kf (x_id-x_jd)^2/ell_d^3,  dK/dsf = 2 Kf/sf,  dK/dsn = 2 sn I.
//   One CTA per 64x64 lower tile of K^-1; partial sums [tile][Nx+2].
// ---------------------------------------------------------------------------------------
template <int NXP>
__global__ void __launch_bounds__(256)
nlml_grad_kernel(const double* __restrict__ XT, int ldx, int N, int Nx,
                 const double* __restrict__ hp, const double* __restrict__ Kinv, int ld,
                 const double* __restrict__ alpha, double* __restrict__ partial)
{
    extern __shared__ double sm[];
    double* Xi = sm; double* Xj = sm + Nx * KB_TILE;
    __shared__ double red[8][NXP + 2];
    const int tt = blockIdx.x;
    int bi = (int)((sqrt(8.0 * (double)tt + 1.0) - 1.0) * 0.5);
    while (bi * (bi + 1) / 2 > tt) --bi;
    while ((bi + 1) * (bi + 2) / 2 <= tt) ++bi;
    const int bj = tt - bi * (bi + 1) / 2;
    const int i0 = bi * KB_TILE, j0 = bj * KB_TILE;
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    for (int idx = tid; idx < Nx * KB_TILE; idx += 256) {
        const int d = idx / KB_TILE, r = idx % KB_TILE;
        Xi[idx] = XT[(long long)d * ldx + i0 + r];
        Xj[idx] = XT[(long long)d * ldx + j0 + r];
    }
    __syncthreads();
    const double sf2 = hp[Nx] * hp[Nx];
    double g[NXP + 2];
#pragma unroll
    for (int d = 0; d < NXP + 2; ++d) g[d] = 0.0;
    double ie2[NXP];
#pragma unroll
    for (int d = 0; d < NXP; ++d) ie2[d] = (d < Nx) ? 1.0 / (hp[d] * hp[d]) : 0.0;
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const int row = i0 + ty + 16 * r;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const int col = j0 + tx + 16 * c;
            if (row >= N || col >= N || col > row) continue;
            double dist = 0.0, d2[NXP];
#pragma unroll
            for (int d = 0; d < NXP; ++d) {
                d2[d] = 0.0;
                if (d < Nx) {
                    const double df = Xi[d * KB_TILE + ty + 16 * r] - Xj[d * KB_TILE + tx + 16 * c];
                    d2[d] = df * df;
                    dist = fma(d2[d], ie2[d], dist);
                }
            }
            const double kf = sf2 * exp(-0.5 * dist);
            const double w = Kinv[(long long)row * ld + col] - alpha[row] * alpha[col];
            const double mult = (row == col) ? 1.0 : 2.0;
            const double wk = mult * w * kf;
#pragma unroll
            for (int d = 0; d < NXP; ++d) g[d] = fma(wk, d2[d], g[d]);
            g[NXP] += wk;
            if (row == col) g[NXP + 1] += w;
        }
    }
#pragma unroll
    for (int d = 0; d < NXP + 2; ++d) g[d] = warp_sum(g[d]);
    if ((tid & 31) == 0) {
#pragma unroll
        for (int d = 0; d < NXP + 2; ++d) red[tid >> 5][d] = g[d];
    }
    __syncthreads();
    if (tid < Nx + 2) {
        const int src = (tid < Nx) ? tid : (NXP + (tid - Nx));
        double s = 0.0;
        for (int q = 0; q < 8; ++q) s += red[q][src];
        partial[(long long)tt * (Nx + 2) + tid] = s;
    }
}

// deterministic column sums of partial[ntile][m] -> grad[m], with the theta scalings
__global__ void __launch_bounds__(256)
nlml_grad_final_kernel(const double* __restrict__ partial, int ntile, int Nx,
                       const double* __restrict__ hp, double* __restrict__ grad)
{
    __shared__ double red[8];
    const int q = blockIdx.x;
    double s = 0.0;
    for (int t = threadIdx.x; t < ntile; t += 256) s += partial[(long long)t * (Nx + 2) + q];
    s = warp_sum(s);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        double r = 0.0;
        for (int w = 0; w < 8; ++w) r += red[w];
        if (q < Nx) r = 0.5 * r / (hp[q] * hp[q] * hp[q]);
        else if (q == Nx) r = 0.5 * r * 2.0 / hp[Nx];
        else r = 0.5 * r * 2.0 * hp[Nx + 1];
        grad[q] = r;
    }
}

// extract an N x N block out of a padded slab; mode 0 = as is, 1 = lower triangle with
// exact zeros above the diagonal (the stored-model convention, SURVEY 8a-a3),
// 2 = symmetric from the lower triangle
__global__ void extract_kernel(const double* __restrict__ src, int ld, double* __restrict__ dst, int N, int mode)
{
    const int c = blockIdx.x * blockDim.x + threadIdx.x, r = blockIdx.y;
    if (c >= N) return;
    double v;
    if (mode == 1) v = (c <= r) ? src[(long long)r * ld + c] : 0.0;
    else if (mode == 2) v = (c <= r) ? src[(long long)r * ld + c] : src[(long long)c * ld + r];
    else v = src[(long long)r * ld + c];
    dst[(long long)r * N + c] = v;
}

// Gram matrix of the solved columns: out[a][h1][h2] = sf2_a - sum_i V[a][h1][i] V[a][h2][i]
// (GP.covar, gp_class.py:380: kss - v.T @ v with the scalar kss).  grid (H, H, outputs).
__global__ void __launch_bounds__(256)
gram_cov_kernel(const double* __restrict__ V, int ldv, long long sV, int n,
                const double* __restrict__ hyp, int hyp_ld, int Nx, int H, double* __restrict__ out)
{
    __shared__ double red[8];
    const int a = blockIdx.z, h1 = blockIdx.y, h2 = blockIdx.x;
    if (h2 > h1) return;                                   // symmetric: lower half computed, both written
    const double* v1 = V + (long long)a * sV + (long long)h1 * ldv;
    const double* v2 = V + (long long)a * sV + (long long)h2 * ldv;
    double s = 0.0;
    for (int i = threadIdx.x; i < n; i += 256) s = fma(v1[i], v2[i], s);
    s = warp_sum(s);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        double r = 0.0;
        for (int q = 0; q < 8; ++q) r += red[q];
        const double sf = hyp[(long long)a * hyp_ld + Nx];
        const double c = sf * sf - r;
        out[((long long)a * H + h1) * H + h2] = c;
        out[((long long)a * H + h2) * H + h1] = c;
    }
}

// ---------------------------------------------------------------------------------------
// 'EM' exact moment matching  (gp_exact_moment, gp_functions.py:344-418), one test point
// per launch set.  Host prepares the Nx x Nx quantities (gpmpc.cu, em_prepare_point):
//   per output a :  iR_a = (Sigma + Lambda_a)^-1 ,  c_a = sf2_a prod(ell_a) / sqrt(det(Sigma+Lambda_a))
//   per pair a>=b:  Qm = (Sigma (iL_a+iL_b) + I)^-1 Sigma/2 ,  t_ab = det(...)^-1/2
// EMP layout (doubles): [a: iR (Nx*Nx), c, G_a (Nx*Nx), lc_a] * Ny, then [pair: Qm (Nx*Nx), t, a, b, const_ab] * npairs
// ---------------------------------------------------------------------------------------
template <int NXP>
__global__ void __launch_bounds__(256)
em_prep_kernel(const double* __restrict__ XT, int ldx, int N, int Nx, int Ny, int npairs,
               const double* __restrict__ hyp, int hyp_ld, const double* __restrict__ alpha, long long sal,
               const double* __restrict__ z, const double* __restrict__ EMP,
               double* __restrict__ meanPart, int nblk,
               double* __restrict__ E, double* __restrict__ F, double* __restrict__ W, double* __restrict__ IJ, int ldn,
               double* __restrict__ LQ, double* __restrict__ E2, double* __restrict__ F2)
{
    __shared__ double M[NXP * NXP], Ga[NXP * NXP], Gb[NXP * NXP];
    __shared__ double red[8];
    const int role = blockIdx.y, tid = threadIdx.x;
    const int i = blockIdx.x * 256 + tid;
    const int nn = Nx * Nx;
    double v[NXP];
#pragma unroll
    for (int d = 0; d < NXP; ++d) v[d] = (d < Nx && i < N) ? XT[(long long)d * ldx + i] - z[d] : 0.0;
    if (role < Ny) {                                        // mean of output a (:381-388)
        const int a = role;
        const double* P = EMP + (long long)a * (2 * nn + 2);
        for (int q = tid; q < nn; q += 256) M[q] = P[q];
        __syncthreads();
        double quad = 0.0;
#pragma unroll
        for (int d = 0; d < NXP; ++d) {
            if (d < Nx) {
                double tacc = 0.0;
#pragma unroll
                for (int e = 0; e < NXP; ++e) if (e < Nx) tacc = fma(M[d * Nx + e], v[e], tacc);
                quad = fma(v[d], tacc, quad);
            }
        }
        // log q_i = log c_a - 1/2 v^T (Sigma+Lambda_a)^-1 v: kept so the pair sums can form
        // t Q_ij - q_i q_j = q_i q_j expm1(.) without cancellation (em_pair_kernel)
        if (i < ldn) LQ[(long long)a * ldn + i] = (i < N) ? log(P[nn]) - 0.5 * quad : 0.0;
        double q = (i < N) ? P[nn] * exp(-0.5 * quad) * alpha[(long long)a * sal + i] : 0.0;
        q = warp_sum(q);
        if ((tid & 31) == 0) red[tid >> 5] = q;
        __syncthreads();
        if (tid == 0) {
            double r = 0.0;
            for (int w = 0; w < 8; ++w) r += red[w];
            meanPart[(long long)a * nblk + blockIdx.x] = r;
        }
        return;
    }
    const int p = role - Ny;
    const double* P = EMP + (long long)Ny * (2 * nn + 2) + (long long)p * (nn + 4);
    const int a = (int)P[nn + 1], b = (int)P[nn + 2];
    for (int q = tid; q < nn; q += 256) {
        M[q] = P[q];
        Ga[q] = EMP[(long long)a * (2 * nn + 2) + nn + 1 + q];      // G_a = Lambda_a^-1 Sigma (Sigma + Lambda_a)^-1
        Gb[q] = EMP[(long long)b * (2 * nn + 2) + nn + 1 + q];
    }
    __syncthreads();
    if (i >= ldn) return;
    const double* ha = hyp + (long long)a * hyp_ld;
    const double* hb = hyp + (long long)b * hyp_ld;
    double lka = 2.0 * log(ha[Nx]), lkb = 2.0 * log(hb[Nx]);      // log_k (:389-391)
    double ii[NXP], ij[NXP];
#pragma unroll
    for (int d = 0; d < NXP; ++d) {
        ii[d] = 0.0; ij[d] = 0.0;
        if (d < Nx) {
            const double sa = v[d] / ha[d], sb = v[d] / hb[d];
            lka = fma(-0.5 * sa, sa, lka); lkb = fma(-0.5 * sb, sb, lkb);
            ii[d] = v[d] / (ha[d] * ha[d]); ij[d] = v[d] / (hb[d] * hb[d]);
        }
    }
    // e2 / f2: the SMALL parts only, for the cancellation-free pair sums:
    //   log(t Q_ij) - log q_i - log q_j = const_ab + e2_i + f2_j + 2 ii^T M ij,
    //   e2_i = ii^T M ii - 1/2 v^T G_a v   (log k_a(x_i) - log q^a_i = const - 1/2 v^T G_a v by Woodbury)
    double e2 = 0.0, f2 = 0.0;
#pragma unroll
    for (int e = 0; e < NXP; ++e) {
        if (e < Nx) {
            double wi = 0.0, wj = 0.0, ga = 0.0, gb = 0.0;
#pragma unroll
            for (int d = 0; d < NXP; ++d)
                if (d < Nx) {
                    wi = fma(ii[d], M[d * Nx + e], wi); wj = fma(ij[d], M[d * Nx + e], wj);
                    ga = fma(v[d], Ga[d * Nx + e], ga); gb = fma(v[d], Gb[d * Nx + e], gb);
                }
            e2 = fma(wi, ii[e], e2); f2 = fma(wj, ij[e], f2);
            e2 = fma(-0.5 * ga, v[e], e2); f2 = fma(-0.5 * gb, v[e], f2);
            W[((long long)p * Nx + e) * ldn + i] = wi;
            IJ[((long long)p * Nx + e) * ldn + i] = ij[e];
        }
    }
    // E / F (with the big log k terms) serve the Q matrix of the trace term only
    double ei = lka, fj = lkb;
#pragma unroll
    for (int e = 0; e < NXP; ++e)
        if (e < Nx) {
            double wi = 0.0, wj = 0.0;
#pragma unroll
            for (int d = 0; d < NXP; ++d) if (d < Nx) { wi = fma(ii[d], M[d * Nx + e], wi); wj = fma(ij[d], M[d * Nx + e], wj); }
            ei = fma(wi, ii[e], ei); fj = fma(wj, ij[e], fj);
        }
    E[(long long)p * ldn + i] = ei;
    F[(long long)p * ldn + i] = fj;
    E2[(long long)p * ldn + i] = (i < N) ? e2 : 0.0;
    F2[(long long)p * ldn + i] = (i < N) ? f2 : 0.0;
}

// sum_ij beta_a,i beta_b,j (t Q_ij - q_i q_j) for one pair; 64x64 tile per CTA, 4x4 per thread (:394-416).
// The reference subtracts invK from beta beta^T on the diagonal pairs before the sum (:410-411),
// which cancels 6-8 digits at cond(K) ~ 1e8-1e10 (negative variances on the car fixture, SURVEY
// q18).  Here that term is evaluated separately and stably as tr(L^-1 Q L^-T) (em_q_kernel +
// DMMA product + em_trdot_kernel): a trace of a positive semi-definite matrix, formed from the
// Cholesky factor like var = sf2 - |L^-1 ks|^2 -- no explicit K^-1 anywhere.
// mode 0: partial sums of beta_i beta_j q_ij into `part`; mode 1: q_ij itself into Qout (ld ldq,
// zero outside N) for the pair's output a == b.
__global__ void __launch_bounds__(256)
em_pair_kernel(int N, int Nx, int Ny, const double* __restrict__ EMP,
               const double* __restrict__ alpha, long long sal,
               const double* __restrict__ E, const double* __restrict__ F, const double* __restrict__ W,
               const double* __restrict__ IJ, int ldn, const double* __restrict__ LQ,
               const double* __restrict__ E2, const double* __restrict__ F2, double* __restrict__ part,
               int mode, int pair_q, double* __restrict__ Qout, int ldq)
{
    extern __shared__ double sm[];
    double* Ws = sm; double* Js = sm + Nx * 64;
    __shared__ double red[8];
    const int p = mode ? pair_q : blockIdx.z, nn = Nx * Nx;
    const double* P = EMP + (long long)Ny * (2 * nn + 2) + (long long)p * (nn + 4);
    const int a = (int)P[nn + 1], b = (int)P[nn + 2];
    const double cab = P[nn + 3];       // log t + (log sf2_a - log c_a) + (log sf2_b - log c_b), from determinants of I + small
    const int i0 = blockIdx.y * 64, j0 = blockIdx.x * 64;
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    for (int idx = tid; idx < Nx * 64; idx += 256) {
        const int d = idx >> 6, r = idx & 63;
        Ws[idx] = (i0 + r < ldn) ? W[((long long)p * Nx + d) * ldn + i0 + r] : 0.0;
        Js[idx] = (j0 + r < ldn) ? IJ[((long long)p * Nx + d) * ldn + j0 + r] : 0.0;
    }
    __syncthreads();
    double acc[4][4];
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int c = 0; c < 4; ++c) acc[r][c] = 0.0;
    for (int d = 0; d < Nx; ++d) {
        double wv[4], jv[4];
#pragma unroll
        for (int r = 0; r < 4; ++r) wv[r] = Ws[d * 64 + ty + 16 * r];
#pragma unroll
        for (int c = 0; c < 4; ++c) jv[c] = Js[d * 64 + tx + 16 * c];
#pragma unroll
        for (int r = 0; r < 4; ++r)
#pragma unroll
            for (int c = 0; c < 4; ++c) acc[r][c] = fma(wv[r], jv[c], acc[r][c]);
    }
    double s = 0.0;
#pragma unroll
    for (int r = 0; r < 4; ++r) {
        const int i = i0 + ty + 16 * r;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const int j = j0 + tx + 16 * c;
            const double lq = (i < N && j < N) ? E[(long long)p * ldn + i] + F[(long long)p * ldn + j] + 2.0 * acc[r][c] : 0.0;
            // mode 1 stores only the part of Q beyond its rank-one backbone: Q_ij = e^{E_i} e^{F_j} (1 + expm1(2 acc_ij));
            // the backbone's trace term |L^-1 e^E|^2 is formed like the ME variance (em_qvec_kernel + trmv), which keeps
            // EM -> ME exact to ~1e-11 as Sigma -> 0 instead of amplifying the full Q through L^-1 twice
            if (mode) { if (i < ldq && j < ldq) Qout[(long long)i * ldq + j] = (i < N && j < N) ? exp(E[(long long)p * ldn + i] + F[(long long)p * ldn + j]) * expm1(2.0 * acc[r][c]) : 0.0; }
            else if (i < N && j < N) {
                // beta_i beta_j (t Q_ij - q_i q_j) = (beta_i q_i)(beta_j q_j) expm1(log t + log Q_ij - log q_i - log q_j):
                // the reference's  t beta^T Q beta - mean_a mean_b  (:412,416) term by term, before the sums cancel
                const double la = LQ[(long long)a * ldn + i], lb = LQ[(long long)b * ldn + j];
                const double wgt = (alpha[(long long)a * sal + i] * exp(la)) * (alpha[(long long)b * sal + j] * exp(lb));
                // the exponent is assembled from its small parts only (never as a difference of O(10) logarithms)
                s = fma(wgt, expm1(cab + E2[(long long)p * ldn + i] + F2[(long long)p * ldn + j] + 2.0 * acc[r][c]), s);
            }
        }
    }
    if (mode) return;
    s = warp_sum(s);
    if ((tid & 31) == 0) red[tid >> 5] = s;
    __syncthreads();
    if (tid == 0) {
        double r = 0.0;
        for (int w = 0; w < 8; ++w) r += red[w];
        part[((long long)p * gridDim.y + blockIdx.y) * gridDim.x + blockIdx.x] = r;
    }
}

// rank-one backbone of Q_aa: qv_i = exp(E_i) (i < N, else 0)
__global__ void em_qvec_kernel(const double* __restrict__ E, int N, int n, double* __restrict__ qv)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) qv[i] = (i < N) ? exp(E[i]) : 0.0;
}

// out[0] = sum_i v_i^2 (single block, fixed order)
__global__ void __launch_bounds__(256)
sumsq_kernel(const double* __restrict__ v, int n, double* __restrict__ out)
{
    __shared__ double red[8];
    double s = 0.0;
    for (int i = threadIdx.x; i < n; i += 256) s = fma(v[i], v[i], s);
    s = warp_sum(s);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        double r = 0.0;
        for (int w = 0; w < 8; ++w) r += red[w];
        out[0] = r;
    }
}

// tr(L^-1 Q L^-T) = sum_{k >= j} Wm[k][j] Li[k][j] with Wm = L^-1 Q (lower tiles): block partial sums,
// grid (n/64 * (n/64+1)/2) lower 64x64 tiles
__global__ void __launch_bounds__(256)
em_trdot_kernel(const double* __restrict__ Wm, const double* __restrict__ Li, int ld, double* __restrict__ part)
{
    __shared__ double red[8];
    const int tt = blockIdx.x;
    int bi = (int)((sqrt(8.0 * (double)tt + 1.0) - 1.0) * 0.5);
    while (bi * (bi + 1) / 2 > tt) --bi;
    while ((bi + 1) * (bi + 2) / 2 <= tt) ++bi;
    const int bj = tt - bi * (bi + 1) / 2;
    const int tid = threadIdx.x, tx = tid & 63, ty = tid >> 6;
    double s = 0.0;
    for (int r = ty; r < 64; r += 4) {
        const int row = bi * 64 + r, col = bj * 64 + tx;
        if (col <= row) s = fma(Wm[(long long)row * ld + col], Li[(long long)row * ld + col], s);
    }
    s = warp_sum(s);
    if ((tid & 31) == 0) red[tid >> 5] = s;
    __syncthreads();
    if (tid == 0) {
        double r = 0.0;
        for (int w = 0; w < 8; ++w) r += red[w];
        part[tt] = r;
    }
}

// mean (Ny), cov (Ny,Ny): t_ab * sum (+ sf2 on the diagonal) - mean mean^T   (:412-416)
__global__ void em_finalize_kernel(int Nx, int Ny, int npairs, const double* __restrict__ EMP,
                                   const double* __restrict__ hyp, int hyp_ld,
                                   const double* __restrict__ meanPart, int nblk,
                                   const double* __restrict__ part, int ntile2,
                                   const double* __restrict__ trPart, int ntr, const double* __restrict__ trVec,
                                   double* __restrict__ mean, double* __restrict__ var, double* __restrict__ cov)
{
    __shared__ double mu[64];
    const int tid = threadIdx.x, nn = Nx * Nx;
    if (tid < Ny) {
        double s = 0.0;
        for (int b = 0; b < nblk; ++b) s += meanPart[(long long)tid * nblk + b];
        mu[tid] = s;
        if (mean) mean[tid] = s;
    }
    __syncthreads();
    if (tid < npairs) {
        const double* P = EMP + (long long)Ny * (2 * nn + 2) + (long long)tid * (nn + 4);
        const int a = (int)P[nn + 1], b = (int)P[nn + 2];
        double s = 0.0;
        for (int q = 0; q < ntile2; ++q) s += part[(long long)tid * ntile2 + q];
        double c = s;       // = t beta_a^T Q beta_b - mean_a mean_b, summed term by term without the cancellation
        if (a == b) {
            // + expected variance  sf2 - t tr(K^-1 Q_aa)  from the Cholesky-based trace (two positive numbers)
            double tr = trVec[a];                                 // |L^-1 e^E|^2: the rank-one backbone
            for (int q = 0; q < ntr; ++q) tr += trPart[(long long)a * ntr + q];
            const double sf = hyp[(long long)a * hyp_ld + Nx];
            c += sf * sf - P[nn] * tr;
        }
        if (cov) { cov[a * Ny + b] = c; cov[b * Ny + a] = c; }
        if (a == b && var) var[a] = c;
    }
}

// ---------------------------------------------------------------------------------------
// Rank-1 append of one training point (SURVEY 8f row 3; the reference's update_data,
// gp_class.py:384-471, is self-declared broken -- this is the textbook update):
//   l = L^-1 k(X, x_new);  lambda = sqrt(k(x_new,x_new) + sn2 - l^T l)
//   L    <- [[L, 0], [l^T, lambda]]          L^-1 <- [[L^-1, 0], [-(l^T L^-1)/lambda, 1/lambda]]
// lvec = L^-1 k, rvec = (L^-1)^T lvec are produced by the trmv kernels; this kernel writes
// row N of both factors (the identity tail row it replaces).  One CTA per output.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
append_row_kernel(double* __restrict__ L, double* __restrict__ Li, int ld, long long sL,
                  const double* __restrict__ lvec, const double* __restrict__ rvec, long long sv,
                  const double* __restrict__ hyp, int hyp_ld, int Nx, int N, int* __restrict__ info)
{
    __shared__ double red[8];
    __shared__ double lam_s;
    const int a = blockIdx.x, tid = threadIdx.x;
    const double* lv = lvec + (long long)a * sv;
    const double* rv = rvec + (long long)a * sv;
    double s = 0.0;
    for (int i = tid; i < N; i += 256) s = fma(lv[i], lv[i], s);
    s = warp_sum(s);
    if ((tid & 31) == 0) red[tid >> 5] = s;
    __syncthreads();
    if (tid == 0) {
        double r = 0.0;
        for (int w = 0; w < 8; ++w) r += red[w];
        const double sf = hyp[(long long)a * hyp_ld + Nx], sn = hyp[(long long)a * hyp_ld + Nx + 1];
        const double d = sf * sf + sn * sn - r;
        if (!(d > 0.0)) atomicCAS(info + a, 0, N + 1);
        lam_s = sqrt(d);
    }
    __syncthreads();
    const double lam = lam_s, il = 1.0 / lam;
    double* Lr = L + (long long)a * sL + (long long)N * ld;
    double* Lir = Li + (long long)a * sL + (long long)N * ld;
    for (int j = tid; j < N; j += 256) { Lr[j] = lv[j]; Lir[j] = -rv[j] * il; }
    if (tid == 0) { Lr[N] = lam; Lir[N] = il; }
}

// ---------------------------------------------------------------------------------------
// First derivatives of the prediction w.r.t. the test input z (SURVEY 8f row 1: what CasADi's
// AD produces for the MPC's NLP from the symbolic build_gp / build_TA_cov graphs,
// gp_functions.py:111-173; mpc_class.py:390-412 differentiates them inside nlpsol):
//   d ks_i / d z_d = ks_i (X_id - z_d)/ell_d^2
//   d var / d z_d  = -2 sum_i beta_i ks_i (X_id - z_d)/ell_d^2 ,  beta = K^-1 ks = L^-T (L^-1 ks)
//   Hm_de = d^2 mean / dz_d dz_e = sum_i alpha_i ks_i s_id s_ie - delta_de mean/ell_d^2 ,
//           s_id = (X_id - z_d)/ell_d^2
// Stage 1 (this kernel): per (output, test point, 1024-point block) partial sums
//   PDV[d] = sum_i beta_i ks_i s_id            PH[q(d<=e)] = sum_i alpha_i ks_i s_id s_ie
// ks is read back from KST (written by ks_mean_jac_kernel), beta rows from the second product.
// grid (Npad/1024, Hc, outputs), 256 threads.
// ---------------------------------------------------------------------------------------
#define GR_CHUNK 1024
template <int NXP>
__global__ void __launch_bounds__(256)
grad_reduce_kernel(const double* __restrict__ XT, int ldx, int N, int Nx,
                   const double* __restrict__ hyp, int hyp_ld,
                   const double* __restrict__ alpha, long long sal,
                   const double* __restrict__ Z,
                   const double* __restrict__ KST, const double* __restrict__ BETA, int ldk, long long sK,
                   double* __restrict__ PDV, double* __restrict__ PH, int nblk, int Hc)
{
    extern __shared__ double gsm[];                 // S[Nx][257], WA[256]
    __shared__ double red[8][NXP];
    __shared__ double zs[NXP], ie2[NXP];
    const int a = blockIdx.z, h = blockIdx.y, blk = blockIdx.x, tid = threadIdx.x;
    double* S = gsm; double* WA = gsm + Nx * 257;
    const double* hp = hyp + (long long)a * hyp_ld;
    if (tid < NXP) {
        const double e = (tid < Nx) ? hp[tid] : 1.0;
        zs[tid] = (tid < Nx) ? Z[(long long)h * Nx + tid] : 0.0;
        ie2[tid] = 1.0 / (e * e);
    }
    __syncthreads();
    const int npairs = Nx * (Nx + 1) / 2;
    const double* ks = KST + (long long)a * sK + (long long)h * ldk;
    const double* be = BETA + (long long)a * sK + (long long)h * ldk;
    const double* al = alpha + (long long)a * sal;
    double dv[NXP];
#pragma unroll
    for (int d = 0; d < NXP; ++d) dv[d] = 0.0;
    double hacc[3] = {0.0, 0.0, 0.0};               // pairs tid, tid+256, tid+512 (NX_MAX = 32: 528 pairs)
    for (int sub = 0; sub < GR_CHUNK / 256; ++sub) {
        const int i = blk * GR_CHUNK + sub * 256 + tid;
        double k = 0.0, wb = 0.0, wa = 0.0;
        if (i < N) { k = ks[i]; wb = be[i] * k; wa = al[i] * k; }
#pragma unroll
        for (int d = 0; d < NXP; ++d) {
            if (d < Nx) {
                const double sd = (i < N) ? (XT[(long long)d * ldx + i] - zs[d]) * ie2[d] : 0.0;
                S[d * 257 + tid] = sd;
                dv[d] = fma(wb, sd, dv[d]);
            }
        }
        WA[tid] = wa;
        __syncthreads();
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            const int q = tid + 256 * r;
            if (q < npairs) {
                // q -> (d <= e), row-major upper packing: q = d*Nx - d(d-1)/2 + (e - d)
                int d = 0, base = 0;
                while (base + (Nx - d) <= q) { base += Nx - d; ++d; }
                const int e = d + (q - base);
                const double* sd = S + d * 257; const double* se = S + e * 257;
                double acc = 0.0;
                for (int t = 0; t < 256; ++t) acc = fma(WA[t] * sd[t], se[t], acc);
                hacc[r] += acc;
            }
        }
        __syncthreads();
    }
#pragma unroll
    for (int d = 0; d < NXP; ++d) dv[d] = warp_sum(dv[d]);
    if ((tid & 31) == 0) {
#pragma unroll
        for (int d = 0; d < NXP; ++d) red[tid >> 5][d] = dv[d];
    }
    __syncthreads();
    const long long rec = ((long long)a * Hc + h) * nblk + blk;
    if (tid < Nx) {
        double sacc = 0.0;
        for (int w = 0; w < 8; ++w) sacc += red[w][tid];
        PDV[rec * Nx + tid] = sacc;
    }
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        const int q = tid + 256 * r;
        if (q < npairs) PH[rec * npairs + q] = hacc[r];
    }
}

// Stage 2: per (test point h of the chunk, output a): dvar_dz (Nx) and the mean Hessian (Nx,Nx)
// from the block partials; grid (Hc, outputs), 128 threads.  mean comes from the gather record.
__global__ void __launch_bounds__(128)
grad_finalize_kernel(const double* __restrict__ PDV, const double* __restrict__ PH, int nblk, int Hc,
                     const double* __restrict__ hyp, int hyp_ld, int Nx, int Ny,
                     const double* __restrict__ G, int Htot, int h0,
                     double* __restrict__ dvar, double* __restrict__ hess)
{
    const int h = blockIdx.x, a = blockIdx.y, tid = threadIdx.x;
    const int npairs = Nx * (Nx + 1) / 2;
    const long long rec = ((long long)a * Hc + h) * nblk;
    const double* hp = hyp + (long long)a * hyp_ld;
    const double mean = G[(((long long)a) * Htot + h0 + h) * (Nx + 2)];
    for (int d = tid; d < Nx; d += 128) {
        double sacc = 0.0;
        for (int b = 0; b < nblk; ++b) sacc += PDV[(rec + b) * Nx + d];
        dvar[(((long long)(h0 + h)) * Ny + a) * Nx + d] = -2.0 * sacc;
    }
    for (int q = tid; q < npairs; q += 128) {
        int d = 0, base = 0;
        while (base + (Nx - d) <= q) { base += Nx - d; ++d; }
        const int e = d + (q - base);
        double sacc = 0.0;
        for (int b = 0; b < nblk; ++b) sacc += PH[(rec + b) * npairs + q];
        if (d == e) sacc -= mean / (hp[d] * hp[d]);
        double* Hm = hess + (((long long)(h0 + h)) * Ny + a) * Nx * Nx;
        Hm[d * Nx + e] = sacc;
        Hm[e * Nx + d] = sacc;
    }
}

// Stage 3: d cov[a][b] / d z_e for every test point (grid H, 128 threads):
//   'ME': delta_ab dvar_a[e]
//   'TA': delta_ab dvar_a[e] + sum_d Hm_a[d][e] (Sigma J_b)[d] + sum_d (J_a Sigma)[d] Hm_b[d][e]
//   (derivative of diag(var) + J Sigma J^T, gp_functions.py:167-171; Sigma need not be symmetric)
__global__ void __launch_bounds__(128)
grad_cov_kernel(int Ny, int Nx, int method_ta, const double* __restrict__ Sigma, int sigma_per_point,
                const double* __restrict__ J, const double* __restrict__ dvar, const double* __restrict__ hess,
                double* __restrict__ dcov)
{
    extern __shared__ double sh[];                  // SJ[Ny][Nx] = Sigma J_b, JS[Ny][Nx] = J_a Sigma
    double* SJ = sh; double* JS = sh + Ny * Nx;
    const int h = blockIdx.x, tid = threadIdx.x;
    const double* Jh = J + (long long)h * Ny * Nx;
    if (method_ta) {
        const double* Sg = Sigma + (sigma_per_point ? (long long)h * Nx * Nx : 0);
        for (int idx = tid; idx < Ny * Nx; idx += 128) {
            const int a = idx / Nx, d = idx % Nx;
            double s1 = 0.0, s2 = 0.0;
            for (int e = 0; e < Nx; ++e) {
                s1 = fma(Sg[d * Nx + e], Jh[a * Nx + e], s1);          // (Sigma J_a)[d]
                s2 = fma(Jh[a * Nx + e], Sg[e * Nx + d], s2);          // (J_a Sigma)[d]
            }
            SJ[idx] = s1; JS[idx] = s2;
        }
    }
    __syncthreads();
    const double* dv = dvar + (long long)h * Ny * Nx;
    const double* Hh = hess + (long long)h * Ny * Nx * Nx;
    double* out = dcov + (long long)h * Ny * Ny * Nx;
    for (int idx = tid; idx < Ny * Ny * Nx; idx += 128) {
        const int e = idx % Nx, b = (idx / Nx) % Ny, a = idx / (Nx * Ny);
        double s = (a == b) ? dv[a * Nx + e] : 0.0;
        if (method_ta) {
            const double* Ha = Hh + (long long)a * Nx * Nx; const double* Hb = Hh + (long long)b * Nx * Nx;
            for (int d = 0; d < Nx; ++d) {
                s = fma(Ha[d * Nx + e], SJ[b * Nx + d], s);
                s = fma(JS[a * Nx + d], Hb[d * Nx + e], s);
            }
        }
        out[idx] = s;
    }
}

// ---------------------------------------------------------------------------------------
// Second derivatives of the prediction w.r.t. the test input z (the next level of CasADi's exact
// Hessian for the MPC's NLP: mpc_class.py:496-513 leaves IPOPT on its default exact Hessian).
// Per output a and test point z, with s_id = (X_id - z_d)/ell_d^2, beta = K^-1 ks, alpha, J, Hm:
//   d2var_de = -2 [ w_d^T w_e + sum_i beta_i ks_i s_id s_ie - delta_de (sf2 - var)/ell_d^2 ],
//              w_d = L^-1 (ks o s_.d)                     (beta^T ks = sum v^2 = sf2 - var)
//   T_fde    = d^3 mean / dz_f dz_d dz_e
//            = sum_i alpha_i ks_i s_if s_id s_ie - delta_fd J_e/ell_f^2 - delta_fe J_d/ell_f^2 - delta_de J_f/ell_d^2
//   'TA' d2cov_ab,de = delta_ab d2var_a,de + sum_f [ T_a,fde (Sigma J_b)_f + Hm_a,fd (Sigma Hm_b)_fe
//                                                + Hm_a,fe (Sigma Hm_b)_fd + (J_a Sigma)_f T_b,fde ]
//   'ME' d2cov_ab,de = delta_ab d2var_a,de
// Pairs (d <= e) are packed row-major: q = d*Nx - d(d-1)/2 + (e - d).
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ void pair_de(int q, int Nx, int& d, int& e)
{
    int base = 0;
    d = 0;
    while (base + (Nx - d) <= q) { base += Nx - d; ++d; }
    e = d + (q - base);
}
__device__ __forceinline__ int pair_q(int d, int e, int Nx) { return d * Nx - d * (d - 1) / 2 + (e - d); }

// A operand of the W = L^-1 dks product: row r = pl*Nx + d holds ks_i s_id of chunk point p0 + pl (columns i < N;
// the padding columns and the rows r >= nrows up to the fragment height are zero).  grid (Npad/128, bm, outputs).
__global__ void __launch_bounds__(128)
hess_wrows_kernel(const double* __restrict__ XT, int ldx, int N, int Nx,
                  const double* __restrict__ hyp, int hyp_ld, const double* __restrict__ Z,
                  const double* __restrict__ KST, int ldk, long long sK, int p0, int nrows,
                  double* __restrict__ A, long long sA)
{
    const int i = blockIdx.x * 128 + threadIdx.x, r = blockIdx.y, a = blockIdx.z;
    double v = 0.0;
    if (r < nrows && i < N) {
        const int pl = r / Nx, d = r - pl * Nx, hl = p0 + pl;
        const double e = hyp[(long long)a * hyp_ld + d];
        const double sd = (XT[(long long)d * ldx + i] - Z[(long long)hl * Nx + d]) * (1.0 / (e * e));
        v = KST[(long long)a * sK + (long long)hl * ldk + i] * sd;
    }
    A[(long long)a * sA + (long long)r * ldk + i] = v;
}

// Gram step: GRAM[a][p0+pl][q(d<=e)] = w_d^T w_e over the Npad columns of the solved rows pl*Nx + d.
// grid (points of the pass, outputs), 256 threads; columns staged 128 at a time.
__global__ void __launch_bounds__(256)
hess_gram_kernel(const double* __restrict__ W, int ldw, long long sW, int np, int Nx, int p0, int Hc,
                 double* __restrict__ GRAM)
{
    extern __shared__ double gsm[];                 // S[Nx][129]
    const int pl = blockIdx.x, a = blockIdx.y, tid = threadIdx.x;
    const int npairs = Nx * (Nx + 1) / 2;
    const double* Wp = W + (long long)a * sW + (long long)pl * Nx * ldw;
    double acc[3] = {0.0, 0.0, 0.0};                // pairs tid, tid+256, tid+512 (NX_MAX = 32: 528 pairs)
    for (int c0 = 0; c0 < np; c0 += 128) {
        for (int idx = tid; idx < Nx * 128; idx += 256) {
            const int d = idx >> 7, t = idx & 127;
            gsm[d * 129 + t] = Wp[(long long)d * ldw + c0 + t];
        }
        __syncthreads();
#pragma unroll
        for (int r = 0; r < 3; ++r) {
            const int q = tid + 256 * r;
            if (q < npairs) {
                int d, e;
                pair_de(q, Nx, d, e);
                const double* sd = gsm + d * 129; const double* se = gsm + e * 129;
                double s = 0.0;
                for (int t = 0; t < 128; ++t) s = fma(sd[t], se[t], s);
                acc[r] += s;
            }
        }
        __syncthreads();
    }
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        const int q = tid + 256 * r;
        if (q < npairs) GRAM[((long long)a * Hc + p0 + pl) * npairs + q] = acc[r];
    }
}

// Per (output, test point, GR_CHUNK-point block): for every pair q = (d <= e), the (pairs x N).(N x (1+Nx)) product
//   HP[q][0] = sum_i beta_i ks_i s_id s_ie          HP[q][1+f] = sum_i alpha_i ks_i s_id s_ie s_if
// A thread owns whole pairs; its 1 + Nx sums live in registers over one 256-point sub-block and in its own slice of
// the block's partial record between sub-blocks (no other thread touches it).  grid (Npad/GR_CHUNK, Hc, outputs).
template <int NXP>
__global__ void __launch_bounds__(256)
hess_reduce_kernel(const double* __restrict__ XT, int ldx, int N, int Nx,
                   const double* __restrict__ hyp, int hyp_ld,
                   const double* __restrict__ alpha, long long sal,
                   const double* __restrict__ Z,
                   const double* __restrict__ KST, const double* __restrict__ BETA, int ldk, long long sK,
                   double* __restrict__ HP, int nblk, int Hc)
{
    extern __shared__ double hsm[];                 // S[Nx][257], WA[256], WB[256]
    __shared__ double zs[NXP], ie2[NXP];
    const int a = blockIdx.z, h = blockIdx.y, blk = blockIdx.x, tid = threadIdx.x;
    double* S = hsm; double* WA = hsm + Nx * 257; double* WB = WA + 256;
    const double* hp = hyp + (long long)a * hyp_ld;
    if (tid < NXP) {
        const double e = (tid < Nx) ? hp[tid] : 1.0;
        zs[tid] = (tid < Nx) ? Z[(long long)h * Nx + tid] : 0.0;
        ie2[tid] = 1.0 / (e * e);
    }
    __syncthreads();
    const int npairs = Nx * (Nx + 1) / 2, F1 = Nx + 1;
    const double* ks = KST + (long long)a * sK + (long long)h * ldk;
    const double* be = BETA + (long long)a * sK + (long long)h * ldk;
    const double* al = alpha + (long long)a * sal;
    double* out = HP + (((long long)a * Hc + h) * nblk + blk) * npairs * F1;
    for (int sub = 0; sub < GR_CHUNK / 256; ++sub) {
        const int i = blk * GR_CHUNK + sub * 256 + tid;
        double k = 0.0, wa = 0.0, wb = 0.0;
        if (i < N) { k = ks[i]; wa = al[i] * k; wb = be[i] * k; }
        for (int d = 0; d < Nx; ++d)
            S[d * 257 + tid] = (i < N) ? (XT[(long long)d * ldx + i] - zs[d]) * ie2[d] : 0.0;
        WA[tid] = wa; WB[tid] = wb;
        __syncthreads();
        for (int q = tid; q < npairs; q += 256) {
            int d, e;
            pair_de(q, Nx, d, e);
            double* o = out + (long long)q * F1;
            double accb = (sub == 0) ? 0.0 : o[0];
            double acc[NXP];
#pragma unroll
            for (int f = 0; f < NXP; ++f) acc[f] = (sub == 0 || f >= Nx) ? 0.0 : o[1 + f];
            const double* sd = S + d * 257; const double* se = S + e * 257;
            for (int t = 0; t < 256; ++t) {
                const double pde = sd[t] * se[t];
                accb = fma(WB[t], pde, accb);
                const double pa = WA[t] * pde;
#pragma unroll
                for (int f = 0; f < NXP; ++f)
                    if (f < Nx) acc[f] = fma(pa, S[f * 257 + t], acc[f]);
            }
            o[0] = accb;
#pragma unroll
            for (int f = 0; f < NXP; ++f)
                if (f < Nx) o[1 + f] = acc[f];
        }
        __syncthreads();
    }
}

// Per (chunk point h, output a): the block partials summed in block order into HS[a][h][q][1+Nx], and
// d2var (H,Ny,Nx,Nx) from the Gram, the beta pair sums and var of the gather record; (d,e) and (e,d) get one value.
// grid (Hc, outputs), 128 threads.
__global__ void __launch_bounds__(128)
hess_finalize_kernel(const double* __restrict__ HP, int nblk, int Hc, const double* __restrict__ GRAM,
                     const double* __restrict__ hyp, int hyp_ld, int Nx, int Ny,
                     const double* __restrict__ G, int Htot, int h0,
                     double* __restrict__ HS, double* __restrict__ d2var)
{
    const int h = blockIdx.x, a = blockIdx.y, tid = threadIdx.x;
    const int npairs = Nx * (Nx + 1) / 2, nent = npairs * (Nx + 1);
    const long long rec = (long long)a * Hc + h;
    const double* src = HP + rec * nblk * nent;
    double* dst = HS + rec * nent;
    for (int k = tid; k < nent; k += 128) {
        double s = 0.0;
        for (int b = 0; b < nblk; ++b) s += src[(long long)b * nent + k];
        dst[k] = s;
    }
    const double* hp = hyp + (long long)a * hyp_ld;
    const double sf = hp[Nx];
    const double c = sf * sf - G[(((long long)a) * Htot + h0 + h) * (Nx + 2) + 1];      // beta^T ks = sf2 - var
    double* out = d2var + (((long long)(h0 + h)) * Ny + a) * Nx * Nx;
    for (int q = tid; q < npairs; q += 128) {
        int d, e;
        pair_de(q, Nx, d, e);
        double pb = 0.0;
        for (int b = 0; b < nblk; ++b) pb += src[(long long)b * nent + (long long)q * (Nx + 1)];
        double v = GRAM[rec * npairs + q] + pb;
        if (d == e) v -= c / (hp[d] * hp[d]);
        v *= -2.0;
        out[d * Nx + e] = v;
        out[e * Nx + d] = v;
    }
}

// T_fde of output a at chunk point h from the summed third-order sums (see the block comment above)
__device__ __forceinline__ double hess_T(const double* HSa, const double* Ja, const double* hp, int Nx, int f, int d, int e)
{
    double t = HSa[(long long)pair_q(min(d, e), max(d, e), Nx) * (Nx + 1) + 1 + f];
    if (f == d) t -= Ja[e] / (hp[f] * hp[f]);
    if (f == e) t -= Ja[d] / (hp[f] * hp[f]);
    if (d == e) t -= Ja[f] / (hp[d] * hp[d]);
    return t;
}

// d2cov (H,Ny,Ny,Nx,Nx) of the chunk's points: grid (Hc), 256 threads.  J comes from the gather records, Hm from
// grad_finalize_kernel; SH[b][f][e] = (Sigma Hm_b)[f][e] is staged in global scratch (Ny Nx^2 per point).
__global__ void __launch_bounds__(256)
hess_cov_kernel(int Ny, int Nx, int method_ta, const double* __restrict__ Sigma, int sigma_per_point,
                const double* __restrict__ G, int Htot, int h0, const double* __restrict__ hyp, int hyp_ld,
                const double* __restrict__ HS, int Hc, const double* __restrict__ hess,
                const double* __restrict__ d2var, double* __restrict__ SH, double* __restrict__ d2cov)
{
    extern __shared__ double csm[];                 // Jh[Ny][Nx], SJ[Ny][Nx] = Sigma J_b, JS[Ny][Nx] = J_a Sigma
    double* Jh = csm; double* SJ = csm + Ny * Nx; double* JS = csm + 2 * Ny * Nx;
    const int h = blockIdx.x, hg = h0 + h, tid = threadIdx.x;
    const int nxx = Nx * Nx;
    const double* dv = d2var + (long long)hg * Ny * nxx;
    double* out = d2cov + (long long)hg * Ny * Ny * nxx;
    if (!method_ta) {
        for (long long idx = tid; idx < (long long)Ny * Ny * nxx; idx += 256) {
            const int de = (int)(idx % nxx), b = (int)((idx / nxx) % Ny), a = (int)(idx / ((long long)nxx * Ny));
            out[idx] = (a == b) ? dv[(long long)a * nxx + de] : 0.0;
        }
        return;
    }
    for (int idx = tid; idx < Ny * Nx; idx += 256) {
        const int a = idx / Nx, d = idx - a * Nx;
        Jh[idx] = G[(((long long)a) * Htot + hg) * (Nx + 2) + 2 + d];
    }
    __syncthreads();
    const double* Sg = Sigma + (sigma_per_point ? (long long)hg * nxx : 0);
    const double* Hh = hess + (long long)hg * Ny * nxx;
    double* SHh = SH + (long long)h * Ny * nxx;
    for (int idx = tid; idx < Ny * Nx; idx += 256) {
        const int a = idx / Nx, d = idx - a * Nx;
        double s1 = 0.0, s2 = 0.0;
        for (int e = 0; e < Nx; ++e) {
            s1 = fma(Sg[d * Nx + e], Jh[a * Nx + e], s1);          // (Sigma J_a)[d]
            s2 = fma(Jh[a * Nx + e], Sg[e * Nx + d], s2);          // (J_a Sigma)[d]
        }
        SJ[idx] = s1; JS[idx] = s2;
    }
    for (int idx = tid; idx < Ny * nxx; idx += 256) {
        const int b = idx / nxx, f = (idx / Nx) % Nx, e = idx % Nx;
        const double* Hb = Hh + (long long)b * nxx;
        double s = 0.0;
        for (int g = 0; g < Nx; ++g) s = fma(Sg[f * Nx + g], Hb[g * Nx + e], s);
        SHh[idx] = s;
    }
    __syncthreads();
    const int npairs = Nx * (Nx + 1) / 2, nent = npairs * (Nx + 1);
    for (int idx = tid; idx < Ny * Ny * npairs; idx += 256) {
        const int q = idx % npairs, b = (idx / npairs) % Ny, a = idx / (npairs * Ny);
        int d, e;
        pair_de(q, Nx, d, e);
        const double* hpa = hyp + (long long)a * hyp_ld; const double* hpb = hyp + (long long)b * hyp_ld;
        const double* HSa = HS + ((long long)a * Hc + h) * nent; const double* HSb = HS + ((long long)b * Hc + h) * nent;
        const double* Ha = Hh + (long long)a * nxx; const double* SHb = SHh + (long long)b * nxx;
        double s = (a == b) ? dv[(long long)a * nxx + d * Nx + e] : 0.0;
        for (int f = 0; f < Nx; ++f) {
            s = fma(hess_T(HSa, Jh + a * Nx, hpa, Nx, f, d, e), SJ[b * Nx + f], s);
            s = fma(Ha[f * Nx + d], SHb[f * Nx + e], s);
            s = fma(Ha[f * Nx + e], SHb[f * Nx + d], s);
            s = fma(JS[a * Nx + f], hess_T(HSb, Jh + b * Nx, hpb, Nx, f, d, e), s);
        }
        double* o = out + ((long long)a * Ny + b) * nxx;
        o[d * Nx + e] = s;
        o[e * Nx + d] = s;
    }
}

// ---------------------------------------------------------------------------------------
// FITC sparse build (gpmpc_fitc; the reference's GP.sparse, gp_class.py:682-689).  The M inducing points are the
// handle's own points U; the N training points stream through in column panels of Nb.
// ---------------------------------------------------------------------------------------
// Cross-covariance panel  Kuf[:, panel] = sf2 exp(-1/2 |(u_i - x_j)/ell|^2)  (Mpad x Nb, row-major, ld = ldk): the K
// build's scheme (centred, scaled coordinates on the handle's dMu, rank-Nx DMMA product, table exp2) on a rectangular
// grid of 128x128 tiles, rows from U (ld ldu, M valid) and columns from the panel's X^T (ld ldf, ncols valid).  No
// mirroring, no noise or jitter; rows >= M and columns >= ncols are exact zeros.  log2 k is clamped to log2 sf2 from
// above everywhere (a training point that is also an inducing point has distance 0 up to rounding).
__global__ void __launch_bounds__(256)
kcross_dmma_kernel(const double* __restrict__ UT, int ldu, int M, const double* __restrict__ FT, long long ldf, int ncols,
                   int Nx, const double* __restrict__ mu, const double* __restrict__ hyp, int hyp_ld,
                   double* __restrict__ K, int ldk, long long sK, int ntj)
{
    extern __shared__ double sm[];
    const int KD = (Nx + 3) & ~3;
    const int S = ((KD >> 2) & 1) ? KD : KD + 4;
    double* Ui = sm;                                      // [128][S] rows (inducing points)
    double* Uj = Ui + KB2_TILE * S;                       // [128][S] columns (training points of the panel)
    double* qi = Uj + KB2_TILE * S;
    double* qj = qi + KB2_TILE;
    double* T32 = qj + KB2_TILE;

    const int a = blockIdx.z;
    const double* hp = hyp + (long long)a * hyp_ld;
    const int bi = blockIdx.x / ntj, bj = blockIdx.x - bi * ntj;
    const int i0 = bi * KB2_TILE, j0 = bj * KB2_TILE;
    const int tid = threadIdx.x;
    const double sf2 = hp[Nx] * hp[Nx];
    const double l2sf2 = log2(sf2);

    __shared__ double sc[36], mus[36];
    if (tid < S) {
        sc[tid] = (tid < Nx) ? 1.2011224087864498 / hp[tid] : 0.0;
        mus[tid] = (tid < Nx) ? mu[tid] : 0.0;
    }
    if (tid < 16) T32[tid] = c_exp2_tab[tid];
    else if (tid < 32) T32[tid] = c_exp2_tab2[tid - 16];
    __syncthreads();
    {
        const bool rowpt = tid < KB2_TILE;
        const int l = tid & (KB2_TILE - 1);
        double* U = rowpt ? Ui + l * S : Uj + l * S;
        double nrm = 0.0;
        for (int d = 0; d < S; ++d) {
            double u = 0.0;
            if (d < Nx) u = ((rowpt ? UT[(long long)d * ldu + i0 + l] : FT[(long long)d * ldf + j0 + l]) - mus[d]) * sc[d];
            U[d] = u;
            nrm = fma(u, u, nrm);
        }
        (rowpt ? qi : qj)[l] = fma(-0.5, nrm, 0.5 * l2sf2);
    }
    __syncthreads();

    const int warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
    double* Ka = K + (long long)a * sK;
    const int nk4 = KD >> 2;
#pragma unroll 1
    for (int mi = 0; mi < 2; ++mi) {
        const int rl = warp * 16 + mi * 8 + g;
        const int row = i0 + rl;
        const double* ua = Ui + rl * S + t;
        const double qr = qi[rl];
        double* drow = Ka + (long long)row * ldk + j0 + 2 * t;
#pragma unroll 1
        for (int ng = 0; ng < 4; ++ng) {
            double acc[4][2];
#pragma unroll
            for (int q = 0; q < 4; ++q) { acc[q][0] = 0.0; acc[q][1] = 0.0; }
            const double* ub = Uj + (ng * 32 + g) * S + t;
            for (int kk = 0; kk < nk4; ++kk) {
                const double av = ua[kk * 4];
#pragma unroll
                for (int q = 0; q < 4; ++q) dmma884(acc[q][0], acc[q][1], av, ub[q * 8 * S + kk * 4]);
            }
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const int cl0 = ng * 32 + q * 8;
                const double2 qc = *reinterpret_cast<const double2*>(qj + cl0 + 2 * t);
                double t0 = (qr + qc.x) + acc[q][0], t1 = (qr + qc.y) + acc[q][1];
                t0 = (t0 < -1020.0) ? -1020.0 : t0;
                t1 = (t1 < -1020.0) ? -1020.0 : t1;
                t0 = (t0 > l2sf2) ? l2sf2 : t0;
                t1 = (t1 > l2sf2) ? l2sf2 : t1;
                double v0 = exp2_t2lvl(t0, T32), v1 = exp2_t2lvl(t1, T32);
                const int col = j0 + cl0 + 2 * t;
                if (row >= M || col >= ncols) v0 = 0.0;
                if (row >= M || col + 1 >= ncols) v1 = 0.0;
                *reinterpret_cast<double2*>(drow + cl0) = make_double2(v0, v1);
            }
        }
    }
}

// FITC column pass over one panel of V = Luu^-1 Kuf (Mpad x Nb, ld = ld): for every column i < ncols
//   Lambda_i = max(sf2 - |V_:i|^2, 0) + sn2       (the clamp absorbs rounding when x_i is itself an inducing point)
//   V_:i *= Lambda_i^-1/2 (in place),  w_i = y_i Lambda_i^-1/2,  partials {sum log Lambda_i, sum y_i^2 / Lambda_i}
// Columns >= ncols (zero in V) get w = 0 and contribute nothing.  CTA = 32 columns x 8 row groups; the row-group sums and
// the per-CTA partials are combined in a fixed order (deterministic).  grid (Nb / 32, outputs).
__global__ void __launch_bounds__(256)
fitc_column_kernel(double* __restrict__ V, int ld, long long sV, int Mpad, int ncols,
                   const double* __restrict__ hyp, int hyp_ld, int Nx, const double* __restrict__ y, long long sy,
                   double* __restrict__ w, long long sw, double* __restrict__ part, long long spart)
{
    __shared__ double red[8][33];
    __shared__ double scl[32];
    const int lane = threadIdx.x & 31, grp = threadIdx.x >> 5, a = blockIdx.y;
    const int col = blockIdx.x * 32 + lane;
    double* Va = V + (long long)a * sV;
    double s = 0.0;
    for (int r = grp; r < Mpad; r += 8) { const double v = Va[(long long)r * ld + col]; s = fma(v, v, s); }
    red[grp][lane] = s;
    __syncthreads();
    if (grp == 0) {
        double q = 0.0;
#pragma unroll
        for (int k = 0; k < 8; ++k) q += red[k][lane];
        const double* hp = hyp + (long long)a * hyp_ld;
        const double sf2 = hp[Nx] * hp[Nx], sn2 = hp[Nx + 1] * hp[Nx + 1];
        const bool valid = col < ncols;
        double lam = sf2 - q;
        lam = (lam > 0.0 ? lam : 0.0) + sn2;
        const double is = valid ? 1.0 / sqrt(lam) : 0.0;
        const double yv = valid ? y[(long long)a * sy + col] : 0.0;
        scl[lane] = is;
        w[(long long)a * sw + col] = yv * is;
        double lp = valid ? log(lam) : 0.0, yy = valid ? yv * yv / lam : 0.0;
        lp = warp_sum(lp); yy = warp_sum(yy);
        if (lane == 0) {
            part[(long long)a * spart + 2 * blockIdx.x] = lp;
            part[(long long)a * spart + 2 * blockIdx.x + 1] = yy;
        }
    }
    __syncthreads();
    const double is = scl[lane];
    for (int r = grp; r < Mpad; r += 8) Va[(long long)r * ld + col] *= is;
}

// b += Vs w  (b = V Lambda^-1 y accumulated panel by panel): one warp per row, lanes stride the Nb columns, fixed-order
// warp reduction; panels are added in stream order (deterministic).  grid (Mpad / 8, outputs).
__global__ void __launch_bounds__(256)
fitc_bvec_kernel(const double* __restrict__ V, int ld, long long sV, int Nb, const double* __restrict__ w, long long sw,
                 double* __restrict__ b, long long sb)
{
    const int row = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31, a = blockIdx.y;
    const double* Vr = V + (long long)a * sV + (long long)row * ld;
    const double* wa = w + (long long)a * sw;
    double s = 0.0;
    for (int i = lane; i < Nb; i += 32) s = fma(Vr[i], wa[i], s);
    s = warp_sum(s);
    if (lane == 0) b[(long long)a * sb + row] += s;
}

// A[i][i] += 1 for i < n (A = I + Phi; Phi's padded rows are zero, so the tail becomes the identity)
__global__ void fitc_add_identity_kernel(double* __restrict__ A, int ld, long long sA, int n)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) A[(long long)blockIdx.y * sA + (long long)i * ld + i] += 1.0;
}

// Exchange-matrix flip of the leading M x M block, lower triangle only:
//   dst[i][j] = scale * src[M-1-j][M-1-i] + (i == j ? dadd : 0)   for j <= i < M   (reads src's lower triangle)
// zeros above the diagonal, identity tail.  scale = -1, dadd = 1 (+ eps): J (I - X) J from X = LA^-T LA^-1 (lower);
// scale = 1, dadd = 0: S = J G^T J from the Cholesky factor G.  grid (ld / 32, ld / 32, batch), block (32, 8).
__global__ void fitc_flip_kernel(const double* __restrict__ src, double* __restrict__ dst, int ld, long long s, int M,
                                 double scale, double dadd)
{
    const int j = blockIdx.x * 32 + threadIdx.x;
    const double* sa = src + (long long)blockIdx.z * s;
    double* da = dst + (long long)blockIdx.z * s;
    for (int i = blockIdx.y * 32 + threadIdx.y; i < blockIdx.y * 32 + 32; i += 8) {
        double v;
        if (i < M && j < M) v = (j <= i) ? scale * sa[(long long)(M - 1 - j) * ld + (M - 1 - i)] + (i == j ? dadd : 0.0) : 0.0;
        else v = (i == j) ? 1.0 : 0.0;
        da[(long long)i * ld + j] = v;
    }
}

// FITC negative log marginal likelihood per output (reference convention, no N/2 log 2 pi):
//   1/2 (y^T Lambda^-1 y - |LA^-1 b|^2) + 1/2 (sum log Lambda_i + 2 sum log LA_ii)
// from the column-pass partials (nparts pairs), t = LA^-1 b and LA's diagonal.  One CTA per output, fixed-order sums.
__global__ void __launch_bounds__(256)
fitc_nll_kernel(const double* __restrict__ part, long long spart, int nparts, const double* __restrict__ LA, int ld,
                long long sL, const double* __restrict__ t, long long st, int n, double* __restrict__ nll)
{
    __shared__ double r[4][8];
    const int a = blockIdx.x, tid = threadIdx.x;
    const double* pa = part + (long long)a * spart;
    const double* La = LA + (long long)a * sL;
    const double* ta = t + (long long)a * st;
    double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
    for (int k = tid; k < nparts; k += 256) { s0 += pa[2 * k]; s1 += pa[2 * k + 1]; }
    for (int i = tid; i < n; i += 256) { s2 = fma(ta[i], ta[i], s2); s3 += log(La[(long long)i * ld + i]); }
    s0 = warp_sum(s0); s1 = warp_sum(s1); s2 = warp_sum(s2); s3 = warp_sum(s3);
    if ((tid & 31) == 0) { r[0][tid >> 5] = s0; r[1][tid >> 5] = s1; r[2][tid >> 5] = s2; r[3][tid >> 5] = s3; }
    __syncthreads();
    if (tid == 0) {
        double q[4] = {0.0, 0.0, 0.0, 0.0};
        for (int k = 0; k < 4; ++k) for (int w8 = 0; w8 < 8; ++w8) q[k] += r[k][w8];
        nll[a] = 0.5 * (q[1] - q[2]) + 0.5 * (q[0] + 2.0 * q[3]);
    }
}
