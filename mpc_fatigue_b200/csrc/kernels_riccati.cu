// kernels_riccati.cu — batched Riccati solve of the multiple-shooting LQ subproblem (DESIGN.md §4f).
//
// Per scenario b (units u = k B + b), x = (q, qd, f) (3n, the row order of the step Jacobian), u = tau (n):
//   min  sum_k 1/2 z_k^T W_k z_k + g_k^T z_k + 1/2 dx_N^T W_N dx_N + g_N^T dx_N,   z_k = (dx_k, du_k)
//   s.t. dx_0 = dx0,  dx_{k+1} = A_k dx_k + B_k du_k + d_k.
// One warp per scenario; the nodes run serially.  Inside a node the x and u components are merged into one index
// c = (u_0 .. u_{n-1}, x_0 .. x_{3n-1}), u first, so that eliminating the first n pivots of the node's KKT block
// Z = [[R + B'PB, S + B'PA, qu], [.., Q + A'PA, qx]] leaves the new cost-to-go (P, p) as the trailing block.  Lanes own
// the columns of Z; every row operand is a shared-memory broadcast.
#include "launch.cuh"

namespace mpcf {

namespace {

// shared-memory doubles of one warp (one scenario): P [nx][nx], p, AB [nx][nc + 1], Z [nc][nc + 1], five vectors
MPCF_HD int riccati_warp_doubles(int n)
{
    const int nx = 3 * n, nc = 4 * n;
    return nx * nx + nx + nx * (nc + 1) + nc * (nc + 1) + 5 * (nc + 1);
}

// column of the step Jacobian / Hessian (z = (q, qd, tau, f, dt)) that holds merged index c
MPCF_DI int zcol(int c, int n) { return c < n ? 2 * n + c : (c - n < 2 * n ? c - n : c); }

MPCF_DI double ld_or0(const double *p, long i) { return p ? __ldg(p + i) : 0.0; }

// A_k and B_k of unit u into AB (row r = state row, column c = merged index; row stride nc + 1, odd: conflict-free columns)
MPCF_DI void load_ab(const RiccatiArgs &a, long u, long U, double *AB, int lane)
{
    const int n = a.n, nx = 3 * n, nc = 4 * n, ldab = nc + 1, P4 = 4 * n + 1;
    for (int idx = lane; idx < nx * nc; idx += 32) {
        const int r = idx / nc, c = idx - r * nc;
        AB[r * ldab + c] = __ldg(a.jac + ((long)r * P4 + zcol(c, n)) * U + u);
    }
}

// W_k entry (i, c) of the merged index, read from the upper triangle of H in merged order, plus the diagonal planes
MPCF_DI double w_entry(const RiccatiArgs &a, int i, int c, long u, long U)
{
    const int n = a.n, P4 = 4 * n + 1;
    const int lo = i < c ? i : c, hi = i < c ? c : i;
    double w = a.H ? __ldg(a.H + ((long)zcol(lo, n) * P4 + zcol(hi, n)) * U + u) : 0.0;
    if (i == c) w += i < n ? ld_or0(a.wu, (long)i * U + u) : ld_or0(a.wx, (long)(i - n) * U + u);
    return w;
}

}  // namespace

// PLANES = false: mpcf_riccati_batch, the gains go to the chunk-local workspace and the forward pass always runs.  PLANES = true:
// mpcf_riccati_gains_batch, the gains go to the caller's planes a.ws = K [n][3n+1][N B] (plane t (3n+1) + j, unit k B + b; b0 = 0) and
// the forward pass and the costates run only when a.dx is given.
template <int MAXN, int WPC, bool PLANES = false>
__global__ void __launch_bounds__(32 * WPC) k_riccati(const RiccatiArgs a, long b0, long cnt)
{
    constexpr int MX = 3 * MAXN;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const long bl = (long)blockIdx.x * WPC + w;  // scenario within the chunk
    if (bl >= cnt) return;                       // warp-uniform: only warp-level barriers below
    const long b = b0 + bl, B = a.B;
    const int n = a.n, N = a.N, nx = 3 * n, nu = n, nc = 4 * n, ld = nc + 1, ldk = nx + 1;
    const long U = (long)N * B;
    extern __shared__ double smem[];
    double *P = smem + (long)w * riccati_warp_doubles(n);
    double *p = P + nx * nx;
    double *AB = p + nx;
    double *Z = AB + nx * ld;
    double *v = Z + nc * ld;  // p + P d | the scaled pivot row
    double *dd = v + ld;      // d_k
    double *xs = dd + ld;     // dx_k (forward), dx_k (reverse)
    double *us = xs + ld;     // du_k
    double *ls = us + ld;     // lambda_{k+1}

    // ---- backward pass: P_N = W_N, p_N = g_N ----
    for (int idx = lane; idx < nx * nx; idx += 32) {
        const int r = idx / nx, m = idx - r * nx;
        P[idx] = ld_or0(a.HN, (long)idx * B + b) + (r == m ? ld_or0(a.wN, (long)r * B + b) : 0.0);
    }
    for (int r = lane; r < nx; r += 32) p[r] = ld_or0(a.gN, (long)r * B + b);
    __syncwarp();
    bool bad = false;
    for (int k = N - 1; k >= 0; --k) {
        const long u = (long)k * B + b;
        load_ab(a, u, U, AB, lane);
        for (int r = lane; r < nx; r += 32) dd[r] = ld_or0(a.d, (long)r * U + u);
        __syncwarp();
        // v = p + P d (P symmetric: column r read as row r, stride 1 over the lanes)
        for (int r = lane; r < nx; r += 32) {
            double s = p[r];
            for (int m = 0; m < nx; ++m) s = fma(P[m * nx + r], dd[m], s);
            v[r] = s;
        }
        // Z = W + [B A]^T P [B A] (upper triangle computed, mirrored so that Z and every P stay exactly symmetric)
        for (int c = lane; c < nc; c += 32) {
            double pab[MX];
#pragma unroll
            for (int r = 0; r < MX; ++r) {
                if (r < nx) {
                    double s = 0.0;
                    for (int m = 0; m < nx; ++m) s = fma(P[r * nx + m], AB[m * ld + c], s);
                    pab[r] = s;
                }
            }
            for (int i = 0; i <= c; ++i) {
                double s = w_entry(a, i, c, u, U);
#pragma unroll
                for (int r = 0; r < MX; ++r)
                    if (r < nx) s = fma(AB[r * ld + i], pab[r], s);
                Z[i * ld + c] = s;
                Z[c * ld + i] = s;
            }
        }
        __syncwarp();
        // right-hand column: g + [B A]^T (p + P d)
        for (int i = lane; i < nc; i += 32) {
            double s = i < nu ? ld_or0(a.gu, (long)i * U + u) : ld_or0(a.gx, (long)(i - nu) * U + u);
            for (int r = 0; r < nx; ++r) s = fma(AB[r * ld + i], v[r], s);
            Z[i * ld + nc] = s;
        }
        __syncwarp();
        // Cholesky of Quu by row elimination: row t becomes (L^T | L^-1 Qux | L^-1 qu), the trailing block P - Y^T Y
        for (int t = 0; t < nu; ++t) {
            const double piv = Z[t * ld + t];
            bad |= !(piv > 0.0);
            const double sq = sqrt(piv);
            for (int c = t + lane; c <= nc; c += 32) {
                const double s = Z[t * ld + c] / sq;
                Z[t * ld + c] = s;
                v[c] = s;
            }
            __syncwarp();
            for (int c = t + 1 + lane; c <= nc; c += 32) {
                const double sc = v[c];
                for (int r = t + 1; r < nc; ++r) Z[r * ld + c] = fma(-v[r], sc, Z[r * ld + c]);
            }
            __syncwarp();
        }
        // K = -L^-T Y_x and k = -L^-T y_u by back substitution (lane = column), into the workspace or the planes; the new (P, p)
        double *K = a.ws + (PLANES ? u : ((bl * N + k) * (long)nu) * ldk);
        const long sk = PLANES ? U : 1;  // stride of the gain entries
        for (int c = nu + lane; c <= nc; c += 32) {
            double kc[MAXN];
#pragma unroll
            for (int t = MAXN - 1; t >= 0; --t) {
                if (t < nu) {
                    double s = Z[t * ld + c];
#pragma unroll
                    for (int q = t + 1; q < MAXN; ++q)
                        if (q < nu) s = fma(Z[t * ld + q], kc[q], s);
                    kc[t] = -s / Z[t * ld + t];
                    K[(t * ldk + (c - nu)) * sk] = kc[t];
                }
            }
            if (c < nc)
                for (int r = 0; r < nx; ++r) P[r * nx + (c - nu)] = Z[(nu + r) * ld + c];
            else
                for (int r = 0; r < nx; ++r) p[r] = Z[(nu + r) * ld + nc];
        }
        __syncwarp();
    }

    // ---- forward pass ----
    const double qnan = __longlong_as_double(0x7ff8000000000000LL);
    if (bad) {  // Quu not positive definite at some node: the whole scenario is NaN
        if constexpr (PLANES) {
            for (int idx = lane; idx < nu * ldk; idx += 32)
                for (int k = 0; k < N; ++k) a.ws[(long)idx * U + (long)k * B + b] = qnan;
            if (!a.dx) return;
        }
        for (int r = lane; r < nx; r += 32)
            for (int k = 0; k <= N; ++k) {
                a.dx[(long)r * (N + 1) * B + (long)k * B + b] = qnan;
                if (a.lam) a.lam[(long)r * (N + 1) * B + (long)k * B + b] = qnan;
            }
        for (int t = lane; t < nu; t += 32)
            for (int k = 0; k < N; ++k) a.du[(long)t * U + (long)k * B + b] = qnan;
        return;
    }
    if (PLANES && !a.dx) return;
    const long UX = (long)(N + 1) * B;
    for (int r = lane; r < nx; r += 32) {
        const double x0 = ld_or0(a.dx0, (long)r * B + b);
        xs[r] = x0;
        a.dx[(long)r * UX + b] = x0;
    }
    for (int k = 0; k < N; ++k) {
        const long u = (long)k * B + b;
        const double *K = a.ws + (PLANES ? u : ((bl * N + k) * (long)nu) * ldk);
        for (int idx = lane; idx < nu * ldk; idx += 32) Z[idx] = K[idx * (PLANES ? U : 1)];
        load_ab(a, u, U, AB, lane);
        for (int r = lane; r < nx; r += 32) dd[r] = ld_or0(a.d, (long)r * U + u);
        __syncwarp();
        for (int t = lane; t < nu; t += 32) {
            double s = Z[t * ldk + nx];
            for (int j = 0; j < nx; ++j) s = fma(Z[t * ldk + j], xs[j], s);
            us[t] = s;
            a.du[(long)t * U + u] = s;
        }
        __syncwarp();
        double xn[(MX + 31) / 32];
#pragma unroll
        for (int q = 0; q < (MX + 31) / 32; ++q) {
            const int r = lane + 32 * q;
            if (r < nx) {
                double s = dd[r];
                for (int c = 0; c < nu; ++c) s = fma(AB[r * ld + c], us[c], s);
                for (int j = 0; j < nx; ++j) s = fma(AB[r * ld + nu + j], xs[j], s);
                xn[q] = s;
                a.dx[(long)r * UX + u + B] = s;
            }
        }
        __syncwarp();
#pragma unroll
        for (int q = 0; q < (MX + 31) / 32; ++q)
            if (lane + 32 * q < nx) xs[lane + 32 * q] = xn[q];
        __syncwarp();
    }
    if (!a.lam) return;

    // ---- costates by a reverse sweep: lambda_N = W_N dx_N + g_N, lambda_k = Q dx + S^T du + gx + A^T lambda_{k+1} ----
    for (int r = lane; r < nx; r += 32) {
        double s = ld_or0(a.gN, (long)r * B + b) + ld_or0(a.wN, (long)r * B + b) * xs[r];
        for (int m = 0; m < nx; ++m) s = fma(ld_or0(a.HN, ((long)r * nx + m) * B + b), xs[m], s);
        ls[r] = s;
        a.lam[(long)r * UX + (long)N * B + b] = s;
    }
    __syncwarp();
    for (int k = N - 1; k >= 0; --k) {
        const long u = (long)k * B + b;
        load_ab(a, u, U, AB, lane);
        for (int r = lane; r < nx; r += 32) xs[r] = a.dx[(long)r * UX + u];  // written by this lane in the forward pass
        for (int t = lane; t < nu; t += 32) us[t] = a.du[(long)t * U + u];
        __syncwarp();
        double lk[(MX + 31) / 32];
#pragma unroll
        for (int q = 0; q < (MX + 31) / 32; ++q) {
            const int r = lane + 32 * q;
            if (r < nx) {
                const int i = nu + r;
                double s = ld_or0(a.gx, (long)r * U + u);
                for (int c = 0; c < nc; ++c) s = fma(w_entry(a, i, c, u, U), c < nu ? us[c] : xs[c - nu], s);
                for (int m = 0; m < nx; ++m) s = fma(AB[m * ld + i], ls[m], s);
                lk[q] = s;
                a.lam[(long)r * UX + u] = s;
            }
        }
        __syncwarp();
#pragma unroll
        for (int q = 0; q < (MX + 31) / 32; ++q)
            if (lane + 32 * q < nx) ls[lane + 32 * q] = lk[q];
        __syncwarp();
    }
}

int riccati_warps_per_cta(int n) { return n <= 8 ? 4 : 2; }

size_t riccati_ws_bytes_per_scenario(int n, int N) { return (size_t)N * n * (3 * n + 1) * sizeof(double); }

template <int MAXN, int WPC, bool PLANES = false>
static cudaError_t launch_bucket(const RiccatiArgs &a, long b0, long cnt, cudaStream_t s)
{
    // the limit is set once per device, for the largest n of the bucket
    if (cudaError_t e = raise_smem_limit<k_riccati<MAXN, WPC, PLANES>>(WPC * riccati_warp_doubles(MAXN) * (int)sizeof(double))) return e;
    const unsigned grid = (unsigned)((cnt + WPC - 1) / WPC);
    k_riccati<MAXN, WPC, PLANES><<<grid, 32 * WPC, (size_t)WPC * riccati_warp_doubles(a.n) * sizeof(double), s>>>(a, b0, cnt);
    g_launches.fetch_add(1);
    return cudaGetLastError();
}

cudaError_t launch_riccati(const RiccatiArgs &a, long b0, long cnt, cudaStream_t s)
{
    if (cnt <= 0) return cudaSuccess;
    if (a.n <= 4) return launch_bucket<4, 4>(a, b0, cnt, s);
    if (a.n <= 8) return launch_bucket<8, 4>(a, b0, cnt, s);
    return launch_bucket<16, 2>(a, b0, cnt, s);
}

cudaError_t launch_riccati_gains(const RiccatiArgs &a, cudaStream_t s)
{
    if (a.B <= 0) return cudaSuccess;
    if (a.n <= 4) return launch_bucket<4, 4, true>(a, 0, a.B, s);
    if (a.n <= 8) return launch_bucket<8, 4, true>(a, 0, a.B, s);
    return launch_bucket<16, 2, true>(a, 0, a.B, s);
}

}  // namespace mpcf
