// sketch.cu — the projection sketch of an fp32 data set (see F32Sketch in kernels.h), built once per data set.
//
// Basis: the top SKETCH_K eigenvectors of the Gram matrix S^T S of an evenly spaced sample S of the rows (one device kernel), found on
// the host by subspace iteration in double with SKETCH_L - SKETCH_K extra columns, modified Gram-Schmidt and a Rayleigh-Ritz step.
// How good the basis is decides only how many candidates the bound drops, never whether the bound holds: the bound's identity
// needs P orthonormal up to the fp32 rounding of its entries, and r = x - P^T fp32(P x) is measured per row.
// Rows: one warp per row computes P x and ||r|| in double (fp32 sums over 768 terms would cost the bound up to ~5e-4 of ||x||).
#include <math.h>

#include <algorithm>
#include <vector>

#include "kernels.h"

namespace jv {

namespace {

constexpr int SKETCH_SAMPLE = 16384;  // rows in the basis sample
constexpr int SKETCH_L = 40;          // columns of the subspace iteration (8 beyond SKETCH_K: the gap after the 32nd value converges fast)
constexpr int SKETCH_ITERS = 8;
constexpr int GT = 64;                // Gram tile edge
constexpr int GR = 16;                // sample rows staged per tile step

// C = S^T S over the sample rows (row k of S = data row k * n / ns); 16 x 16 threads per 64 x 64 tile of C, 4 x 4 entries each
__global__ void __launch_bounds__(256) sketch_gram_kernel(const float *__restrict__ rows, long long n, int stride, int ns, float *__restrict__ C)
{
    __shared__ float a[GR][GT], b[GR][GT];
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const int i0 = blockIdx.y * GT, j0 = blockIdx.x * GT;
    float acc[4][4] = {};
    for (int r0 = 0; r0 < ns; r0 += GR) {
        for (int t = threadIdx.x; t < GR * GT; t += 256) {
            const int r = t / GT, c = t - r * GT;
            const float *row = rows + (size_t)((long long)(r0 + r) * n / ns) * stride;
            const bool in = r0 + r < ns;
            a[r][c] = in && i0 + c < stride ? row[i0 + c] : 0.f;
            b[r][c] = in && j0 + c < stride ? row[j0 + c] : 0.f;
        }
        __syncthreads();
#pragma unroll
        for (int r = 0; r < GR; r++) {
            float av[4], bv[4];
#pragma unroll
            for (int u = 0; u < 4; u++) { av[u] = a[r][ty + 16 * u]; bv[u] = b[r][tx + 16 * u]; }
#pragma unroll
            for (int u = 0; u < 4; u++)
#pragma unroll
                for (int v = 0; v < 4; v++) acc[u][v] = fmaf(av[u], bv[v], acc[u][v]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int u = 0; u < 4; u++)
#pragma unroll
        for (int v = 0; v < 4; v++) {
            const int i = i0 + ty + 16 * u, j = j0 + tx + 16 * v;
            if (i < stride && j < stride) C[(size_t)i * stride + j] = acc[u][v];
        }
}

// one warp per row: proj = fp32(P x), norms = {||x - P^T proj||, ||x||} rounded up
__global__ void __launch_bounds__(256) sketch_project_kernel(const float *__restrict__ rows, long long n, int stride, const float *__restrict__ basis,
                                                             float *__restrict__ proj, float2 *__restrict__ norms)
{
    const int lane = threadIdx.x & 31;
    const long long warps = (long long)gridDim.x * (blockDim.x >> 5);
    for (long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); row < n; row += warps) {
        const float *x = rows + (size_t)row * stride;
        double u[SKETCH_K];
#pragma unroll
        for (int j = 0; j < SKETCH_K; j++) u[j] = 0.0;
        for (int i = lane; i < stride; i += 32) {
            const double xv = x[i];
#pragma unroll
            for (int j = 0; j < SKETCH_K; j++) u[j] = fma((double)__ldg(basis + (size_t)j * stride + i), xv, u[j]);
        }
        float mine = 0.f;
#pragma unroll
        for (int j = 0; j < SKETCH_K; j++) {
            const float uj = (float)warp_sum_d(u[j]);
            u[j] = uj;  // from here on: the stored (rounded) projection, which r is measured against
            if (lane == j) mine = uj;
        }
        proj[(size_t)row * SKETCH_K + lane] = mine;
        double rr = 0.0, xx = 0.0;
        for (int i = lane; i < stride; i += 32) {
            const double xv = x[i];
            double r = xv;
#pragma unroll
            for (int j = 0; j < SKETCH_K; j++) r = fma(-(double)__ldg(basis + (size_t)j * stride + i), u[j], r);
            rr = fma(r, r, rr);
            xx = fma(xv, xv, xx);
        }
        rr = warp_sum_d(rr);
        xx = warp_sum_d(xx);
        if (lane == 0) norms[row] = make_float2(__double2float_ru(sqrt(rr)), __double2float_ru(sqrt(xx)));
    }
}

// columns j of the D x L column-major Y: modified Gram-Schmidt, twice (the second pass removes what rounding left of the first)
void mgs(std::vector<double> &Y, int D, int L)
{
    for (int pass = 0; pass < 2; pass++)
        for (int j = 0; j < L; j++) {
            double *yj = &Y[(size_t)j * D];
            for (int k = 0; k < j; k++) {
                const double *yk = &Y[(size_t)k * D];
                double d = 0.0;
                for (int i = 0; i < D; i++) d += yk[i] * yj[i];
                for (int i = 0; i < D; i++) yj[i] -= d * yk[i];
            }
            double nn = 0.0;
            for (int i = 0; i < D; i++) nn += yj[i] * yj[i];
            nn = sqrt(nn);
            const double inv = nn > 0.0 ? 1.0 / nn : 0.0;
            for (int i = 0; i < D; i++) yj[i] *= inv;
        }
}

// Z = C Y (C symmetric D x D row-major, Y / Z column-major D x L)
void gram_times(const std::vector<double> &Cd, const std::vector<double> &Y, std::vector<double> &Z, int D, int L)
{
    Z.assign((size_t)D * L, 0.0);
    for (int i = 0; i < D; i++) {  // one row of C at a time: it stays in cache across the L columns
        const double *c = &Cd[(size_t)i * D];
        for (int j = 0; j < L; j++) {
            const double *y = &Y[(size_t)j * D];
            double s = 0.0;
            for (int k = 0; k < D; k++) s += c[k] * y[k];
            Z[(size_t)j * D + i] = s;
        }
    }
}

// cyclic Jacobi on the symmetric L x L matrix A (row-major): eigenvalues on A's diagonal, eigenvectors in the columns of V
void jacobi_eigen(std::vector<double> &A, std::vector<double> &V, int L)
{
    V.assign((size_t)L * L, 0.0);
    for (int i = 0; i < L; i++) V[(size_t)i * L + i] = 1.0;
    for (int sweep = 0; sweep < 50; sweep++) {
        double off = 0.0, diag = 0.0;
        for (int p = 0; p < L; p++)
            for (int q = 0; q < L; q++) (p == q ? diag : off) += A[(size_t)p * L + q] * A[(size_t)p * L + q];
        if (off <= 1e-30 * diag) break;
        for (int p = 0; p < L - 1; p++)
            for (int q = p + 1; q < L; q++) {
                const double apq = A[(size_t)p * L + q];
                if (apq == 0.0) continue;
                const double theta = (A[(size_t)q * L + q] - A[(size_t)p * L + p]) / (2.0 * apq);
                const double t = (theta >= 0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
                const double c = 1.0 / sqrt(t * t + 1.0), s = t * c;
                for (int k = 0; k < L; k++) {  // A <- A J (columns p, q)
                    const double akp = A[(size_t)k * L + p], akq = A[(size_t)k * L + q];
                    A[(size_t)k * L + p] = c * akp - s * akq;
                    A[(size_t)k * L + q] = s * akp + c * akq;
                }
                for (int k = 0; k < L; k++) {  // A <- J^T A (rows p, q)
                    const double apk = A[(size_t)p * L + k], aqk = A[(size_t)q * L + k];
                    A[(size_t)p * L + k] = c * apk - s * aqk;
                    A[(size_t)q * L + k] = s * apk + c * aqk;
                }
                for (int k = 0; k < L; k++) {
                    const double vkp = V[(size_t)k * L + p], vkq = V[(size_t)k * L + q];
                    V[(size_t)k * L + p] = c * vkp - s * vkq;
                    V[(size_t)k * L + q] = s * vkp + c * vkq;
                }
            }
    }
}

struct SketchLayout {
    size_t basis, gram, proj, norms, C, total;
};
SketchLayout layout_of(const DataDesc &d)
{
    auto up = [](size_t v) { return (v + 255) & ~(size_t)255; };
    SketchLayout l;
    l.basis = 0;
    l.gram = up(l.basis + (size_t)SKETCH_K * d.stride * 4);
    l.proj = up(l.gram + (size_t)SKETCH_K * SKETCH_K * 8);
    l.norms = up(l.proj + (size_t)d.n * SKETCH_K * 4);
    l.C = up(l.norms + (size_t)d.n * 8);
    l.total = up(l.C + (size_t)d.stride * d.stride * 4);
    return l;
}

}  // namespace

size_t f32_sketch_bytes(const DataDesc &d) { return layout_of(d).total; }

cudaError_t build_f32_sketch(const DataDesc &d, void *mem, F32Sketch *sk, double *captured, cudaStream_t s)
{
    const SketchLayout l = layout_of(d);
    char *base = static_cast<char *>(mem);
    float *basis = reinterpret_cast<float *>(base + l.basis);
    double *gram = reinterpret_cast<double *>(base + l.gram);
    float *proj = reinterpret_cast<float *>(base + l.proj);
    float2 *norms = reinterpret_cast<float2 *>(base + l.norms);
    float *C = reinterpret_cast<float *>(base + l.C);
    const int D = d.stride, ns = (int)std::min<long long>(SKETCH_SAMPLE, d.n);

    const dim3 gg((D + GT - 1) / GT, (D + GT - 1) / GT);
    sketch_gram_kernel<<<gg, 256, 0, s>>>(d.rows, d.n, D, ns, C);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    g_launches++;
    std::vector<float> Cf((size_t)D * D);
    if ((e = cudaMemcpyAsync(Cf.data(), C, Cf.size() * 4, cudaMemcpyDeviceToHost, s)) != cudaSuccess) return e;
    if ((e = cudaStreamSynchronize(s)) != cudaSuccess) return e;
    std::vector<double> Cd(Cf.begin(), Cf.end());
    double trace = 0.0;
    for (int i = 0; i < D; i++) trace += Cd[(size_t)i * D + i];

    // subspace iteration from a fixed-seed start (the sketch, and so the rows read, are the same from run to run)
    std::vector<double> Y((size_t)D * SKETCH_L), Z;
    unsigned long long st = 0x2545F4914F6CDD1Dull;
    for (auto &y : Y) {
        st ^= st << 13; st ^= st >> 7; st ^= st << 17;
        y = (double)(st >> 11) * (1.0 / 9007199254740992.0) - 0.5;
    }
    mgs(Y, D, SKETCH_L);
    for (int it = 0; it < SKETCH_ITERS; it++) {
        gram_times(Cd, Y, Z, D, SKETCH_L);
        Y.swap(Z);
        mgs(Y, D, SKETCH_L);
    }
    // Rayleigh-Ritz: B = Y^T C Y, its eigenvectors rotate Y onto the Ritz vectors
    gram_times(Cd, Y, Z, D, SKETCH_L);
    std::vector<double> B((size_t)SKETCH_L * SKETCH_L), V;
    for (int a = 0; a < SKETCH_L; a++)
        for (int b = 0; b < SKETCH_L; b++) {
            double v = 0.0;
            for (int i = 0; i < D; i++) v += Y[(size_t)a * D + i] * Z[(size_t)b * D + i];
            B[(size_t)a * SKETCH_L + b] = v;
        }
    for (int a = 0; a < SKETCH_L; a++)
        for (int b = a + 1; b < SKETCH_L; b++) B[(size_t)a * SKETCH_L + b] = B[(size_t)b * SKETCH_L + a] = 0.5 * (B[(size_t)a * SKETCH_L + b] + B[(size_t)b * SKETCH_L + a]);
    jacobi_eigen(B, V, SKETCH_L);
    std::vector<int> order(SKETCH_L);
    for (int i = 0; i < SKETCH_L; i++) order[i] = i;
    std::sort(order.begin(), order.end(), [&](int a, int b) { return B[(size_t)a * SKETCH_L + a] > B[(size_t)b * SKETCH_L + b]; });
    std::vector<double> P((size_t)D * SKETCH_K, 0.0);
    double top = 0.0;
    for (int j = 0; j < SKETCH_K; j++) {
        const int c = order[j];
        top += B[(size_t)c * SKETCH_L + c];
        for (int a = 0; a < SKETCH_L; a++) {
            const double w = V[(size_t)a * SKETCH_L + c];
            for (int i = 0; i < D; i++) P[(size_t)j * D + i] += w * Y[(size_t)a * D + i];
        }
    }
    mgs(P, D, SKETCH_K);
    *captured = trace > 0.0 ? top / trace : 0.0;

    std::vector<float> Pf(P.begin(), P.end());
    std::vector<double> G((size_t)SKETCH_K * SKETCH_K);
    for (int a = 0; a < SKETCH_K; a++)
        for (int b = 0; b < SKETCH_K; b++) {
            double v = 0.0;
            for (int i = 0; i < D; i++) v += (double)Pf[(size_t)a * D + i] * (double)Pf[(size_t)b * D + i];
            G[(size_t)a * SKETCH_K + b] = v;
        }
    if ((e = cudaMemcpyAsync(basis, Pf.data(), Pf.size() * 4, cudaMemcpyHostToDevice, s)) != cudaSuccess) return e;
    if ((e = cudaMemcpyAsync(gram, G.data(), G.size() * 8, cudaMemcpyHostToDevice, s)) != cudaSuccess) return e;
    int dev = 0, sms = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    sketch_project_kernel<<<std::max(1, sms) * 8, 256, 0, s>>>(d.rows, d.n, D, basis, proj, norms);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    g_launches++;
    if ((e = cudaStreamSynchronize(s)) != cudaSuccess) return e;  // Pf / G are host temporaries of this call
    sk->basis = basis;
    sk->gram = gram;
    sk->proj = reinterpret_cast<const float4 *>(proj);
    sk->norms = norms;
    return cudaSuccess;
}

}  // namespace jv
