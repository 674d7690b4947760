// Small hand-written support kernels: checksum, row-wise max |x| (constraint violation), elementwise
// accumulation, packing of the rigid-contact inputs, FMA peak micro-benchmark (the FP64 / FP32 roofline denominators are measured, not assumed).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace grbda_kernels
{
    // out[0] += sum x, out[1] += sum |x|   (out zeroed by the caller)
    __global__ void __launch_bounds__(256) checksumKernel(const double *__restrict__ x, int64_t n, double *out)
    {
        double s = 0.0, a = 0.0;
        for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        {
            const double v = x[i];
            s += v;
            a += fabs(v);
        }
        for (int o = 16; o > 0; o >>= 1)
        {
            s += __shfl_down_sync(0xffffffffu, s, o);
            a += __shfl_down_sync(0xffffffffu, a, o);
        }
        __shared__ double ws[8], wa[8];
        const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
        if (l == 0)
        {
            ws[w] = s;
            wa[w] = a;
        }
        __syncthreads();
        if (threadIdx.x == 0)
        {
            for (int i = 1; i < 8; i++)
            {
                s += ws[i];
                a += wa[i];
            }
            atomicAdd(out, s);
            atomicAdd(out + 1, a);
        }
    }

    // y[b] = max_i |x[b * n + i]|
    __global__ void rowMaxAbsKernel(const double *__restrict__ x, int n, int64_t rows, double *__restrict__ y)
    {
        const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
        if (b >= rows)
            return;
        double m = 0.0;
        for (int i = 0; i < n; i++)
            m = fmax(m, fabs(x[b * n + i]));
        y[b] = m;
    }

    // y0[i] += x0[i] (i < n0), y1[i] += x1[i] (i < n1): sums the two contributions to q_bar of the vector-Jacobian
    // products with external forces (n1 = 0), and to q_bar and yd_bar of the simulation step's
    __global__ void __launch_bounds__(256) accumulateKernel(double *__restrict__ y0, const double *__restrict__ x0, int64_t n0,
                                                            double *__restrict__ y1, const double *__restrict__ x1, int64_t n1)
    {
        for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n0 + n1; i += (int64_t)gridDim.x * blockDim.x)
            if (i < n0)
                y0[i] += x0[i];
            else
                y1[i - n0] += x1[i - n0];
    }

    // Input array 2 of the rigid-contact programs, row b = [tau[b] (nt values); s (ncp); x0 (, x1)] with s_k = 1.0 where
    // active[b][k] != 0, 0.0 elsewhere, all 1.0 without a mask (active = NULL); ns = 1 or 2 scalars broadcast to every
    // row: [tau; s; eps] (nt = nv, ns = 1) for the contact dynamics, [s; e; eps] (nt = 0, ns = 2) for the impulse
    __global__ void __launch_bounds__(256) packContactRowsKernel(double *__restrict__ packed, const double *__restrict__ tau,
                                                                 int nt, const uint8_t *__restrict__ active, int ncp,
                                                                 double x0, double x1, int ns, int64_t batch)
    {
        const int row = nt + ncp + ns;
        for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < batch * row; i += (int64_t)gridDim.x * blockDim.x)
        {
            const int64_t b = i / row;
            const int k = (int)(i - b * row);
            double v;
            if (k < nt)
                v = tau[b * nt + k];
            else if (k < nt + ncp)
                v = !active || active[b * ncp + (k - nt)] ? 1.0 : 0.0;
            else
                v = k == nt + ncp ? x0 : x1;
            packed[i] = v;
        }
    }

    // Dependent-free FMA streams: 8 independent accumulators per thread, `iters` rounds of 8 FMAs.
    template <typename real>
    __global__ void __launch_bounds__(256) fmaPeakKernel(real *out, int iters, real a, real b)
    {
        real x0 = threadIdx.x, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5, x6 = x0 + 6,
             x7 = x0 + 7;
        for (int i = 0; i < iters; i++)
        {
#pragma unroll 8
            for (int k = 0; k < 8; k++)
            {
                x0 = fma(x0, a, b);
                x1 = fma(x1, a, b);
                x2 = fma(x2, a, b);
                x3 = fma(x3, a, b);
                x4 = fma(x4, a, b);
                x5 = fma(x5, a, b);
                x6 = fma(x6, a, b);
                x7 = fma(x7, a, b);
            }
        }
        const real s = x0 + x1 + x2 + x3 + x4 + x5 + x6 + x7;
        if (s == (real)-1.2345)
            out[0] = s;
    }

} // namespace grbda_kernels
