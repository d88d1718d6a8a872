// denoise.cu — the edge-avoiding a-trous wavelet filter (Dammertz, Sewtz, Hanika, Lensch, HPG 2010) over the accumulation sums,
// guided by the buffers of pt_render_aov (trace_kernels.cu aovKernel).  One launch per iteration, float32; every tap reads four
// float4 (colour, albedo, normal, position), so the pass is bound by L2 / HBM traffic.
#include "trace_kernels.h"
#include <cfloat>

namespace ptb
{

// the colour of pixel i as the iteration filters it: the first iteration divides the sums by the albedo (the filter then smooths
// illumination, and texture detail comes back with the albedo in the last iteration)
static __device__ __forceinline__ float3 colourAt(const AtrousParams &p, const float4 c, const float4 a)
{
	if (!p.demodulate) return make_float3(c.x, c.y, c.z);
	return make_float3(c.x / fmaxf(a.x, 0.01f), c.y / fmaxf(a.y, 0.01f), c.z / fmaxf(a.z, 0.01f));
}

// one iteration: 5 x 5 taps of the B3 spline kernel h = [1 4 6 4 1] / 16 (outer product), `step` pixels apart; taps outside the image
// are skipped and the weights renormalised.  Weight of tap q for pixel p:
//   h * exp(-|c_p - c_q|^2 / sigma_c^2 - |n_p - n_q|^2 / sigma_n^2 - |x_p - x_q|^2 / (sigma_x t_p)^2)
// A pixel none of whose camera rays hit anything is passed through; a tap counts only where p and q agree on that.
__global__ void __launch_bounds__(256) atrousKernel(const __grid_constant__ AtrousParams p)
{
	const uint32_t x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
	if (x >= p.width || y >= p.height) return;
	const uint32_t i = y * p.width + x;
	const float4 in = __ldg(p.in + i), ap = __ldg(p.albedo + i);
	if (ap.w == 0.0f)
	{
		p.out[i] = in;
		return;
	}
	const float4 np = __ldg(p.normal + i), xp = __ldg(p.position + i);
	const float3 cp = colourAt(p, in, ap);
	// (a sigma of 0 admits equal values only: the inverse is clamped to the largest float, so that 0 x it stays 0)
	const float xs = p.sigmaPosition * xp.w;
	const float invX2 = fminf(1.0f / (xs * xs), FLT_MAX);
	const float h[5] = { 1.0f / 16.0f, 4.0f / 16.0f, 6.0f / 16.0f, 4.0f / 16.0f, 1.0f / 16.0f };
	float sw = 0.0f, r = 0.0f, g = 0.0f, b = 0.0f;
#pragma unroll
	for (int dy = -2; dy <= 2; ++dy)
	{
		const int qy = int(y) + dy * int(p.step);
		if (qy < 0 || qy >= int(p.height)) continue;
#pragma unroll
		for (int dx = -2; dx <= 2; ++dx)
		{
			const int qx = int(x) + dx * int(p.step);
			if (qx < 0 || qx >= int(p.width)) continue;
			const uint32_t q = uint32_t(qy) * p.width + uint32_t(qx);
			const float4 aq = __ldg(p.albedo + q);
			if (aq.w == 0.0f) continue;
			const float3 cq = colourAt(p, __ldg(p.in + q), aq);
			const float4 nq = __ldg(p.normal + q), xq = __ldg(p.position + q);
			const float c0 = cp.x - cq.x, c1 = cp.y - cq.y, c2 = cp.z - cq.z;
			const float n0 = np.x - nq.x, n1 = np.y - nq.y, n2 = np.z - nq.z;
			const float x0 = xp.x - xq.x, x1 = xp.y - xq.y, x2 = xp.z - xq.z;
			const float e = (c0 * c0 + c1 * c1 + c2 * c2) * p.invColor2 + (n0 * n0 + n1 * n1 + n2 * n2) * p.invNormal2 + (x0 * x0 + x1 * x1 + x2 * x2) * invX2;
			const float w = h[dx + 2] * h[dy + 2] * expf(-e);
			sw += w;
			r += w * cq.x;
			g += w * cq.y;
			b += w * cq.z;
		}
	}
	// (the centre tap always counts: sw >= 36 / 256)
	float3 o = make_float3(r / sw, g / sw, b / sw);
	if (p.remodulate) o = make_float3(o.x * fmaxf(ap.x, 0.01f), o.y * fmaxf(ap.y, 0.01f), o.z * fmaxf(ap.z, 0.01f));
	p.out[i] = make_float4(o.x, o.y, o.z, in.w);
}

int launchAtrous(const AtrousParams &p, cudaStream_t stream)
{
	const dim3 block(32, 8), grid((p.width + 31) / 32, (p.height + 7) / 8);
	atrousKernel<<<grid, block, 0, stream>>>(p);
	return 1;
}

} // namespace ptb
