/* tests/adaptive_oracle.c — the CPU restatement of option "adaptive" (include/pt_b200.h) that tests/test_adaptive.py checks the trace
 * kernel against.  NOT THE REFERENCE, like the env_is / light_is sections of the oracle: it adds one entry point on top of the oracle
 * (oracle/pt_oracle.c, included whole and unchanged) and uses the oracle's own camera rays, Philox draws, stratification rule and path
 * loop (getColor), so every sample is the oracle's.  Built by the test with the oracle's compiler flags. */
#include "../oracle/pt_oracle.c"

/* ---- NOT THE REFERENCE: adaptive sampling (the product's option "adaptive", include/pt_b200.h).  A pixel's samples come in intervals
 * [0, c0), [c0, c1), ... that end at its checkpoints c0 = min(m, spp), c_{j+1} = min(2 c_j, spp); each interval is stratified on its own
 * by the oracle's rule (strataFor) applied to its length.  At a checkpoint below spp the pixel stops when the standard error of the mean luminance of
 * its samples is at most tau x max(mean, PT_ADAPTIVE_FLOOR), evaluated here in float64; the sum of its n samples is stored x spp / n. */
uint64_t orc_render_adaptive(const orc_scene *s, const pt_camera_desc *cam, uint32_t w, uint32_t h, uint32_t spp, uint32_t min_spp, double tau,
                             uint64_t seed, int max_bounces, float *accum, uint32_t *counts, double *margin)
{
	cam_t k = makeCamera(cam);
	uint64_t rays = 0;
	const uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma omp parallel for schedule(dynamic, 1) reduction(+ : rays)
	for (int y = 0; y < (int)h; ++y)
		for (uint32_t x = 0; x < w; ++x)
		{
			const uint32_t pixel = x + (uint32_t)y * w;
			v3 color = V(0.0f, 0.0f, 0.0f);
			double s1 = 0.0, s2 = 0.0, marg = INFINITY;
			uint32_t start = 0, end = min_spp < spp ? min_spp : spp;
			for (;;)
			{
				uint32_t per, bitsA, bitsB;
				strataFor(end - start, &per, &bitsA, &bitsB);
				for (uint32_t i = start; i < end; ++i)
				{
					uint32_t rng[4];
					orc_philox(pixel, i, 0, 0, k0, k1, rng);
					const uint32_t m = i - start;
					if (per && m < (per << (bitsA + bitsB)))
					{
						const uint32_t cell = m / per, a = cell >> bitsB, bMask = (1u << bitsB) - 1u;
						const uint32_t b = (a & 1u) ? bMask - (cell & bMask) : (cell & bMask);
						rng[2] = (a << (32u - bitsA)) | (rng[2] >> bitsA);
						rng[3] = (b << (32u - bitsB)) | (rng[3] >> bitsB);
					}
					float u = (x + orc_uniform(rng[0])) / (float)w;
					float v = (y + orc_uniform(rng[1])) / (float)h;
					ray_t r = cameraRay(&k, u, v);
					const v3 c = s->nodeCount ? getColor(s, r, pixel, i, k0, k1, rng, max_bounces, &rays) : V(0.0f, 0.0f, 0.0f);
					color = vadd(color, c);
					const double lum = 0.2126 * c.x + 0.7152 * c.y + 0.0722 * c.z;
					s1 += lum;
					s2 += lum * lum;
				}
				if (end == spp) break;
				const double n = end, lhs = sqrt(fmax(s2 - s1 * s1 / n, 0.0) / (n * (n - 1.0))), rhs = tau * fmax(s1 / n, (double)PT_ADAPTIVE_FLOOR);
				const double d = fabs(lhs / rhs - 1.0);
				if (d < marg) marg = d;
				if (lhs <= rhs) break;
				start = end;
				end = end > spp / 2u ? spp : 2u * end;
			}
			if (end != spp) color = vscale((float)spp / (float)end, color);
			float *a = accum + (size_t)pixel * 4;
			a[0] = color.x; a[1] = color.y; a[2] = color.z; a[3] = 1.0f;
			counts[pixel] = end;
			margin[pixel] = marg;
		}
	return rays;
}
