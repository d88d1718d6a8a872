#include "light_sampling.h"
#include <algorithm>
#include <cmath>
#include <utility>

namespace ptb
{
double localArea(uint32_t type)
{
	const double pi = 3.14159265358979323846;
	switch (type)
	{
	case PT_SPHERE: return 4.0 * pi;
	case PT_CYLINDER: return 4.0 * pi;
	case PT_DISK: return pi;
	case PT_CONE: return 2.0 * std::sqrt(2.0) * pi;
	case PT_PARABOLOID: return pi * (5.0 * std::sqrt(5.0) - 1.0) / 6.0;
	case PT_QUAD: return 4.0;
	default: return 24.0; // PT_CUBE
	}
}

void buildLightTable(CompiledScene &cs, LightTable &out)
{
	out.recs.clear();
	out.sceneIndex.clear();
	out.probability.clear();
	std::vector<std::pair<uint32_t, uint32_t>> em; // (scene index, primitive index)
	for (size_t i = 0; i < cs.prims.size(); ++i)
	{
		cs.mats[i].pad[0] = 0;
		const float *e = cs.mats[i].emissive;
		if (e[0] != 0.0f || e[1] != 0.0f || e[2] != 0.0f) em.emplace_back(cs.prims[i].packed & kPrimSceneMask, uint32_t(i));
	}
	std::sort(em.begin(), em.end());
	const size_t n = em.size();
	std::vector<LightRec> recs(n);
	std::vector<double> w(n, 0.0), det(n, 0.0);
	double total = 0.0;
	for (size_t k = 0; k < n; ++k)
	{
		const Prim &p = cs.prims[em[k].second];
		const uint32_t type = (p.packed >> kPrimTypeShift) & 7u;
		const float *rows[3] = { p.row0, p.row1, p.row2 };
		double W[3][3], t[3];
		for (int r = 0; r < 3; ++r)
		{
			for (int c = 0; c < 3; ++c) W[r][c] = rows[r][c];
			t[r] = rows[r][3];
		}
		const double dW = W[0][0] * (W[1][1] * W[2][2] - W[1][2] * W[2][1]) - W[0][1] * (W[1][0] * W[2][2] - W[1][2] * W[2][0]) +
		                  W[0][2] * (W[1][0] * W[2][1] - W[1][1] * W[2][0]);
		LightRec &L = recs[k];
		for (float &x : L.m) x = 0.0f;
		L.packed = em[k].second | (type << kPrimTypeShift);
		if (!(std::isfinite(dW) && dW != 0.0)) continue; // a degenerate transform: weight 0, never selected
		// M = W^-1 (adjugate / determinant), translation -M t
		double M[3][3];
		M[0][0] = (W[1][1] * W[2][2] - W[1][2] * W[2][1]) / dW;
		M[0][1] = (W[0][2] * W[2][1] - W[0][1] * W[2][2]) / dW;
		M[0][2] = (W[0][1] * W[1][2] - W[0][2] * W[1][1]) / dW;
		M[1][0] = (W[1][2] * W[2][0] - W[1][0] * W[2][2]) / dW;
		M[1][1] = (W[0][0] * W[2][2] - W[0][2] * W[2][0]) / dW;
		M[1][2] = (W[0][2] * W[1][0] - W[0][0] * W[1][2]) / dW;
		M[2][0] = (W[1][0] * W[2][1] - W[1][1] * W[2][0]) / dW;
		M[2][1] = (W[0][1] * W[2][0] - W[0][0] * W[2][1]) / dW;
		M[2][2] = (W[0][0] * W[1][1] - W[0][1] * W[1][0]) / dW;
		for (int r = 0; r < 3; ++r)
		{
			for (int c = 0; c < 3; ++c) L.m[4 * r + c] = float(M[r][c]);
			L.m[4 * r + 3] = float(-(M[r][0] * t[0] + M[r][1] * t[1] + M[r][2] * t[2]));
		}
		const double dM = std::fabs(1.0 / dW);
		// world area: flat faces by Nanson's formula (|det M| |W^T n_l| per unit of local area; W^T e_k = row k of W), curved shapes by the
		// uniform-scale value - any positive estimate keeps the estimator unbiased, only P_sel enters the pdf
		auto rowLen = [&](int r) { return std::sqrt(W[r][0] * W[r][0] + W[r][1] * W[r][1] + W[r][2] * W[r][2]); };
		double area;
		if (type == PT_QUAD || type == PT_DISK) area = localArea(type) * dM * rowLen(1);
		else if (type == PT_CUBE) area = 8.0 * dM * (rowLen(0) + rowLen(1) + rowLen(2));
		else area = localArea(type) * std::cbrt(dM * dM);
		const float *e = cs.mats[em[k].second].emissive;
		const double mean = (double(e[0]) + double(e[1]) + double(e[2])) / 3.0;
		w[k] = mean > 0.0 && std::isfinite(area) ? mean * area : 0.0;
		det[k] = dM;
		total += w[k];
	}
	if (!(total > 0.0 && std::isfinite(total))) return; // nothing that emits: the option leaves the render alone
	std::vector<double> scaled(n);
	out.probability.resize(n);
	out.sceneIndex.resize(n);
	for (size_t k = 0; k < n; ++k)
	{
		const double P = w[k] / total;
		const uint32_t type = (recs[k].packed >> kPrimTypeShift) & 7u;
		recs[k].pdfScale = P > 0.0 ? float(P / (localArea(type) * det[k])) : 0.0f;
		out.probability[k] = float(P);
		out.sceneIndex[k] = em[k].first;
		scaled[k] = P * double(n);
		cs.mats[em[k].second].pad[0] = uint32_t(k) + 1u;
	}
	// Vose's alias method; the work lists are filled in index order and used as stacks
	std::vector<uint32_t> small, large;
	auto put = [&](uint32_t i, double q, uint32_t other)
	{
		recs[i].aliasQ = float(q < 0.0 ? 0.0 : (q > 1.0 ? 1.0 : q));
		recs[i].alias = other;
	};
	for (size_t i = 0; i < n; ++i) (scaled[i] < 1.0 ? small : large).push_back(uint32_t(i));
	while (!small.empty() && !large.empty())
	{
		const uint32_t s = small.back(), l = large.back();
		small.pop_back();
		put(s, scaled[s], l);
		scaled[l] = (scaled[l] + scaled[s]) - 1.0;
		if (scaled[l] < 1.0) { large.pop_back(); small.push_back(l); }
	}
	for (uint32_t i : large) put(i, 1.0, i);
	for (uint32_t i : small) put(i, 1.0, i); // only through rounding
	out.recs = std::move(recs);
}
} // namespace ptb
