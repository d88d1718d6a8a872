// light_sampling.h — the emitter table of option "light_is": next-event estimation of emissive objects with multiple importance
// sampling.  Not in the reference, which finds an emitter only when a BSDF-sampled ray happens to hit it (kernels/trace.cu:136-151).
//
// With "light_is" every scattering vertex also draws one point on an emissive primitive - the emitter by an alias table over
// selection weights, the point uniformly by LOCAL area on the primitive's canonical surface, mapped to the world by the primitive's
// local->world map M - and traces a shadow ray to it.  The two strategies are combined by the balance heuristic.  Same integral as
// the reference's estimator (paths of at most max_bounces segments, emission added at hits 1..5), so the image converges to the
// reference's picture.
//
// Area pdf in world space of a point sampled uniformly by local area A_l (Nanson's formula, exact for any invertible M):
//   p_A(x) = 1 / (A_l |det M| |W^T n_l|),  W = M^-1 (the world->local rows of the Prim record), n_l the UNIT local normal at x;
// solid-angle pdf seen from p with unit direction w and distance d:  P_sel p_A d^2 / |cos_l| = P_sel / (A_l |det M|) * d^2 / |(W^T n_l) . w|.
// The record keeps the constant factor P_sel / (A_l |det M|), so both the light sample and the MIS weight at a BSDF hit need
// one dot product with the (unnormalised) world normal W^T n_l.
#pragma once
#include "scene_compile.h"
#include <cstdint>
#include <vector>

namespace ptb
{
// One emitter = 64 bytes, read with __ldg (trace_device.cuh sampleLight / lightPdf):
//   m[0..11]  local->world map M, three rows of four (inverted in double from the primitive's world->local rows)
//   pdfScale  P_sel / (A_l |det M|)
//   aliasQ    acceptance threshold of this emitter's alias-table entry (Vose)
//   alias     alias emitter of the entry
//   packed    primitive index (BVH order, bits 0..23) | shape type << 24
struct alignas(16) LightRec
{
	float m[12];
	float pdfScale;
	float aliasQ;
	uint32_t alias;
	uint32_t packed;
};
static_assert(sizeof(LightRec) == 64, "LightRec must be 64 bytes");

struct LightTable
{
	std::vector<LightRec> recs;      // emitters in scene order (the index of the object in the caller's array)
	std::vector<uint32_t> sceneIndex; // per emitter: its scene index
	std::vector<float> probability;   // per emitter: selection probability P_sel
};

// Local surface area of the canonical shapes: sphere 4 pi, cylinder 4 pi, disk pi, cone 2 sqrt(2) pi, paraboloid pi (5 sqrt 5 - 1) / 6,
// quad 4, cube 24 (indexed by PT_SPHERE .. PT_CUBE)
double localArea(uint32_t type);

// Every primitive with a non-zero emissive channel is one emitter.  Selection weight = mean emissive x world area (exact for
// disk / quad / cube; |det M|^(2/3) A_l for the curved shapes, exact under uniform scale).  One alias table over the emitters
// (Vose's method, work lists filled in index order and used as stacks, as buildEnvDistribution): deterministic, the oracle
// restatement gets the same bits.  Also stores each primitive's emitter index + 1 in Mat::pad[0] (0: not an emitter).
void buildLightTable(CompiledScene &cs, LightTable &out);
} // namespace ptb
