// Host-side state of the IPA producers (include/speechPlayer_ipa.h), shared by the host producer (ipa_frames.cpp) and the
// device producer (ipa_device.cu): the phoneme table as sorted arrays, and the pitch factors of one call.
#pragma once
#include <cstdint>
#include <vector>

#include "ipa_core.h"

struct speechPlayer_ipaTable {
	uint64_t id = 0;               // unique per table for the life of the process (device copies are cached by it)
	std::vector<uint64_t> keys;    // sorted packed keys (ipa::packKey)
	std::vector<uint8_t> flags;
	std::vector<uint64_t> present;
	std::vector<double> values;    // [n][47]
	int h = -1;
	ipa::TableView view() const {
		return ipa::TableView{keys.data(), flags.data(), present.data(), values.data(), (int)keys.size(), h};
	}
};

namespace ipa {

// pitchPath's factors for one call.  table: the percents of every clause type ([kClauseTypes][kMaxPercents], ipaPercents),
// then the factors of every distinct (clause type, inflection) of the call ([groups][kMaxPercents], std::pow).  group[i]
// is text i's row (empty when every text uses row 0).
struct PitchPlan {
	std::vector<double> table;
	std::vector<int32_t> group;
	int groups = 0;
	const double *pct(int clause) const { return table.data() + (size_t)clause * kMaxPercents; }
	const double *factor(int g) const { return table.data() + (size_t)(kClauseTypes + g) * kMaxPercents; }
	Factors factors(unsigned int text, int clause) const {
		return Factors{pct(clause), factor(group.empty() ? 0 : group[text])};
	}
};
void planPitches(PitchPlan &plan, const double *inflection, const char *clauseType, unsigned int numTexts);

}  // namespace ipa
