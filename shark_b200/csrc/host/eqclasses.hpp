// --eqclasses: the per-context class tables of shk_eq_classes merged into one, and its text form.
#pragma once
#include <algorithm>
#include <cstdint>
#include <string>
#include <vector>

namespace shkhost {

// One class table as shk_eq_classes returns it: class i is ids[offsets[i], offsets[i+1]), counts[i] reads.
struct EqTable {
    std::vector<uint64_t> offsets{0};
    std::vector<uint32_t> ids;
    std::vector<uint64_t> counts;
    size_t size() const { return counts.size(); }
};

// The classes of every table, equal id lists summed, in lexicographic order of the lists (the order of each input).
inline EqTable eq_merge(const std::vector<EqTable> &tables)
{
    struct Ref {
        const uint32_t *p;
        uint64_t n, count;
    };
    std::vector<Ref> all;
    for (const EqTable &t : tables)
        for (size_t i = 0; i < t.size(); ++i)
            all.push_back({t.ids.data() + t.offsets[i], t.offsets[i + 1] - t.offsets[i], t.counts[i]});
    auto less = [](const Ref &x, const Ref &y) { return std::lexicographical_compare(x.p, x.p + x.n, y.p, y.p + y.n); };
    std::stable_sort(all.begin(), all.end(), less);
    EqTable out;
    for (size_t i = 0; i < all.size();) {
        size_t j = i + 1;
        uint64_t count = all[i].count;
        for (; j < all.size() && !less(all[i], all[j]); ++j) count += all[j].count;
        if (count) {
            out.ids.insert(out.ids.end(), all[i].p, all[i].p + all[i].n);
            out.offsets.push_back(out.ids.size());
            out.counts.push_back(count);
        }
        i = j;
    }
    return out;
}

// `<count> <name_1> ... <name_n>` per class, the name of index g the one the ssv prints for it (legend[g], empty past
// the legend: SURVEY.md App. C Q1).
inline std::string eq_format(const EqTable &t, const std::vector<std::string> &legend)
{
    std::string txt;
    for (size_t i = 0; i < t.size(); ++i) {
        txt += std::to_string(t.counts[i]);
        for (uint64_t k = t.offsets[i]; k < t.offsets[i + 1]; ++k) {
            txt += ' ';
            if (t.ids[k] < legend.size()) txt += legend[t.ids[k]];
        }
        txt += '\n';
    }
    return txt;
}

}  // namespace shkhost
