// Host-side test tool for the CLI's --eqclasses merge and text form (eqclasses.hpp; no device code, no CUDA): used by
// tests/test_eqclasses.py.  stdin:
//   <n_names> then one name per line (a name may be empty)
//   <n_tables>, then per table <n_classes> and per class a line `<count> <len> <id_1> ... <id_len>`
// stdout: eq_format(eq_merge(tables), names).
#include <cstdio>
#include <iostream>
#include <string>

#include "eqclasses.hpp"

int main()
{
    size_t n_names = 0, n_tables = 0;
    std::cin >> n_names;
    std::string line;
    std::getline(std::cin, line);
    std::vector<std::string> names(n_names);
    for (auto &nm : names) std::getline(std::cin, nm);
    std::cin >> n_tables;
    std::vector<shkhost::EqTable> tables(n_tables);
    for (auto &t : tables) {
        size_t n = 0;
        std::cin >> n;
        for (size_t i = 0; i < n; ++i) {
            uint64_t count = 0, len = 0;
            std::cin >> count >> len;
            for (uint64_t k = 0; k < len; ++k) {
                uint32_t id = 0;
                std::cin >> id;
                t.ids.push_back(id);
            }
            t.offsets.push_back(t.ids.size());
            t.counts.push_back(count);
        }
    }
    if (!std::cin) return 2;
    const std::string txt = shkhost::eq_format(shkhost::eq_merge(tables), names);
    fwrite(txt.data(), 1, txt.size(), stdout);
    return 0;
}
