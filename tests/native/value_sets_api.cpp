// zkb.hpp mirror of value sets: the golden `example` relation checked for its own witness and for the witness of
// `example_incorrect` in one batch, on one context (argv[1]: tests/golden).
#include <cstdio>
#include <string>
#include <vector>

#include "zkb.hpp"

int main(int argc, char** argv) {
    if (argc < 2) return 2;
    const std::string g = argv[1];
    zkb::GpuBackend b(0);
    zkb::Evaluator e(b);
    e.add_value_set(zkb::Source::from_dirs_and_files({g + "/example/001_witness.sieve"}));
    e.add_value_set(zkb::Source::from_dirs_and_files({g + "/example_incorrect/001_witness.sieve"}));
    e.from_messages(zkb::Source::from_dirs_and_files({g + "/example/000_instance.sieve", g + "/example/002_relation.sieve"}));
    auto r = e.get_batch_violations();
    if (r.size() != 2 || r[0].status != ZKB_OK || !r[0].violations.empty() || r[1].status != ZKB_OK || r[1].violations.size() != 1 ||
        r[1].violations[0] != "Wire_9 (may be weighted) should be 0, while it is not") {
        fprintf(stderr, "unexpected batch result\n");
        return 1;
    }
    zkb::GpuBackend single(0);
    zkb::Evaluator one(single);
    one.from_messages(zkb::Source::from_directory(g + "/example"));
    if (!one.get_violations().empty()) return 1;
    int codes[2] = {0, 0};  // every wire of the example is freed at the end: no value, in both
    try { one.get(8); } catch (const zkb::Error& err) { codes[0] = err.code; }
    try { e.get(0, 8); } catch (const zkb::Error& err) { codes[1] = err.code; }
    if (codes[0] != ZKB_E_SEMANTIC || codes[1] != ZKB_E_SEMANTIC) {
        fprintf(stderr, "Evaluator::get of a freed wire: %d / %d\n", codes[0], codes[1]);
        return 1;
    }
    try {
        e.get(2, 8);
        return 1;
    } catch (const zkb::Error& err) {
        if (err.code != ZKB_E_ARG) return 1;
    }
    printf("value_sets_api ok\n");
    return 0;
}
