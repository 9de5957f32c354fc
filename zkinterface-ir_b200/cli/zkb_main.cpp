// zkb — verbs of zki_sieve (rust/src/cli.rs) on the GPU backend.
//   zkb evaluate [--device N] <workspace dir | *.sieve ... | ->       cli.rs:130, 315-320, 557-571
//   zkb evaluate [--device N | --devices a,b,...] --sets DIR <paths...>
//                                                                     one statement per subdirectory of DIR (its value set)
//   zkb flatten --out <dir | -> <workspace dir | *.sieve ... | ->     cli.rs:442-472 (host only)
//   zkb expand-definable --gate-set <s> --out <dir | -> <paths...>    cli.rs:513-553 (host only)
//   zkb validate <workspace dir | *.sieve ... | ->                    cli.rs:297-313 (host only)
//   zkb metrics <workspace dir | *.sieve ... | ->                     cli.rs:322-330 (host only; JSON on stdout)
//   zkb valid-eval-metrics [--device N] <paths...>                    cli.rs:333-363 (all three in one go)
// `evaluate` / `validate` print exactly what the reference prints on stderr ("The statement is TRUE!" /
// "The statement is COMPLIANT with the specification!" / the violation lists) and exit non-zero with
// "Found N violations." when there are any.
#include <dirent.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/stat.h>

#include <algorithm>
#include <string>
#include <vector>

#include "zkb.h"

static int usage(const char* argv0) {
    fprintf(stderr,
            "usage: %s evaluate [--device N | --devices a,b,...] [--sets DIR] <paths...>\n"
            "       %s flatten --out <dir|-> <paths...>\n"
            "       %s expand-definable --gate-set <gateset> --out <dir|-> <paths...>\n"
            "       %s validate <paths...>\n"
            "       %s metrics <paths...>\n"
            "       %s valid-eval-metrics [--device N] <paths...>\n",
            argv0, argv0, argv0, argv0, argv0, argv0);
    fprintf(stderr,
            "  --sets DIR      every subdirectory of DIR is one value set (instance / witness .sieve files); <paths> hold the\n"
            "                  relation and the values common to all sets\n"
            "  --devices LIST  split the sets over these device ordinals (repeats share one device)\n");
    return 2;
}

// print_violations, cli.rs:557-571
static int print_violations(size_t n, const std::vector<std::string>& v, const char* what_it_is_supposed_to_be) {
    fprintf(stderr, "\n");
    if (n > 0) {
        fprintf(stderr, "The statement is NOT %s!\n", what_it_is_supposed_to_be);
        fprintf(stderr, "Violations:\n");
        for (const auto& s : v) fprintf(stderr, "- %s\n", s.c_str());
        fprintf(stderr, "\nError: Found %zu violations.\n", n);
        return 1;
    }
    fprintf(stderr, "The statement is %s!\n", what_it_is_supposed_to_be);
    return 0;
}

// "0,1,1": device ordinals, at least one
static bool parse_devices(const char* list, std::vector<int>& out) {
    std::string s = list;
    size_t pos = 0;
    while (true) {
        size_t comma = s.find(',', pos);
        std::string item = s.substr(pos, comma == std::string::npos ? std::string::npos : comma - pos);
        char* end = nullptr;
        long d = strtol(item.c_str(), &end, 10);
        if (item.empty() || *end != '\0' || d < 0 || d > 1024) return false;
        out.push_back((int)d);
        if (comma == std::string::npos) return true;
        pos = comma + 1;
    }
}

static int fail_with(const char* msg) {
    fprintf(stderr, "Error: %s\n", msg);
    return 1;
}

// zkb evaluate --sets DIR <paths...>: one statement per subdirectory of DIR, each printed as `zkb evaluate <paths...>
// DIR/<name>` prints it, after a "== <name> ==" line
static int evaluate_sets(const char* sets_dir, const std::vector<int>& devs, bool comm, const std::vector<const char*>& paths) {
    std::vector<std::string> names;
    DIR* d = opendir(sets_dir);
    if (!d) {
        fprintf(stderr, "Error: cannot read directory %s\n", sets_dir);
        return 1;
    }
    while (dirent* e = readdir(d)) {
        std::string name = e->d_name;
        struct stat st;
        if (name == "." || name == ".." || stat((std::string(sets_dir) + "/" + name).c_str(), &st) != 0 || !S_ISDIR(st.st_mode)) continue;
        names.push_back(name);
    }
    closedir(d);
    std::sort(names.begin(), names.end());
    if (names.empty()) {
        fprintf(stderr, "Error: no value set (subdirectory) in %s\n", sets_dir);
        return 1;
    }
    std::vector<zkb_ctx*> ctxs;
    for (int dev : devs) {
        ctxs.push_back(zkb_create(dev));
        if (zkb_last_error(ctxs.back())[0]) return fail_with(zkb_last_error(ctxs.back()));
    }
    zkb_evaluator* ev = zkb_evaluator_create(ctxs[0]);
    if (comm) {  // --devices: the contexts form one communicator, the sets are split over them
        if (zkb_comm_init(ctxs.data(), (int)ctxs.size()) != ZKB_OK) return fail_with(zkb_last_error(ctxs[0]));
        if (zkb_evaluator_use_devices(ev, ctxs.data(), (int)ctxs.size()) != ZKB_OK) return fail_with(zkb_evaluator_last_error(ev));
    }
    for (const auto& name : names) {
        const std::string dir = std::string(sets_dir) + "/" + name;
        const char* p = dir.c_str();
        if (zkb_evaluator_add_value_set_paths(ev, &p, 1) != ZKB_OK) return fail_with(zkb_evaluator_last_error(ev));
    }
    if (zkb_evaluator_ingest_paths(ev, paths.data(), paths.size()) != ZKB_OK) return fail_with(zkb_evaluator_last_error(ev));
    size_t not_true = 0;
    for (size_t j = 0; j < names.size(); j++) {
        int status = ZKB_OK;
        size_t n = 0;
        if (zkb_evaluator_batch_result(ev, j, &status, &n) != ZKB_OK) return fail_with(zkb_evaluator_last_error(ev));
        fprintf(stderr, "== %s ==\n", names[j].c_str());
        if (status != ZKB_OK) {
            fprintf(stderr, "Error: %s\n", zkb_evaluator_batch_violation(ev, j, 0));
            not_true++;
            continue;
        }
        std::vector<std::string> v;
        for (size_t i = 0; i < n; i++) v.push_back(zkb_evaluator_batch_violation(ev, j, i));
        not_true += print_violations(n, v, "TRUE") != 0;
    }
    zkb_evaluator_destroy(ev);
    for (auto c : ctxs) zkb_destroy(c);
    if (not_true) {
        fprintf(stderr, "Error: %zu of %zu statements are NOT TRUE.\n", not_true, names.size());
        return 1;
    }
    return 0;
}

int main(int argc, char** argv) {
    if (argc < 3) return usage(argv[0]);
    const std::string verb = argv[1];
    int device = 0;
    bool device_given = false;
    const char* out = nullptr;
    const char* gate_set = nullptr;
    const char* sets_dir = nullptr;
    const char* devices_list = nullptr;
    std::vector<const char*> paths;
    for (int i = 2; i < argc; i++) {
        if (strcmp(argv[i], "--device") == 0 && i + 1 < argc) device = atoi(argv[++i]), device_given = true;
        else if (strcmp(argv[i], "--out") == 0 && i + 1 < argc) out = argv[++i];
        else if (strcmp(argv[i], "--gate-set") == 0 && i + 1 < argc) gate_set = argv[++i];
        else if (verb == "evaluate" && strcmp(argv[i], "--sets") == 0 && i + 1 < argc) sets_dir = argv[++i];
        else if (verb == "evaluate" && strcmp(argv[i], "--devices") == 0 && i + 1 < argc) devices_list = argv[++i];
        else paths.push_back(argv[i]);
    }
    if (verb == "evaluate" && (sets_dir || devices_list)) {
        if (!sets_dir || device_given) return usage(argv[0]);  // --devices needs --sets, and excludes --device
        std::vector<int> devs;
        if (devices_list && !parse_devices(devices_list, devs)) return usage(argv[0]);
        if (devs.empty()) devs.push_back(device);
        return evaluate_sets(sets_dir, devs, devices_list != nullptr, paths);
    }
    if (verb == "evaluate") {
        zkb_ctx* ctx = zkb_create(device);
        if (zkb_last_error(ctx)[0]) {
            fprintf(stderr, "Error: %s\n", zkb_last_error(ctx));
            return 1;
        }
        zkb_evaluator* ev = zkb_evaluator_create(ctx);
        int rc = zkb_evaluator_ingest_paths(ev, paths.data(), paths.size());
        size_t n = 0;
        if (rc == ZKB_OK) rc = zkb_evaluator_get_violations(ev, &n);
        if (rc != ZKB_OK) {
            fprintf(stderr, "Error: %s\n", zkb_evaluator_last_error(ev));
            return 1;
        }
        std::vector<std::string> v;
        for (size_t i = 0; i < n; i++) v.push_back(zkb_evaluator_violation(ev, i));
        int status = print_violations(n, v, "TRUE");
        zkb_evaluator_destroy(ev);
        zkb_destroy(ctx);
        return status;
    }
    if (verb == "flatten" || verb == "expand-definable") {
        if (!out) return usage(argv[0]);
        if (verb == "expand-definable" && !gate_set) return 0;  // main_expand_definable does nothing without --gate-set (cli.rs:521)
        zkb_ctx* ctx = zkb_create(-1);
        zkb_evaluator* ev = zkb_evaluator_create(ctx);
        int rc = verb == "flatten" ? zkb_evaluator_set_flatten(ev, 1) : zkb_evaluator_set_expand_definable(ev, gate_set);
        if (rc == ZKB_OK) rc = zkb_evaluator_ingest_paths(ev, paths.data(), paths.size());
        if (rc == ZKB_OK) {
            if (strcmp(out, "-") == 0) {  // MemorySink, then instance / witness / relation messages to stdout
                const uint8_t* p[3];
                size_t n[3];
                rc = zkb_evaluator_flatten(ev, &p[0], &n[0], &p[1], &n[1], &p[2], &n[2]);
                for (int i = 0; i < 3 && rc == ZKB_OK; i++)
                    if (n[i]) fwrite(p[i], 1, n[i], stdout);
            } else {
                rc = zkb_evaluator_flatten_to_dir(ev, out);
            }
        }
        if (rc != ZKB_OK) {
            fprintf(stderr, "Error: %s\n", zkb_evaluator_last_error(ev));
            return 1;
        }
        zkb_evaluator_destroy(ev);
        zkb_destroy(ctx);
        return 0;
    }
    if (verb == "validate") {
        zkb_validator* val = zkb_validator_create(1);  // main_validate validates as prover (cli.rs:301)
        int rc = zkb_validator_ingest_paths(val, paths.data(), paths.size());
        size_t n = 0;
        if (rc == ZKB_OK) rc = zkb_validator_get_violations(val, &n);
        if (rc != ZKB_OK) {
            fprintf(stderr, "Error: %s\n", zkb_validator_last_error(val));
            return 1;
        }
        std::vector<std::string> v;
        for (size_t i = 0; i < n; i++) v.push_back(zkb_validator_violation(val, i));
        int status = print_violations(n, v, "COMPLIANT with the specification");
        zkb_validator_destroy(val);
        return status;
    }
    if (verb == "metrics") {
        zkb_metrics* m = zkb_metrics_create();
        if (zkb_metrics_ingest_paths(m, paths.data(), paths.size()) != ZKB_OK) {
            fprintf(stderr, "Error: %s\n", zkb_metrics_last_error(m));
            return 1;
        }
        printf("%s\n", zkb_metrics_json(m));
        zkb_metrics_destroy(m);
        return 0;
    }
    if (verb == "valid-eval-metrics") {  // main_valid_eval_metrics: validator (as prover), evaluator and stats on the same messages
        zkb_validator* val = zkb_validator_create(1);
        zkb_metrics* m = zkb_metrics_create();
        zkb_ctx* ctx = zkb_create(device);
        if (zkb_last_error(ctx)[0]) {
            fprintf(stderr, "Error: %s\n", zkb_last_error(ctx));
            return 1;
        }
        zkb_evaluator* ev = zkb_evaluator_create(ctx);
        const bool from_stdin = paths.size() == 1 && strcmp(paths[0], "-") == 0;
        std::vector<uint8_t> piped;  // stdin can be read only once: the three consumers share the bytes
        if (from_stdin) {
            uint8_t chunk[1 << 16];
            size_t got;
            while ((got = fread(chunk, 1, sizeof chunk, stdin)) > 0) piped.insert(piped.end(), chunk, chunk + got);
        }
        int rc = from_stdin ? zkb_validator_ingest_buffer(val, piped.data(), piped.size())
                            : zkb_validator_ingest_paths(val, paths.data(), paths.size());
        if (rc != ZKB_OK) {
            fprintf(stderr, "Error: %s\n", zkb_validator_last_error(val));
            return 1;
        }
        rc = from_stdin ? zkb_evaluator_ingest_buffer(ev, piped.data(), piped.size())
                        : zkb_evaluator_ingest_paths(ev, paths.data(), paths.size());
        if (rc != ZKB_OK) {
            fprintf(stderr, "Error: %s\n", zkb_evaluator_last_error(ev));
            return 1;
        }
        rc = from_stdin ? zkb_metrics_ingest_buffer(m, piped.data(), piped.size())
                        : zkb_metrics_ingest_paths(m, paths.data(), paths.size());
        if (rc != ZKB_OK) {
            fprintf(stderr, "Error: %s\n", zkb_metrics_last_error(m));
            return 1;
        }
        size_t n1 = 0, n2 = 0;
        if (zkb_validator_get_violations(val, &n1) != ZKB_OK) {
            fprintf(stderr, "Error: %s\n", zkb_validator_last_error(val));
            return 1;
        }
        if (zkb_evaluator_get_violations(ev, &n2) != ZKB_OK) {
            fprintf(stderr, "Error: %s\n", zkb_evaluator_last_error(ev));
            return 1;
        }
        std::vector<std::string> v1, v2;
        for (size_t i = 0; i < n1; i++) v1.push_back(zkb_validator_violation(val, i));
        for (size_t i = 0; i < n2; i++) v2.push_back(zkb_evaluator_violation(ev, i));
        int res1 = print_violations(n1, v1, "COMPLIANT with the specification");
        int res2 = print_violations(n2, v2, "TRUE");
        printf("%s\n", zkb_metrics_json(m));
        return res1 ? res1 : res2;
    }
    return usage(argv[0]);
}
