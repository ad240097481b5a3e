// `aligner` — drop-in for the binary nimble's front end execs (nimble/__main__.py:154,195-196):
//   aligner --input F [--input F2] -c N --strand_filter S { -r LIB.json -o OUT }... [-t TRIM]   [--gpus N | $NB200_GPUS]
// -r also takes an index file written by `python -m nimble_b200 index` (LIB.nb200idx): no index build at start-up.
// (argv built at nimble/__main__.py:177-192).  Copy it to <site-packages>/nimble/aligner next to
// libnimble_b200.so and the unmodified `python -m nimble align` runs on the B200 backend.
// Exit code 0 on success, non-zero otherwise (forwarded by nimble, __main__.py:198,211).
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "nimble_b200.h"

int main(int argc, char **argv) {
    std::vector<const char *> inputs, libs, outs;
    const char *strand = "unstranded", *trim = "";
    int cores = 0, k = 0, gpus = getenv("NB200_GPUS") ? atoi(getenv("NB200_GPUS")) : 1;
    for (int i = 1; i < argc; i++) {
        const std::string a = argv[i];
        auto need = [&](const char *what) -> const char * {
            if (i + 1 >= argc) { fprintf(stderr, "aligner: %s needs a value\n", what); exit(2); }
            return argv[++i];
        };
        if (a == "--input" || a == "-i") inputs.push_back(need("--input"));
        else if (a == "-c" || a == "--cores") cores = atoi(need("-c"));
        else if (a == "--strand_filter") strand = need("--strand_filter");
        else if (a == "-r" || a == "--reference") libs.push_back(need("-r"));
        else if (a == "-o" || a == "--output") outs.push_back(need("-o"));
        else if (a == "-t" || a == "--trim") trim = need("-t");
        else if (a == "-k" || a == "--kmer") k = atoi(need("-k"));
        else if (a == "--gpus") gpus = atoi(need("--gpus"));
        else { fprintf(stderr, "aligner: unknown argument %s\n", a.c_str()); return 2; }
    }
    if (inputs.empty() || inputs.size() > 2 || libs.empty() || libs.size() != outs.size()) {
        fprintf(stderr, "usage: aligner --input F [--input F2] -c N --strand_filter S {-r LIB.json -o OUT}... [-t TRIM]\n");
        return 2;
    }
    if (gpus > 1) {      // one process, one context per GPU: reads dealt to the GPUs in slabs, outputs in input order
        std::vector<int32_t> devs;
        for (int d = 0; d < gpus; d++) devs.push_back(d);
        char err[1024] = "";
        const int32_t rc = nb200_align_files_multi(devs.data(), gpus, cores, inputs.data(), (int32_t)inputs.size(), libs.data(), (int32_t)libs.size(),
                                                   strand, k, outs.data(), trim, err, sizeof err, nullptr);
        if (rc != NB200_OK) fprintf(stderr, "aligner: %s\n", err);
        return rc == NB200_OK ? 0 : (rc == NB200_ENODEVICE ? 3 : 1);
    }
    nb200_ctx *ctx = nullptr;
    const char *dev = getenv("LOCAL_RANK");
    if (nb200_create(dev ? atoi(dev) : 0, cores, &ctx) != NB200_OK) {
        fprintf(stderr, "aligner: %s\n", nb200_last_error(nullptr));
        return 3;
    }
    std::vector<int32_t> ids(libs.size());
    for (size_t i = 0; i < libs.size(); i++)
        if (nb200_load_library(ctx, libs[i], strand, k, &ids[i]) != NB200_OK) {
            fprintf(stderr, "aligner: %s: %s\n", libs[i], nb200_last_error(ctx));
            nb200_destroy(ctx);
            return 1;
        }
    if (*trim) {     // "<TARGET_LENGTH>:<STRICTNESS>[,...]", one entry per library (nimble/__main__.py:400)
        std::string t(trim);
        size_t a = 0, li = 0;
        bool ok = true;
        while (ok && li < libs.size()) {
            const size_t e = t.find(',', a);
            int tl = 0; double st = 0.0; char tail = 0;
            const std::string item = t.substr(a, e == std::string::npos ? std::string::npos : e - a);
            ok = sscanf(item.c_str(), "%d:%lf%c", &tl, &st, &tail) == 2 && tl >= 0 && nb200_library_set_trim(ctx, ids[li], tl, st) == NB200_OK;
            li++;
            if (e == std::string::npos) break;
            a = e + 1;
        }
        if (!ok || li != libs.size() || t.find(',', a) != std::string::npos) {
            fprintf(stderr, "aligner: -t expects <TARGET_LENGTH>:<STRICTNESS> (strictness 0..1), comma-separated, one entry per library\n");
            nb200_destroy(ctx);
            return 2;
        }
    }
    const int32_t rc = nb200_align_files(ctx, inputs.data(), (int32_t)inputs.size(), ids.data(), outs.data(), (int32_t)libs.size());
    if (rc != NB200_OK) fprintf(stderr, "aligner: %s\n", nb200_last_error(ctx));
    nb200_destroy(ctx);
    return rc == NB200_OK ? 0 : 1;
}
