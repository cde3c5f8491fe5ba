// gen_classes.cpp -- writes pokegym_b200/csrc/gb_classes.inc (tools/gen_classes.sh) from the per-opcode base table of
// gb_predecode.h and the class mix of the benchmark workloads (tools/class_counts.txt, tools/class_mix.py).
#include <cstdio>
#include <map>
#include <string>
#include <vector>
#define GB_NO_CLASS_LOOKUP 1
#include "gb_predecode.h"

struct Cls { unsigned h, f; double n; };
static std::vector<Cls> cls;
static std::vector<double> wsum;  // wsum[i] = weight of ids < i
static std::map<std::pair<int, int>, std::pair<double, int>> memo;  // (lo, hi) -> (expected tests, choice: 0 = peel lo, m = split at m)

// Least expected number of tests that find the id c in [lo, hi) (hi == N: c may also be >= N, an instruction without a class),
// each test being `c == lo` (peel the hottest id of the range: ids are in order of frequency) or `c < m` (split).
static double cost(int lo, int hi) {
    const int N = (int)cls.size();
    if (hi - lo == 1 && hi < N) return 0.0;
    auto it = memo.find({lo, hi});
    if (it != memo.end()) return it->second.first;
    const double w = wsum[hi] - wsum[lo] + (hi == N ? 1.0 : 0.0);  // weight 1 for the out-of-class instructions
    double best = w + (hi - lo == 1 ? 0.0 : cost(lo + 1, hi));
    int choice = 0;
    for (int m = lo + 1; m < hi; m++) {
        const double c = w + cost(lo, m) + cost(m, hi);
        if (c < best) { best = c; choice = m; }
    }
    memo[{lo, hi}] = {best, choice};
    return best;
}

static void emit(int lo, int hi, int depth) {
    const int N = (int)cls.size();
    const std::string in(4 * depth, ' ');
    if (hi - lo == 1 && hi < N) {
        printf("%s  L(%d, %u, 0x%04xu) \\\n", in.c_str(), lo, cls[lo].h, cls[lo].f);
        return;
    }
    const int m = memo.at({lo, hi}).second;
    if (m == 0) {
        printf("%sif (GB_CLS_TEST((c) == %du)) { \\\n%s  L(%d, %u, 0x%04xu) \\\n%s} else { \\\n", in.c_str(), lo, in.c_str(), lo, cls[lo].h, cls[lo].f, in.c_str());
        if (hi - lo == 1) printf("%s  OTHER \\\n", in.c_str());
        else emit(lo + 1, hi, depth + 1);
    } else {
        printf("%sif (GB_CLS_TEST((c) < %du)) { \\\n", in.c_str(), m);
        emit(lo, m, depth + 1);
        printf("%s} else { \\\n", in.c_str());
        emit(m, hi, depth + 1);
    }
    printf("%s} \\\n", in.c_str());
}

int main(int argc, char **argv) {
    pd_desc_t t[512];
    pd_build_base(t);
    std::map<std::pair<unsigned, unsigned>, int> m;
    for (int i = 0; i < 512; i++) {
        unsigned h = t[i].x & 0xFF, f = t[i].w & 0xFFF0u;
        if (h < H_RARE) m[{h, f}]++;
    }
    FILE *in = argc > 1 ? fopen(argv[1], "r") : nullptr;
    if (!in) { fprintf(stderr, "usage: gen_classes tools/class_counts.txt\n"); return 1; }
    char line[256];
    while (fgets(line, sizeof line, in)) {  // "handler flags count", hottest first
        unsigned h, f;
        double n;
        if (line[0] == '#' || sscanf(line, "%u %x %lf", &h, &f, &n) != 3) continue;
        auto it = m.find({h, f});
        if (it == m.end()) { fprintf(stderr, "counted pair h=%u f=%04x is not a class\n", h, f); return 1; }
        cls.push_back({h, f, n});
        m.erase(it);
    }
    fclose(in);
    for (auto &kv : m) cls.push_back({kv.first.first, kv.first.second, 0.0});  // never seen in the benchmark workloads
    const int N = (int)cls.size();
    wsum.assign(N + 1, 0.0);
    for (int i = 0; i < N; i++) wsum[i + 1] = wsum[i] + cls[i].n;
    const double expected = cost(0, N) / wsum[N];

    printf("// gb_classes.inc -- GENERATED (tools/gen_classes.sh): every (handler, operand flags) pair the per-opcode base table of\n"
           "// gb_predecode.h produces for the fast set, one dense id each, in order of frequency in the benchmark workloads\n"
           "// (tools/class_counts.txt): nvcc lays the class bodies out in id order, so the bodies a game runs sit next to each other.\n"
           "// GB_CLS(id, handler, flags): the single-lane build of the interpreter dispatches on the id to an instance of the\n"
           "// instruction body in which both are compile-time constants.\n"
           "#if defined(GB_CLS)\n");
    for (int i = 0; i < N; i++) printf("GB_CLS(%d, %u, 0x%04xu)\n", i, cls[i].h, cls[i].f);
    printf("#endif\n#define GB_CLS_COUNT %d\n", N);
    printf("// GB_CLS_DISPATCH(c, L, OTHER): L(id, handler, flags) for the class id c, OTHER when c >= GB_CLS_COUNT.  A tree of tests\n"
           "// shaped by the class counts for the fewest expected tests (%.2f per instruction of the workloads counted): the hottest\n"
           "// ids are peeled off first by `c == id`, ranges of colder ones are split by `c < m`.  GB_CLS_TEST wraps every test.\n"
           "#define GB_CLS_DISPATCH(c, L, OTHER) \\\n", expected);
    emit(0, N, 0);
    printf("\n");
}
