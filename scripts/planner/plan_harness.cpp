// plan digest + timing harness (no CUDA).  Build: g++ -O3 -std=c++17 -DPLAN_CPP='"path/plan.cpp"' harness.cpp -lpthread
#include PLAN_CPP
#include <chrono>
#include <cstdio>
#include <cstring>
#include <fstream>
namespace genlib { int set_error(int code, const std::string &) { return code; } }
using namespace genlib;
int main(int argc, char **argv) {
    // args: file world schedule reps [stream]
    const char *file = argv[1]; int world = atoi(argv[2]), sched = atoi(argv[3]), reps = atoi(argv[4]); bool stream = argc > 5 && atoi(argv[5]);
    const char *name = strrchr(file, '/') ? strrchr(file, '/') + 1 : file;   // (a bare file name has no '/')
    std::ifstream fh(file, std::ios::binary);
    int64_t hd[2]; fh.read((char *)hd, 16);
    std::vector<int32_t> fa(hd[0]), mo(hd[0]), pro(hd[1]); std::vector<int64_t> ids(hd[0]);
    fh.read((char *)fa.data(), 4 * hd[0]); fh.read((char *)mo.data(), 4 * hd[0]); fh.read((char *)ids.data(), 8 * hd[0]); fh.read((char *)pro.data(), 4 * hd[1]);
    // schedule 4 (pairs): every proband with the one a third of the list further on, every fifth with itself
    const bool pairs = sched == 4;
    std::vector<int32_t> pa, pb;
    for (int64_t i = 0; pairs && i < hd[1]; i++) { pa.push_back(pro[i]); pb.push_back(i % 5 ? pro[(i + hd[1] / 3) % hd[1]] : pro[i]); }
    const PairList pl{(int64_t)pa.size(), pa.data(), pb.data()};
    const int32_t n_pro = pairs ? 0 : (int32_t)hd[1];
    double best = 1e30, best_first = 1e30; uint64_t dg = 0; int rc = 0; std::string err;
    for (int r = 0; r < reps; r++) {
        Plan P; adopt_retired_storage(P);
        PlanStream ps;
        auto t0 = std::chrono::steady_clock::now();
        double first = 0;
        if (stream) {
            std::thread w([&] { rc = build_plan((int32_t)hd[0], fa.data(), mo.data(), sched ? ids.data() : nullptr, n_pro, pro.data(), world, sched, P, err, &ps, 0, pl); });
            ps.wait([&] { return ps.layers_done.load() >= 1 || ps.stage.load() == 2; });
            first = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
            w.join();
        } else rc = build_plan((int32_t)hd[0], fa.data(), mo.data(), sched ? ids.data() : nullptr, n_pro, pro.data(), world, sched, P, err, nullptr, 0, pl);
        double ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
        best = std::min(best, ms); best_first = std::min(best_first, first);
        dg = plan_digest(P, !stream);
        retire_storage(P);
    }
    std::printf("%s w%d s%d%s rc %d digest %016llx", name, world, sched, stream ? " stream" : "", rc, (unsigned long long)dg);
    std::fprintf(stderr, "   %s w%d s%d: best %.1f ms, first layer after %.1f ms\n", name, world, sched, best, best_first);
    std::printf("\n");
    return 0;
}
