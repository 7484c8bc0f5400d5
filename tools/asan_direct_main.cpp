#include "../include/ibo_b200.h"
#include "../ibo_b200/csrc/options.h"
#include <cstdio>
#include <cmath>
#include <string>
#include <vector>
#include <random>
namespace ibo { void set_error(const std::string&) {} int eval_neg_acq(ibo_model*, const double*, long, int, double, double, int, ScoreForce, double*) { return -2; } }
extern "C" int ibo_comm_size(void) { return 1; }
extern "C" int ibo_comm_rank(void) { return 0; }
extern "C" int ibo_comm_allgather(const double*, long, double*) { return -5; }
extern "C" int ibo_model_dim(const ibo_model*) { return 0; }
struct Obj { int d; std::vector<double> c; int kind; long calls; };
static void cb(void* u, long n, int nd, const double* X, double* y) {
    Obj* o = (Obj*)u; o->calls += n;
    for (long p = 0; p < n; p++) {
        double s = 0;
        for (int j = 0; j < nd; j++) { double t = X[p * nd + j] - o->c[j]; s += (1 + j) * t * t + 0.2 * std::sin(9 * X[p * nd + j]); }
        if (o->kind == 1) s = std::floor(4 * s) / 4;
        if (o->kind == 2) s = 1.0;
        y[p] = s;
    }
}
int main() {
    std::mt19937 g(1);
    std::uniform_real_distribution<double> U(0, 1);
    for (int rep = 0; rep < 60; rep++) {
        int d = 1 + rep % 24;
        std::vector<double> lb(d), ub(d);
        Obj o{d, std::vector<double>(d), rep % 3, 0};
        for (int j = 0; j < d; j++) { lb[j] = (rep % 2) ? 0.0 : -1.0 + U(g); ub[j] = lb[j] + 0.5 + 2 * U(g); o.c[j] = (rep % 4 == 0) ? lb[j] : lb[j] + U(g) * (ub[j] - lb[j]); }
        if (d > 2 && rep % 5 == 0) ub[d - 1] = lb[d - 1];
        double res[3][2]; long ns[3];
        int flagsv[3] = {0, IBO_FLAG_DIRECT_SEQ, IBO_FLAG_DIRECT_SPECULATE};
        for (int m = 0; m < 3; m++) {
            std::vector<double> xmin(d); double fmin; int it;
            int rc = ibo_direct_batched(cb, &o, d, lb.data(), ub.data(), 8 + rep % 30, 100000, (rep % 7 == 0) ? 500 : 1000000, flagsv[m], &fmin, xmin.data(), &ns[m], &it);
            if (rc) { printf("rc %d\n", rc); return 1; }
            res[m][0] = fmin; res[m][1] = xmin[0];
        }
        if (res[0][0] != res[1][0] || res[0][0] != res[2][0] || ns[0] != ns[1] || ns[0] != ns[2] || res[0][1] != res[2][1]) { printf("MISMATCH rep %d\n", rep); return 1; }
    }
    printf("asan run ok\n");
    return 0;
}
extern "C" int ibo_model_create_from_inverse(int, int, const double*, int, const double*, const double*, int, int, double, const double*, double, int, const double*, const double*, double, const double*, const double*, ibo_model**, int*) { return -2; }
extern "C" int ibo_model_destroy(ibo_model*) { return 0; }
