// Batched DIRECT: the reference's rectangle rules (cpp/direct.cpp:49-65 Rectangle, :111-141 samplef,
// :146-235 divrec, :372-498 selection + division order) restructured so that every iteration issues
// one batch -- all probe points of all potentially-optimal rectangles together with every child centre that does
// not depend on the division order (all but a few per thousand), the rest in a second, small batch --
// instead of one objective call per sample.  Floating-point expressions that decide control flow
// (side lengths, centre-to-vertex distances, slopes, the epsilon test) are written exactly as the
// reference writes them so that, on identical objective values, the trajectory is identical:
// same samples, same rectangles, same (FMIN, XMIN, nsamples).
//
// The potentially-optimal test is evaluated once per distance class (O(C^2) per iteration) instead of
// the reference's O(R^2) pair scan, on the same slope expressions, with bit-identical accept / reject
// decisions (see select(); SURVEY.md section 3.3).
#include "../../include/ibo_b200.h"
#include "options.h"
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <ctime>
#include <limits>
#include <map>
#include <memory>
#include <set>
#include <unordered_map>
#include <string>
#include <utility>
#include <vector>
#include <chrono>
#include <cstdio>
#include <thread>

namespace ibo {
void set_error(const std::string& s);
int eval_neg_acq(ibo_model* m, const double* Xs, long n, int acq, double ymax, double parm, int flags, ScoreForce force, double* y);
int batch_uses_i8(ibo_model* m, long n, int flags);
bool tiny_server_fits(const ibo_model* m, long n);
int tiny_server_eval(ibo_model* m, const double* X, long n, int acq, double ymax, double parm, int flags, double* y);
void tiny_server_stop(ibo_model* m);

namespace {

typedef std::pair<unsigned, double> ind_val;
bool sort_by_val(const ind_val& a, const ind_val& b) { return a.second < b.second; }   // cpp/direct.cpp:44-47

const double MAX_DOUBLE = std::numeric_limits<double>::max();
const double MIN_DOUBLE = std::numeric_limits<double>::min();   // +2.2e-308, as in cpp/direct.h:19

// Append-only rectangle store (unit-cube coordinates).  The reference keeps a std::vector<Rectangle>, erases
// divided rectangles and appends their children, so the relative order of live rectangles is their creation
// order -- which is what ids are here.  Rectangles are grouped by their exact centre-to-vertex distance d
// ("classes"); each class keeps its members in a min-heap on y so that the class minimum and its ties are O(log R).
struct Store {
    int N = 0;
    std::vector<double> lb, ub, center, d, y;
    std::vector<int> cls;
    std::vector<char> alive;
    // members: binary min-heap on (y, id).  Only class minima are ever taken out (they are the rectangles that get
    // divided), so a heap -- contiguous, no node allocation -- is all the order structure DIRECT needs.
    struct Class { double d; std::vector<std::pair<double, unsigned> > heap; };
    std::vector<Class> classes;          // only the first `ncls` entries are in use (the rest keep their heap capacity)
    size_t ncls = 0;
    std::unordered_map<unsigned long long, int> cls_of_d;
    std::vector<int> by_d;               // class ids in ascending d (select() walks them in this order)
    size_t live = 0;

    // The store is kept per host thread and reused by successive queries (sequential BO / the gallery issue one DIRECT
    // run per step): clearing keeps the capacity, so only the first query pays for growing ~25 MB of rectangle
    // geometry through fresh pages (that growth was ~40 % of the host driver time at d = 20, 200 iterations).
    void reset(int ndim) {
        N = ndim;
        if (lb.capacity() > ((size_t)1 << 27)) {      // > 1 GiB per array: give the memory back
            std::vector<double>().swap(lb); std::vector<double>().swap(ub); std::vector<double>().swap(center);
        }
        lb.clear(); ub.clear(); center.clear(); d.clear(); y.clear(); cls.clear(); alive.clear();
        for (size_t k = 0; k < ncls; k++) classes[k].heap.clear();
        ncls = 0;
        cls_of_d.clear();
        by_d.clear();
        live = 0;
    }

    static double key(double y) { return y != y ? MAX_DOUBLE : y; }   // NaN sorts last
    static bool heap_gt(const std::pair<double, unsigned>& a, const std::pair<double, unsigned>& b) { return a > b; }
    unsigned add(const double* l, const double* u, const double* c, double dd, double yy) {
        unsigned id = (unsigned)d.size();
        lb.insert(lb.end(), l, l + N); ub.insert(ub.end(), u, u + N); center.insert(center.end(), c, c + N);
        d.push_back(dd); y.push_back(yy); alive.push_back(1);
        unsigned long long bits; std::memcpy(&bits, &dd, 8);
        auto it = cls_of_d.find(bits);
        int k;
        if (it == cls_of_d.end()) {
            k = (int)ncls++;
            if (classes.size() < ncls) classes.push_back(Class());
            classes[k].d = dd; cls_of_d[bits] = k;
            by_d.insert(std::upper_bound(by_d.begin(), by_d.end(), dd, [this](double v, int c) { return v < classes[c].d; }), k);
        }
        else k = it->second;
        cls.push_back(k);
        auto& h = classes[k].heap;
        h.push_back(std::make_pair(key(yy), id));
        std::push_heap(h.begin(), h.end(), heap_gt);
        live++;
        return id;
    }
    // takes every member tying the class minimum out of class k (ascending id not guaranteed)
    void pop_minima(int k, std::vector<unsigned>& out) {
        auto& h = classes[k].heap;
        const double kmin = h.front().first;
        while (!h.empty() && h.front().first == kmin) {
            out.push_back(h.front().second);
            std::pop_heap(h.begin(), h.end(), heap_gt);
            h.pop_back();
        }
    }
    void retire(unsigned id) { alive[id] = 0; live--; }     // the id was taken out of its heap by pop_minima
};

struct Driver {
    ibo_batch_objective_t f; void* user;
    int N;
    std::vector<double> lowerb, upperb;
    std::vector<char> fixed;
    double FMIN = MAX_DOUBLE;
    std::vector<double> XMIN;
    long nsamples = 0;
    bool timed_out = false;     // maxtime ran out in the middle of an iteration (rectangle-by-rectangle mode)
    bool failed = false;        // the objective reported a failed evaluation (NaN): the run stops, nothing else is evaluated
    std::vector<double> xbuf;   // batch staging (box coordinates)

    // unit cube -> box (cpp/direct.cpp:113-120)
    void to_box(const double* x, double* out) const {
        for (int i = 0; i < N; i++) out[i] = fixed[i] ? lowerb[i] : x[i] * (upperb[i] - lowerb[i]) + lowerb[i];
    }
    // bookkeeping half of samplef (cpp/direct.cpp:122-129): strict <, first sample in call order wins
    void account(const double* x, double y) {
        nsamples += 1;
        if (y < FMIN) {
            FMIN = y;
            XMIN.resize(N);
            for (int i = 0; i < N; i++) XMIN[i] = lowerb[i] + (upperb[i] - lowerb[i]) * x[i];
        }
    }
    void eval(const std::vector<double>& unit_pts, long n, std::vector<double>& y) {
        xbuf.resize((size_t)n * N);
        y.resize(n);
        for (long p = 0; p < n; p++) to_box(&unit_pts[(size_t)p * N], &xbuf[(size_t)p * N]);
        // NaN is how a batch objective says "this evaluation failed" (a CUDA error, a failed peer rank, a Python exception in the
        // callback): DIRECT on NaN values is meaningless, so the first one ends the run with IBO_E_OBJECTIVE instead of iterating
        // on garbage until maxiter.  Under IBO_FLAG_SHARD every rank sees the same values, hence stops at the same batch.
        if (failed) { for (long p = 0; p < n; p++) y[p] = 0.0; return; }
        if (n > 0) f(user, n, N, xbuf.data(), y.data());
        for (long p = 0; p < n; p++)
            if (y[p] != y[p]) { failed = true; break; }
        if (failed) for (long p = 0; p < n; p++) y[p] = 0.0;
    }
};

// centre and centre-to-vertex distance exactly as Rectangle::Rectangle (cpp/direct.cpp:54-61)
inline double center_and_d(const double* lb, const double* ub, double* c, int N) {
    double d = 0.0;
    for (int i = 0; i < N; i++) {
        c[i] = lb[i] + (ub[i] - lb[i]) / 2.;
        d += std::pow((lb[i] - c[i]), 2);
    }
    return std::sqrt(d);
}

struct Pending {           // one rectangle being divided
    unsigned src;          // id in the store
    int ndims = 0;         // number of longest, non-fixed sides
    long dim0 = 0;         // offset of its dims in the flat dims array
    long probe0 = 0;       // offset of its 2*k probe values in the phase-A batch
    long child0 = 0;       // offset of its 2*k children in the flat child arrays
    long spec0 = -1;       // first entry of its (long side, variant) table in Scratch::specMap (-1: children wait for phase B)
    int nu = 0;            // number of unclean long sides (<= 2 when spec0 >= 0), see divide()
    int udim[2] = {0, 0};
    double old_d = 0;      // d of the shrunk middle rectangle
};

// Scratch reused across iterations (no per-rectangle allocations in the hot loop).
struct Scratch {
    std::vector<Pending> P;
    std::vector<unsigned> dims;
    std::vector<ind_val> I;
    std::vector<double> pts, ptsB, yA, yB;       // probe points / child centres (unit cube) and their values
    std::vector<double> spec, ptsB2, yB2;        // speculative child centres (phase A) / children left for phase B
    std::vector<long> lateIdx;                   // child index of every point of the phase-B batch
    std::vector<long> specMap;                   // (rectangle, long side, variant) -> first of its two points in `spec`, or -1
    std::vector<int> posOfDim;                   // dim -> position among the rectangle's long dims
    std::vector<double> clb, cub, cd;            // children, in the reference's return order
    std::vector<double> mid_lb, mid_ub;          // shrunk middle rectangles, one per Pending
};

// phase timers of the host driver (printed by run_direct when IBO_DIRECT_TIMING is set)
struct PhaseTimes { double select = 0, probes = 0, children = 0, replay = 0, sel_build = 0; long scans = 0, scan_steps = 0; };
static thread_local PhaseTimes g_pt;
static inline double now_s() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

// Divides the given rectangles (already in processing order): appends the new rectangles in the reference's
// order and retires the sources.  seq: one rectangle per batch pair (the reference's exact call order).
void divide(Driver& D, Store& R, const std::vector<unsigned>& order, bool seq, bool speculate, Scratch& W,
            time_t start = 0, int maxtime = -1) {
    const int N = D.N;
    size_t g0 = 0;
    while (g0 < order.size()) {
        size_t g1 = seq ? g0 + 1 : order.size();
        const size_t np_rect = g1 - g0;
        W.P.assign(np_rect, Pending());
        W.dims.clear(); W.pts.clear();
        // ---- phase A: probe points at lb + w/3, lb + 2w/3 along every longest side (cpp/direct.cpp:156-192)
        double tA = now_s();
        long np = 0;
        for (size_t t = g0; t < g1; t++) {
            Pending& p = W.P[t - g0];
            p.src = order[t];
            const double* lb = &R.lb[(size_t)p.src * N];
            const double* ub = &R.ub[(size_t)p.src * N];
            const double* c = &R.center[(size_t)p.src * N];
            double maxlength = ub[0] - lb[0];          // dim 0 even if fixed (reference quirk, SURVEY 3.3)
            for (int i = 1; i < N; i++)
                if (!D.fixed[i] && ub[i] - lb[i] > maxlength) maxlength = ub[i] - lb[i];
            p.probe0 = np;
            p.dim0 = (long)W.dims.size();
            for (int i = 0; i < N; i++) {
                if (!D.fixed[i] && ub[i] - lb[i] == maxlength) {
                    W.dims.push_back((unsigned)i);
                    size_t o = W.pts.size();
                    W.pts.insert(W.pts.end(), c, c + N);
                    W.pts.insert(W.pts.end(), c, c + N);
                    W.pts[o + i] = lb[i] + maxlength / 3.;
                    W.pts[o + N + i] = lb[i] + 2. * maxlength / 3.;
                    np += 2;
                    p.ndims++;
                }
            }
        }
        // ---- child centres ride in the same batch.  A child of side A is centred at lb + (ub - lb)/2 of ITS bounds
        // (cpp/direct.cpp:54-58): along A that is the centre of the outer third, along every other long side B it is the
        // centre of B's full extent if B is split after A and of B's middle third if B was split before A (:201-232) --
        // and the order is only known once the probe values are back.  The two expressions agree bit for bit for almost
        // every DIRECT interval that does not start at 0 (a few per ten thousand differ); intervals touching the lower
        // face of the box (lb = 0: full relative precision) often differ in the last place.  Sides where they differ are
        // the rectangle's "unclean" sides U.
        //   U empty            -> the 2k child centres are order independent and are evaluated now;
        //   |U| <= 2, spec     -> every child is evaluated now for each subset of U \ {A} that may precede A (<= 4
        //                         variants; the values of the variants that did not occur are discarded);
        //   otherwise          -> the children wait for phase B as before.
        // `spec` (IBO_FLAG_DIRECT_SPECULATE) is for pure objectives only: the callback sees points the reference never
        // samples.  The samples that count, their values and the replay order are the reference's in every case; an
        // iteration costs one GPU batch instead of two.
        long nspec = 0;
        W.spec.clear(); W.specMap.clear();
        if (!seq) {
            static thread_local std::vector<double> cu, cs;
            cu.resize(N); cs.resize(N);
            for (size_t t = 0; t < np_rect; t++) {
                Pending& p = W.P[t];
                const double* lb = &R.lb[(size_t)p.src * N];
                const double* ub = &R.ub[(size_t)p.src * N];
                for (int i = 0; i < N; i++) cu[i] = lb[i] + (ub[i] - lb[i]) / 2.;
                int nu = 0;
                for (int a = 0; a < p.ndims; a++) {
                    const unsigned i = W.dims[p.dim0 + a];
                    const double w = ub[i] - lb[i];
                    const double s1 = lb[i] + w / 3., s2 = lb[i] + 2. * w / 3.;
                    cs[i] = s1 + (s2 - s1) / 2.;
                    if (cu[i] != cs[i]) { if (nu < 2) p.udim[nu] = (int)i; nu++; }
                }
                if (nu > (speculate ? 2 : 0)) continue;
                p.nu = nu;
                p.spec0 = (long)W.specMap.size();
                const int nvar = 1 << nu;
                for (int a = 0; a < p.ndims; a++) {
                    const unsigned i = W.dims[p.dim0 + a];
                    const double w = ub[i] - lb[i];
                    const double s1 = lb[i] + w / 3., s2 = lb[i] + 2. * w / 3.;
                    for (int mask = 0; mask < nvar; mask++) {
                        // bit j of mask: unclean side udim[j] was split before this one (its own bit is never set)
                        bool own = false;
                        for (int j2 = 0; j2 < nu; j2++) own = own || (((mask >> j2) & 1) && p.udim[j2] == (int)i);
                        if (own) { W.specMap.push_back(-1); continue; }
                        W.specMap.push_back(nspec);
                        const size_t o = W.spec.size();
                        W.spec.resize(o + 2 * (size_t)N);
                        double* c1 = &W.spec[o];
                        double* c3 = c1 + N;
                        std::memcpy(c1, cu.data(), sizeof(double) * N);
                        for (int j2 = 0; j2 < nu; j2++) if ((mask >> j2) & 1) c1[p.udim[j2]] = cs[p.udim[j2]];
                        std::memcpy(c3, c1, sizeof(double) * N);
                        c1[i] = lb[i] + (s1 - lb[i]) / 2.;
                        c3[i] = s2 + (ub[i] - s2) / 2.;
                        nspec += 2;
                    }
                }
            }
            W.pts.insert(W.pts.end(), W.spec.begin(), W.spec.end());
        }
        g_pt.probes += now_s() - tA;
        D.eval(W.pts, np + nspec, W.yA);
        double tB = now_s();
        // ---- sort the dims by min(sf1, sf2) and build the children (cpp/direct.cpp:181-232)
        const size_t nchild = (size_t)np;            // two children per probed side
        W.clb.resize(nchild * N); W.cub.resize(nchild * N); W.ptsB.resize(nchild * N); W.cd.resize(nchild);
        W.mid_lb.resize(np_rect * N); W.mid_ub.resize(np_rect * N);
        long nc = 0;
        W.yB.resize(nchild);
        W.lateIdx.clear();
        W.posOfDim.resize(N);
        for (size_t t = 0; t < np_rect; t++) {
            Pending& p = W.P[t];
            W.I.clear();
            for (int a = 0; a < p.ndims; a++) W.posOfDim[W.dims[p.dim0 + a]] = a;
            for (int a = 0; a < p.ndims; a++) {
                double sf1 = W.yA[p.probe0 + 2 * a], sf2 = W.yA[p.probe0 + 2 * a + 1];
                unsigned dim = W.dims[p.dim0 + a];
                if (sf1 < sf2) W.I.push_back(ind_val(dim, sf1));
                else W.I.push_back(ind_val(dim, sf2));
            }
            std::sort(W.I.begin(), W.I.end(), sort_by_val);
            double* olb = &W.mid_lb[t * N];
            double* oub = &W.mid_ub[t * N];
            std::memcpy(olb, &R.lb[(size_t)p.src * N], sizeof(double) * N);
            std::memcpy(oub, &R.ub[(size_t)p.src * N], sizeof(double) * N);
            p.child0 = nc;
            int doneMask = 0;      // unclean sides already split
            for (size_t a = 0; a < W.I.size(); a++) {
                unsigned dd = W.I[a].first;
                double dwidth = oub[dd] - olb[dd];
                double split1 = olb[dd] + dwidth / 3.;
                double split2 = olb[dd] + 2. * dwidth / 3.;
                double* lb1 = &W.clb[(size_t)nc * N];       double* ub1 = &W.cub[(size_t)nc * N];
                double* lb3 = &W.clb[(size_t)(nc + 1) * N]; double* ub3 = &W.cub[(size_t)(nc + 1) * N];
                std::memcpy(lb1, olb, sizeof(double) * N); std::memcpy(ub1, oub, sizeof(double) * N);
                std::memcpy(lb3, olb, sizeof(double) * N); std::memcpy(ub3, oub, sizeof(double) * N);
                ub1[dd] = split1;
                lb3[dd] = split2;
                W.cd[nc] = center_and_d(lb1, ub1, &W.ptsB[(size_t)nc * N], N);
                olb[dd] = split1;
                oub[dd] = split2;
                W.cd[nc + 1] = center_and_d(lb3, ub3, &W.ptsB[(size_t)(nc + 1) * N], N);
                // value from the phase-A batch when the child's centre is bit for bit one of those evaluated there
                long sp = -1;
                if (p.spec0 >= 0) sp = W.specMap[(size_t)p.spec0 + ((size_t)W.posOfDim[dd] << p.nu) + doneMask];
                for (int c2 = 0; c2 < 2; c2++) {
                    if (sp >= 0 && !std::memcmp(&W.ptsB[(size_t)(nc + c2) * N], &W.spec[(size_t)(sp + c2) * N], sizeof(double) * N))
                        W.yB[nc + c2] = W.yA[np + sp + c2];
                    else W.lateIdx.push_back(nc + c2);
                }
                for (int j2 = 0; j2 < p.nu; j2++) if (p.udim[j2] == (int)dd) doneMask |= 1 << j2;
                nc += 2;
            }
            // the middle third keeps the old centre and y; d is recomputed from the shrunk bounds (:226-231)
            double d = 0.0;
            const double* ocp = &R.center[(size_t)p.src * N];
            for (int i = 0; i < N; i++) d += std::pow((olb[i] - ocp[i]), 2);
            p.old_d = std::sqrt(d);
        }
        g_pt.children += now_s() - tB;
        if ((long)W.lateIdx.size() == nc) D.eval(W.ptsB, nc, W.yB);
        else if (!W.lateIdx.empty()) {
            const size_t nl = W.lateIdx.size();
            W.ptsB2.resize(nl * N);
            for (size_t q = 0; q < nl; q++) std::memcpy(&W.ptsB2[q * N], &W.ptsB[(size_t)W.lateIdx[q] * N], sizeof(double) * N);
            D.eval(W.ptsB2, (long)nl, W.yB2);
            for (size_t q = 0; q < nl; q++) W.yB[W.lateIdx[q]] = W.yB2[q];
        }
        double tC = now_s();
        // ---- replay the reference's call order for FMIN / nsamples, then append the rectangles
        std::vector<double> oc(N);
        for (size_t t = 0; t < np_rect; t++) {
            Pending& p = W.P[t];
            const long k2 = 2L * p.ndims;
            for (long a = 0; a < k2; a++) D.account(&W.pts[(size_t)(p.probe0 + a) * N], W.yA[p.probe0 + a]);
            for (long a = 0; a < k2; a++) D.account(&W.ptsB[(size_t)(p.child0 + a) * N], W.yB[p.child0 + a]);
            for (long a = 0; a < k2; a++) {
                const size_t o = (size_t)(p.child0 + a);
                R.add(&W.clb[o * N], &W.cub[o * N], &W.ptsB[o * N], W.cd[o], W.yB[o]);
            }
            // middle rectangle (copy of the source with shrunk bounds)
            std::memcpy(oc.data(), &R.center[(size_t)p.src * N], sizeof(double) * N);
            double oy = R.y[p.src];
            R.retire(p.src);
            R.add(&W.mid_lb[t * N], &W.mid_ub[t * N], oc.data(), p.old_d, oy);
        }
        g_pt.replay += now_s() - tC;
        g0 = g1;
        // rectangle-by-rectangle mode (a scalar callback, possibly slow): the wall-clock budget is checked after every rectangle,
        // as the reference does (cpp/direct.cpp:493-497); the batched modes check once per iteration
        if (seq && maxtime >= 0 && time(NULL) - start > maxtime) { D.timed_out = true; break; }
    }
}

// potentially-optimal rectangles, ascending creation order (cpp/direct.cpp:378-456).
// The reference's pair scan decides rectangle j from (d_j, y_j) and the multiset of the others only through
//   I3: reject if some rectangle of the same size has a smaller y      -> y_j must equal its class minimum
//   I1/I2: extremal slopes towards smaller / larger classes            -> attained at those classes' minima
//          (fl(x - c) and fl(x / c), c > 0, are monotone in x, so the extremal slope is the slope of the minimum)
// so the decision is a function of the class alone and is evaluated once per class: O(C^2 + #selected log R),
// with accept / reject decisions bit-identical to the O(R^2) scan.
void select(Store& R, double FMIN, std::vector<unsigned>& potopts) {
    const double epsilon = 10e-10;
    potopts.clear();
    // live classes in ascending d (distinct by construction; the store keeps the order up to date as classes appear, a few
    // per iteration, so nothing is sorted here): sd / sy / sk are what the slope scans stream through
    static thread_local std::vector<double> sd, sy;
    static thread_local std::vector<int> sk;
    static thread_local std::vector<char> dominated;
    sd.clear(); sy.clear(); sk.clear();
    const double tb0 = now_s();
    for (int k : R.by_d) {
        if (R.classes[k].heap.empty()) continue;
        unsigned id = R.classes[k].heap.front().second;
        sd.push_back(R.classes[k].d); sy.push_back(R.y[id]); sk.push_back(k);
    }
    const size_t C = sd.size();
    g_pt.sel_build += now_s() - tb0;
    // Quick reject (exactly the reference's `minI2 <= 0` break): a larger class whose minimum is <= y_j makes the
    // slope (y_c - y_j)/(d_c - d_j) non-positive.  With classes sorted by d, that is a suffix-minimum lookup, so
    // only the few classes on the lower-right staircase pay for a slope scan.
    dominated.assign(C, 0);
    {
        double sufmin = MAX_DOUBLE; bool have = false;
        for (size_t t = C; t-- > 0;) {
            if (have && sufmin - sy[t] <= 0.) dominated[t] = 1;      // sign of fl(y_c - y_j) is exact
            if (!have || sy[t] < sufmin) { sufmin = sy[t]; have = true; }
        }
    }
    // Only the classes that survive (the lower-right "staircase": strictly below every larger class) can attain the extremal
    // slopes of a surviving class j.  A dominated class c (some larger c' has y_c' <= y_c) is never the argmin of
    // (y_c - y_j)/(d_c - d_j) over the larger classes: num' <= num and den' >= den > 0, and correctly rounded subtraction and
    // division are monotone, so fl(slope_c') <= fl(slope_c).  It is never the argmax of (y_j - y_c)/(d_j - d_c) over the smaller
    // classes either: its dominator is smaller than j (a dominator >= j would dominate j) and gives fl(slope) >= by the same
    // argument.  So the scans stream through the compacted staircase (a sixth of the classes at d = 20) with bit-identical
    // maxI1 / minI2.
    {
        size_t w = 0;
        for (size_t t = 0; t < C; t++)
            if (!dominated[t]) { sd[w] = sd[t]; sy[w] = sy[t]; sk[w] = sk[t]; ++w; }
        sd.resize(w); sy.resize(w); sk.resize(w);
    }
    const size_t S = sd.size();
    for (size_t t = 0; t < S; t++) {
        const double dj = sd[t], yj = sy[t];
        double maxI1 = MIN_DOUBLE, minI2 = MAX_DOUBLE;
        bool breaked = false;
        // maxI1 = max over smaller classes of (yj - yc)/(dj - dc), minI2 = min over larger classes of (yc - yj)/(dc - dj):
        // max / min do not depend on the visiting order, so the scan walks outwards from the class's own position, where
        // the steepest slopes usually are, and stops at the first moment the reference's final test `minI2 < maxI1` is
        // already decided (maxI1 only grows, minI2 only shrinks) -- same accept / reject, a fraction of the divisions.
        // (`minI2 <= 0` cannot occur here: that is the `dominated` case above.)
        size_t l = t, r = t + 1;
        long steps = 0;
        while ((l > 0 || r < S) && !breaked) {
            ++steps;
            if (l > 0) {
                --l;
                double val = (yj - sy[l]) / (dj - sd[l]);
                if (val > maxI1) maxI1 = val;
            }
            if (r < S) {
                double val = (sy[r] - yj) / (sd[r] - dj);
                if (val < minI2) minI2 = val;
                ++r;
            }
            if (maxI1 != MIN_DOUBLE && minI2 != MAX_DOUBLE && minI2 < maxI1) breaked = true;
        }
        g_pt.scans++; g_pt.scan_steps += steps;
        if (breaked) continue;
        bool ok = false;
        if (minI2 == MAX_DOUBLE) ok = true;
        else if (FMIN == 0.0) ok = (yj <= dj * minI2);
        else ok = (epsilon <= (FMIN - yj) / std::abs(FMIN) + (dj / std::abs(FMIN)) * minI2);
        if (!ok) continue;
        // every member tying the class minimum is potentially optimal; they leave the heap here and are divided
        // (or the run ends) before the next selection
        R.pop_minima(sk[t], potopts);
    }
    std::sort(potopts.begin(), potopts.end());
}

int run_direct(ibo_batch_objective_t f, void* user, int ndim, const double* lb, const double* ub, int maxiter, int maxtime,
               int maxsample, int flags, double* fmin, double* xmin, long* nsamples, int* iterations) {
    if (!f || ndim < 1 || !lb || !ub) { set_error("bad argument"); return IBO_E_BADARG; }
    const bool seq = (flags & IBO_FLAG_DIRECT_SEQ) != 0;
    const bool speculate = !seq && (flags & IBO_FLAG_DIRECT_SPECULATE) != 0;
    time_t start = time(NULL);
    Driver D;
    D.f = f; D.user = user; D.N = ndim;
    D.lowerb.assign(lb, lb + ndim); D.upperb.assign(ub, ub + ndim);
    D.fixed.resize(ndim);
    for (int i = 0; i < ndim; i++) D.fixed[i] = (lb[i] == ub[i]);
    // The per-thread store is reused by successive queries; a nested query (an objective callback that itself runs
    // DIRECT on this thread) gets a private one.
    static thread_local Store tlsR;
    static thread_local Scratch tlsW;
    static thread_local bool tlsBusy = false;
    const bool nested = tlsBusy;
    std::unique_ptr<Store> ownR(nested ? new Store() : nullptr);
    std::unique_ptr<Scratch> ownW(nested ? new Scratch() : nullptr);
    Store& R = nested ? *ownR : tlsR;
    Scratch& W = nested ? *ownW : tlsW;
    struct BusyGuard { bool& b; bool set; ~BusyGuard() { if (set) b = false; } } guard{tlsBusy, !nested};
    if (!nested) tlsBusy = true;
    R.reset(ndim);
    // first rectangle: the unit cube, sampled at its centre (cpp/direct.cpp:349-357)
    {
        std::vector<double> l(ndim, 0.0), u(ndim, 1.0), c(ndim);
        double d = center_and_d(l.data(), u.data(), c.data(), ndim);
        std::vector<double> y;
        D.eval(c, 1, y);
        D.account(c.data(), y[0]);
        R.add(l.data(), u.data(), c.data(), d, y[0]);
    }
    std::vector<unsigned> potopts, order;
    order.clear();
    R.pop_minima(R.cls[0], order);      // the unit cube leaves its heap like any rectangle about to be divided
    divide(D, R, order, seq, speculate, W);
    int iteration = 0;
    bool done = false;
    while (iteration < maxiter && !done) {
        iteration++;
        double tS = now_s();
        select(R, D.FMIN, potopts);
        g_pt.select += now_s() - tS;
        if (potopts.empty()) break;    // "could not divide any more" (cpp/direct.cpp:473-477)
        // division order: highest index first; stop after the rectangle that pushes nsamples past
        // maxsample (cpp/direct.cpp:479-492).  Each rectangle costs 4 samples per longest side, which is
        // known before evaluating, so the cut is taken up front.
        order.clear();
        long ns = D.nsamples;
        for (size_t t = potopts.size(); t-- > 0;) {
            unsigned j = potopts[t];
            const double* l = &R.lb[(size_t)j * ndim];
            const double* u = &R.ub[(size_t)j * ndim];
            double maxlength = u[0] - l[0];
            for (int i = 1; i < ndim; i++)
                if (!D.fixed[i] && u[i] - l[i] > maxlength) maxlength = u[i] - l[i];
            int k = 0;
            for (int i = 0; i < ndim; i++)
                if (!D.fixed[i] && u[i] - l[i] == maxlength) k++;
            order.push_back(j);
            ns += 4L * k;
            if (ns > (long)(unsigned)maxsample) { done = true; break; }
        }
        divide(D, R, order, seq, speculate, W, start, maxtime);
        if (D.failed || D.timed_out) break;
        if (time(NULL) - start > maxtime) break;
        if (D.nsamples > (long)(unsigned)maxsample) break;
    }
    if (ibo::get_option(ibo::OPT_DIRECT_TIMING))
        fprintf(stderr, "[run_direct] host phases: select %.3f ms, probe build %.3f ms, child build %.3f ms, replay+append %.3f ms; "
                        "%zu rectangles, %zu classes; select: class table %.3f ms, %ld slope scans, %ld scan steps\n", 1e3 * g_pt.select, 1e3 * g_pt.probes, 1e3 * g_pt.children, 1e3 * g_pt.replay,
                R.d.size(), R.ncls, 1e3 * g_pt.sel_build, g_pt.scans, g_pt.scan_steps);
    g_pt = PhaseTimes();
    if (D.failed) { set_error("DIRECT: the objective reported a failed evaluation (NaN)"); return IBO_E_OBJECTIVE; }
    if (fmin) *fmin = D.FMIN;
    if (xmin) for (int i = 0; i < ndim; i++) xmin[i] = D.XMIN.empty() ? lb[i] : D.XMIN[i];
    if (nsamples) *nsamples = D.nsamples;
    if (iterations) *iterations = iteration;
    return IBO_OK;
}

struct ScalarAdapter { objective_t f; };
void scalar_batch(void* user, long n, int ndim, const double* X, double* y) {
    ScalarAdapter* a = static_cast<ScalarAdapter*>(user);
    std::vector<double> x(ndim);
    for (long p = 0; p < n; p++) {
        std::memcpy(x.data(), X + (size_t)p * ndim, sizeof(double) * ndim);
        y[p] = a->f(ndim, x.data());
    }
}

struct GpuObjective {
    ibo_model* m; int acq; double ymax, parm; int flags; int rc; double t_eval; long batches, points;
    long shard_min = 0; long sharded_batches = 0; std::vector<double> mine, all;
    bool server = false;      // a model of one row-block: batches go to the resident kernel of tiny.cu
};
void gpu_batch(void* user, long n, int ndim, const double* X, double* y) {
    GpuObjective* g = static_cast<GpuObjective*>(user);
    const double nan = std::numeric_limits<double>::quiet_NaN();
    // (the driver stops calling after the first NaN; under IBO_FLAG_SHARD all ranks are then in the same state)
    if (g->rc != IBO_OK) { for (long i = 0; i < n; i++) y[i] = nan; return; }
    auto t0 = std::chrono::steady_clock::now();
    const int world = (g->flags & IBO_FLAG_SHARD) ? ibo_comm_size() : 1;
    if (world > 1 && n >= g->shard_min) {
        // Every rank runs the same deterministic driver on the same model; a batch is cut into `world` contiguous slices
        // of `per` points, rank r evaluates slice r, and the values are all-gathered (NCCL over NVLink).  A candidate's
        // value does not depend on the batch it is evaluated in (DESIGN.md "Determinism"), so the trajectory is the
        // single-GPU one bit for bit.  Slot `per` of every rank's block carries its status: a local failure reaches
        // every rank in the same collective, and all of them end the query (nobody is left waiting in the next all-gather).
        const long per = (n + world - 1) / world;
        const int rank = ibo_comm_rank();
        const long lo = std::min((long)rank * per, n), hi = std::min(lo + per, n);
        g->mine.assign((size_t)per + 1, 0.0);
        g->all.resize((size_t)(per + 1) * world);
        int rcLocal = IBO_OK;
        // INT8 or FP64 kernels: decided from the size of the whole batch, exactly as the unsharded query decides it, so that every
        // candidate gets the same bits on whatever rank and in whatever slice it is evaluated
        const bool i8 = batch_uses_i8(g->m, n, g->flags) != 0;
        const int sliceFlags = i8 ? g->flags : g->flags | IBO_FLAG_FP64;
        const ScoreForce force = i8 ? ScoreForce::I8 : ScoreForce::None;
        if (hi > lo) rcLocal = eval_neg_acq(g->m, X + (size_t)lo * ndim, hi - lo, g->acq, g->ymax, g->parm, sliceFlags, force, g->mine.data());
        g->mine[(size_t)per] = rcLocal == IBO_OK ? 0.0 : 1.0;
        int rc2 = ibo_comm_allgather(g->mine.data(), per + 1, g->all.data());
        g->rc = rcLocal != IBO_OK ? rcLocal : rc2;
        if (g->rc == IBO_OK) {
            for (int r = 0; r < world; r++)
                if (g->all[(size_t)r * (per + 1) + per] != 0.0) { g->rc = IBO_E_COMM; set_error("sharded DIRECT: rank " + std::to_string(r) + " failed to evaluate its slice"); break; }
        }
        if (g->rc == IBO_OK)
            for (int r = 0; r < world; r++) {
                const long a = std::min((long)r * per, n), b = std::min(a + per, n);
                if (b > a) std::memcpy(y + a, g->all.data() + (size_t)r * (per + 1), sizeof(double) * (size_t)(b - a));
            }
        g->sharded_batches++;
    } else if (g->server && tiny_server_fits(g->m, n)) {
        g->rc = tiny_server_eval(g->m, X, n, g->acq, g->ymax, g->parm, g->flags, y);
    } else {
        if (g->server) tiny_server_stop(g->m);      // the resident kernel owns the model's stream: it leaves before anything else is launched
        g->rc = eval_neg_acq(g->m, X, n, g->acq, g->ymax, g->parm, g->flags, ScoreForce::None, y);
    }
    g->t_eval += std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    g->batches++; g->points += n;
    if (g->rc != IBO_OK) for (long i = 0; i < n; i++) y[i] = nan;
}

}  // namespace
}  // namespace ibo

using namespace ibo;

extern "C" int ibo_direct_batched(ibo_batch_objective_t f, void* user, int ndim, const double* lb, const double* ub, int maxiter,
                                  int maxtime, int maxsample, int flags, double* fmin, double* xmin, long* nsamples, int* iterations) {
    return run_direct(f, user, ndim, lb, ub, maxiter, maxtime, maxsample, flags, fmin, xmin, nsamples, iterations);
}

extern "C" int ibo_acqmax(ibo_model* m, const double* lb, const double* ub, int acq, double ymax, double parm, int flags,
                          int maxiter, int maxtime, int maxsample, double* opt, double* optx, long* nsamples, int* iterations) {
    if (!m || acq < 0 || acq > 2) { set_error("bad argument"); return IBO_E_BADARG; }
    GpuObjective g{m, acq, ymax, parm, flags, IBO_OK, 0.0, 0, 0};
    if (flags & IBO_FLAG_SHARD) {
        const long sm = ibo::get_option(ibo::OPT_SHARD_MIN);       // batches below this many points stay on every rank (latency)
        g.shard_min = sm > 0 ? sm : 64L * ibo_comm_size();
    }
    g.server = !(flags & IBO_FLAG_SHARD);
    double fmin = 0;
    auto t0 = std::chrono::steady_clock::now();
    // the GPU objective is a pure function of the point (DESIGN.md "Determinism"): the driver may speculate
    int rc = run_direct(gpu_batch, &g, ibo_model_dim(m), lb, ub, maxiter, maxtime, maxsample, flags | IBO_FLAG_DIRECT_SPECULATE, &fmin, optx, nsamples, iterations);
    tiny_server_stop(m);
    if (ibo::get_option(ibo::OPT_DIRECT_TIMING)) {
        double tt = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
        fprintf(stderr, "[ibo_acqmax] total %.3f ms, GPU batches %.3f ms (%ld batches, %ld sharded, %ld points, %.1f us/batch), host driver %.3f ms\n",
                1e3 * tt, 1e3 * g.t_eval, g.batches, g.sharded_batches, g.points, g.batches ? 1e6 * g.t_eval / g.batches : 0.0, 1e3 * (tt - g.t_eval));
    }
    if (rc) return rc;
    if (g.rc) return g.rc;
    if (opt) *opt = -fmin;
    return IBO_OK;
}

// ---- legacy symbols ---------------------------------------------------------------------------
// Independent queries side by side: one host thread per query, each driving its own model handle (own stream, own device
// workspace; the rectangle store of the driver is per thread).  Queries on different devices use the GPUs of a box for
// throughput -- a single DIRECT query is a chain of ~200 dependent small batches and does not get faster with more GPUs --;
// queries on the same device overlap each other's launch and round-trip latencies.
extern "C" int ibo_acqmax_many(int nq, ibo_model* const* models, const double* lb, const double* ub, int acq, const double* ymax,
                               const double* parm, int flags, int maxiter, int maxtime, int maxsample,
                               double* opt, double* optx, long* nsamples, int* iterations, int* status) {
    if (nq < 1 || !models || !lb || !ub || !ymax || !parm || !opt || !optx) { set_error("bad argument"); return IBO_E_BADARG; }
    const int ndim = ibo_model_dim(models[0]);
    for (int q = 0; q < nq; q++) {
        if (!models[q] || ibo_model_dim(models[q]) != ndim) { set_error("ibo_acqmax_many: models must share the dimension"); return IBO_E_BADARG; }
        for (int p = 0; p < q; p++)
            if (models[p] == models[q]) { set_error("ibo_acqmax_many: every query needs its own model handle"); return IBO_E_BADARG; }
    }
    if (flags & IBO_FLAG_SHARD) { set_error("ibo_acqmax_many: queries are independent, IBO_FLAG_SHARD does not apply"); return IBO_E_BADARG; }
    std::vector<int> rc(nq, IBO_OK);
    std::vector<std::string> err(nq);
    std::vector<std::thread> th;
    for (int q = 0; q < nq; q++)
        th.emplace_back([&, q]() {
            long ns = 0; int it = 0;
            rc[q] = ibo_acqmax(models[q], lb, ub, acq, ymax[q], parm[q], flags, maxiter, maxtime, maxsample, &opt[q], optx + (size_t)q * ndim, &ns, &it);
            if (rc[q]) err[q] = ibo_last_error();
            if (nsamples) nsamples[q] = ns;
            if (iterations) iterations[q] = it;
        });
    for (auto& t : th) t.join();
    int first = IBO_OK;
    for (int q = 0; q < nq; q++) {
        if (status) status[q] = rc[q];
        if (rc[q] && !first) { first = rc[q]; set_error("query " + std::to_string(q) + ": " + err[q]); }
    }
    return first;
}

extern "C" const double* direct(objective_t objective, int ndim, double* lb, double* ub, int maxiter, int maxtime, int maxsample) {
    if (!objective || ndim < 1) return NULL;
    ScalarAdapter a{objective};
    double* res = (double*)malloc(sizeof(double) * (ndim + 1));   // caller frees (cpp/direct.cpp:564-569)
    if (!res) return NULL;
    int rc = run_direct(scalar_batch, &a, ndim, lb, ub, maxiter, maxtime, maxsample, IBO_FLAG_DIRECT_SEQ, &res[0], &res[1], NULL, NULL);
    if (rc) { free(res); return NULL; }
    return res;
}

extern "C" const double* acqmaxGP(int ndim, double* lb, double* ub, double* invR, double* X, double* Y, int nx, int acqfunc,
                                  int kerneltype, double* hyperparams, int npbases, double* pbasismeans, double* pbasisbeta,
                                  double pbasistheta, double* pbasislowerb, double* pbasiswidth, double parm, double noise,
                                  int maxiter, int maxtime, int maxsample) {
    if (acqfunc < 0 || acqfunc > 2) {                     // cpp/optimizeGP.cpp:342-346
        set_error("[C++] unknown acquisition function");
        return NULL;
    }
    if (kerneltype < 0 || kerneltype > 3 || nx < 1 || ndim < 1) return NULL;
    // hyper-parameter layout as GP_Maximizer::posterior reads it (cpp/optimizeGP.cpp:70-112);
    // sf2 = 1 for kernels 0-2 (:303-310); for Matern-5/2 the reference takes exp(2 log(hyperparams[ndim])) (:313) -- the
    // magnitude slot of the kernel's [theta, magnitude] array only when ndim == 1.  The drop-in reads the same element: a caller
    // with ndim > 1 gets defined behaviour from the reference only by passing ndim + 1 values with the magnitude last, and gets
    // the same answer here (tests/golden: matern5_2d / 4d / 10d).
    double sf2 = 1.0;
    int nh = (kerneltype == 0) ? ndim : 1;
    if (kerneltype == 3) sf2 = std::exp(2.0 * std::log(hyperparams[ndim]));
    ibo_model* m = NULL;
    int info = 0;
    int rc = ibo_model_create_from_inverse(0, kerneltype, hyperparams, nh, X, Y, nx, ndim, noise, invR, sf2, npbases, pbasismeans,
                                           pbasisbeta, pbasistheta, pbasislowerb, pbasiswidth, &m, &info);
    if (rc) return NULL;
    double maxY = Y[0];
    for (int i = 0; i < nx; i++) if (Y[i] > maxY) maxY = Y[i];      // cpp/optimizeGP.cpp:317-322
    double* res = (double*)malloc(sizeof(double) * (ndim + 1));
    double opt = 0;
    rc = res ? ibo_acqmax(m, lb, ub, acqfunc, maxY, parm, IBO_FLAG_MODE_CPP, maxiter, maxtime, maxsample, &opt, &res[1], NULL, NULL) : IBO_E_NOMEM;
    ibo_model_destroy(m);
    if (rc) { free(res); return NULL; }
    res[0] = -opt;     // the reference returns FMIN of the negated acquisition
    return res;
}
