// ps_api.cu -- the C ABI (include/polystokes_b200.h).  No exception crosses the boundary: every entry
// point catches, stores the message for ps_last_error() and returns PS_FAILED / PS_INVALID, mirroring the
// reference's "return false + addError" convention (exec/HDK_PolyStokes.C:251-314, 597-608).
#include "ps_solver.hpp"
#include <map>
#include <array>
#include <fstream>
#include <limits>
#include <thread>
#include <mutex>
#include <condition_variable>
#include <functional>
#include <memory>
#include <chrono>

using namespace ps;

struct MultiGroup;
// S: the solver (for the handle of ps_create_multi: rank 0's, not owned); tm: the CUDA events of ps_timer
struct ps_solver { Solver* S; void* tm[2] = {nullptr, nullptr}; Scratch scratch; MultiGroup* multi = nullptr; };

// ps_create_multi: one process drives several GPUs.  The handle owns one ordinary single-GPU handle ("rank") per device and one
// persistent host thread per rank; a collective entry point (ps_step, ps_setup, ps_solve, ps_time_kernel, ps_timer) runs on all
// ranks at once -- the ranks talk to each other exactly as separate processes would (NCCL for the plumbing, peer memory for
// the halos / reductions; ps_comm.hpp, ps_peer.hpp) -- and returns when the last rank is done.
struct MultiGroup {
    struct Worker {
        std::thread th; std::mutex m; std::condition_variable cv;
        std::function<int()> task; bool has = false, quit = false, done = true; int rc = 0; std::string err;
        std::vector<void*> graveyard;            // device buffers the rank let go of during a collective call (ps_rt.hpp, g_deferredFree)
        const char* volatile where = "idle";     // breadcrumb of the rank thread (PS_WHERE), read by the watchdog below
    };
    std::vector<ps_solver*> kids;
    std::vector<std::unique_ptr<Worker>> workers;
    void start(int n) {
        for (int k = 0; k < n; ++k) {
            workers.emplace_back(new Worker);
            Worker* w = workers.back().get();
            w->th = std::thread([w] {
                g_deferredFree = &w->graveyard;
                g_where = &w->where;
                for (;;) {
                    std::function<int()> job;
                    { std::unique_lock<std::mutex> lk(w->m); w->cv.wait(lk, [w] { return w->has || w->quit; }); if (w->quit) return; job = w->task; w->has = false; }
                    int rc; std::string err;
                    try { rc = job(); if (rc == PS_FAILED || rc == PS_INVALID) err = g_lastError; }
                    catch (const std::exception& e) { rc = PS_FAILED; err = e.what(); }
                    catch (...) { rc = PS_FAILED; err = "unknown error"; }
                    w->where = "idle";
                    { std::lock_guard<std::mutex> lk(w->m); w->rc = rc; w->err = err; w->done = true; }
                    w->cv.notify_all();
                }
            });
        }
    }
    // every rank is idle (its collective call has returned): the parked frees cannot wait on anybody any more
    void bury() {
#ifndef PS_EMULATE
        for (auto& w : workers) { for (void* p : w->graveyard) cudaFree(p); w->graveyard.clear(); }
#endif
    }
    // f(rank) on every rank's thread; returns rank 0's result, or the first failure (its message goes to the caller's ps_last_error)
    int run(const std::function<int(int)>& f) {
        for (size_t k = 0; k < workers.size(); ++k) {
            Worker* w = workers[k].get();
            { std::lock_guard<std::mutex> lk(w->m); w->task = [f, k] { return f((int)k); }; w->has = true; w->done = false; }
            w->cv.notify_all();
        }
        // A rank that failed never joins the collectives its peers are waiting in: once one rank has returned with an error and
        // another is still busy 5 s later, that rank's communicator is aborted (its kernels give up, the rank fails with a message)
        // and its peer-memory waits run into their own time-out.  PS_MULTI_WATCHDOG_S (default 120): a collective call that long
        // is reported once on stderr with every rank's position.
        static const int watchdog = getenv("PS_MULTI_WATCHDOG_S") ? atoi(getenv("PS_MULTI_WATCHDOG_S")) : 120;
        bool barked = false, aborted = false;
        const auto t0 = std::chrono::steady_clock::now();
        // (called with no worker mutex held: every look at another worker's state takes that worker's mutex)
        auto failedRank = [&]() -> int {
            for (size_t j = 0; j < workers.size(); ++j) { Worker* q = workers[j].get(); std::lock_guard<std::mutex> g2(q->m); if (q->done && (q->rc == PS_FAILED || q->rc == PS_INVALID)) return (int)j; }
            return -1;
        };
        double failSeen = -1.;
        int rc0 = PS_SUCCESS; bool failed = false;
        for (size_t k = 0; k < workers.size(); ++k) {
            Worker* w = workers[k].get();
            std::unique_lock<std::mutex> lk(w->m);
            while (!w->done) {
                w->cv.wait_for(lk, std::chrono::milliseconds(500), [w] { return w->done; });
                if (w->done) break;
                const double el = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
                lk.unlock();
                if (!aborted && failedRank() >= 0) {
                    if (failSeen < 0.) failSeen = el;
                    else if (el - failSeen > 5.) {
                        aborted = true;
                        for (size_t j = 0; j < workers.size(); ++j) {
                            bool busy; { std::lock_guard<std::mutex> g2(workers[j]->m); busy = !workers[j]->done; }
                            if (busy && kids[j]->S && kids[j]->S->comm) kids[j]->S->comm->abort();
                        }
                    }
                }
                if (watchdog > 0 && !barked && el > watchdog) {
                    barked = true;
                    fprintf(stderr, "[polystokes_b200] a collective call on the multi-GPU handle has been running for %d s:", watchdog);
                    for (size_t j = 0; j < workers.size(); ++j) {
                        Worker* q = workers[j].get();
                        std::lock_guard<std::mutex> g2(q->m);
                        if (q->done) fprintf(stderr, " rank %zu done (rc %d%s%s);", j, q->rc, q->err.empty() ? "" : ": ", q->err.c_str());
                        else fprintf(stderr, " rank %zu in %s;", j, q->where);
                    }
                    fprintf(stderr, "\n");
                }
                lk.lock();
            }
            if (k == 0) rc0 = w->rc;
            if ((w->rc == PS_FAILED || w->rc == PS_INVALID) && !failed) { failed = true; rc0 = w->rc; g_lastError = "rank " + std::to_string(k) + ": " + w->err; }
        }
        if (aborted) g_lastError += " (the other ranks' communicators were aborted: destroy the handle)";
        bury();
        return rc0;
    }
    void stop() {
        for (auto& w : workers) { { std::lock_guard<std::mutex> lk(w->m); w->quit = true; } w->cv.notify_all(); if (w->th.joinable()) w->th.join(); }
        bury();
        workers.clear();
    }
};

namespace {

template <class Fn>
int guarded(Fn&& fn) {
    try { return fn(); }
    catch (const std::exception& e) { g_lastError = e.what(); return PS_FAILED; }
    catch (...) { g_lastError = "unknown error"; return PS_FAILED; }
}
// Every entry point that takes a handle runs on the handle's device with the handle's scratch buffers, whatever thread calls it
// (Houdini cooks a DOP on arbitrary worker threads whose current device is 0), and leaves the caller's current device untouched.
struct Enter {
    int prev = -1; Scratch* prevScratch;
    explicit Enter(ps_solver* h) : prevScratch(g_scratch) {
        g_scratch = &h->scratch;
#ifndef PS_EMULATE
        if (h->S) { if (cudaGetDevice(&prev) != cudaSuccess) prev = -1; if (prev != h->S->P.device) PS_CUDA(cudaSetDevice(h->S->P.device)); else prev = -1; }
#endif
    }
    ~Enter() {
        g_scratch = prevScratch;
#ifndef PS_EMULATE
        if (prev >= 0) cudaSetDevice(prev);
#endif
    }
};
template <class Fn>
int guarded(ps_solver* h, Fn&& fn) {
    try { Enter e(h); return fn(); }
    catch (const std::exception& e) { g_lastError = e.what(); return PS_FAILED; }
    catch (...) { g_lastError = "unknown error"; return PS_FAILED; }
}

// host CSR (export / parity only -- never on the solve path)
struct HostCsr { int64_t rows = 0, cols = 0; std::vector<int64_t> ptr; std::vector<int32_t> idx; std::vector<double> val; };

HostCsr diag_csr(const std::vector<double>& d) {
    HostCsr m; m.rows = m.cols = (int64_t)d.size(); m.ptr.resize(d.size() + 1); m.idx.resize(d.size()); m.val = d;
    for (size_t i = 0; i < d.size(); ++i) { m.ptr[i] = (int64_t)i; m.idx[i] = (int32_t)i; }
    m.ptr[d.size()] = (int64_t)d.size();
    return m;
}
HostCsr blockdiag_csr(const std::vector<double>& blocks, int R) {
    HostCsr m; m.rows = m.cols = (int64_t)R * RDOF;
    m.ptr.resize(m.rows + 1); m.idx.resize((size_t)R * RDOF * RDOF); m.val = blocks;
    for (int64_t r = 0; r <= m.rows; ++r) m.ptr[r] = r * RDOF;
    for (int b = 0; b < R; ++b) for (int i = 0; i < RDOF; ++i) for (int j = 0; j < RDOF; ++j) m.idx[((size_t)b * RDOF + i) * RDOF + j] = b * RDOF + j;
    return m;
}

// ---- several ranks: the global objects, assembled on rank 0 from the pieces their owners hold ----
// Every entry is copied from the one rank that owns it, never summed over the ranks: a sum would turn an owner's -0.0 into +0.0,
// and the exported files print the two differently.

// index ranges [lo, hi) of a table that one rank owns, ascending
typedef std::vector<std::pair<int64_t, int64_t>> Spans;
template <int N>
Spans spans_in(const RangeSetN<N>& s, int64_t lo, int64_t hi) {      // the ranges of s inside [lo, hi), relative to lo
    Spans o;
    for (int i = 0; i < s.n; ++i) { const int64_t a = std::max(s.lo[i], lo), b = std::min(s.lo[i] + s.count(i), hi); if (b > a) o.push_back({a - lo, b - lo}); }
    return o;
}
Spans region_spans(const Solver& S, int64_t per, int64_t off = 0) { return {{off + S.RG.regLo * per, off + S.RG.regHi * per}}; }

template <class T> void put(std::vector<uint8_t>& b, const T* p, size_t n) { const size_t o = b.size(); b.resize(o + n * sizeof(T)); if (n) memcpy(b.data() + o, p, n * sizeof(T)); }
template <class T> const uint8_t* take(const uint8_t* q, T* p, size_t n) { if (n) memcpy(p, q, n * sizeof(T)); return q + n * sizeof(T); }

// Collective: rank 0 receives every rank's bytes in rank order, the other ranks an empty list.  The sizes travel in one all-reduce
// (Solver::hostAllgather), the payload in one grouped send / receive towards rank 0 through a staging buffer of the solver's device.
std::vector<std::vector<uint8_t>> gather_bytes(Solver& S, const std::vector<uint8_t>& mine) {
    PS_WHERE("export / view: gather");
    const int N = S.part.nranks;
    const std::vector<double> sz = S.hostAllgather({(double)mine.size()});
    DBuf<uint8_t>& buf = scratch().gather;
    std::vector<std::vector<uint8_t>> all;
    if (S.part.rank == 0) {
        std::vector<size_t> off((size_t)N + 1, 0);
        for (int k = 0; k < N; ++k) off[k + 1] = off[k] + (k ? (size_t)std::llround(sz[k]) : 0);
        buf.alloc(off[N] + 1);
        std::vector<int> peers; std::vector<const void*> sb; std::vector<void*> rb; std::vector<size_t> sby, rby;
        for (int k = 1; k < N; ++k) { peers.push_back(k); sb.push_back(nullptr); sby.push_back(0); rb.push_back(buf.p + off[k]); rby.push_back(off[k + 1] - off[k]); }
        S.comm->sendrecv(N - 1, peers.data(), sb.data(), sby.data(), rb.data(), rby.data(), S.st);
        all.resize((size_t)N);
        all[0] = mine;
        for (int k = 1; k < N; ++k) { all[k].resize(off[k + 1] - off[k]); copy_d2h(all[k].data(), buf.p + off[k], all[k].size(), S.st); }
        stream_sync(S.st);
    } else {
        buf.alloc(mine.size() + 1);
        copy_h2d(buf.p, mine.data(), mine.size(), S.st);
        const int root = 0; const void* sb = buf.p; void* rb = nullptr; const size_t sby = mine.size(), rby = 0;
        S.comm->sendrecv(1, &root, &sb, &sby, &rb, &rby, S.st);
        stream_sync(S.st);      // the staging buffer is reused by the next gather
    }
    return all;
}

// Collective: a table of n items of `stride` values on rank 0, every item copied from the rank that owns it (`own`: the items of
// this rank's copy `local` that it owns); the other ranks get an empty table
template <class T>
std::vector<T> gather_owned(Solver& S, const std::vector<T>& local, const Spans& own, int64_t n, int stride = 1) {
    std::vector<uint8_t> mine;
    const int64_t ns = (int64_t)own.size();
    put(mine, &ns, 1);
    for (const auto& s : own) { put(mine, &s.first, 1); put(mine, &s.second, 1); put(mine, local.data() + s.first * stride, (size_t)(s.second - s.first) * stride); }
    const std::vector<std::vector<uint8_t>> all = gather_bytes(S, mine);
    std::vector<T> out;
    if (S.part.rank != 0) return out;
    out.assign((size_t)n * stride, T());
    for (const auto& piece : all) {
        const uint8_t* q = piece.data();
        int64_t m; q = take(q, &m, 1);
        for (int64_t i = 0; i < m; ++i) { int64_t a, b; q = take(q, &a, 1); q = take(q, &b, 1); q = take(q, out.data() + a * stride, (size_t)(b - a) * stride); }
    }
    return out;
}

// Rows of K_ext in the compact form of CompactOp (code word, then the 6 stored columns of each row): the active rows (G / D^T), or
// the coupled reduced rows (JG / JD^T) with their packed faces, the rows of region r at [regStart[r], regStart[r+1]), and the
// regions' centres of mass.  This rank's rows, or (`global`, several ranks, collective) every row from its owner, on rank 0.
struct KRows { std::vector<uint64_t> code; std::vector<int32_t> col; std::vector<int32_t> face; std::vector<int64_t> regStart; std::vector<double> com; };

KRows k_rows(Solver& S, bool reduced, bool global) {
    const Counts& C = S.C;
    const int R = S.RG.count;
    const int64_t nRows = C.nRowsExt, lo = reduced ? C.nActiveVs : 0, n = reduced ? nRows - C.nActiveVs : C.nActiveVs;
    KRows K;
    const std::vector<uint64_t> code = S.Op.kcode.to_host(S.st, (size_t)nRows);
    const std::vector<int32_t> col = S.Op.kcol.to_host(S.st, (size_t)6 * nRows);      // [6][nRows]
    K.code.assign(code.begin() + lo, code.begin() + lo + n);
    K.col.resize((size_t)6 * n);
    for (int64_t i = 0; i < n; ++i) for (int k = 0; k < 6; ++k) K.col[(size_t)6 * i + k] = col[(size_t)k * nRows + lo + i];
    if (reduced && R > 0) {
        K.face = S.RG.rowFace.to_host(S.st, (size_t)n);
        K.com = S.RG.com.to_host(S.st, (size_t)3 * R);
        const std::vector<int32_t> start = S.RG.rowStart.to_host(S.st, (size_t)R + 1);
        K.regStart.assign(start.begin(), start.end());
    }
    if (!global || !S.part.multi()) return K;
    const Spans own = spans_in(S.ownK, lo, lo + n);
    K.code = gather_owned(S, K.code, own, n);
    K.col = gather_owned(S, K.col, own, n, 6);
    if (!reduced || R == 0) return K;
    std::vector<int32_t> region = S.RG.rowRegion.to_host(S.st, (size_t)n);
    region = gather_owned(S, region, own, n);
    K.face = gather_owned(S, K.face, own, n);
    K.com = gather_owned(S, K.com, region_spans(S, 3), (int64_t)3 * R);
    if (S.part.rank != 0) return K;
    // The rows come in the ranks' order: by region, face axis and voxel order within each rank.  A shared region (ps_part.hpp) has rows
    // on several ranks; the cuts are whole tile layers and the tiles are numbered z-slowest, so its rows of one axis are in voxel
    // order when taken rank after rank.  A stable sort by (region, axis) thus restores the row order of one GPU, and the duplicate
    // columns of k_block are summed in the same order.
    std::vector<int64_t> ord((size_t)n);
    for (int64_t i = 0; i < n; ++i) ord[i] = i;
    auto key = [&](int64_t i) { return (int64_t)region[i] * 4 + ((K.face[i] >> 29) & 3); };
    std::stable_sort(ord.begin(), ord.end(), [&](int64_t a, int64_t b) { return key(a) < key(b); });
    KRows G;
    G.code.resize((size_t)n); G.col.resize((size_t)6 * n); G.face.resize((size_t)n); G.com = std::move(K.com);
    G.regStart.assign((size_t)R + 1, 0);
    for (int64_t i = 0; i < n; ++i) {
        const int64_t j = ord[i];
        G.code[i] = K.code[j]; G.face[i] = K.face[j];
        std::copy(K.col.begin() + 6 * j, K.col.begin() + 6 * j + 6, G.col.begin() + 6 * i);
        ++G.regStart[region[j] + 1];
    }
    for (int r = 0; r < R; ++r) G.regStart[r + 1] += G.regStart[r];
    return G;
}

// G / D^T (active rows) and JG / JD^T (26 rows per region) rebuilt from the compact rows of K_ext with the reference's CSR
// conventions (sorted columns, duplicates summed in traversal order, explicit zeros kept: S_CMB:454-455, 524-525, 612-613;
// SURVEY.md section 8c)
HostCsr k_block(const Solver& S, const KRows& K, const std::string& name) {
    const Counts& C = S.C;
    const int64_t nP = C.nPressures, nT = C.nStresses;
    const double sc = S.g.invDx / 64.;
    // the 8 (value, column) slots of row i: the compact form expanded as the operator kernels read it
    auto slots = [&](size_t i, double* v, int32_t* c) {
        const int32_t* col = K.col.data() + 6 * i;
        const int32_t c0w = col[0];
        const int64_t cOff = nP + (int64_t)((uint32_t)c0w >> 30) * C.nCenter;
        const int64_t c0 = c0w & OP_COL_MASK, c1 = col[1];
        const int64_t cc[8] = {c0, c1, cOff + c0, cOff + c1, col[2], col[3], col[4], col[5]};
        for (int k = 0; k < 8; ++k) { v[k] = (double)op_code(K.code[i], k) * sc; c[k] = (int32_t)cc[k]; }
    };
    const bool pressure = (name == "G" || name == "JG");
    const int64_t colLo = pressure ? 0 : nP, colHi = pressure ? nP : nP + nT;
    HostCsr m; m.cols = colHi - colLo;
    double v[8]; int32_t c[8];
    if (name == "G" || name == "Dt") {
        m.rows = C.nActiveVs; m.ptr.assign(m.rows + 1, 0);
        for (int64_t r = 0; r < m.rows; ++r) {
            std::vector<std::pair<int32_t, double>> e;
            slots((size_t)r, v, c);
            for (int k = 0; k < 8; ++k) if (v[k] != 0. && c[k] >= colLo && c[k] < colHi) e.push_back({(int32_t)(c[k] - colLo), v[k]});
            std::sort(e.begin(), e.end(), [](auto& a, auto& b) { return a.first < b.first; });
            for (auto& x : e) { m.idx.push_back(x.first); m.val.push_back(x.second); }
            m.ptr[r + 1] = (int64_t)m.idx.size();
        }
        return m;
    }
    const int R = S.RG.count;
    m.rows = (int64_t)R * RDOF; m.ptr.assign(m.rows + 1, 0);
    if (R == 0) return m;
    for (int r = 0; r < R; ++r) {
        std::map<int32_t, std::array<double, RDOF>> cols;
        for (int64_t row = K.regStart[r]; row < K.regStart[r + 1]; ++row) {
            const int32_t packed = K.face[row];
            const int axis = (packed >> 29) & 3;
            const I3 f = delin(S.g, SL_FACE + axis, (int64_t)(packed & 0x1fffffff));
            double p[3] = {(double)f.x, (double)f.y, (double)f.z};
            p[axis] -= 0.5;
            double cf[RDOF];
            conversion_coefficients(p[0] * S.g.dx - K.com[3 * r], p[1] * S.g.dx - K.com[3 * r + 1], p[2] * S.g.dx - K.com[3 * r + 2], axis, cf);
            slots((size_t)row, v, c);
            for (int k = 0; k < 8; ++k) {
                if (v[k] == 0. || c[k] < colLo || c[k] >= colHi) continue;
                auto it = cols.find((int32_t)(c[k] - colLo));
                if (it == cols.end()) { std::array<double, RDOF> a; for (int n = 0; n < RDOF; ++n) a[n] = v[k] * cf[n]; cols.emplace((int32_t)(c[k] - colLo), a); }
                else for (int n = 0; n < RDOF; ++n) it->second[n] += v[k] * cf[n];
            }
        }
        for (int n = 0; n < RDOF; ++n) {
            for (auto& kvp : cols) { m.idx.push_back(kvp.first); m.val.push_back(kvp.second[n]); }
            m.ptr[(int64_t)r * RDOF + n + 1] = (int64_t)m.idx.size();
        }
    }
    return m;
}

// A vector as this rank holds it, and the entries of it this rank owns.  `share`: distributed data whose per-rank view keeps only the
// owned entries (zero elsewhere, so the sum over the ranks is the global vector); the other vectors are returned as held.
struct Piece { std::vector<double> v; Spans own; bool share = false; };

bool vector_piece(Solver& S, const std::string& n, Piece& p) {
    const Counts& C = S.C; const int R = S.RG.count; const size_t NN = (size_t)RDOF * RDOF;
    const int64_t nA = C.nActiveVs, nP = C.nPressures, nSys = C.nSystemSize;
    auto reg = [&](const DBuf<double>& d, size_t per, bool share) { p.v = R ? d.to_host(S.st, (size_t)R * per) : std::vector<double>(); p.own = region_spans(S, (int64_t)per); p.share = share; };
    auto sys = [&](std::vector<double>&& v) { p.v = std::move(v); p.own = spans_in(S.ownSys, 0, nSys); p.share = true; };
    if (n == "activeRHS") { p.v = S.rhsU.to_host(S.st, (size_t)nA); p.own = spans_in(S.ownK, 0, nA); }
    else if (n == "oldActiveVs") { p.v = S.oldVs.to_host(S.st, (size_t)nA); p.own = spans_in(S.ownK, 0, nA); }
    else if (n == "reducedRHS") reg(S.RG.rhsR, RDOF, true);
    else if (n == "pressureRHS") { p.v = S.rhsPT.to_host(S.st, (size_t)nP); p.own = spans_in(S.ownSys, 0, nP); }
    else if (n == "stressRHS") { auto v = S.rhsPT.to_host(S.st, (size_t)nSys); p.v.assign(v.begin() + nP, v.end()); p.own = spans_in(S.ownSys, nP, nSys); }
    else if (n == "b") sys(S.b.to_host(S.st, (size_t)nSys));
    else if (n == "solution") sys(S.x.to_host(S.st, (size_t)nSys));
    else if (n == "guess") sys(S.haveGuess ? S.guess.to_host(S.st, (size_t)nSys) : std::vector<double>((size_t)nSys, 0.));
    else if (n == "velSolution") {
        p.v = S.velSol.to_host(S.st, (size_t)(nA + C.nReducedVs));
        p.own = spans_in(S.ownK, 0, nA); p.own.push_back(region_spans(S, RDOF, nA)[0]); p.share = true;
    }
    else if (n == "com") reg(S.RG.com, 3, false);
    else if (n == "bestFit") reg(S.RG.bestFit, RDOF, true);
    else if (n == "MrDense") reg(S.RG.Mr, NN, true);
    else if (n == "ViscDense") reg(S.RG.Visc, NN, true);
    else if (n == "BinvDense") reg(S.RG.Binv, NN, true);
    else return false;
    return true;
}
// the vector as the caller sees it: this rank's view, or with `global` on a decomposed handle the whole vector on rank 0 (collective;
// the other ranks get an empty vector)
std::vector<double> view(Solver& S, Piece&& p, bool global) {
    if (!S.part.multi()) return std::move(p.v);
    if (global) return gather_owned(S, p.v, p.own, (int64_t)p.v.size());
    if (!p.share) return std::move(p.v);
    std::vector<double> m(p.v.size(), 0.);
    for (const auto& s : p.own) std::copy(p.v.begin() + s.first, p.v.begin() + s.second, m.begin() + s.first);
    return m;
}

bool get_vector(Solver& S, const std::string& n, std::vector<double>& out, bool global) {
    // replicated on every rank: the same answer from any rank, no collective
    if (n == "unitLoad") { out = S.unitLoad; return true; }
    if (n == "unitCounts") { out.assign(S.unitCounts.begin(), S.unitCounts.end()); return true; }
    if (n == "diagA") { if (S.part.multi()) return false; S.computeDiagonal(); out = S.diagA.to_host(S.st, (size_t)S.C.nSystemSize); return true; }
    if (n == "guess" && global && S.part.multi()) S.constructGuessVectors();      // several ranks: formed where it is read (collective)
    Piece p;
    if (!vector_piece(S, n, p)) return false;
    out = view(S, std::move(p), global);
    return true;
}

bool is_matrix(const std::string& n) {
    for (const char* m : {"G", "Dt", "JG", "JDt", "A", "Mc", "McInv", "uInv", "u", "Mr", "B", "BInv"}) if (n == m) return true;
    return false;
}
// a matrix by name: this rank's view (on a rank of a decomposed handle the region blocks of its own regions only), or with `global`
// the whole matrix on rank 0 (collective; the other ranks leave `out` empty).  The explicit A is built on one GPU only.
void get_matrix(Solver& S, const std::string& name, HostCsr& out, bool global) {
    const Counts& C = S.C;
    const int R = S.RG.count;
    const bool here = !global || !S.part.multi() || S.part.rank == 0;
    if (name == "G" || name == "Dt" || name == "JG" || name == "JDt") {
        const KRows K = k_rows(S, name == "JG" || name == "JDt", global);
        if (here) out = k_block(S, K, name);
        return;
    }
    if (name == "A") {     // explicit system matrix, built on the device (ps_explicit.cu)
        if (global && S.part.multi()) throw Error("the explicit A is built on one GPU");
        S.buildExplicitA();
        out.rows = out.cols = S.Aexp.n;
        out.ptr = S.Aexp.ptr.to_host(S.st, (size_t)S.Aexp.n + 1);
        out.idx = S.Aexp.nnz ? S.Aexp.idx.to_host(S.st, (size_t)S.Aexp.nnz) : std::vector<int32_t>();
        out.val = S.Aexp.nnz ? S.Aexp.val.to_host(S.st, (size_t)S.Aexp.nnz) : std::vector<double>();
        return;
    }
    auto diag = [&](const DBuf<double>& d, int64_t n, const Spans& own) {
        Piece p; p.v = d.to_host(S.st, (size_t)n); p.own = own;
        const std::vector<double> v = view(S, std::move(p), global);
        if (here) out = diag_csr(v);
    };
    const Spans active = spans_in(S.ownK, 0, C.nActiveVs), stress = spans_in(S.ownSys, C.nPressures, C.nSystemSize);
    if (name == "Mc") diag(S.mc, C.nActiveVs, active);
    else if (name == "McInv") diag(S.mcInv, C.nActiveVs, active);
    else if (name == "uInv") diag(S.uInv, C.nStresses, stress);
    else if (name == "u") diag(S.uDiag, C.nStresses, stress);
    else {
        // the region blocks; a rank's own view holds those of its own regions only (the blocks of the other regions are zero)
        std::vector<double> a, v;
        get_vector(S, name == "BInv" ? "BinvDense" : "MrDense", a, global);
        if (name == "B") {
            get_vector(S, "ViscDense", v, global);
            for (size_t i = 0; i < a.size(); ++i) a[i] = S.g.invDt * a[i] + 2. * v[i];
        }
        if (here) out = blockdiag_csr(a, R);
    }
}

// Eigen::saveMarket / saveMarketVector format (extern/eigen/unsupported/Eigen/src/SparseExtra/MarketIO.h:311-372)
bool save_market(const HostCsr& m, const std::string& path) {
    std::ofstream out(path.c_str(), std::ios::out);
    if (!out) return false;
    out.flags(std::ios_base::scientific); out.precision(std::numeric_limits<double>::digits10 + 2);
    out << "%%MatrixMarket matrix coordinate  real general" << std::endl;
    out << m.rows << " " << m.cols << " " << m.idx.size() << "\n";
    for (int64_t r = 0; r < m.rows; ++r) for (int64_t p = m.ptr[r]; p < m.ptr[r + 1]; ++p) out << (r + 1) << " " << (m.idx[p] + 1) << " " << m.val[p] << "\n";
    return true;
}
bool save_market_vector(const std::vector<double>& v, const std::string& path) {
    std::ofstream out(path.c_str(), std::ios::out);
    if (!out) return false;
    out.flags(std::ios_base::scientific); out.precision(std::numeric_limits<double>::digits10 + 2);
    out << "%%MatrixMarket matrix array real general\n" << v.size() << " " << 1 << "\n";
    for (double x : v) out << x << "\n";
    return true;
}

// The views of a ps_create_multi handle are the global objects: fn(S, global = true, answer) runs on every rank (collective) and
// rank 0 answers the caller.  A single-GPU handle, or one rank of a job with one process per GPU, answers with its own view.
template <class Fn>
int views(ps_handle h, Fn&& fn) {
    if (!h->multi) return guarded(h, [&] { return fn(*h->S, false, true); });
    MultiGroup* G = h->multi;
    return G->run([&](int k) { ps_solver* kid = G->kids[(size_t)k]; return guarded(kid, [&] { return fn(*kid->S, true, k == 0); }); });
}

}  // namespace

extern "C" {

const char* ps_last_error(void) { return g_lastError.c_str(); }

int ps_create(const ps_params* params, ps_handle* out) {
    if (!params || !out) { g_lastError = "ps_create: null argument"; return PS_INVALID; }
    *out = nullptr;
    return guarded([&] {
        ps_solver* h = new ps_solver; h->S = nullptr;
        int prev = -1;
#ifndef PS_EMULATE
        if (cudaGetDevice(&prev) != cudaSuccess) { cudaGetLastError(); prev = -1; }
#endif
        try { h->S = new Solver(*params); } catch (...) { delete h; throw; }
#ifndef PS_EMULATE
        if (prev >= 0 && prev != params->device) cudaSetDevice(prev);      // the constructor selected the handle's device
#endif
        *out = h; return (int)PS_SUCCESS; });
}
void ps_destroy(ps_handle h) {
    if (!h) return;
    if (h->multi) {
        MultiGroup* G = h->multi;
        G->run([G](int k) { ps_destroy(G->kids[(size_t)k]); return (int)PS_SUCCESS; });     // every rank on its own thread: a rank's teardown may wait for its peers' streams
        G->stop();
        delete G;
        h->S = nullptr; h->multi = nullptr;
        delete h;
        return;
    }
#ifndef PS_EMULATE
    for (void* e : h->tm) if (e) cudaEventDestroy((cudaEvent_t)e);
#endif
    try { Enter e(h); delete h->S; h->S = nullptr; } catch (...) {}
    delete h;      // the scratch buffers go with it (cudaFree finds the owning device from the pointer)
}

#ifndef PS_EMULATE
int ps_comm_unique_id(void* id128) {
    if (!id128) { g_lastError = "ps_comm_unique_id: null argument"; return PS_INVALID; }
    return guarded([&] { nccl_unique_id(id128); return (int)PS_SUCCESS; });  // no handle
}
int ps_comm_init(ps_handle h, int rank, int nranks, const void* id128) {
    if (!h || !id128) { g_lastError = "ps_comm_init: null argument"; return PS_INVALID; }
    if (h->multi) { g_lastError = "ps_comm_init: a ps_create_multi handle is already decomposed"; return PS_INVALID; }
    return guarded(h, [&] {
        h->S->initComm(make_nccl_comm(rank, nranks, id128));
        h->S->setupPeer();
        return (int)PS_SUCCESS;
    });
}
// SURVEY.md section 8b: the caller is ONE cook thread (exec/HDK_PolyStokes.C:222); it cannot run one process per GPU.
int ps_create_multi(const ps_params* params, int ndev, const int* devs, ps_handle* out) {
    if (!params || !out || ndev < 1 || ndev > PEER_MAX_RANKS) { g_lastError = "ps_create_multi: bad argument (1 <= ndev <= 8)"; return PS_INVALID; }
    *out = nullptr;
    return guarded([&] {
        std::unique_ptr<MultiGroup> G(new MultiGroup);
        auto cleanup = [&] { for (ps_solver* k : G->kids) ps_destroy(k); G->kids.clear(); G->stop(); };
        for (int r = 0; r < ndev; ++r) {
            ps_params P = *params;
            P.device = devs ? devs[r] : r;
            ps_handle k = nullptr;
            if (ps_create(&P, &k) != PS_SUCCESS) { const std::string e = g_lastError; cleanup(); throw Error("ps_create_multi: device " + std::to_string(P.device) + ": " + e); }
            G->kids.push_back(k);
        }
        if (ndev > 1) {
            unsigned char id[128];
            nccl_unique_id(id);                  // also loads libnccl once, before the rank threads need it
            G->start(ndev);
            MultiGroup* g = G.get();
            const int rc = g->run([g, ndev, &id](int k) { return ps_comm_init(g->kids[(size_t)k], k, ndev, id); });
            if (rc != PS_SUCCESS) { const std::string e = g_lastError; cleanup(); throw Error("ps_create_multi: " + e); }
        } else G->start(1);
        ps_solver* h = new ps_solver;
        h->S = G->kids[0]->S;
        h->multi = G.release();
        *out = h;
        return (int)PS_SUCCESS;
    });
}
#else
int ps_create_multi(const ps_params*, int, const int*, ps_handle* out) { if (out) *out = nullptr; g_lastError = "ps_create_multi: needs CUDA devices (the emulation twin is single process per rank)"; return PS_FAILED; }
// the emulation twin has no NCCL: tests/ hand it host callbacks (torch.distributed / gloo) instead
int ps_comm_unique_id(void* id128) { if (id128) memset(id128, 0, 128); return PS_SUCCESS; }
int ps_comm_init(ps_handle, int, int, const void*) { g_lastError = "ps_comm_init: the emulation twin takes ps_comm_init_callbacks"; return PS_FAILED; }
int ps_comm_init_callbacks(ps_handle h, int rank, int nranks, ps_allreduce_cb ar, ps_sendrecv_cb sr, void* ctx) {
    if (!h || !ar || !sr) return PS_INVALID;
    return guarded(h, [&] { h->S->initComm(make_callback_comm(rank, nranks, ar, sr, ctx)); return (int)PS_SUCCESS; });
}
#endif
int ps_get_partition(ps_handle h, int32_t* rank, int32_t* zLo, int32_t* zHi, int32_t* zCut) {
    if (!h) return -1;
    const Partition& p = h->S->part;
    if (rank) *rank = p.rank;
    if (zLo) *zLo = p.zCut[p.rank];
    if (zHi) *zHi = p.zCut[p.rank + 1];
    if (zCut) for (int k = 0; k <= p.nranks; ++k) zCut[k] = p.zCut[k];
    return p.nranks;
}

int ps_set_partition(ps_handle h, const int32_t* zCut) {
    if (!h) { g_lastError = "ps_set_partition: null handle"; return PS_INVALID; }
    if (h->multi) { MultiGroup* G = h->multi; return G->run([&](int k) { return ps_set_partition(G->kids[(size_t)k], zCut); }); }
    return guarded(h, [&] { return h->S->setPartition(zCut); });
}
int ps_rebalance(ps_handle h, int32_t* zCut) {
    if (!h) { g_lastError = "ps_rebalance: null handle"; return PS_INVALID; }
    if (h->multi) { MultiGroup* G = h->multi; return G->run([&](int k) { return ps_rebalance(G->kids[(size_t)k], k == 0 ? zCut : nullptr); }); }
    return guarded(h, [&] { return h->S->rebalance(zCut); });
}

int ps_set_params(ps_handle h, const ps_params* params) {
    if (!h || !params) { g_lastError = "ps_set_params: null argument"; return PS_INVALID; }
    if (h->multi) { MultiGroup* G = h->multi; return G->run([&](int k) { return ps_set_params(G->kids[(size_t)k], params); }); }
    return guarded(h, [&] { h->S->setParams(*params); return (int)PS_SUCCESS; });
}
// pinned host memory for callers without CUDA headers (the node adaptor's staging arrays): copies from / to it overlap with kernels
void* ps_alloc_pinned(size_t bytes) {
#ifndef PS_EMULATE
    void* p = nullptr;
    if (cudaMallocHost(&p, bytes ? bytes : 16) != cudaSuccess) { cudaGetLastError(); g_lastError = "ps_alloc_pinned: cudaMallocHost failed"; return nullptr; }
    return p;
#else
    return malloc(bytes ? bytes : 16);
#endif
}
void ps_free_pinned(void* p) {
#ifndef PS_EMULATE
    if (p) cudaFreeHost(p);
#else
    free(p);
#endif
}

// stats of a collective call: rank 0's, with the slowest rank's stage times and the launches of all ranks
static void merge_stats(ps_stats* dst, const std::vector<ps_stats>& all) {
    if (!dst || all.empty()) return;
    *dst = all[0];
    dst->gpu_launches = 0;
    for (const ps_stats& s : all) { dst->gpu_launches += s.gpu_launches; for (int i = 0; i < PS_NUM_STAGES; ++i) dst->stage_ms[i] = std::max(dst->stage_ms[i], s.stage_ms[i]); }
}

int ps_step(ps_handle h, const ps_fields_in* in, ps_fields_out* out, ps_stats* stats) {
    if (!h || !in) { g_lastError = "ps_step: null argument"; return PS_INVALID; }
    if (h->multi) {
        MultiGroup* G = h->multi;
        std::vector<ps_stats> st(G->kids.size());
        const int rc = G->run([&](int k) { return ps_step(G->kids[(size_t)k], in, out, &st[(size_t)k]); });
        merge_stats(stats, st);
        return rc;
    }
    return guarded(h, [&] {
        Solver& S = *h->S;
        const int res = S.step(*in, out, stats);
        if (S.P.exportMatrices || S.P.exportComponentMatrices || S.P.exportStats)
            ps_export(h, S.P.exportDataPrefix, (S.P.exportMatrices ? 1 : 0) | (S.P.exportComponentMatrices ? 2 : 0) | (S.P.exportStats ? 4 : 0));
        return res;
    });
}
int ps_setup(ps_handle h, const ps_fields_in* in) {
    if (!h || !in) { g_lastError = "ps_setup: null argument"; return PS_INVALID; }
    if (h->multi) { MultiGroup* G = h->multi; return G->run([&](int k) { return ps_setup(G->kids[(size_t)k], in); }); }
    return guarded(h, [&] { Solver& S = *h->S; for (double& m : S.stageMs) m = 0; g_launches = 0; 
        try { S.setInputsAndSetup(*in); }
        catch (...) { stream_sync(S.stIn); S.lateInputsPending = false; throw; }   // no copy may outlive the error return
        return (int)PS_SUCCESS; });
}
int ps_solve(ps_handle h, ps_fields_out* out, ps_stats* stats) {
    if (!h) { g_lastError = "ps_solve: null handle"; return PS_INVALID; }
    if (h->multi) {
        MultiGroup* G = h->multi;
        std::vector<ps_stats> st(G->kids.size());
        const int rc = G->run([&](int k) { return ps_solve(G->kids[(size_t)k], out, &st[(size_t)k]); });
        merge_stats(stats, st);
        return rc;
    }
    return guarded(h, [&] {
        Solver& S = *h->S;
        if (!S.haveSetup) throw Error("ps_solve: call ps_setup first");
        S.stageMs[PS_STAGE_SOLVE] = 0; S.stageMs[PS_STAGE_WRITEBACK] = 0;
        const int res = S.solve();
        if (out && res != PS_UNSUPPORTED_SOLVER) {
            if (res == PS_SUCCESS || S.P.keepNonConvergedResults) S.recoverVelocityFromPressureStress();
            S.applySolutionToVelocity(*out);
        }
        if (stats) S.fillStats(stats);
        return res;
    });
}

int64_t ps_get_count(ps_handle h, const char* name) {
    if (!h || !name) return INT64_MIN;
    const Solver& S = *h->S; const Counts& C = S.C; const std::string n(name);
    if (n == "nCenter") return C.nCenter;
    if (n == "nFaceX") return C.nFace[0]; if (n == "nFaceY") return C.nFace[1]; if (n == "nFaceZ") return C.nFace[2];
    if (n == "nEdgeYZ") return C.nEdge[0]; if (n == "nEdgeXZ") return C.nEdge[1]; if (n == "nEdgeXY") return C.nEdge[2];
    if (n == "nActiveVs") return C.nActiveVs; if (n == "nReducedVs") return C.nReducedVs;
    if (n == "nPressures") return C.nPressures; if (n == "nStresses") return C.nStresses;
    if (n == "nTotalDOFs") return C.nTotalDOFs; if (n == "nSystemSize") return C.nSystemSize;
    if (n == "regionCount") return S.RG.count; if (n == "iterations") return S.solveIterations;
    if (n == "peerTransport") return S.peer.on ? 1 : 0;
    if (n == "slabLocal") return S.part.local ? 1 : 0;
    if (n == "sharedRegions") return S.RG.nShared;
    if (n == "sharedPeerExchanges") return S.sharedPeerExchanges;      // moment sums of shared regions since the last setup, peer transport
    if (n == "sharedCommExchanges") return S.sharedCommExchanges;      // ... and by the communicator's all-reduce
    if (n == "peerSharedCap") return PEER_SH_CAP;      // shared regions the peer moment area holds; a step with more takes the communicator
    if (n == "directHalo") return S.fusedHalo ? 1 : 0;      // boundary entries stored straight into the neighbours' vectors (ps_peer.hpp, VecLink)
    if (n == "result") return S.result; if (n == "usedBiCGStab") return S.usedBiCGStab;
    if (n == "nRowsExt") return C.nRowsExt; if (n == "fixLoops") return S.fixLoops;
    // the shape of the reduced regions and the kernels their term of an apply takes (ps_pcg.cu, region_path)
    if (n == "maxRegionRows") return S.RG.maxRegionRows; if (n == "maxRegionAxisRows") return S.RG.maxRegionAxisRows;
    if (n == "maxRegionCells") return S.RG.maxRegionCells; if (n == "minRegionCells") return S.RG.minRegionCells;
    if (n == "regionPath") return region_path(S.RG);
    return INT64_MIN;
}
double ps_get_real(ps_handle h, const char* name) {
    if (!h || !name) return NAN;
    const std::string n(name);
    if (n == "solveError") return h->S->solveError;
    if (n == "xmag") return h->S->solveXmag;
    return NAN;
}

int64_t ps_get_index_field(ps_handle h, int kind, int slot, int32_t* out) {
    if (!h || slot < 0 || slot >= N_SLOTS || kind < 0 || kind > 2) return -1;
    if (h->multi) { g_lastError = "ps_get_index_field: per-voxel views of a ps_create_multi handle live on several GPUs; use a single-GPU handle"; return -1; }
    Solver& S = *h->S;
    const size_t n = (size_t)S.g.n[slot];
    if (!out) return (int64_t)n;
    int rc = guarded(h, [&] {
        if (kind == 0) { std::vector<int8_t> v = S.dLabel[slot].to_host(S.st, n); for (size_t i = 0; i < n; ++i) out[i] = v[i]; }
        else { std::vector<int32_t> v = (kind == 1 ? S.dAidx[slot] : S.dRidx[slot]).to_host(S.st, n); std::copy(v.begin(), v.end(), out); }
        return 0;
    });
    return rc == 0 ? (int64_t)n : -1;
}
int64_t ps_get_weight_field(ps_handle h, int liquid, int slot, float* out) {
    if (!h || slot < 0 || slot >= N_SLOTS) return -1;
    if (h->multi) { g_lastError = "ps_get_weight_field: per-voxel views of a ps_create_multi handle live on several GPUs; use a single-GPU handle"; return -1; }
    Solver& S = *h->S;
    const size_t n = (size_t)S.g.n[slot];
    if (!out) return (int64_t)n;
    int rc = guarded(h, [&] { std::vector<uint8_t> v = (liquid ? S.dLiqW[slot] : S.dFluW[slot]).to_host(S.st, n); for (size_t i = 0; i < n; ++i) out[i] = (float)v[i] * 0.125f; return 0; });
    return rc == 0 ? (int64_t)n : -1;
}

int ps_get_csr(ps_handle h, const char* name, int64_t* rows, int64_t* cols, int64_t* nnz, int64_t* rowptr, int32_t* colidx, double* vals) {
    if (!h || !name) return PS_INVALID;
    const std::string nm(name);
    if (!is_matrix(nm)) { g_lastError = "ps_get_csr: unknown matrix " + nm; return PS_INVALID; }
    return views(h, [&](Solver& S, bool global, bool answer) {
        HostCsr m;
        get_matrix(S, nm, m, global);
        if (!answer) return (int)PS_SUCCESS;
        if (rows) *rows = m.rows;
        if (cols) *cols = m.cols;
        if (nnz) *nnz = (int64_t)m.idx.size();
        if (rowptr) std::copy(m.ptr.begin(), m.ptr.end(), rowptr);
        if (colidx) std::copy(m.idx.begin(), m.idx.end(), colidx);
        if (vals) std::copy(m.val.begin(), m.val.end(), vals);
        return (int)PS_SUCCESS;
    });
}
int64_t ps_get_vector(ps_handle h, const char* name, double* out) {
    if (!h || !name) return -1;
    int64_t n = -1;
    const int rc = views(h, [&](Solver& S, bool global, bool answer) {
        std::vector<double> v;
        if (!get_vector(S, name, v, global)) { g_lastError = std::string("ps_get_vector: no vector ") + name + " on this handle"; return (int)PS_INVALID; }
        if (answer) { n = (int64_t)v.size(); if (out) std::copy(v.begin(), v.end(), out); }
        return (int)PS_SUCCESS;
    });
    return rc == PS_SUCCESS ? n : -1;
}

int ps_apply(ps_handle h, const double* x, double* y) {
    if (!h || !x || !y) return PS_INVALID;
    return views(h, [&](Solver& S, bool global, bool answer) {
        if (!S.haveSetup) throw Error("ps_apply: call ps_setup first");
        const size_t n = (size_t)S.C.nSystemSize;
        DBuf<double>& dx = scratch().applyX; DBuf<double>& dy = scratch().applyY;
        dx.alloc(n); dy.alloc(n);
        copy_h2d(dx.p, x, n * sizeof(double), S.st);
        dy.zero(S.st, n);                       // several ranks: rows of other ranks stay 0 (sum over ranks = A x)
        S.applyOperator(dx.p, dy.p, nullptr);
        if (!global || !S.part.multi()) { copy_d2h(y, dy.p, n * sizeof(double), S.st); return (int)PS_SUCCESS; }
        const std::vector<double> all = gather_owned(S, dy.to_host(S.st, n), spans_in(S.ownSys, 0, (int64_t)n), (int64_t)n);
        if (answer) std::copy(all.begin(), all.end(), y);
        return (int)PS_SUCCESS;
    });
}

double ps_kernel_bytes(ps_handle h, const char* name) {
    if (!h || !name) return 0;
    const Solver& S = *h->S; const Counts& C = S.C; const std::string nm(name);
    // DESIGN.md section 5; the byte model itself is OpBytes (ps_solver.hpp), also behind the unit loads of ps_rebalance
    OpCounts c;
    c.nCenter = C.nCenter; c.nActiveVs = C.nActiveVs; c.nEdges = C.nEdge[0] + C.nEdge[1] + C.nEdge[2]; c.nRedRows = S.RG.nRows; c.nRegions = S.RG.count;
    const OpBytes b(c);
    if (nm == "csr_pass1") return b.csrPass1;
    if (nm == "csr_pass2") return b.csrPass2;
    if (nm == "csr_apply") return b.csrApply;
    if (nm == "pass1") return b.pass1;
    if (nm == "pass1_sweep") return b.pass1Sweep;
    if (nm == "pass2") return b.pass2;
    if (nm == "pass2_dots") return b.pass2Dots;
    if (nm == "reduced") return b.reduced;
    if (nm == "apply") return b.pass1 + b.pass2;
    if (nm == "cg_update") return b.cgUpdate;
    if (nm == "cg_iteration") return b.cgIteration;
    return 0;
}

double ps_time_kernel(ps_handle h, const char* name, int reps) {
    if (!h || !name || reps <= 0) return -1;
    if (h->multi) {     // collective; the slowest rank's time
        MultiGroup* G = h->multi;
        std::vector<double> t(G->kids.size(), -1.);
        G->run([&](int k) { t[(size_t)k] = ps_time_kernel(G->kids[(size_t)k], name, reps); return t[(size_t)k] < 0 ? (int)PS_FAILED : (int)PS_SUCCESS; });
        double worst = -1; bool bad = false;
        for (double v : t) { if (v < 0) bad = true; worst = std::max(worst, v); }
        return bad ? -1 : worst;
    }
    double ms = -1;
    guarded(h, [&] {
        Solver& S = *h->S; const std::string nm(name);
        if (!S.haveSetup) throw Error("ps_time_kernel: call ps_setup first");
        if (nm == "cg_iteration") {
            const int savedMax = S.P.maxSolverIterations, savedEvery = S.P.checkEvery; const double savedTol = S.P.tolerance;
            S.P.maxSolverIterations = reps; S.P.checkEvery = reps; S.P.tolerance = 0.0;   // never converges: exactly `reps` iterations
            S.stageMs[PS_STAGE_SOLVE] = 0;
            S.cgOnly = true;
            try { S.solve(); } catch (...) { S.cgOnly = false; throw; }
            S.cgOnly = false;
            ms = S.stageMs[PS_STAGE_SOLVE] / reps;
            S.P.maxSolverIterations = savedMax; S.P.checkEvery = savedEvery; S.P.tolerance = savedTol;
            return 0;
        }
        const int which = nm == "pass1" ? 1 : nm == "pass2" ? 2 : nm == "apply" ? 0 : nm == "pass1_sweep" ? 3 : nm == "pass2_dots" ? 4 : nm == "cg_update" ? 5 : nm == "reduced" ? 6 : -1;
        if (which < 0) throw Error("ps_time_kernel: unknown kernel name");
        // the CG kernels look at the device scalars: a fresh state that cannot converge or run out of iterations while timed (the iterates are
        // garbage -- only the memory traffic matters here)
        k_cg_init(S.st, S.ownSys, S.b.p, S.x.p, S.r.p, S.p.p, S.dotPartial.p, S.scal.p, 0.0, reps + 8, PeerCtx());
#ifndef PS_EMULATE
        cudaEvent_t a, b; PS_CUDA(cudaEventCreate(&a)); PS_CUDA(cudaEventCreate(&b));
        S.timedOperator(which);
        PS_CUDA(cudaEventRecord(a, S.st));
        for (int i = 0; i < reps; ++i) S.timedOperator(which);
        PS_CUDA(cudaEventRecord(b, S.st)); PS_CUDA(cudaEventSynchronize(b));
        float t = 0; PS_CUDA(cudaEventElapsedTime(&t, a, b)); ms = t / reps;
        cudaEventDestroy(a); cudaEventDestroy(b);
#else
        S.timedOperator(which); ms = 0;
#endif
        return 0;
    });
    return ms;
}

// Device-side stopwatch for callers that time whole steps: the solver works on its own stream, which an outside event
// (e.g. torch.cuda.Event on torch's current stream) does not see.
double ps_timer(ps_handle h, int stop) {
    if (!h) return -1;
    if (h->multi) {     // every rank's own stream; the slowest rank's time
        MultiGroup* G = h->multi;
        std::vector<double> t(G->kids.size(), -1.);
        G->run([&](int k) { t[(size_t)k] = ps_timer(G->kids[(size_t)k], stop); return t[(size_t)k] < 0 ? (int)PS_FAILED : (int)PS_SUCCESS; });
        double worst = -1; bool bad = false;
        for (double v : t) { if (v < 0) bad = true; worst = std::max(worst, v); }
        return bad ? -1 : worst;
    }
    double ms = -1;
    guarded(h, [&] {
#ifndef PS_EMULATE
        Solver& S = *h->S;
        for (void*& e : h->tm) if (!e) { cudaEvent_t ev; PS_CUDA(cudaEventCreate(&ev)); e = ev; }
        if (!stop) { PS_CUDA(cudaEventRecord((cudaEvent_t)h->tm[0], S.st)); ms = 0; return 0; }
        PS_CUDA(cudaEventRecord((cudaEvent_t)h->tm[1], S.st)); PS_CUDA(cudaEventSynchronize((cudaEvent_t)h->tm[1]));
        float t = 0; PS_CUDA(cudaEventElapsedTime(&t, (cudaEvent_t)h->tm[0], (cudaEvent_t)h->tm[1])); ms = t;
#else
        ms = 0;
#endif
        return 0;
    });
    return ms;
}

// On a decomposed handle (several ranks, either front end) ps_export is collective: the objects are assembled on rank 0 from their
// owners (gather_owned), rank 0 alone writes, and one all-reduce of a status word gives every rank the same return code.
int ps_export(ps_handle h, const char* prefix, int what) {
    if (!h || !prefix) return PS_INVALID;
    if (h->multi) { MultiGroup* G = h->multi; return G->run([&](int k) { return ps_export(G->kids[(size_t)k], prefix, what); }); }
    return guarded(h, [&] {
        Solver& S = *h->S; const std::string pre(prefix);
        const bool multi = S.part.multi(), writer = S.part.rank == 0;
        bool ok = true;
        std::vector<double> v;
        auto vec = [&](const char* name, const char* file) { if (get_vector(S, name, v, true) && writer) ok &= save_market_vector(v, pre + file); };
        if (what & 1) {   // exportMatrices / exportMatricesPostSolve (S.cpp:533-541, 568-572); A is implicit on this path
            vec("b", "Vec_b.mtx");
            vec("guess", "Vec_guess.mtx");
            // Mat_A.mtx: the explicit matrix exists only for solverType EIGEN (S_AS:7-27); the factored path leaves A an
            // empty nSystemSize x nSystemSize matrix (A.resize only, S_AS:446) and that is what the reference writes
            HostCsr Am;
            if (S.P.solverType == 1 && !multi) get_matrix(S, "A", Am, true);
            else { Am.rows = Am.cols = S.C.nSystemSize; Am.ptr.assign((size_t)Am.rows + 1, 0); }
            if (writer) ok &= save_market(Am, pre + "Mat_A.mtx");
            vec("solution", "solutionVector.mtx");
        }
        if (what & 2) {   // exportComponentMatrices (S.cpp:543-566)
            const char* mats[] = {"Mc", "McInv", "Mr", "B", "BInv", "u", "uInv", "G", "Dt", "JG", "JDt"};
            const char* files[] = {"Mat_Mc.mtx", "Mat_McInv.mtx", "Mat_Mr.mtx", "Mat_Mr_plus_2JDtuDJ.mtx", "Mat_Inv_Mr_plus_2JDtuDJ.mtx", "Mat_u.mtx", "Mat_uInv.mtx",
                                   "Mat_G.mtx", "Mat_Dt.mtx", "Mat_JG.mtx", "Mat_JDt.mtx"};
            for (int i = 0; i < 11; ++i) { HostCsr m; get_matrix(S, mats[i], m, true); if (writer) ok &= save_market(m, pre + files[i]); }
            const char* vecs[] = {"activeRHS", "reducedRHS", "pressureRHS", "stressRHS"};
            const char* vfiles[] = {"Vec_activeRHS.mtx", "Vec_reducedRHS.mtx", "Vec_pressureRHS.mtx", "Vec_stressRHS.mtx"};
            for (int i = 0; i < 4; ++i) vec(vecs[i], vfiles[i]);
        }
        if (what & 4) {   // exportStats (S.cpp:574-606)
            ps_stats st; S.fillStats(&st);
            if (multi) {  // the counts are global already; the "thread count" is the SMs of all ranks, the times are the slowest rank's
                const std::vector<double> all = S.hostAllgather({st.dimData[22], st.solveData[2], st.solveData[3], st.solveData[4], st.solveData[5]});
                st.dimData[22] = 0.;
                for (int k = 0; k < S.part.nranks; ++k) {
                    st.dimData[22] += all[(size_t)5 * k];
                    for (int j = 1; j < 5; ++j) st.solveData[1 + j] = std::max(st.solveData[1 + j], all[(size_t)5 * k + j]);
                }
            }
            if (writer) {
                ok &= save_market_vector(std::vector<double>(st.dimData, st.dimData + 27), pre + "dimData.mtx");
                ok &= save_market_vector(std::vector<double>(st.solveData, st.solveData + 6), pre + "solveData.mtx");
            }
        }
        if (multi) ok = S.hostAllreduceSum(ok ? 0. : 1.) < 0.5;
        if (!ok) { g_lastError = "ps_export: could not write under prefix " + pre; return (int)PS_FAILED; }
        return (int)PS_SUCCESS;
    });
}

}  // extern "C"
