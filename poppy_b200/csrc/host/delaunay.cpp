#include "delaunay.hpp"

#include <emmintrin.h>

#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstring>
#include <thread>
#include <unordered_map>

#include <sys/mman.h>

#include <cstdlib>

namespace poppy {

namespace {
constexpr size_t kHugePage = 2u << 20, kHugeMin = 256u << 10;
struct HugeCache {          // the blocks a thread freed last (one per size class seen), reused by its next mesh
    static constexpr int kSlots = 4;
    void* ptr[kSlots] = {nullptr, nullptr, nullptr, nullptr};
    size_t size[kSlots] = {0, 0, 0, 0};
    ~HugeCache() { for (void* p : ptr) std::free(p); }
};
thread_local HugeCache g_huge_cache;
size_t huge_round(size_t bytes) { return (bytes + kHugePage - 1) / kHugePage * kHugePage; }
}  // namespace

void* huge_alloc(size_t bytes) {
    if (bytes < kHugeMin) {
        void* p = std::malloc(bytes ? bytes : 1);
        if (!p) throw std::bad_alloc();
        return p;
    }
    const size_t size = huge_round(bytes);
    HugeCache& c = g_huge_cache;
    for (int i = 0; i < HugeCache::kSlots; ++i)
        if (c.ptr[i] && c.size[i] == size) { void* p = c.ptr[i]; c.ptr[i] = nullptr; return p; }
    void* p = std::aligned_alloc(kHugePage, size);
    if (!p) throw std::bad_alloc();
    madvise(p, size, MADV_HUGEPAGE);          // advisory: ordinary pages serve equally well, only slower
    return p;
}

void huge_free(void* p, size_t bytes) {
    if (!p) return;
    if (bytes < kHugeMin) { std::free(p); return; }
    HugeCache& c = g_huge_cache;
    const size_t size = huge_round(bytes);
    for (int i = 0; i < HugeCache::kSlots; ++i)
        if (!c.ptr[i]) { c.ptr[i] = p; c.size[i] = size; return; }
    std::free(c.ptr[0]);                      // cache full: drop the oldest entry
    for (int i = 0; i + 1 < HugeCache::kSlots; ++i) { c.ptr[i] = c.ptr[i + 1]; c.size[i] = c.size[i + 1]; }
    c.ptr[HugeCache::kSlots - 1] = p; c.size[HugeCache::kSlots - 1] = size;
}

void clip_points(std::vector<Point2f>& pts, int cols, int rows) {
    for (Point2f& p : pts) {
        p.x = p.x > cols ? cols - 1 : p.x;
        p.y = p.y > rows ? rows - 1 : p.y;
        p.x = p.x < 0 ? 0 : p.x;
        p.y = p.y < 0 ? 0 : p.y;
    }
}

namespace {
uint64_t point_key(Point2f p) {
    // exact float equality classes: +0 and -0 compare equal
    float x = p.x == 0.f ? 0.f : p.x, y = p.y == 0.f ? 0.f : p.y;
    uint32_t a, b;
    std::memcpy(&a, &x, 4);
    std::memcpy(&b, &y, 4);
    return ((uint64_t)a << 32) | b;
}
}  // namespace

void make_uniq(const std::vector<Point2f>& pts, std::vector<Point2f>& out, std::vector<int32_t>* first_index) {
    // open-addressing set of the bit patterns seen so far (slot = index + 1 of the first occurrence, 0 = empty)
    size_t cap = 16;
    while (cap < pts.size() * 2 + 2) cap <<= 1;
    std::vector<int32_t> slot(cap, 0);
    out.reserve(out.size() + pts.size());
    if (first_index) first_index->reserve(first_index->size() + pts.size());
    for (size_t i = 0; i < pts.size(); ++i) {
        const uint64_t key = point_key(pts[i]);
        size_t h = (size_t)((key * 0x9E3779B97F4A7C15ull) >> 17) & (cap - 1);
        bool seen = false;
        for (; slot[h]; h = (h + 1) & (cap - 1))
            if (point_key(pts[slot[h] - 1]) == key) { seen = true; break; }
        if (seen) continue;
        slot[h] = (int32_t)i + 1;
        out.push_back(pts[i]);
        if (first_index) first_index->push_back((int32_t)i);
    }
}

// ---------------------------------------------------------------------------------------------------------------
DelaunayMesh::DelaunayMesh(int width, int height, int expected_points) {
    const float big = 3.f * (float)(width > height ? width : height);
    top_left_ = {0.f, 0.f};
    bottom_right_ = {(float)width, (float)height};
    q_.reserve((size_t)3 * (expected_points > 0 ? expected_points : 64) + 16);
    org_.reserve(2 * q_.capacity());
    pt_.reserve((size_t)(expected_points > 0 ? expected_points : 64) + 8);
    // slot 0 of both tables is the null element
    q_.push_back(Quad{});
    org_.assign(2, 0);
    pt_.push_back({0.f, 0.f});
    const int a = new_vertex({big, 0.f}), b = new_vertex({0.f, big}), c = new_vertex({-big, -big});
    const int ab = new_quad(), bc = new_quad(), ca = new_quad();
    set_ends(ab, a, b);
    set_ends(bc, b, c);
    set_ends(ca, c, a);
    splice(ab, sym(ca));
    splice(bc, sym(ab));
    splice(ca, sym(bc));
    recent_ = ab;
}

int DelaunayMesh::new_quad() {
    if (free_quad_ <= 0) {
        q_.push_back(Quad{});
        org_.insert(org_.end(), 2, 0);
        free_quad_ = (int)q_.size() - 1;
    }
    const int e = free_quad_ * 4;
    Quad& q = q_[free_quad_];
    free_quad_ = q.next[1];
    q.next[0] = e; q.next[1] = e + 3; q.next[2] = e + 2; q.next[3] = e + 1;
    org_[e >> 1] = org_[(e >> 1) + 1] = 0;
    q.opt[0] = q.opt[1] = pt_[0];
    return e;
}

void DelaunayMesh::free_quad_of(int e) {
    splice(e, oprev(e));
    const int s = sym(e);
    splice(s, oprev(s));
    Quad& q = q_[e >> 2];
    q.next[0] = 0;
    q.next[1] = free_quad_;
    free_quad_ = e >> 2;
}

int DelaunayMesh::new_vertex(Point2f p) {
    pt_.push_back(p);
    return (int)pt_.size() - 1;
}

void DelaunayMesh::splice(int a, int b) {
    int& an = next_of(a);
    int& bn = next_of(b);
    int& arn = next_of(rot(an, 1));
    int& brn = next_of(rot(bn, 1));
    std::swap(an, bn);
    std::swap(arn, brn);
}

void DelaunayMesh::set_ends(int e, int o, int d) {
    Quad& q = q_[e >> 2];
    const int r = e & 3;                    // primal: 0 or 2
    org_[e >> 1] = o;
    org_[(e >> 1) ^ 1] = d;
    q.opt[r >> 1] = pt_[o];
    q.opt[(r >> 1) ^ 1] = pt_[d];
}

int DelaunayMesh::connect(int a, int b) {
    const int e = new_quad();
    splice(e, lnext(a));
    splice(sym(e), b);
    set_ends(e, dst(a), org(b));
    return e;
}

void DelaunayMesh::flip(int e) {
    const int s = sym(e), a = oprev(e), b = oprev(s);
    splice(e, a);
    splice(s, b);
    set_ends(e, dst(a), dst(b));
    splice(e, lnext(a));
    splice(s, lnext(b));
}

namespace {
double tri_area(Point2f a, Point2f b, Point2f c) {
    return ((double)b.x - a.x) * ((double)c.y - a.y) - ((double)b.y - a.y) * ((double)c.x - a.x);
}

int in_circle(Point2f pt, Point2f a, Point2f b, Point2f c) {
    const double eps = FLT_EPSILON * 0.125;
    double v = ((double)a.x * a.x + (double)a.y * a.y) * tri_area(b, c, pt);
    v -= ((double)b.x * b.x + (double)b.y * b.y) * tri_area(a, c, pt);
    v += ((double)c.x * c.x + (double)c.y * c.y) * tri_area(a, b, pt);
    v -= ((double)pt.x * pt.x + (double)pt.y * pt.y) * tri_area(a, b, c);
    return v > eps ? 1 : v < -eps ? -1 : 0;
}
}  // namespace

int DelaunayMesh::side_of(Point2f p, int e) const {
    const Quad& q = q_[e >> 2];
    const int k = (e >> 1) & 1;
    const double cw = tri_area(p, q.opt[k ^ 1], q.opt[k]);
    return (cw > 0) - (cw < 0);
}

bool DelaunayMesh::begin_walk(Point2f p, Walk& w) const {
    w.p = p;
    w.e = 0;
    w.r_cur = 0;
    w.budget = (int)q_.size() * 4;
    w.where = kOutside;
    if (p.x < top_left_.x || p.y < top_left_.y || p.x >= bottom_right_.x || p.y >= bottom_right_.y) return false;
    w.where = kError;
    w.e = recent_;
    w.r_cur = side_of(p, w.e);
    if (w.r_cur > 0) { w.e = sym(w.e); w.r_cur = -w.r_cur; }
    return true;
}

bool DelaunayMesh::walk_step(Walk& w) const {
    if (w.budget-- <= 0) return false;                 // Subdiv2D::locate gives up after 4 * quads steps
    const Quad* __restrict__ q = q_.data();
    const Point2f p = w.p;
    const int e = w.e;
    const Quad& qe = q[e >> 2];
    const int on = qe.next[e & 3], dp = rot(qe.next[(e + 3) & 3], 3);
    const Quad& qon = q[on >> 2];
    const Quad& qdp = q[dp >> 2];
    const int kon = (on >> 1) & 1, kdp = (dp >> 1) & 1;
    const double a_on = tri_area(p, qon.opt[kon ^ 1], qon.opt[kon]), a_dp = tri_area(p, qdp.opt[kdp ^ 1], qdp.opt[kdp]);
    if (w.r_cur != 0 && a_on != 0 && a_dp != 0) {
        // general position (the common case): the four sign combinations of Subdiv2D::locate collapse to
        // "inside" or one conditional move, so the walk has no data-dependent branch to mispredict
        if (a_on > 0 && a_dp > 0) { w.where = kInside; return false; }
        const int go_dp = -(int)(a_on > 0);          // right of onext (then not right of dprev): cross dprev, else onext
        w.e = on ^ ((on ^ dp) & go_dp);
        w.r_cur = -1;
        return true;
    }
    const int r_on = (a_on > 0) - (a_on < 0), r_dp = (a_dp > 0) - (a_dp < 0);
    if (r_dp > 0) {
        if (r_on > 0 || (r_on == 0 && w.r_cur == 0)) { w.where = kInside; return false; }
        w.r_cur = r_on;
        w.e = on;
    } else if (r_on > 0) {
        if (r_dp == 0 && w.r_cur == 0) { w.where = kInside; return false; }
        w.r_cur = r_dp;
        w.e = dp;
    } else if (w.r_cur == 0 && side_of(pt_[dst(on)], e) >= 0) {
        w.e = sym(e);
    } else {
        w.r_cur = r_on;
        w.e = on;
    }
    return true;
}

namespace {
// A walk state with everything its step needs already in hand: the edge, its onext / dprev edges, and the coordinate
// differences (B - p, C - p) of their two orientation predicates tri_area(p, B, C).
struct WalkCand {
    int e, on, dp, pad;
    double on_bx, on_by, on_cx, on_cy, dp_bx, dp_by, dp_cx, dp_cy;
};
}  // namespace

void DelaunayMesh::MoveLog::open(WalkTrace* trace) {
    t = trace;
    acc = 0;
    pos = limit = 0;
    if (!t) return;
    pos = t->first[t->points];
    const uint64_t capacity = (uint64_t)t->bits.size() * 64;
    limit = (uint32_t)std::min<uint64_t>((uint64_t)pos + WalkTrace::kMaxSteps, capacity > 64 ? capacity - 64 : 0);
    if (limit < pos) limit = pos;
    acc = (pos & 63) ? __atomic_load_n(&t->bits[pos >> 6], __ATOMIC_RELAXED) & ((1ull << (pos & 63)) - 1) : 0;
}

void DelaunayMesh::MoveLog::close() {
    if (!t) return;
    if ((size_t)t->points + 1 >= t->first.size()) return;                 // more points than begin() was told: not recorded
    if (pos & 63) __atomic_store_n(&t->bits[pos >> 6], acc & ((1ull << (pos & 63)) - 1), __ATOMIC_RELAXED);
    t->first[t->points + 1] = pos;
    ++t->points;
}

namespace {
// Bit pattern of tri_area(p, q.opt[1], q.opt[0]) = (o1.x - p.x) * (o0.y - p.y) - (o1.y - p.y) * (o0.x - p.x), evaluated with
// the same double operations in the same order as tri_area() (SSE2: both differences of a point in one instruction).
// The predicate of the edge's other direction, tri_area(p, opt[0], opt[1]), is its exact negation (the products commute
// and rounding is symmetric), i.e. the sign bit flipped.
inline int64_t area_bits(const float* opt, __m128d P) {
    const __m128 v = _mm_load_ps(opt);                                  // o0.x o0.y o1.x o1.y
    const __m128d d0 = _mm_sub_pd(_mm_cvtps_pd(v), P);                  // o0 - p
    const __m128d d1 = _mm_sub_pd(_mm_cvtps_pd(_mm_movehl_ps(v, v)), P);     // o1 - p
    const __m128d m = _mm_mul_pd(d1, _mm_shuffle_pd(d0, d0, 1));        // d1.x * d0.y , d1.y * d0.x
    const __m128d a = _mm_sub_sd(m, _mm_unpackhi_pd(m, m));
    return _mm_cvtsi128_si64(_mm_castpd_si128(a));
}
}  // namespace

void DelaunayMesh::walk_guided(Walk& w, const uint64_t* bits, uint32_t first, int count, MoveLog* log) const {
    if (w.r_cur == 0 || count <= 0 || w.budget <= 0) return;
    const Quad* __restrict__ q = q_.data();
    const __m128d P = _mm_set_pd((double)w.p.y, (double)w.p.x);
    const int steps = std::min(count, w.budget);
    int e = w.e, j = 0;
    // the guide's bits pass through one register; the moves taken are appended to the log in bulk afterwards (they are
    // the guide's bits except at the - at most 9 - steps noted in wrong_at)
    uint64_t word = __atomic_load_n(&bits[first >> 6], __ATOMIC_RELAXED) >> (first & 63);
    int left = 64 - (int)(first & 63);
    uint16_t wrong_at[kMaxWrong + 1];
    int wrong = 0;
    for (; j < steps; ++j) {
        const int bit = (int)(word & 1);
        word >>= 1;
        if (--left == 0) { word = __atomic_load_n(&bits[(first + (uint32_t)j + 1) >> 6], __ATOMIC_RELAXED); left = 64; }
        const Quad& qe = q[e >> 2];
        const int on = qe.next[e & 3], dp = rot(qe.next[(e + 3) & 3], 3);
        int nxt = bit ? dp : on;                // the only value the next step's loads wait for
        // the two orientation predicates of the step, off that chain
        const int64_t ion = area_bits(&q[on >> 2].opt[0].x, P) ^ (int64_t)((uint64_t)((on >> 1) & 1) << 63);
        const int64_t idp = area_bits(&q[dp >> 2].opt[0].x, P) ^ (int64_t)((uint64_t)((dp >> 1) & 1) << 63);
        // what walk_step / walk_run do here: general position (neither predicate zero), not inside (not both > 0),
        // move = (a_on > 0). Integer operations on the bit patterns: a compare-and-branch on a_on > 0 would mispredict
        // every other step and throw away the loads the next steps have already started.
        const int g_on = ion > 0, g_dp = idp > 0;                        // x > 0 (no NaNs; -0.0 and +0.0 are not > 0)
        const int z = (int)(((uint64_t)ion << 1) == 0) | (int)(((uint64_t)idp << 1) == 0);
        if (__builtin_expect(z | (g_on & g_dp), 0)) break;               // degenerate or inside: the ordinary walk decides
        if (__builtin_expect(g_on ^ bit, 0)) {
            // wrong prediction (an edge flipped since the guide was recorded): take the real move; the paths usually
            // rejoin a step or two later with the same number of moves, so the following bits still apply
            asm volatile("" ::: "memory");      // keeps this a branch: as a conditional move it would tie nxt to the predicates
            nxt = g_on ? dp : on;
            wrong_at[wrong++] = (uint16_t)j;
            if (wrong > kMaxWrong) { e = nxt; ++j; break; }              // the guide no longer describes this walk
        }
        e = nxt;
    }
    if (j == 0) return;
    w.e = e;
    w.budget -= j;
    w.r_cur = -1;
    if (log) log->append(bits, first, j, wrong_at, wrong);
}

// n moves = bits first .. first + n - 1 of src with the positions listed in flips inverted
void DelaunayMesh::MoveLog::append(const uint64_t* src, uint32_t first, int n, const uint16_t* flips, int n_flips) {
    if (!t) return;
    int f = 0;
    for (int done = 0; done < n && pos < limit;) {
        const uint32_t sb = first + (uint32_t)done;
        const int take = std::min({n - done, 64 - (int)(sb & 63), 64 - (int)(pos & 63), (int)(limit - pos)});
        uint64_t chunk = __atomic_load_n(&src[sb >> 6], __ATOMIC_RELAXED) >> (sb & 63);
        if (take < 64) chunk &= (1ull << take) - 1;
        while (f < n_flips && (int)flips[f] < done + take) { chunk ^= 1ull << (flips[f] - done); ++f; }
        acc |= chunk << (pos & 63);
        pos += (uint32_t)take;
        done += take;
        if ((pos & 63) == 0) { __atomic_store_n(&t->bits[(pos >> 6) - 1], acc, __ATOMIC_RELAXED); acc = 0; }
    }
}

bool DelaunayMesh::walk_run(Walk& w) const { return walk_run(w, nullptr); }

bool DelaunayMesh::walk_run(Walk& w, MoveLog* log) const {
    if (w.r_cur == 0) return false;
    const Quad* __restrict__ q = q_.data();
    const double px = w.p.x, py = w.p.y;
    auto fill = [&](int x, WalkCand& c) {
        const Quad& qx = q[x >> 2];
        const int on = qx.next[x & 3], dp = rot(qx.next[(x + 3) & 3], 3);
        const Quad& qo = q[on >> 2];
        const Quad& qd = q[dp >> 2];
        // one level further: the records fill(on) / fill(dp) will read their coordinates from (the quads of onext and
        // dprev of both successors) start their way from L2 now, a whole step before the loads that need them
        __builtin_prefetch(&q[qo.next[on & 3] >> 2]);
        __builtin_prefetch(&q[qo.next[(on + 3) & 3] >> 2]);
        __builtin_prefetch(&q[qd.next[dp & 3] >> 2]);
        __builtin_prefetch(&q[qd.next[(dp + 3) & 3] >> 2]);
        const int ko = (on >> 1) & 1, kd = (dp >> 1) & 1;
        c.e = x; c.on = on; c.dp = dp;
        c.on_bx = (double)qo.opt[ko ^ 1].x - px; c.on_by = (double)qo.opt[ko ^ 1].y - py;
        c.on_cx = (double)qo.opt[ko].x - px;     c.on_cy = (double)qo.opt[ko].y - py;
        c.dp_bx = (double)qd.opt[kd ^ 1].x - px; c.dp_by = (double)qd.opt[kd ^ 1].y - py;
        c.dp_cx = (double)qd.opt[kd].x - px;     c.dp_cy = (double)qd.opt[kd].y - py;
    };
    WalkCand buf[2][2];
    fill(w.e, buf[0][0]);
    const WalkCand* cur = &buf[0][0];
    for (int side = 1;; side ^= 1) {
        if (w.budget <= 0) { w.e = cur->e; w.r_cur = -1; return false; }     // walk_step reports the exhausted budget
        // both successors, speculatively (independent of the predicates below)
        WalkCand* nxt = buf[side];
        fill(cur->on, nxt[0]);
        fill(cur->dp, nxt[1]);
        const double a_on = cur->on_bx * cur->on_cy - cur->on_by * cur->on_cx;      // tri_area(p, B, C) of onext
        const double a_dp = cur->dp_bx * cur->dp_cy - cur->dp_by * cur->dp_cx;      // ... of dprev
        if (a_on == 0 || a_dp == 0) { w.e = cur->e; w.r_cur = -1; return false; }   // degenerate: the generic step decides
        --w.budget;
        if (a_on > 0 && a_dp > 0) {
            w.e = cur->e; w.r_cur = -1; w.where = kInside;
            return true;
        }
        if (log) log->push(a_on > 0);
        cur = &nxt[a_on > 0];      // right of onext (then not right of dprev): cross dprev, else onext
    }
}

DelaunayMesh::Where DelaunayMesh::classify(const Walk& w, int& out_edge, int& out_vertex) {
    out_edge = 0;
    out_vertex = 0;
    if (w.where == kOutside) return kOutside;
    const int e = w.e;
    const Point2f p = w.p;
    Where where = w.where;
    recent_ = e;
    if (where == kInside) {
        const Point2f o = pt_[org(e)], d = pt_[dst(e)];
        double t1 = std::fabs(p.x - o.x);
        t1 += std::fabs(p.y - o.y);
        double t2 = std::fabs(p.x - d.x);
        t2 += std::fabs(p.y - d.y);
        double t3 = std::fabs(o.x - d.x);
        t3 += std::fabs(o.y - d.y);
        if (t1 < FLT_EPSILON) { out_vertex = org(e); return kVertex; }
        if (t2 < FLT_EPSILON) { out_vertex = dst(e); return kVertex; }
        if ((t1 < t3 || t2 < t3) && std::fabs(tri_area(p, o, d)) < FLT_EPSILON) where = kOnEdge;
    }
    if (where == kError) return kError;
    out_edge = e;
    return where;
}

int DelaunayMesh::insert(Point2f p) { return insert(p, nullptr, 0, nullptr); }

int DelaunayMesh::insert(Point2f p, const WalkTrace* guide, int index, WalkTrace* record, int guide_points) {
    Walk w;
    MoveLog log;
    if (record) log.open(record);
    MoveLog* lg = record ? &log : nullptr;
    if (begin_walk(p, w)) {
        if (guide && index < (guide_points >= 0 ? guide_points : guide->points)) {
            const uint32_t f0 = guide->first[index];
            walk_guided(w, guide->bits.data(), f0, (int)(guide->first[index + 1] - f0), lg);
        }
        // general-position stretches run in the dependence-cut loop; a degenerate predicate is decided by one generic
        // step, after which the fast loop resumes
        while (!walk_run(w, lg)) {
            if (lg) lg->stop();
            if (!walk_step(w)) break;
        }
    }
    if (record) log.close();
    return finish_insert(w);
}

int DelaunayMesh::finish_insert(Walk& w) {
    const Point2f p = w.p;
    int cur = 0, vtx = 0;
    const Where where = classify(w, cur, vtx);
    if (where == kOutside) { err_ = "point outside the subdivision rectangle (cv::Subdiv2D: StsOutOfRange)"; return -1; }
    if (where == kError) { err_ = "point location failed (cv::Subdiv2D: StsBadSize)"; return -1; }
    if (where == kVertex) return vtx;
    if (where == kOnEdge) {
        const int doomed = cur;
        recent_ = cur = oprev(cur);
        free_quad_of(doomed);
    }
    const int v = new_vertex(p);
    int base = new_quad();
    const int first = org(cur);
    set_ends(base, first, v);
    splice(base, cur);
    do {
        base = connect(cur, sym(base));
        cur = oprev(base);
    } while (dst(cur) != first);
    cur = oprev(base);
    const int budget = (int)q_.size() * 4;
    // The swap loop reads every coordinate from the quad records it is walking anyway (Quad::opt mirrors pt_[org]); the
    // vertex tables (org_ -> pt_, two more dependent loads per point) are not touched. Vertices of a mesh have pairwise
    // different coordinates (insert() returns the existing vertex for a repeated point), so "org(cur) == first" can be
    // decided on the coordinates as well.
    const Point2f first_pt = pt_[first];
    for (int i = 0; i < budget; ++i) {
        const int t = oprev(cur);
        const Quad& qc = q_[cur >> 2];
        const Quad& qt = q_[t >> 2];
        const int kc = (cur >> 1) & 1, kt = (t >> 1) & 1;
        const Point2f c_org = qc.opt[kc], c_dst = qc.opt[kc ^ 1], t_dst = qt.opt[kt ^ 1];
        const double cw = tri_area(t_dst, c_dst, c_org);                 // side_of(t_dst, cur)
        if (cw > 0 && in_circle(c_org, t_dst, c_dst, p) < 0) {
            flip(cur);
            cur = oprev(cur);
        } else if (c_org.x == first_pt.x && c_org.y == first_pt.y) {
            break;
        } else {
            cur = lprev(onext(cur));
        }
    }
    return v;
}

void DelaunayMesh::triangles(std::vector<int32_t>& ids) const {
    ids.clear();
    const int total = (int)q_.size() * 4;
    std::vector<char> seen(total, 0);
    for (int e = 4; e < total; e += 2) {
        if (seen[e]) continue;
        const int a = org(e);
        if (a < 4) continue;                  // null / bounding-triangle vertex: outside the rect
        const int eb = lnext(e), b = org(eb);
        if (b < 4) continue;
        const int ec = lnext(eb), c = org(ec);
        if (c < 4) continue;
        seen[e] = seen[eb] = seen[ec] = 1;
        ids.push_back(a);
        ids.push_back(b);
        ids.push_back(c);
    }
}

bool triangulate_points(std::vector<Point2f> points, int width, int height, std::vector<int32_t>& tri_idx,
                        std::string* error, const WalkTrace* guide, WalkTrace* record, const WalkPace* pace) {
    tri_idx.clear();
    // whatever happens, a follower waiting on this triangulation is released when it ends
    struct Release {
        std::atomic<int>* p;
        ~Release() { if (p) p->store(INT_MAX, std::memory_order_release); }
    } release{pace ? pace->publish : nullptr};
    clip_points(points, width, height);
    std::vector<Point2f> uniq;
    std::vector<int32_t> first;
    make_uniq(points, uniq, &first);
    if (record) record->begin((int)uniq.size());
    DelaunayMesh mesh(width, height, (int)uniq.size());
    std::vector<int32_t> owner(4, -1);        // mesh vertex id -> index of its first occurrence in `points`
    int guide_ready = (pace && pace->follow) ? 0 : -1;      // points of the guide known to be published (-1: all of guide->points)
    for (size_t i = 0; i < uniq.size(); ++i) {
        if (guide_ready >= 0 && guide_ready != INT_MAX && (int)i >= guide_ready) {
            // stay behind the triangulation that records the guide: its point i must be published before ours is predicted
            for (int spins = 0;; ++spins) {
                guide_ready = pace->follow->load(std::memory_order_acquire);
                if (guide_ready > (int)i) break;
                if (spins < 256) _mm_pause(); else std::this_thread::yield();
            }
        }
        const int avail = guide_ready == INT_MAX ? -1 : guide_ready;
        const int v = mesh.insert(uniq[i], guide, (int)i, record, avail);
        if (v < 0) {
            if (error) *error = mesh.error();
            if (record) record->points = 0;       // (not freed: a follower may still be reading what was published)
            return false;
        }
        if (pace && pace->publish) pace->publish->store((int)i + 1, std::memory_order_release);
        if (v >= (int)owner.size()) owner.resize(v + 1, -1);
        if (owner[v] < 0) owner[v] = first[i];
    }
    std::vector<int32_t> ids;
    mesh.triangles(ids);
    tri_idx.resize(ids.size());
    for (size_t i = 0; i < ids.size(); ++i) tri_idx[i] = owner[ids[i]];
    return true;
}

bool triangulate_points_next(std::vector<Point2f> points, int width, int height, std::vector<int32_t>& tri_idx,
                             std::string* error) {
    thread_local WalkTrace traces[2];
    thread_local int cur = 0;
    const bool ok = triangulate_points(std::move(points), width, height, tri_idx, error, traces[cur].empty() ? nullptr : &traces[cur],
                                       &traces[cur ^ 1]);
    if (ok) cur ^= 1;
    return ok;
}

}  // namespace poppy
