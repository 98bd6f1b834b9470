// Host topology stage: incremental Delaunay triangulation of the morphed points with the exact insertion,
// point-location and enumeration behaviour of cv::Subdiv2D 4.6.0, because the *order* of the triangle list decides
// which triangle owns a shared pixel (reference src/algo.cpp:60-81,95-106,205-213).
//
// Restated from the published quad-edge algorithm (Guibas & Stolfi 1985) as OpenCV instantiates it:
//   OCV imgproc/src/subdivision2d.cpp:45-110 (edge algebra), :222-248 (splice / connect / swap), :264-404 (locate),
//   :412-490 (insert), :492-540 (bounding triangle), :756-785 (getTriangleList).
// The topology stays on the host by design (north-star); this file replaces only the O(T*N) std::find lookup of
// get_triangle_indices by an O(1) table that returns the same first-occurrence index.
#pragma once

#include <atomic>
#include <climits>
#include <cstddef>
#include <cstdint>
#include <string>
#include <vector>

namespace poppy {

struct Point2f {
    float x, y;
};

// clip_points(), reference src/util.cpp:453-460 (note: ">" — a coordinate equal to cols/rows passes)
void clip_points(std::vector<Point2f>& pts, int cols, int rows);

// make_uniq(), reference src/util.cpp:541-548: first occurrences in order. first_index[i] is the position in
// `pts` of unique point i.
void make_uniq(const std::vector<Point2f>& pts, std::vector<Point2f>& out, std::vector<int32_t>* first_index = nullptr);

// The moves of the point-location walks of one triangulation, one bit per general-position step (0: the walk crossed to
// onext, 1: to dprev), per inserted point. Consecutive frames of a sequence move every point by a fraction of a pixel, so
// the walks of frame f are an almost perfect PREDICTION of the walks of frame f + 1: DelaunayMesh::insert follows the
// recorded moves speculatively and only checks each step's two orientation predicates against them, which turns the
// walk's chain of dependent loads and compares (load -> load -> convert -> multiply -> compare -> select, ~25 ns per step)
// into one dependent load per step with the predicates off the critical path. A wrong prediction is detected at the step
// where it happens and the ordinary walk takes over from that very state, so any trace - stale, foreign or garbage -
// yields exactly the triangulation an unguided insertion yields.
struct WalkTrace {
    static constexpr int kMaxSteps = 4096;       // recorded moves per point (longer walks are simply not predicted further)
    std::vector<uint32_t> first;                 // per point: index of its first bit; first[points] = total
    std::vector<uint64_t> bits;
    int points = 0;
    // Sized once per triangulation and never reallocated while it is recorded (moves that do not fit are dropped), so that
    // another thread may read the points already published (WalkPace) while the rest is still being written.
    void begin(int expected_points) {
        points = 0;
        first.assign((size_t)expected_points + 2, 0);
        bits.assign((size_t)expected_points * 6 + kMaxSteps / 64 + 2, 0);       // 384 moves per point on average
    }
    void clear() { first.clear(); bits.clear(); points = 0; }
    bool empty() const { return points == 0; }
};

// Lets the triangulation of frame f + 1 run a few points behind the triangulation of frame f on another thread, predicted by
// the very walks frame f is recording: `follow` is the number of points the guide has published (INT_MAX when it is
// complete), `publish` is where this triangulation reports its own progress.
struct WalkPace {
    const std::atomic<int>* follow = nullptr;
    std::atomic<int>* publish = nullptr;
};

// Allocator of the mesh tables: blocks of 256 KB and more are 2 MB-aligned and advised as transparent huge pages, so that the
// point-location walk - one dependent load into the 1.9 MB quad table per step - stops missing the first-level TLB (4 KB
// pages cover 384 KB of it); the last block a thread freed is kept for its next mesh (a fresh block is zero-filled by the
// kernel on first touch). Falls back to ordinary pages wherever the kernel does not grant huge ones.
void* huge_alloc(size_t bytes);
void huge_free(void* p, size_t bytes);
template <class T>
struct HugeAlloc {
    using value_type = T;
    HugeAlloc() = default;
    template <class U> HugeAlloc(const HugeAlloc<U>&) {}
    T* allocate(size_t n) { return static_cast<T*>(huge_alloc(n * sizeof(T))); }
    void deallocate(T* p, size_t n) { huge_free(p, n * sizeof(T)); }
    template <class U> bool operator==(const HugeAlloc<U>&) const { return true; }
    template <class U> bool operator!=(const HugeAlloc<U>&) const { return false; }
};

class DelaunayMesh {
public:
    // bounding rect [0,w) x [0,h), as Subdiv2D(Rect(0,0,w,h))
    // expected_points: capacity hint (the tables never move while points are inserted when it is large enough)
    DelaunayMesh(int width, int height, int expected_points = 0);

    // Subdiv2D::insert. Returns the vertex id (>= 4 for real points) or -1 when the point is outside the rect
    // (where cv::Subdiv2D throws StsOutOfRange); error() then describes it.
    int insert(Point2f pt);
    // the same with the walk predicted by point `index` of `guide` (nullable) and recorded as the next point of `record`
    // (nullable); identical results whatever the guide holds
    int insert(Point2f pt, const WalkTrace* guide, int index, WalkTrace* record, int guide_points = -1);

    enum Where { kError = -2, kOutside = -1, kInside = 0, kVertex = 1, kOnEdge = 2 };
    struct Walk {
        Point2f p;
        int e, r_cur, budget;
        Where where;
    };

    // The general-position steps of the same walk as one loop with the data dependences cut: while the two orientation
    // predicates of the current edge are evaluated, the links and end points of BOTH possible successors are already
    // being loaded and their coordinate differences formed, so a step costs one predicate latency instead of
    // load -> load -> predicate. Identical decisions to walk_step (same double arithmetic, same order); stops at the
    // first degenerate predicate. Returns true when the walk ended (w.where set), false when walk_step must continue.
    bool walk_run(Walk& w) const;

    // Appends the moves of one walk to a WalkTrace (register accumulator, flushed per 64 moves).
    struct MoveLog {
        WalkTrace* t = nullptr;
        uint64_t acc = 0;
        uint32_t pos = 0, limit = 0;
        void open(WalkTrace* trace);
        void push(int bit) {
            if (pos >= limit) return;
            acc |= (uint64_t)bit << (pos & 63);
            if ((++pos & 63) == 0) { __atomic_store_n(&t->bits[(pos >> 6) - 1], acc, __ATOMIC_RELAXED); acc = 0; }
        }
        void append(const uint64_t* src, uint32_t first, int n, const uint16_t* flips, int n_flips);
        void stop() { limit = pos; }            // a degenerate step: what follows is not a prefix of general-position moves
        void close();
    };
    bool walk_run(Walk& w, MoveLog* log) const;
    static constexpr int kMaxWrong = 8;         // wrong predictions after which a walk gives up on its guide
    // Follows up to `count` predicted moves (bits first .. first + count - 1 of `bits`), verifying each; stops in front of
    // the first step whose predicates disagree with the prediction (or end the walk, or are degenerate).
    void walk_guided(Walk& w, const uint64_t* bits, uint32_t first, int count, MoveLog* log) const;

    // Subdiv2D::getTriangleList order; each triangle as three vertex ids (all >= 4).
    void triangles(std::vector<int32_t>& vertex_ids) const;

    Point2f vertex(int id) const { return pt_[id]; }
    int vertex_count() const { return (int)pt_.size(); }
    const std::string& error() const { return err_; }

private:
    // insert() cut at the boundaries of its point-location walk, which insert() runs in between (walk_guided, walk_run,
    // and walk_step wherever a predicate is degenerate):
    //   begin_walk(p, w)   false: p is outside the rectangle (w.where = kOutside)
    //   walk_step(w)       one step of Subdiv2D::locate, degenerate predicates included; false when the walk has ended
    //   finish_insert(w)   classification of the final edge + the topology update; returns what insert() returns
    bool begin_walk(Point2f pt, Walk& w) const;
    bool walk_step(Walk& w) const;
    int finish_insert(Walk& w);

    // One quad-edge record = half a cache line: the four onext links and a copy of the origin coordinates of the two
    // primal edges, so that the point-location walk (latency-bound pointer chasing, ~120 steps per inserted point at
    // 20k points; three records per step: the current edge's, its onext's and its dprev's) never chases vertex
    // indices and its working set (32 B x 3 quads per point) stays inside a 2 MB L2. Vertex ids live in a cold table.
    struct alignas(32) Quad {
        int next[4];
        Point2f opt[2];     // coordinates of org(4q) and org(4q + 2)
    };
    // edge id = 4 * quad + rot
    int& next_of(int e) { return q_[e >> 2].next[e & 3]; }
    int onext(int e) const { return q_[e >> 2].next[e & 3]; }
    static int rot(int e, int r) { return (e & ~3) + ((e + r) & 3); }
    static int sym(int e) { return e ^ 2; }
    int oprev(int e) const { return rot(onext(rot(e, 1)), 1); }
    int lnext(int e) const { return rot(onext(rot(e, 3)), 1); }
    int lprev(int e) const { return sym(onext(e)); }
    int dprev(int e) const { return rot(onext(rot(e, 3)), 3); }
    int org(int e) const { return org_[e >> 1]; }          // primal edges only (e even)
    int dst(int e) const { return org_[(e >> 1) ^ 1]; }

    int new_quad();
    void free_quad_of(int e);
    int new_vertex(Point2f p);
    void splice(int a, int b);
    void set_ends(int e, int o, int d);
    int connect(int a, int b);
    void flip(int e);
    int side_of(Point2f p, int e) const;      // sign of "p is right of e" (primal edges only)
    Where classify(const Walk& w, int& edge, int& vertex);

    std::vector<Quad, HugeAlloc<Quad>> q_;
    std::vector<int, HugeAlloc<int>> org_;      // 2 per quad: origin vertex of edges 4q and 4q + 2
    std::vector<Point2f, HugeAlloc<Point2f>> pt_;
    int free_quad_ = 0;
    int recent_ = 0;
    Point2f top_left_{0, 0}, bottom_right_{0, 0};
    std::string err_;
};

// The host stage of morph_images for one frame (reference src/algo.cpp:205-213): clip, dedupe, triangulate, and
// return triangle vertex indices into `points` (first exact-equal occurrence), in getTriangleList order.
// Returns false (with `error`) where the reference would throw.
// guide / record (nullable): the walk traces of a neighbouring frame to predict from, and where to record this frame's.
bool triangulate_points(std::vector<Point2f> points, int width, int height, std::vector<int32_t>& tri_idx,
                        std::string* error = nullptr, const WalkTrace* guide = nullptr, WalkTrace* record = nullptr,
                        const WalkPace* pace = nullptr);

// triangulate_points for callers that triangulate the frames of a sequence one call at a time (the reference's own pattern:
// morph_images() once per frame): each call is predicted by the calling thread's previous call and records for the next.
bool triangulate_points_next(std::vector<Point2f> points, int width, int height, std::vector<int32_t>& tri_idx,
                             std::string* error = nullptr);

}  // namespace poppy
