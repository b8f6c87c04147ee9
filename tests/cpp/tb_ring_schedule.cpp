// tests/cpp/tb_ring_schedule.cpp -- CPU-only check of the shared-memory ring of the temporally blocked kernel
// (csrc/lbm_tb.cuh: tb_ring_at, tb_slots, tb_ring_put, tb_ring_pull), against the schedule of both marches.
//   tb_ring_schedule          -> prints "ok <checked pulls>" or the first violation (exit 1)
//   tb_ring_schedule bytes    -> prints the ring bytes per block for depth 3, 128 rows
//
// The marches of tb_thread are replayed step by step for a chunk: every stage k < T stores its column into its ring
// (tb_ring_put, one value per row and population that names stage, column, population and row), every stage k > 1
// pulls its column (tb_ring_pull, every row that has both neighbours).  A pull must return what stage k-1 computed for
// the columns c+1 / c / c-1 and rows y-1 / y / y+1 it pulls from; no slot may be read and written between the same two
// barriers (the skewed march has one barrier per step, the one-column-lag march one before each stage k > 1); and the
// pulls of the first and last row stay inside the slot of their group.  Also: tb_ring_fill (the ghost rows' constants,
// written once before the march) reaches every double of the ring, so every later pull returns them.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <map>
#include <vector>

#include "lbm_tb.cuh"

using namespace lbm;

namespace {

constexpr int B = 16;

double tag(int k, int c, int i, int y) { return (double)((((long long)k * 100000 + (c + 1000)) * 16 + i) * 1024 + y); }

struct Replay {
    int T;
    bool skew;
    std::vector<double> ring;
    std::vector<int> wrote_in, read_in;  // barrier interval of the last store / pull of each double (-1: none)
    std::map<double, int> where;         // tag -> index it was stored at
    long long pulls = 0;
    int epoch = 0;

    Replay(int T_, bool skew_) : T(T_), skew(skew_), ring(tb_ring_at<B>(T_, 0, 0), -1.0),
                                 wrote_in(ring.size(), -1), read_in(ring.size(), -1) {}

    bool fail(const char* what, int k, int c, int s, int y, int i) {
        std::printf("%s march, depth %d: %s (stage %d, column %d, step %d, row %d, population %d)\n",
                    skew ? "skewed" : "one-column-lag", T, what, k, c, s, y, i);
        return false;
    }

    bool store(int k, int c, int s, const TbSlots& o) {
        for (int y = 0; y < B; ++y) {
            double f[Q];
            for (int i = 0; i < Q; ++i) f[i] = tag(k, c, i, y);
            std::vector<double> before = ring;
            tb_ring_put<B>(ring.data() + y, k, o.st[0], o.st[1], o.st[2], f);
            int n = 0;
            for (size_t j = 0; j < ring.size(); ++j) {
                if (ring[j] == before[j]) continue;
                ++n;
                if (read_in[j] == epoch) return fail("store into a slot pulled from between the same barriers", k, c, s, y, -1);
                wrote_in[j] = epoch;
                where[ring[j]] = (int)j;
            }
            if (n != Q) return fail("store did not write nine distinct doubles", k, c, s, y, -1);
        }
        return true;
    }

    bool pull(int k, int c, int s, const TbSlots& o) {
        for (int y = 1; y < B - 1; ++y) {
            double f[Q];
            tb_ring_pull<B>(ring.data() + y, k - 1, o.pl[0], o.pl[1], o.pl[2], f);
            for (int i = 0; i < Q; ++i) {
                const double want = tag(k - 1, c - cxi(i), i, y - cyi(i));
                if (f[i] != want) return fail("pull got another cell's population", k, c, s, y, i);
                const int j = where.at(want);
                if (wrote_in[j] == epoch) return fail("pull of a slot stored into between the same barriers", k, c, s, y, i);
                read_in[j] = epoch;
            }
            ++pulls;
        }
        // the first and last row: every population from the slot of its group (rows outside the block are dead)
        std::vector<double> idx(ring.size());
        for (size_t j = 0; j < idx.size(); ++j) idx[j] = (double)j;
        for (int y : {0, B - 1}) {
            double f[Q];
            tb_ring_pull<B>(idx.data() + y, k - 1, o.pl[0], o.pl[1], o.pl[2], f);
            for (int i = 0; i < Q; ++i) {
                const int g = cxi(i) == -1 ? 0 : (cxi(i) == 0 ? 1 : 2);
                const int lo = tb_ring_at<B>(k - 1, g, 0) + o.pl[g];
                if (f[i] < lo || f[i] >= lo + 3 * B) return fail("edge row reads outside its slot", k, c, s, y, i);
            }
        }
        return true;
    }

    // columns [x0, x1) of one chunk; stage k works on the columns [x0 - (T-k), x1 + (T-k)) (tb_col_kind)
    bool chunk(int x0, int x1) {
        auto on = [&](int k, int c) { return c >= x0 - (T - k) && c < x1 + (T - k); };
        if (skew) {
            for (int s = x0 - (T - 1); s <= x1 - 1 + 2 * (T - 1); ++s) {
                const TbSlots o = tb_slots<B>(s, true);
                for (int k = T; k >= 2; --k) {
                    const int c = s - 2 * (k - 1);
                    if (!on(k, c)) continue;
                    if (!pull(k, c, s, o)) return false;
                    if (k < T && !store(k, c, s, o)) return false;
                }
                if (on(1, s) && !store(1, s, s, o)) return false;
                ++epoch;  // the step's barrier
            }
        } else {
            for (int s = x0 - (T - 1); s <= x1 + (T - 2); ++s) {
                const TbSlots o = tb_slots<B>(s, false);
                if (on(1, s) && !store(1, s, s, o)) return false;
                for (int k = 2; k <= T; ++k) {
                    ++epoch;  // the barrier before stage k
                    const int c = s - (k - 1);
                    if (!on(k, c)) continue;
                    if (!pull(k, c, s, o)) return false;
                    if (k < T && !store(k, c, s, o)) return false;
                }
            }
        }
        return true;
    }
};

// tb_ring_fill of every stage and row into a NaN ring: no double left unwritten, every pull of every step returns f
bool fill_reaches_every_slot(int T) {
    std::vector<double> ring(tb_ring_at<B>(T, 0, 0), std::numeric_limits<double>::quiet_NaN());
    double f[Q];
    for (int i = 0; i < Q; ++i) f[i] = 1.0 + i;
    for (int k = 1; k < T; ++k)
        for (int y = 0; y < B; ++y) tb_ring_fill<B>(ring.data() + y, k, f);
    for (size_t j = 0; j < ring.size(); ++j)
        if (ring[j] != ring[j]) {
            std::printf("depth %d: tb_ring_fill leaves ring double %zu unwritten\n", T, j);
            return false;
        }
    for (int skew = 0; skew < 2; ++skew)
        for (int s = -5; s < 13; ++s)
            for (int k = 1; k < T; ++k)
                for (int y = 1; y < B - 1; ++y) {
                    const TbSlots o = tb_slots<B>(s, skew != 0);
                    double g[Q];
                    tb_ring_pull<B>(ring.data() + y, k, o.pl[0], o.pl[1], o.pl[2], g);
                    for (int i = 0; i < Q; ++i)
                        if (g[i] != f[i]) {
                            std::printf("depth %d: after tb_ring_fill, step %d pulls %g for population %d\n", T, s, g[i], i);
                            return false;
                        }
                }
    return true;
}

}  // namespace

int main(int argc, char** argv) {
    if (argc > 1 && std::strcmp(argv[1], "bytes") == 0) {
        std::printf("%zu\n", (size_t)TbShape<3, 128>::RING_DOUBLES * sizeof(double));
        return 0;
    }
    for (int T = 2; T <= TB_MAX_DEPTH; ++T)
        if (!fill_reaches_every_slot(T)) return 1;
    long long pulls = 0;
    for (int skew = 0; skew < 2; ++skew)
        for (int T = 2; T <= TB_MAX_DEPTH; ++T)
            for (int x0 : {0, 5, 64})
                for (int w : {1, 2, 3, 4, 7, 64}) {
                    Replay r(T, skew != 0);
                    if (!r.chunk(x0, x0 + w)) return 1;
                    pulls += r.pulls;
                }
    std::printf("ok %lld\n", pulls);
    return 0;
}
