// Host-side construction of the acquisition operator: sampling masks and the lookup
// tables the K1 kernel walks.  Header-only so the CPU emulation of K1 can share it.
//
// Mask constructors follow (maths only; written from scratch in C++):
//   main_files/subsampling_patterns/setup_subsampling_spiralgrided.m:7-34
//   main_files/subsampling_patterns/setup_subsampling_epi.m:20-30
#pragma once
#include <math.h>
#include <stdint.h>

#include <algorithm>
#include <vector>

namespace optab {

// MATLAB round(): halves away from zero
static inline double matlab_round(double x) { return x < 0 ? -floor(-x + 0.5) : floor(x + 0.5); }

// frames[i] = ascending 0-based column-major indices n + N*m (MATLAB find order - 1)
static inline void spiral_frames(int N, int S, int L, std::vector<std::vector<int32_t>>& frames) {
    const double PI = 3.14159265358979323846;
    const double delta = PI / 180.0 * 7.5;
    std::vector<double> theta(S), r(S);
    double rmin = 1e300, rmax = -1e300;
    for (int i = 0; i < S; ++i) {
        // linspace(0, 2*pi, S): MATLAB computes d1 + (0:n1)*(d2-d1)/n1 and pins the last point
        double t = (S > 1) ? (double)i * (2.0 * PI) / (double)(S - 1) : 2.0 * PI;
        if (i == S - 1) t = 2.0 * PI;
        theta[i] = 8.0 * t;
        r[i] = pow(1.05, theta[i]);
        rmin = std::min(rmin, r[i]);
        rmax = std::max(rmax, r[i]);
    }
    for (int i = 0; i < S; ++i) r[i] = (r[i] - rmin) / (rmax - rmin);
    frames.assign(L, {});
    std::vector<uint8_t> img((size_t)N * N);
    for (int f = 0; f < L; ++f) {
        std::fill(img.begin(), img.end(), 0);
        for (int i = 0; i < S; ++i) {
            double cx = r[i] * cos(theta[i] + f * delta);
            double cy = r[i] * sin(theta[i] + f * delta);
            double gx = matlab_round(cx * N / 2) + N / 2 + 1;
            double gy = matlab_round(cy * N / 2) + N / 2 + 1;
            gx = std::min(gx, (double)N);
            gy = std::min(gy, (double)N);
            int n = (int)gx - 1, m = (int)gy - 1;  // 0-based (row, col)
            // fftshift of an even-sized image: circular shift by N/2 in both dims
            int ns = (n + N / 2) % N, ms = (m + N / 2) % N;
            img[(size_t)ms * N + ns] = 1;
        }
        for (int k = 0; k < N * N; ++k)
            if (img[k]) frames[f].push_back(k);
    }
}

static inline void epi_frames(int N, int M, double percentage, int L, std::vector<std::vector<int32_t>>& frames) {
    int step = (int)matlab_round(1.0 / percentage);
    int no_of_steps = N / step;
    std::vector<uint8_t> comb(N, 0);
    for (int i = 0; i < step * no_of_steps; i += step) comb[i] = 1;
    frames.assign(L, {});
    for (int f = 0; f < L; ++f) {
        std::vector<uint8_t> sh(N);
        for (int n = 0; n < N; ++n) sh[(n + 1) % N] = comb[n];  // comb([N,1:N-1])
        comb = sh;
        for (int m = 0; m < M; ++m)
            for (int n = 0; n < N; ++n)
                if (comb[n]) frames[f].push_back(n + N * m);
    }
}

struct K1Tables {
    int C = 0, nmeas = 0, ns_max = 0;
    std::vector<int> frame_ptr;       // [C+1]
    std::vector<int32_t> idx;         // [nmeas]
    std::vector<uint16_t> samp;       // [nmeas]
    std::vector<uint32_t> p4tab;      // [C][8][p4_len] flat work lists of the sparse inverse pass (see build_k1_tables)
    int p4_len = 0;
    std::vector<float> tw;            // [N][2]
    // streaming kernel (xupdate_stream.cu): work items of the sparse m-direction sums (see build_stream_tables)
    bool stream_ok = false;           // false: some frame needs more than N items / too many overflow partials
    std::vector<uint32_t> itA;        // [C][N] k1 | cnt << 8 | start << 16   (cnt == 0: thread has no item; the word is then 255)
    std::vector<uint32_t> itB;        // [C][N] slot | novf << 8 | ovf0 << 16
    std::vector<uint32_t> ent;        // [nmeas] j | k2 << 16, frame-major, grouped by item
    std::vector<uint16_t> rowmask;    // [C][16] bit a of entry b: row R a + b (R = N / 16) holds samples (inverse FFT stage 1 skips empty rows)
    int n_ovf = 0;                    // largest number of overflow partials in one frame
    int max_row = 0;                  // largest number of samples in one row of one frame
    // real-image variant of the streaming kernels (xupdate_real.cu): the same work-item tables over FOLDED rows.  For a real image
    // the n-direction transform is Hermitian, T(N - k1, m) = conj T(k1, m), so a sample (k1 > N/2, k2) is carried by row N - k1 as
    // (N - k2) mod N with its value conjugated: entries j | k2' << 16 | conj << 31, rows 0 .. N/2 only.
    bool real_ok = false;             // N == 224 only
    std::vector<uint32_t> r_itA, r_itB, r_ent;
    std::vector<uint16_t> r_rowmask;  // [C][16] like rowmask, symmetric: row k and row N - k are set together
    int r_n_ovf = 0;
    std::vector<float> tw2;           // [16][16][2]  e^{-2 pi i (i j) / N}
    std::vector<float> tw448;         // [2N][2]      e^{-2 pi i t / (2N)} (448 entries at N = 224, 512 at N = 256)
};

constexpr int K1_PHASES = 8;          // row phases of the sparse inverse pass = THREADS / MC of the kernel
// p4tab entry: k2 | k1 << 8 | j << 16 | last_of_row << 31; j == ns_max addresses a zero coefficient (empty rows, padding)
static inline uint32_t p4_entry(int k2, int k1, int j, bool last) {
    return (uint32_t)k2 | ((uint32_t)k1 << 8) | ((uint32_t)j << 16) | (last ? 0x80000000u : 0u);
}


constexpr int STREAM_QMAX = 64;      // == k1::QMAX_STREAM
constexpr int STREAM_OVF_MAX = 96;   // == k1::OVF_MAX_STREAM

// Work items of the streaming kernel (N = 224 or 256 threads, one per k-space row).  Every item carries at least one sample, so
// cnt == 0 marks a thread without an item (k1 takes all 8 bits: row 255 is a real row at N = 256).
// The samples of a k-space row k1 are cut into chunks of at most Q samples (Q = the
// smallest value for which the frame needs no more than N items, so a thread never carries more than one); the row's first
// chunk is its PRIMARY item (it writes the row in the inverse pass), the others are OVERFLOW items whose partial sums go
// through numbered shared-memory slots and are added by the primary in slot order (deterministic, no atomics).  Rows
// without samples are zero-filled by a thread that is handed the row as a side duty.  Lane placement: thread 16 h + l takes
// an item of residue class l (k1 = l mod 16) whenever one is left, heaviest first, so the 16 lanes of a half-warp address 16
// different bank pairs in the [column][k1] workspace and the items of a warp carry similar sample counts.
// Core of the work-item construction for one frame: `rows[k]` holds the entry words of row k (any row numbering < N).
// Returns false when the frame does not fit (more than N items or too many overflow partials).
static inline bool stream_items_for_frame(int N, const std::vector<std::vector<uint32_t>>& rows, int q_min, int ent_base, uint32_t* itA,
                                          uint32_t* itB, std::vector<uint32_t>& ent, int& n_ovf) {
    struct Item { int k1, first, cnt, chunk, nchunks, ovf0; };
    int Q = 0;
    for (int q = std::max(1, q_min); q <= STREAM_QMAX && !Q; ++q) {
        int items = 0, ovf = 0;
        for (int k = 0; k < N; ++k) {
            int n = ((int)rows[k].size() + q - 1) / q;
            items += n;
            ovf += std::max(0, n - 1);
        }
        if (items <= N && ovf <= STREAM_OVF_MAX && ovf <= 254) Q = q;
    }
    if (!Q) return false;
    std::vector<Item> items;
    int slots = 0;
    for (int k = 0; k < N; ++k) {
        const int sz = (int)rows[k].size();
        if (!sz) continue;
        const int n = (sz + Q - 1) / Q;
        int first = 0;
        for (int ch = 0; ch < n; ++ch) {
            const int cnt = sz / n + (ch < sz % n ? 1 : 0);  // even split
            items.push_back({k, first, cnt, ch, n, slots});
            first += cnt;
        }
        slots += n - 1;
    }
    n_ovf = std::max(n_ovf, slots);
    // lane placement
    std::vector<std::vector<int>> bucket(16);
    for (int i = 0; i < (int)items.size(); ++i) bucket[items[i].k1 % 16].push_back(i);
    for (auto& b : bucket) std::stable_sort(b.begin(), b.end(), [&](int a, int b2) { return items[a].cnt > items[b2].cnt; });
    std::vector<int> place(N, -1), left;
    const int H = N / 16;
    for (int l = 0; l < 16; ++l)
        for (int h = 0; h < (int)bucket[l].size(); ++h) {
            if (h < H) place[16 * h + l] = bucket[l][h];
            else left.push_back(bucket[l][h]);
        }
    std::stable_sort(left.begin(), left.end(), [&](int a, int b2) { return items[a].cnt > items[b2].cnt; });
    for (int tid = 0, q = 0; tid < N && q < (int)left.size(); ++tid)
        if (place[tid] < 0) place[tid] = left[q++];
    // (rows without samples are skipped by the inverse FFT through `rowmask`: no zero fill)
    size_t pos = 0;
    for (int tid = 0; tid < N; ++tid) {
        uint32_t A = 255u, B = 0u;
        if (place[tid] >= 0) {
            const Item& it = items[place[tid]];
            A = (uint32_t)it.k1 | ((uint32_t)it.cnt << 8) | ((uint32_t)pos << 16);
            const int slot = it.chunk == 0 ? 0 : it.ovf0 + it.chunk;  // overflow slots are numbered from 1
            const int novf = it.chunk == 0 ? it.nchunks - 1 : 0;
            B |= (uint32_t)slot | ((uint32_t)novf << 8) | ((uint32_t)it.ovf0 << 16);
            for (int q = 0; q < it.cnt; ++q) ent[ent_base + pos++] = rows[it.k1][it.first + q];
        }
        itA[tid] = A;
        itB[tid] = B;
    }
    return true;
}

static inline void build_stream_tables(int N, const std::vector<std::vector<int32_t>>& frames, K1Tables& t, int q_min = 1) {
    t.stream_ok = N == 224 || N == 256;  // the sides the streaming kernels are instantiated for
    t.itA.assign((size_t)t.C * N, 255u);
    t.itB.assign((size_t)t.C * N, 0u);
    t.ent.assign(std::max(t.nmeas, 1), 0);
    t.rowmask.assign((size_t)t.C * 16, 0);
    t.n_ovf = 0;
    t.max_row = 0;
    t.real_ok = t.stream_ok && N == 224;
    t.r_itA.assign((size_t)t.C * N, 255u);
    t.r_itB.assign((size_t)t.C * N, 0u);
    t.r_ent.assign(std::max(t.nmeas, 1), 0);
    t.r_rowmask.assign((size_t)t.C * 16, 0);
    t.r_n_ovf = 0;
    if (!t.stream_ok) return;
    for (int c = 0; c < t.C; ++c) {
        const auto& f = frames[c];
        std::vector<std::vector<uint32_t>> rows(N), folded(N);
        for (int j = 0; j < (int)f.size(); ++j) {
            const int k1 = f[j] % N, k2 = f[j] / N;
            rows[k1].push_back((uint32_t)j | ((uint32_t)k2 << 16));
            if (2 * k1 <= N) folded[k1].push_back((uint32_t)j | ((uint32_t)k2 << 16));
            else folded[N - k1].push_back((uint32_t)j | ((uint32_t)((N - k2) % N) << 16) | 0x80000000u);
        }
        for (int k = 0; k < N; ++k) {
            t.max_row = std::max(t.max_row, (int)rows[k].size());
            if (!rows[k].empty()) t.rowmask[(size_t)c * 16 + k % (N / 16)] |= (uint16_t)(1u << (k / (N / 16)));
            if (!folded[k].empty() && N == 224) {
                const int kn = (N - k) % N;
                t.r_rowmask[(size_t)c * 16 + k % 14] |= (uint16_t)(1u << (k / 14));
                t.r_rowmask[(size_t)c * 16 + kn % 14] |= (uint16_t)(1u << (kn / 14));
            }
        }
        if (!stream_items_for_frame(N, rows, q_min, t.frame_ptr[c], t.itA.data() + (size_t)c * N, t.itB.data() + (size_t)c * N, t.ent, t.n_ovf)) {
            t.stream_ok = false;
            t.real_ok = false;
            return;
        }
        if (t.real_ok && !stream_items_for_frame(N, folded, q_min, t.frame_ptr[c], t.r_itA.data() + (size_t)c * N, t.r_itB.data() + (size_t)c * N,
                                                 t.r_ent, t.r_n_ovf))
            t.real_ok = false;
    }
}

static inline void build_k1_tables(int N, const std::vector<std::vector<int32_t>>& frames, K1Tables& t, int stream_q_min = 1) {
    t.C = (int)frames.size();
    t.frame_ptr.assign(t.C + 1, 0);
    for (int c = 0; c < t.C; ++c) t.frame_ptr[c + 1] = t.frame_ptr[c] + (int)frames[c].size();
    t.nmeas = t.frame_ptr[t.C];
    t.ns_max = 0;
    t.p4_len = 0;
    t.idx.clear();
    t.samp.clear();
    std::vector<std::vector<std::vector<uint32_t>>> lists(t.C, std::vector<std::vector<uint32_t>>(K1_PHASES));
    for (int c = 0; c < t.C; ++c) t.ns_max = std::max(t.ns_max, (int)frames[c].size());
    for (int c = 0; c < t.C; ++c) {
        const auto& f = frames[c];
        int ns = (int)f.size();
        std::vector<std::vector<std::pair<int, int>>> rows(N);  // per k1: (k2, j), ascending j keeps k2 ascending
        for (int j = 0; j < ns; ++j) {
            int k1 = f[j] % N, k2 = f[j] / N;
            t.idx.push_back(f[j]);
            t.samp.push_back((uint16_t)(k1 | (k2 << 8)));
            rows[k1].push_back({k2, j});
        }
        // Sparse inverse pass: every row k1 of the slab must be written (rows without samples with zero).  Rows are dealt
        // to K1_PHASES work lists of equal cost (largest first onto the lightest list); a thread owns one column and one
        // list and walks it with a single uniform loop: accumulate c_j e^{+2 pi i k2 m / N}, store at the row's last entry.
        std::vector<int> order(N);
        for (int k = 0; k < N; ++k) order[k] = k;
        std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return rows[a].size() > rows[b].size(); });
        std::vector<size_t> cost(K1_PHASES, 0);
        for (int k1 : order) {
            int ph = (int)(std::min_element(cost.begin(), cost.end()) - cost.begin());
            auto& L = lists[c][ph];
            if (rows[k1].empty()) {
                L.push_back(p4_entry(0, k1, t.ns_max, true));
            } else {
                for (size_t e = 0; e < rows[k1].size(); ++e)
                    L.push_back(p4_entry(rows[k1][e].first, k1, rows[k1][e].second, e + 1 == rows[k1].size()));
            }
            cost[ph] = L.size();
        }
        for (int ph = 0; ph < K1_PHASES; ++ph) t.p4_len = std::max(t.p4_len, (int)lists[c][ph].size());
    }
    t.p4tab.assign((size_t)t.C * K1_PHASES * t.p4_len, p4_entry(0, 0, t.ns_max, false));  // padding: adds zero, stores nothing
    for (int c = 0; c < t.C; ++c)
        for (int ph = 0; ph < K1_PHASES; ++ph)
            std::copy(lists[c][ph].begin(), lists[c][ph].end(), t.p4tab.begin() + ((size_t)c * K1_PHASES + ph) * t.p4_len);
    build_stream_tables(N, frames, t, stream_q_min);
    t.tw.resize(2 * N);
    const double PI = 3.14159265358979323846;
    t.tw448.resize(4 * N);
    for (int i = 0; i < 2 * N; ++i) {
        t.tw448[2 * i] = (float)cos(-PI * i / N);
        t.tw448[2 * i + 1] = (float)sin(-PI * i / N);
    }
    t.tw2.resize(2 * 256);
    for (int i = 0; i < 16; ++i)
        for (int j = 0; j < 16; ++j) {
            t.tw2[2 * (16 * i + j)] = (float)cos(-2.0 * PI * (i * j) / N);
            t.tw2[2 * (16 * i + j) + 1] = (float)sin(-2.0 * PI * (i * j) / N);
        }
    for (int i = 0; i < N; ++i) {
        t.tw[2 * i] = (float)cos(-2.0 * PI * i / N);
        t.tw[2 * i + 1] = (float)sin(-2.0 * PI * i / N);
    }
}

// ---- general V (SURVEY.md 7.3-1, 8f-2) ------------------------------------------------------------------------------------
// P = vertical stack of S_i kron(conj(V(i,:)), I): frame i samples sum_c V(i,c) X^_c on its own mask Omega_i.  The normal matrix
// is block diagonal in k-space: at location k the C x C block G_k = sum_{i: k in Omega_i} V(i,:)^T V(i,:).  All channels are
// therefore transformed on the UNION of the masks (one shared work-item table), and small per-location kernels mix channels.
constexpr int GENERAL_PART_MAX = 3400;   // union locations per part (shared memory: 12 bytes per location in the forward kernel)
struct GeneralTables {
    int L = 0, C = 0, nU = 0;
    std::vector<int32_t> ulist;        // [nU] union of the sampled locations, ascending k = k1 + N k2
    std::vector<int32_t> memb_ptr;     // [nU + 1] CSR over union locations
    std::vector<int32_t> memb_frame;   // [nmeas] frame i of each (location, frame) incidence
    std::vector<int32_t> memb_meas;    // [nmeas] its row in y (frame-major measurement index)
    std::vector<int32_t> meas_u;       // [nmeas] union slot of measurement j
    std::vector<int32_t> meas_frame;   // [nmeas] frame of measurement j
    std::vector<float> V;              // [L][C] row-major
    // The union is cut into contiguous parts (bands of k2) small enough for the streaming kernels' work-item tables and shared
    // memory; part p covers union slots [part_off[p], part_off[p+1]).  The transforms are linear in the mask, so the forward
    // kernel runs once per part and the adjoint passes accumulate.
    std::vector<K1Tables> parts;
    std::vector<int32_t> part_off;     // [P + 1]
    bool ok = false;
};

static inline void build_general_tables(int N, const std::vector<std::vector<int32_t>>& frames, const double* Vcm /*L x C col-major*/,
                                        int L, int C, GeneralTables& g, int stream_q_min = 1) {
    g.L = L;
    g.C = C;
    g.V.resize((size_t)L * C);
    for (int i = 0; i < L; ++i)
        for (int c = 0; c < C; ++c) g.V[(size_t)i * C + c] = (float)Vcm[i + (size_t)L * c];
    std::vector<uint8_t> seen((size_t)N * N, 0);
    for (const auto& f : frames)
        for (int32_t k : f) seen[k] = 1;
    g.ulist.clear();
    std::vector<int32_t> slot((size_t)N * N, -1);
    for (int k = 0; k < N * N; ++k)
        if (seen[k]) {
            slot[k] = (int32_t)g.ulist.size();
            g.ulist.push_back(k);
        }
    g.nU = (int)g.ulist.size();
    std::vector<std::vector<std::pair<int32_t, int32_t>>> inc(g.nU);
    g.meas_u.clear();
    g.meas_frame.clear();
    int32_t j = 0;
    for (int i = 0; i < L; ++i)
        for (int32_t k : frames[i]) {
            inc[slot[k]].push_back({i, j});
            g.meas_u.push_back(slot[k]);
            g.meas_frame.push_back(i);
            ++j;
        }
    g.memb_ptr.assign(g.nU + 1, 0);
    g.memb_frame.clear();
    g.memb_meas.clear();
    for (int u = 0; u < g.nU; ++u) {
        for (auto& e : inc[u]) {
            g.memb_frame.push_back(e.first);
            g.memb_meas.push_back(e.second);
        }
        g.memb_ptr[u + 1] = (int32_t)g.memb_frame.size();
    }
    // parts: as few as possible, each within the streaming kernels' limits
    g.ok = false;
    for (int P = std::max(1, (g.nU + GENERAL_PART_MAX - 1) / GENERAL_PART_MAX); P <= 32 && !g.ok; ++P) {
        g.parts.assign(P, K1Tables());
        g.part_off.assign(P + 1, 0);
        bool all = true;
        for (int pi = 0; pi < P; ++pi) {
            const int a = (int)((int64_t)g.nU * pi / P), b = (int)((int64_t)g.nU * (pi + 1) / P);
            g.part_off[pi] = a;
            g.part_off[pi + 1] = b;
            std::vector<std::vector<int32_t>> one(1, std::vector<int32_t>(g.ulist.begin() + a, g.ulist.begin() + b));
            build_k1_tables(N, one, g.parts[pi], stream_q_min);
            all = all && g.parts[pi].stream_ok;
        }
        g.ok = all;
    }
}

// (G_u + rho I)^{-1} for every union location, row-major C x C, computed in double (Gauss-Jordan with partial pivoting on an SPD matrix)
static inline void general_inverses(const GeneralTables& g, double rho, std::vector<float>& Minv) {
    const int C = g.C;
    Minv.assign((size_t)g.nU * C * C, 0.f);
    std::vector<double> A((size_t)C * 2 * C);
    for (int u = 0; u < g.nU; ++u) {
        for (int r = 0; r < C; ++r)
            for (int c = 0; c < 2 * C; ++c) A[(size_t)r * 2 * C + c] = (c == r ? rho : 0.0) + (c == C + r ? 1.0 : 0.0);
        for (int e = g.memb_ptr[u]; e < g.memb_ptr[u + 1]; ++e) {
            const float* v = &g.V[(size_t)g.memb_frame[e] * C];
            for (int r = 0; r < C; ++r)
                for (int c = 0; c < C; ++c) A[(size_t)r * 2 * C + c] += (double)v[r] * (double)v[c];
        }
        for (int col = 0; col < C; ++col) {
            int piv = col;
            for (int r = col + 1; r < C; ++r)
                if (fabs(A[(size_t)r * 2 * C + col]) > fabs(A[(size_t)piv * 2 * C + col])) piv = r;
            if (piv != col)
                for (int c = 0; c < 2 * C; ++c) std::swap(A[(size_t)piv * 2 * C + c], A[(size_t)col * 2 * C + c]);
            const double d = 1.0 / A[(size_t)col * 2 * C + col];
            for (int c = 0; c < 2 * C; ++c) A[(size_t)col * 2 * C + c] *= d;
            for (int r = 0; r < C; ++r) {
                if (r == col) continue;
                const double f = A[(size_t)r * 2 * C + col];
                if (f != 0.0)
                    for (int c = 0; c < 2 * C; ++c) A[(size_t)r * 2 * C + c] -= f * A[(size_t)col * 2 * C + c];
            }
        }
        for (int r = 0; r < C; ++r)
            for (int c = 0; c < C; ++c) Minv[((size_t)u * C + r) * C + c] = (float)A[(size_t)r * 2 * C + C + c];
    }
}

}  // namespace optab
