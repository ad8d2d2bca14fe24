// Reference for the edit-distance search (sccg_archive_search_edits, include/sccg.h), written from the header's contract alone:
// an O(m * n) Sellers DP per window, pattern and strand with the 256 x 256 match rule, and for every end within k edits the
// largest start found by computing ed(P, D[x:e]) anew for each x from e down to max(window start, e - m - k).
//
// Input (one file, argv[1]):  "k strands" / n_patterns / one pattern per line in hex / n_sequences / one D per line in hex /
// n_windows / "sequence start end" per line.  Output: one hit per line, "window start end pattern strand edits", in the order
// windows, patterns, strands, ends (the caller sorts).
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <fstream>
#include <string>
#include <vector>

static bool M[256][256];

static int up(int b) { return b >= 'a' && b <= 'z' ? b - 32 : b; }

static void match_table() {
    const char* codes[] = {"RAG", "YCT", "SCG", "WAT", "KGT", "MAC", "BCGT", "DAGT", "HACT", "VACG", "NACGT"};
    for (int p = 0; p < 256; ++p)
        for (int d = 0; d < 256; ++d) {
            bool m = up(d) == up(p);
            for (const char* c : codes)
                if (up(p) == c[0])
                    for (const char* q = c + 1; *q; ++q) m = m || up(d) == *q;
            M[p][d] = m;
        }
}

static int comp(int c) {
    const char* pairs = "ATCGRYKMBVDH";
    for (int i = 0; pairs[i]; ++i) {
        if (c == pairs[i]) return pairs[i ^ 1];
        if (c == pairs[i] + 32) return pairs[i ^ 1] + 32;
    }
    return c;
}

static std::string unhex(const std::string& h) {
    std::string s(h.size() / 2, '\0');
    for (size_t i = 0; i < s.size(); ++i) s[i] = (char)std::stoi(h.substr(2 * i, 2), nullptr, 16);
    return s;
}

// ed(P, T): both ends anchored
static int edit_distance(const std::string& P, const unsigned char* T, int n) {
    const int m = (int)P.size();
    std::vector<int> prev(m + 1), cur(m + 1);
    for (int i = 0; i <= m; ++i) prev[i] = i;
    for (int y = 0; y < n; ++y) {
        cur[0] = y + 1;
        for (int i = 1; i <= m; ++i)
            cur[i] = std::min({prev[i - 1] + !M[(unsigned char)P[i - 1]][T[y]], prev[i] + 1, cur[i - 1] + 1});
        std::swap(prev, cur);
    }
    return prev[m];
}

int main(int argc, char** argv) {
    if (argc != 2) { fprintf(stderr, "usage: edit_probe <input>\n"); return 2; }
    match_table();
    std::ifstream in(argv[1]);
    int k, strands, np, nd;
    long nw;
    in >> k >> strands >> np;
    std::vector<std::string> pats(np);
    for (auto& p : pats) { std::string h; in >> h; p = unhex(h); }
    in >> nd;
    std::vector<std::string> Ds(nd);
    for (auto& d : Ds) { std::string h; in >> h; d = h == "-" ? std::string() : unhex(h); }
    in >> nw;
    for (long w = 0; w < nw; ++w) {
        long a, s, e;
        in >> a >> s >> e;
        const unsigned char* D = (const unsigned char*)Ds[a].data();
        for (int i = 0; i < np; ++i)
            for (int st = 0; st < 2; ++st) {
                if (!((strands >> st) & 1)) continue;
                std::string P = pats[i];
                if (st) { std::reverse(P.begin(), P.end()); for (auto& c : P) c = (char)comp((unsigned char)c); }
                const int m = (int)P.size();
                // Sellers: C[i] = min over x of ed(P[0:i], D[x:y]) with x free
                std::vector<int> C(m + 1), N(m + 1);
                for (int r = 0; r <= m; ++r) C[r] = r;
                for (long y = s; y < e; ++y) {
                    N[0] = 0;
                    for (int r = 1; r <= m; ++r) N[r] = std::min({C[r - 1] + !M[(unsigned char)P[r - 1]][D[y]], C[r] + 1, N[r - 1] + 1});
                    std::swap(C, N);
                    if (C[m] > k) continue;
                    const long end = y + 1;
                    long start = -1;
                    for (long x = end; x >= std::max(s, end - m - k); --x)
                        if (edit_distance(P, D + x, (int)(end - x)) == C[m]) { start = x; break; }
                    printf("%ld %ld %ld %d %d %d\n", w, start, end, i, st, C[m]);
                }
            }
    }
    return 0;
}
