// Test probe: the record-body token loop of the reference's reconstruct_genome (decompression.cpp:210-236) with the real
// std::string::find, substr and std::stoi of libstdc++, exceptions caught.  It gives test_emu_token_grammar.py a witness
// for the oracle's restatement (orc_reconstruct with its orc_stoi) that does not rest on that restatement.
//
//   stoi_probe <cases>    one case per line: "<reference hex> <body hex>"
// prints one line per case: "ok <decoded record hex>" (token decode only: no run lists, no 50-column wrap), or
// "fail <class>" with class invalid_argument / out_of_range (stoi or substr threw), bounds (the reference's
// "exceeds reference genome size" exit) or endless (a token without ')': the reference's loop starts over at 0).
#include <cstdio>
#include <fstream>
#include <iostream>
#include <stdexcept>
#include <string>

static std::string unhex(const std::string& h) {
    std::string s;
    for (size_t i = 0; i + 1 < h.size(); i += 2) s.push_back((char)std::stoi(h.substr(i, 2), nullptr, 16));
    return s;
}

static std::string hex(const std::string& s) {
    static const char* d = "0123456789abcdef";
    std::string h;
    for (unsigned char c : s) { h.push_back(d[c >> 4]); h.push_back(d[c & 15]); }
    return h;
}

// the loop as decompression.cpp:210-236 writes it; int arithmetic wraps (built with -fwrapv)
static std::string decode(const std::string& ref, const std::string& enc) {
    std::string rec;
    size_t i = 0;
    int prev_abs_start = 0;
    while (i < enc.size()) {
        if (enc[i] == '(') {
            size_t end_pos = enc.find(')', i);
            size_t comma_pos = enc.find(',', i);
            int delta = std::stoi(enc.substr(i + 1, comma_pos - i - 1));
            int length = std::stoi(enc.substr(comma_pos + 1, end_pos - comma_pos - 1));
            int absolute_start = prev_abs_start + delta;
            prev_abs_start = absolute_start;
            if (absolute_start + length > (int)ref.size()) return "fail bounds";
            rec += ref.substr(absolute_start, length);
            if (end_pos == std::string::npos) return "fail endless";
            i = end_pos + 1;
        } else {
            rec += enc[i];
            ++i;
        }
    }
    return "ok " + hex(rec);
}

int main(int argc, char** argv) {
    if (argc != 2) { std::fprintf(stderr, "usage: stoi_probe <cases>\n"); return 2; }
    std::ifstream in(argv[1], std::ios::binary);
    std::string line;
    while (std::getline(in, line)) {
        const size_t sp = line.find(' ');
        const std::string ref = unhex(line.substr(0, sp)), enc = unhex(line.substr(sp + 1));
        std::string r;
        try {
            r = decode(ref, enc);
        } catch (const std::invalid_argument&) {
            r = "fail invalid_argument";
        } catch (const std::out_of_range&) {
            r = "fail out_of_range";
        }
        std::cout << r << '\n';
    }
    return 0;
}
