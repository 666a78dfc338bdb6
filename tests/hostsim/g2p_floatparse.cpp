// g2p_floatparse — the gaffilter's float parse (parse_float_text, csrc/g2p_filter.cuh: how k_filter_parse reads gi:f:
// values) next to std::stof, which the reference reads them with.  TEST INFRASTRUCTURE ONLY.
//
// usage: g2p_floatparse < values      one value per line; prints "<product> <stof>" per line, each the float's bits in
//                                     hex or "throw" (product: false, i.e. the record aborts; stof: an exception)
#define HS_IMPLEMENTATION
#include "cuda_shim.hpp"

#include <iostream>
#include <string>

#include "../../cactus-gfa-tools_b200/csrc/g2p_kernels.cuh"

using namespace g2p;

static std::string bits(float f) {
    u32 u;
    std::memcpy(&u, &f, 4);
    char buf[16];
    std::snprintf(buf, sizeof buf, "%08x", u);
    return buf;
}

int main() {
    std::string line, out;
    while (std::getline(std::cin, line)) {
        float f = 0.f;
        out += parse_float_text(reinterpret_cast<const u8*>(line.data()), (u32)line.size(), f) ? bits(f) : "throw";
        out += ' ';
        try {
            out += bits(std::stof(line));
        } catch (const std::exception&) {
            out += "throw";
        }
        out += '\n';
    }
    std::fwrite(out.data(), 1, out.size(), stdout);
    return 0;
}
