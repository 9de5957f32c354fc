// zkb.hpp mirror of the capture list: GpuBackend::capture / read_captured against GpuBackend::read_values, and against the
// values computed here, for a small program over p = 101 evaluated for 300 witnesses.
#include <cstdio>
#include <cstring>
#include <vector>

#include "zkb.hpp"

int main() {
    zkb::GpuBackend b(0);
    b.set_field(zkb::Value{101});
    auto x = b.witness(), y = b.witness();
    auto s = b.add(x, y);
    auto t = b.multiply(s, x);
    auto u = b.add_constant(t, zkb::Value{7});
    b.finalize(1);
    const std::vector<zkb::GpuBackend::Wire> wires = {x, y, s, t, u};
    b.capture(wires);
    const uint32_t n = 300;
    std::vector<uint8_t> wit(n * 2);
    for (uint32_t j = 0; j < n; j++) {
        wit[2 * j] = (uint8_t)(j % 101);
        wit[2 * j + 1] = (uint8_t)((3 * j + 1) % 101);
    }
    auto v = b.evaluate(nullptr, 0, wit.data(), 2, 1, n);
    if (v.size() != n) return 1;
    const size_t stride = 4;
    auto cap = b.read_captured(0, n, wires.size(), stride);
    for (uint32_t j = 0; j < n; j++) {
        const uint32_t a = wit[2 * j], c = wit[2 * j + 1], sum = (a + c) % 101, prod = sum * a % 101;
        const uint32_t want[5] = {a, c, sum, prod, (prod + 7) % 101};
        auto rv = b.read_values(j, wires, stride);
        for (size_t i = 0; i < wires.size(); i++) {
            const uint8_t* got = &cap[(j * wires.size() + i) * stride];
            const uint32_t g = got[0] | got[1] << 8 | got[2] << 16 | (uint32_t)got[3] << 24;
            if (g != want[i] || memcmp(got, &rv[i * stride], stride) != 0) {
                fprintf(stderr, "witness %u value %zu: captured %u, expected %u\n", j, i, g, want[i]);
                return 1;
            }
        }
    }
    auto part = b.read_captured(100, 5, wires.size(), stride);
    if (memcmp(part.data(), &cap[100 * wires.size() * stride], part.size()) != 0) return 1;
    printf("capture_api ok\n");
    return 0;
}
