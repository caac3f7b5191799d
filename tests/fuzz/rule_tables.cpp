// Harness of tests/test_rule_tables.py: the shared Philox4x32-10 and every form of the deficit-key order, printed from the
// headers the library compiles.
//   rule_tables c0 c1 c2 c3 k0 k1 [...]   one "philox" line per counter/key sextuple (hex), then the key tables
#include <cstdio>
#include <cstdlib>
#include "update_rule.hpp"

int main(int argc, char** argv) {
  for (int i = 1; i + 6 <= argc; i += 6) {
    uint32_t x[4], k[2];
    for (int j = 0; j < 4; j++) x[j] = (uint32_t)std::strtoul(argv[i + j], nullptr, 16);
    for (int j = 0; j < 2; j++) k[j] = (uint32_t)std::strtoul(argv[i + 4 + j], nullptr, 16);
    egm::philox4x32_10(x, k[0], k[1]);
    std::printf("philox %08x %08x %08x %08x uniform %.17g\n", x[0], x[1], x[2], x[3], egm::uniform53(x[0], x[1]));
  }
  for (uint32_t k = 0; k < 15; k++) std::printf("key_action %u %d\n", k, egrule::deficit_key_action(k));
  for (int c = 0; c < 256; c++) std::printf("action_key %d %d\n", c, egrule::deficit_key_of_action(c));
  std::printf("nibbles %llx %llx\n", (unsigned long long)egrule::kKeyOfType, (unsigned long long)egrule::kTypeOfKey);
  return 0;
}
