// Prints the route choose_standard_route takes for each query line on stdin:
//     B K D N derivative sms coeffs_aligned16 inputs_aligned16 forced     (forced: a route name or "-")
// Instantiates no kernel and needs no device (tests/test_standard_routes.py).
#include <cstdio>
#include <cstring>

#include "../../mav_trajectory_generation_cmake_b200/csrc/minsnap_standard_route.cuh"

int main() {
  using minsnap::StandardRoute;
  long B, sms;
  int K, D, N, derivative, coeffs_aligned, inputs_aligned;
  char forced[32];
  while (std::scanf("%ld %d %d %d %d %ld %d %d %31s", &B, &K, &D, &N, &derivative, &sms, &coeffs_aligned,
                    &inputs_aligned, forced) == 9) {
    minsnap::StandardRouteQuery q{B, K, D, N, derivative, sms, coeffs_aligned != 0, inputs_aligned != 0, {}};
    for (int r = 0; r < static_cast<int>(StandardRoute::Unsupported); ++r)
      if (std::strcmp(forced, minsnap::standard_route_name(static_cast<StandardRoute>(r))) == 0)
        q.forced = static_cast<StandardRoute>(r);
    std::printf("%s\n", minsnap::standard_route_name(minsnap::choose_standard_route(q)));
  }
  return 0;
}
