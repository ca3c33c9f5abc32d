// erl.h -- elastic rate limit (ERL) controller, product side.
//
// The Go hypervisor runs this loop itself
// (pkg/hypervisor/worker/computing/quota_controller.go:378-458); the
// hypervisor-facing C-ABI of the limiter (provider/limiter.h:98-100,
// LimiterUpdateERL) exposes the same step so that a CGO-free host can hand it
// to the provider.  This is an independent restatement in C++ (the oracle's is
// oracle/erl_oracle.c); tests diff the two bit for bit.
#pragma once
#include <stdint.h>

#include <cmath>
#include <string>

#include "shm_quota.h"

namespace tferl {

struct Config {            // quota_controller.go:20-47,118-131
  double burst_window = 0.5;
  double rate_min = 10.0, rate_max = 200000.0;
  double capacity_min = 200.0, capacity_max = 200000.0;
  double util_alpha = 0.25;
  double kp = 0.9, ki = 0.35, kd = 0.10;
  double integral_decay = 0.85;
  // TF_HYPERVISOR_SCHEDULING_CONFIG JSON (:143-178); unknown / non-positive values keep defaults
  static Config from_json(const char* json);
};

struct State {             // erlState :64-70, initial values :253-268
  double current_rate = 100.0;
  double smoothed_util = 0.0;
  double integral_err = 0.0;
  double last_error = 0.0;
  bool initialized = false;
};

constexpr double kTickSeconds = 0.5;  // erlUpdateInterval

double slew(double current, double target, double up_ratio, double down_ratio);                 // :314-319
double desired_rate(double current_rate, double target, double smoothed, double dt, State& st,
                    const Config& cfg);                                                          // :321-347
double rebalance(tfq::QuotaFile& q, uint32_t idx, double now_secs, double rate, double capacity,
                 double target, double smoothed);                                                // :349-376
// One controller step for one (worker, device): EMA, rate, capacity, quota-file writes, rebalance.
// Returns the token balance after the step.
double tick(tfq::QuotaFile& q, uint32_t idx, State& st, const Config& cfg, uint32_t up_limit,
            double util_percent, double now_secs);                                               // :412-446
// controller.go:307-325.  Inline: the worker executable uses it without linking the controller (and QuotaFile).
inline uint32_t up_limit_percent(int64_t compute_percent, double tflops_limit, double max_tflops) {
  if (compute_percent > 0) return (uint32_t)compute_percent;
  if (tflops_limit > 0 && max_tflops > 0) {
    const double pct = std::ceil(tflops_limit / max_tflops * 100.0);
    if (pct < 1) return 1;
    if (pct > 100) return 100;
    return (uint32_t)pct;
  }
  return 100;
}

}  // namespace tferl
