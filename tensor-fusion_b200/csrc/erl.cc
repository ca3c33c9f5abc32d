// erl.cc -- see erl.h.  Built with -ffp-contract=off: Go/amd64 never fuses a*b+c.
#include "erl.h"

#include <cmath>
#include <cstdlib>
#include <cstring>

namespace tferl {

namespace {
constexpr double kDeadband = 0.03;          // utilDeadband
constexpr double kIntegralClamp = 1.5;
constexpr double kUpRatio = 0.35;           // maxRateIncreaseRatio
constexpr double kDownRatio = 0.25;         // maxRateDecreaseRatio
constexpr double kReserveRatio = 0.35;      // tokenReserveRatio
constexpr double kDrainRatio = 0.80;        // tokenDrainRatio
constexpr double kDrainMin = 25.0;          // tokenDrainMin

inline double clamp(double v, double lo, double hi) { return tfq::go_min(tfq::go_max(v, lo), hi); }

// value of "key":"<number>" inside the elasticRateLimitParameters object, or fallback
double positive_field(const std::string& obj, const char* key, double fallback) {
  const std::string pat = std::string("\"") + key + "\"";
  size_t k = obj.find(pat);
  if (k == std::string::npos) return fallback;
  k = obj.find(':', k + pat.size());
  if (k == std::string::npos) return fallback;
  const size_t q0 = obj.find('"', k);
  if (q0 == std::string::npos) return fallback;
  const size_t q1 = obj.find('"', q0 + 1);
  if (q1 == std::string::npos) return fallback;
  std::string v = obj.substr(q0 + 1, q1 - q0 - 1);
  const size_t a = v.find_first_not_of(" \t\r\n");
  if (a == std::string::npos) return fallback;
  const size_t b = v.find_last_not_of(" \t\r\n");
  v = v.substr(a, b - a + 1);
  char* end = nullptr;
  const double x = std::strtod(v.c_str(), &end);
  if (end == v.c_str() || *end != '\0' || !(x > 0)) return fallback;
  return x;
}
}  // namespace

Config Config::from_json(const char* json) {
  Config c;
  if (!json || !*json) return c;
  const std::string all(json);
  const size_t at = all.find("\"elasticRateLimitParameters\"");
  if (at == std::string::npos) return c;
  const size_t open = all.find('{', at);
  const size_t close = open == std::string::npos ? std::string::npos : all.find('}', open);
  if (close == std::string::npos) return c;
  const std::string obj = all.substr(open, close - open + 1);
  c.rate_max = positive_field(obj, "maxRefillRate", c.rate_max);
  c.rate_min = positive_field(obj, "minRefillRate", c.rate_min);
  c.util_alpha = positive_field(obj, "filterAlpha", c.util_alpha);
  c.kp = positive_field(obj, "kp", c.kp);
  c.ki = positive_field(obj, "ki", c.ki);
  c.kd = positive_field(obj, "kd", c.kd);
  c.burst_window = positive_field(obj, "burstWindow", c.burst_window);
  c.capacity_min = positive_field(obj, "capacityMin", c.capacity_min);
  c.capacity_max = positive_field(obj, "capacityMax", c.capacity_max);
  c.integral_decay = positive_field(obj, "integralDecayFactor", c.integral_decay);
  if (c.rate_min > c.rate_max) c.rate_min = c.rate_max;
  if (c.capacity_min > c.capacity_max) c.capacity_min = c.capacity_max;
  c.util_alpha = clamp(c.util_alpha, 0.01, 0.95);
  c.integral_decay = clamp(c.integral_decay, 0.01, 0.999);
  return c;
}

double slew(double current, double target, double up_ratio, double down_ratio) {
  return target > current ? tfq::go_min(target, current * (1.0 + up_ratio))
                          : tfq::go_max(target, current * (1.0 - down_ratio));
}

double desired_rate(double current_rate, double target, double smoothed, double dt, State& st, const Config& cfg) {
  if (smoothed <= 0.01) return tfq::go_min(current_rate * (1.0 + kUpRatio), cfg.rate_max);  // idle: ramp up
  const double err = target - smoothed;
  if (std::fabs(err) < kDeadband) {
    st.integral_err *= cfg.integral_decay;
    return current_rate;
  }
  st.integral_err = clamp(st.integral_err * cfg.integral_decay + err * dt, -kIntegralClamp, kIntegralClamp);
  const double deriv = dt > 0 ? (err - st.last_error) / dt : 0.0;
  st.last_error = err;
  const double feed_forward = current_rate * (target / tfq::go_max(smoothed, 0.05));
  const double factor = clamp(1.0 + cfg.kp * err + cfg.ki * st.integral_err + cfg.kd * deriv, 0.5, 1.5);
  return slew(current_rate, clamp(feed_forward * factor, cfg.rate_min, cfg.rate_max), kUpRatio, kDownRatio);
}

double rebalance(tfq::QuotaFile& q, uint32_t idx, double now_secs, double rate, double capacity, double target,
                 double smoothed) {
  double tokens = q.tokens(idx);
  const double last = q.last_update(idx);
  if (last > 0) {
    const double elapsed = now_secs - last;
    if (elapsed > 0 && elapsed < 5.0) {
      q.fetch_add(idx, rate * elapsed);
      tokens = q.tokens(idx);
    }
  }
  const double reserve = clamp(capacity * kReserveRatio, 0.0, capacity);
  const double drain = tfq::go_max(kDrainMin, capacity * kDrainRatio) * kTickSeconds;
  if (tokens > capacity) {
    tokens = tfq::go_max(capacity, tokens - drain);
    q.set_tokens(idx, tokens);
  } else if (smoothed > target + kDeadband && tokens > reserve) {
    tokens = tfq::go_max(reserve, tokens - drain);
    q.set_tokens(idx, tokens);
  }
  q.set_last_update(idx, now_secs);
  return tokens;
}

double tick(tfq::QuotaFile& q, uint32_t idx, State& st, const Config& cfg, uint32_t up_limit, double util_percent,
            double now_secs) {
  const double target = (double)up_limit / 100.0;
  const double util = util_percent / 100.0;
  if (!st.initialized) {
    st.smoothed_util = util;
    st.initialized = true;
  } else {
    st.smoothed_util = cfg.util_alpha * util + (1 - cfg.util_alpha) * st.smoothed_util;
  }
  st.current_rate = desired_rate(st.current_rate, target, st.smoothed_util, kTickSeconds, st, cfg);
  const double capacity = clamp(st.current_rate * cfg.burst_window, cfg.capacity_min, cfg.capacity_max);
  q.set_rate(idx, st.current_rate);
  q.set_capacity(idx, capacity);
  return rebalance(q, idx, now_secs, st.current_rate, capacity, target, st.smoothed_util);
}

}  // namespace tferl
