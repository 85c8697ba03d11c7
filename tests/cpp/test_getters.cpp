// The members of the reference's taylor_adaptive_batch<T> added at the end of round 2 (include/heyoka/taylor.hpp:
// is_variational(), get_n_orig_sv(), get_dtime_data(), get_state_range(), get_pars_range(), get_te_cooldowns();
// continuous_output_batch::operator()(const T *)).
// Run by tests/test_zz_gpu_late_additions.py (needs a CUDA device: the class owns a device-resident batch).
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <limits>
#include <stdexcept>
#include <string>
#include <vector>

#include <heyoka_b200/heyoka_b200.hpp>

using namespace heyoka_b200;

static int n_fail = 0;
#define REQUIRE(cond)                                                                                                  \
    do {                                                                                                               \
        if (!(cond)) {                                                                                                 \
            std::printf("REQUIRE failed at %s:%d: %s\n", __FILE__, __LINE__, #cond);                                   \
            ++n_fail;                                                                                                  \
        }                                                                                                              \
    } while (0)

int main()
{
    auto [x, v] = make_vars("x", "v");
    using t_ev_t = t_event_batch<double>;

    // No events: plain getters; the ranges are writable views of the host mirrors, like the non-const data pointers.
    {
        taylor_adaptive_batch<double> ta{{prime(x) = v, prime(v) = -par[0] * sin(x)},
                                         {0.05, 0.06, 0.07, 0.08, 0.025, 0.026, 0.027, 0.028},
                                         4u,
                                         kw::pars = {9.8, 9.9, 10., 10.1},
                                         kw::time = {0.5, 1., 1.5, 2.}};
        REQUIRE(!ta.is_variational());
        REQUIRE(ta.get_n_orig_sv() == 2u && ta.get_n_orig_sv() == ta.get_dim());
        const auto [hi, lo] = ta.get_dtime_data();
        REQUIRE(hi == ta.get_time_data());
        for (int i = 0; i < 4; ++i) {
            REQUIRE(hi[i] == 0.5 * (i + 1) && lo[i] == 0.);
        }
        auto sr = ta.get_state_range();
        auto pr = ta.get_pars_range();
        REQUIRE(sr.size() == 8u && pr.size() == 4u && !sr.empty());
        REQUIRE(&*sr.begin() == ta.get_state_data() && &*pr.begin() == ta.get_pars_data());
        REQUIRE(sr[5] == 0.026 && pr[2] == 10.);
        // Writes through the ranges are picked up by the next step, like writes through get_state_data().
        taylor_adaptive_batch<double> tb = ta;
        for (auto &val : ta.get_state_range()) {
            val *= 2.;
        }
        ta.get_pars_range()[1] = 12.;
        for (std::size_t i = 0; i < 8u; ++i) {
            tb.get_state_data()[i] *= 2.;
        }
        tb.get_pars_data()[1] = 12.;
        ta.step();
        tb.step();
        REQUIRE(ta.get_state() == tb.get_state());
        REQUIRE(ta.get_last_h() == tb.get_last_h());
        REQUIRE(ta.get_dtime_data().first[3] == tb.get_time()[3]);
        bool thrown = false;
        try {
            (void)ta.get_te_cooldowns();
        } catch (const std::invalid_argument &e) {
            thrown = std::string(e.what()).find("No events were defined for this integrator") != std::string::npos;
        }
        REQUIRE(thrown);
    }
    // Terminal events without callbacks stop the lanes at v = 0 and start a cooldown there; an event that never
    // triggers stays out of cooldown; reset_cooldowns() clears the state.
    {
        taylor_adaptive_batch<double> ta{{prime(x) = v, prime(v) = -9.8 * sin(x)},
                                         {0, 0.01, 0.02, 0.03, .25, .26, .27, .28},
                                         4u,
                                         kw::t_events = {t_ev_t(v), t_ev_t(x - 100.)}};
        {
            const auto &cd0 = ta.get_te_cooldowns();
            REQUIRE(cd0.size() == 4u);
            for (const auto &lane : cd0) {
                REQUIRE(lane.size() == 2u && !lane[0] && !lane[1]);
            }
        }
        ta.propagate_for(100.);
        // (The lock-step loop ends at the first iteration in which a lane is stopped by its terminal event: a lane that
        // has not reached its own yet ends with `success` and no cooldown.)
        std::vector<bool> stopped(4u);
        unsigned n_stopped = 0;
        for (std::uint32_t i = 0; i < 4u; ++i) {
            const auto oc = std::get<0>(ta.get_propagate_res()[i]);
            stopped[i] = static_cast<std::int64_t>(oc) == -1;
            REQUIRE(stopped[i] || oc == taylor_outcome::success);
            n_stopped += stopped[i];
        }
        REQUIRE(n_stopped >= 3u);
        const auto before = ta.get_te_cooldowns(); // (a copy)
        REQUIRE(before.size() == 4u);
        for (std::uint32_t i = 0; i < 4u; ++i) {
            REQUIRE(before[i].size() == 2u && !before[i][1]);
            REQUIRE(static_cast<bool>(before[i][0]) == stopped[i]);
            if (before[i][0]) {
                // (time spent in cooldown, cooldown): just triggered, automatically deduced cooldown.
                REQUIRE(before[i][0]->first == 0.);
                REQUIRE(std::isfinite(before[i][0]->second) && before[i][0]->second > 0.);
            }
        }
        ta.reset_cooldowns(2u);
        {
            const auto &cd = ta.get_te_cooldowns();
            REQUIRE(!cd[2][0] && !cd[2][1]);
            for (std::uint32_t i : {0u, 1u, 3u}) {
                REQUIRE(cd[i] == before[i]);
            }
        }
        ta.reset_cooldowns();
        for (const auto &lane : ta.get_te_cooldowns()) {
            REQUIRE(!lane[0] && !lane[1]);
        }
    }
    // continuous_output_batch: the pointer overload of the call operator (include/heyoka/continuous_output.hpp:191).
    {
        taylor_adaptive_batch<double> ta{{prime(x) = v, prime(v) = -x}, {0., 0.1, 0.2, 0.3, 1., 1.1, 1.2, 1.3}, 4u};
        auto [co, cb] = ta.propagate_until(5., kw::c_output = true);
        REQUIRE(co.has_value());
        if (co) {
            const std::vector<double> tm{0.5, 1.5, 2.5, 4.75};
            const auto by_vec = (*co)(tm);
            const auto by_ptr = (*co)(tm.data());
            REQUIRE(by_vec == by_ptr && by_ptr.size() == 8u);
            // x(t) = x0 cos t + v0 sin t
            REQUIRE(std::abs(by_ptr[1] - (0.1 * std::cos(1.5) + 1.1 * std::sin(1.5))) < 1e-13);
            // get_times() / get_tcs() (include/heyoka/continuous_output.hpp:198-199): (n_steps + 2) rows of times (start,
            // the end of every iteration, the padding), [n_steps][dim][order + 1][batch] Taylor coefficients. At the
            // start of an iteration the output is the order-0 coefficients of that iteration: bit for bit at the
            // starting time 0; elsewhere get_times() holds the high parts of double-length times, and the output at
            // the high part is off by the low part lo (|lo| <= ulp(hi) / 2) times the order-1 coefficient, plus rounding.
            const auto n_steps = co->get_n_steps();
            const auto &tms = co->get_times();
            const auto &tcs = co->get_tcs();
            const std::size_t ord1 = ta.get_order() + 1u;
            REQUIRE(tms.size() == (n_steps + 2u) * 4u && tcs.size() == n_steps * 2u * ord1 * 4u);
            for (std::size_t i = 0; i < 4u; ++i) {
                REQUIRE(tms[i] == 0. && tms[n_steps * 4u + i] == 5. && std::isinf(tms[(n_steps + 1u) * 4u + i]));
            }
            const auto c_at = [&](std::size_t k, std::size_t var, std::size_t o, std::size_t i) {
                return tcs[((k * 2u + var) * ord1 + o) * 4u + i];
            };
            for (std::size_t k = 0; k < n_steps; ++k) {
                const auto out = (*co)(tms.data() + k * 4u);
                for (std::size_t var = 0; var < 2u; ++var) {
                    for (std::size_t i = 0; i < 4u; ++i) {
                        double amp = 0.;
                        for (std::size_t j = 0; j < n_steps; ++j) {
                            amp = std::max(amp, std::abs(c_at(j, var, 0, i)));
                        }
                        const double t = std::abs(tms[k * 4u + i]);
                        const double ulp = std::nextafter(t, std::numeric_limits<double>::infinity()) - t;
                        const double tol = std::abs(c_at(k, var, 1, i)) * ulp
                                           + 4. * std::numeric_limits<double>::epsilon() * amp;
                        REQUIRE(std::abs(out[var * 4u + i] - c_at(k, var, 0, i)) <= tol);
                        REQUIRE(k != 0u || out[var * 4u + i] == c_at(k, var, 0, i));
                    }
                }
            }
            // The last recorded iteration holds the integrator's current Taylor coefficients.
            const auto &tc = ta.get_tc();
            REQUIRE(tc.size() == 2u * ord1 * 4u);
            REQUIRE(std::equal(tc.begin(), tc.end(), tcs.end() - static_cast<std::ptrdiff_t>(tc.size())));
        }
    }
    // doc/tut_ensemble.rst (tutorial/ensemble.cpp), GOLDEN: ensemble_propagate_until(20) over the ten initial conditions
    // (0.05 + i / 100, 0.025 + i / 100); the reference prints member 9: state [0.12257736827306077,
    // 0.24068377640981869], 124 steps, time_limit. Here: five members of batch size 2 (member k holds the initial
    // conditions 2k and 2k + 1), through ensemble_propagate_until_batch().
    {
        taylor_adaptive_batch<double> ta{{prime(x) = v, prime(v) = -9.8 * sin(x)}, {0., 0., 0., 0.}, 2u};
        const auto gen = [](taylor_adaptive_batch<double> tc, std::size_t k) {
            for (std::size_t l = 0; l < 2u; ++l) {
                const auto i = static_cast<double>(2u * k + l);
                tc.get_state_data()[l] = 0.05 + i / 100.;
                tc.get_state_data()[2u + l] = 0.025 + i / 100.;
            }
            return tc;
        };
        const auto ret = ensemble_propagate_until_batch(ta, 20., 5u, gen);
        REQUIRE(ret.size() == 5u);
        if (ret.size() == 5u) {
            const auto &m = std::get<0>(ret[4]);
            REQUIRE(m.get_time()[1] == 20.);
            const auto &pr = m.get_propagate_res()[1];
            REQUIRE(std::get<0>(pr) == taylor_outcome::time_limit);
            REQUIRE(std::get<3>(pr) == 124u);
            REQUIRE(std::abs(std::get<1>(pr) - 0.158147) < 6e-7 && std::abs(std::get<2>(pr) - 0.167025) < 6e-7);
            REQUIRE(std::abs(m.get_state()[1] / 0.12257736827306077 - 1.) < 1e-12);
            REQUIRE(std::abs(m.get_state()[3] / 0.24068377640981869 - 1.) < 1e-12);
            REQUIRE(!std::get<1>(ret[4]).has_value());
        }
    }
    // test/taylor_adaptive_batch.cpp:2244-2267 ("empty init state", "scalar time ctor"): construction without initial
    // conditions gives a zeroed state; a scalar kw::time is splatted over the batch. A one-element state list still
    // means (state, batch size).
    {
        const auto dyn = model::pendulum();
        taylor_adaptive_batch<double> t0{dyn, 2u};
        REQUIRE((t0.get_state() == std::vector<double>{0., 0., 0., 0.}));
        taylor_adaptive_batch<double> t1{dyn, 2u, kw::time = 42};
        REQUIRE((t1.get_time() == std::vector<double>{42., 42.}));
        REQUIRE((t1.get_state() == std::vector<double>{0., 0., 0., 0.}));
        taylor_adaptive_batch<double> t2{{prime(x) = x}, {1.}, 1u};
        REQUIRE((t2.get_batch_size() == 1u && t2.get_state() == std::vector<double>{1.}));
    }
    // test/taylor_adaptive_batch.cpp:1864-1941 ("get_set_dtime"): sizes, normalisation and the reference's dtime_checks()
    // (finite components, |hi| >= |lo|), made before the times are touched.
    {
        taylor_adaptive_batch<double> ta{{prime(x) = v, prime(v) = -9.8 * sin(x)}, {0, 0.01, 0.1, 0.11}, 2u};
        const double eps = std::numeric_limits<double>::epsilon(), inf = std::numeric_limits<double>::infinity();
        ta.step();
        REQUIRE(ta.get_dtime().first[0] != 0. && ta.get_dtime().second[0] == 0.);
        const auto throws = [&](auto &&f, const char *msg) {
            try {
                f();
            } catch (const std::invalid_argument &e) {
                return std::string(e.what()).find(msg) != std::string::npos;
            }
            return false;
        };
        REQUIRE(throws([&] { ta.set_dtime(std::vector<double>{}, std::vector<double>{1.}); },
                       "the batch size is 2, but the number of specified times is (0, 1)"));
        ta.set_dtime({3., -7.}, {2., 5.});
        REQUIRE((ta.get_dtime().first == std::vector<double>{5., -2.} && ta.get_dtime().second == std::vector<double>{0., 0.}));
        ta.set_dtime(3., eps);
        REQUIRE((ta.get_dtime().first == std::vector<double>{3., 3.} && ta.get_dtime().second == std::vector<double>{eps, eps}));
        ta.set_dtime({3., 4.}, {1., 2.});
        const char *finite = "The components of the double-length representation of the time coordinate must both be finite";
        const char *order = "must not be smaller in magnitude than the second component";
        REQUIRE(throws([&] { ta.set_dtime(inf, 1.); }, finite));
        REQUIRE(throws([&] { ta.set_dtime(1., inf); }, finite));
        REQUIRE(throws([&] { ta.set_dtime(3., 4.); }, order));
        REQUIRE(throws([&] { ta.set_dtime({1., inf}, {1., 2.}); }, finite));
        REQUIRE(throws([&] { ta.set_dtime({1., 2.}, {1., 3.}); }, order));
        REQUIRE((ta.get_dtime().first == std::vector<double>{4., 6.} && ta.get_dtime().second == std::vector<double>{0., 0.}));
    }
    if (n_fail == 0) {
        std::printf("ALL PASSED (getters)\n");
    }
    return n_fail == 0 ? 0 : 1;
}
