#!/bin/bash
# Builds stan/mock/run_stan_mock: stan/gp_lml_stan.hpp + the functional mock of Stan Math, linked against libgpb200.so.
set -e
cd "$(dirname "$0")/../.."
g++ -std=c++11 -O1 -g -Wall -Werror -Istan/mock stan/mock/run.cpp -Lgp_b200/lib -lgpb200 -Wl,-rpath,'$ORIGIN/../../gp_b200/lib' -o stan/mock/run_stan_mock
g++ -std=c++11 -O1 -g -Wall -Werror -Istan/mock stan/mock/run_groups.cpp -Lgp_b200/lib -lgpb200 -Wl,-rpath,'$ORIGIN/../../gp_b200/lib' -o stan/mock/run_stan_groups_mock
echo stan/mock/run_stan_mock stan/mock/run_stan_groups_mock
