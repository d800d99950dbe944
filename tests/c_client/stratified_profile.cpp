// stratified_profile.cpp — EvaluationProfile::Stratified of include/echo_b200.hpp, driven from the CPU suite (tests/test_stratified.py):
// RenderParameters maps it to ECHO_DISTRIBUTION_STRATIFIED beside the evaluator's own bits, and Validate refuses an Extend the
// stratified sequence cannot take. Prints "stratified_profile ok".
#include <cstdio>
#include <cstring>

#include "echo_b200.hpp"

using namespace echo_b200;

static bool rejects(const EvaluationProfile& profile)
{
	try { profile.Validate(); }
	catch (const std::invalid_argument&) { return true; }
	return false;
}

int main()
{
	RenderTexture texture({ 40, 24 }, 8);
	EvaluationProfile uniform;
	EvaluationProfile stratified = uniform;
	stratified.Stratified = true;

	if (RenderParameters(uniform, texture).evaluator != ECHO_EVALUATOR_PATH_TRACED) return 2;
	if (RenderParameters(stratified, texture).evaluator != ECHO_DISTRIBUTION_STRATIFIED) return 3;

	EvaluationProfile albedo = stratified;
	albedo.Evaluator = ECHO_EVALUATOR_ALBEDO | ECHO_EVALUATOR_DIVERGE_ONCE;
	if (RenderParameters(albedo, texture).evaluator != (ECHO_EVALUATOR_ALBEDO | ECHO_EVALUATOR_DIVERGE_ONCE | ECHO_DISTRIBUTION_STRATIFIED)) return 4;

	EchoRenderParams a = RenderParameters(uniform, texture), b = RenderParameters(stratified, texture);
	b.evaluator = a.evaluator;
	if (std::memcmp(&a, &b, sizeof(a)) != 0) return 5; // the flag is the only difference

	EvaluationProfile largest = stratified, beyond = stratified, wide = uniform;
	largest.Extend = ECHO_DISTRIBUTION_STRATIFIED_EXTEND_MAX;
	beyond.Extend = ECHO_DISTRIBUTION_STRATIFIED_EXTEND_MAX + 1;
	wide.Extend = ECHO_DISTRIBUTION_STRATIFIED_EXTEND_MAX + 1;
	if (rejects(stratified) || rejects(largest) || !rejects(beyond) || rejects(wide)) return 6;

	std::printf("stratified_profile ok\n");
	return 0;
}
