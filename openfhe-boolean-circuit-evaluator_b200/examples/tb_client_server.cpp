// tb_client_server.cpp -- evaluation without the secret key, through host/binfhecontext.h and host/circuit.h.
// The key holder (client) generates the keys on the host and hands the evaluator (server) the evaluation keys only; the evaluator runs
// an adder circuit on the holder's ciphertexts on the GPU and returns ciphertexts; the holder decrypts and checks them against a ripple
// adder computed in plain C++.  Exit code 0 and "ALL PASSED" when every check passes.
//     usage: tb_client_server <adder .out file> [-s TOY|STD128_OPT] [-m AP|GINX] [-n loops]
#include "../host/circuit.h"
#include <cstdio>
#include <cstring>

int main(int argc, char **argv) {
  if (argc < 2) { std::fprintf(stderr, "usage: %s <adder .out file> [-s set] [-m method] [-n loops]\n", argv[0]); return 2; }
  lbcrypto::BINFHE_PARAMSET set = lbcrypto::STD128_OPT;
  lbcrypto::BINFHE_METHOD method = lbcrypto::GINX;
  unsigned loops = 4;
  for (int i = 2; i + 1 < argc; i += 2) {
    if (!std::strcmp(argv[i], "-s")) set = !std::strcmp(argv[i + 1], "TOY") ? lbcrypto::TOY : lbcrypto::STD128_OPT;
    else if (!std::strcmp(argv[i], "-m")) method = !std::strcmp(argv[i + 1], "AP") ? lbcrypto::AP : lbcrypto::GINX;
    else if (!std::strcmp(argv[i], "-n")) loops = (unsigned)std::atoi(argv[i + 1]);
  }
  // key holder: no GPU needed, keys from OS entropy
  lbcrypto::BinFHEContext holder;
  holder.GenerateBinFHEContext(set, method, -1);
  auto sk = holder.KeyGen();
  holder.BTKeyGen(sk);
  const std::vector<uint8_t> eval_keys = holder.ExportKeys(false);

  // evaluator: the evaluation keys, no secret key
  lbcrypto::BinFHEContext server;
  server.GenerateBinFHEContext(set, method, 0);
  server.ImportKeys(eval_keys);
  Circuit circ(server);
  if (!circ.ReadFile(argv[1])) return 1;
  uint32_t nin = 0, bits[8], nout = 0;
  bfhe_circuit_info(circ.raw(), &nin, bits, &nout, nullptr, nullptr, nullptr, nullptr);
  if (nin != 2 || bits[0] != bits[1] || nout != bits[0] + 1) { std::fprintf(stderr, "not an adder circuit\n"); return 2; }
  const unsigned n = bits[0];

  bool passed = true;
  for (unsigned t = 0; t < loops; t++) {
    srand(t);
    std::vector<unsigned> in1(n), in2(n);
    std::vector<std::vector<lbcrypto::LWECiphertext>> cts(2);
    for (unsigned ix = 0; ix < n; ix++) {
      in1[ix] = rand() % 2;
      in2[ix] = rand() % 2;
      cts[0].push_back(holder.Encrypt(sk, in1[ix], lbcrypto::FRESH)); // level 0 of the circuit bootstraps them
      cts[1].push_back(holder.Encrypt(sk, in2[ix], lbcrypto::FRESH));
    }
    std::vector<unsigned> golden(n + 1, 0);
    unsigned c = 0;
    for (unsigned ix = 0; ix < n; ix++) {
      unsigned a = in1[ix], b = in2[ix], tmp = a ^ b;
      golden[ix] = c ^ tmp;
      c = (a & b) | (c & tmp);
    }
    golden[n] = c;
    circ.Reset();
    circ.setEncrypted(true);
    circ.SetInput(cts);
    const std::vector<lbcrypto::LWECiphertext> out = circ.ClockCiphertexts();
    bool ok = out.size() == n + 1;
    for (unsigned ix = 0; ok && ix <= n; ix++) {
      lbcrypto::LWEPlaintext r = 0;
      holder.Decrypt(sk, out[ix], &r);
      ok = (unsigned)r == golden[ix];
    }
    std::printf("test %u %s\n", t, ok ? "passed" : "FAILED");
    passed = passed && ok;
  }
  // the evaluator cannot decrypt
  bool threw = false;
  try {
    lbcrypto::LWEPlaintext r;
    server.Decrypt(sk, holder.Encrypt(sk, 1, lbcrypto::FRESH), &r);
  } catch (const std::exception &) {
    threw = true;
  }
  passed = passed && threw;
  std::printf("%s\n", passed ? "ALL PASSED" : "SOME FAILED");
  return passed ? 0 : 1;
}
