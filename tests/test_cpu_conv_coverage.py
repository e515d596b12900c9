"""The conv parity matrix cannot silently fall behind the library: every conv / pointwise kernel instance compiled into
libtwg.so (read from its symbol table) has a case in tests/conv_coverage.py, or is excluded there by name with a reason."""
import subprocess

from tests.conv_coverage import COVERAGE, EXCLUDED, canonical, instances_from_symbols


def _library_instances():
  from twingan_b200 import _lib
  out = subprocess.run(['nm', '--defined-only', _lib.LIB_PATH], check=True, capture_output=True, text=True).stdout
  return instances_from_symbols(out.splitlines())


def test_every_compiled_conv_instance_has_a_parity_case(built_lib):
  found = _library_instances()
  assert len(found) > 100, sorted(found)
  table = set(COVERAGE)
  assert not table & set(EXCLUDED), table & set(EXCLUDED)
  assert found == table | set(EXCLUDED), {'compiled, no case': sorted(found - table - set(EXCLUDED)),
                                          'in the table, not compiled': sorted((table | set(EXCLUDED)) - found)}
  for key, cases in COVERAGE.items():
    assert cases, key
  for key, why in EXCLUDED.items():
    assert why.strip(), key


def test_table_keys_are_canonical_and_cases_well_formed():
  for key, cases in COVERAGE.items():
    assert canonical(key) == key, key
    for c in cases:
      N, H, W, Ci, Co, k, pad = c.geom
      assert min(N, H, W, Ci, Co, k) > 0 and 0 <= pad < k, (key, c)
      assert set(c.opts) <= {1, 2, 3, 4, 6, 7, 8, 9}, (key, c)


def test_kernel_names_normalise_alike():
  """The profiler's demangled names and the symbol table's mangled ones map to the same key."""
  assert canonical('void twg::k_conv_fwd_tc<64, 128, false, 1>(CUtensorMap_st, CUtensorMap_st, float*)') == \
      'k_conv_fwd_tc<64,128,0,1>'
  assert canonical('void twg::k_conv_halo_tc<32, 16, 2, 0>(CUtensorMap_st const, int)') == 'k_conv_halo_tc<32,16,2,0>'
  assert canonical('twg::k_pw_expand(float const*, float const*, float*, long, int, int, int, int)') == 'k_pw_expand'
  assert canonical('void twg::k_split_act(float const*, __nv_bfloat16*, __nv_bfloat16*, long)') is None
  syms = ['0000000000123456 T _ZN3twg13k_conv_fwd_tcILi64ELi128ELb0ELi1EEEv14CUtensorMap_stS1_S1_S1_PfNS_6TcGeomEPKfiiPv',
          '0000000000123456 t _ZL56__device_stub__ZN3twg11k_pw_reduceILi2EEEvPKfS2_PfliiiiiPKfS0_Pfliiiii',
          '0000000000123456 T _ZN3twg11k_pw_expandEPKfS1_Pfliiii',
          '0000000000123456 T _ZN3twg11k_split_actEPKfP13__nv_bfloat16S3_l']
  assert instances_from_symbols(syms) == {'k_conv_fwd_tc<64,128,0,1>', 'k_pw_reduce<2>', 'k_pw_expand'}
